"""Generate tests/golden/reference_networks.json: the state-dict layout ([parameter name, shape] in state-dict order) of
the reference's two networks (utils/network.py: LightActorCritic, ActorCritic at (4, 42, 42) and 3 actions) and of the
"model" state dict in each of its shipped checkpoints (resources/pong/checkpoint-{weak,medium}.pkl).  Needs the
reference tree (CRL_REFERENCE_ROOT).

The trained weights stay the reference's data and are not stored.  What the tests pin with this file: our networks load
every layout strictly (the names DevicePolicy needs to load the real checkpoint files), and the tournament fixture's
synthetic weights are assigned in the reference's own parameter order (tests/test_builtin_policies.py)."""
import importlib.util
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_loader  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden", "reference_networks.json")


def layout(state_dict):
    return [[name, list(p.shape)] for name, p in state_dict.items()]


def main():
    import torch
    root = ref_loader.REFERENCE_ROOT
    spec = importlib.util.spec_from_file_location("_ref_network", os.path.join(root, "competitive_rl", "utils", "network.py"))
    R = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(R)            # the file imports torch only
    out = {"LightActorCritic": layout(R.LightActorCritic((4, 42, 42), 3).state_dict()),
           "ActorCritic": layout(R.ActorCritic((4, 42, 42), 3).state_dict())}
    for name in ("weak", "medium"):
        ckpt = torch.load(os.path.join(root, "resources", "pong", "checkpoint-%s.pkl" % name), map_location="cpu",
                          weights_only=False)
        out["checkpoint-%s.pkl" % name] = layout(ckpt["model"])
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", OUT, {k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
