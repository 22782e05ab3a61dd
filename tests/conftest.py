import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")
ATLAS = os.path.join(ROOT, "competitive-rl_b200", "data", "scoreboard_atlas.npz")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def atlas():
    import numpy as np
    return np.load(ATLAS)["strips"]


def load_golden(name):
    import numpy as np
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def reference_layout(key):
    """[(parameter name, shape)] in state-dict order of the reference's network or checkpoint `key`
    (tests/golden/reference_networks.json, oracle/gen_golden_networks.py)."""
    import json
    with open(os.path.join(GOLDEN, "reference_networks.json")) as f:
        return [(name, tuple(shape)) for name, shape in json.load(f)[key]]


def synthetic_state_dict(layout):
    """The weights of tests/golden/tournament_synth.npz: parameter k of `layout` ([(name, shape)] in state-dict order),
    element i = float32(0.08 * sin(0.37 * i + k))."""
    import numpy as np
    import torch
    sd = {}
    for k, (name, shape) in enumerate(layout):
        i = np.arange(int(np.prod(shape)), dtype=np.float64)
        sd[name] = torch.from_numpy((0.08 * np.sin(0.37 * i + k)).astype(np.float32).reshape(tuple(shape)))
    return sd
