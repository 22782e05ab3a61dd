"""Real 84x84 Pong observation frames for compressible_store_probe.cu, from the CPU oracle: 128 cPongDouble envs under
random actions, both agents' 4-frame stacks taken every 50 steps up to step 200, written as raw uint8 frames.
    python tools/probes/oracle_frames.py frames.bin"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
from pong_oracle import PongOracleVec, make_serve_table  # noqa: E402

N, STEPS, EVERY = 128, 200, 50
atlas = np.load(os.path.join(ROOT, "competitive-rl_b200", "data", "scoreboard_atlas.npz"))["strips"]
env = PongOracleVec("cPongDouble-v0", N, 84, 4, 21, atlas, make_serve_table(N, 64, seed=1))
env.reset()
rng = np.random.default_rng(0)
frames = []
for t in range(1, STEPS + 1):
    obs, _, _, _ = env.step(rng.integers(0, 3, (N, 2)).astype(np.int32))
    if t % EVERY == 0:
        frames += [obs[0].reshape(-1, 84, 84), obs[1].reshape(-1, 84, 84)]
out = np.ascontiguousarray(np.concatenate(frames))
out.tofile(sys.argv[1])
print("%d frames, %.1f %% zero bytes, %.1f %% 255 bytes -> %s" % (len(out), 100 * (out == 0).mean(), 100 * (out == 255).mean(), sys.argv[1]))
