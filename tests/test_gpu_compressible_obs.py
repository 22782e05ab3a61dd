"""Pong observation buffers in compressible memory (crl_obs_alloc / crl_obs_free, ext.obs_empty): what the device grants,
that the vec-env's buffers come from there, that the rasterisers write the same bytes into it as into ordinary memory,
that copies out of it return those bytes, and that closing an env gives the memory back."""
import ctypes
import gc

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

# CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED (cuda.h)
GENERIC_COMPRESSION_SUPPORTED = 107


@pytest.fixture(scope="module")
def lib():
    from competitive_rl_b200 import _native
    return _native.load()


@pytest.fixture(scope="module")
def ext():
    from competitive_rl_b200 import _native
    return _native.ext()


@pytest.fixture(scope="module")
def supported(lib):
    """whether the device supports generic memory compression (the B200 does)"""
    cudart = ctypes.CDLL("libcudart.so.12")
    v = ctypes.c_int(0)
    assert cudart.cudaDeviceGetAttribute(ctypes.byref(v), GENERIC_COMPRESSION_SUPPORTED, 0) == 0
    return v.value != 0


def test_obs_alloc_grants_compressible_memory(lib, supported):
    name = torch.cuda.get_device_name(0)
    p, comp = ctypes.c_void_p(), ctypes.c_int32(-1)
    assert lib.crl_obs_alloc(0, 3 << 20, ctypes.byref(p), ctypes.byref(comp)) == 0, lib.crl_last_error()
    try:
        assert p.value and p.value % 16 == 0
        if not supported:
            assert comp.value == 0
            pytest.skip("%s does not support generic memory compression: ordinary memory" % name)
        assert comp.value == 1, "%s supports generic compression but did not grant it (driver: ordinary memory)" % name
    finally:
        assert lib.crl_obs_free(p) == 0, lib.crl_last_error()
    assert lib.crl_obs_free(None) == 0
    bad = torch.empty(16, dtype=torch.uint8, device="cuda")
    assert lib.crl_obs_free(ctypes.c_void_p(bad.data_ptr())) != 0     # not one of crl_obs_alloc's


@pytest.mark.parametrize("stack_mode", ["stack", "ring"])
def test_make_envs_buffers_come_from_obs_alloc(stack_mode, supported):
    from competitive_rl_b200 import make_envs
    env = make_envs("cPongDouble-v0", num_envs=64, resized_dim=84, frame_stack=4, log_dir=None, stack_mode=stack_mode)
    assert env.obs_compressed == supported
    env.close()


def _zeroed(ext, shape, compressible):
    t, comp = ext.obs_empty(list(shape), torch.uint8, 0, compressible)
    t.zero_()
    return t, comp


@pytest.mark.parametrize("dim,stack_mode", [(84, "stack"), (84, "ring"), (42, "stack"), (42, "ring")])
def test_render_into_compressible_equals_ordinary(dim, stack_mode, lib, ext, supported):
    from competitive_rl_b200 import make_envs
    N, C = 4096, 4
    env = make_envs("cPongDouble-v0", num_envs=N, resized_dim=dim, frame_stack=C, log_dir=None, seed=7,
                    stack_mode=stack_mode, max_num_rounds=2)
    env.reset()
    rng = np.random.default_rng(1)
    for _ in range(60):
        env.step(rng.integers(0, 3, (N, 2)))
    shape = (N, 2 * C if stack_mode == "ring" else C, dim, dim)
    out = {}
    for compressible in (True, False):
        bufs = [_zeroed(ext, shape, compressible) for _ in range(2)]
        assert all(c == (compressible and supported) for _, c in bufs)
        s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        rc = lib.crl_pong_render_obs(env._h, ctypes.c_void_p(bufs[0][0].data_ptr()), ctypes.c_void_p(bufs[1][0].data_ptr()), s)
        assert rc == 0, lib.crl_last_error()
        torch.cuda.synchronize()
        out[compressible] = [b.cpu().numpy() for b, _ in bufs]
    for k in range(2):
        assert out[False][k].any()
        assert np.array_equal(out[True][k], out[False][k]), k
    env.close()


def test_copies_out_of_compressible_memory(ext):
    shape = (4096, 4, 84, 84)
    g = torch.Generator().manual_seed(3)
    src = torch.randint(0, 256, shape, dtype=torch.uint8, generator=g)
    src[: shape[0] // 2] = 0                          # half constant (compresses), half random bytes (does not)
    src[: shape[0] // 4, :, 10:20] = 255
    t, _ = ext.obs_empty(list(shape), torch.uint8, 0)
    t.copy_(src.cuda())
    assert torch.equal(t.cpu(), src)
    pinned = torch.empty(shape, dtype=torch.uint8, pin_memory=True)
    pinned.copy_(t, non_blocking=True)               # cudaMemcpyAsync into page-locked memory
    torch.cuda.synchronize()
    assert torch.equal(pinned, src)
    v = t[100:200, 1:3]                               # a strided view of the buffer
    assert torch.equal(v.cpu(), src[100:200, 1:3])


def test_close_gives_the_memory_back(ext):
    from competitive_rl_b200 import make_envs
    N, C, D = 16384, 4, 84
    obs_bytes = 2 * 2 * N * C * D * D                # two buffer sets (n_buffers=2) x two agents
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    env = make_envs("cPongDouble-v0", num_envs=N, resized_dim=D, frame_stack=C, log_dir=None)
    obs = env.reset()
    torch.cuda.synchronize()
    free1 = torch.cuda.mem_get_info(0)[0]
    assert free0 - free1 >= 0.9 * obs_bytes
    del obs
    env.close()
    del env
    gc.collect()
    torch.cuda.synchronize()
    free2 = torch.cuda.mem_get_info(0)[0]
    assert free2 - free1 >= 0.9 * obs_bytes, (free0, free1, free2)
