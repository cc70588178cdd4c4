"""Which engine runs each DFNet call.  A call resolves one tile size -- PNDF_TILE in the environment, else the pinned tile policy,
else the batch-size rule of pndf_tile_for_batch -- and a launch that cannot take it runs the fused 32-pose kernel instead.  The
engine that ran is identified two ways: the launch count (tensor-core engine: 8 kernels per forward, 15 per forward + gradient,
prior evaluation or projection step, per pass of at most 131 072 poses; fused FFMA kernel: one launch per call) and bit equality
with the same call under the expected PNDF_TILE.  Where the tile size decides the result, the forced 8- and 32-pose runs are also
checked to differ on that input, so that the bit comparison tells the two tilings apart."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from posendf_b200 import _lib, synth
from posendf_b200.engine import Engine

pytestmark = pytest.mark.gpu

TC_CHUNK = 131072                    # poses per pass of the tensor-core engine
SIZES = ["10", "8sms", "8sms+1", "16sms+1", "131073"]
# (PNDF_TILE, pinned policy): the batch-size rule, each pinned policy, and the environment overriding a pinned policy
SETTINGS = [(None, 0), (None, 8), (None, 32), (None, 128), ("32", 128), ("8", 128), ("128", 8)]


@pytest.fixture(scope="module")
def eng():
    e = Engine(device=0)
    e.set_weights_flat(synth.flatten_params(synth.make_params(1)))
    yield e
    e.close()


@pytest.fixture
def run(eng, monkeypatch):
    """run(fn, env, policy): fn() under that PNDF_TILE / pinned policy -> (outputs on the host, launches it made)"""
    def go(fn, env=None, policy=0):
        if env is None:
            monkeypatch.delenv("PNDF_TILE", raising=False)
        else:
            monkeypatch.setenv("PNDF_TILE", env)
        eng.set_tile_policy(policy)
        try:
            n0 = eng.launch_count()
            out = fn()
            torch.cuda.synchronize()
            return [t.cpu() for t in out], eng.launch_count() - n0
        finally:
            eng.set_tile_policy(0)
            monkeypatch.delenv("PNDF_TILE", raising=False)
    return go


def batch_size(eng, name):
    s = eng.num_sms()
    return {"10": 10, "8sms": 8 * s, "8sms+1": 8 * s + 1, "16sms+1": 16 * s + 1, "131073": TC_CHUNK + 1}[name]


def requested(eng, B, env, policy):
    if env is not None:
        return {"8": 8, "128": 128}.get(env, 32)
    return policy or eng.tile_for_batch(B)


def same(a, b):
    return len(a) == len(b) and all(torch.equal(x, y) for x, y in zip(a, b))


def stream():
    return torch.cuda.current_stream().cuda_stream


def project_gather(eng, x, steps):
    """pndf_project_gather without peers"""
    d = torch.empty(x.shape[0], 1, device=x.device, dtype=torch.float32)
    _lib.check(eng.lib.pndf_project_gather(eng._h, x.data_ptr(), x.shape[0], steps, 0, d.data_ptr(), None, None, 0, stream()))
    return d


def test_tile_for_batch_is_the_batch_size_rule(eng, run):
    s = eng.num_sms()
    want = {10: 8, 8 * s: 8, 8 * s + 1: 128, 16 * s + 1: 128, TC_CHUNK + 1: 128}
    for env, policy in SETTINGS:
        got, _ = run(lambda: [torch.tensor([eng.tile_for_batch(B) for B in want])], env, policy)
        assert got[0].tolist() == list(want.values()), (env, policy)


# quaternion calls: every tile size is available; tensor-core kernels per pass of TC_CHUNK poses
QUAT_OPS = {
    "forward": (lambda eng, x: [eng.forward(x)], 8),
    "forward_grad": (lambda eng, x: list(eng.forward_grad(x)), 15),
    "project": (lambda eng, x: (lambda y: [eng.project_(y, steps=2), y])(x.clone()), 2 * 15),
    "project_gather": (lambda eng, x: (lambda y: [project_gather(eng, y, 2), y])(x.clone()), 2 * 15),
}


@pytest.mark.parametrize("op", list(QUAT_OPS))
@pytest.mark.parametrize("size", SIZES)
def test_quaternion_calls(eng, run, op, size):
    fn, tc_launches = QUAT_OPS[op]
    B = batch_size(eng, size)
    x = torch.from_numpy(synth.make_poses(31, B)).cuda()
    ref = {t: run(lambda: fn(eng, x), str(t))[0] for t in (8, 32, 128)}
    assert not same(ref[8], ref[32])
    for env, policy in SETTINGS:
        tile = requested(eng, B, env, policy)
        out, n = run(lambda: fn(eng, x), env, policy)
        assert n == (tc_launches * math.ceil(B / TC_CHUNK) if tile == 128 else 1), (env, policy, tile, n)
        assert same(out, ref[tile]), (env, policy, tile)


@pytest.mark.parametrize("size", SIZES)
def test_prior_grad(eng, run, size):
    """the prior mode takes the tensor-core engine in ONE pass: above TC_CHUNK poses a requested 128 runs the fused 32-pose kernel"""
    B = batch_size(eng, size)
    aa = torch.from_numpy(synth.make_axis_angle(32, B)).cuda()
    fn = lambda: list(eng.prior_grad(aa))
    ref = {t: run(fn, str(t))[0] for t in (8, 32, 128)}
    assert not same(ref[8], ref[32])
    for env, policy in SETTINGS:
        tile = requested(eng, B, env, policy)
        if tile == 128 and B > TC_CHUNK:
            tile = 32
        out, n = run(fn, env, policy)
        assert n == (15 if tile == 128 else 1), (env, policy, tile, n)
        assert same(out, ref[tile]), (env, policy, tile)


def export_calls(eng, x):
    B = x.shape[0]
    tiles = (B + 31) // 32
    n = C.c_size_t()
    _lib.check(eng.lib.pndf_debug_dump_floats(C.byref(n)))
    rows = n.value // 32
    tan = torch.from_numpy(synth.normal(33, tiles * 128 * 32).astype(np.float32)).cuda()

    def export():
        dist = torch.empty(B, 1, device=x.device)
        grad = torch.empty(B, 21, 4, device=x.device)
        dump = torch.zeros(tiles * 32, rows, device=x.device)
        _lib.check(eng.lib.pndf_forward_grad_export(eng._h, x.data_ptr(), B, 1, dist.data_ptr(), grad.data_ptr(), dump.data_ptr(),
                                                    None, stream()))
        return [dist, grad, dump]

    def tangent():
        dump = torch.zeros(tiles * 32, rows, device=x.device)
        _lib.check(eng.lib.pndf_forward_tangent_export(eng._h, x.data_ptr(), B, 1, tan.data_ptr(), dump.data_ptr(), None, stream()))
        return [dump]

    return {"debug": lambda: list(eng.forward_grad_debug(x)), "export": export, "tangent": tangent}


@pytest.mark.parametrize("op", ["debug", "export", "tangent"])
@pytest.mark.parametrize("size", ["10", "8sms+1"])
def test_debug_and_training_exports_run_fused_32(eng, run, op, size):
    B = batch_size(eng, size)
    x = torch.from_numpy(synth.make_poses(34, B)).cuda()
    fn = export_calls(eng, x)[op]
    ref, _ = run(fn, "32")
    for env, policy in SETTINGS + [("8", 0), ("128", 0)]:
        out, n = run(fn, env, policy)
        assert n == 1 and same(out, ref), (env, policy, n)


def tc_host_chunks(B):
    """chunks of pndf_project_host on the tensor-core engine: 8 192-pose head and tail, body chunks of at most 49 152 poses"""
    if B <= 2 * 8192:
        return math.ceil(B / 8192)
    mid = B - 2 * 8192
    per = math.ceil(math.ceil(mid / math.ceil(mid / 49152)) / 128) * 128
    return 2 + math.ceil(mid / per)


@pytest.mark.parametrize("B", [20000, 1000])
def test_project_host(eng, run, B):
    """every chunk runs the tile the whole batch resolves to: the result equals pndf_project on the whole batch"""
    poses = torch.from_numpy(synth.make_poses(35, B)).pin_memory()
    x = poses.cuda()
    dev = lambda: (lambda y: [y, eng.project_(y, steps=2)])(x.clone())
    ref = {t: run(dev, str(t))[0] for t in (8, 32, 128)}
    assert not same(ref[8], ref[32])
    for env, policy in SETTINGS[:4]:
        tile = requested(eng, B, env, policy)
        out, n = run(lambda: list(eng.project_host(poses, steps=2)), env, policy)
        chunks = tc_host_chunks(B) if tile == 128 else math.ceil(B / (eng.num_sms() * 4 * 32))
        assert n == chunks * (2 * 15 if tile == 128 else 1), (policy, tile, n)
        assert same(out, ref[tile]), (policy, tile)


@pytest.mark.parametrize("S,T", [(3, 40), (2, 1000), (2, 70000)])
def test_denoise_prior(eng, run, S, T):
    """one tensor-core chain iff S*T resolves to 128 and fits one pass; else two fused sequence groups, each at the tile its own
    size resolves to (128 -> 32)"""
    B = S * T
    aa0 = torch.from_numpy(synth.make_axis_angle(36, B).reshape(S, T, 21, 3)).cuda()
    nsteps = 2

    def fn():
        aa = aa0.clone()
        d, hist = eng.denoise_prior_(aa, iterations=1, steps_per_iter=nsteps, lr=0.02, want_loss=True)
        return [aa, d, hist]

    ref = {t: run(fn, str(t))[0] for t in (8, 32, 128)}
    assert not same(ref[8], ref[32])
    groups = [S // 2 * T, (S - S // 2) * T]
    for env, policy in SETTINGS:
        if requested(eng, B, env, policy) == 128 and B <= TC_CHUNK:
            tile, launches = 128, 15 * nsteps + 1
        else:
            tiles = {32 if t == 128 else t for t in (requested(eng, Bg, env, policy) for Bg in groups)}
            assert len(tiles) == 1
            tile, launches = tiles.pop(), (nsteps + 1) * 2
        out, n = run(fn, env, policy)
        assert n == launches, (env, policy, tile, n)
        assert same(out, ref[tile]), (env, policy, tile)
