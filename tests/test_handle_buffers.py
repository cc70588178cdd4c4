"""A failed grow of a handle's device buffers leaves the handle usable.  Each entry point below is asked once for a batch whose
buffers are far beyond any GPU's memory: cudaMalloc fails at once, the call returns an error that names the allocation, and the
same small call as before then runs again and returns the same bits.  Each failing call fails before it enqueues any work sized
by its batch."""
import numpy as np
import pytest
import torch

from posendf_b200 import _lib, synth, train
from posendf_b200.engine import Engine

pytestmark = pytest.mark.gpu

HUGE_B = 1 << 40


@pytest.fixture(scope="module")
def eng():
    e = Engine(device=0)
    e.set_weights_flat(synth.flatten_params(synth.make_params(1)))
    yield e
    e.close()


def stream():
    return torch.cuda.current_stream().cuda_stream


def fails_for_memory(rc, lib):
    torch.cuda.synchronize()
    assert rc != 0
    assert "memory" in lib.pndf_last_error().decode().lower()


def test_denoise_prior_after_a_failed_grow(eng):
    aa0 = torch.from_numpy(synth.make_axis_angle(12, 2 * 50).reshape(2, 50, 63)).cuda()

    def small():
        aa = aa0.clone()
        d, hist = eng.denoise_prior_(aa, iterations=2, steps_per_iter=3, lr=0.02, want_loss=True)
        torch.cuda.synchronize()
        return aa, d, hist

    first = small()
    aa = aa0.clone()
    fails_for_memory(eng.lib.pndf_denoise_prior(eng._h, aa.data_ptr(), 1 << 31, 100, 2, 3, 0.02, None, None, stream()), eng.lib)
    assert torch.equal(aa, aa0)
    again = small()
    for a, b in zip(first, again):
        assert torch.equal(a, b)


def test_wgrad_accumulate_after_a_failed_grow(eng):
    """one training step's exports (pose batch with the Eikonal term, as FusedTrainLosses runs it) reduced into the flat gradient"""
    B = 64
    x = torch.from_numpy(synth.make_poses(2001, B, kind="noisy", sigma=0.25)).cuda().contiguous()
    gt = torch.from_numpy((synth.uniform01(4001, B) * 0.5).astype(np.float32)).cuda()
    ex = train._Exports(eng, x, True, want_masks=True)
    ex.coef = torch.empty(B, device=x.device, dtype=torch.float32)
    ex.v = torch.empty(B, 21, 4, device=x.device, dtype=torch.float32)
    losses = torch.empty(3, device=x.device, dtype=torch.float32)
    _lib.check(eng.lib.pndf_train_losses(eng._h, ex.dist.data_ptr(), gt.data_ptr(), ex.grad.data_ptr(), B, B, 0, 0, 1,
                                         ex.coef.data_ptr(), ex.v.data_ptr(), losses.data_ptr(), stream()))
    ex.tangent_launch(eng)
    gd = torch.ones(1, device=x.device, dtype=torch.float32)
    ge = torch.full((1,), 1.3, device=x.device, dtype=torch.float32)
    flat = torch.empty(eng.param_count, device=x.device, dtype=torch.float32)

    def wgrad(n):
        return eng.lib.pndf_wgrad_accumulate(eng._h, ex.x.data_ptr(), ex.v.data_ptr(), 1, ex.dump.data_ptr(), ex.dump_t.data_ptr(),
                                             ex.coef.data_ptr(), 0.0, ex.dist.data_ptr(), n, gd.data_ptr(), ge.data_ptr(), None,
                                             flat.data_ptr(), 1, stream())

    _lib.check(wgrad(B))
    first = flat.clone()
    assert first.abs().sum().item() > 0
    fails_for_memory(wgrad(HUGE_B), eng.lib)
    flat.fill_(float("nan"))
    _lib.check(wgrad(B))
    torch.cuda.synchronize()
    assert torch.equal(flat, first)


def test_encoder_param_grads_after_a_failed_grow(eng):
    B = 64
    x = torch.from_numpy(synth.make_poses(5, B, kind="noisy", sigma=0.25)).cuda().contiguous()
    gen = torch.Generator(device="cuda").manual_seed(0)
    v = torch.randn(B, 84, device="cuda", generator=gen)
    up1 = torch.randn(B, 126, device="cuda", generator=gen)
    upt = torch.randn(B, 126, device="cuda", generator=gen)
    grads = torch.empty(2, 3516, device="cuda", dtype=torch.float32)

    def enc_grads(n):
        return eng.lib.pndf_encoder_param_grads(eng._h, x.data_ptr(), v.data_ptr(), n, 1, up1.data_ptr(), upt.data_ptr(), None,
                                                grads.data_ptr(), stream())

    _lib.check(enc_grads(B))
    first = grads.clone()
    assert first[0].abs().sum().item() > 0 and first[1].abs().sum().item() > 0
    fails_for_memory(enc_grads(HUGE_B), eng.lib)
    assert not grads.any()          # the call zeroes grads_dev before it grows its buffers
    _lib.check(enc_grads(B))
    torch.cuda.synchronize()
    assert torch.equal(grads, first)
