"""GPU parity tests proper: the fused sm_100a kernel, called through the C ABI (libpndf.so), against the
oracle on the same seeded inputs and against the committed golden vectors of the real reference."""
import numpy as np
import pytest
import torch

from conftest import (assert_grad_parity, assert_pose_parity, case_cfg, case_inputs, golden_case_names, load_golden,
                      per_pose_rel, rel_err)
from oracle import posendf_numpy as onp
from posendf_b200 import synth

pytestmark = pytest.mark.gpu
CASES = golden_case_names()


@pytest.fixture(autouse=True, params=["auto", "32", "8", "128"])
def tile_size(request, monkeypatch):
    """every test of this file runs with the library's own choice of path (tensor-core DFNet for large batches, 32-pose FFMA tiles,
    8-pose small-tile kernels for batches that cannot fill the SMs) and with each of them forced (PNDF_TILE = 128 / 32 / 8,
    csrc/pndf_capi.cu::tile_for)"""
    if request.param == "auto":
        monkeypatch.delenv("PNDF_TILE", raising=False)
    else:
        monkeypatch.setenv("PNDF_TILE", request.param)
    return request.param


def make_engine(meta, params):
    from posendf_b200.engine import Engine
    cfg = case_cfg(meta)
    eng = Engine(device=0, use_enc=cfg["use_enc"], enc_act=cfg["enc_act"], enc_beta=cfg["enc_beta"],
                 df_act=cfg["df_act"], df_beta=cfg["df_beta"])
    in_dim = 126 if cfg["use_enc"] else 84
    eng.set_weights_flat(synth.flatten_params(params, in_dim=in_dim, use_enc=cfg["use_enc"]))
    return eng


def oracle_intermediates(params, poses, cfg):
    """every tile the kernel's debug hook dumps, from the fp64 oracle: list of (name, row0, array[rows, B])"""
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    x = poses.astype(np.float64)
    q, _ = onp.normalise_columns(x)
    if cfg["use_enc"]:
        z0, _ = onp.encoder_forward(p64, q, cfg)
    else:
        z0 = q.reshape(len(q), -1)
    d, pres = onp.dfnet_forward(p64, z0, cfg)
    zs = [onp.act(pr, cfg["df_act"], cfg["df_beta"]) for pr in pres[:-1]]
    out = [("z0", 0, z0.T), ("z1", 128, zs[0].T), ("z2", 384, zs[1].T), ("z3a", 896, zs[2][:, :512].T),
           ("z3b", 1408, zs[2][:, 512:].T), ("z4", 1920, zs[3].T), ("z5", 2432, zs[4].T), ("z6", 2688, zs[5].T)]
    g = np.ones((len(x), 1)) * onp.dact(pres[-1], onp.out_act_kind(cfg["df_act"]), cfg["df_beta"])
    g = g @ p64["dfnet.lin6.weight"]
    gm = {}
    for l in range(5, -1, -1):
        gm[l + 1] = g * onp.dact(pres[l], cfg["df_act"], cfg["df_beta"])     # masked gradient wrt pre_l
        g = gm[l + 1] @ p64[f"dfnet.lin{l}.weight"]
    out += [("g6m", 2752, gm[6].T), ("g5m", 2816, gm[5].T), ("g4m", 3072, gm[4].T), ("g3a", 3584, gm[3][:, :512].T),
            ("g3b", 4096, gm[3][:, 512:].T), ("g2m", 4608, gm[2].T), ("g1m", 5120, gm[1].T), ("g0", 5376, g.T)]
    return out


@pytest.mark.parametrize("name", ["lrelu_enc_s1", "softplus_enc_s3", "lrelu_noenc_s6"])
def test_every_layer_tile_matches_oracle(name):
    meta, z = load_golden(name)
    cfg = case_cfg(meta)
    params, poses = case_inputs(meta)
    poses = poses[:32]
    eng = make_engine(meta, params)
    dist, grad, dump = eng.forward_grad_debug(torch.from_numpy(poses).cuda())
    torch.cuda.synchronize()
    dump = dump.cpu().numpy().T          # pose-major export -> [row][pose]
    lines = []
    worst = 0.0
    for nm, row0, ref in oracle_intermediates(params, poses, cfg):
        got = dump[row0:row0 + ref.shape[0]]
        scale = np.abs(ref).max() + 1e-30
        err = np.abs(got - ref).max() / scale
        lines.append(f"{name:24s} {nm:5s} rows {ref.shape[0]:4d} max|ref| {scale:.3e} max err/scale {err:.3e}")
        worst = max(worst, err)
    print("\n".join(lines))
    assert worst < 2e-5, "\n".join(lines)
    assert np.max(rel_err(dist.cpu().numpy(), z["d64"][:32])) < 1e-5


@pytest.mark.parametrize("name", CASES)
def test_forward_distance_vs_reference_golden(name):
    meta, z = load_golden(name)
    params, poses = case_inputs(meta)
    eng = make_engine(meta, params)
    d = eng.forward(torch.from_numpy(poses).cuda()).cpu().numpy()
    assert d.shape == (64, 1)
    assert np.max(rel_err(d, z["d64"])) < 1e-5      # north-star bar: 1e-5 relative on the distance


@pytest.mark.parametrize("name", CASES)
def test_forward_grad_vs_reference_golden(name):
    meta, z = load_golden(name)
    params, poses = case_inputs(meta)
    eng = make_engine(meta, params)
    d, g = eng.forward_grad(torch.from_numpy(poses).cuda())
    assert np.max(rel_err(d.cpu().numpy(), z["d64"])) < 1e-5
    # outliers (if any) must be kink flips: reproduced by the fp64 oracle with a near-zero pre-activation on its other branch
    assert_grad_parity(g.cpu().numpy(), z["g64"], explain=(params, poses, case_cfg(meta)))


@pytest.mark.parametrize("name", CASES)
def test_projection_10_steps_vs_reference_golden(name):
    """experiments/sample_poses.py:70-74, ten steps fused in ONE launch."""
    meta, z = load_golden(name)
    params, poses = case_inputs(meta)
    eng = make_engine(meta, params)
    x = torch.from_numpy(poses).cuda().contiguous()
    dlast = eng.project_(x, steps=10)
    assert_pose_parity(x.cpu().numpy(), z["proj64"])
    assert np.max(rel_err(dlast.cpu().numpy(), z["proj_d64"][-1])) < 2e-5
    # ten single-step launches == one ten-step launch, bit for bit
    y = torch.from_numpy(poses).cuda().contiguous()
    for _ in range(10):
        eng.project_(y, steps=1)
    assert torch.equal(x, y)


@pytest.mark.parametrize("name", ["lrelu_enc_s1", "softplus_enc_s3"])
def test_projection_50_steps_vs_reference_golden(name):
    """BASELINE configs[2]: the loop of experiments/sample_poses.py:70-74 run to K = 50 by the REAL reference (fp64 golden),
    against ONE 50-step launch; also 5 launches of 10 steps == 1 launch of 50, bit for bit."""
    meta, z = load_golden(name)
    params, poses = case_inputs(meta)
    eng = make_engine(meta, params)
    x = torch.from_numpy(poses).cuda().contiguous()
    dlast = eng.project_(x, steps=50)
    assert_pose_parity(x.cpu().numpy(), z["proj50_64"])
    assert z["proj50_d64"].shape[0] == 50
    assert np.max(rel_err(dlast.cpu().numpy(), z["proj50_d64"][-1])) < 2e-5
    y = torch.from_numpy(poses).cuda().contiguous()
    for _ in range(5):
        eng.project_(y, steps=10)
    assert torch.equal(x, y)


@pytest.mark.parametrize("B,sub", [(1024, 1024), (65536, 2048)])
def test_baseline_config_batches_vs_fp64_oracle(B, sub):
    """BASELINE configs[0] (1 024 poses) and configs[1] (65 536 poses) at their exact sizes: distances of EVERY pose against the
    fp64 oracle; gradient and one projection step against it on `sub` poses spread over the batch (all of them at 1 024)."""
    meta, _ = load_golden("lrelu_enc_s1")
    cfg = case_cfg(meta)
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    poses = synth.make_poses(1234, B)
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    x = torch.from_numpy(poses).cuda()
    d = eng.forward(x)
    d2, g = eng.forward_grad(x)
    xp = x.clone()
    dl = eng.project_(xp, steps=1)
    torch.cuda.synchronize()
    assert torch.equal(d, d2) and torch.equal(d, dl)
    dref = np.concatenate([onp.forward(p64, poses[i:i + 8192].astype(np.float64), cfg) for i in range(0, B, 8192)])
    assert np.max(rel_err(d.cpu().numpy(), dref)) < 1e-5
    idx = np.arange(B) if sub >= B else np.unique(np.linspace(0, B - 1, sub).astype(np.int64))
    _, gref = onp.forward_grad(p64, poses[idx].astype(np.float64), cfg)
    assert_grad_parity(g.cpu().numpy()[idx], gref, explain=(params, poses[idx], cfg))
    xref, _ = onp.project(p64, poses[idx].astype(np.float64), cfg, steps=1)
    assert_pose_parity(xp.cpu().numpy()[idx], xref)


@pytest.mark.parametrize("B", [1, 31, 32, 33, 1000, 4736 + 17])
def test_ragged_batches_and_tile_independence(B):
    """per-pose independence: any batch size, any position in the batch -> identical bits."""
    meta, _ = load_golden("lrelu_enc_s1")
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    poses = synth.make_poses(5, B)
    x = torch.from_numpy(poses).cuda()
    d, g = eng.forward_grad(x)
    dref, gref = onp.forward_grad({k: v.astype(np.float64) for k, v in params.items()}, poses.astype(np.float64), case_cfg(meta))
    assert np.max(rel_err(d.cpu().numpy(), dref)) < 1e-5
    assert_grad_parity(g.cpu().numpy(), gref, explain=(params, poses, case_cfg(meta)))
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(0)).cuda()
    d2, g2 = eng.forward_grad(x[perm].contiguous())
    assert torch.equal(d2, d[perm]) and torch.equal(g2, g[perm])
    assert torch.equal(eng.forward(x), d)           # forward-only kernel == forward of the grad kernel


def test_empty_batch():
    meta, _ = load_golden("lrelu_enc_s1")
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    d = eng.forward(torch.empty(0, 21, 4, device="cuda"))
    assert d.shape == (0, 1)


def test_upstream_gradient_vjp_and_no_normalise():
    meta, _ = load_golden("relu_enc_s2")
    cfg = case_cfg(meta)
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    poses = synth.make_poses(21, 96, kind="noisy", sigma=0.25)
    gup = (synth.normal(3, 96) * 3.0).astype(np.float32).reshape(96, 1)
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    d, g = eng.forward_grad(torch.from_numpy(poses).cuda(), g_up=torch.from_numpy(gup).cuda())
    dref, gref = onp.forward_grad(p64, poses.astype(np.float64), cfg, g_up=gup.astype(np.float64))
    assert np.max(rel_err(d.cpu().numpy(), dref)) < 1e-5
    assert_grad_parity(g.cpu().numpy(), gref)
    # manifold branch of the train path: no column normalisation (model/posendf.py:80-83)
    d, g = eng.forward_grad(torch.from_numpy(poses).cuda(), normalise=False)
    dref, gref = onp.forward_grad(p64, poses.astype(np.float64), cfg, normalise=False)
    assert np.max(rel_err(d.cpu().numpy(), dref)) < 1e-5
    assert_grad_parity(g.cpu().numpy(), gref)


def test_renormalised_projection_option():
    meta, _ = load_golden("lrelu_enc_s1")
    cfg = case_cfg(meta)
    params, poses = case_inputs(meta)
    eng = make_engine(meta, params)
    x = torch.from_numpy(poses).cuda().contiguous()
    eng.project_(x, steps=5, renorm=True)
    xref, _ = onp.project({k: v.astype(np.float64) for k, v in params.items()}, poses.astype(np.float64), cfg, steps=5, renorm=True)
    assert_pose_parity(x.cpu().numpy(), xref)
    assert np.allclose(np.linalg.norm(x.cpu().numpy(), axis=2), 1.0, atol=1e-6)


@pytest.mark.parametrize("name", ["lrelu_enc_s1", "softplus_enc_s3"])
def test_prior_term_axis_angle(name):
    """experiments/motion_denoise.py:81-83 + backward to the axis-angle pose."""
    meta, _ = load_golden(name)
    cfg = case_cfg(meta)
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    aa = synth.make_axis_angle(4, 200)
    aa[0, 0] = 0.0
    gup = np.full((200, 1), 1e7 * 2 * 0.5 / 200, dtype=np.float32)
    d, g = eng.prior_grad(torch.from_numpy(aa).cuda(), g_up=torch.from_numpy(gup).cuda())
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    a64 = aa.astype(np.float64)
    quat = onp.axis_angle_to_quaternion(a64)
    dref, qbar = onp.forward_grad(p64, quat, cfg, g_up=gup.astype(np.float64))
    gref = onp.axis_angle_to_quaternion_vjp(a64, qbar)
    assert np.max(rel_err(d.cpu().numpy(), dref)) < 1e-5
    assert_grad_parity(g.cpu().numpy(), gref, tol=2e-5)


@pytest.mark.parametrize("B", [148 * 4 * 32 + 1234, 70000 + 77])
def test_host_buffer_projection_matches_device_projection(B):
    """pndf_project_host (pinned host buffers, chunked upload / compute / download overlap; head / body / tail chunk schedule on the
    tensor-core engine) == pndf_project on the same batch, bit for bit"""
    meta, _ = load_golden("lrelu_enc_s1")
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    poses = torch.from_numpy(synth.make_poses(8, B)).pin_memory()
    out, dist = eng.project_host(poses, steps=2)
    x = poses.cuda().contiguous()
    d = eng.project_(x, steps=2)
    assert torch.equal(out, x.cpu()) and torch.equal(dist, d.cpu())


def test_large_batch_properties():
    """config-2 size (65 536 poses): d >= 0, finite, chunk results identical to the full-batch run."""
    meta, _ = load_golden("lrelu_enc_s1")
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    B = 65536
    x = torch.from_numpy(synth.make_poses(123, B)).cuda()
    d, g = eng.forward_grad(x)
    assert torch.isfinite(d).all() and torch.isfinite(g).all() and (d >= 0).all()
    # a caller that evaluates a slice of a batch on its own pins the tile size the whole batch gets (include/pndf.h)
    eng.set_tile_policy(eng.tile_for_batch(B))
    d2, g2 = eng.forward_grad(x[20000:20000 + 777].contiguous())
    eng.set_tile_policy(0)
    assert torch.equal(d2, d[20000:20777]) and torch.equal(g2, g[20000:20777])
    y = x.clone()
    eng.project_(y, steps=1)
    assert torch.equal(y, x - d.reshape(-1, 1, 1) * g)


def test_tensor_core_passes_of_a_very_large_batch(tile_size):
    """the tensor-core engine walks batches above 131 072 poses in passes (its activations live in HBM between the layer kernels):
    a 2-step projection over 131 072 + 333 poses equals the same call on the two parts, bit for bit, and follows the fp64 oracle"""
    if tile_size not in ("auto", "128"):
        pytest.skip("one pass structure per engine: the fused kernel has none")
    meta, _ = load_golden("lrelu_enc_s1")
    cfg = case_cfg(meta)
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    B = 131072 + 333
    poses = synth.make_poses(77, B)
    x = torch.from_numpy(poses).cuda()
    y = x.clone()
    d = eng.project_(y, steps=2)
    parts = []
    eng.set_tile_policy(eng.tile_for_batch(B))
    for lo, hi in ((0, 131072), (131072, B)):
        z = x[lo:hi].clone()
        dz = eng.project_(z, steps=2)
        parts.append((z, dz))
    eng.set_tile_policy(0)
    torch.cuda.synchronize()
    assert torch.equal(y, torch.cat([p[0] for p in parts])) and torch.equal(d, torch.cat([p[1] for p in parts]))
    idx = np.unique(np.concatenate([np.linspace(0, B - 1, 192).astype(np.int64), np.arange(131072 - 8, 131072 + 8), np.arange(B - 8, B)]))
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    xref, _ = onp.project(p64, poses[idx].astype(np.float64), cfg, steps=2)
    assert_pose_parity(y.cpu().numpy()[idx], xref)


# ---------------------------------------------------------------------------- reference call surface on the GPU
def _opt(meta):
    cfg = case_cfg(meta)
    return {"train": {"device": "cuda", "loss_type": meta.get("loss_type", "l1"), "batch_size": 4},
            "model": {"StrEnc": {"use": cfg["use_enc"], "act": cfg["enc_act"], "beta": cfg["enc_beta"]},
                      "DFNet": {"in_dim": 126 if cfg["use_enc"] else 84, "dims": [256, 512, 1024, 512, 256, 64],
                                "act": cfg["df_act"], "beta": cfg["df_beta"]}}}


@pytest.mark.parametrize("name", ["lrelu_enc_s1", "softplus_enc_s3", "lrelu_noenc_s6"])
def test_module_drop_in_forward_and_autograd(name):
    """the exact call pattern of experiments/sample_poses.py:66-74 against the reference's golden output."""
    from posendf_b200 import PoseNDF, gradient
    meta, z = load_golden(name)
    params, poses = case_inputs(meta)
    net = PoseNDF(_opt(meta))
    net.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()})
    net.eval()
    noisy = torch.from_numpy(poses).cuda()
    noisy.requires_grad = True
    for _ in range(10):
        pred = net(noisy, train=False)
        grad = gradient(noisy, pred["dist_pred"]).reshape(-1, 84)
        noisy = noisy - (pred["dist_pred"] * grad).reshape(-1, 21, 4)
    assert_pose_parity(noisy.detach().cpu().numpy(), z["proj64"])
    # fused K-step projection gives the same trajectory
    x, d = net.project(torch.from_numpy(poses), steps=10)
    assert_pose_parity(x.cpu().numpy(), z["proj64"])
    assert np.max(per_pose_rel(x.cpu().numpy(), noisy.detach().cpu().numpy())) < 1e-6
    # no-grad forward, any leading shape, CPU input moved like the reference's .to(device)
    with torch.no_grad():
        d0 = net(torch.from_numpy(poses).reshape(8, 8, 84), train=False)["dist_pred"]
    assert d0.shape == (64, 1) and np.max(rel_err(d0.cpu().numpy(), z["d64"])) < 1e-5


def test_module_backward_with_upstream_gradient_and_weight_refresh():
    """motion_denoise-style: loss = w * mean(dist)^2 ; backward() reaches the pose through the fused gradient."""
    from posendf_b200 import PoseNDF
    meta, z = load_golden("lrelu_enc_s1")
    cfg = case_cfg(meta)
    params, poses = case_inputs(meta)
    net = PoseNDF(_opt(meta))
    net.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()})
    x = torch.from_numpy(poses).cuda().requires_grad_(True)
    d = net(x, train=False)["dist_pred"]
    loss = 1e7 * torch.mean(d) ** 2
    loss.backward()
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    dref, gref = onp.forward_grad(p64, poses.astype(np.float64), cfg)
    up = 1e7 * 2 * dref.mean() / len(dref)
    assert_grad_parity(x.grad.cpu().numpy(), up * gref)
    # in-place weight update (an optimiser step) must invalidate the packed device copy
    with torch.no_grad():
        net.dfnet.lin6.bias.add_(0.25)
    d2 = net(x.detach(), train=False)["dist_pred"]
    assert torch.allclose(d2, d.detach() + 0.25, atol=1e-6)


def test_denoise_prior_loop_vs_oracle():
    """experiments/motion_denoise.py:70-99 restricted to the prior term: fused prior kernel + per-sequence Adam."""
    meta, _ = load_golden("softplus_enc_s3")
    cfg = case_cfg(meta)
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    S, T = 3, 40
    aa = synth.make_axis_angle(11, S * T).reshape(S, T, 21, 3)
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    xref, dref, href = onp.denoise_prior(p64, aa.astype(np.float64), cfg, iterations=2, steps_per_iter=4)
    x = torch.from_numpy(aa).cuda().contiguous()
    d, hist = eng.denoise_prior_(x, iterations=2, steps_per_iter=4, lr=0.02, want_loss=True)
    x = x.cpu().numpy(); d = d.cpu().numpy(); hist = hist.cpu().numpy()
    assert np.max(np.abs(hist - href) / np.abs(href)) < 2e-5
    assert np.max(rel_err(d, dref)) < 1e-5
    # Adam normalises the step by sqrt(v): every element moves ~lr per step whatever the gradient scale, so the
    # comparison is absolute against the 0.02-per-step move (8 steps); kink flips show up as a few outliers
    err = np.abs(x - xref)
    assert np.abs(xref - aa).max() > 0.05
    assert np.median(err) < 2e-6 and (err > 1e-4).mean() < 0.01, (np.median(err), err.max(), (err > 1e-4).mean())


def test_two_handles_and_side_stream_do_not_interfere():
    """two engines with different weights / activations alive at once, one driven from a non-default stream"""
    from posendf_b200.engine import Engine
    pa, pb = synth.make_params(1), synth.make_params(2)
    ea = Engine(device=0, enc_act="lrelu", df_act="lrelu")
    eb = Engine(device=0, enc_act="softplus", df_act="softplus")
    ea.set_weights_flat(synth.flatten_params(pa)); eb.set_weights_flat(synth.flatten_params(pb))
    poses = synth.make_poses(17, 300)
    x = torch.from_numpy(poses).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        db, gb = eb.forward_grad(x)
    da, ga = ea.forward_grad(x)
    side.synchronize(); torch.cuda.synchronize()
    p64 = lambda p: {k: v.astype(np.float64) for k, v in p.items()}
    ra, _ = onp.forward_grad(p64(pa), poses.astype(np.float64), onp.default_cfg())
    rb, _ = onp.forward_grad(p64(pb), poses.astype(np.float64), onp.default_cfg(enc_act="softplus", df_act="softplus"))
    assert np.max(rel_err(da.cpu().numpy(), ra)) < 1e-5 and np.max(rel_err(db.cpu().numpy(), rb)) < 1e-5


def test_api_misuse_fails_loudly():
    from posendf_b200.engine import Engine
    eng = Engine(device=0)
    x = torch.zeros(4, 21, 4, device="cuda")
    with pytest.raises(RuntimeError, match="pndf_set_weights"):
        eng.forward(x)                                     # no weights yet
    with pytest.raises(RuntimeError, match="wrong parameter count"):
        eng.set_weights_flat(np.zeros(10, dtype=np.float32))
    eng.set_weights_flat(synth.flatten_params(synth.make_params(1)))
    with pytest.raises(RuntimeError):
        eng.forward(torch.zeros(4, 21, 4))                 # CPU tensor
    with pytest.raises(RuntimeError):
        eng.project_(torch.zeros(8, 21, 4, device="cuda")[::2])   # non-contiguous in-place target
    with pytest.raises(RuntimeError, match="steps"):
        eng.project_(x.clone(), steps=0)
    with pytest.raises(RuntimeError, match="amass.yaml"):
        Engine(device=0, dims=(128, 128))
    # fp64 / non-contiguous inputs of the out-of-place entry points are converted, not rejected
    d = eng.forward(torch.zeros(8, 21, 4, device="cuda", dtype=torch.float64)[::2] + 0.1)
    assert d.shape == (4, 1) and torch.isfinite(d).all()


@pytest.mark.parametrize("S,T", [(3, 40), (70, 1), (5, 7), (2, 300)])
def test_denoise_one_launch_per_step_graph_equals_plain_launches(S, T, monkeypatch, tile_size):
    """f1: steps + 1 launches per sequence group (the Adam update of step t-1 rides in the prologue of launch t; two groups of
    sequences run as parallel chains so that one group's tail round overlaps the other's next launch), replayed as one CUDA graph;
    the graph replay and plain launches give identical bits, also when a tile holds many short sequences (T = 1, 7) or a
    sequence spans many tiles (T = 300), and the result follows the fp64 oracle."""
    meta, _ = load_golden("softplus_enc_s3")       # smooth network: no kink flips between fp32 and the fp64 oracle
    cfg = case_cfg(meta)
    params, _ = case_inputs(meta)
    eng = make_engine(meta, params)
    aa = synth.make_axis_angle(21, S * T).reshape(S, T, 21, 3)
    outs = []
    for no_graph in (False, True):
        if no_graph:
            monkeypatch.setenv("PNDF_NO_GRAPH", "1")
        else:
            monkeypatch.delenv("PNDF_NO_GRAPH", raising=False)
        x = torch.from_numpy(aa).cuda().contiguous()
        n0 = eng.launch_count()
        d, hist = eng.denoise_prior_(x, iterations=2, steps_per_iter=3, lr=0.02, want_loss=True)
        torch.cuda.synchronize()
        if eng.tile_for_batch(S * T) == 128 or tile_size == "128":
            assert eng.launch_count() - n0 == 2 * 3 * 15 + 1      # tensor-core engine: ONE chain, 15 kernels per step + the last update
        else:
            assert eng.launch_count() - n0 == (2 * 3 + 1) * (2 if S >= 2 else 1)      # two sequence groups = two parallel chains
        outs.append((x.clone(), d.clone(), hist.clone()))
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    xref, dref, href = onp.denoise_prior(p64, aa.astype(np.float64), cfg, iterations=2, steps_per_iter=3)
    x, d, hist = (t.cpu().numpy() for t in outs[0])
    assert np.max(np.abs(hist - href) / np.abs(href)) < 2e-5
    assert np.max(rel_err(d, dref)) < 1e-5
    err = np.abs(x - xref)
    assert np.median(err) < 2e-6 and (err > 1e-4).mean() < 0.01, (np.median(err), err.max())
