"""Thin host-side wrapper of one libpndf handle working on torch CUDA tensors (device memory + streams are
PyTorch's; all arithmetic is the library's fused sm_100a kernel)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class Engine:
    """One pndf_handle.  Inputs must be CUDA fp32 tensors on the handle's device (made contiguous here)."""

    def __init__(self, device=0, **cfg_kw):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("posendf_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.cfg = _lib.make_config(device=self.device.index, **cfg_kw)
        h = C.c_void_p()
        _lib.check(self.lib.pndf_create(C.byref(self.cfg), C.byref(h)))
        self._h = h
        n = C.c_size_t()
        _lib.check(self.lib.pndf_param_count(C.byref(self.cfg), C.byref(n)))
        self.param_count = n.value

    def close(self):
        if getattr(self, "_h", None):
            self.lib.pndf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights
    def set_weights_flat(self, flat):
        flat = np.ascontiguousarray(np.asarray(flat, dtype=np.float32).reshape(-1))
        _lib.check(self.lib.pndf_set_weights(self._h, flat.ctypes.data_as(C.c_void_p), flat.size))

    def set_weights_device(self, flat):
        """flat fp32 CUDA tensor in state_dict order; repacked by a gather kernel on the current stream (no host sync)"""
        flat = self._prep(flat, 1)
        _lib.check(self.lib.pndf_set_weights_device(self._h, flat.data_ptr(), flat.numel(), _stream_ptr(self.device)))
        self._flat_keepalive = flat     # the gather may still be in flight when the caller drops its reference

    # ---- helpers
    def _prep(self, t, last):
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.device == self.device):
            raise RuntimeError(f"expected a CUDA tensor on {self.device}")
        t = t.detach().to(torch.float32).reshape(-1, last).contiguous()
        return t

    def forward(self, pose, normalise=True):
        x = self._prep(pose, 84)
        B = x.shape[0]
        dist = torch.empty(B, 1, device=self.device, dtype=torch.float32)
        _lib.check(self.lib.pndf_forward(self._h, x.data_ptr(), B, int(normalise), dist.data_ptr(), _stream_ptr(self.device)))
        return dist

    def forward_grad(self, pose, g_up=None, normalise=True):
        x = self._prep(pose, 84)
        B = x.shape[0]
        dist = torch.empty(B, 1, device=self.device, dtype=torch.float32)
        grad = torch.empty(B, 21, 4, device=self.device, dtype=torch.float32)
        gp = None
        if g_up is not None:
            g_up = self._prep(g_up, 1)
            gp = g_up.data_ptr()
        _lib.check(self.lib.pndf_forward_grad(self._h, x.data_ptr(), B, int(normalise), gp, dist.data_ptr(), grad.data_ptr(),
                                              _stream_ptr(self.device)))
        return dist, grad

    def project_(self, pose, steps=1, renorm=False):
        """in place on a contiguous fp32 CUDA tensor; returns the distance at the start of the last step."""
        if not (pose.is_cuda and pose.dtype == torch.float32 and pose.is_contiguous() and pose.device == self.device):
            raise RuntimeError("project_ needs a contiguous fp32 CUDA tensor on the engine's device")
        B = pose.numel() // 84
        dist = torch.empty(B, 1, device=self.device, dtype=torch.float32)
        _lib.check(self.lib.pndf_project(self._h, pose.data_ptr(), B, int(steps), int(renorm), dist.data_ptr(),
                                         _stream_ptr(self.device)))
        return dist

    def project_host(self, pose_host, steps=1, renorm=False, out=None, dist_out=None):
        """HOST tensors in, HOST tensors out (pinned memory gives copy/compute overlap)."""
        if pose_host.is_cuda or pose_host.dtype != torch.float32 or not pose_host.is_contiguous():
            raise RuntimeError("project_host needs a contiguous fp32 CPU tensor")
        B = pose_host.numel() // 84
        out = out if out is not None else torch.empty_like(pose_host)
        dist_out = dist_out if dist_out is not None else torch.empty(B, 1, dtype=torch.float32)
        _lib.check(self.lib.pndf_project_host(self._h, pose_host.data_ptr(), out.data_ptr(), dist_out.data_ptr(), B, int(steps),
                                              int(renorm)))
        return out, dist_out

    def prior_grad(self, aa, g_up=None):
        a = self._prep(aa, 63)
        B = a.shape[0]
        dist = torch.empty(B, 1, device=self.device, dtype=torch.float32)
        grad = torch.empty(B, 21, 3, device=self.device, dtype=torch.float32)
        gp = None
        if g_up is not None:
            g_up = self._prep(g_up, 1)
            gp = g_up.data_ptr()
        _lib.check(self.lib.pndf_prior_grad(self._h, a.data_ptr(), B, gp, dist.data_ptr(), grad.data_ptr(), _stream_ptr(self.device)))
        return dist, grad

    def denoise_prior_(self, aa, iterations=10, steps_per_iter=50, lr=0.02, want_loss=False):
        """in place on a contiguous fp32 CUDA tensor (S,T,21,3) / (S,T,63); returns (dist (S,T), loss history or None)."""
        if not (aa.is_cuda and aa.dtype == torch.float32 and aa.is_contiguous() and aa.device == self.device and aa.dim() >= 3):
            raise RuntimeError("denoise_prior_ needs a contiguous fp32 CUDA tensor shaped (S, T, 63) or (S, T, 21, 3)")
        S, T = aa.shape[0], aa.shape[1]
        if aa.numel() != S * T * 63:
            raise RuntimeError("denoise_prior_: last dims must hold 21 joints x 3")
        dist = torch.empty(S, T, device=self.device, dtype=torch.float32)
        hist = torch.empty(iterations * steps_per_iter, S, device=self.device, dtype=torch.float32) if want_loss else None
        _lib.check(self.lib.pndf_denoise_prior(self._h, aa.data_ptr(), S, T, int(iterations), int(steps_per_iter), float(lr),
                                               dist.data_ptr(), hist.data_ptr() if want_loss else None, _stream_ptr(self.device)))
        return dist, hist

    def forward_grad_debug(self, pose, normalise=True):
        x = self._prep(pose, 84)
        B = min(x.shape[0], 32)
        n = C.c_size_t()
        _lib.check(self.lib.pndf_debug_dump_floats(C.byref(n)))
        dump = torch.zeros(32, n.value // 32, device=self.device, dtype=torch.float32)     # pose-major: [pose][5504]
        dist = torch.empty(B, 1, device=self.device, dtype=torch.float32)
        grad = torch.empty(B, 21, 4, device=self.device, dtype=torch.float32)
        _lib.check(self.lib.pndf_forward_grad_debug(self._h, x.data_ptr(), B, int(normalise), dist.data_ptr(), grad.data_ptr(),
                                                    dump.data_ptr(), _stream_ptr(self.device)))
        return dist, grad, dump

    def tile_for_batch(self, B) -> int:
        """tile size the library's batch-size rule picks for B poses: 8 or 32 (fused FFMA kernel) or 128 (tensor-core engine)"""
        t = C.c_int()
        _lib.check(self.lib.pndf_tile_for_batch(self._h, int(B), C.byref(t)))
        return t.value

    def set_tile_policy(self, tile=0):
        """0 = per launch from its batch size; 8 / 32 / 128 = pinned (split batches that must match the unsplit run bit for bit)"""
        _lib.check(self.lib.pndf_set_tile_policy(self._h, int(tile)))

    def launch_count(self) -> int:
        n = C.c_int64()
        _lib.check(self.lib.pndf_launch_count(self._h, C.byref(n)))
        return n.value

    def num_sms(self) -> int:
        n = C.c_int()
        _lib.check(self.lib.pndf_num_sms(self._h, C.byref(n)))
        return n.value


def fp32_peak_tflops(device=0, variant=0) -> float:
    lib = _lib.load()
    v = C.c_double()
    _lib.check(lib.pndf_fp32_peak(int(device), int(variant), C.byref(v)))
    return v.value


def knn_rerank(query, database, cand_idx, metric="geo", weighted=False):
    """data/dist_utils.py `geo` / `euc` .dist_calc + topk(5): CUDA tensors query (Q,21,4) fp32, database (N,21,4) fp32,
    cand_idx (Q,K) int32 -> (distances (Q,5) ascending, positions inside the candidate lists (Q,5) int32)."""
    lib = _lib.load()
    q = query.detach().to(torch.float32).reshape(-1, 84).contiguous()
    db = database.detach().to(torch.float32).reshape(-1, 84).contiguous()
    ci = cand_idx.detach().to(torch.int32).contiguous()
    if not (q.is_cuda and db.is_cuda and ci.is_cuda):
        raise RuntimeError("knn_rerank needs CUDA tensors (there is no CPU fallback)")
    Q, K = ci.shape
    val = torch.empty(Q, 5, device=q.device, dtype=torch.float32)
    pos = torch.empty(Q, 5, device=q.device, dtype=torch.int32)
    _lib.check(lib.pndf_knn_rerank(q.device.index or 0, q.data_ptr(), Q, db.data_ptr(), ci.data_ptr(), K,
                                   {"geo": 0, "euc": 1}[metric], int(weighted), val.data_ptr(), pos.data_ptr(), _stream_ptr(q.device)))
    return val, pos


def knn_exact(query, database, metric="geo", weighted=False):
    """exact 5 nearest database poses of every query under the reference's `geo` / `euc` metric (data/dist_utils.py:19-50)
    over the WHOLE database -- the labels data/prepare_traindata.py:138-170 approximates through faiss candidates.
    CUDA tensors query (Q,21,4), database (N,21,4) fp32 -> (distances (Q,5) ascending, database row indices (Q,5) int32)."""
    lib = _lib.load()
    q = query.detach().to(torch.float32).reshape(-1, 84).contiguous()
    db = database.detach().to(torch.float32).reshape(-1, 84).contiguous()
    if not (q.is_cuda and db.is_cuda):
        raise RuntimeError("knn_exact needs CUDA tensors (there is no CPU fallback)")
    Q, N = q.shape[0], db.shape[0]
    val = torch.empty(Q, 5, device=q.device, dtype=torch.float32)
    idx = torch.empty(Q, 5, device=q.device, dtype=torch.int32)
    _lib.check(lib.pndf_knn_exact(q.device.index or 0, q.data_ptr(), Q, db.data_ptr(), N, {"geo": 0, "euc": 1}[metric],
                                  int(weighted), val.data_ptr(), idx.data_ptr(), _stream_ptr(q.device)))
    return val, idx


def axis_angle_to_quaternion(aa):
    """pytorch3d.transforms.axis_angle_to_quaternion on a CUDA tensor (..., 3) -> (..., 4), real part first"""
    lib = _lib.load()
    a = aa.detach().to(torch.float32).contiguous()
    if not a.is_cuda:
        raise RuntimeError("axis_angle_to_quaternion needs a CUDA tensor (there is no CPU fallback)")
    out = torch.empty(*a.shape[:-1], 4, device=a.device, dtype=torch.float32)
    _lib.check(lib.pndf_axis_angle_to_quaternion(a.device.index or 0, a.data_ptr(), a.numel() // 3, out.data_ptr(), _stream_ptr(a.device)))
    return out


def quaternion_to_axis_angle(quat):
    """pytorch3d.transforms.quaternion_to_axis_angle on a CUDA tensor (..., 4) -> (..., 3)"""
    lib = _lib.load()
    q = quat.detach().to(torch.float32).contiguous()
    if not q.is_cuda:
        raise RuntimeError("quaternion_to_axis_angle needs a CUDA tensor (there is no CPU fallback)")
    out = torch.empty(*q.shape[:-1], 3, device=q.device, dtype=torch.float32)
    _lib.check(lib.pndf_quaternion_to_axis_angle(q.device.index or 0, q.data_ptr(), q.numel() // 4, out.data_ptr(), _stream_ptr(q.device)))
    return out
