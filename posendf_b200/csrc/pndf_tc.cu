// pndf_tc.cu -- the tensor-core DFNet path: PoseNDF distance, its analytic gradient and the projection step for LARGE batches with
// the seven DFNet layers (99.8 % of the flops) on the 5th-gen tensor cores.
//
// Reference semantics: PoseNDF.forward(train=False) + gradient() + the projection step, model/posendf.py:62-76,100-101,18-27 and
// experiments/sample_poses.py:70-74 -- identical to the FFMA kernel's (pndf_kernel.cuh); only where the DFNet GEMMs run changes.
//
// One projection step of B poses is a sequence of launches on one stream:
//   tc_enc_fwd_kernel     32-pose tiles: column normalise, structure encoder along the kinematic tree (the same device code as the
//                         fused kernel, 8 lanes per pose) -> z0 as tf32 hi / lo pairs, pose-major [pose][128]
//   6 x tc_gemm_kernel    z_{l+1} = act(z_l W_l^T + b_l): 3xTF32 tcgen05 GEMM (pndf_tc_gemm.cuh), epilogue = bias + activation +
//                         hi / lo split, activations stay pose-major in HBM / L2 (43 KB per pose for the whole chain)
//   tc_head_kernel        layer 6 (64 -> 1), output activation, dist; seeds the reverse chain t_5 = g_up phi_out'(s) w_6 phi'(pre_5)
//   6 x tc_gemm_kernel    t_{l-1} = (t_l W_l) * phi'(pre_{l-1}): the same GEMM on the transposed weight copies, epilogue multiplies
//                         by the activation derivative recovered from the stored activation z_l (sign for relu / lrelu,
//                         1 - exp(-beta z) for softplus); the last one leaves g0 = dd/dz0 in fp32
//   tc_enc_bwd_kernel     32-pose tiles: encoder forward again (cheaper than storing its intermediates), encoder reverse sweep,
//                         Jacobian of the column normalisation, x <- x - d * g, optional renormalisation, write-back (+ the fused
//                         gather: the same values to every peer GPU's gathered buffer)
// K-step projections repeat the sequence K times (the FFMA kernel keeps the tile on chip instead; here the step is 2x faster).
//
// Numerics: tools/tc_chain_probe.cu measured the chain (split accumulators + 128-deep K chunks) at the accuracy of the fp32 FMA
// chain; tests/test_gpu_parity.py runs the golden / oracle comparisons on this path too (tile policy 128).
#include "pndf_tc.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <array>
#include <map>
#include <vector>

#include "pndf_host.h"
#include "pndf_kernel.cuh"
#include "pndf_tc_gemm.cuh"

namespace pndf {

namespace {

__device__ __forceinline__ float tf32_rna(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}
// ---- GEMM epilogues (called by the thread owning output row `row` for each 32-column group; the kernel stores the outputs)
// The activation kind is a template parameter: with a run-time flag every element carried both branches and the epilogue of a
// 128 x 128 tile ran to ~2 400 SASS instructions per thread -- at two drain warps per scheduler that is longer than the two
// accumulator pairs of runway the MMA warp has, and the tensor pipe stalled on it (profiles/README.md, "epilogue exposure").
template <bool SOFT>
struct FwdEpi {          // z = act(acc + bias) -> hi / lo
    static constexpr int kOutputs = 2;
    const float* bias;
    float* out_hi;
    float* out_lo;
    int ldo;
    float par;           // slope (relu 0 / lrelu 0.01) or softplus beta
    uint32_t* mask;      // piecewise-linear kinds: bit j of word [tiled_offset(row, col0) / 32] = (pre-activation of column col0 + j > 0),
                         // all the reverse pass needs (128 coalesced bytes per warp instead of re-reading 4 KB of z); may be null
    __host__ __device__ float* out(int w) const { return w == 0 ? out_hi : out_lo; }
    const float* out_host(int w) const { return w == 0 ? out_hi : out_lo; }
    __device__ int ld() const { return ldo; }
    // the running sums start at the bias (16-byte aligned: csrc/pndf_capi.cu pads every small-parameter block)
    __device__ void init4(int col, float* r) const {
        const float4 b = __ldg(reinterpret_cast<const float4*>(bias + col));
        r[0] = b.x; r[1] = b.y; r[2] = b.z; r[3] = b.w;
    }
    __device__ void operator()(int row, int col0, const float (&v)[32], float (&hi)[32], float (&lo)[32]) const {
        const float inv_beta = SOFT ? 1.0f / par : 0.0f;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const float x = v[j];
            float dv;
            const float z = SOFT ? softplus_fast(x, par, inv_beta, dv) : (x > 0.0f ? x : x * par);
            hi[j] = tf32_rna(z);
            lo[j] = tf32_rna(z - hi[j]);
        }
        if (!SOFT && mask) {
            uint32_t bits = 0;
#pragma unroll
            for (int j = 0; j < 32; ++j) bits |= (v[j] > 0.0f ? 1u : 0u) << j;
            mask[pndf_tc::tiled_offset(row, col0, ldo) >> 5] = bits;      // consecutive lanes = consecutive rows = consecutive words
        }
    }
};
template <bool SOFT>
struct BwdEpi {          // t = acc * act'(pre) with act' recovered from the stored activation z -> hi / lo
    static constexpr int kOutputs = 2;
    const float* z_hi;
    const float* z_lo;
    float* out_hi;
    float* out_lo;
    int ldo;
    float par;
    const uint32_t* mask;      // piecewise-linear kinds: the forward epilogue's sign bits (see FwdEpi); softplus reads z instead
    __host__ __device__ float* out(int w) const { return w == 0 ? out_hi : out_lo; }
    const float* out_host(int w) const { return w == 0 ? out_hi : out_lo; }
    __device__ int ld() const { return ldo; }
    __device__ void init4(int, float* r) const { r[0] = r[1] = r[2] = r[3] = 0.0f; }
    __device__ void operator()(int row, int col0, const float (&v)[32], float (&hi)[32], float (&lo)[32]) const {
        const size_t off = pndf_tc::tiled_offset(row, col0, ldo);      // 32 contiguous floats (all operands are in the tiled layout)
        if (!SOFT) {
            const uint32_t bits = __ldg(mask + (off >> 5));
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const float t = v[j] * (((bits >> j) & 1u) ? 1.0f : par);
                hi[j] = tf32_rna(t);
                lo[j] = tf32_rna(t - hi[j]);
            }
            return;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float zz[8], zl[8];
            pndf_tc::ld_global_nc_v8(z_hi + off + 8 * j, zz);
            pndf_tc::ld_global_nc_v8(z_lo + off + 8 * j, zl);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const float d = -expm1f(-par * (zz[k] + zl[k]));
                const float t = v[8 * j + k] * d;
                hi[8 * j + k] = tf32_rna(t);
                lo[8 * j + k] = tf32_rna(t - hi[8 * j + k]);
            }
        }
    }
};
struct G0Epi {           // the last reverse op: dd/dz0 in fp32
    static constexpr int kOutputs = 1;
    float* o;
    int ldo;
    __host__ __device__ float* out(int) const { return o; }
    const float* out_host(int) const { return o; }
    __device__ int ld() const { return ldo; }
    __device__ void init4(int, float* r) const { r[0] = r[1] = r[2] = r[3] = 0.0f; }
    __device__ void operator()(int, int, const float (&v)[32], float (&o0)[32], float (&)[32]) const {
#pragma unroll
        for (int j = 0; j < 32; ++j) o0[j] = v[j];
    }
};

// ---- weights: flat fp32 parameter vector -> tf32 hi / lo copies, forward layout W_l [n_out][k_pad] and reverse layout W_l^T [n_in_pad][n_out]
struct SplitParams {
    const float* flat;
    float* hi;
    float* lo;
    long long w_off[6];      // offset of W_l in the flat vector
    long long f_off[6];      // offset of the forward copy of layer l in hi / lo
    long long r_off[6];      // offset of the reverse copy
    int n_in[6], n_out[6], k_pad[6], n_in_pad[6];
    int f_tile[6];           // row tile of the forward copy (= the N tile of its GEMM: 128, 64 for the 64-wide layer)
    long long total;
};
__global__ void __launch_bounds__(256) tc_split_weights_kernel(const SplitParams p) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < p.total; i += (long long)gridDim.x * blockDim.x) {
        int l = 0;
        bool rev = false;
        long long base = 0;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            if (i >= p.f_off[k]) { l = k; rev = false; base = p.f_off[k]; }
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            if (i >= p.r_off[k]) { l = k; rev = true; base = p.r_off[k]; }
        }
        // element e of a TILED [rows][cols] matrix (pndf_tc_gemm.cuh::tiled_offset): e = ((rt * cols/32 + cb) * T + r) * 32 + c
        const long long e = i - base;
        const int cols = rev ? p.n_out[l] : p.k_pad[l], T = rev ? 128 : p.f_tile[l];
        const int c = (int)(e & 31);
        const long long q = e >> 5;
        const int r = (int)(q % T);
        const long long q2 = q / T;
        const int cb = (int)(q2 % (cols / 32)), rt = (int)(q2 / (cols / 32));
        const int row = rt * T + r, col = cb * 32 + c;
        float w = 0.0f;
        if (!rev) {      // forward copy: row = output unit n, column = input feature k
            if (col < p.n_in[l]) w = p.flat[p.w_off[l] + (long long)row * p.n_in[l] + col];
        } else {         // reverse copy: row = input feature k, column = output unit n
            if (row < p.n_in[l]) w = p.flat[p.w_off[l] + (long long)col * p.n_in[l] + row];
        }
        const float h = tf32_rna(w);
        p.hi[i] = h;
        p.lo[i] = tf32_rna(w - h);
    }
}

// ---- encoder head of a step: 32-pose tile -> z0 hi / lo
struct EncParams {
    const float* pose;       // [B][84]
    const float* encw;       // 3516 floats or nullptr
    float* z0_hi;            // [P][z0_ld]
    float* z0_lo;
    const float* g0;         // [P][128] (reverse kernel)
    const float* feat;       // [P][128] fp32 encoder features of the forward kernel (reverse kernel; tiled layout)
    float* feat_out;         // same buffer, written by the forward kernel when a reverse pass follows
    const float* dist;       // [B]      (reverse kernel: d of this step)
    float* pose_out;         // [B][84] or nullptr
    float* grad;             // [B][84] or nullptr
    float* peer_pose[kMaxPeers];
    long long B;
    int z0_ld, normalise, use_enc, enc_act, do_step, renorm, n_peers;
    float enc_beta;
    // prior mode (experiments/motion_denoise.py:81-83): `pose` is [B][63] axis-angle, `grad` its [B][63] VJP; the forward kernel applies
    // the pending Adam update of a denoise loop first (same prologue as the fused kernel's, pndf_kernel.cuh)
    int input_kind;
    DenoiseFuse dn;
};
// shared-memory layout: the forward kernel needs no gradient buffer (5 CTAs per SM), the reverse kernel no encoder recomputation
// (3 CTAs per SM): both are latency-bound prologue -> tree walk -> epilogue pipelines, occupancy is what overlaps them
constexpr int kEncSmX = 0;                               // [128][32] features (swizzled, as the fused kernel)
template <bool REVERSE> __host__ __device__ constexpr int enc_sm_y() { return kEncSmX + 128 * 32 * 4; }      // reverse: [224][32] gradients: rows [0,128) dd/dz0 (then the
                                                                                         // projected pose), rows [128,212) qbar
template <bool REVERSE> __host__ __device__ constexpr int enc_sm_w() { return enc_sm_y<REVERSE>() + (REVERSE ? 224 * 32 * 4 : 0); }
template <bool REVERSE> __host__ __device__ constexpr int enc_sm_qs() { return enc_sm_w<REVERSE>() + ((kEncFloats * 4 + 127) / 128) * 128; }
template <bool REVERSE> __host__ __device__ constexpr int enc_sm_nrm() { return enc_sm_qs<REVERSE>() + kTileM * kXS * 4; }
template <bool REVERSE> __host__ __device__ constexpr int enc_sm_total() { return enc_sm_nrm<REVERSE>() + 4 * 32 * 4; }

template <bool ESOFT, bool REVERSE>
__global__ void __launch_bounds__(256) tc_enc_kernel(const EncParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    float* X = reinterpret_cast<float*>(smem + kEncSmX);
    float* Y = reinterpret_cast<float*>(smem + enc_sm_y<REVERSE>());
    float* encw = reinterpret_cast<float*>(smem + enc_sm_w<REVERSE>());
    float* qs = reinterpret_cast<float*>(smem + enc_sm_qs<REVERSE>());
    float* nrm = reinterpret_cast<float*>(smem + enc_sm_nrm<REVERSE>());
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long pose0 = (long long)blockIdx.x * kTileM;
    const int nvalid = (int)min((long long)kTileM, p.B - pose0);
    EncLane enc;
    enc.l = lane & 7; enc.base = lane & 24; enc.m = warp * 4 + (lane >> 3);
    const float apar = ESOFT ? p.enc_beta : ((p.enc_act == ACT_RELU) ? 0.0f : 0.01f);

    const bool aa_in = (p.input_kind != IN_QUAT);
    if (!aa_in) {
        for (int idx = tid; idx < kTileM * 84; idx += 256) qs[idx] = (idx < nvalid * 84) ? __ldg(p.pose + pose0 * 84 + idx) : 0.0f;      // raw x, scaled in place
    } else {
        __shared__ float s_red[8];
        __shared__ float s_scale[kTileM + 1];
        const float* src = p.pose + pose0 * 63;
        const bool dn = !REVERSE && (p.dn.pending != 0);
        if (dn) {
            // per-sequence loss scale of the PREVIOUS step for every sequence that has a frame in this tile:
            // c = mean_t dist_prev[s][t] (same summation order as seq_adam_kernel), scale = weight * 2 c / T
            const int T = p.dn.T;
            const long long s_lo = pose0 / T, s_hi = (pose0 + nvalid - 1) / T;
            for (long long sq = s_lo; sq <= s_hi; ++sq) {
                const float* dp = p.dn.dist_prev + sq * T;
                float acc = 0.0f;
                for (int t = tid; t < T; t += 256) acc += dp[t];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                if (lane == 0) s_red[warp] = acc;
                __syncthreads();
                if (tid == 0) {
                    float tot = 0.0f;
                    for (int w = 0; w < 8; ++w) tot += s_red[w];
                    const float cmean = tot / (float)T;
                    s_scale[sq - s_lo] = p.dn.ap.weight * 2.0f * cmean / (float)T;
                    if (p.dn.loss_out != nullptr && sq * T >= pose0) p.dn.loss_out[sq] = p.dn.ap.weight * cmean * cmean;
                }
                __syncthreads();
            }
        }
        for (int idx = tid; idx < kTileM * 21; idx += 256) {
            const int m = idx / 21, j = idx - m * 21;
            float a[3] = {0.f, 0.f, 0.f}, q[4];
            if (m < nvalid) {
                if (dn) {
                    const long long e0 = (pose0 * 21 + idx) * 3;
                    const float scale = s_scale[(pose0 + m) / p.dn.T - pose0 / p.dn.T];
#pragma unroll
                    for (int k3 = 0; k3 < 3; ++k3) {
                        float av = p.dn.pose_rw[e0 + k3], mv = p.dn.m[e0 + k3], vv = p.dn.v[e0 + k3];
                        dn_adam_update(av, mv, vv, p.dn.graw[e0 + k3], scale, p.dn.ap);
                        p.dn.pose_rw[e0 + k3] = av; p.dn.m[e0 + k3] = mv; p.dn.v[e0 + k3] = vv;
                        a[k3] = av;
                    }
                } else {
                    // plain loads: in a denoise step the forward kernel of this step has just rewritten these values
                    a[0] = src[idx * 3]; a[1] = src[idx * 3 + 1]; a[2] = src[idx * 3 + 2];
                }
            }
            aa_to_quat(a, q);
#pragma unroll
            for (int cpt = 0; cpt < 4; ++cpt) qs[m * kXS + j * 4 + cpt] = (m < nvalid) ? q[cpt] : 0.0f;
        }
    }
    if (p.use_enc)
        for (int i = tid; i < kEncFloats; i += 256) encw[i] = __ldg(p.encw + i);
    if (REVERSE) {      // dd/dz0 and the features of this tile, pose-major in HBM -> [feature][pose]
        for (int idx = tid; idx < kTileM * 128; idx += 256) {
            const int m = idx >> 7, f = idx & 127;
            const size_t off = pndf_tc::tiled_offset(pose0 + m, f, 128);
            Y[swz(f, m)] = (m < nvalid) ? __ldg(p.g0 + off) : 0.0f;
            if (p.use_enc) X[swz(f, m)] = (m < nvalid) ? __ldg(p.feat + off) : 0.0f;
        }
    }
    __syncthreads();
    // ---- column norms, q = x / n (8 lanes per pose)
    {
        const int cpt = enc.l & 3, hf = enc.l >> 2;
        if (p.normalise) {
            float sq = 0.0f;
            for (int j = hf; j < 21; j += 2) {
                const float x = qs[enc.m * kXS + j * 4 + cpt];
                sq = fmaf(x, x, sq);
            }
            sq += __shfl_xor_sync(0xffffffffu, sq, 4);
            const float n = fmaxf(sqrtf(sq), 1e-12f);
            if (hf == 0) nrm[cpt * 32 + enc.m] = n;
            for (int j = hf; j < 21; j += 2) qs[enc.m * kXS + j * 4 + cpt] = qs[enc.m * kXS + j * 4 + cpt] / n;
        }
        __syncwarp();
        if (!REVERSE) {
            if (p.use_enc) {
                encoder_forward<ESOFT>(encw, qs, X, nullptr, enc, apar);
                if (enc.l < 2) X[swz(126 + enc.l, enc.m)] = 0.0f;
            } else {
                for (int e = enc.l; e < 128; e += 8) X[swz(e, enc.m)] = (e < 84) ? qs[enc.m * kXS + e] : 0.0f;
            }
        }
    }
    if (!REVERSE) {
        __syncthreads();
        // z0 -> pose-major tf32 hi / lo rows of width z0_ld (128 with the encoder, 96 without) + the fp32 features for the reverse kernel
        const int cols = p.z0_ld;
        for (int idx = tid; idx < kTileM * (cols / 4); idx += 256) {
            const int m = idx / (cols / 4), c4 = (idx - m * (cols / 4)) * 4;
            if (m >= nvalid) continue;
            float z[4], h[4], l[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                z[k] = X[swz(c4 + k, m)];
                h[k] = tf32_rna(z[k]);
                l[k] = tf32_rna(z[k] - h[k]);
            }
            const size_t off = pndf_tc::tiled_offset(pose0 + m, c4, cols);
            *reinterpret_cast<float4*>(p.z0_hi + off) = make_float4(h[0], h[1], h[2], h[3]);
            *reinterpret_cast<float4*>(p.z0_lo + off) = make_float4(l[0], l[1], l[2], l[3]);
            if (p.feat_out != nullptr && p.use_enc)
                *reinterpret_cast<float4*>(p.feat_out + pndf_tc::tiled_offset(pose0 + m, c4, 128)) = make_float4(z[0], z[1], z[2], z[3]);
        }
        return;
    }
    // ---- reverse: encoder adjoint sweep, Jacobian of the column normalisation, projection step
    {
        const int m = enc.m;
        if (p.use_enc) {
            encoder_backward<ESOFT>(encw, qs, X, Y, enc, apar);      // qbar -> Y rows [128, 212)
        } else {
            for (int e = enc.l; e < 84; e += 8) Y[swz(128 + e, m)] = Y[swz(e, m)];
            __syncwarp();
        }
        const float d = (m < nvalid) ? __ldg(p.dist + pose0 + m) : 0.0f;
        const int cpt = enc.l & 3, hf = enc.l >> 2;
        float n = 1.0f, dot = 0.0f;
        if (p.normalise) {
            n = nrm[cpt * 32 + m];
            for (int j = hf; j < 21; j += 2) dot = fmaf(qs[m * kXS + j * 4 + cpt], Y[swz(128 + j * 4 + cpt, m)], dot);
            dot += __shfl_xor_sync(0xffffffffu, dot, 4);
            if (n <= 1e-12f) dot = 0.0f;
        }
        __syncwarp();
        for (int j = hf; j < 21; j += 2) {
            const int e = j * 4 + cpt;
            float g = Y[swz(128 + e, m)];
            if (p.normalise) g = (g - qs[m * kXS + e] * dot) / n;
            Y[swz(128 + e, m)] = g;
            if (p.do_step) {      // the projected pose takes the place of dd/dz0 (rows [0, 84) of this warp's columns)
                const float x = (m < nvalid) ? __ldg(p.pose + (pose0 + m) * 84 + e) : 0.0f;
                Y[swz(e, m)] = __fsub_rn(x, __fmul_rn(d, g));
            }
        }
        if (p.do_step && p.renorm) {
            __syncwarp();
            for (int j = enc.l; j < 21; j += 8) {
                float sq = 0.0f;
#pragma unroll
                for (int c4 = 0; c4 < 4; ++c4) sq = fmaf(Y[swz(j * 4 + c4, m)], Y[swz(j * 4 + c4, m)], sq);
                const float inv = 1.0f / sqrtf(sq);
#pragma unroll
                for (int c4 = 0; c4 < 4; ++c4) Y[swz(j * 4 + c4, m)] *= inv;
            }
        }
    }
    __syncthreads();
    if (aa_in) {      // prior mode: the VJP through aa -> quat, no step
        if (p.grad != nullptr) {
            const float* src = p.pose + pose0 * 63;
            float* dst = p.grad + pose0 * 63;
            for (int idx = tid; idx < nvalid * 21; idx += 256) {
                const int m = idx / 21, j = idx - m * 21;
                const float a[3] = {src[idx * 3], src[idx * 3 + 1], src[idx * 3 + 2]};
                const float qb[4] = {Y[swz(128 + j * 4, m)], Y[swz(128 + j * 4 + 1, m)], Y[swz(128 + j * 4 + 2, m)], Y[swz(128 + j * 4 + 3, m)]};
                float ab[3];
                aa_to_quat_vjp(a, qb, ab);
                dst[idx * 3] = ab[0]; dst[idx * 3 + 1] = ab[1]; dst[idx * 3 + 2] = ab[2];
            }
        }
        return;
    }
    for (int idx = tid; idx < nvalid * 84; idx += 256) {
        const int m = idx / 84, e = idx - m * 84;
        if (p.grad != nullptr) p.grad[pose0 * 84 + idx] = Y[swz(128 + e, m)];
        if (p.pose_out != nullptr) {
            const float v = Y[swz(e, m)];
            p.pose_out[pose0 * 84 + idx] = v;
            for (int r = 0; r < p.n_peers; ++r) p.peer_pose[r][pose0 * 84 + idx] = v;
        }
    }
}

// ---- layer 6 + output activation + seed of the reverse chain, one thread per pose
struct HeadParams {
    const float* z6_hi;      // [P][64]
    const float* z6_lo;
    const float* w6;         // 64
    const float* b6;         // 1
    const float* g_up;       // [B] or nullptr
    float* dist;             // [B] or nullptr
    float* dist_keep;        // [B] internal copy for the reverse kernel (always written)
    float* peer_dist[kMaxPeers];
    float* t5_hi;            // [P][64] or nullptr (forward only)
    float* t5_lo;
    long long B;
    int soft, n_peers;
    float slope, beta;
};
__global__ void __launch_bounds__(128) tc_head_kernel(const HeadParams p) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.B) return;
    float z[64];
    float s = 0.0f;
#pragma unroll
    for (int k4 = 0; k4 < 16; ++k4) {
        const size_t off = pndf_tc::tiled_offset(b, 4 * k4, 64);
        const float4 h = __ldg(reinterpret_cast<const float4*>(p.z6_hi + off));
        const float4 l = __ldg(reinterpret_cast<const float4*>(p.z6_lo + off));
        z[4 * k4] = h.x + l.x; z[4 * k4 + 1] = h.y + l.y; z[4 * k4 + 2] = h.z + l.z; z[4 * k4 + 3] = h.w + l.w;
    }
    // the fused kernel sums 8 lanes x 8 terms and then a 3-level butterfly; any fixed order is as good against the fp64 oracle
#pragma unroll
    for (int k = 0; k < 64; ++k) s = fmaf(__ldg(p.w6 + k), z[k], s);
    s += __ldg(p.b6);
    float dv;
    const float d = act_eval(s, p.soft ? ACT_SOFTPLUS : ACT_RELU, p.beta, dv);
    p.dist_keep[b] = d;
    if (p.dist != nullptr) p.dist[b] = d;
    for (int r = 0; r < p.n_peers; ++r)
        if (p.peer_dist[r] != nullptr) p.peer_dist[r][b] = d;
    if (p.t5_hi == nullptr) return;
    const float gs = (p.g_up != nullptr ? __ldg(p.g_up + b) : 1.0f) * dv;
#pragma unroll
    for (int k4 = 0; k4 < 16; ++k4) {
        float h[4], l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float zz = z[4 * k4 + k];
            const float d5 = p.soft ? -expm1f(-p.beta * zz) : (zz > 0.0f ? 1.0f : p.slope);
            const float t = gs * __ldg(p.w6 + 4 * k4 + k) * d5;
            h[k] = tf32_rna(t);
            l[k] = tf32_rna(t - h[k]);
        }
        const size_t off = pndf_tc::tiled_offset(b, 4 * k4, 64);
        *reinterpret_cast<float4*>(p.t5_hi + off) = make_float4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<float4*>(p.t5_lo + off) = make_float4(l[0], l[1], l[2], l[3]);
    }
}

}  // namespace

// ------------------------------------------------------------------------------------------------ host side
struct TcState {
    explicit TcState(const pndf_config& c) : cfg(c), L(c) {}
    pndf_config cfg;
    ParamLayout L;                 // where W_l sits in the flat parameter vector; L.width = in_dim, 256, 512, 1024, 512, 256, 64, 1
    int kpad[6], ninpad[6];        // K of the forward op l (n_in padded to 32), N of the reverse op l (n_in padded to 128)
    int zw[7];                     // width of the stored activation z_l: z_0 padded to kpad[0], then the layer widths
    DevBuf<float> w_hi, w_lo;
    long long f_off[6], r_off[6], w_total = 0;
    // activations, for as many poses (a multiple of 128) as `act` holds act_per_pose floats: forward z_0..z_6 (hi, lo), reverse
    // t_5..t_0 (hi, lo), g0, dist, encoder features, sign masks.  The offsets are per pose: buffer x of a P-pose allocation starts at
    // float P * x_off
    DevBuf<float> act;
    long long z_off[7], t_off[6], g0_off = 0, dist_off = 0, mask_off[7] = {0, 0, 0, 0, 0, 0, 0}, feat_off = 0, act_per_pose = 0;
    int num_sms = 148;
    // tensor maps of the GEMM launches, keyed by (operand / output addresses, shape): a step repeats the same twelve launches, and
    // six cuTensorMapEncodeTiled calls per launch are host time the 15-launch step of a small batch does not have
    std::map<std::array<unsigned long long, 8>, pndf_tc::GemmMaps> maps;
    std::string err;
};

static int tc_fail(TcState* s, const std::string& m) { s->err = m; return 1; }
// 0 if the last launch was accepted, else records `what` + the CUDA error string
static int tc_check(TcState* s, const char* what) {
    const cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) return 0;
    return tc_fail(s, std::string(what) + ": " + cudaGetErrorString(e));
}
const char* tc_last_error(TcState* s) { return s ? s->err.c_str() : "null tc state"; }

int tc_create(TcState** out, const pndf_config* cfg) {
    TcState* s = new TcState(*cfg);
    const int* w = s->L.width;
    long long tot = 0;
    for (int l = 0; l < 6; ++l) {
        s->kpad[l] = (w[l] + 31) / 32 * 32;
        s->ninpad[l] = (w[l] + 127) / 128 * 128;
    }
    for (int l = 0; l < 6; ++l) { s->f_off[l] = tot; tot += (long long)w[l + 1] * s->kpad[l]; }
    for (int l = 0; l < 6; ++l) { s->r_off[l] = tot; tot += (long long)s->ninpad[l] * w[l + 1]; }
    s->w_total = tot;
    s->zw[0] = s->kpad[0];
    for (int l = 1; l < 7; ++l) s->zw[l] = w[l];
    long long off = 0;
    for (int l = 0; l < 7; ++l) { s->z_off[l] = off; off += 2 * s->zw[l]; }
    for (int l = 0; l < 6; ++l) { s->t_off[l] = off; off += 2 * w[l + 1]; }      // t_l has the width of layer l's output
    s->g0_off = off; off += 128;
    s->dist_off = off; off += 1;
    s->feat_off = off; off += 128;                                                 // fp32 encoder features (forward -> reverse kernel)
    for (int l = 1; l <= 5; ++l) { s->mask_off[l] = off; off += s->zw[l] / 32; }  // sign bits of the pre-activations of z_1 .. z_5
    s->act_per_pose = off;
    cudaDeviceGetAttribute(&s->num_sms, cudaDevAttrMultiProcessorCount, cfg->device);
    if (s->w_hi.reserve(tot, "tf32 weights (hi)") || s->w_lo.reserve(tot, "tf32 weights (lo)") || !pndf_tc::encode_fn()) {
        delete s;
        return 1;
    }
    *out = s;
    return 0;
}

void tc_destroy(TcState* s) { delete s; }

int tc_set_weights(TcState* s, const float* flat_dev, cudaStream_t st) {
    SplitParams p{};
    p.flat = flat_dev; p.hi = s->w_hi.get(); p.lo = s->w_lo.get(); p.total = s->w_total;
    for (int l = 0; l < 6; ++l) {
        p.w_off[l] = s->L.w_off[l]; p.f_off[l] = s->f_off[l]; p.r_off[l] = s->r_off[l];
        p.n_in[l] = s->L.width[l]; p.n_out[l] = s->L.width[l + 1]; p.k_pad[l] = s->kpad[l]; p.n_in_pad[l] = s->ninpad[l];
        p.f_tile[l] = (s->L.width[l + 1] % 128 == 0) ? 128 : 64;
    }
    tc_split_weights_kernel<<<148 * 8, 256, 0, st>>>(p);
    return tc_check(s, "tc_split_weights_kernel launch");
}

int tc_reserve(TcState* s, long long B) {
    const size_t need = (size_t)((B + 127) / 128 * 128 * s->act_per_pose);
    if (need <= s->act.size()) return 0;
    s->maps.clear();      // the cached tensor maps point into the buffer being replaced
    if (s->act.reserve(need, "tensor-core activations", true)) return tc_fail(s, pndf_last_error());
    return 0;
}

template <int NT, class Epi>
static int launch_gemm(TcState* s, const float* a_hi, const float* a_lo, long long P, int K, const float* b_hi, const float* b_lo, int N,
                       const Epi& epi, cudaStream_t st) {
    using namespace pndf_tc;
    const std::array<unsigned long long, 8> key = {(unsigned long long)(uintptr_t)a_hi, (unsigned long long)(uintptr_t)a_lo,
                                                   (unsigned long long)(uintptr_t)b_hi, (unsigned long long)(uintptr_t)epi.out_host(0),
                                                   (unsigned long long)(uintptr_t)epi.out_host(Epi::kOutputs - 1), (unsigned long long)P,
                                                   (unsigned long long)K, ((unsigned long long)N << 32) | (unsigned)NT};
    auto it = s->maps.find(key);
    if (it == s->maps.end()) {
        GemmMaps m;
        if (!make_map(&m.a_hi, a_hi, P, K, pndf_tc::kTM) || !make_map(&m.a_lo, a_lo, P, K, pndf_tc::kTM) || !make_map(&m.b_hi, b_hi, N, K, NT) ||
            !make_map(&m.b_lo, b_lo, N, K, NT))
            return tc_fail(s, "cuTensorMapEncodeTiled failed");
        for (int w = 0; w < Epi::kOutputs; ++w)
            if (!make_out_map(&m.out[w], epi.out_host(w), P, epi.ldo)) return tc_fail(s, "cuTensorMapEncodeTiled failed (output)");
        if (Epi::kOutputs == 1) m.out[1] = m.out[0];
        if (s->maps.size() > 256) s->maps.clear();      // batch sizes come and go; a map is cheap to rebuild
        it = s->maps.emplace(key, m).first;
    }
    const GemmMaps& maps = it->second;
    auto kern = tc_gemm_kernel<NT, Epi>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, pndf_tc::smem_bytes<NT>()) != cudaSuccess)
        return tc_fail(s, "cudaFuncSetAttribute failed");
    // (pndf::kThreads is the fused kernel's 256; this kernel is compiled for pndf_tc::kThreads = 320)
    const int m_tiles = (int)(P / pndf_tc::kTM), n_tiles = N / NT;
    const int grid = std::min(m_tiles * n_tiles, s->num_sms);
    kern<<<grid, pndf_tc::kThreads, pndf_tc::smem_bytes<NT>(), st>>>(maps, K, m_tiles, n_tiles, epi);
    return tc_check(s, "tc_gemm_kernel launch");
}

int tc_run(TcState* s, const KParams& a, int want_grad, cudaStream_t st, int64_t* launches) {
    if (a.input_kind != IN_QUAT && (a.steps != 1 || a.do_step || a.pose_out != nullptr))
        return tc_fail(s, "tensor-core path: axis-angle input is the prior mode (one evaluation, no step)");
    if (tc_reserve(s, a.B)) return 1;
    const long long P = (a.B + 127) / 128 * 128;
    const pndf_config& cfg = s->cfg;
    const bool dsoft = cfg.df_act == PNDF_ACT_SOFTPLUS, esoft = cfg.enc_act == PNDF_ACT_SOFTPLUS;
    const float dpar = dsoft ? cfg.df_beta : (cfg.df_act == PNDF_ACT_RELU ? 0.0f : 0.01f);
    const int* zw = s->zw;
    const int* widths = s->L.width;
    const long long cap = (long long)(s->act.size() / s->act_per_pose);      // poses the activation buffers hold (>= P)
    float* act = s->act.get();
    auto zhi = [&](int l) { return act + cap * s->z_off[l]; };
    auto zlo = [&](int l) { return zhi(l) + P * zw[l]; };
    auto thi = [&](int l) { return act + cap * s->t_off[l]; };
    auto tlo = [&](int l) { return thi(l) + P * widths[l + 1]; };
    auto maskp = [&](int l) { return reinterpret_cast<uint32_t*>(act + cap * s->mask_off[l]); };
    float* g0 = act + cap * s->g0_off;
    float* featp = act + cap * s->feat_off;
    float* dkeep = act + cap * s->dist_off;
    cudaFuncSetAttribute(tc_enc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, enc_sm_total<false>());
    cudaFuncSetAttribute(tc_enc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, enc_sm_total<true>());
    cudaFuncSetAttribute(tc_enc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, enc_sm_total<false>());
    cudaFuncSetAttribute(tc_enc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, enc_sm_total<true>());
    const unsigned tiles32 = (unsigned)((a.B + kTileM - 1) / kTileM);
    const float* pose_cur = a.pose_in;
    for (int step = 0; step < a.steps; ++step) {
        const bool last = (step == a.steps - 1);
        EncParams ep{};
        ep.pose = pose_cur; ep.encw = a.encw; ep.z0_hi = zhi(0); ep.z0_lo = zlo(0); ep.B = a.B; ep.z0_ld = zw[0];
        ep.normalise = a.normalise; ep.use_enc = cfg.use_enc; ep.enc_act = cfg.enc_act; ep.enc_beta = cfg.enc_beta;
        ep.input_kind = a.input_kind;
        if (a.dn.pending) ep.dn = a.dn;
        ep.feat_out = want_grad ? featp : nullptr;
        if (esoft) tc_enc_kernel<true, false><<<tiles32, 256, enc_sm_total<false>(), st>>>(ep);
        else tc_enc_kernel<false, false><<<tiles32, 256, enc_sm_total<false>(), st>>>(ep);
        if (tc_check(s, "tc_enc_kernel (forward) launch")) return 1;
        // ---- forward chain
        for (int l = 0; l < 6; ++l) {
            const float* bh = s->w_hi.get() + s->f_off[l];
            const float* bl = s->w_lo.get() + s->f_off[l];
            const int N = widths[l + 1];
            auto fwd = [&](auto fe) {
                return (N % 128 == 0) ? launch_gemm<128>(s, zhi(l), zlo(l), P, s->kpad[l], bh, bl, N, fe, st)
                                      : launch_gemm<64>(s, zhi(l), zlo(l), P, s->kpad[l], bh, bl, N, fe, st);
            };
            uint32_t* mk = (l < 5 && want_grad) ? maskp(l + 1) : nullptr;
            const int rc = dsoft ? fwd(FwdEpi<true>{a.bias[l], zhi(l + 1), zlo(l + 1), zw[l + 1], dpar, nullptr})
                                 : fwd(FwdEpi<false>{a.bias[l], zhi(l + 1), zlo(l + 1), zw[l + 1], dpar, mk});
            if (rc) return 1;
        }
        HeadParams hp{};
        hp.z6_hi = zhi(6); hp.z6_lo = zlo(6); hp.w6 = a.w6; hp.b6 = a.bias[6]; hp.g_up = a.g_up; hp.B = a.B;
        hp.dist = last ? a.dist : nullptr; hp.dist_keep = dkeep; hp.soft = dsoft ? 1 : 0; hp.slope = dsoft ? 0.0f : dpar; hp.beta = cfg.df_beta;
        if (last) { hp.n_peers = a.n_peers; for (int r = 0; r < a.n_peers; ++r) hp.peer_dist[r] = a.peer_dist[r]; }
        if (want_grad) { hp.t5_hi = thi(5); hp.t5_lo = tlo(5); }
        tc_head_kernel<<<(unsigned)((a.B + 127) / 128), 128, 0, st>>>(hp);
        if (tc_check(s, "tc_head_kernel launch")) return 1;
        if (launches) *launches += 8;
        if (!want_grad) break;
        // ---- reverse chain: op l maps t_l (width n_out[l]) through W_l to the input side (width n_in[l])
        for (int l = 5; l >= 0; --l) {
            const float* bh = s->w_hi.get() + s->r_off[l];
            const float* bl = s->w_lo.get() + s->r_off[l];
            const int K = widths[l + 1], N = s->ninpad[l];
            int rc;
            if (l > 0) {
                rc = dsoft ? launch_gemm<128>(s, thi(l), tlo(l), P, K, bh, bl, N, BwdEpi<true>{zhi(l), zlo(l), thi(l - 1), tlo(l - 1), zw[l], dpar, nullptr}, st)
                           : launch_gemm<128>(s, thi(l), tlo(l), P, K, bh, bl, N, BwdEpi<false>{zhi(l), zlo(l), thi(l - 1), tlo(l - 1), zw[l], dpar, maskp(l)}, st);
            } else {
                G0Epi ge{g0, 128};
                rc = launch_gemm<128>(s, thi(0), tlo(0), P, K, bh, bl, N, ge, st);
            }
            if (rc) return 1;
        }
        EncParams rp = ep;
        rp.g0 = g0; rp.dist = dkeep; rp.do_step = a.do_step; rp.renorm = a.renorm;
        rp.grad = last ? a.grad : nullptr;
        rp.pose_out = a.do_step ? a.pose_out : nullptr;
        if (last && a.do_step) { rp.n_peers = a.n_peers; for (int r = 0; r < a.n_peers; ++r) rp.peer_pose[r] = a.peer_pose[r]; }
        rp.feat = featp; rp.feat_out = nullptr; rp.pose = pose_cur;
        rp.dn = DenoiseFuse{};      // the update was applied by the forward kernel
        if (esoft) tc_enc_kernel<true, true><<<tiles32, 256, enc_sm_total<true>(), st>>>(rp);
        else tc_enc_kernel<false, true><<<tiles32, 256, enc_sm_total<true>(), st>>>(rp);
        if (tc_check(s, "tc_enc_kernel (reverse) launch")) return 1;
        if (launches) *launches += 7;
        pose_cur = a.pose_out;       // the next step starts from the projected poses
    }
    return 0;
}

}  // namespace pndf
