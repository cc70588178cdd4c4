// pndf_capi.cu -- C ABI (include/pndf.h) over the fused sm_100a kernel: handle management, host-side
// repacking of the reference state_dict into the kernel's slab stream, launches, host-buffer pipeline.
#include "../../include/pndf.h"
#include "pndf_kernel.cuh"
#include "pndf_denoise.cuh"
#include "pndf_encoder_train.cuh"
#include "pndf_train_ops.cuh"
#include "pndf_wgrad.cuh"
#include "pndf_feed.cuh"
#include "pndf_tc.h"
#include "pndf_host.h"
#include "pndf_knn.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace pndf;

namespace pndf {
using FusedFn = void (*)(const KParams);
FusedFn pndf_fused_entry_00(int mode, int small_tile);
FusedFn pndf_fused_entry_01(int mode, int small_tile);
FusedFn pndf_fused_entry_10(int mode, int small_tile);
FusedFn pndf_fused_entry_11(int mode, int small_tile);
}  // namespace pndf

namespace {
thread_local std::string g_err;
}  // namespace

int pndf::fail(const std::string& msg) {
    g_err = msg;
    return 1;
}

namespace {

#define CUDA_OK(expr)                                                                                     \
    do {                                                                                                  \
        cudaError_t _e = (expr);                                                                          \
        if (_e != cudaSuccess) return fail(std::string(#expr) + ": " + cudaGetErrorString(_e));          \
    } while (0)

const int kAmassDims[6] = {256, 512, 1024, 512, 256, 64};
const double kSmallTileCost = 0.40;      // time of an 8-pose tile relative to a 32-pose tile (measured, DESIGN.md)
const long long kTcChunk = 131072;       // poses per pass of the tensor-core path (5.7 GB of activations)

}  // namespace

struct pndf_handle {
    pndf_config cfg;
    int num_sms = 0;
    bool have_weights = false;
    DevBuf<float> d_wstream;      // slab stream
    DevBuf<float> d_small;        // biases (2625) + w6 (64) + encoder (3516), each 16B-aligned
    // device-side packing: slab stream / small buffer element -> index into the flat parameter vector (-1 = zero pad)
    DevBuf<int32_t> d_map_w, d_map_s;
    DevBuf<float> d_flat;         // staging copy of the flat parameter vector (host uploads)
    cudaEvent_t w_event = nullptr; // recorded after the last repack; launches on other streams wait for it
    cudaStream_t w_stream = nullptr;
    bool w_pending = false;
    size_t off_bias[7];
    size_t off_w6 = 0, off_enc = 0;
    // per-CTA scratch (softplus derivatives: num_sms * kUnits * 32 floats; encoder feature stash: num_sms * 128 * 32
    // floats), indexed by blockIdx only -- so every stream that may have a launch in flight needs its own copy:
    // slot 0 = the caller's stream (a handle is driven from ONE caller stream, include/pndf.h), slots 1, 2 = the two
    // pipeline streams of pndf_project_host (allocated on first use)
    DevBuf<float> d_scratch[3];
    DevBuf<float> d_z0[3];
    cudaEvent_t use_event = nullptr;   // recorded after every launch: a repack on another stream waits for it (WAR on the weights)
    cudaStream_t use_stream = nullptr;
    bool used = false;
    int f0_slabs = 0, z0_rows = 0;
    int64_t launches = 0;
    // host pipeline (pndf_project_host)
    cudaStream_t hs[2] = {nullptr, nullptr};
    cudaEvent_t hs_ev = nullptr;
    DevBuf<float> d_chunk[2];         // [chunk poses][84]
    DevBuf<float> d_chunk_dist[2];
    // training (pndf_train_losses / pndf_wgrad_accumulate / pndf_adam_step)
    DevBuf<int32_t> d_pos[3];         // flat parameter index -> slab-stream position (forward / reverse copy), small-buffer position
    DevBuf<float> d_ws;               // split-K workspace [slots][n_params]
    DevBuf<float> d_encrows;          // encoder-gradient rows [2][warps][kEncFloats] + first-level partial sums [2][kEncChunks][kEncFloats]
    DevBuf<float> d_loss_partial;     // [blocks][2]
    DevBuf<unsigned int> d_loss_counter;
    DevBuf<double> d_loss_totals;     // [3]
    // denoise loop state (pndf_denoise_prior): raw gradient, Adam moments ([poses][63] each), dist + second distance buffer
    DevBuf<float> d_dn[5];
    cudaStream_t cap_stream = nullptr;   // graph capture of the denoise loop
    cudaStream_t dn_stream2 = nullptr;   // second sequence group of the denoise loop (parallel branch)
    cudaEvent_t dn_ev[2] = {nullptr, nullptr};
    cudaGraphExec_t dn_exec = nullptr;
    bool in_capture = false;
    int tile_policy = 0;                 // 0: per launch from its batch size, 8 / 32 / 128: pinned (pndf_set_tile_policy); 128 = tensor-core path
    TcState* tc = nullptr;               // tensor-core DFNet path (pndf_tc.cu); nullptr if it could not be set up
};

namespace {

int validate(const pndf_config* c) {
    if (!c) return fail("null config");
    if (c->num_hidden != 6) return fail("fused kernel implements DFNet dims [256,512,1024,512,256,64] (configs/amass.yaml) only");
    for (int i = 0; i < 6; ++i)
        if (c->dims[i] != kAmassDims[i]) return fail("fused kernel implements DFNet dims [256,512,1024,512,256,64] (configs/amass.yaml) only");
    if (c->use_enc && c->in_dim != 126) return fail("with the structure encoder DFNet.in_dim must be 126");
    if (!c->use_enc && c->in_dim != 84) return fail("without the structure encoder DFNet.in_dim must be 84");
    for (int a : {c->enc_act, c->df_act})
        if (a < 0 || a > 2) return fail("activation must be PNDF_ACT_RELU / LRELU / SOFTPLUS");
    return 0;
}

size_t param_count(const pndf_config* c) { return (size_t)ParamLayout(*c).total; }

// Append one op's weights in the per-warp slab order the kernel consumes (pndf_kernel.cuh): for each slab index,
// for each of the 8 warps, R rows x FW feature columns (R*FW = 1024).  TN = features per thread, KG = K-groups.
//   TN == 8: warp columns = [32 features starting at cg*32 | 32 features starting at N/2 + cg*32], cg = warp (KG 1) or
//            warp & 3 (KG 2, N = 256; warps 4-7 hold the second half of the K rows)
//   TN == 2: 16 features starting at warp*16;   TN == 1: 8 features starting at warp*8.
// get(k, n) returns w[k][n] (0 outside the real matrix).
template <class F>
void pack_op(std::vector<float>& out, int K, int TN, int KG, F get) {
    const int FW = 8 * TN, R = kSlabFloats / FW, N = 64 * TN / KG;
    const int rows_per_group = K / KG, nslabs = rows_per_group / R;
    for (int s = 0; s < nslabs; ++s)
        for (int w = 0; w < kWarps; ++w) {
            const int kg = (KG == 1) ? 0 : (w >> 2), cg = (KG == 1) ? w : (w & 3);
            for (int r = 0; r < R; ++r) {
                const int k = kg * rows_per_group + s * R + r;
                for (int c = 0; c < FW; ++c) {
                    int n;
                    if (TN == 8) n = (c < 32) ? (cg * 32 + c) : (N / 2 + cg * 32 + (c - 32));
                    else n = cg * FW + c;
                    out.push_back(get(k, n));
                }
            }
        }
}

// Lay the flat parameter vector (reference state_dict order) out as (slab stream, small-parameter buffer) and record the
// offsets in the handle.  Run once at create time on the vector 1,2,3,... so that the result is an index map; the
// actual packing of weights is then a device-side gather (pack_gather_kernel), which keeps a training step free of
// host round trips.
int build_streams(pndf_handle* h, const float* flat, std::vector<float>& s, std::vector<float>& sm) {
    const ParamLayout L(h->cfg);
    const int* widths = L.width;
    const float* W[7];
    const float* Bv[7];
    for (int l = 0; l < 7; ++l) {
        W[l] = flat + L.w_off[l];
        Bv[l] = flat + L.b_off[l];
    }
    // ---- slab stream, in consumption order (pndf_kernel.cuh)
    s.clear();
    s.reserve((size_t)340 * kWarps * kSlabFloats);
    auto fwd = [&](int l, int k_off, int n_off) {   // w(k,n) = W_l[n_off+n][k_off+k]
        const float* w = W[l]; const int in = widths[l], out = widths[l + 1];
        return [=](int k, int n) { return (k_off + k < in && n_off + n < out) ? w[(size_t)(n_off + n) * in + (k_off + k)] : 0.0f; };
    };
    auto bwd = [&](int l, int k_off, int n_off) {   // w(k,n) = W_l[k_off+k][n_off+n]
        const float* w = W[l]; const int in = widths[l], out = widths[l + 1];
        return [=](int k, int n) { return (k_off + k < out && n_off + n < in) ? w[(size_t)(k_off + k) * in + (n_off + n)] : 0.0f; };
    };
    pack_op(s, h->z0_rows, 8, 2, fwd(0, 0, 0));   // F0  (N = 256, split-K)
    pack_op(s, 256, 8, 1, fwd(1, 0, 0));          // F1
    pack_op(s, 512, 8, 1, fwd(2, 0, 0));          // F2a : out features [0,512)
    pack_op(s, 512, 8, 1, fwd(3, 0, 0));          // F3a : in  features [0,512)
    pack_op(s, 512, 8, 1, fwd(2, 0, 512));        // F2b : out features [512,1024)
    pack_op(s, 512, 8, 1, fwd(3, 512, 0));        // F3b : in  features [512,1024)
    pack_op(s, 512, 8, 2, fwd(4, 0, 0));          // F4  (N = 256, split-K)
    pack_op(s, 256, 1, 1, fwd(5, 0, 0));          // F5  (N = 64)
    pack_op(s, 64, 8, 2, bwd(5, 0, 0));           // B5  (N = 256, split-K)
    pack_op(s, 256, 8, 1, bwd(4, 0, 0));          // B4
    pack_op(s, 512, 8, 1, bwd(3, 0, 0));          // B3a : in  features [0,512) of layer 3
    pack_op(s, 512, 8, 1, bwd(2, 0, 0));          // B2a : out features [0,512) of layer 2
    pack_op(s, 512, 8, 1, bwd(3, 0, 512));        // B3b
    pack_op(s, 512, 8, 1, bwd(2, 512, 0));        // B2b
    pack_op(s, 512, 8, 2, bwd(1, 0, 0));          // B1  (N = 256, split-K)
    pack_op(s, 256, 2, 1, bwd(0, 0, 0));          // B0  (N = 128: in_dim padded)
    const size_t expect = (size_t)(h->f0_slabs + 2 * slabs_of(256, 1, 64) + 8 * slabs_of(512, 1, 64) + 2 * slabs_of(512, 2, 64) +
                                   slabs_of(256, 1, 8) + slabs_of(64, 2, 64) + slabs_of(256, 1, 16)) * kWarps * kSlabFloats;
    if (s.size() != expect) return fail("internal: slab stream size mismatch");
    // ---- small parameters
    sm.clear();
    auto align4 = [&]() { while (sm.size() % 4) sm.push_back(0.0f); };
    for (int l = 0; l < 7; ++l) {
        align4();
        h->off_bias[l] = sm.size();
        sm.insert(sm.end(), Bv[l], Bv[l] + widths[l + 1]);
    }
    align4(); h->off_w6 = sm.size(); sm.insert(sm.end(), W[6], W[6] + 64);
    align4(); h->off_enc = sm.size();
    sm.insert(sm.end(), flat, flat + L.enc_floats);
    align4();
    return 0;
}

__global__ void pack_gather_kernel(const float* __restrict__ flat, const int32_t* __restrict__ map, float* __restrict__ out, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int32_t m = map[i];
        out[i] = (m >= 0) ? flat[m] : 0.0f;
    }
}

// Rewrite the weights on `st`: `write()` enqueues the kernels that change the packed buffers, then the tensor-core copies are split
// from the flat vector d_flat.  Launches still reading the old weights on another stream finish first; launches on another stream
// wait for w_event (order_after_weights).
template <class Write>
int write_weights(pndf_handle* h, const float* d_flat, cudaStream_t st, Write write) {
    if (h->used && h->use_stream != st) CUDA_OK(cudaStreamWaitEvent(st, h->use_event, 0));
    write();
    CUDA_OK(cudaGetLastError());
    if (h->tc && tc_set_weights(h->tc, d_flat, st)) return fail(std::string("tensor-core path: ") + tc_last_error(h->tc));
    if (!h->w_event) CUDA_OK(cudaEventCreateWithFlags(&h->w_event, cudaEventDisableTiming));
    CUDA_OK(cudaEventRecord(h->w_event, st));
    h->w_stream = st;
    h->w_pending = true;
    h->have_weights = true;
    return 0;
}

int pack_on_device(pndf_handle* h, const float* d_flat, cudaStream_t st) {
    return write_weights(h, d_flat, st, [&] {
        pack_gather_kernel<<<h->num_sms * 4, 256, 0, st>>>(d_flat, h->d_map_w.get(), h->d_wstream.get(), h->d_wstream.size());
        pack_gather_kernel<<<8, 256, 0, st>>>(d_flat, h->d_map_s.get(), h->d_small.get(), h->d_small.size());
    });
}

// a launch on a stream other than the one the weights were last repacked on has to wait for that repack
int order_after_weights(pndf_handle* h, cudaStream_t st) {
    if (h->w_pending && st != h->w_stream) CUDA_OK(cudaStreamWaitEvent(st, h->w_event, 0));
    return 0;
}

// Record that a launch on `st` reads the weights: a repack on another stream waits for it.  Not inside a stream capture (events
// must not be recorded into one): the caller records after the graph launch.
int mark_used(pndf_handle* h, cudaStream_t st) {
    if (h->in_capture) return 0;
    CUDA_OK(cudaEventRecord(h->use_event, st));
    h->use_stream = st;
    h->used = true;
    return 0;
}

int build_maps(pndf_handle* h) {
    const size_t n = param_count(&h->cfg);
    std::vector<float> iota(n), s, sm;
    for (size_t i = 0; i < n; ++i) iota[i] = (float)(i + 1);      // exact in fp32 (n < 2^24); 0 marks padding
    if (build_streams(h, iota.data(), s, sm)) return 1;
    std::vector<int32_t> mw(s.size()), ms(sm.size());
    for (size_t i = 0; i < s.size(); ++i) mw[i] = (int32_t)s[i] - 1;
    for (size_t i = 0; i < sm.size(); ++i) ms[i] = (int32_t)sm[i] - 1;
    if (h->d_wstream.reserve(s.size(), "slab stream") || h->d_small.reserve(sm.size(), "small-parameter buffer") ||
        h->d_map_w.reserve(mw.size(), "slab-stream map") || h->d_map_s.reserve(ms.size(), "small-parameter map") ||
        h->d_flat.reserve(n, "flat parameter staging buffer"))
        return 1;
    CUDA_OK(cudaMemcpy(h->d_map_w.get(), mw.data(), mw.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    CUDA_OK(cudaMemcpy(h->d_map_s.get(), ms.data(), ms.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    // inverse maps for the optimizer kernel: where does flat parameter i live in the packed buffers?
    std::vector<int32_t> pos[3];
    for (auto& v : pos) v.assign(n, -1);
    for (size_t i = 0; i < mw.size(); ++i) {
        if (mw[i] < 0) continue;
        if (pos[0][mw[i]] < 0) pos[0][mw[i]] = (int32_t)i;
        else if (pos[1][mw[i]] < 0) pos[1][mw[i]] = (int32_t)i;
        else return fail("internal: a weight appears more than twice in the slab stream");
    }
    for (size_t i = 0; i < ms.size(); ++i)
        if (ms[i] >= 0) pos[2][ms[i]] = (int32_t)i;
    for (size_t i = 0; i < n; ++i)
        if (pos[0][i] < 0 && pos[2][i] < 0) return fail("internal: a parameter is missing from the packed buffers");
    for (int k = 0; k < 3; ++k) {
        if (h->d_pos[k].reserve(n, "optimizer position map")) return 1;
        CUDA_OK(cudaMemcpy(h->d_pos[k].get(), pos[k].data(), n * sizeof(int32_t), cudaMemcpyHostToDevice));
    }
    return 0;
}

// Barrier between the GPUs of one node over peer memory: every rank owns a flag array [world + 1] inside its IPC buffer;
// lane r stores `epoch` into rank r's array at index `rank` (release, system scope: everything this stream wrote to peer
// memory before -- the fused gather stores of the preceding kernel -- is visible first) and then waits until rank r's
// epoch has arrived in the local array.  Bounded spin: after ~10 s the error slot [world] is set instead of hanging.
struct PeerFlags {
    uint32_t* flags[kMaxPeers + 1];
};
__global__ void peer_barrier_kernel(PeerFlags f, int world, int rank, uint32_t epoch) {
    const int r = threadIdx.x;
    if (r >= world) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f.flags[r] + rank), "r"(epoch) : "memory");
    const uint32_t* mine = f.flags[rank] + r;
    for (long long spin = 0;; ++spin) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
        if ((int32_t)(v - epoch) >= 0) break;
        if (spin > (1LL << 26)) {
            f.flags[rank][world] = 1u;
            break;
        }
        __nanosleep(128);
    }
}

// the 12 instances of the fused kernel (MODE x softplus DFNet x softplus encoder) live in four translation units
// (pndf_fused_inst.cu, compiled in parallel)
FusedFn fused_fn(int mode, bool dsoft, bool esoft, bool small_tile = false) {
    if (dsoft) return esoft ? pndf_fused_entry_11(mode, small_tile) : pndf_fused_entry_10(mode, small_tile);
    return esoft ? pndf_fused_entry_01(mode, small_tile) : pndf_fused_entry_00(mode, small_tile);
}

// Tile size of a launch: 8 or 32 poses per tile on the fused FFMA kernel, 128 = the tensor-core engine.  The engines and tilings
// differ in fp32 summation order, so every bit-for-bit guarantee (sharded == unsharded, pndf_project_host == pndf_project, graph
// replay == plain launches) rests on this one choice.
//
// The batch-size rule (pndf_tile_for_batch).  A 32-pose tile per SM is the latency floor of the fused kernel (~0.46 ms forward +
// reverse), so a batch that cannot give every SM a tile runs the small-tile variant: 8 poses per tile, four times as many CTAs,
// each ~0.3-0.4 of the time (the four lane groups split K).  It streams the weights once per 8 poses, so it only pays while the
// 32-pose tiling needs a single round.  From one pose more than a single round of 8-pose tiles covers (8 x SMs = 1 184) the DFNet
// GEMMs run on the tensor cores (pndf_tc.cu), ~3x the FFMA kernel (DESIGN.md 3b).  Measured, forward + d(dist)/d(pose) + step,
// lrelu (tools/small_batch_bench.py): 1 024 poses 195 us (8-pose tiles) vs 252 us; 1 536: 389 vs 270 us; 4 736: 459 (32-pose
// tiles) vs 301 us; 8 192: 917 vs 412 us.
bool small_tile_for(const pndf_handle* h, long long B) {
    const long long t32 = (B + kTileM - 1) / kTileM, t8 = (B + 7) / 8;
    const long long r32 = (t32 + h->num_sms - 1) / h->num_sms, r8 = (t8 + h->num_sms - 1) / h->num_sms;
    return r32 == 1 && (double)r8 * kSmallTileCost < 0.9;
}
int batch_tile(const pndf_handle* h, long long B) {
    if (h->tc && B > 8LL * h->num_sms) return 128;
    return small_tile_for(h, B) ? 8 : 32;
}
// the tile a call over B poses asks for: `PNDF_TILE=8|32|128` in the environment (tests, tuning), else the pinned policy
// (pndf_set_tile_policy), else the batch-size rule.  launch() narrows it to what the launch can take.
int tile_for(const pndf_handle* h, long long B) {
    if (const char* e = getenv("PNDF_TILE")) {
        const int t = atoi(e);
        return t == 8 ? 8 : (t == 128 && h->tc) ? 128 : 32;
    }
    if (h->tile_policy != 0) return h->tile_policy;
    return batch_tile(h, B);
}
// Can the tensor-core engine take this launch?  Forward, forward + gradient and projection steps on quaternions, and the prior mode
// (axis-angle input: one evaluation + VJP, optionally with a denoise loop's pending Adam update in the prologue) as ONE pass: the
// sequence bookkeeping does not survive the chunking of very large batches.  Training exports, tangent launches and the debug dump
// stay on the fused kernel.
bool tc_capable(const pndf_handle* h, const KParams& p, int mode) {
    if (!h->tc || mode == 2 || p.dbg != nullptr || p.act_masks != nullptr || p.tan_in != nullptr) return false;
    if (p.input_kind == IN_QUAT && p.dn.pending == 0) return !(mode == 1 && p.steps > 1 && p.pose_out == nullptr);
    return mode == 1 && p.steps == 1 && !p.do_step && p.pose_out == nullptr && p.n_peers == 0 && p.B <= kTcChunk;
}

int ensure_slot(pndf_handle* h, int slot) {
    if (h->d_z0[slot].reserve((size_t)h->num_sms * 128 * 32, "per-CTA encoder scratch")) return 1;
    if (h->cfg.df_act == PNDF_ACT_SOFTPLUS && h->d_scratch[slot].reserve((size_t)h->num_sms * kUnits * 32, "per-CTA softplus scratch"))
        return 1;
    return 0;
}

// per-warp rows [2][nwarps][E] followed by the first-level partial sums [2][kEncChunks][E]
int ensure_encrows(pndf_handle* h, long long nwarps) {
    return h->d_encrows.reserve(((size_t)2 * nwarps + 2 * kEncChunks) * kEncFloats, "encoder-gradient rows");
}

// One DFNet call at the tile its caller resolved (tile_for), narrowed to what the launch can take: 128 on a launch the tensor-core
// engine cannot take runs the fused kernel with 32-pose tiles, and so does 8 on a tangent, export or debug launch.
int launch(pndf_handle* h, KParams& p, int mode, int tile, cudaStream_t st, int slot = 0) {
    if (!h->have_weights) return fail("pndf_set_weights has not been called");
    if (p.B <= 0) return 0;
    if ((tile == 128 && !tc_capable(h, p, mode)) || (tile == 8 && (mode == 2 || p.dbg != nullptr || p.act_masks != nullptr)))
        tile = 32;
    p.wstream = h->d_wstream.get();
    for (int l = 0; l < 7; ++l) p.bias[l] = h->d_small.get() + h->off_bias[l];
    p.w6 = h->d_small.get() + h->off_w6;
    p.encw = h->cfg.use_enc ? h->d_small.get() + h->off_enc : nullptr;
    p.dscratch = h->d_scratch[slot].get();
    p.z0scratch = h->d_z0[slot].get();
    if (!h->in_capture && order_after_weights(h, st)) return 1;
    if (tile == 128) {
        // the activations of the whole DFNet chain live in HBM between the layer kernels (43.5 KB per pose): bound them by walking
        // very large batches in chunks of kTcChunk poses (every pose is independent; all steps of a chunk run before the next chunk).
        // The prior mode is one pass (tc_capable): its sequence bookkeeping (p.dn) is never sliced.
        const long long row = (p.input_kind == IN_QUAT) ? 84 : 63;
        for (long long off = 0; off < p.B; off += kTcChunk) {
            KParams c = p;
            c.B = std::min<long long>(kTcChunk, p.B - off);
            c.pose_in = p.pose_in + off * row;
            if (p.pose_out) c.pose_out = p.pose_out + off * row;
            if (p.dist) c.dist = p.dist + off;
            if (p.grad) c.grad = p.grad + off * row;
            if (p.g_up) c.g_up = p.g_up + off;
            for (int r = 0; r < p.n_peers; ++r) {
                c.peer_pose[r] = p.peer_pose[r] + off * row;
                if (p.peer_dist[r]) c.peer_dist[r] = p.peer_dist[r] + off;
            }
            if (tc_run(h->tc, c, mode == 1, st, &h->launches)) return fail(std::string("tensor-core path: ") + tc_last_error(h->tc));
        }
        return mark_used(h, st);
    }
    p.ntiles = (int)(tile == 8 ? (p.B + 7) / 8 : (p.B + kTileM - 1) / kTileM);
    p.use_enc = h->cfg.use_enc; p.enc_act = h->cfg.enc_act; p.df_act = h->cfg.df_act;
    p.enc_beta = h->cfg.enc_beta; p.df_beta = h->cfg.df_beta;
    p.f0_slabs = h->f0_slabs; p.z0_rows = h->z0_rows; p.in_dim = h->cfg.in_dim;
    const int grid = std::min(p.ntiles, h->num_sms);
    fused_fn(mode, h->cfg.df_act == PNDF_ACT_SOFTPLUS, h->cfg.enc_act == PNDF_ACT_SOFTPLUS, tile == 8)<<<grid, kThreads, kSmTotal, st>>>(p);
    CUDA_OK(cudaGetLastError());
    h->launches++;
    return mark_used(h, st);
}

}  // namespace

extern "C" {

const char* pndf_last_error(void) { return g_err.c_str(); }
const char* pndf_version(void) { return "posendf_b200 0.1 (sm_100a fused FFMA kernel)"; }

int pndf_param_count(const pndf_config* cfg, size_t* n) {
    if (validate(cfg)) return 1;
    *n = param_count(cfg);
    return 0;
}

int pndf_create(const pndf_config* cfg, pndf_handle** out) {
    if (!out) return fail("null out pointer");
    if (validate(cfg)) return 1;
    int ndev = 0;
    CUDA_OK(cudaGetDeviceCount(&ndev));
    if (cfg->device < 0 || cfg->device >= ndev) return fail("no such CUDA device");
    CUDA_OK(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CUDA_OK(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10) return fail(std::string("libpndf is built for sm_100a (B200); device is ") + prop.name);
    pndf_handle* h = new pndf_handle();
    h->cfg = *cfg;
    h->num_sms = prop.multiProcessorCount;
    h->z0_rows = cfg->use_enc ? 128 : 96;
    h->f0_slabs = slabs_of(h->z0_rows, 2, 64);
    for (int mode = 0; mode < 3; ++mode)
        for (int small = 0; small < (mode == 2 ? 1 : 2); ++small)
            CUDA_OK(cudaFuncSetAttribute(fused_fn(mode, cfg->df_act == PNDF_ACT_SOFTPLUS, cfg->enc_act == PNDF_ACT_SOFTPLUS, small != 0),
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, kSmTotal));
    if (ensure_slot(h, 0)) { pndf_destroy(h); return 1; }
    if (cudaEventCreateWithFlags(&h->use_event, cudaEventDisableTiming) != cudaSuccess) { pndf_destroy(h); return fail("cudaEventCreate failed"); }
    if (build_maps(h)) { pndf_destroy(h); return 1; }
    if (tc_create(&h->tc, cfg)) { h->tc = nullptr; cudaGetLastError(); }      // without it everything runs on the FFMA kernels
    *out = h;
    return 0;
}

int pndf_destroy(pndf_handle* h) {
    if (!h) return 0;
    cudaSetDevice(h->cfg.device);
    if (h->w_event) cudaEventDestroy(h->w_event);
    if (h->use_event) cudaEventDestroy(h->use_event);
    tc_destroy(h->tc);
    if (h->dn_exec) cudaGraphExecDestroy(h->dn_exec);
    if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
    if (h->dn_stream2) cudaStreamDestroy(h->dn_stream2);
    for (int i = 0; i < 2; ++i)
        if (h->dn_ev[i]) cudaEventDestroy(h->dn_ev[i]);
    for (int i = 0; i < 2; ++i)
        if (h->hs[i]) cudaStreamDestroy(h->hs[i]);
    if (h->hs_ev) cudaEventDestroy(h->hs_ev);
    delete h;      // frees the device buffers
    return 0;
}

int pndf_set_weights(pndf_handle* h, const float* flat, size_t n) {
    if (!h || !flat) return fail("null argument");
    if (n != param_count(&h->cfg)) return fail("pndf_set_weights: wrong parameter count");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    CUDA_OK(cudaMemcpy(h->d_flat.get(), flat, n * sizeof(float), cudaMemcpyHostToDevice));
    if (pack_on_device(h, h->d_flat.get(), nullptr)) return 1;
    CUDA_OK(cudaStreamSynchronize(nullptr));
    return 0;
}

int pndf_set_weights_device(pndf_handle* h, const float* flat_dev, size_t n, void* stream) {
    if (!h || !flat_dev) return fail("null argument");
    if (n != param_count(&h->cfg)) return fail("pndf_set_weights_device: wrong parameter count");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    return pack_on_device(h, flat_dev, (cudaStream_t)stream);
}

int pndf_forward(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, float* dist_dev, void* stream) {
    if (!h) return fail("null handle");
    if (B == 0) return 0;
    if (B < 0 || !pose_dev || !dist_dev) return fail("null argument");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    KParams p{};
    p.pose_in = pose_dev; p.dist = dist_dev; p.B = B; p.steps = 1; p.normalise = normalise; p.input_kind = IN_QUAT;
    return launch(h, p, 0, tile_for(h, p.B), (cudaStream_t)stream);
}

int pndf_forward_grad(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, const float* g_up_dev,
                      float* dist_dev, float* grad_dev, void* stream) {
    if (!h) return fail("null handle");
    if (B == 0) return 0;
    if (B < 0 || !pose_dev || !grad_dev) return fail("null argument");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    KParams p{};
    p.pose_in = pose_dev; p.dist = dist_dev; p.grad = grad_dev; p.g_up = g_up_dev; p.B = B; p.steps = 1;
    p.normalise = normalise; p.input_kind = IN_QUAT;
    return launch(h, p, 1, tile_for(h, p.B), (cudaStream_t)stream);
}

int pndf_project(pndf_handle* h, float* pose_dev, int64_t B, int steps, int renorm, float* dist_dev, void* stream) {
    if (!h) return fail("null handle");
    if (steps < 1) return fail("steps must be >= 1");
    if (B == 0) return 0;
    if (B < 0 || !pose_dev) return fail("null argument");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    KParams p{};
    p.pose_in = pose_dev; p.pose_out = pose_dev; p.dist = dist_dev; p.B = B; p.steps = steps; p.do_step = 1;
    p.renorm = renorm; p.normalise = 1; p.input_kind = IN_QUAT;
    return launch(h, p, 1, tile_for(h, p.B), (cudaStream_t)stream);
}

int pndf_project_gather(pndf_handle* h, float* pose_dev, int64_t B, int steps, int renorm, float* dist_dev,
                        float* const* peer_pose_dev, float* const* peer_dist_dev, int n_peers, void* stream) {
    if (!h) return fail("null handle");
    if (steps < 1) return fail("steps must be >= 1");
    if (n_peers < 0 || n_peers > kMaxPeers) return fail("pndf_project_gather: at most 7 peers (8 GPUs of one node)");
    if (n_peers > 0 && !peer_pose_dev) return fail("null argument");
    if (B == 0) return 0;
    if (B < 0 || !pose_dev) return fail("null argument");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    KParams p{};
    p.pose_in = pose_dev; p.pose_out = pose_dev; p.dist = dist_dev; p.B = B; p.steps = steps; p.do_step = 1;
    p.renorm = renorm; p.normalise = 1; p.input_kind = IN_QUAT;
    p.n_peers = n_peers;
    for (int r = 0; r < n_peers; ++r) {
        if (!peer_pose_dev[r] || (reinterpret_cast<uintptr_t>(peer_pose_dev[r]) & 15)) return fail("pndf_project_gather: peer pointers must be 16-byte aligned");
        p.peer_pose[r] = peer_pose_dev[r];
        p.peer_dist[r] = peer_dist_dev ? peer_dist_dev[r] : nullptr;
    }
    return launch(h, p, 1, tile_for(h, p.B), (cudaStream_t)stream);
}

// ---- peer memory (one process per GPU): cudaMalloc + cudaIpc handles; the handle bytes travel through the caller's
// own channel (torch.distributed all_gather in posendf_b200/dist.py)
int pndf_peer_alloc(int device, size_t bytes, void** dev_ptr, unsigned char* handle64) {
    if (!dev_ptr || !handle64 || bytes == 0) return fail("pndf_peer_alloc: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    CUDA_OK(cudaSetDevice(device));
    void* ptr = nullptr;
    CUDA_OK(cudaMalloc(&ptr, bytes));
    CUDA_OK(cudaMemset(ptr, 0, bytes));
    cudaIpcMemHandle_t hd;
    cudaError_t e = cudaIpcGetMemHandle(&hd, ptr);
    if (e != cudaSuccess) {
        cudaFree(ptr);
        return fail(std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
    }
    memcpy(handle64, &hd, 64);
    *dev_ptr = ptr;
    return 0;
}
int pndf_peer_open(int device, const unsigned char* handle64, void** dev_ptr) {
    if (!dev_ptr || !handle64) return fail("pndf_peer_open: bad argument");
    CUDA_OK(cudaSetDevice(device));
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handle64, 64);
    CUDA_OK(cudaIpcOpenMemHandle(dev_ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
int pndf_peer_close(int device, void* dev_ptr) {
    if (!dev_ptr) return 0;
    CUDA_OK(cudaSetDevice(device));
    CUDA_OK(cudaIpcCloseMemHandle(dev_ptr));
    return 0;
}
int pndf_peer_free(int device, void* dev_ptr) {
    if (!dev_ptr) return 0;
    CUDA_OK(cudaSetDevice(device));
    CUDA_OK(cudaFree(dev_ptr));
    return 0;
}
int pndf_peer_barrier(int device, uint32_t* const* flags_dev, int world, int rank, uint32_t epoch, void* stream) {
    if (!flags_dev || world < 1 || world > kMaxPeers + 1 || rank < 0 || rank >= world) return fail("pndf_peer_barrier: bad argument");
    CUDA_OK(cudaSetDevice(device));
    PeerFlags f{};
    for (int r = 0; r < world; ++r) {
        if (!flags_dev[r]) return fail("pndf_peer_barrier: null flag array");
        f.flags[r] = flags_dev[r];
    }
    peer_barrier_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(f, world, rank, epoch);
    CUDA_OK(cudaGetLastError());
    return 0;
}

int pndf_prior_grad(pndf_handle* h, const float* aa_dev, int64_t B, const float* g_up_dev, float* dist_dev,
                    float* grad_aa_dev, void* stream) {
    if (!h) return fail("null handle");
    if (B == 0) return 0;
    if (B < 0 || !aa_dev || !grad_aa_dev) return fail("null argument");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    KParams p{};
    p.pose_in = aa_dev; p.dist = dist_dev; p.grad = grad_aa_dev; p.g_up = g_up_dev; p.B = B; p.steps = 1;
    p.normalise = 1; p.input_kind = IN_AXIS_ANGLE;
    return launch(h, p, 1, tile_for(h, p.B), (cudaStream_t)stream);
}

int pndf_project_host(pndf_handle* h, const float* pose_in_host, float* pose_out_host, float* dist_host, int64_t B,
                      int steps, int renorm) {
    if (!h) return fail("null handle");
    if (steps < 1) return fail("steps must be >= 1");
    if (B == 0) return 0;
    if (B < 0 || !pose_in_host || !pose_out_host) return fail("null argument");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    for (int i = 0; i < 2; ++i)
        if (!h->hs[i]) CUDA_OK(cudaStreamCreateWithFlags(&h->hs[i], cudaStreamNonBlocking));
    if (!h->hs_ev) CUDA_OK(cudaEventCreateWithFlags(&h->hs_ev, cudaEventDisableTiming));
    if (ensure_slot(h, 1) || ensure_slot(h, 2)) return 1;   // the two streams overlap: each needs its own per-CTA scratch
    // one tile size for all chunks, the one the whole batch gets: the result equals pndf_project on the same batch bit for bit
    const int tile = tile_for(h, B);
    // Chunk schedule.  Fused engine: uniform chunks of 4 tiles per SM (its time is linear in the tiles).  Tensor-core engine: its 15
    // launches per chunk want LARGE chunks (8 192 poses 0.41 ms, 49 152 poses 1.65 ms), but only the first chunk's upload and the
    // last chunk's download cannot hide under compute -- so a small head, large body chunks, a small tail.
    std::vector<int64_t> sizes;
    if (tile == 128) {
        const int64_t kEdge = 8192, kBody = 49152;
        if (B <= 2 * kEdge) {
            for (int64_t off = 0; off < B; off += kEdge) sizes.push_back(std::min(kEdge, B - off));
        } else {
            sizes.push_back(kEdge);
            const int64_t mid = B - 2 * kEdge, parts = (mid + kBody - 1) / kBody;
            const int64_t per = ((mid + parts - 1) / parts + 127) / 128 * 128;
            for (int64_t done = 0; done < mid; done += per) sizes.push_back(std::min(per, mid - done));
            sizes.push_back(kEdge);
        }
    } else {
        const int64_t chunk = (int64_t)h->num_sms * 4 * kTileM;
        for (int64_t off = 0; off < B; off += chunk) sizes.push_back(std::min(chunk, B - off));
    }
    const size_t need = (size_t)*std::max_element(sizes.begin(), sizes.end());
    bool grow = false;
    for (int i = 0; i < 2; ++i) grow |= h->d_chunk[i].size() < need * 84 || h->d_chunk_dist[i].size() < need;
    if (grow) {
        CUDA_OK(cudaStreamSynchronize(h->hs[0]));
        CUDA_OK(cudaStreamSynchronize(h->hs[1]));
        for (int i = 0; i < 2; ++i)
            if (h->d_chunk[i].reserve(need * 84, "host pipeline chunk") || h->d_chunk_dist[i].reserve(need, "host pipeline chunk distances"))
                return 1;
    }
    int which = 0;
    int64_t off = 0;
    for (size_t ci = 0; ci < sizes.size(); off += sizes[ci], ++ci, which ^= 1) {
        const int64_t nb = sizes[ci];
        cudaStream_t st = h->hs[which];
        float* chunk = h->d_chunk[which].get();
        float* chunk_dist = h->d_chunk_dist[which].get();
        CUDA_OK(cudaMemcpyAsync(chunk, pose_in_host + off * 84, nb * 84 * sizeof(float), cudaMemcpyHostToDevice, st));
        KParams p{};
        p.pose_in = chunk; p.pose_out = chunk; p.dist = chunk_dist; p.B = nb;
        p.steps = steps; p.do_step = 1; p.renorm = renorm; p.normalise = 1; p.input_kind = IN_QUAT;
        // the tensor-core path keeps its activations in ONE set of buffers per handle: its launches of consecutive chunks must not
        // overlap (the copies of the two streams still do)
        if (tile == 128 && off > 0) CUDA_OK(cudaStreamWaitEvent(st, h->hs_ev, 0));
        if (launch(h, p, 1, tile, st, 1 + which)) return 1;
        if (tile == 128) CUDA_OK(cudaEventRecord(h->hs_ev, st));
        CUDA_OK(cudaMemcpyAsync(pose_out_host + off * 84, chunk, nb * 84 * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (dist_host) CUDA_OK(cudaMemcpyAsync(dist_host + off, chunk_dist, nb * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    CUDA_OK(cudaStreamSynchronize(h->hs[0]));
    CUDA_OK(cudaStreamSynchronize(h->hs[1]));
    return 0;
}

int pndf_denoise_prior(pndf_handle* h, float* aa_dev, int64_t S, int64_t T, int iterations, int steps_per_iter, float lr,
                       float* dist_dev, float* loss_hist_dev, void* stream) {
    if (!h) return fail("null handle");
    if (S == 0 || T == 0) return 0;
    if (S < 0 || T < 0 || !aa_dev) return fail("null argument");
    if (iterations < 1 || steps_per_iter < 1) return fail("iterations and steps_per_iter must be >= 1");
    if (T > (1 << 24) / 63) return fail("sequence too long");
    if (!h->have_weights) return fail("pndf_set_weights has not been called");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t B = S * T;
    for (int i = 0; i < 5; ++i)
        if (h->d_dn[i].reserve((size_t)B * (i < 3 ? 63 : 1), "denoise loop state")) return 1;
    if (!h->dn_stream2) {
        if (cudaStreamCreateWithFlags(&h->dn_stream2, cudaStreamNonBlocking) != cudaSuccess) h->dn_stream2 = nullptr;
        for (int i = 0; i < 2 && h->dn_stream2; ++i)
            if (cudaEventCreateWithFlags(&h->dn_ev[i], cudaEventDisableTiming) != cudaSuccess) {
                cudaStreamDestroy(h->dn_stream2);
                h->dn_stream2 = nullptr;
            }
        cudaGetLastError();
    }
    if (h->dn_stream2 && ensure_slot(h, 1)) return 1;
    float* graw = h->d_dn[0].get();
    float* m = h->d_dn[1].get();
    float* v = h->d_dn[2].get();
    // distances are double-buffered (the update prologue of step t reads whole sequences of step t-1 while other CTAs already
    // write step t); the buffers alternate so that the LAST step lands in the caller's array
    float* dbuf[2] = {dist_dev ? dist_dev : h->d_dn[3].get(), h->d_dn[4].get()};
    const int nsteps = iterations * steps_per_iter;
    const double b1 = 0.9, b2 = 0.999;
    auto adam_of = [&](int t1, int it) {      // parameters of update number t1 (1-based), loss weight of outer iteration `it`
        AdamParams ap;
        ap.lr = lr; ap.beta1 = (float)b1; ap.beta2 = (float)b2; ap.eps = 1e-8f;
        ap.bias1 = (float)(1.0 - std::pow(b1, (double)t1)); ap.bias2 = (float)(1.0 - std::pow(b2, (double)t1));
        ap.weight = 1e7f / (1.0f + (float)it);
        return ap;
    };
    // ONE launch per optimisation step and sequence group (prior + gradient, with the previous step's Adam update fused into its
    // prologue) and one trailing update kernel per group; the whole loop is captured into a CUDA graph and replayed as a single
    // graph launch.  Sequences are independent of each other, so they are split into two groups whose launch chains run side by
    // side (second internal stream = a parallel branch of the graph, its own per-CTA scratch slot): when the persistent CTAs of
    // one group's launch run out of tiles, the other group's next launch takes over their SMs -- without it 1 200 tiles on 148
    // SMs (config C4) leave the ninth round 90 % empty in every one of the 100 steps.
    // On the tensor-core engine (one set of activation buffers per handle) the loop is ONE chain over all sequences; its buffers
    // are reserved before the capture starts.
    const bool on_tc = tile_for(h, B) == 128 && B <= kTcChunk;
    if (on_tc && tc_reserve(h->tc, B)) return fail(std::string("tensor-core path: ") + tc_last_error(h->tc));
    const int G = (!on_tc && S >= 2 && h->dn_stream2 != nullptr) ? 2 : 1;
    auto enqueue = [&](cudaStream_t s0) -> int {
        if (cudaMemsetAsync(m, 0, (size_t)B * 63 * sizeof(float), s0) != cudaSuccess) return fail("cudaMemsetAsync failed");
        if (cudaMemsetAsync(v, 0, (size_t)B * 63 * sizeof(float), s0) != cudaSuccess) return fail("cudaMemsetAsync failed");
        cudaStream_t sg[2] = {s0, h->dn_stream2};
        const int64_t seq0[3] = {0, G == 2 ? S / 2 : S, S};
        if (G == 2) {
            if (cudaEventRecord(h->dn_ev[0], s0) != cudaSuccess || cudaStreamWaitEvent(sg[1], h->dn_ev[0], 0) != cudaSuccess)
                return fail("denoise: fork failed");
        }
        for (int t = 0; t < nsteps; ++t) {
            for (int g = 0; g < G; ++g) {
                const int64_t o = seq0[g] * T, Bg = (seq0[g + 1] - seq0[g]) * T;      // first pose / poses of the group
                KParams p{};
                p.pose_in = aa_dev + o * 63; p.dist = dbuf[(nsteps - 1 - t) & 1] + o; p.grad = graw + o * 63; p.B = Bg; p.steps = 1;
                p.normalise = 1; p.input_kind = IN_AXIS_ANGLE;
                if (t > 0) {
                    p.dn.pending = 1; p.dn.m = m + o * 63; p.dn.v = v + o * 63; p.dn.graw = graw + o * 63;
                    p.dn.dist_prev = dbuf[(nsteps - t) & 1] + o; p.dn.pose_rw = aa_dev + o * 63; p.dn.T = (int)T;
                    p.dn.ap = adam_of(t, (t - 1) / steps_per_iter);
                    p.dn.loss_out = loss_hist_dev ? loss_hist_dev + (size_t)(t - 1) * S + seq0[g] : nullptr;
                }
                // off the tensor-core chain the groups run side by side: fused engine only
                const int tile = tile_for(h, Bg);
                if (launch(h, p, 1, (!on_tc && tile == 128) ? 32 : tile, sg[g], g)) return 1;
            }
        }
        for (int g = 0; g < G; ++g) {
            const int64_t o = seq0[g] * T;
            seq_adam_kernel<<<(unsigned)(seq0[g + 1] - seq0[g]), 256, 0, sg[g]>>>(
                aa_dev + o * 63, graw + o * 63, dbuf[0] + o, m + o * 63, v + o * 63,
                loss_hist_dev ? loss_hist_dev + (size_t)(nsteps - 1) * S + seq0[g] : nullptr, (int)T,
                adam_of(nsteps, (nsteps - 1) / steps_per_iter));
            if (cudaGetLastError() != cudaSuccess) return fail("seq_adam_kernel launch failed");
            h->launches++;
        }
        if (G == 2) {
            if (cudaEventRecord(h->dn_ev[1], sg[1]) != cudaSuccess || cudaStreamWaitEvent(s0, h->dn_ev[1], 0) != cudaSuccess)
                return fail("denoise: join failed");
        }
        return 0;
    };
    if (order_after_weights(h, st)) return 1;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    CUDA_OK(cudaStreamIsCapturing(st, &cs));
    bool graphed = false;
    // (the tensor-core chain is 15 kernels of ~0.1 ms per step: the host stays far ahead of the GPU with plain launches, while
    //  capturing + instantiating a 1 501-node graph costs tens of milliseconds per call)
    if (cs == cudaStreamCaptureStatusNone && !getenv("PNDF_NO_GRAPH") && !on_tc) {
        // capture on an internal stream (the caller's may be the legacy default stream, which cannot be captured), replay on the caller's
        if (!h->cap_stream && cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking) != cudaSuccess) h->cap_stream = nullptr;
        if (h->cap_stream && cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            h->in_capture = true;
            const int64_t launches0 = h->launches;
            const int rc = enqueue(h->cap_stream);
            h->in_capture = false;
            cudaGraph_t g = nullptr;
            const cudaError_t e = cudaStreamEndCapture(h->cap_stream, &g);
            if (rc == 0 && e == cudaSuccess && g) {
                if (h->dn_exec) { cudaGraphExecDestroy(h->dn_exec); h->dn_exec = nullptr; }
                if (cudaGraphInstantiate(&h->dn_exec, g, 0) == cudaSuccess && cudaGraphLaunch(h->dn_exec, st) == cudaSuccess) graphed = true;
            }
            if (g) cudaGraphDestroy(g);
            if (!graphed) { cudaGetLastError(); h->launches = launches0; }
        } else {
            cudaGetLastError();
        }
    }
    if (!graphed && enqueue(st)) return 1;
    return mark_used(h, st);
}

int pndf_debug_dump_floats(size_t* n) {
    *n = (size_t)kDumpRows * 32;
    return 0;
}

int pndf_forward_grad_debug(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, float* dist_dev,
                            float* grad_dev, float* dump_dev, void* stream) {
    if (!h || !pose_dev || !grad_dev || !dump_dev) return fail("null argument");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    KParams p{};
    p.pose_in = pose_dev; p.dist = dist_dev; p.grad = grad_dev; p.B = std::min<int64_t>(B, 32); p.steps = 1;
    p.normalise = normalise; p.input_kind = IN_QUAT; p.dbg = dump_dev;
    return launch(h, p, 1, tile_for(h, p.B), (cudaStream_t)stream);
}

int pndf_act_handoff_bytes(const pndf_handle* h, int64_t B, size_t* n) {
    if (!h || B < 0 || !n) return fail("bad argument");
    const size_t tiles = (size_t)((B + kTileM - 1) / kTileM);
    *n = tiles * (h->cfg.df_act == PNDF_ACT_SOFTPLUS ? (size_t)kUnits * 32 * sizeof(float) : (size_t)4 * kMaskStride);
    return 0;
}

int pndf_forward_grad_export(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, float* dist_dev, float* grad_dev,
                             float* dump_dev, void* act_handoff_dev, void* stream) {
    if (!h) return fail("null handle");
    if (B == 0) return 0;
    if (B < 0 || !pose_dev || !grad_dev || !dump_dev) return fail("null argument");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    KParams p{};
    p.pose_in = pose_dev; p.dist = dist_dev; p.grad = grad_dev; p.B = B; p.steps = 1;
    p.normalise = normalise; p.input_kind = IN_QUAT; p.dbg = dump_dev; p.dump_all = 1;
    p.act_masks = (uint8_t*)act_handoff_dev;
    return launch(h, p, 1, tile_for(h, p.B), (cudaStream_t)stream);
}

int pndf_forward_tangent_export(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, const float* tan_dev,
                                float* dump_dev, const void* act_handoff_dev, void* stream) {
    if (!h) return fail("null handle");
    if (B == 0) return 0;
    if (B < 0 || !pose_dev || !tan_dev || !dump_dev) return fail("null argument");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    KParams p{};
    p.pose_in = pose_dev; p.B = B; p.steps = 1; p.normalise = normalise; p.input_kind = IN_QUAT;
    p.dbg = dump_dev; p.dump_all = 1; p.tan_in = tan_dev;
    p.act_masks = (uint8_t*)act_handoff_dev;
    return launch(h, p, 2, tile_for(h, p.B), (cudaStream_t)stream);
}

int pndf_encoder_tangent(pndf_handle* h, const float* pose_dev, const float* v_dev, int64_t B, int normalise,
                         float* zdot_tiles_dev, void* stream) {
    if (!h) return fail("null handle");
    if (B == 0) return 0;
    if (B < 0 || !pose_dev || !v_dev || !zdot_tiles_dev) return fail("null argument");
    if (!h->have_weights) return fail("pndf_set_weights has not been called");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    EncTrainParams p{};
    p.x = pose_dev; p.v = v_dev; p.encw = h->d_small.get() + h->off_enc; p.zdot_tiles = zdot_tiles_dev; p.B = B;
    p.normalise = normalise; p.act = h->cfg.enc_act; p.beta = h->cfg.enc_beta; p.use_enc = h->cfg.use_enc;
    if (order_after_weights(h, (cudaStream_t)stream)) return 1;
    enc_tangent_kernel<<<(unsigned)((B + 127) / 128), 128, 0, (cudaStream_t)stream>>>(p);
    CUDA_OK(cudaGetLastError());
    h->launches++;
    return 0;
}

int pndf_encoder_param_grads(pndf_handle* h, const float* pose_dev, const float* v_dev, int64_t B, int normalise,
                             const float* up_first_dev, const float* up_tangent_dev, const float* up_second_dev,
                             float* grads_dev, void* stream) {
    if (!h) return fail("null handle");
    if (!h->cfg.use_enc) return fail("this configuration has no structure encoder");
    if (B < 0 || !pose_dev || !grads_dev) return fail("null argument");
    if (!h->have_weights) return fail("pndf_set_weights has not been called");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_OK(cudaMemsetAsync(grads_dev, 0, 2 * kEncFloats * sizeof(float), st));
    if (B == 0) return 0;
    const long long nwarps = ((B + 127) / 128) * 4;
    if (ensure_encrows(h, nwarps)) return 1;
    EncTrainParams p{};
    p.x = pose_dev; p.v = v_dev; p.encw = h->d_small.get() + h->off_enc; p.up1 = up_first_dev; p.upt = up_tangent_dev;
    p.upz = up_second_dev; p.grads = h->d_encrows.get(); p.B = B; p.normalise = normalise; p.act = h->cfg.enc_act;
    p.beta = h->cfg.enc_beta; p.use_enc = 1;
    if (order_after_weights(h, st)) return 1;
    enc_grad_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(p);
    CUDA_OK(cudaGetLastError());
    const int nsets = (up_tangent_dev || up_second_dev) ? 2 : 1;
    enc_rows_reduce_kernel<<<(nsets * kEncFloats + 255) / 256, 256, 0, st>>>(h->d_encrows.get(), nwarps, nsets, grads_dev);
    CUDA_OK(cudaGetLastError());
    h->launches += 2;
    return 0;
}

int pndf_softplus_adjoint(int device, const float* z_next_dev, const float* zdot_next_dev, const float* adj_dev, int64_t ld,
                          const float* zbar_dev, const float* w_eik_dev, float beta, int64_t B, int n, float* pbar_dev,
                          void* stream) {
    if (B == 0) return 0;
    if (B < 0 || n <= 0 || (n & 3) || (ld & 3) || !z_next_dev || !zdot_next_dev || !adj_dev || !zbar_dev || !pbar_dev)
        return fail("pndf_softplus_adjoint: bad argument");
    CUDA_OK(cudaSetDevice(device));
    SoftplusAdjParams p{};
    p.z_next = z_next_dev; p.zdot_next = zdot_next_dev; p.adj = adj_dev; p.zbar = zbar_dev; p.w = w_eik_dev; p.pbar = pbar_dev;
    p.ld = ld; p.B = B; p.n = n; p.beta = beta;
    const long long total = B * (long long)(n >> 2);
    const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, 148LL * 16);
    softplus_adjoint_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p);
    CUDA_OK(cudaGetLastError());
    return 0;
}

int pndf_train_losses(pndf_handle* h, const float* dist_dev, const float* dist_gt_dev, const float* grad_dev, int64_t B,
                      int64_t B_total, int mode, int l2, int reset, float* coef_dev, float* v_dev, float* losses_dev, void* stream) {
    if (!h) return fail("null handle");
    if (B <= 0 || B_total < B || !dist_dev || !losses_dev) return fail("pndf_train_losses: bad argument");
    if (mode != 0 && mode != 1) return fail("pndf_train_losses: mode must be 0 (pose batch) or 1 (manifold batch)");
    if (mode == 0 && (!dist_gt_dev || !coef_dev)) return fail("pndf_train_losses: pose mode needs dist_gt and coef");
    if (mode == 0 && grad_dev && !v_dev) return fail("pndf_train_losses: Eikonal term needs the tangent output");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    const int blocks = (int)((B + 255) / 256);
    // the counter and the totals are zeroed once, when they are allocated: from then on the kernel resets the counter itself, and
    // the totals on a call with `reset`
    if (h->d_loss_partial.reserve((size_t)blocks * 2, "loss partial sums") || h->d_loss_counter.reserve(1, "loss counter", true) ||
        h->d_loss_totals.reserve(3, "loss totals", true))
        return 1;
    LossParams p{};
    p.dist = dist_dev; p.dist_gt = dist_gt_dev; p.grad = grad_dev; p.coef = coef_dev; p.v = v_dev;
    p.partial = h->d_loss_partial.get(); p.counter = h->d_loss_counter.get(); p.totals = h->d_loss_totals.get(); p.losses = losses_dev;
    p.B = B; p.inv_n = 1.0 / (double)B_total; p.mode = mode; p.l2 = l2; p.reset = reset;
    if (reset && mode == 0) CUDA_OK(cudaMemsetAsync(losses_dev, 0, 3 * sizeof(float), (cudaStream_t)stream));
    train_loss_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(p);
    CUDA_OK(cudaGetLastError());
    h->launches++;
    return 0;
}

int pndf_wgrad_accumulate(pndf_handle* h, const float* pose_dev, const float* v_dev, int normalise, const float* dump_dev,
                          const float* dump_t_dev, const float* coef_dev, float uniform, const float* dist_dev, int64_t B,
                          const float* up_dev, const float* w_eik_dev, const float* upz_dev, float* grad_flat_dev, int overwrite,
                          void* stream) {
    if (!h) return fail("null handle");
    if (B == 0) return 0;
    if (B < 0 || !pose_dev || !dump_dev || !dist_dev || !up_dev || !grad_flat_dev) return fail("pndf_wgrad_accumulate: null argument");
    if (!h->have_weights) return fail("pndf_set_weights has not been called");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const ParamLayout L(h->cfg);
    const size_t n_params = (size_t)L.total;
    const size_t ws_stride = (n_params + 3) & ~(size_t)3;      // 16-byte aligned workspace slots (vector stores)
    // K-split length: 84 output tiles per split, 2 CTAs per SM -- pick the multiple of 32 poses in [768, 1536] that wastes the
    // least of the last wave (B = 32 768: 864 poses -> 38 splits, 3 192 CTAs = 10.8 waves of 296)
    const int kTiles = 84;
    int kc = 1024;
    {
        const long long slots = 2LL * h->num_sms;
        long long best = -1;
        for (int cand = 768; cand <= 1536; cand += kWgBK) {
            const long long splits = (B + cand - 1) / cand;
            const long long waves = (kTiles * splits + slots - 1) / slots;
            const long long cost = waves * cand;
            if (best < 0 || cost < best) { best = cost; kc = cand; }
        }
    }
    const int ksplits = (int)((B + kc - 1) / kc);
    const long long nwarps = ((B + 127) / 128) * 4;      // of the encoder-gradient kernel
    if (h->d_ws.reserve((size_t)ksplits * ws_stride, "split-K workspace")) return 1;
    if (h->cfg.use_enc && ensure_encrows(h, nwarps)) return 1;
    static bool attr_set[64] = {};
    if (h->cfg.device < 64 && !attr_set[h->cfg.device]) {
        CUDA_OK(cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem));
        attr_set[h->cfg.device] = true;
    }
    // export column map (DESIGN.md): layer inputs z_l, adjoints of pre_l
    const int z_col[7] = {0, 128, 384, 896, 1920, 2432, 2688};
    const int a_col[6] = {5120, 4608, 3584, 3072, 2816, 2752};
    WgParams p{};
    p.dump = dump_dev; p.dump_t = dump_t_dev; p.coef = coef_dev; p.up = up_dev; p.w_eik = w_eik_dev; p.uniform = uniform;
    p.ws = h->d_ws.get(); p.B = B; p.ws_stride = (long long)ws_stride; p.kc = kc; p.slot0 = 0; p.nprob = 6;
    int tiles = 0;
    // big layers first: their CTAs start first inside every K-split
    const int order[6] = {2, 3, 1, 4, 0, 5};
    for (int i = 0; i < 6; ++i) {
        const int l = order[i];
        WgProblem& q = p.prob[i];
        q.a_col = a_col[l]; q.z_col = z_col[l]; q.n_out = L.width[l + 1]; q.n_in = L.width[l];
        q.m_tiles = (q.n_out + kWgTile - 1) / kWgTile; q.n_tiles = (q.n_in + kWgTile - 1) / kWgTile;
        q.tile0 = tiles; q.w_off = L.w_off[l]; q.b_off = L.b_off[l];
        tiles += q.m_tiles * q.n_tiles;
    }
    if (order_after_weights(h, st)) return 1;
    wgrad_kernel<<<dim3((unsigned)tiles, (unsigned)ksplits), kWgThreads, kWgSmem, st>>>(p);
    CUDA_OK(cudaGetLastError());
    WgLastParams lp{};
    lp.dump = dump_dev; lp.dump_t = dump_t_dev; lp.coef = coef_dev; lp.up = up_dev; lp.w_eik = w_eik_dev; lp.dist = dist_dev;
    lp.uniform = uniform; lp.ws = h->d_ws.get(); lp.B = B; lp.ws_stride = (long long)ws_stride; lp.w6_off = L.w_off[6]; lp.b6_off = L.b_off[6];
    lp.kc = kc; lp.slot0 = 0; lp.z6_col = z_col[6]; lp.softplus = (h->cfg.df_act == PNDF_ACT_SOFTPLUS); lp.beta = h->cfg.df_beta;
    wgrad_last_kernel<<<(unsigned)ksplits, 256, 0, st>>>(lp);
    CUDA_OK(cudaGetLastError());
    int n_enc_rows = 0;
    float* enc_part = nullptr;
    if (h->cfg.use_enc) {
        EncTrainParams ep{};
        ep.x = pose_dev; ep.v = (w_eik_dev || upz_dev) ? v_dev : nullptr; ep.encw = h->d_small.get() + h->off_enc; ep.upz = upz_dev;
        ep.g0 = dump_dev + 5376; ep.g0_ld = kDumpRows; ep.coef = coef_dev; ep.uniform = uniform; ep.up = up_dev;
        ep.weik = dump_t_dev ? w_eik_dev : nullptr;
        ep.grads = h->d_encrows.get(); ep.B = B; ep.normalise = normalise; ep.act = h->cfg.enc_act; ep.beta = h->cfg.enc_beta; ep.use_enc = 1;
        enc_grad_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(ep);
        CUDA_OK(cudaGetLastError());
        const int nsets = (ep.weik || ep.upz) ? 2 : 1;
        enc_part = h->d_encrows.get() + (size_t)2 * nwarps * kEncFloats;      // after this call's per-warp rows (ensure_encrows)
        enc_rows_partial_kernel<<<dim3((unsigned)((nsets * kEncFloats + 255) / 256), kEncChunks), 256, 0, st>>>(h->d_encrows.get(), nwarps, nsets, enc_part);
        CUDA_OK(cudaGetLastError());
        n_enc_rows = kEncChunks * nsets;     // [set][chunk] rows, summed in this order by the reduce kernel
        h->launches++;
    }
    wgrad_reduce_kernel<<<(unsigned)((n_params + 255) / 256), 256, 0, st>>>(h->d_ws.get(), ksplits, (long long)ws_stride, (long long)n_params,
                                                                           L.enc_floats, enc_part, n_enc_rows, grad_flat_dev, overwrite);
    CUDA_OK(cudaGetLastError());
    h->launches += 3;
    return 0;
}

int pndf_adam_step(pndf_handle* h, float* param_flat_dev, const float* grad_flat_dev, float* exp_avg_dev, float* exp_avg_sq_dev,
                   size_t n, double lr, double beta1, double beta2, double eps, double weight_decay, double grad_scale,
                   int64_t step, void* stream) {
    if (!h) return fail("null handle");
    if (!param_flat_dev || !grad_flat_dev || !exp_avg_dev || !exp_avg_sq_dev) return fail("pndf_adam_step: null argument");
    if (n != param_count(&h->cfg)) return fail("pndf_adam_step: wrong parameter count");
    if (step < 1) return fail("pndf_adam_step: step counts from 1");
    CUDA_OK(cudaSetDevice(h->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    AdamStepParams p{};
    p.param = param_flat_dev; p.grad = grad_flat_dev; p.m = exp_avg_dev; p.v = exp_avg_sq_dev; p.n = (long long)n;
    p.lr_over_bias1 = (float)(lr / (1.0 - std::pow(beta1, (double)step)));
    p.bias2_sqrt = (float)std::sqrt(1.0 - std::pow(beta2, (double)step));
    p.one_minus_beta1 = (float)(1.0 - beta1); p.beta2 = (float)beta2; p.one_minus_beta2 = (float)(1.0 - beta2);
    p.eps = (float)eps; p.weight_decay = (float)weight_decay; p.grad_scale = (float)grad_scale;
    p.pos_a = h->d_pos[0].get(); p.pos_b = h->d_pos[1].get(); p.pos_s = h->d_pos[2].get();
    p.wstream = h->d_wstream.get(); p.small = h->d_small.get();
    if (write_weights(h, param_flat_dev, st, [&] { adam_step_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p); })) return 1;
    h->launches++;
    return 0;
}

int pndf_feed_batch(int device, const float* pose_table_dev, const float* dist_table_dev, const int64_t* file_off_dev,
                    const float* amass_table_dev, const int64_t* amass_off_dev, const int32_t* item_file_dev,
                    const int32_t* item_amass_dev, int b, int num_pts, int flip, int fix_flip_bug, uint64_t seed,
                    const int64_t* rows_dev, const int64_t* amass_rows_dev, float* pose_out_dev, float* dist_out_dev,
                    float* man_out_dev, void* stream) {
    if (b == 0 || num_pts == 0) return 0;
    if (b < 0 || num_pts < 0 || !pose_table_dev || !dist_table_dev || !file_off_dev || !amass_table_dev || !amass_off_dev ||
        !item_file_dev || !item_amass_dev || !pose_out_dev || !dist_out_dev || !man_out_dev)
        return fail("pndf_feed_batch: null argument");
    static_assert(sizeof(long long) == sizeof(int64_t), "int64_t is long long");
    CUDA_OK(cudaSetDevice(device));
    FeedParams p{};
    p.pose_table = pose_table_dev; p.dist_table = dist_table_dev; p.file_off = (const long long*)file_off_dev;
    p.amass_table = amass_table_dev; p.amass_off = (const long long*)amass_off_dev; p.item_file = item_file_dev;
    p.item_amass = item_amass_dev; p.rows = (const long long*)rows_dev; p.amass_rows = (const long long*)amass_rows_dev;
    p.pose_out = pose_out_dev; p.dist_out = dist_out_dev; p.man_out = man_out_dev;
    p.b = b; p.num_pts = num_pts; p.flip = flip; p.fix_flip_bug = fix_flip_bug; p.seed = seed;
    const long long warps = (long long)b * num_pts;
    const unsigned grid = (unsigned)std::min<long long>((warps + 7) / 8, 148LL * 16);
    feed_batch_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p);
    CUDA_OK(cudaGetLastError());
    return 0;
}

int pndf_axis_angle_to_quaternion(int device, const float* aa_dev, int64_t n, float* quat_dev, void* stream) {
    if (n == 0) return 0;
    if (n < 0 || !aa_dev || !quat_dev) return fail("pndf_axis_angle_to_quaternion: bad argument");
    CUDA_OK(cudaSetDevice(device));
    aa_to_quat_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(aa_dev, quat_dev, n);
    CUDA_OK(cudaGetLastError());
    return 0;
}

int pndf_quaternion_to_axis_angle(int device, const float* quat_dev, int64_t n, float* aa_dev, void* stream) {
    if (n == 0) return 0;
    if (n < 0 || !aa_dev || !quat_dev) return fail("pndf_quaternion_to_axis_angle: bad argument");
    CUDA_OK(cudaSetDevice(device));
    quat_to_aa_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(quat_dev, aa_dev, n);
    CUDA_OK(cudaGetLastError());
    return 0;
}

int pndf_knn_rerank(int device, const float* query_dev, int64_t Q, const float* database_dev, const int32_t* cand_dev, int K,
                    int metric, int weighted, float* out_val_dev, int32_t* out_pos_dev, void* stream) {
    if (Q == 0) return 0;
    if (Q < 0 || K < kKnnK || !query_dev || !database_dev || !cand_dev || !out_val_dev || !out_pos_dev)
        return fail("pndf_knn_rerank: null argument or K < 5");
    if (metric != 0 && metric != 1) return fail("pndf_knn_rerank: metric must be 0 (geo) or 1 (euc)");
    CUDA_OK(cudaSetDevice(device));
    KnnParams p{};
    p.query = query_dev; p.database = database_dev; p.cand = cand_dev; p.out_val = out_val_dev; p.out_pos = out_pos_dev;
    p.Q = Q; p.K = K; p.metric = metric; p.weighted = weighted;
    knn_rerank_kernel<<<(unsigned)((Q + 3) / 4), 128, 0, (cudaStream_t)stream>>>(p);
    CUDA_OK(cudaGetLastError());
    return 0;
}

int pndf_knn_exact(int device, const float* query_dev, int64_t Q, const float* database_dev, int64_t N, int metric, int weighted,
                   float* out_val_dev, int32_t* out_idx_dev, void* stream) {
    if (Q == 0) return 0;
    if (Q < 0 || N < kKnnK || N > 0x7fffffffLL || !query_dev || !database_dev || !out_val_dev || !out_idx_dev)
        return fail("pndf_knn_exact: null argument or fewer than 5 database poses");
    if (metric != 0 && metric != 1) return fail("pndf_knn_exact: metric must be 0 (geo) or 1 (euc)");
    if ((reinterpret_cast<uintptr_t>(database_dev) & 15) != 0) return fail("pndf_knn_exact: database must be 16-byte aligned");
    CUDA_OK(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    static bool attr_set[64] = {};
    if (device < 64 && !attr_set[device]) {
        CUDA_OK(cudaFuncSetAttribute(knn_exact_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kExSmem));
        CUDA_OK(cudaFuncSetAttribute(knn_exact_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kExSmem));
        attr_set[device] = true;
    }
    int sms = 148;
    CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    // database slices: enough CTAs for ~4 per SM, slices are whole 128-row tiles
    const long long gx = (Q + kExQ - 1) / kExQ;
    const long long tiles = (N + kExD - 1) / kExD;
    long long want = std::max<long long>(1, (4LL * sms + gx - 1) / gx);
    want = std::min(want, tiles);
    const long long tiles_per_split = (tiles + want - 1) / want;
    const int nsplit = (int)((tiles + tiles_per_split - 1) / tiles_per_split);
    float* part_val = nullptr;
    int32_t* part_idx = nullptr;
    const size_t nelem = (size_t)Q * nsplit * kKnnK;
    CUDA_OK(cudaMallocAsync(&part_val, nelem * sizeof(float), st));
    CUDA_OK(cudaMallocAsync(&part_idx, nelem * sizeof(int32_t), st));
    KnnExactParams p{};
    p.query = query_dev; p.database = database_dev; p.part_val = part_val; p.part_idx = part_idx;
    p.Q = Q; p.N = N; p.rows_per_split = tiles_per_split * kExD; p.nsplit = nsplit; p.weighted = weighted;
    const dim3 grid((unsigned)gx, (unsigned)nsplit);
    if (metric == 0) knn_exact_kernel<0><<<grid, kExThreads, kExSmem, st>>>(p);
    else knn_exact_kernel<1><<<grid, kExThreads, kExSmem, st>>>(p);
    CUDA_OK(cudaGetLastError());
    knn_merge_kernel<<<(unsigned)((Q + 127) / 128), 128, 0, st>>>(part_val, part_idx, Q, nsplit, out_val_dev, out_idx_dev);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaFreeAsync(part_val, st));
    CUDA_OK(cudaFreeAsync(part_idx, st));
    return 0;
}

int pndf_set_tile_policy(pndf_handle* h, int tile) {
    if (!h) return fail("null handle");
    if (tile != 0 && tile != 8 && tile != 32 && tile != 128) return fail("pndf_set_tile_policy: tile must be 0 (auto), 8, 32 or 128");
    if (tile == 128 && !h->tc) return fail("pndf_set_tile_policy: the tensor-core path is not available on this handle");
    h->tile_policy = tile;
    return 0;
}
int pndf_tile_for_batch(pndf_handle* h, int64_t B, int* tile) {
    if (!h || !tile || B < 0) return fail("bad argument");
    *tile = batch_tile(h, B);
    return 0;
}

int pndf_launch_count(pndf_handle* h, int64_t* n) {
    if (!h || !n) return fail("null argument");
    *n = h->launches;
    return 0;
}
int pndf_num_sms(pndf_handle* h, int* n) {
    if (!h || !n) return fail("null argument");
    *n = h->num_sms;
    return 0;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// fp32 FMA peak micro-benchmark (roofline denominator for an FFMA-bound kernel; measured, not nominal)
namespace {

template <int VARIANT>
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters, float seed) {
    // 8x8 register tile like the GEMM inner loop: 64 independent accumulators.
    // VARIANT 0: scalar FFMA, operands in registers      1: packed FFMA2 (fma.rn.f32x2)
    //         2: half FFMA2 + half scalar FFMA           3: FFMA2 with the GEMM's shared-memory operand traffic
    //            (4 LDS.128 per 32 FFMA2, broadcast pattern of the fused kernel)
    __shared__ float4 sm[1152];
    float a[8], b[8], acc[8][8];
    if (VARIANT == 3 || VARIANT == 4) {
        for (int i = threadIdx.x; i < 1152; i += blockDim.x) sm[i] = make_float4(seed, -seed, 0.5f * seed, 0.25f * seed);
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        a[i] = seed + 0.001f * (threadIdx.x + i);
        b[i] = seed - 0.002f * (threadIdx.x + i);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int mg = (VARIANT == 4) ? (lane & 3) : (lane >> 3), ngl = (VARIANT == 4) ? (lane >> 2) : (lane & 7);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int rep = 0; rep < 4; ++rep) {
            if (VARIANT == 3 || VARIANT == 4) {
                const int k = (it * 4 + rep) & 7;
                const float4 a0 = sm[k * 8 + ((2 * mg) ^ k)], a1 = sm[k * 8 + ((2 * mg + 1) ^ k)];
                const float4 b0 = sm[64 + k * 128 + warp * 8 + ngl], b1 = sm[64 + k * 128 + 64 + warp * 8 + ngl];
                a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
                b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w; b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
            }
            if (VARIANT == 0) {
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            } else if (VARIANT == 5) {
                // same FMAs, feature pair outermost (the b pair is the reused operand, 8 pose scalars stream past it)
#pragma unroll
                for (int j = 0; j < 8; j += 2) {
                    unsigned long long bb;
                    asm("mov.b64 %0, {%1, %2};" : "=l"(bb) : "f"(b[j]), "f"(b[j + 1]));
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        unsigned long long aa, cc;
                        asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(a[i]));
                        asm("mov.b64 %0, {%1, %2};" : "=l"(cc) : "f"(acc[i][j]), "f"(acc[i][j + 1]));
                        asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(cc) : "l"(aa), "l"(bb));
                        asm("mov.b64 {%0, %1}, %2;" : "=f"(acc[i][j]), "=f"(acc[i][j + 1]) : "l"(cc));
                    }
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    unsigned long long aa;
                    asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(a[i]));
#pragma unroll
                    for (int j = 0; j < 8; j += 2) {
                        if (VARIANT == 2 && j >= 4) {
                            acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
                            acc[i][j + 1] = fmaf(a[i], b[j + 1], acc[i][j + 1]);
                        } else {
                            unsigned long long bb, cc;
                            asm("mov.b64 %0, {%1, %2};" : "=l"(bb) : "f"(b[j]), "f"(b[j + 1]));
                            asm("mov.b64 %0, {%1, %2};" : "=l"(cc) : "f"(acc[i][j]), "f"(acc[i][j + 1]));
                            asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(cc) : "l"(aa), "l"(bb));
                            asm("mov.b64 {%0, %1}, %2;" : "=f"(acc[i][j]), "=f"(acc[i][j + 1]) : "l"(cc));
                        }
                    }
                }
            }
        }
    }
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) s += acc[i][j];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// legacy warp-level tensor-core path (mma.sync) throughput probes: variant 10 = tf32 m16n8k8, 11 = bf16 m16n8k16.
// 16 independent accumulator tiles per warp (32 poses x 64 features), fragments in registers.
template <int VARIANT>
__global__ void __launch_bounds__(256) mma_peak_kernel(float* out, int iters, float seed) {
    float c[16][4];
    unsigned a[2][4], b[8][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int r = 0; r < 4; ++r) a[i][r] = __float_as_uint(seed + 0.001f * (threadIdx.x + r + i));
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int r = 0; r < 2; ++r) b[j][r] = __float_as_uint(seed - 0.002f * (threadIdx.x + r + j));
#pragma unroll
    for (int t = 0; t < 16; ++t)
#pragma unroll
        for (int r = 0; r < 4; ++r) c[t][r] = 0.0f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float* d = c[i * 8 + j];
                if (VARIANT == 10) {
                    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                                 : "r"(a[i][0]), "r"(a[i][1]), "r"(a[i][2]), "r"(a[i][3]), "r"(b[j][0]), "r"(b[j][1]));
                } else {
                    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                                 : "r"(a[i][0]), "r"(a[i][1]), "r"(a[i][2]), "r"(a[i][3]), "r"(b[j][0]), "r"(b[j][1]));
                }
            }
    }
    float s = 0.0f;
#pragma unroll
    for (int t = 0; t < 16; ++t)
#pragma unroll
        for (int r = 0; r < 4; ++r) s += c[t][r];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace

extern "C" int pndf_fp32_peak(int device, int variant, double* tflops) {
    if (!tflops) return fail("null argument");
    CUDA_OK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_OK(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * ((variant == 3 || variant == 4) ? 1 : 4), threads = 256, iters = ((variant == 3 || variant == 4) ? 8192 : 2048);
    float* out = nullptr;
    CUDA_OK(cudaMalloc(&out, (size_t)blocks * threads * sizeof(float)));
    cudaEvent_t e0, e1;
    CUDA_OK(cudaEventCreate(&e0));
    CUDA_OK(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CUDA_OK(cudaEventRecord(e0));
        if (variant == 0) fp32_peak_kernel<0><<<blocks, threads>>>(out, iters, 0.5f);
        else if (variant == 1) fp32_peak_kernel<1><<<blocks, threads>>>(out, iters, 0.5f);
        else if (variant == 2) fp32_peak_kernel<2><<<blocks, threads>>>(out, iters, 0.5f);
        else if (variant == 3) fp32_peak_kernel<3><<<blocks, threads>>>(out, iters, 0.5f);
        else if (variant == 4) fp32_peak_kernel<4><<<blocks, threads>>>(out, iters, 0.5f);
        else if (variant == 5) fp32_peak_kernel<5><<<blocks, threads>>>(out, iters, 0.5f);
        else if (variant == 10) mma_peak_kernel<10><<<blocks, threads>>>(out, iters, 0.5f);
        else mma_peak_kernel<11><<<blocks, threads>>>(out, iters, 0.5f);
        CUDA_OK(cudaEventRecord(e1));
        CUDA_OK(cudaEventSynchronize(e1));
        CUDA_OK(cudaGetLastError());
        float ms = 0.0f;
        CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
        const double per_thread = (variant >= 10) ? 2.0 * 16.0 * (16 * 8 * (variant == 10 ? 8 : 16)) / 32.0 * iters
                                                  : 2.0 * 64.0 * 4.0 * iters;
        const double flops = per_thread * (double)blocks * threads;
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    *tflops = best;
    return 0;
}
