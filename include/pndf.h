/*
 * pndf.h -- C ABI of the B200-native PoseNDF distance-field / projection engine (libpndf.so).
 *
 * The reference (garvita-tiwari/PoseNDF) has no plugin / FFI interface; its boundary for this path is
 * the Python class surface of PoseNDF(nn.Module).  Every entry point below names the reference
 * interface it replaces (file:line under the reference root).  All signatures are plain C: pointers,
 * sizes, ints.  No torch types, no exceptions across the ABI.
 *
 * Conventions
 *   - return value: 0 = ok, non-zero = error (message via pndf_last_error(), thread-local).  An error return, a failed
 *     allocation included, leaves the handle usable.
 *   - "dev" pointers are CUDA device pointers on the handle's device, contiguous fp32, 16-byte aligned.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); all device work is enqueued
 *     on it, nothing synchronises implicitly, the caller owns every buffer it passes in.
 *   - the library owns only what hangs off the handle (packed weight stream, per-CTA scratch).
 *   - a pose is 21 joints x 4 quaternion components, row-major, 84 floats = 336 bytes.
 *   - a handle is not thread-safe; use one handle per device per thread, and drive it from ONE caller stream at a
 *     time: the per-CTA scratch hanging off the handle is indexed by block only, so two launches of the same handle
 *     must not overlap (launches on the same stream never do; pndf_project_host's two internal streams have their
 *     own scratch copies).  Ordering that the library does handle across streams: a launch waits for the last weight
 *     repack, and a weight repack waits for the last launch (events).
 */
#ifndef PNDF_H_
#define PNDF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PNDF_ACT_RELU 0     /* nn.ReLU                       model/network/net_modules.py:34-36,86-92  */
#define PNDF_ACT_LRELU 1    /* nn.LeakyReLU() slope 0.01     model/network/net_modules.py:30-32,94-100 */
#define PNDF_ACT_SOFTPLUS 2 /* nn.Softplus(beta), thr 20     model/network/net_modules.py:39-41,101-107 */

#define PNDF_NUM_JOINTS 21
#define PNDF_POSE_FLOATS 84
#define PNDF_MAX_HIDDEN 8

/* The slice of the reference's `opt` dict the hot path reads (model/posendf.py:35-55,
 * model/network/net_modules.py:14-15,30-41,128). */
typedef struct pndf_config {
    int32_t use_enc;               /* opt['model']['StrEnc']['use']                                    */
    int32_t enc_act;               /* opt['model']['StrEnc']['act']   -> PNDF_ACT_*                    */
    float enc_beta;                /* opt['model']['StrEnc']['beta']                                   */
    int32_t df_act;                /* opt['model']['DFNet']['act']                                     */
    float df_beta;                 /* opt['model']['DFNet']['beta']                                    */
    int32_t in_dim;                /* opt['model']['DFNet']['in_dim'] (126 with encoder, 84 without)   */
    int32_t num_hidden;            /* len(opt['model']['DFNet']['dims'])                               */
    int32_t dims[PNDF_MAX_HIDDEN]; /* opt['model']['DFNet']['dims']                                    */
    int32_t device;                /* CUDA ordinal (opt['train']['device'])                            */
} pndf_config;

typedef struct pndf_handle pndf_handle;

/* PoseNDF.__init__  (model/posendf.py:32-55).  Fails (non-zero) for architectures the fused kernel does
 * not implement -- there is no fallback path. */
int pndf_create(const pndf_config* cfg, pndf_handle** out);
int pndf_destroy(pndf_handle* h);

/* Number of fp32 parameters for cfg (1 365 565 for configs/amass.yaml), i.e. the length of the flat
 * vector pndf_set_weights expects. */
int pndf_param_count(const pndf_config* cfg, size_t* n);

/* load_state_dict (experiments/sample_poses.py:90-91, model/train_posendf.py:158-176).
 * `flat` is a HOST pointer to the state_dict tensors concatenated in the reference's own order:
 *   enc.net.{i}.net.0.weight, .0.bias, .2.weight, .2.bias  for i = 0..20   (only if use_enc)
 *   dfnet.lin{l}.weight (out,in row-major), dfnet.lin{l}.bias              for l = 0..num_hidden
 * The library repacks it into the slab stream the kernel consumes and uploads it (synchronous). */
int pndf_set_weights(pndf_handle* h, const float* flat, size_t n);

/* The same for a DEVICE pointer (the trainer's parameters after optimizer.step(), model/train_posendf.py:99):
 * the repacking is a gather kernel enqueued on `stream`, no host round trip, no synchronisation.  Launches that
 * use the handle afterwards must be ordered after it (same stream or an event). */
int pndf_set_weights_device(pndf_handle* h, const float* flat_dev, size_t n, void* stream);

/* PoseNDF.forward(pose, train=False)['dist_pred']  (model/posendf.py:62-76,100-101).
 * normalise != 0 applies F.normalize(pose, dim=1) (posendf.py:71); normalise == 0 is the manifold
 * branch of the train path (posendf.py:80-83).  dist_dev: B floats. */
int pndf_forward(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, float* dist_dev, void* stream);

/* forward + gradient(pose, dist_pred)  (model/posendf.py:18-27 / experiments/sample_poses.py:25-34,73;
 * with an upstream gradient it is the backward of experiments/motion_denoise.py:98 through the prior).
 * g_up_dev: B floats or NULL (= ones).  grad_dev: B*84 floats = g_up[b] * d dist[b] / d pose[b]. */
int pndf_forward_grad(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, const float* g_up_dev,
                      float* dist_dev, float* grad_dev, void* stream);

/* The projection loop body, `steps` times, in one launch (experiments/sample_poses.py:70-74):
 *     pose <- pose - dist * d dist / d pose
 * renorm != 0 re-normalises every quaternion after each step (north-star option; the reference does
 * not, SURVEY Q6).  pose_dev is updated in place; dist_dev (B floats, may be NULL) receives the
 * distance evaluated at the start of the last step, as the reference's loop leaves it. */
int pndf_project(pndf_handle* h, float* pose_dev, int64_t B, int steps, int renorm, float* dist_dev, void* stream);

/* Same as pndf_project but with HOST buffers (what a non-CUDA caller of the reference's
 * SamplePose.project would hold): pinned staging, chunked H2D / kernel / D2H overlap inside.
 * pose_out_host may alias pose_in_host.  Synchronous. */
int pndf_project_host(pndf_handle* h, const float* pose_in_host, float* pose_out_host, float* dist_host,
                      int64_t B, int steps, int renorm);

/* Multi-GPU projection run (BASELINE configs[2]: the loop of experiments/sample_poses.py:70-74 over a pose batch sharded
 * across the GPUs of one node, ONE gather of the projected poses at the end; the reference itself has no distributed
 * code).  pndf_project on this rank's shard, fused with the gather: the kernel's write-back also stores every projected
 * tile (and its distance) straight into the gathered buffers of `n_peers` other GPUs through NVLink-mapped pointers
 * (peer_pose_dev[r] / peer_dist_dev[r] = where THIS rank's slice starts inside peer r's gathered buffer; peer_dist_dev may
 * be NULL), so the transfer overlaps the arithmetic tile by tile.  Completion on the peers = this stream reaching a
 * pndf_peer_barrier.  n_peers <= 7. */
int pndf_project_gather(pndf_handle* h, float* pose_dev, int64_t B, int steps, int renorm, float* dist_dev,
                        float* const* peer_pose_dev, float* const* peer_dist_dev, int n_peers, void* stream);

/* Peer memory for the fused gather, one process per GPU: cudaMalloc'ed, zero-filled buffer + its 64-byte cudaIpc handle
 * (the caller ships the handle bytes to the other ranks -- torch.distributed in posendf_b200/dist.py); open / close map
 * another rank's buffer into this process (peer access enabled lazily). */
int pndf_peer_alloc(int device, size_t bytes, void** dev_ptr, unsigned char* handle64);
int pndf_peer_open(int device, const unsigned char* handle64, void** dev_ptr);
int pndf_peer_close(int device, void* dev_ptr);
int pndf_peer_free(int device, void* dev_ptr);
/* Barrier of the `world` ranks over peer memory, enqueued on `stream`: flags_dev[r] = rank r's flag array (world + 1
 * uint32, zero-initialised, inside its peer buffer; flags_dev[rank] is the local one).  Stores `epoch` (increasing,
 * same on all ranks) into every rank's array with release/system semantics -- ordered after all earlier peer stores of
 * this stream -- and waits for every rank's epoch.  A rank that never arrives sets the local error slot [world] after
 * ~10 s instead of hanging the GPU. */
int pndf_peer_barrier(int device, uint32_t* const* flags_dev, int world, int rank, uint32_t epoch, void* stream);

/* Motion-denoise prior term (experiments/motion_denoise.py:81-83,97-98):
 *   quat = axis_angle_to_quaternion(aa)   (pytorch3d 0.7.2 formula), dist = PoseNDF(quat),
 *   grad_aa = g_up[b] * d dist[b] / d aa[b]   (g_up NULL = ones).
 * aa_dev: B*63 floats (21 joints x 3).  dist_dev: B floats.  grad_aa_dev: B*63 floats. */
int pndf_prior_grad(pndf_handle* h, const float* aa_dev, int64_t B, const float* g_up_dev, float* dist_dev,
                    float* grad_aa_dev, void* stream);

/* Motion-denoise inner loop restricted to the prior term (experiments/motion_denoise.py:70,74-83,97-99 with the
 * weights of :29-35): for it in range(iterations): for i in range(steps_per_iter):
 *     loss_s = 1e7/(1+it) * mean_t(dist[s,t])^2  per sequence s;  backward to the axis-angle pose;  Adam(lr) step.
 * aa_dev: S*T*63 floats, updated in place (S sequences of T frames, 21 joints x 3).  dist_dev (S*T, may be NULL):
 * distances of the last evaluated step.  loss_hist_dev (iterations*steps_per_iter*S floats, may be NULL): the
 * weighted prior loss per step and sequence.  ONE launch per step: the fused prior kernel of step t applies, in its tile
 * prologue, the Adam update step t-1 asked for (the per-sequence mean of dist couples the tiles of a sequence, so it is read
 * back from the previous launch's distances); a small per-sequence kernel applies the last update.  Sequences are independent,
 * so they run as two groups with their own launch chains side by side (the tail round of one group's launch overlaps the other
 * group's next launch).  The 2 x (steps_total + 1) launches are captured into a CUDA graph and replayed as one graph launch on
 * `stream` (PNDF_NO_GRAPH=1 in the environment: plain launches on `stream` and one internal stream).  When S*T poses select the
 * tensor-core engine (more than 8 x SMs poses, at most 131 072) the loop is ONE chain over all sequences instead -- 15 kernels per
 * step, the pending Adam update in the prologue of the first one -- issued as plain launches on `stream` (the host stays ahead of
 * them; a 1 501-node graph would cost more to build than it saves).  Same results within the parity bars, same arguments.
 * The SMPL temporal / data terms need licensed SMPL files and are out of scope. */
int pndf_denoise_prior(pndf_handle* h, float* aa_dev, int64_t S, int64_t T, int iterations, int steps_per_iter, float lr,
                       float* dist_dev, float* loss_hist_dev, void* stream);

/* Debug / test hook: like pndf_forward_grad for the first 32 poses only, additionally dumping every
 * intermediate activation / gradient tile (layout documented in DESIGN.md) to dump_dev (floats). */
int pndf_debug_dump_floats(size_t* n);
int pndf_forward_grad_debug(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, float* dist_dev,
                            float* grad_dev, float* dump_dev, void* stream);

/* Training support (model/posendf.py:78-99, model/train_posendf.py:93-99; host side in posendf_b200/train.py).
 * pndf_forward_grad_export = pndf_forward_grad (unit upstream gradient) that additionally writes, for EVERY 32-pose
 * pose b (padded to a multiple of 32), all layer inputs z_l and all pre-activation adjoints to dump_dev[b][5504]
 * (column map in DESIGN.md): plain strided (B x width) operands of the weight-gradient GEMMs
 * dW_l = sum_b adj_l[b] (x) z_l[b].
 * pndf_forward_tangent_export recomputes the forward pass and then pushes the tangent tan_dev[t][128][32] of the DFNet
 * input through the linearised network (forward mode), exporting the tangents of all layer inputs to columns
 * [0,2752) of dump_dev[b]: the second operand of the Eikonal term's weight gradients.
 * act_handoff_dev (nullable, pndf_act_handoff_bytes(h, B) bytes): launch 1 stores the activation derivatives of every
 * hidden unit there -- 1 bit per unit and pose for a relu / lrelu DFNet (10.6 KB per 32 poses), fp32 for softplus
 * (10.5 KB per pose) -- and the tangent launch, given the same buffer, skips its own primal forward pass (half of its
 * arithmetic). */
int pndf_act_handoff_bytes(const pndf_handle* h, int64_t B, size_t* n);
int pndf_forward_grad_export(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, float* dist_dev, float* grad_dev,
                             float* dump_dev, void* act_handoff_dev, void* stream);
int pndf_forward_tangent_export(pndf_handle* h, const float* pose_dev, int64_t B, int normalise, const float* tan_dev,
                                float* dump_dev, const void* act_handoff_dev, void* stream);

/* One element-wise step of the softplus second-order adjoint chain of the Eikonal term (the double backward of
 * model/posendf.py:89-96 / model/train_posendf.py:98 for act: softplus):
 *   pbar[b][j] = zbar[b][j] * s + w * beta (1 - s) * adj[b][j] * zdot_next[b][j] / s ,   s = 1 - exp(-beta z_next[b][j])
 * z_next, zdot_next, adj are (B x n) column slices of the pose-major exports (row stride ld floats); zbar, pbar dense;
 * w_eik_dev a device scalar (nullable = 1).  n and ld multiples of 4, pointers 16-byte aligned. */
int pndf_softplus_adjoint(int device, const float* z_next_dev, const float* zdot_next_dev, const float* adj_dev, int64_t ld,
                          const float* zbar_dev, const float* w_eik_dev, float beta, int64_t B, int n, float* pbar_dev,
                          void* stream);

/* Structure-encoder side of the training step (model/network/net_modules.py:140-170, 3 516 parameters).
 * pndf_encoder_tangent: tangent of the encoder output (or of the normalised pose without encoder) along the pose
 *   tangent v_dev (B*84), written as the [tile][128][32] input of pndf_forward_tangent_export.
 * pndf_encoder_param_grads: parameter gradients (reference order, 3 516 floats per set) of
 *     set 0:  sum_b <up_first[b], z0[b]>                      set 1:  sum_b <up_tangent[b], zdot0[b]> + <up_second[b], z0[b]>
 *   into grads_dev[2][3516] (zeroed here; any of the three upstream arrays (B*126) may be NULL), including the
 *   second-derivative terms of a softplus encoder. */
int pndf_encoder_tangent(pndf_handle* h, const float* pose_dev, const float* v_dev, int64_t B, int normalise,
                         float* zdot_tiles_dev, void* stream);
int pndf_encoder_param_grads(pndf_handle* h, const float* pose_dev, const float* v_dev, int64_t B, int normalise,
                             const float* up_first_dev, const float* up_tangent_dev, const float* up_second_dev,
                             float* grads_dev, void* stream);

/* ---- training step, native end to end (model/posendf.py:78-99 losses, model/train_posendf.py:93-99 backward + Adam) ----
 *
 * pndf_train_losses: the per-pose part of the three losses on the outputs of pndf_forward_grad_export, one chunk of the
 * batch at a time (B poses of B_total):
 *   mode 0 (pose batch):     losses[0] = L1|MSE(dist, dist_gt) (l2 selects MSE), coef[b] = dLoss/ddist[b];
 *                            with grad_dev (B*84): losses[1] = mean_{b,j} (|g_{b,j}| - 1)^2 and v[b] = dEikonal/dg[b]
 *                            (zero sub-gradient where |g_{b,j}| == 0, as torch's norm backward)      posendf.py:85,89-96
 *   mode 1 (manifold batch): losses[2] = mean |dist|                                                  posendf.py:86
 * reset != 0 on the first chunk of a step.  losses_dev: 3 device floats, valid after the last chunk (running totals live in
 * the handle); block partials are summed in a fixed order.  Nothing synchronises. */
int pndf_train_losses(pndf_handle* h, const float* dist_dev, const float* dist_gt_dev, const float* grad_dev, int64_t B,
                      int64_t B_total, int mode, int l2, int reset, float* coef_dev, float* v_dev, float* losses_dev, void* stream);

/* loss.backward() for one exported chunk (model/train_posendf.py:98): accumulates into the flat gradient vector
 * (reference parameter order, pndf_set_weights layout)
 *     up * d/dtheta sum_b coef[b] dist(x_b)   +   w_eik * d/dtheta Eikonal      (first-order part of the Eikonal term:
 *     exact for relu / lrelu; a softplus DFNet adds its second-order adjoint chain on top, posendf_b200/train.py)
 * from the exports of pndf_forward_grad_export (dump_dev) and pndf_forward_tangent_export (dump_t_dev or NULL): split-K
 * FFMA2 outer-product GEMMs for the six DFNet layers (wgrad_kernel), the last layer, the encoder reverse sweep, and a
 * fixed-order reduction.  coef_dev NULL = the same weight `uniform` for every pose (manifold term).  up_dev / w_eik_dev are
 * DEVICE scalars (the upstream gradients autograd hands to backward()); upz_dev = second-order adjoint of z0 (B*126,
 * softplus DFNet) or NULL; v_dev = the pose tangent the tangent launch used.  overwrite != 0 stores instead of adding. */
int pndf_wgrad_accumulate(pndf_handle* h, const float* pose_dev, const float* v_dev, int normalise, const float* dump_dev,
                          const float* dump_t_dev, const float* coef_dev, float uniform, const float* dist_dev, int64_t B,
                          const float* up_dev, const float* w_eik_dev, const float* upz_dev, float* grad_flat_dev, int overwrite,
                          void* stream);

/* torch.optim.Adam(params, lr, betas, eps, weight_decay).step() (model/train_posendf.py:30,99) on the flat parameter /
 * gradient / moment vectors, same operation order as torch; the same kernel writes the new values into the engine's packed
 * weight buffers, so the next launch sees them without a repack.  grad_scale multiplies the gradient first (1 / world size
 * after a summing all-reduce).  step counts from 1. */
int pndf_adam_step(pndf_handle* h, float* param_flat_dev, const float* grad_flat_dev, float* exp_avg_dev, float* exp_avg_sq_dev,
                   size_t n, double lr, double beta1, double beta2, double eps, double weight_decay, double grad_scale,
                   int64_t step, void* stream);

/* Training-data feed: one trainer batch of PoseData items (model/load_data.py:43-71 __getitem__, :73-77 DataLoader stacking)
 * assembled in ONE launch from tables resident in device memory: all data files concatenated (pose_table N*84, dist_table N*5
 * raw neighbour distances, file_off n_files+1 row offsets), all AMASS files concatenated (amass_table, amass_off).  Item i of
 * the batch uses data file item_file[i] and AMASS file item_amass[i]; every point draws a row of each WITH replacement
 * (counter-based generator keyed by `seed`, or rows_dev / amass_rows_dev [b*num_pts] to inject the indices), dist = mean of
 * the 5 stored distances, flip negates quaternions with a negative real part; with flip the reference overwrites the manifold
 * poses with the flipped noisy poses (load_data.py:63) -- kept unless fix_flip_bug.  Outputs: pose (b*num_pts*84), dist
 * (b*num_pts), man_poses (b*num_pts*84).  Stateless. */
int pndf_feed_batch(int device, const float* pose_table_dev, const float* dist_table_dev, const int64_t* file_off_dev,
                    const float* amass_table_dev, const int64_t* amass_off_dev, const int32_t* item_file_dev,
                    const int32_t* item_amass_dev, int b, int num_pts, int flip, int fix_flip_bug, uint64_t seed,
                    const int64_t* rows_dev, const int64_t* amass_rows_dev, float* pose_out_dev, float* dist_out_dev,
                    float* man_out_dev, void* stream);

/* Rotation formats on either side of the path: pytorch3d.transforms.axis_angle_to_quaternion / quaternion_to_axis_angle
 * (0.7.2; experiments/sample_poses.py:60,80, experiments/motion_denoise.py:81, model/load_data.py:108) on n rotations
 * (n = poses * 21): aa n*3 floats, quat n*4 floats (real part first, 16-byte aligned).  Formulas restated from the
 * published source -- parity unpinned, pytorch3d is not vendored in the reference.  Stateless. */
int pndf_axis_angle_to_quaternion(int device, const float* aa_dev, int64_t n, float* quat_dev, void* stream);
int pndf_quaternion_to_axis_angle(int device, const float* quat_dev, int64_t n, float* aa_dev, void* stream);

/* Distance-label rerank of the dataset preparation (data/dist_utils.py:19-30 `euc`, :41-50 `geo`, topk at
 * data/prepare_traindata.py:156): for each of Q query poses (Q*84 floats) the 5 nearest of its K candidates, given as
 * int32 indices (Q*K) into a database of unit-quaternion poses (N*84 floats).  metric 0 = geo: mean_j (1 - |<q_j, q'_j>|),
 * 1 = euc: mean_j |q_j - q'_j|; weighted != 0 uses the reference's normalised joint ranks instead of the mean.
 * out_val_dev: Q*5 ascending distances, out_pos_dev: Q*5 positions inside the candidate list (torch.topk's indices).
 * Stateless (no handle); HBM-bound: 336 B read per (query, candidate). */
int pndf_knn_rerank(int device, const float* query_dev, int64_t Q, const float* database_dev, const int32_t* cand_dev, int K,
                    int metric, int weighted, float* out_val_dev, int32_t* out_pos_dev, void* stream);

/* The same labels WITHOUT a candidate stage: exact 5 nearest database poses of every query over the whole database
 * (what data/prepare_traindata.py:138-170 approximates with 500 faiss candidates before its rerank; identical to
 * pndf_knn_rerank whenever the candidate list contains the true neighbours).  out_idx_dev: Q*5 int32 row indices into
 * the database (N <= 2^31-1), ascending distance, ties by lower index.  Brute force on the fp32 pipe: 105 FMA per
 * (query, database pose) pair, database tiles streamed once per 64 queries through shared memory by TMA bulk copies.
 * database_dev must be 16-byte aligned.  Stateless; scratch comes from the stream-ordered allocator. */
int pndf_knn_exact(int device, const float* query_dev, int64_t Q, const float* database_dev, int64_t N, int metric, int weighted,
                   float* out_val_dev, int32_t* out_idx_dev, void* stream);

/* Measurement helpers used by bench.py (not on the data path):
 *   pndf_fp32_peak: in-process FFMA micro-benchmark, dense fp32 FMA TFLOP/s of this GPU right now.
 *     variant 0 = scalar FFMA, 1 / 5 = packed FFMA2 (fma.rn.f32x2) with the pose scalar / the feature pair as the
 *     reused operand, 2-4 / 10-11 = probes used while tuning (operand traffic, legacy mma.sync).
 *   pndf_launch_count: number of kernel launches this handle has enqueued so far. */
/* Tile size / arithmetic engine of the forward / forward+reverse launches.  By default every launch picks it from ITS batch size:
 *   B <= 8 x SMs (1 184 on a B200): the fused FFMA kernel's 8-pose small-tile variant (2.4x lower latency than 32-pose tiles at the
 *     reference's real call sites, B = 10 in experiments/sample_poses.py:96);
 *   larger batches, quaternion input or the axis-angle prior mode (pndf_prior_grad, pndf_denoise_prior): the tensor-core engine
 *     ("tile 128": DFNet GEMMs as 3xTF32 tcgen05 kernels on 128-pose tiles, pndf_tc.cu);
 *   training exports, tangent launches, the debug dump, prior-mode batches above 131 072 poses: the fused FFMA kernel with 32-pose
 *     tiles.
 * The engines differ in fp32 summation order / split arithmetic (same parity bars), so a caller that splits ONE batch over several
 * launches or GPUs and wants bits identical to the unsplit run pins the tile the whole batch would get:
 * tile = pndf_tile_for_batch(h, B_total), pndf_set_tile_policy(h, tile), launches, pndf_set_tile_policy(h, 0).
 * posendf_b200/dist.py does this; pndf_project_host runs all its chunks at the tile of its whole batch by itself.
 * PNDF_TILE=8|32|128 in the environment overrides everything (tests, tuning). */
int pndf_set_tile_policy(pndf_handle* h, int tile);
int pndf_tile_for_batch(pndf_handle* h, int64_t B, int* tile);

int pndf_fp32_peak(int device, int variant, double* tflops);
int pndf_launch_count(pndf_handle* h, int64_t* n);
int pndf_num_sms(pndf_handle* h, int* n);

const char* pndf_last_error(void);
const char* pndf_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PNDF_H_ */
