/*
 * ffb6d_b200.h -- C ABI of libffb6d_b200.so: the B200 (sm_100a) implementation of
 * FFB6D's bidirectional-fusion hot path (KNN index build, gather + max-pool /
 * nearest-feature gather, RandLA set-abstraction ops).
 *
 * Every entry point is extern "C", takes plain pointers and sizes, returns
 * FFB6D_OK (0) or a negative error code, and never throws.  ffb6d_last_error()
 * returns a thread-local, human readable message for the last failure.
 *
 * "Reference" citations below are relative to /root/reference/ffb6d/ of
 * ethnhe/FFB6D @ e90baf73.  NN/ = models/RandLA/utils/nearest_neighbors/,
 * GS/ = models/RandLA/utils/cpp_wrappers/.
 *
 * Pointer conventions
 *   *_host entry points take HOST pointers and have the reference's own C++
 *   signatures (NN/knn_.h:2-26): they are what the reference's Cython shim
 *   (NN/knn.pyx:8-31) would bind instead of cpp_knn*.  They copy in, run the
 *   CUDA kernels on the current device's default stream, copy out and
 *   synchronise before returning -- the caller-visible behaviour of the
 *   reference (blocking, caller-allocated output).
 *   All other entry points take DEVICE pointers plus a cudaStream_t passed as
 *   an opaque void* (NULL = default stream), are asynchronous, and never
 *   allocate: temporary storage is caller-provided (see *_workspace_bytes).
 *
 * Index dtype: idx_is_i64 != 0 means int64 ("long", what NN/knn.pyx:93 allocates
 * and what torch.gather consumes), 0 means int32 (what the datasets store,
 * datasets/ycb/ycb_dataset.py:283-309).
 *
 * Feature layouts for the gather ops (the reference tensors are NCHW
 * [B,C,S,1], models/ffb6d.py:159-194):
 *   FFB6D_LAYOUT_NCS  feat[b][c][s]  (contiguous NCHW; point axis fastest)
 *   FFB6D_LAYOUT_NSC  feat[b][s][c]  (torch channels_last view of the same
 *                                     NCHW tensor; channel axis fastest)
 * The output uses the layout of the input.
 */
#ifndef FFB6D_B200_H_
#define FFB6D_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FFB6D_OK              0
#define FFB6D_ERR_INVALID    -1   /* bad argument (shape, K, null pointer, layout) */
#define FFB6D_ERR_CUDA       -2   /* a CUDA runtime call or kernel launch failed  */
#define FFB6D_ERR_WORKSPACE  -3   /* workspace missing or too small               */
#define FFB6D_ERR_NO_DEVICE  -4   /* no CUDA device visible                       */

#define FFB6D_LAYOUT_NCS 0
#define FFB6D_LAYOUT_NSC 1

#define FFB6D_MAX_K 64            /* largest supported neighbour count */

typedef void *ffb6d_stream_t;     /* cudaStream_t */

/* ---- library ------------------------------------------------------------ */
int ffb6d_version(void);                 /* ABI version, bumped on signature change */
const char *ffb6d_last_error(void);      /* thread-local message of the last failure */
int ffb6d_device_count(void);            /* number of CUDA devices, 0 if none / no driver */
/* number of kernels this library has launched in this process (all threads).
 * bench.py reports it as gpu_launches. */
uint64_t ffb6d_launch_count(void);

/* ---- KNN index build ---------------------------------------------------- */
/*
 * Exact K nearest neighbours of every query among the support points of the
 * same batch item, ascending squared distance, fp32 arithmetic identical to
 * nanoflann's L2_Adaptor for dim 3 (NN/nanoflann.hpp:343-346, no FMA).
 * Replaces cpp_knn_batch / cpp_knn_batch_omp (NN/knn_.cxx:72-135).
 *   support [B,S,3] f32, query [B,Q,3] f32 -> idx_out [B,Q,K] int32|int64
 * Ties (exactly equal fp32 distances) are ordered by ascending support index
 * (the reference orders them by KD-tree traversal; see DESIGN.md "tie contract").
 * K > S: slots >= S are written as 0, as the reference leaves them (NN/knn_.cxx:120-121).
 * Workspace: ffb6d_knn_workspace_bytes(B,S,Q,K) bytes of device memory, 256-byte
 * aligned; may be NULL when that function returns 0.
 */
size_t ffb6d_knn_workspace_bytes(int64_t B, int64_t S, int64_t Q, int K);
int ffb6d_knn_batch(const float *support, const float *query,
                    int64_t B, int64_t S, int64_t Q, int K,
                    void *idx_out, int idx_is_i64,
                    void *workspace, size_t workspace_bytes,
                    ffb6d_stream_t stream);

/* Same, selecting the algorithm explicitly (testing / benchmarking):
 * algo 0 = automatic, 1 = tiled brute force, 2 = uniform-grid search. */
int ffb6d_knn_batch_algo(const float *support, const float *query,
                         int64_t B, int64_t S, int64_t Q, int K,
                         void *idx_out, int idx_is_i64,
                         void *workspace, size_t workspace_bytes,
                         int algo, ffb6d_stream_t stream);

/*
 * Build-once / query-many form of the same search, for callers that search one support
 * cloud several times (the FFB6D schedule searches each pyramid level 2-4 times,
 * datasets/ycb/ycb_dataset.py:275-308).  The grid (uniform-cell index of `support`) is
 * written by ffb6d_knn_grid_build into caller memory of ffb6d_knn_grid_bytes(B,S) bytes and
 * is read-only afterwards: queries may run concurrently on any streams ordered after the
 * build.  K_hint only tunes the cell size (performance); results never depend on it.  Each
 * query call needs its own scratch of ffb6d_knn_grid_query_bytes(B,Q) bytes.  `support`
 * must be the array the grid was built from.  Results are identical to ffb6d_knn_batch.
 */
size_t ffb6d_knn_grid_bytes(int64_t B, int64_t S);
size_t ffb6d_knn_grid_query_bytes(int64_t B, int64_t Q);
int ffb6d_knn_grid_build(const float *support, int64_t B, int64_t S, int K_hint,
                         void *grid, size_t grid_bytes, ffb6d_stream_t stream);
int ffb6d_knn_grid_query(const float *support, const float *query,
                         int64_t B, int64_t S, int64_t Q, int K,
                         void *idx_out, int idx_is_i64,
                         const void *grid, size_t grid_bytes,
                         void *scratch, size_t scratch_bytes, ffb6d_stream_t stream);
/* The same search with a layout hint: the Q queries of every batch item are the pixels of an image with
 * rows of `query_width` points, row after row (the stride pyramids of the organised cloud,
 * ycb_dataset.py:253-267).  For K = 1 the 32 queries of an 8x4 pixel tile then share one candidate set.
 * Results are identical to ffb6d_knn_grid_query; query_width = 0 means "no particular order". */
int ffb6d_knn_grid_query_organized(const float *support, const float *query,
                                   int64_t B, int64_t S, int64_t Q, int K,
                                   void *idx_out, int idx_is_i64,
                                   const void *grid, size_t grid_bytes,
                                   void *scratch, size_t scratch_bytes,
                                   int64_t query_width, ffb6d_stream_t stream);

/*
 * cld_interp_idx{i} (datasets/ycb/ycb_dataset.py:280-282: the nearest level-(i+1) point of every level-i point) read
 * off cld_nei_idx{i} (:275-277) instead of searched.  `query` [B,Q,3] is a cloud level, `support` [B,S,3] its first S
 * rows (the next level, :278), `knn_idx` [B,Q,K_list] the K-neighbour self search of `query` (rows ordered by
 * (distance, index), what ffb6d_knn_batch / ffb6d_knn_grid_query produce, same index dtype as idx_out).  The first
 * entry of a row that is < S is the nearest subset point under the same total order; rows without one are answered
 * by a full scan of the support.  idx_out [B,Q,1]; scratch: ffb6d_knn_grid_query_bytes(B, Q).  Results are identical
 * to ffb6d_knn_batch(support, query, ..., K = 1).
 */
int ffb6d_knn_subset_nn(const float *support, const float *query, int64_t B, int64_t S, int64_t Q,
                        const void *knn_idx, int K_list, void *idx_out, int idx_is_i64,
                        void *scratch, size_t scratch_bytes, ffb6d_stream_t stream);

/*
 * The whole index build of a batch in one call: the 22 searches of datasets/ycb/ycb_dataset.py:269-309
 * (== datasets/linemod/linemod_dataset.py:313-353) on `stream`, one grid per (support set, K class).
 *   cld  [B,N0,3]: the sampled, shuffled clouds; level i of the pyramid = the first N0/4^i rows (:278)
 *   img2/img4/img8 [B,(H/sr)*(W/sr),3]: stride-sr sub-grids of the organised cloud (:253-267;
 *                  ffb6d_backproject writes them), zero rows at holes
 *   out[22]: device buffers in the reference's call order -- for i = 0..3: cld_nei_idx{i} [B,N_i,K],
 *            cld_interp_idx{i} [B,N_i,1], r2p_ds_nei_idx{i} [B,N_{i+1},K], p2r_ds_nei_idx{i} [B,HW(sr_i),1]
 *            (sr = 4,8,8,8); then for i = 0..2: r2p_up_nei_idx{i} [B,N_{3-i},K], p2r_up_nei_idx{i}
 *            [B,HW(sr_i),1] (sr = 4,2,2); int32, or int64 with idx_is_i64.  cld_sub_idx{i} is the
 *            first N_{i+1} rows of cld_nei_idx{i} (:279).
 * N0 a multiple of 256, H and W multiples of 8.  workspace: ffb6d_build_indices_workspace_bytes.
 */
size_t ffb6d_build_indices_workspace_bytes(int64_t B, int64_t N0, int64_t H, int64_t W, int K);
int ffb6d_build_indices(const float *cld, const float *img2, const float *img4, const float *img8,
                        int64_t B, int64_t N0, int64_t H, int64_t W, int K,
                        void *const *out, int idx_is_i64, void *workspace, size_t workspace_bytes,
                        ffb6d_stream_t stream);

/* Performance knobs of the grid search (never affect results): the cell edge is
 * cell_scale x the `quantile`-th smallest (0..31) of 32 sampled K-th-neighbour distances.
 * Non-positive / negative arguments leave a knob unchanged.  Defaults 1.0 and 17. */
void ffb6d_knn_grid_tune(float cell_scale, int quantile);
/* Same knob for the grids built for K = 1 searches (default 2.5). */
void ffb6d_knn_grid_tune_k1(float cell_scale_k1);

/* HOST-pointer twins with the reference's exact signatures (NN/knn_.h:2-16);
 * dim must be 3.  `long` is int64 on LP64, as in the reference. */
int ffb6d_knn_batch_host(const float *batch_data, size_t batch_size, size_t npts, size_t dim,
                         const float *queries, size_t nqueries, size_t K, long *batch_indices);
int ffb6d_knn_host(const float *points, size_t npts, size_t dim,
                   const float *queries, size_t nqueries, size_t K, long *indices);

/* ---- gather + max-pool / nearest gather -------------------------------- */
/*
 * out[b,c,q] = max_k feat[b,c,idx[b,q,k]]                       (K >= 1)
 * Replaces FFB6D.random_sample / Network.random_sample (models/ffb6d.py:159-177,
 * models/RandLA/RandLANet.py:87-102) and, with K == 1, FFB6D.nearest_interpolation
 * (models/ffb6d.py:179-194, RandLANet.py:104-117) and the final `choose` gather
 * (models/ffb6d.py:309-312).  Pure selection: results are bitwise equal to the
 * reference (NaN propagates like torch.max).
 *   feat [B,C,S] f32 in `layout`, idx [B,Q,K] -> out [B,C,Q] f32 in `layout`.
 * Indices must lie in [0,S).  The forward kernels do not check them (an offender reads a stale or
 * foreign element where torch.gather raises a device assert); the backward kernels skip offenders.
 * Debugging aid: ffb6d_check_indices below, or FFB6D_CHECK_INDICES=1 in the environment, which runs
 * that check (and synchronises the stream) in front of every gather entry point.
 */
int ffb6d_gather_max_fwd(const float *feat, const void *idx, int idx_is_i64,
                         int64_t B, int64_t C, int64_t S, int64_t Q, int K,
                         int layout, float *out, ffb6d_stream_t stream);
/* Validates `count` indices against [0,S): returns FFB6D_ERR_INVALID (with the number of offenders
 * in ffb6d_last_error) if any lies outside.  Blocking: synchronises `stream`; not capturable. */
int ffb6d_check_indices(const void *idx, int idx_is_i64, int64_t count, int64_t S, ffb6d_stream_t stream);
/* Name of the kernel ffb6d_gather_max_fwd launches for a shape (for profiling tools). */
const char *ffb6d_gather_kernel_name(int64_t B, int64_t C, int64_t S, int64_t Q, int K, int layout);
/*
 * Backward of the above as autograd defines it for gather + max: grad_feat is
 * zero-filled, then grad_out[b,c,q] is added at the arg-max neighbour (the first
 * maximal k).  fp32 atomic adds: summation order is not deterministic, exactly
 * as the reference's torch.gather backward on CUDA.
 */
int ffb6d_gather_max_bwd(const float *feat, const void *idx, int idx_is_i64,
                         const float *grad_out,
                         int64_t B, int64_t C, int64_t S, int64_t Q, int K,
                         int layout, float *grad_feat, ffb6d_stream_t stream);

/*
 * out[b,n,k,:] = pc[b,idx[b,n,k],:]        channels-last neighbour gather
 * Replaces Building_block.gather_neighbour (models/RandLA/RandLANet.py:225-234).
 *   pc [B,S,D] f32, idx [B,N,K] -> out [B,N,K,D] f32
 */
int ffb6d_gather_neighbour_fwd(const float *pc, const void *idx, int idx_is_i64,
                               int64_t B, int64_t S, int64_t D, int64_t N, int K,
                               float *out, ffb6d_stream_t stream);
int ffb6d_gather_neighbour_bwd(const float *grad_out, const void *idx, int idx_is_i64,
                               int64_t B, int64_t S, int64_t D, int64_t N, int K,
                               float *grad_pc, ffb6d_stream_t stream);

/*
 * Relative position encoding of RandLA's local spatial encoding
 * (models/RandLA/RandLANet.py:216-223):
 *   out[b,n,k,:] = [ ||xyz_n - xyz_j||, xyz_n - xyz_j, xyz_n, xyz_j ],  j = idx[b,n,k]
 *   xyz [B,N,3] f32, idx [B,N,K] -> out [B,N,K,10] f32
 * The norm is sqrt((dx*dx + dy*dy) + dz*dz) with round-to-nearest fp32 ops, the
 * order torch.sum uses for a length-3 reduction.
 */
int ffb6d_relative_pos_encoding_fwd(const float *xyz, const void *idx, int idx_is_i64,
                                    int64_t B, int64_t N, int K,
                                    float *out, ffb6d_stream_t stream);
/* Same values written channel-major, out [B,10,N,K] -- what the reference obtains with
 * .permute((0,3,1,2)).contiguous() before the first LFA conv (RandLANet.py:197-198). */
int ffb6d_relative_pos_encoding_cm_fwd(const float *xyz, const void *idx, int idx_is_i64,
                                       int64_t B, int64_t N, int K,
                                       float *out, ffb6d_stream_t stream);

/* ---- fusion 1x1 MLP (tensor cores) ---------------------------------------- */
/*
 * out[b,co,p] = act( scale[co] * sum_ci W[co,ci] * cat(x1,x2)[b,ci,p] + shift[co] )
 * Replaces torch.cat + pt_utils.Conv2d(kernel_size=(1,1), bn=True) with frozen (eval)
 * BatchNorm statistics (models/pytorch_utils.py:75-129,168-201; built models/ffb6d.py:55-80,
 * 104-129; applied :246-262, 282-298): scale = gamma/sqrt(var+eps), shift = beta - mean*scale.
 * tcgen05 TF32 tensor cores with 3xTF32 operand splitting: agrees with the fp32 path to ~1e-6
 * relative (the 1e-5 contract).  x1 [B,C1,P], x2 [B,C2,P] or NULL (C2 = 0), weight [Co,C1+C2]
 * row-major, out [B,Co,P]; all f32, NCHW (point axis contiguous).
 * act: 0 none, 1 ReLU (the fusion layers), 2 LeakyReLU(negative_slope) (RandLA's pt_utils.Conv2d,
 * models/RandLA/pytorch_utils.py:163-197: conv -> BN(eps 1e-6) -> LeakyReLU(0.2)).
 */
int ffb6d_fusion_mlp_fwd(const float *x1, int64_t C1, const float *x2, int64_t C2,
                         const float *weight, const float *scale, const float *shift,
                         int64_t B, int64_t Co, int64_t P, int act, float negative_slope,
                         float *out, ffb6d_stream_t stream);

/*
 * The same layer with the weights prepared once (inference: weights are constants).
 * ffb6d_fusion_mlp_pack splits weight [Co,Ci] into its TF32 hi/lo parts and lays them out as the
 * kernel's shared-memory tiles (`packed`: device, 16-byte aligned, ffb6d_fusion_mlp_pack_bytes(Co,
 * Ci) bytes); ffb6d_fusion_mlp_fwd_packed then streams those tiles with bulk-async (TMA) copies.
 * ffb6d_fusion_mlp_fwd = pack into a stream-ordered scratch block + fwd_packed.
 */
size_t ffb6d_fusion_mlp_pack_bytes(int64_t Co, int64_t Ci);
int ffb6d_fusion_mlp_pack(const float *weight, int64_t Co, int64_t Ci, void *packed, size_t packed_bytes,
                          ffb6d_stream_t stream);
int ffb6d_fusion_mlp_fwd_packed(const float *x1, int64_t C1, const float *x2, int64_t C2,
                                const void *packed, const float *scale, const float *shift,
                                int64_t B, int64_t Co, int64_t P, int act, float negative_slope,
                                float *out, ffb6d_stream_t stream);

/*
 * The packed layer with the two epilogue extras of the restructured fusion stage (SURVEY.md §8f-3):
 *   out = act( scale * ( W * cat(x1, x2) + addend[b, add_idx[b, p], :] ) + shift )
 * The reference computes rgb' = p2r_fuse(cat(rgb, nearest_interpolation(p2r_pre(p), idx)))
 * (models/ffb6d.py:246-253, 282-289).  The 1x1 conv is linear and the interpolation a pure selection, so
 * W * cat(rgb, y[idx]) = W1 * rgb + (W2 * y)[idx]: the small product Z = W2 * y is computed on the N_{i+1}
 * points (one call with out_layout = FFB6D_LAYOUT_NSC, so that Z is stored [B, NA, Co], a point's channels
 * contiguous), and the big layer runs over K = C_r only and adds Z[idx[p]] in its epilogue -- the
 * interpolated map is never materialised and the layer's FLOPs halve.
 *   addend   [B, NA, Co] f32 channels-last, or NULL;   add_idx [B, P] int32 / int64 (with addend)
 *   out_layout: FFB6D_LAYOUT_NCS -> out [B, Co, P] (NCHW), FFB6D_LAYOUT_NSC -> out [B, P, Co]
 */
int ffb6d_fusion_mlp_fwd_ex(const float *x1, int64_t C1, const float *x2, int64_t C2,
                            const void *packed, const float *scale, const float *shift,
                            int64_t B, int64_t Co, int64_t P, int act, float negative_slope,
                            const float *addend, const void *add_idx, int add_idx_is_i64, int64_t NA,
                            int out_layout, float *out, ffb6d_stream_t stream);

/* ---- training mode of the 1x1 layers (batch-statistics BatchNorm, backward) ---------------------------
 * Reference: pt_utils.Conv2d = conv1x1(bias=False) -> BatchNorm2d -> activation, trained with autograd
 * (models/pytorch_utils.py:75-129; RandLA flavour models/RandLA/pytorch_utils.py:35-111, eps 1e-6,
 * momentum 0.99; train_ycb.py:464-470 runs backward + Adam over them).  The layer is composed of
 *   z = W * cat(x1, x2)                 ffb6d_fusion_mlp_fwd_ex (scale 1, shift 0, act 0), z is kept
 *   y = act(BN_batch(z))                ffb6d_bn_train_fwd   (also updates the running statistics)
 * and backwards
 *   dz, dgamma, dbeta from dy           ffb6d_bn_train_bwd
 *   dW = sum_b dz_b * X_b^T             ffb6d_fusion_mlp_wgrad (tcgen05, split-K, fp32 atomics into dW)
 *   dX = W^T * dz                       ffb6d_fusion_mlp_fwd_ex with the packed transposed weight
 * stats [C][4] f32 = (mean, 1/sqrt(var+eps), gamma/sqrt(var+eps), beta) per channel, written by the forward
 * and read by the backward; workspace: ffb6d_bn_workspace_bytes(C, P) bytes of device memory.
 * act: 0 none, 1 ReLU, 2 LeakyReLU(negative_slope).  gamma / beta / running_* may be NULL. */
size_t ffb6d_bn_workspace_bytes(int64_t C, int64_t P);
int ffb6d_bn_train_fwd(const float *z, int64_t B, int64_t C, int64_t P, const float *gamma, const float *beta,
                       float eps, float momentum, float *running_mean, float *running_var,
                       int act, float negative_slope, float *stats, float *y,
                       void *workspace, size_t workspace_bytes, ffb6d_stream_t stream);
int ffb6d_bn_train_bwd(const float *z, const float *grad_y, const float *stats, int64_t B, int64_t C, int64_t P,
                       int act, float negative_slope, float *grad_gamma, float *grad_beta, float *grad_z,
                       void *workspace, size_t workspace_bytes, ffb6d_stream_t stream);
/* The same two passes split at their per-channel reductions, for synchronised BatchNorm across ranks
 * (the reference converts every BatchNorm to SyncBN before DDP, train_ycb.py:568; torch.nn.SyncBatchNorm
 * semantics).  Per layer and step:
 *   ffb6d_bn_train_stats      sums [C][2] f64 = local (sum z, sum z^2)        -> all-reduce sums, and the counts
 *   ffb6d_bn_train_apply      stats, y, running statistics from the global sums over count elements
 *   ffb6d_bn_train_bwd_stats  sums [C][2] f64 = local (sum g', sum g' * xhat) -> all-reduce sums
 *   ffb6d_bn_train_bwd_apply  grad_z from the global sums over the same count
 * count is the global element count sum over ranks of B_r * P, >= the local B * P (every rank needs >= 1
 * frame).  running_var takes the unbiased variance with the global count.  grad_gamma / grad_beta (may be
 * NULL) are the LOCAL sums, as torch.nn.SyncBatchNorm returns them; DDP's gradient all-reduce averages them
 * with every other parameter gradient.  The sums are added in the order of ffb6d_bn_train_fwd / _bwd and
 * rounded as they are, so with the sums of one rank and count = B * P the split passes reproduce
 * ffb6d_bn_train_fwd / ffb6d_bn_train_bwd bit for bit.  stats and workspace as above; sums 8-byte aligned. */
int ffb6d_bn_train_stats(const float *z, int64_t B, int64_t C, int64_t P, double *sums,
                         void *workspace, size_t workspace_bytes, ffb6d_stream_t stream);
int ffb6d_bn_train_apply(const float *z, int64_t B, int64_t C, int64_t P, const double *sums, double count,
                         const float *gamma, const float *beta, float eps, float momentum,
                         float *running_mean, float *running_var, int act, float negative_slope,
                         float *stats, float *y, ffb6d_stream_t stream);
int ffb6d_bn_train_bwd_stats(const float *z, const float *grad_y, const float *stats, int64_t B, int64_t C,
                             int64_t P, int act, float negative_slope, double *sums, float *grad_gamma,
                             float *grad_beta, void *workspace, size_t workspace_bytes, ffb6d_stream_t stream);
int ffb6d_bn_train_bwd_apply(const float *z, const float *grad_y, const float *stats, const double *sums,
                             double count, int64_t B, int64_t C, int64_t P, int act, float negative_slope,
                             float *grad_z, ffb6d_stream_t stream);
/* grad_z = grad_y * act'(z) for a layer with an activation but no BatchNorm. */
int ffb6d_act_bwd(const float *z, const float *grad_y, int64_t n, int act, float negative_slope, float *grad_z,
                  ffb6d_stream_t stream);
/* grad_w [Co, C1+C2] = sum over frames of grad_z [B,Co,P] * cat(x1, x2)^T; grad_w is overwritten. */
int ffb6d_fusion_mlp_wgrad(const float *grad_z, const float *x1, int64_t C1, const float *x2, int64_t C2,
                           int64_t B, int64_t Co, int64_t P, float *grad_w, ffb6d_stream_t stream);

/*
 * Attentive pooling core of RandLA's Att_pooling (models/RandLA/RandLANet.py:243-248):
 *   out[b,c,n] = sum_k f[b,c,n,k] * softmax_k(att[b,c,n,:])[k],   f = cat(f1, f2) along channels
 *   f1 [B,C1,N,K], f2 [B,C2,N,K] or NULL, att [B,C1+C2,N,K] -> out [B,C1+C2,N]   (f32, K <= 64)
 * (the scores `att` come from the layer's fc = 1x1 conv, i.e. ffb6d_fusion_mlp_fwd with act 0).
 */
int ffb6d_att_pool_fwd(const float *f1, int64_t C1, const float *f2, int64_t C2, const float *att,
                       int64_t B, int64_t N, int K, float *out, ffb6d_stream_t stream);
/* Backward of the above: grad_f[k] = g * s[k], grad_att[k] = s[k] * g * (f[k] - out), s = softmax_k(att).
 * grad_f1 [B,C1,N,K], grad_f2 [B,C2,N,K] (NULL iff C2 == 0), grad_att [B,C1+C2,N,K]; grad_out [B,C1+C2,N,1]. */
int ffb6d_att_pool_bwd(const float *f1, int64_t C1, const float *f2, int64_t C2, const float *att,
                       const float *grad_out, int64_t B, int64_t N, int K,
                       float *grad_f1, float *grad_f2, float *grad_att, ffb6d_stream_t stream);

/*
 * One fused kernel per attentive pooling of RandLA's local feature aggregation (inference, BatchNorm folded):
 *   f_xyz = mlp1(relative_pos_encoding(xyz, idx)) [-> mlp2]          (models/RandLA/RandLANet.py:197-199, 207, 216-223)
 *   f_cat = cat(gather_neighbour(feature, idx), f_xyz)                (:200-205, 208-212)
 *   out   = mlp(sum_K f_cat * softmax_K(fc(f_cat)))                   (:243-250)
 * A warp owns a point; nothing of size N*K is written to memory.
 *   xyz [B,N,3]; idx [B,N,16]; feature [B,Dh,N] (Dh = d/2 in {16, 32, 64}); w_x1 [Dh,10], w_x2 [Dh,Dh] or NULL
 *   (NULL: first pooling of a Building_block), w_fc [2Dh,2Dh], w_out [Do,2Dh] (Do <= 2Dh); scale_* / shift_*: the
 *   folded BatchNorm of mlp1 / mlp2 / the output mlp; LeakyReLU(negative_slope) after each of them.
 *   out [B,Do,N] f32.
 */
int ffb6d_lfa_att_pool_fused(const float *xyz, const void *idx, int idx_is_i64, const float *feature,
                             const float *w_x1, const float *scale_x1, const float *shift_x1,
                             const float *w_x2, const float *scale_x2, const float *shift_x2,
                             const float *w_fc, const float *w_out, const float *scale_out, const float *shift_out,
                             int64_t B, int64_t N, int K, int64_t Dh, int64_t Do, float negative_slope,
                             float *out, ffb6d_stream_t stream);

/* ---- depth map -> searched point sets ------------------------------------- */
/*
 * Back-projection of the depth image and extraction of the four point sets the fusion
 * schedule searches, replacing dpt_2_pcld + the `choose` sampling + the stride pyramids of the
 * datasets (datasets/ycb/ycb_dataset.py:165-176, 237, 253-267).  float64 arithmetic like numpy's,
 * rounded once to float32: bit-identical to the reference's arrays.
 *   depth [B,H,W] f32 metres (0 = hole), intrinsics (fx, fy, cx, cy) as float64: 4 values shared
 *   by the batch (intrinsics_per_frame = 0) or [B,4]; choose [B,N] int32 flat pixel indices
 *   -> cld [B,N,3]; pyr2 [B,(H/2)*(W/2),3]; pyr4; pyr8   (f32; holes are signed zeros)
 */
int ffb6d_backproject(const float *depth, int64_t B, int64_t H, int64_t W,
                      const double *intrinsics, int intrinsics_per_frame,
                      const int *choose, int64_t N,
                      float *cld, float *pyr2, float *pyr4, float *pyr8, ffb6d_stream_t stream);

/*
 * Valid-pixel compaction + seeded point sampling on the device: replaces the reference's CPU recipe
 * (datasets/ycb/ycb_dataset.py:218-235: `nonzero()` of the depth mask, a random subset of N valid pixels --
 * or all of them repeated cyclically ('wrap') when fewer exist --, then a random permutation).
 *   depth [B,H,W] f32 (valid where > min_depth) -> choose [B,N] int32 flat pixel indices, the `choose`
 *   input of ffb6d_backproject; valid_count [B] int32 (device, may be NULL) = number of valid pixels.
 * Deterministic per (seed, frame index).  Same distribution as the reference (uniform subset, uniform order);
 * numpy's own random stream is not reproduced.  workspace: ffb6d_sample_pixels_workspace_bytes(B,H,W) bytes.
 */
size_t ffb6d_sample_pixels_workspace_bytes(int64_t B, int64_t H, int64_t W);
int ffb6d_sample_pixels(const float *depth, int64_t B, int64_t H, int64_t W, float min_depth, int64_t N,
                        uint64_t seed, int *choose, int *valid_count, void *workspace, size_t workspace_bytes,
                        ffb6d_stream_t stream);

/* ---- keypoint voting and pose fitting (the step after the network) -------- */
/*
 * Gaussian mean shift of G independent vote sets, replacing MeanShiftTorch.fit
 * (ffb6d/utils/meanshift_pytorch.py:28-57) as cal_frame_poses / cal_frame_poses_lm call it once per keypoint
 * and once for the centre (ffb6d/utils/pvn3d_eval_utils_kpls.py:89-90, 124-137, 245-258).  One persistent
 * kernel runs all G sets to convergence (max shift < bandwidth * 1e-3, or max_iter + 1 rounds, :30-47) without
 * the N x N matrices and without a host round trip per iteration.
 *   votes [G,N,3] f32; valid: u8 mask of the points that vote (the reference's votes[mask]), [N] shared by the
 *   sets (valid_stride = 0), one row per set (valid_stride >= N elements between rows), or NULL (all vote)
 *   -> centres [G,3] f32: the mode with the most modes within one bandwidth (lowest index on ties);
 *      labels [G,N] u8: 1 where a point's mode lies within one bandwidth of it (0 for non-voting points);
 *      iters [G] i32: rounds run; modes [G,N,3] f32 or NULL: every point's converged position
 *      (`ret_mid_res=True`; rows of non-voting points are 0).
 * A set without voting points gets centre (0,0,0) and 0 rounds.  Floating point: the sums run in another order
 * than torch's, agreement is to about the stop threshold (tests/test_gpu_pose.py), not bitwise.
 * G <= 64.  workspace: ffb6d_mean_shift_workspace_bytes(G, N) bytes.
 */
size_t ffb6d_mean_shift_workspace_bytes(int64_t G, int64_t N);
int ffb6d_mean_shift_fit(const float *votes, const unsigned char *valid, int64_t valid_stride, int64_t G, int64_t N,
                         float bandwidth, int max_iter, float *centres, unsigned char *labels, int *iters,
                         float *modes, void *workspace, size_t workspace_bytes, ffb6d_stream_t stream);

/*
 * Least-squares rigid transform mapping point set A onto B (Kabsch / SVD), replacing best_fit_transform
 * (ffb6d/utils/pvn3d_eval_utils_kpls.py:28-59), batched over G objects; float64 arithmetic like numpy's.
 *   A, B [G,M,3] f32 (mesh keypoints, voted keypoints) -> T [G,3,4] f64 = [R | t], det R = +1.
 */
int ffb6d_best_fit_transform(const float *A, const float *B, int64_t G, int64_t M, double *T, ffb6d_stream_t stream);

/* ---- grid subsampling --------------------------------------------------- */
/*
 * Voxel-grid barycentre subsampling, replaces grid_subsampling()
 * (GS/cpp_subsampling/grid_subsampling/grid_subsampling.cpp:5-106) behind
 * DataProcessing.grid_sub_sampling (models/RandLA/helper_tool.py:199-219).
 * HOST pointers (the reference op is numpy-in / numpy-out).
 *   points [N,3] f32, features [N,fdim] f32 or NULL, classes [N,ldim] i32 or NULL
 *   -> sub_points [M,3], sub_features [M,fdim], sub_classes [M,ldim]; outputs must
 *      have room for N rows; *M_out receives M.
 * Rows are emitted by ascending voxel key (the reference's order is that of a
 * libstdc++ unordered_map and is unspecified).  Per-voxel sums are accumulated in
 * input order, so barycentres and mean features are bitwise equal to the
 * reference; among labels tied for the maximal count the smallest is chosen.
 */
int ffb6d_grid_subsample_host(const float *points, size_t N,
                              const float *features, size_t fdim,
                              const int *classes, size_t ldim,
                              float sampleDl,
                              float *sub_points, float *sub_features, int *sub_classes,
                              size_t *M_out);

#ifdef __cplusplus
}
#endif
#endif /* FFB6D_B200_H_ */
