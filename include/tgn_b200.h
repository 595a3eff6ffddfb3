/*
 * tgn_b200.h -- C ABI of libtgn_b200.so: the B200-native (sm_100a) replacement for the native
 * layer of limhoyeon/ToothGroupNetwork's point-cloud operator hot path.
 *
 * Boundary being replaced (paths relative to /root/reference/external_libs/pointops/src):
 * the reference exposes its kernels to the pybind glue through ten `extern "C"` launchers
 * taking raw device pointers.  Part 1 below exports those ten symbols with identical
 * signatures and semantics (legacy default stream, void return, caller-owned outputs), so
 * the reference's `*_cuda.cpp` glue links against this library unchanged.  Part 2 is the
 * same operations with an explicit stream and a status code, plus the operations the
 * reference runs as PyTorch tensor code on the pointnet2 side (ball query, 3-NN, gather,
 * grouped shared-MLP set abstraction), which this library provides as fused kernels.
 *
 * Conventions: all pointers are DEVICE pointers unless stated otherwise; float = fp32,
 * int = int32; tensors are dense row-major; `stream` is a cudaStream_t passed as void*.
 * Part-2 functions return 0 on success, TGN_ERR_* otherwise (text in tgn_last_error()).
 * No function synchronises the device.  There is no CPU path.
 */
#ifndef TGN_B200_H_
#define TGN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ===================================================================================
 * Part 1 -- drop-in for the reference's extern "C" launchers.
 * =================================================================================== */

/* sampling/sampling_cuda_kernel.h:14 (definition sampling_cuda_kernel.cu:131-171).
 * b clouds packed in xyz (n_total,3) with cumulative ends offset[b]; new_offset[b] cumulative
 * sample counts; n = largest cloud size (selects the reference's block size and therefore its
 * tie-break); tmp (n_total) pre-filled by the caller (1e10), holds the running minima on
 * return; idx (m_total) receives global row ids, first sample of a cloud = its first point. */
void furthestsampling_cuda_launcher(int b, int n, const float *xyz, const int *offset,
                                    const int *new_offset, float *tmp, int *idx);

/* knnquery/knnquery_cuda_kernel.h:14 (definition knnquery_cuda_kernel.cu:111-116).
 * idx (m,nsample), dist2 (m,nsample) = squared distances, ascending; a segment with fewer
 * than nsample points leaves (segment start, 1e10) in the trailing slots. */
void knnquery_cuda_launcher(int m, int nsample, const float *xyz, const float *new_xyz,
                            const int *offset, const int *new_offset, int *idx, float *dist2);

/* grouping/grouping_cuda_kernel.h:13-14 (grouping_cuda_kernel.cu:27-41) */
void grouping_forward_cuda_launcher(int m, int nsample, int c, const float *input, const int *idx, float *output);
void grouping_backward_cuda_launcher(int m, int nsample, int c, const float *grad_output, const int *idx, float *grad_input);

/* interpolation/interpolation_cuda_kernel.h:13-14 (interpolation_cuda_kernel.cu:35-47);
 * output / grad_input are accumulated into and must be pre-zeroed by the caller. */
void interpolation_forward_cuda_launcher(int n, int c, int k, const float *input, const int *idx, const float *weight, float *output);
void interpolation_backward_cuda_launcher(int n, int c, int k, const float *grad_output, const int *idx, const float *weight, float *grad_input);

/* subtraction/subtraction_cuda_kernel.h:13-14 (subtraction_cuda_kernel.cu:32-44) */
void subtraction_forward_cuda_launcher(int n, int nsample, int c, const float *input1, const float *input2, const int *idx, float *output);
void subtraction_backward_cuda_launcher(int n, int nsample, int c, const int *idx, const float *grad_output, float *grad_input1, float *grad_input2);

/* aggregation/aggregation_cuda_kernel.h:12-17 (aggregation_cuda_kernel.cu:41-53) */
void aggregation_forward_cuda_launcher(int n, int nsample, int c, int w_c, const float *input, const float *position,
                                       const float *weight, const int *idx, float *output);
void aggregation_backward_cuda_launcher(int n, int nsample, int c, int w_c, const float *input, const float *position,
                                        const float *weight, const int *idx, const float *grad_output,
                                        float *grad_input, float *grad_position, float *grad_weight);

/* ===================================================================================
 * Part 2 -- stream-taking, status-returning entry points.
 * =================================================================================== */
#define TGN_OK 0
#define TGN_ERR_INVALID 1
#define TGN_ERR_CUDA 2

int tgn_version(void);
const char *tgn_last_error(void);          /* thread-local, valid until the next failing call */
int tgn_launch_count(void);                /* kernels launched by this library in this process */

/* FPS.  Same contract as furthestsampling_cuda_launcher; tmp may be NULL (running minima start
 * at 1e10 and are not written back) when the cloud fits the register-resident kernel.
 * `mode`: 0 = choose by b and n_max: clouds of more than 4096 points go to the bucket-pruned kernel
 *         (Morton-sorted 64-point buckets, exact; 16, 8 or 4 warps per cloud as the batch grows),
 *         smaller ones stay register-resident in one CTA / cluster;
 *         -1 = streaming kernel (needs tmp); -2 = bucket kernel, shape by batch size;
 *         -(10 + W) = bucket kernel with W in {16, 8, 4, 2, 1} warps per cloud;
 *         100*G + CS = register-resident cluster of CS CTAs (1,2,4,8) with G clouds in flight
 *         (1 or 2; G omitted = 1).  Every mode returns the same indices. */
int tgn_furthestsampling(int b, int n_max, const float *xyz, const int *offset, const int *new_offset,
                         float *tmp, int *idx, int mode, void *stream);

/* kNN.  b = number of segments (length of offset / new_offset). */
int tgn_knnquery(int b, int m, int nsample, const float *xyz, const float *new_xyz, const int *offset,
                 const int *new_offset, int *idx, float *dist2, void *stream);

/* Crop extraction: the k (<= 4096) nearest points of each of Q centres per cloud, ascending (float64 distance, index) --
 * replaces ops_utils.get_nearest_neighbor_idx (sklearn KDTree.query(k=3072) on the host, ops_utils.py:146-161).
 * xyz (B,N,3), centres (B,Q,3) -> out_idx (B,Q,k) int32, or int64 when idx64 != 0.  One CTA per centre: radix select of
 * the k-th distance, compaction, bitonic sort. */
int tgn_crop_knn(int B, int N, int Q, int k, const float *xyz, const float *centres, void *out_idx, int idx64, void *stream);

/* DBSCAN labels equal to scikit-learn's DBSCAN(eps, min_samples).fit(xyz).labels_ (float64 reduced-distance predicate, clusters
 * numbered by their smallest core index, border points take the smallest neighbouring label, noise -1): replaces the host-side
 * clustering of ops_utils.get_clustering_labels (ops_utils.py:98).  xyz (n,3) float32 DEVICE; workspace of
 * tgn_dbscan_bytes(n) DEVICE bytes; labels (n) int32, core (n) bytes (1 = core sample), n_clusters DEVICE int or NULL. */
size_t tgn_dbscan_bytes(int n);
int tgn_dbscan(int n, const float *xyz, double eps, int min_samples, void *workspace, int *labels, unsigned char *core, int *n_clusters,
               void *stream);

/* kNN through a per-segment uniform grid: identical answers to tgn_knnquery (distinct distances: order-independent;
 * ties among the k+1 best: the query is re-run with the reference's index-order heap), ~100x fewer distance evaluations
 * on 24k-point clouds.  The grid depends only on (xyz, offset): build it once into a caller-owned DEVICE workspace of
 * tgn_knn_grid_bytes(b, n_total) bytes and reuse it for every query set / k against that point set. */
size_t tgn_knn_grid_bytes(int b, int n_total);
int tgn_knn_grid_build(int b, int n_total, const float *xyz, const int *offset, void *workspace, void *stream);
int tgn_knn_grid_query(int b, int n_total, int m, int nsample, const float *xyz, const float *new_xyz, const int *offset,
                       const int *new_offset, const void *workspace, int *idx, float *dist2, void *stream);

/* Exact float64 kNN with scikit-learn KDTree semantics: replaces the host KDTree searches of the tgnet boundary stage
 * (inference_pipeline_tgn.py:289-330, :107-140).  points (n,3) and queries (m,3) float64 DEVICE; for every query the k <= 64
 * (and k <= n) nearest points in ascending (rdist, index) order, rdist = (dx*dx + dy*dy) + dz*dz in float64 without FMA
 * contraction; exact ties come out lower index first.  Build once per point set into a caller-owned DEVICE workspace of
 * tgn_knn_f64_bytes(n) bytes (it holds the grid of tgn_knn_grid_build plus a float64 copy of the points in cell order) and
 * reuse it for every query set and k.  Outputs, each optional (NULL = not written): idx (m,k) int64, dist (m,k) float64 =
 * sqrt(rdist) correctly rounded.  With labels (n) float64 the query also writes nearest_label (m) = labels[idx[:,0]],
 * is_boundary (m) bytes = (count / k < ratio) with count the neighbours whose label equals nearest_label, and the number
 * of boundary queries to the DEVICE int n_boundary (zeroed by the call); no (m,k) matrix is needed for that. */
size_t tgn_knn_f64_bytes(int n);
int tgn_knn_f64_build(int n, const double *points, void *workspace, void *stream);
int tgn_knn_f64_query(int n, int m, int k, const double *queries, const void *workspace, int64_t *idx, double *dist,
                      const double *labels, double ratio, double *nearest_label, unsigned char *is_boundary, int *n_boundary,
                      void *stream);

int tgn_grouping_forward(int m, int nsample, int c, const float *input, const int *idx, float *output, void *stream);
int tgn_grouping_backward(int m, int nsample, int c, const float *grad_output, const int *idx, float *grad_input, void *stream);
int tgn_interpolation_forward(int n, int c, int k, const float *input, const int *idx, const float *weight, float *output, void *stream);
int tgn_interpolation_backward(int n, int c, int k, const float *grad_output, const int *idx, const float *weight, float *grad_input, void *stream);
/* output[n,:] += sum_i input[idx[n,i],:] * weight[n,i].  fused = 1: the FMA chain of interpolation_cuda_kernel.cu:5-18
 * (== tgn_interpolation_forward); fused = 0: product rounded, then added -- the arithmetic of the torch loop in
 * pointops.interpolation (pointops.py:177-179), which is what the models call. */
int tgn_weighted_gather(int n, int c, int k, const float *input, const int *idx, const float *weight, float *output, int fused, void *stream);
/* Deterministic, ORDER-EXACT scatter-add backwards.  The reference's live callers gather with torch advanced indexing,
 * whose backward (index_put_ accumulate) adds every destination row's contributions sequentially in ascending source
 * position.  tgn_csr_build inverts an index tensor once (keys[M] -> per destination row the ascending list of source
 * positions) into a DEVICE workspace of tgn_csr_bytes(M, n_rows); the two backwards below then reproduce torch's sums
 * bit for bit, without value atomics.
 *   tgn_gather_backward_det:           grad_in[r,:] = sum_{p : keys[p]=r, ascending} grad_out[p,:]      (grad_out (M,c))
 *   tgn_weighted_gather_backward_det:  keys = idx (n,k) flattened; grad_out (n,c), weight (n,k):
 *        per i: G_i[r,:] = sum_{n ascending, idx[n,i]=r} grad_out[n,:]*weight[n,i];  grad_in = ((G_{k-1}+G_{k-2})+...)+G_0
 *        -- the order in which autograd sums the k index_put results of pointops.interpolation (pointops.py:177-179);
 *        single != 0: one accumulation over all (n,i) in ascending n*k+i -- the backward of pointnet2_utils.py:340. */
size_t tgn_csr_bytes(long long M, int n_rows);
int tgn_csr_build(long long M, int n_rows, const int *keys, void *workspace, void *stream);
int tgn_gather_backward_det(long long M, int n_rows, int c, const void *workspace, const float *grad_out, float *grad_in, void *stream);
int tgn_weighted_gather_backward_det(long long M, int n_rows, int c, int k, int single, const void *workspace, const float *grad_out,
                                     const float *weight, float *grad_in, void *stream);

int tgn_subtraction_forward(int n, int nsample, int c, const float *input1, const float *input2, const int *idx, float *output, void *stream);
int tgn_subtraction_backward(int n, int nsample, int c, const int *idx, const float *grad_output, float *grad_input1, float *grad_input2, void *stream);
int tgn_aggregation_forward(int n, int nsample, int c, int w_c, const float *input, const float *position, const float *weight,
                            const int *idx, float *output, void *stream);
int tgn_aggregation_backward(int n, int nsample, int c, int w_c, const float *input, const float *position, const float *weight,
                             const int *idx, const float *grad_output, float *grad_input, float *grad_position,
                             float *grad_weight, void *stream);

/* Ball query: pointnet2_utils.query_ball_point (external_libs/pointnet2_utils/pointnet2_utils.py:120-144).
 * xyz (B,N,3), new_xyz (B,S,3) -> group_idx (B,S,nsample): the first nsample point indices in
 * ascending order whose EXPANDED squared distance (-2ab + |a|^2 + |b|^2, evaluated in the
 * reference's rounding order) is not > r2, padded with the first hit; N in every slot when the
 * ball is empty.  r2 must be float32(radius**2).  idx64 is a bit set: bit 0 writes int64 (the
 * reference's dtype) instead of int32; by default clouds of >= 8192 points whose balls are sparse
 * are answered by a uniform-grid kernel and the rest by an index-order tile scan (same result);
 * bit 2 (4) forces the tile scan, bit 3 (8) the grid, bit 1 (2) a streaming scan (experiments).
 * Bits 4 (16) / 5 (32): |new_xyz|^2 / |xyz|^2 rounded as (x*x + z*z) + y*y instead of (x*x + y*y) + z*z --
 * torch.sum(p ** 2, -1) on CUDA takes the first form for a contiguous (..., 3) operand and the second for a strided
 * view (and always on the CPU); the Python layer sets the bits from the layout the reference's call would see. */
int tgn_ball_query(int B, int N, int S, float r2, int nsample, const float *xyz, const float *new_xyz,
                   void *group_idx, int idx64, void *stream);

/* 3 nearest coarse points by the same expanded distance (pointnet2_utils.py:333-335):
 * xyz1 (B,N,3) fine, xyz2 (B,S,3) coarse, S >= 3 -> dist (B,N,3) ascending, idx (B,N,3) int32. */
int tgn_three_nn(int B, int N, int S, const float *xyz1, const float *xyz2, float *dist, int *idx, void *stream);
/* Same with `order`: bit 0 / bit 1 = |xyz1|^2 / |xyz2|^2 in the contiguous-reduce rounding (see tgn_ball_query). */
int tgn_three_nn_ex(int B, int N, int S, const float *xyz1, const float *xyz2, float *dist, int *idx, int order, void *stream);

/* The matrix itself (pointnet2_utils.square_distance :20-41): src (B,N,3), dst (B,M,3) -> out (B,N,M), expanded form, `order` as in
 * tgn_three_nn_ex (bit 0: src, bit 1: dst).  Forward only; the Python wrapper keeps torch's formulation under autograd. */
int tgn_square_distance(int B, int N, int M, const float *src, const float *dst, float *out, int order, void *stream);

/* Weighted 3-point interpolation (pointnet2_utils.py:337-340): weights 1/(dist+1e-8) normalised,
 * points2 (B,S,C) point-major -> out (B,N,C). */
int tgn_three_interpolate(int B, int N, int S, int C, const float *points2, const float *dist, const int *idx,
                          float *out, void *stream);
/* norm_alt != 0: the normaliser is summed as (r0 + r2) + r1, torch's CUDA reduce order for the contiguous (B,N,3)
 * reciprocal tensor; 0: (r0 + r1) + r2, the CPU order. */
int tgn_three_interpolate_ex(int B, int N, int S, int C, const float *points2, const float *dist, const int *idx,
                             float *out, int norm_alt, void *stream);

/* Batched row gather: pointnet2_utils.index_points (pointnet2_utils.py:44-61).
 * points (B,N,C), idx (B,M) int32 -> out (B,M,C). */
int tgn_gather_rows(int B, int N, int M, int C, const float *points, const int *idx, float *out, void *stream);

/* (B,C,N) -> (B,N,C) and back (the reference permutes with torch; here one tiled kernel). */
int tgn_transpose_cn(int B, int C, int N, const float *in, float *out, void *stream);

/* Fused set-abstraction body: gather -> [xyz_rel | feats] -> L x (1x1 conv + bias + ReLU) -> max
 * over the K neighbours, without materialising the grouped tensor
 * (PointNetSetAbstraction.forward pointnet2_utils.py:213-239 / Msg :261-299, eval-mode BatchNorm
 * folded into weight/bias by the caller).
 *   xyz (B,N,3); feats (B,N,D) point-major or NULL (D = 0); new_xyz (B,S,3); group_idx (B,S,K) int32
 *   xyz_first: 1 -> channels [xyz_rel, feats] (SSG, :169), 0 -> [feats, xyz_rel] (MSG, :285)
 *   n_layers in [1,4]; channels[n_layers+1] HOST array, channels[0] = 3 + D; every width <= 128
 *   weights[l] (C_{l+1}, C_l) row-major DEVICE, biases[l] (C_{l+1}) DEVICE; the two pointer arrays are HOST arrays
 *   out: channel-first (B, out_c_total, S); this branch writes channels [out_c_offset, +C_last)
 *   engine: 0 = auto (2 when the shape fits it, else 3, else 1), 1 = fp32 CUDA-core kernel (exact FMA),
 *           2 = tcgen05 3xTF32 kernel (widths <= 64, ~2^-21), 3 = tcgen05 kernel for wide layers (first layer
 *           3xTF32, later layers as three bf16x2-split MMAs, ~1e-5; at least two layers, K in {16,32,64,128}). */
int tgn_sa_group_mlp_max(int B, int N, int S, int K, int D, const float *xyz, const float *feats, const float *new_xyz,
                         const int *group_idx, int xyz_first, int n_layers, const int *channels,
                         const float *const *weights, const float *const *biases, float *out, int out_c_total,
                         int out_c_offset, int engine, void *stream);

/* ---------------------------------------------------------------------------------------------------
 * 1x1-convolution chains with BATCH-STATISTICS BatchNorm (any width), one launch per layer
 * (PointNetSetAbstraction(Msg).forward pointnet2_utils.py:232-237 / :289-294 and
 * PointNetFeaturePropagation.forward :346-352 with BatchNorm in training mode -- which is how every
 * reference call site, inference included, runs them -- and in eval mode for widths the single-kernel
 * engines above do not take).  Layer l computes the RAW pre-activation, channel-major:
 *      y[c, r] = sum_k W[c, k] * act(x)[r, k] + bias[c],   r in [0, rows)
 * where act() is the previous layer's BatchNorm + ReLU applied while the operand is built
 * (in_affine: 0 none, 1 from the fp64 batch sums `in_stats` = {sum[cin], sumsq[cin]} over `rows` rows,
 * 2 from running statistics).  tcgen05, operands split into three bf16 parts (six MMAs per K step, fp32-grade:
 * batch-statistics BatchNorm amplifies rounding differences) or two (`precision` = 2: three MMAs, ~1e-5).
 * mode 0: the operand row r = (b, n), b = r / rows_per_batch, is read from up to two strided segments,
 *         x[k] = seg_ptr[i][b*seg_batch_stride[i] + n*seg_row_stride[i] + k'*seg_chan_stride[i]] (strides in floats);
 * mode 1: neighbourhood gather, r = ((b*S + s)*K + j): [feats[b, gidx[r], :] | xyz[b, gidx[r]] - new_xyz[b, s]]
 *         (xyz_first = 0, MSG order :285) or [xyz - centre | feats] (xyz_first = 1, SSG order :169); cin = D + 3.
 * Outputs, each optional: y (cout, rows); stats (2*cout doubles, ACCUMULATED: caller zeroes) = per-channel
 * sum / sum of squares of y; ymax / ymin (cout, rows/group) = extrema over groups of `group` consecutive rows
 * (the max over the K neighbours must wait for the BatchNorm scale's sign, so both are kept); with
 * extrema_atomic != 0 they are merged with atomics into buffers the caller pre-filled with -inf / +inf
 * (required when 128 % group != 0).  w_packed: tgn_pw_pack_weights of the (cout, cin) weight.
 * in_update_running != 0 with in_affine == 1 applies torch's momentum update to in_running_mean / _var once. */
typedef struct {
    int rows, rows_per_batch, cin, cout;
    int mode;
    const float *seg_ptr[2];
    int seg_channels[2];
    long long seg_batch_stride[2], seg_row_stride[2], seg_chan_stride[2];
    const float *xyz, *feats, *new_xyz;
    const int *gidx;
    int N, S, K, D, xyz_first;
    int in_affine, in_update_running;
    const double *in_stats;
    const float *in_gamma, *in_beta;
    float *in_running_mean, *in_running_var;
    float in_eps, in_momentum;
    const void *w_packed;
    const float *bias;
    float *y;
    double *stats;
    float *ymax, *ymin;
    int group, extrema_atomic;
    int precision;          /* 0 / 3: three bf16 parts per operand, six MMAs per K step (fp32-grade); 2: two parts, three MMAs (~1e-5) */
} tgn_pw_layer_t;

/* Final BatchNorm (+ ReLU) of a chain into a channel-first tensor:
 *   out[b, out_c_offset + c, n] = relu?(scale_c * v + shift_c),  v = src[c, b*rows_per_batch + n]
 * or, when ymin != NULL, v = (scale_c >= 0 ? src : ymin)[c, ...] (src = the max).  `affine` as in_affine above
 * (0 = identity), statistics over stat_rows rows. */
typedef struct {
    int rows, rows_per_batch, channels, out_channels, out_c_offset, relu;
    const float *src, *ymin;
    float *out;
    int affine, update_running;
    const double *stats;
    long long stat_rows;
    const float *gamma, *beta;
    float *running_mean, *running_var;
    float eps, momentum;
} tgn_pw_apply_t;

/* Fused forward of blocks.PointTransformerLayer (models/modules/cbl_point_transformer/blocks.py:14-44; SURVEY 8(f)-3): vector
 * self-attention over the K neighbours idx[i, :] of every point, share_planes = 8, in up to four passes over the gathers (one per
 * BatchNorm that runs on batch statistics + the output pass); nothing of size (n, K, c) is materialised.
 *   p (n,3); xq, xk, xv (n,c) = linear_q/k/v(x) (left to the caller's GEMMs); idx (n,K) int32 (kNN of p in p); out (n,c)
 *   linear_p = Linear(3,3) [p_w0 (3,3), p_b0] -> BatchNorm1d(3) [p_*] -> ReLU -> Linear(3,c) [p_w1 (c,3), p_b1]
 *   linear_w = BatchNorm1d(c) [a_gamma..] -> ReLU -> Linear(c, c/8) [a_w (c/8,c), a_b] -> BatchNorm1d(c/8) [b_gamma..] -> ReLU
 *              -> Linear(c/8, c/8) [b_w, b_b]
 *   bn_mode[i]: 1 = batch statistics (stats_* = zeroed fp64 {sum[ch], sumsq[ch]} scratch, filled by the passes), 2 = running
 *   statistics; update_running != 0 applies torch's momentum update to the *_rmean / *_rvar of the BatchNorms in mode 1.
 * c in {32, 64, 128, 256, 512}, K <= 64. */
typedef struct {
    int n, c, K;
    const float *p, *xq, *xk, *xv;
    const int *idx;
    float *out;
    const float *p_w0, *p_b0, *p_w1, *p_b1;
    const float *p_gamma, *p_beta; float *p_rmean, *p_rvar; float p_eps, p_momentum;
    const float *a_gamma, *a_beta; float *a_rmean, *a_rvar; float a_eps, a_momentum;
    const float *a_w, *a_b;
    const float *b_gamma, *b_beta; float *b_rmean, *b_rvar; float b_eps, b_momentum;
    const float *b_w, *b_b;
    double *stats_p, *stats_a, *stats_b;
    int bn_mode[3];
    int update_running;
} tgn_pt_layer_t;
int tgn_pt_layer_forward(const tgn_pt_layer_t *layer, void *stream);
int tgn_pt_layer_struct_size(void);
/* layers with fewer queries than this run one CTA per query instead of one warp per query (default 1024); returns the old value */
int tgn_pt_layer_set_cta_threshold(int n_queries);

size_t tgn_pw_packed_bytes(int cout, int cin);
int tgn_pw_struct_size(int which);         /* sizeof(tgn_pw_layer_t) (0) / sizeof(tgn_pw_apply_t) (1): binding self-check */
int tgn_pw_pack_weights(int cout, int cin, const float *w, void *packed, void *stream);
int tgn_pw_layer_forward(const tgn_pw_layer_t *layer, void *stream);
int tgn_pw_apply(const tgn_pw_apply_t *p, void *stream);
int tgn_pw_fill(float *ptr, long long n, float value, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TGN_B200_H_ */
