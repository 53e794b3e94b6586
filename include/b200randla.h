/*
 * b200randla.h -- C ABI of libb200randla.so: the B200 (sm_100a) RandLA-Net hot path
 * of IGNF/myria3d, as hand-written CUDA kernels behind plain pointers and sizes.
 *
 * Conventions (SURVEY.md section 8b):
 *   - every pointer is a DEVICE pointer unless named host_*; the caller owns every
 *     buffer (outputs and workspaces are pre-allocated by the caller);
 *   - no allocation, no synchronisation, no global state inside: every entry point
 *     only enqueues kernels on `stream` (a cudaStream_t passed as void*), so calls
 *     are re-entrant, graph-capturable and safe from the autograd engine thread;
 *   - floating tensors are fp32 row-major; neighbour tables are int32 [rows, kt]
 *     with kt the TABLE WIDTH (16 or 32 for the LFA kernels), -1 padded: clouds
 *     smaller than k give min(k, n_cloud) neighbours (torch_cluster semantics);
 *     `ptr` arrays are int64 [B+1] exactly as PyG's Batch.ptr;
 *   - return value 0 = ok; non-zero = error (B200_E_*), message via b200_last_error().
 *     Asynchronous CUDA errors surface at the caller's next synchronisation.
 *
 * Each entry point cites the reference call it replaces (paths relative to the
 * myria3d repository root).
 */
#ifndef B200RANDLA_H_
#define B200RANDLA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_ABI_VERSION 6

#define B200_OK 0
#define B200_E_INVALID 1     /* bad argument (null pointer, unsupported size/alignment) */
#define B200_E_UNSUPPORTED 2 /* valid request this build has no kernel for */
#define B200_E_CUDA 3        /* a CUDA runtime call failed at enqueue time */

int b200_abi_version(void);
/* Thread-local message of the last failing call on this thread ("" if none). */
const char* b200_last_error(void);
/* Number of kernels this library has enqueued since load (all threads). */
int64_t b200_launch_count(void);
/* cudaGetDeviceProperties-based sanity check: 0 iff the current device is sm_100. */
int b200_check_device(void);
/* Process-wide switches (the library reads no environment variables).  Together with the launch counter these are
 * the only mutable global state; compute entry points are otherwise pure functions of their arguments.
 *   "tensor_cores"  1 (default) / 0: A/B switch that routes every tcgen05 kernel to its fp32-FMA counterpart
 *                   (tests and profiles compare the two; no reference counterpart).
 *   "tensor_core_paths"  bitmask (default 31) of the kernel families allowed on the tensor cores while "tensor_cores" is 1:
 *                   1 Linear forward, 2 Linear input gradient, 4 wide weight gradient, 8 narrow weight gradient,
 *                   16 fused LFA forward/backward.  Used to attribute numerical differences to one family.
 *   "tma_rows"      bitmask of the Linear kernels of the 16/32/64-channel layers on >= 8192 rows that run as TMA-fed
 *                   persistent row-streaming kernels (tma_rows.cu; 2-D tensor maps, mbarrier ring): 1 forward,
 *                   2 input gradient, 4 weight gradient (default 7); cleared bits select the register-staged kernels.
 *   "bn_backward_fused"  0 (default) / 1: b200_affine_act_bwd runs reduce + apply of the small levels as ONE launch with a
 *                   grid barrier (measured on a B200: 16.8 us against 8.0 + 5.5 us for the two kernels -- a grid of
 *                   #SMs / 2 CTAs is too small for either phase -- so it is off; kept as an A/B switch).
 *   "knn_points_per_cell"  average occupancy of the bucket grid of b200_knn_grid; 0 (default) = automatic
 *                   (6 for k < 8, 8 for k < 24, 16 above); results do not depend on it (exact search).
 *   "tc_timeline"   device pointer (as integer) to 128 int64 receiving clock64() marks of CTA 0 of the tcgen05 GEMMs
 *                   (scripts/tc_timeline.py); 0 (default) = off.
 * b200_get_option returns the current value, -1 for an unknown key. */
int b200_set_option(const char* key, int64_t value);
int64_t b200_get_option(const char* key);

/* ---------------------------------------------------------------- kNN ------------------
 * Replaces torch_cluster knn()/knn_graph() as called by
 *   knn_graph(pos, k, batch=batch, loop=True)   myria3d/models/modules/pyg_randla_net.py:180
 *   knn_interpolate(..., k=1)                   myria3d/models/modules/pyg_randla_net.py:250
 *   knn_interpolate(..., k=interpolation_k)     myria3d/models/model.py:90
 * For every query y (cloud b = the segment [ptr_y[b], ptr_y[b+1])) the k nearest x of
 * the SAME cloud, ascending by fp32 squared distance ((dx*dx+dy*dy)+dz*dz, no FMA),
 * ties to the lower x index; self is included when x == y.
 *   nbr   int32 [ny, kt]  global x indices, -1 padded beyond min(k, n_cloud) and beyond k
 *   dist2 fp32  [ny, kt]  matching squared distances (+inf padded); may be NULL
 * max_queries_per_cloud bounds the launch grid (host knows ptr).
 */
int b200_knn(const float* pos_x, const int64_t* ptr_x, int64_t nx,
             const float* pos_y, const int64_t* ptr_y, int64_t ny,
             int32_t num_clouds, int64_t max_queries_per_cloud,
             int32_t k, int32_t kt, int32_t* nbr, float* dist2, void* stream);

/* Replaces the same reference calls as b200_knn (knn_graph, pyg_randla_net.py:180; knn inside knn_interpolate,
 * pyg_randla_net.py:250, models/model.py:90).
 * Same contract and bit-identical output as b200_knn, but each query only visits the cells of a per-cloud
 * uniform 2-D bucket grid (over the two widest axes) that can still contain one of its k nearest
 * neighbours: O(n k) instead of O(n^2) distance evaluations.  Needs a caller-owned, 256-byte aligned
 * workspace of b200_knn_grid_workspace_bytes(nx, num_clouds, max_x_per_cloud) bytes (contents are
 * scratch).  max_x_per_cloud / max_y_per_cloud must be the exact maxima of the cloud sizes (or larger).
 */
int64_t b200_knn_grid_workspace_bytes(int64_t nx, int32_t num_clouds, int64_t max_x_per_cloud);
int b200_knn_grid(const float* pos_x, const int64_t* ptr_x, int64_t nx,
                  const float* pos_y, const int64_t* ptr_y, int64_t ny,
                  int32_t num_clouds, int64_t max_x_per_cloud, int64_t max_y_per_cloud,
                  int32_t k, int32_t kt, int32_t* nbr, float* dist2,
                  void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------- LocSE / attentive pooling -----
 * Together these replace LocalFeatureAggregation.propagate()+message()
 * (myria3d/models/modules/pyg_randla_net.py:121-152): gather, relative position
 * encoding, encoder SharedMLP, concat, attention Linear, neighbourhood softmax
 * (torch_geometric.utils.softmax), weighting and the aggr="add" scatter.
 *
 * b200_edge_moments: first and second moments of q = (p_i, p_j, |p_j-p_i|) in R^7 over
 * all valid edges, in fp64: out[0]=edge count, out[1..7]=sum q, out[8..56]=sum q q^T
 * (row-major 7x7).  `out` (57 doubles) must be zeroed by the caller.  With them the
 * train-mode BatchNorm of mlp_encoder (statistics over all E edges, pyg_randla_net.py:117,144)
 * folds into an affine map, so the fused kernels below are single-pass in training too.
 */
int b200_edge_moments(const float* pos, const int32_t* nbr, int64_t n, int32_t kt,
                      double* out, void* stream);

/* Fold mlp_encoder = Linear(10 -> h) + BatchNorm1d(momentum .01, eps 1e-6) (pyg_randla_net.py:117,144)
 * into the affine map of q the fused kernels consume:  enc_w [h,7], enc_b [h].
 *   w fp32 [h,10], b fp32 [h] or NULL, gamma/beta fp32 [h] (BatchNorm affine),
 *   moments fp64 [57] from b200_edge_moments (training) or NULL (eval: running statistics are used).
 * Training also updates running_mean / running_var (unbiased variance) and increments
 * *num_batches_tracked (int64, may be NULL) exactly like torch.nn.BatchNorm1d.
 * The backward returns the exact train-mode gradients through the batch statistics:
 *   grad_w [h,10], grad_b [h] (may be NULL; identically 0 in training), grad_gamma, grad_beta: written when
 *   accumulate == 0, added to (+=) when accumulate != 0 (the buffers are then the parameters' .grad). */
int b200_encoder_fold_fwd(const float* w, const float* b, const float* gamma, const float* beta,
                          const double* moments, float* running_mean, float* running_var,
                          int64_t* num_batches_tracked, float momentum, float eps,
                          float* enc_w, float* enc_b, int32_t h, void* stream);
int b200_encoder_fold_bwd(const float* w, const float* b, const float* gamma, const double* moments,
                          const float* running_mean, const float* running_var, float eps,
                          const float* g_enc_w, const float* g_enc_b,
                          float* grad_w, float* grad_b, float* grad_gamma, float* grad_beta,
                          int32_t h, int32_t accumulate, void* stream);

/* Fused forward of LocalFeatureAggregation.propagate()+message() (pyg_randla_net.py:121-152: x_j / pos gathers :121-124,
 * relative position encoding :141-143, mlp_encoder :144, concat :145, mlp_attention :149, softmax :150, weighting :152,
 * aggr="add").  c = channels of the LFA (x has h = c/2 features).
 *   x       fp32 [n, h]        pos fp32 [n, 3]      nbr int32 [n, kt]
 *   enc_w   fp32 [h, 7]        encoder weight acting on q=(p_i,p_j,dist), BatchNorm folded in
 *   enc_b   fp32 [h]           folded bias
 *   att_wt  fp32 [c, c]        TRANSPOSE of mlp_attention.lins.0.weight (att_wt[m][n] = W[n][m])
 *   out     fp32 [n, c]        sum_j softmax_j(W f_ij) * f_ij,  f_ij = [x_j ; lrelu(enc_w q_ij + enc_b)]
 */
int b200_lfa_fwd(const float* x, const float* pos, const int32_t* nbr,
                 const float* enc_w, const float* enc_b, const float* att_wt,
                 float* out, int64_t n, int32_t c, int32_t kt, void* stream);

/* Fused backward of the same block (autograd of pyg_randla_net.py:121-152; recomputes the forward per tile).
 * grad_x / grad_enc_w / grad_enc_b /
 * grad_att_w are ACCUMULATED into (atomics): the caller zero-fills them.
 *   att_w   fp32 [c, c]  mlp_attention.lins.0.weight as stored ([out, in])
 *   grad_att_w fp32 [c, c] in the same [out, in] layout
 *   workspace: b200_lfa_bwd_workspace_bytes(n, c, kt) bytes of scratch (16-byte aligned; 0 bytes / NULL for
 *   c <= 32).  For c >= 64 the per-edge softmax gradients and features are streamed there and the
 *   attention-weight gradient is reduced by a split-K GEMM instead of per-tile atomics.
 */
int64_t b200_lfa_bwd_workspace_bytes(int64_t n, int32_t c, int32_t kt);
int b200_lfa_bwd(const float* x, const float* pos, const int32_t* nbr,
                 const float* enc_w, const float* enc_b, const float* att_wt, const float* att_w,
                 const float* grad_out,
                 float* grad_x, float* grad_enc_w, float* grad_enc_b, float* grad_att_w,
                 void* workspace, int64_t workspace_bytes,
                 int64_t n, int32_t c, int32_t kt, void* stream);

/* ------------------------------------------------------- index / scatter kernels -------
 * b200_gather_rows: out[i, :] = src[idx[i], :]          (decimate, pyg_randla_net.py:237)
 * b200_scatter_rows_add: dst[idx[i], :] += src[i, :]    (its backward; dst pre-zeroed)
 * idx is int64 (what torch.randperm yields at pyg_randla_net.py:221).
 */
int b200_gather_rows(const float* src, const int64_t* idx, float* out,
                     int64_t n_out, int32_t c, void* stream);
int b200_scatter_rows_add(const float* src, const int64_t* idx, float* dst,
                          int64_t n_src, int32_t c, void* stream);

/* Inverse-squared-distance kNN interpolation = torch_geometric knn_interpolate's tail
 * (pyg_randla_net.py:250 with k=1; model.py:90-98 with k=10):
 *   w_e = 1 / max(d2_e, 1e-16);  y_i = (sum_e x[nbr_e] * w_e) / (sum_e w_e)
 * with the reference's rounding sequence (products, sequential sums in ascending-distance
 * order, one IEEE division) so that k=1 reproduces (x*w)/w bit for bit.
 *   nbr int32 [ny, kt], dist2 fp32 [ny, kt] from b200_knn; -1 entries are skipped.
 *   out fp32 [ny, ld_out] written at columns [0, c)  (ld_out >= c lets the caller
 *   interpolate straight into the left part of a concat buffer).
 * Backward: grad_x[nbr_e, :] += grad_y[i, :] * w_e / sum_e w_e   (grad_x pre-zeroed).
 */
int b200_knn_interp_fwd(const float* x, const int32_t* nbr, const float* dist2,
                        float* out, int64_t ny, int32_t c, int32_t k, int32_t kt,
                        int64_t ld_out, void* stream);
int b200_knn_interp_bwd(const float* grad_y, int64_t ld_grad, const int32_t* nbr, const float* dist2,
                        float* grad_x, int64_t ny, int32_t c, int32_t k, int32_t kt, void* stream);

/* ------------------------------------------------------- per-point shared MLP ----------
 * Replace SharedMLP = PyG MLP(Linear -> BatchNorm1d(momentum .01, eps 1e-6) -> LeakyReLU(.2))
 * (pyg_randla_net.py:97-109) on [n, c] rows, torch.nn.Linear for fc0 / fc_classif
 * (pyg_randla_net.py:42,53) and the block tail lrelu(mlp2(x) + shortcut(x)) (:186-187).
 *
 * b200_linear_fwd:  y[n, cout] = [a1 | a2] W^T + bias
 *   a1 fp32 [n, c1] (row stride ld1), a2 fp32 [n, c2] (row stride ld2) or NULL with c2 = 0:
 *   the K dimension is the concatenation (FPModule's torch.cat, pyg_randla_net.py:251).
 *   w fp32 [cout, c1+c2] row-major, bias fp32 [cout] or NULL.
 *   If colstats != NULL the epilogue also produces, for the BatchNorm that follows, per-ROW-TILE partial
 *   sums: colstats fp64 [P, 2*cout] with P = b200_linear_fwd_num_stat_partials(n, c1, c2, cout); row p holds
 *   (sum_i y[i,ch], sum_i y[i,ch]^2) over the rows of tile p.  Rows are WRITTEN (no zero-fill, no atomics);
 *   b200_bn_finalize adds them up.
 */
int64_t b200_linear_fwd_num_stat_partials(int64_t n, int32_t c1, int32_t c2, int32_t cout);
int b200_linear_fwd(const float* a1, int64_t ld1, int32_t c1, const float* a2, int64_t ld2, int32_t c2,
                    const float* w, const float* bias, float* y, int64_t n, int32_t cout,
                    double* colstats, void* stream);
/* Autograd of the Linear layers of SharedMLP / fc0 / fc_classif (pyg_randla_net.py:42,53,97-109), input side:
 * grad_a[n, c1+c2 split as ga1|ga2] = grad_y W ; either output may be NULL (skipped).
 * workspace (16-byte aligned, b200_linear_bwd_input_workspace_bytes(), may be NULL / 0): holds W^T for the
 * tensor-core path (layers with >= 64 input and output channels); without it the fp32-FMA kernel runs.
 * Layers with >= 64 input and output channels (and c1 % 32 == 0) run on tcgen05 (3xTF32) in b200_linear_fwd /
 * b200_linear_bwd_input and then require 16-byte aligned rows. */
int64_t b200_linear_bwd_input_workspace_bytes(int64_t n, int32_t c1, int32_t c2, int32_t cout);
int b200_linear_bwd_input(const float* grad_y, const float* w, float* ga1, int64_t ldg1, int32_t c1,
                          float* ga2, int64_t ldg2, int32_t c2, void* workspace, int64_t workspace_bytes,
                          int64_t n, int32_t cout, void* stream);
/* Autograd of the same Linear layers (pyg_randla_net.py:42,53,97-109), parameter side:
 * grad_w[cout, c1+c2] += grad_y^T [a1|a2];  grad_bias[cout] += column sums of grad_y
 * (both ACCUMULATED: caller zero-fills; grad_bias may be NULL).  >= 64 x 64 weights run on the tensor cores
 * (tcgen05, 3xTF32 split: fp32-grade accuracy).  `workspace` (optional; 16-byte aligned,
 * b200_linear_bwd_weight_workspace_bytes() bytes) lets the split-K partial tiles be reduced by a second
 * kernel instead of global atomics (faster and deterministic); NULL selects the atomic path. */
int64_t b200_linear_bwd_weight_workspace_bytes(int64_t n, int32_t c1, int32_t c2, int32_t cout, int32_t has_bias);
int b200_linear_bwd_weight(const float* grad_y, const float* a1, int64_t ld1, int32_t c1,
                           const float* a2, int64_t ld2, int32_t c2,
                           float* grad_w, float* grad_bias, void* workspace, int64_t workspace_bytes,
                           int64_t n, int32_t cout, void* stream);

/* BatchNorm1d(momentum 0.01, eps 1e-6) of SharedMLP (pyg_randla_net.py:94-109; PyG MLP norm="batch_norm"):
 * statistics -> per-channel affine.  colstats fp64 [num_partials, 2*c] = partial (sum, sum of
 * squares) rows that add up to the statistics over `count` rows.  Writes scale = gamma*invstd, shift = beta - mean*scale, and
 * mean / invstd (saved for backward).  If running_mean != NULL updates the running
 * statistics in place: r = (1-momentum) r + momentum * stat (unbiased variance).
 * and increments *num_batches_tracked (int64, may be NULL).
 * With colstats == NULL (eval mode) uses the running statistics instead. */
int b200_bn_finalize(const double* colstats, int32_t num_partials, int64_t count, const float* gamma, const float* beta,
                     float* running_mean, float* running_var, int64_t* num_batches_tracked,
                     float momentum, float eps,
                     float* scale, float* shift, float* mean, float* invstd, int32_t c, void* stream);

/* BatchNorm apply + LeakyReLU(0.2) of SharedMLP (pyg_randla_net.py:92,97-109) and, with the second branch, the residual
 * tail lrelu(mlp2(x) + shortcut(x)) of DilatedResidualBlock (pyg_randla_net.py:186-187):
 * out = act(y1*scale1 + shift1 [+ y2*scale2 + shift2]) ; act = LeakyReLU(slope) (slope = 1: identity). */
int b200_affine_act_fwd(const float* y1, const float* scale1, const float* shift1,
                        const float* y2, const float* scale2, const float* shift2,
                        float slope, float* out, int64_t n, int32_t c, void* stream);

/* Backward of the same block (autograd of pyg_randla_net.py:97-109,186-187), pass 1: g = grad_out * act'(out);
 * accumulates (fp64, pre-zeroed)
 *   red1[0:c] = sum g,  red1[c:2c] = sum g * (y1 - mean1) * invstd1   (and red2 likewise for y2). */
int b200_affine_act_bwd_reduce(const float* grad_out, const float* out, float slope,
                               const float* y1, const float* mean1, const float* invstd1, double* red1,
                               const float* y2, const float* mean2, const float* invstd2, double* red2,
                               int64_t n, int32_t c, void* stream);
/* Backward of the same block, pass 2 (train-mode BatchNorm): with xhat = (y - mean) * invstd,
 *   grad_y = gamma*invstd * (g - red[0:c]/n - xhat * red[c:2c]/n),
 *   grad_gamma += red[c:2c], grad_beta += red[0:c]  (ACCUMULATED when the pointers are given: pass the parameters'
 *   .grad buffers, or zero-filled temporaries).
 * Eval mode / plain affine (red == NULL): grad_y = g * scale.
 * grad_y2 (second branch) is produced when y2 != NULL. */
int b200_affine_act_bwd_apply(const float* grad_out, const float* out, float slope,
                              const float* y1, const float* gamma1, const float* mean1, const float* invstd1,
                              const double* red1, const float* scale1, float* grad_y1,
                              float* grad_gamma1, float* grad_beta1,
                              const float* y2, const float* gamma2, const float* mean2, const float* invstd2,
                              const double* red2, const float* scale2, float* grad_y2,
                              float* grad_gamma2, float* grad_beta2,
                              int64_t n, int32_t c, void* stream);
/* Train-mode backward of the same block in ONE call: b200_affine_act_bwd_reduce followed by b200_affine_act_bwd_apply
 * (autograd of BatchNorm1d + LeakyReLU inside SharedMLP, pyg_randla_net.py:97-109, and of the block tail :186-187).
 * red1 / red2 (fp64 [2c] each) and `barrier` (one uint32) must be ZERO on entry; they are scratch.  When n * c <= 2^21,
 * c % 4 == 0, the rows are 16-byte aligned and option "bn_backward_fused" is 1 (default 0), both passes run as one kernel with a
 * grid barrier in between (at most #SMs / 2 CTAs, two fit an SM: always co-resident); otherwise, or with
 * barrier == NULL, as the two launches.  Results are those of the two-call sequence. */
int b200_affine_act_bwd(const float* grad_out, const float* out, float slope,
                        const float* y1, const float* gamma1, const float* mean1, const float* invstd1, double* red1,
                        float* grad_y1, float* grad_gamma1, float* grad_beta1,
                        const float* y2, const float* gamma2, const float* mean2, const float* invstd2, double* red2,
                        float* grad_y2, float* grad_gamma2, float* grad_beta2,
                        uint32_t* barrier, int64_t n, int32_t c, void* stream);

/* ------------------------------------------------------- loss --------------------------
 * torch.nn.CrossEntropyLoss(weight | NULL, ignore_index, label_smoothing=0, reduction="mean") on [n, c] logits and
 * int64 targets (configs/model/criterion/{CrossEntropyLoss,WeightedCrossEntropyLoss}.yaml; models/model.py:117-118,135-136,152-153); c <= 32.
 *   fwd: acc (fp64 [2]) and counter (uint32 [1]) are zero-filled scratch; loss_out fp32 [2] = {mean loss, sum of the
 *        weights of the rows that count} (the second value feeds the backward).  0 counted rows -> NaN like torch; a
 *        target outside [0, c) other than ignore_index also yields NaN (torch: device-side assert).
 *   bwd: grad_logits [n, c] = *grad_loss * w[t] * (softmax(x) - onehot(t)) / loss_out[1]; ignored rows get 0. */
int b200_cross_entropy_fwd(const float* logits, const int64_t* target, const float* weight, int64_t n, int32_t c,
                           int64_t ignore_index, double* acc, uint32_t* counter, float* loss_out, void* stream);
int b200_cross_entropy_bwd(const float* logits, const int64_t* target, const float* weight, int64_t n, int32_t c,
                           int64_t ignore_index, const float* loss_and_wsum, const float* grad_loss,
                           float* grad_logits, void* stream);

/* ------------------------------------------------------- optimizer ----------------------
 * One Adam update over FLAT fp32 buffers (parameters, gradients, first and second moments), the arithmetic of
 * torch.optim.Adam(lr, betas, eps) without weight decay / amsgrad (configs/model/optimizer/Adam.yaml uses the
 * defaults).  *step (device int64) is incremented first and used for the bias corrections, so the call is
 * CUDA-graph capturable.  lr_dev (device float, may be NULL) overrides lr: a captured graph then follows a
 * learning-rate scheduler (configs/model/lr_scheduler/).  All buffers 16-byte aligned. */
int b200_adam_flat(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                   const float* lr_dev, float beta1, float beta2, float eps, int64_t* step, void* stream);

/* ------------------------------------------------------- sliding-window stitch (SURVEY 8f-2) ---
 * b200_stitch_segment_sum replaces torch_scatter.scatter_sum(logits, idx_in_full_cloud, out=zeros(nb_points, C))
 * (myria3d/models/interpolation.py:113-116).  `order` is a STABLE argsort of the destination indices and
 * `sorted_idx = idx[order]`; every destination row is summed sequentially in input order (bit-identical to the
 * reference's CPU scatter, deterministic, no atomics).  `out` is pre-zeroed by the caller; rows without a
 * prediction stay zero.
 * b200_stitch_finalize replaces reduced_logits[idx] (:121), Softmax(dim=1) (:142), argmax (:145) and
 * Categorical(probs).entropy() (:166) in one pass; logits / probas / preds / entropy may each be NULL.
 * c <= 32 classes. */
int b200_stitch_segment_sum(const float* rows, const int64_t* order, const int64_t* sorted_idx, float* out,
                            int64_t m, int32_t c, int64_t nb_points, void* stream);
int b200_stitch_finalize(const float* reduced, const int64_t* idx, float* logits, float* probas, int64_t* preds,
                         float* entropy, int64_t m, int32_t c, void* stream);

/* ------------------------------------------------------- decimation draw ----------------
 * Replaces decimation_indices() (myria3d/models/modules/pyg_randla_net.py:192-231): per cloud b, a uniformly random
 * ORDERED subset of new_ptr[b+1] - new_ptr[b] of its ptr[b+1] - ptr[b] points (the distribution of
 * ptr[b] + torch.randperm(n_b)[:n_b // decimation]), all clouds of the batch in one launch, no host sync.
 * Random stream: Philox4x32-10 keyed by (seed, salt) and counted by (global point index, *counter); `counter`
 * (device int64, may be NULL = 0) is read, never written: advance it with b200_counter_add between draws (both are
 * CUDA-graph capturable).  idx_out[new_ptr[b] + t] (int64) receives the t-th drawn point of cloud b as an index into
 * the batch.  max_kept = max_b (new_ptr[b+1] - new_ptr[b]) <= 25600 (B200_E_UNSUPPORTED beyond). */
int b200_decimation_draw(const int64_t* ptr, const int64_t* new_ptr, int32_t num_clouds, int64_t max_kept, uint64_t seed,
                         const int64_t* counter, uint32_t salt, int64_t* idx_out, void* stream);
/* *counter += delta (single-thread kernel; device-side step / draw counters of captured graphs). */
int b200_counter_add(int64_t* counter, int64_t delta, void* stream);

/* ------------------------------------------------------- predict-time sample preparation (SURVEY 8f-4) ------
 * What myria3d does on the CPU between reading a tile and batching receptive fields, as kernels.  Caller owns all
 * buffers; *_tmp buffers have the size of their partner; offsets01 is a device int64[2] = {0, n}.
 *
 * b200_segmented_sort_pairs: stable ascending LSB radix sort of (key, val) pairs by the low key_bits bits, segment s =
 *   [offsets[s], offsets[s+1]), one CTA per segment; result in keys / vals (building block of the entries below).
 * b200_receptive_fields_per_axis / _count / _fill replace split_cloud_into_samples (myria3d/pctl/dataset/utils.py:
 *   126-158) + get_mosaic_of_centers (:29-38): field f = ix * per_axis + iy has centre (w/2 + ix * (w - overlap),
 *   w/2 + iy * (w - overlap)) relative to (min_x, min_y) of the cloud; a point belongs to it iff its Chebyshev distance
 *   to the centre is <= floor(w / 2) (scipy query_ball_point(r = subtile_width // 2, p = inf), tested in float64 like
 *   scipy).  _count fills counts[per_axis^2] (int64); the caller turns them into offsets (exclusive scan, per_axis^2 + 1
 *   entries) and _fill writes every field's point indices in ASCENDING order (uint32) at idx[offsets[f] ...]; cursors =
 *   per_axis^2 uint64 of scratch, pay / pay_tmp / idx_tmp = scratch of sum(counts) uint32.
 * b200_grid_sampling_sort / _pool replace torch_geometric.transforms.GridSampling(size) for ONE sample
 *   (configs/datamodule/transforms/preparations/points_budget.yaml:76-79; PyG 2.4 semantics: voxel_grid over
 *   [pos.min(0), pos.max(0)] = start_end[6] (device), consecutive_cluster -> voxels in ascending id order, scatter MEAN
 *   of pos and x, majority vote (ties: lowest class) of y).  _sort leaves (voxel id, point index) sorted in key / val,
 *   head[i] = 1 at the first point of every voxel and *num_voxels; the caller compacts the head positions into
 *   run_start[num_voxels] (int32) and calls _pool, which writes pos_out / x_out / y_out [num_voxels rows].
 * b200_random_permutation: perm = a uniformly random permutation of 0..n-1 (Philox keys of b200_decimation_draw +
 *   sort): perm[:num] is torch.randperm(n)[:num] of MaximumNumNodes / MinimumNumNodes (transforms.py:48-84).
 * b200_center_pos: pos -= pos.mean(0) for one sample (torch_geometric.transforms.Center, points_budget.yaml:96-97). */
int b200_segmented_sort_pairs(uint32_t* keys, uint32_t* vals, uint32_t* keys_tmp, uint32_t* vals_tmp,
                              const int64_t* offsets, int32_t num_segments, int32_t key_bits, void* stream);
int32_t b200_receptive_fields_per_axis(float tile_width, float subtile_width, float subtile_overlap);
int b200_receptive_fields_count(const float* pos, int64_t n, float min_x, float min_y, float tile_width,
                                float subtile_width, float subtile_overlap, int64_t* counts, void* stream);
int b200_receptive_fields_fill(const float* pos, int64_t n, float min_x, float min_y, float tile_width,
                               float subtile_width, float subtile_overlap, const int64_t* offsets, uint64_t* cursors,
                               uint32_t* idx, uint32_t* idx_tmp, uint32_t* pay, uint32_t* pay_tmp, void* stream);
int b200_grid_sampling_sort(const float* pos, int32_t n, float size, const float* start_end, uint32_t* key, uint32_t* val,
                            uint32_t* key_tmp, uint32_t* val_tmp, const int64_t* offsets01, int32_t* head,
                            int32_t* num_voxels, void* stream);
int b200_grid_sampling_pool(const uint32_t* key, const uint32_t* val, const int32_t* run_start, int32_t num_voxels, int32_t n,
                            const float* pos, const float* x, int32_t cx, const int64_t* y, int32_t num_classes,
                            float* pos_out, float* x_out, int64_t* y_out, int32_t* count_out, void* stream);
int b200_random_permutation(int64_t n, uint64_t seed, const int64_t* counter, uint32_t salt, uint32_t* key, uint32_t* perm,
                            uint32_t* key_tmp, uint32_t* perm_tmp, const int64_t* offsets01, void* stream);
int b200_center_pos(float* pos, int32_t n, void* stream);

/* ------------------------------------------------------- batch preparation (train / eval / predict) ------
 * myria3d's per-sample transform chain, run on a whole raw batch of B samples (sample b = rows [ptr[b], ptr[b+1]) of
 * pos fp32 [n, 3], x fp32 [n, cx], y int64 [n] raw LAS codes, idx int64 [n] = idx_in_original_cloud), in the order of
 * pctl/datamodule/hdf5.py:76-89 (preparations + normalizations [+ augmentations in train]).  mode: 0 train, 1 eval,
 * 2 predict.  Buffers *_c, key / val / *_tmp, run_start and the pooled *_p have the raw layout (n rows, sample b at
 * ptr[b]); stats is int32 [b200_batch_prep_stats_len(B)]:
 *   [0] error flags (B200_BATCH_PREP_E_*), [1..8] bitmask of the unknown codes 0..255, [9 + b] rows kept by
 *   DropPointsByClass, [9 + B + b] voxels after GridSampling.
 * The caller reads stats once, after _pool, and sizes the rest from it.
 *
 * b200_batch_prep_compact replaces TargetTransform (pctl/transforms/transforms.py:168-232: lut[code] = rank in
 *   classification_dict of preprocessing_dict.get(code, code), 65 for 65, -1 for an unknown code; train / eval only) and
 *   DropPointsByClass (:235-248: rows labelled 65 dropped, order kept; idx subsampled alike), then computes each sample's
 *   GridSampling voxel ids over its bounding box (x fastest; B200_BATCH_PREP_E_VOXEL_OVERFLOW when they do not fit
 *   below 2^32 - 1).  In predict mode lut is ignored and rows with the raw code 65 are dropped.  y / idx may be NULL in
 *   predict mode.
 * b200_batch_prep_voxelize: stable per-sample sort of (voxel id, row) and run heads -> run_start, voxel counts.
 * b200_batch_prep_pool replaces torch_geometric.transforms.GridSampling(grid_size) (points_budget.yaml:76-79): per
 *   voxel, fp64 mean of pos and x, majority label (ties: lowest class < num_classes); per sample bit-identical to
 *   b200_grid_sampling_sort / _pool on that sample alone.
 * b200_batch_prep_budget_draw: the permutations of MinimumNumNodes / MaximumNumNodes (transforms.py:48-84) for the whole
 *   batch: segment g = [seg_off[g], seg_off[g+1]) (device int64 [num_segments + 1], total = seg_off[num_segments])
 *   receives a uniformly random permutation of 0 .. length - 1 in perm; seg_ids = int32 [num_segments][2] = (sample,
 *   repetition) of each segment.  Philox keys of (seed, sample) counted by (row, repetition, *counter) as
 *   b200_decimation_draw, then b200_segmented_sort_pairs.
 * b200_batch_prep_finalize: one CTA per sample: rows r < out_ptr[b+1] - out_ptr[b] are pooled rows
 *   perm[choice_off[b] + r] (choice_off[b] = -1: row r) of sample b; Center (torch_geometric, fp64 mean), NullifyLowestZ,
 *   NormalizePos (pos * scale, scale = (float)(1 / (subtile_width / 2)), transforms.py:141-165),
 *   StandardizeRGBAndIntensity on columns col_intensity (log(v + 1) first) and col_rgb (:117-138: fp64 mean and
 *   unbiased std + 1e-6, NaN std -> 1, clamp to +-3 std), and in train mode RandomFlip(0, flip_p), RandomFlip(1, flip_p)
 *   (flip_p < 0: none) and RandomRotate(rotate_degrees, axis=2) (0: none; pos @ M^T, M = [[cos, sin, 0], [-sin, cos, 0],
 *   [0, 0, 1]], cos / sin rounded to fp32) with Philox draws of (seed, *counter, b).  Writes pos_out, x_out, y_out (if
 *   y_p), batch_out (int64) at out_ptr[b]; eval / predict: pos_sampled_copy (CopySampledPos) and the rows kept by
 *   DropPointsByClass, pos_c -> pos_copy (CopyFullPos) and, in eval, y_c -> y_copy (CopyFullPreparedTargets) at
 *   full_ptr[b].  draws (may be NULL) = fp64 [B, 3]: flip x, flip y, angle in degrees. */
#define B200_BATCH_PREP_E_UNKNOWN_CODE 1
#define B200_BATCH_PREP_E_CODE_RANGE 2
#define B200_BATCH_PREP_E_VOXEL_OVERFLOW 4
int64_t b200_batch_prep_stats_len(int32_t num_samples);
int b200_batch_prep_compact(int32_t mode, const float* pos, const float* x, int32_t cx, const int64_t* y, const int64_t* idx,
                            const int64_t* ptr, int32_t num_samples, int64_t n, const int32_t* lut, float grid_size,
                            float* pos_c, float* x_c, int64_t* y_c, int64_t* idx_c, uint32_t* key, uint32_t* val,
                            int32_t* stats, void* stream);
int b200_batch_prep_voxelize(uint32_t* key, uint32_t* val, uint32_t* key_tmp, uint32_t* val_tmp, const int64_t* ptr,
                             int32_t num_samples, int32_t* run_start, int32_t* stats, void* stream);
int b200_batch_prep_pool(const uint32_t* val, const int32_t* run_start, const int64_t* ptr, int32_t num_samples, int64_t n,
                         const int32_t* stats, const float* pos_c, const float* x_c, int32_t cx, const int64_t* y_c,
                         int32_t num_classes, float* pos_p, float* x_p, int64_t* y_p, void* stream);
int b200_batch_prep_budget_draw(const int64_t* seg_off, const int32_t* seg_ids, int32_t num_segments, int64_t total,
                                uint64_t seed, const int64_t* counter, uint32_t* key, uint32_t* perm, uint32_t* key_tmp,
                                uint32_t* perm_tmp, void* stream);
int b200_batch_prep_finalize(int32_t mode, const float* pos_p, const float* x_p, int32_t cx, const int64_t* y_p,
                             const int64_t* ptr, int32_t num_samples, const uint32_t* perm, const int64_t* choice_off,
                             const int64_t* out_ptr, int32_t col_intensity, int32_t col_rgb, float scale, float flip_p,
                             float rotate_degrees, uint64_t seed, const int64_t* counter, float* pos_out, float* x_out,
                             int64_t* y_out, int64_t* batch_out, float* pos_sampled_copy, const float* pos_c,
                             const int64_t* y_c, const int32_t* stats, const int64_t* full_ptr, float* pos_copy,
                             int64_t* y_copy, double* draws, void* stream);

/* ------------------------------------------------------- tcgen05 self-test --------------
 * d[128, n] (+)= a[128, k] * b[n, k]^T on the 5th-generation tensor cores (tcgen05.mma, TMEM accumulator):
 * passes = 1 plain TF32, 3 = 3xTF32 split (kind::tf32), 6 = bf16 x 3 split (kind::f16, six cross products: the
 * arithmetic of tc_skinny.cu), 2 = fp16 x 2 split (kind::f16, three cross products: the arithmetic of the fused LFA
 * kernels); 2, 3 and 6 are fp32-grade.  Pins the shared-memory descriptor / TMEM
 * conventions of the fused kernels (no reference counterpart: test infrastructure of the kernels that replace
 * pyg_randla_net.py:97-152).  flags: bit 0 / bit 1 = stage A / B transposed and read it through the MN-major
 * descriptor (passes = 2 or 6); bit 2 = pre-initialise the accumulator from d with tcgen05.st and accumulate.
 * *status (device int32): 0 = ok, 1 = the MMA completion barrier timed out.
 * 16 <= n <= 256, n % 16 == 0, k % 8 == 0 (k % 16 == 0 for passes = 2 or 6); flags < 16 (bit 3: A in tensor memory). */
int b200_tc_gemm_selftest(const float* a, const float* b, float* d, int32_t n, int32_t k, int32_t passes,
                          int32_t flags, int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200RANDLA_H_ */
