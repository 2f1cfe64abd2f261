/*
 * grafp_b200.h - C ABI of the B200-native GraFP GraphEncoder hot path.
 *
 * One shared library (libgrafp_b200.so, sm_100a only) replaces the PyTorch-eager op
 * sequences of the reference's dynamic k-NN graph and graph-convolution aggregation.
 * Citations are into the upstream chymaera96/GraFP checkout.
 *
 * Conventions
 *  - Every tensor is a plain device pointer owned by the caller; the library never
 *    allocates, frees or retains device memory.  All work is enqueued on `stream`
 *    (a cudaStream_t / CUstream passed as void*); calls return after launch and are
 *    CUDA-graph capturable.  There is NO CPU path: host pointers are an error.
 *  - Node features are stored as rows: x[b][n][c] contiguous ("channels last" of the
 *    reference's logical (B, C, N, 1) tensors).  dtype: 0 = float32, 1 = bfloat16.
 *  - Index tensors are (B, N, k) contiguous, int64 (the reference's edge_index
 *    element type) when idx_is_i64 != 0, else int32.  Neighbour ids address the key
 *    set (y when given, else x) of the same batch item, in [0, M).
 *  - Return value: 0 = success; < 0 = GRAFP_E* argument/shape error; > 0 = the
 *    cudaError_t of a failed launch.  grafp_last_error() returns a thread-local
 *    message for the last failing call on this thread.
 */
#ifndef GRAFP_B200_H_
#define GRAFP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GRAFP_ABI_VERSION 7

#define GRAFP_OK 0
#define GRAFP_EINVAL (-1)       /* null / misaligned pointer, non-positive size, k > M ... */
#define GRAFP_EUNSUPPORTED (-2) /* shape or dtype outside what the kernels implement      */
#define GRAFP_EWORKSPACE (-3)   /* workspace smaller than grafp_knn_workspace_bytes()     */
#define GRAFP_ENODEVICE (-4)    /* no sm_100 device is current                            */

#define GRAFP_F32 0
#define GRAFP_BF16 1

/* k-NN kernel selection for grafp_knn_fwd */
#define GRAFP_KNN_AUTO 0 /* tcgen05 path when the shape allows it, else the SIMT path */
#define GRAFP_KNN_SIMT 1 /* exact-fp32 CUDA-core Gram + fused top-k                   */
#define GRAFP_KNN_TC 2   /* TMA + tcgen05 + fused top-k: the f16x3 kernels when K <= 8, else the tf32x3 kernel */
#define GRAFP_KNN_TC_TF32 3 /* force the first-generation tf32x3 tcgen05 kernel (cross-check)          */

#define GRAFP_KNN_MAX_K 128 /* k * dilation: the reference caps dilation at 128 // k (graph_encoder.py:128) */

int grafp_abi_version(void);
const char* grafp_last_error(void);

/*
 * Kernel-selection / diagnostic options (process-wide, atomically readable from any thread).  Defaults are read
 * ONCE, when the first option is consulted, from the environment variable GRAFP_<NAME IN CAPITALS>; after that only
 * grafp_set_option changes them (tests and benchmarks use this for A/B runs).  Names and values:
 *   "mr_fwd_form"  K2: 0 generic, 1 register-prefetch kernel, 2 cp.async-pipelined persistent kernel (default)
 *   "mr_bwd_form"  K3: 0 dense + scatter pair, 1 cluster kernel with a device-scope fence, 2 cluster kernel (default),
 *                  3 deterministic gather over the reverse graph (fp32, k == 3, needs the workspace)
 *   "knn_epilogue" K1 selection: 0 auto (default), 1 vote-gated scan, 2 candidate queues, 3 group maxima (K <= 4)
 *   "edge_bwd_row" / "gather_row" / "edge_row" / "maxk_row": 1 = row-form kernels (default), 0 = per-edge forms
 *   "bn_reverse"   K5: 1 = first pass back to front (its input was just written front to back: the tail is in L2), second
 *                  pass front to back (default); 0 = the other way round
 *   "bn_persistent" K5: 1 = statistics + apply in ONE cooperative launch with a grid barrier (default), 0 = two launches
 *   "bn_l2_keep_mb" K5: megabytes of the first pass's input loaded "evict last" so the second pass finds them in L2
 *                  (the rest of both passes is loaded "evict first"); default 80, 0 = no cache hints
 *   "check_index"  1 = grafp_check_index is run on user-supplied graphs by the Python layer (default 0)
 *   "conv_gemm"    1 = the Python layer runs dense 1x1 convolutions in front of a train-mode BatchNorm through
 *                  grafp_conv1x1_bn_stats_fwd when TF32 convolutions are allowed and a row of x is at most 2 KB
 *                  (default 1); 2 = whatever the row size; 0 = cuDNN + full BatchNorm
 * grafp_set_option returns GRAFP_EINVAL for an unknown name; grafp_get_option returns the value, or GRAFP_EINVAL.
 */
int grafp_set_option(const char* name, int value);
int grafp_get_option(const char* name);

/*
 * Range check of an index tensor (the reference's advanced indexing raises IndexError for ids outside [0, M),
 * torch_nn.py:92-96; the aggregation kernels address rows with them unchecked).  Counts the entries of
 * idx[0 .. count) (int64 when idx_is_i64 != 0, else int32) outside [0, limit) into *bad_count (device int32, zeroed
 * by the call).  The caller synchronises and reads it.
 */
int grafp_check_index(const void* idx, int idx_is_i64, long long count, int limit, int* bad_count, void* stream);

/* Diagnostic: name of the k-NN kernel the last grafp_knn_fwd call on this thread launched
 * ("simt", "tcgen05"). */
const char* grafp_knn_last_algo(void);
/* Diagnostic: which arithmetic the last k-NN call used: "f16x3" (fp16 hi/lo planes, kind::f16),
 * "tf32x3" (tf32 hi/lo planes, kind::tf32) or "fp32" (CUDA cores). */
const char* grafp_knn_last_variant(void);

/*
 * Dilated k-NN graph.  Replaces DenseDilatedKnnGraph.forward
 * (encoder/gcn_lib/torch_edge.py:270-284) = F.normalize (:274-275,281) +
 * pairwise_distance / xy_pairwise_distance (:7-18, :37-53) + optional relative_pos
 * bias (:97-99, :160-162) + topk (:100, :163) + DenseDilated [..., ::d] (:252-254),
 * without ever writing the N x M distance matrix to HBM.
 *
 *  x        (B, N, C) query node features.
 *  normalize != 0: L2-normalise every node over C first (what DenseDilatedKnnGraph.forward does);
 *           0: use the features as given (dense_knn_matrix / xy_dense_knn_matrix called directly).
 *  y        (B, M, C) key node features or NULL (keys = x, M must equal N).
 *  relpos   (N, M) float32 bias added to the squared distances, or NULL.
 *  nn_idx   (B, N, k_out) int64 out: neighbour ids sorted by ascending distance, ties by
 *           lowest id; k_out = k (ranks 0, d, 2d, ...) or k*dilation when emit_all != 0
 *           (the caller then applies DenseDilated's stochastic branch, :246-250).
 *  nn_idx32 optional int32 copy of nn_idx (same shape) or NULL.
 *  The centre ids (edge_index[1], :102) are arange(N) and are not produced here.
 *  metric   GRAFP_METRIC_L2: squared Euclidean distance |x|^2 - 2 x.y + |y|^2 (pairwise_distance).
 *           GRAFP_METRIC_COSINE: 1 - x.y (+ relpos), the distance of the cosine variants dense_knn_matrix_plg /
 *           xy_dense_knn_matrix_plg(_new) (:106-141, :166-219; SURVEY 8f row 3).  Evaluated as 2 (1 - x.y) through the
 *           same kernels with both squared norms forced to 1 - a power-of-two rescaling, so the order is the
 *           reference's up to ties; the caller passes relpos already doubled.
 */
#define GRAFP_METRIC_L2 0
#define GRAFP_METRIC_COSINE 1
size_t grafp_knn_workspace_bytes(int B, int N, int M, int C, int K, int dtype);
int grafp_knn_fwd(const void* x, const void* y, const float* relpos, int64_t* nn_idx, int32_t* nn_idx32,
                  int B, int N, int M, int C, int k, int dilation, int emit_all, int normalize, int dtype,
                  int algo, int metric, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Max-relative aggregation.  Replaces the body of MRConv2d.forward before self.nn
 * (encoder/gcn_lib/torch_vertex.py:21-32): two batched_index_select gathers
 * (torch_nn.py:79-98), x_j - x_i, max over k, and the channel-interleaving cat.
 *
 *  out[b][n][2c] = x[b][n][c]
 *  out[b][n][2c+1] = max_j ( src[b][nbr[b][n][j]][c] - x[b][ctr[b][n][j]][c] ),  src = y ? y : x
 *  argmax[b][n][c] = first j attaining the max (uint8; NULL when no backward is needed)
 *  ctr == NULL means ctr[b][n][j] = n (what the k-NN graph produces, torch_edge.py:102).
 *
 * The backward overwrites grad_x (B, N, C) and, when y was given, grad_y (B, M, C):
 *  grad_x[b][n][c]  = g[b][n][2c] + sum over (m, j = argmax[b][m][c]) of
 *                     ( -g[b][m][2c+1] if ctr[b][m][j] == n )  ( +g[b][m][2c+1] if y == NULL and nbr[b][m][j] == n )
 * `workspace` (optional, grafp_mr_aggregate_bwd_workspace_bytes(B, N, k) bytes, caller-owned scratch):
 * when given, and the graph is the k-NN op's (ctr == NULL, y == NULL, k == 3, fp32), the backward runs
 * in gather form over the reverse graph built into the workspace: no atomics, fixed summation order
 * (bit-reproducible).  Without it (or outside that envelope) the scatter uses vector reductions
 * (red.global.add) and the floating-point accumulation order is not fixed.
 */
int grafp_mr_aggregate_fwd(const void* x, const void* y, const void* nbr_idx, const void* ctr_idx, int idx_is_i64,
                           void* out, uint8_t* argmax, int B, int N, int M, int C, int k, int dtype, void* stream);
size_t grafp_mr_aggregate_bwd_workspace_bytes(int B, int N, int k);
int grafp_mr_aggregate_bwd(const void* grad_out, const uint8_t* argmax, const void* nbr_idx, const void* ctr_idx,
                           int idx_is_i64, void* grad_x, void* grad_y, int B, int N, int M, int C, int k, int dtype,
                           void* workspace, size_t workspace_bytes, void* stream);

/*
 * Plain neighbour gather.  Replaces batched_index_select (torch_nn.py:79-98).
 *  out[b][n][j][c] = src[b][idx[b][n][j]][c]          out is (B, N, k, C)
 * Backward (index_put_ accumulate of the reference's autograd) overwrites grad_src (B, M, C).
 */
int grafp_gather_fwd(const void* src, const void* idx, int idx_is_i64, void* out, int B, int N, int M, int C, int k,
                     int dtype, void* stream);
int grafp_gather_bwd(const void* grad_out, const void* idx, int idx_is_i64, void* grad_src, int B, int N, int M, int C,
                     int k, int dtype, void* stream);

/*
 * Neighbour sum.  Replaces batched_index_select + torch.sum(x_j, -1, keepdim=True) of GINConv2d.forward
 * (torch_vertex.py:84-88) without the (B, C, N, k) intermediate.
 *  out[b][n][c] = sum_j src[b][idx[b][n][j]][c]        out is (B, N, C), summed in the order j = 0 .. k-1
 * Backward overwrites grad_src (B, M, C):  grad_src[b][m][c] = sum over edges (n, j) with idx[b][n][j] = m of
 * grad_out[b][n][c].
 */
int grafp_neighbor_sum_fwd(const void* src, const void* idx, int idx_is_i64, void* out, int B, int N, int M, int C, int k,
                           int dtype, void* stream);
int grafp_neighbor_sum_bwd(const void* grad_out, const void* idx, int idx_is_i64, void* grad_src, int B, int N, int M,
                           int C, int k, int dtype, void* stream);

/*
 * EdgeConv feature construction.  Replaces cat([x_i, x_j - x_i], dim=1) of
 * EdgeConv2d.forward (torch_vertex.py:46-51).
 *  out[b][n][j][c]     = x[b][ctr[b][n][j]][c]
 *  out[b][n][j][C + c] = src[b][nbr[b][n][j]][c] - x[b][ctr[b][n][j]][c]      out is (B, N, k, 2C)
 * Backward overwrites grad_x (and grad_y when y was given).
 */
int grafp_edge_gather_fwd(const void* x, const void* y, const void* nbr_idx, const void* ctr_idx, int idx_is_i64,
                          void* out, int B, int N, int M, int C, int k, int dtype, void* stream);
int grafp_edge_gather_bwd(const void* grad_out, const void* nbr_idx, const void* ctr_idx, int idx_is_i64, void* grad_x,
                          void* grad_y, int B, int N, int M, int C, int k, int dtype, void* stream);

/*
 * Max over the neighbour axis.  Replaces torch.max(h, -1, keepdim=True) of
 * EdgeConv2d.forward (torch_vertex.py:51) and GraphSAGE.forward (:69).
 *  out[b][n][c] = max_j h[b][n][j][c],  argmax = first such j.   h is (B, N, k, C)
 * Backward overwrites grad_h with grad_out routed to the argmax slot and zeros elsewhere.
 */
int grafp_max_over_k_fwd(const void* h, void* out, uint8_t* argmax, int B, int N, int C, int k, int dtype, void* stream);
int grafp_max_over_k_bwd(const void* grad_out, const uint8_t* argmax, void* grad_h, int B, int N, int C, int k, int dtype,
                         void* stream);

/*
 * Train-mode BatchNorm over node rows fused with what follows it in the Grapher / FFN blocks
 * (SURVEY 8f row 2).  Replaces nn.BatchNorm2d (training) + nn.ReLU of BasicConv
 * (encoder/gcn_lib/torch_nn.py:52-64) and of FFN.fc1 + act (encoder/graph_encoder.py:56-66), and
 * nn.BatchNorm2d + the residual add of Grapher.fc2 / FFN.fc2 (torch_vertex.py:158-162,194;
 * graph_encoder.py:60-66).  x, residual, out, dy, dx are (R, C) rows of `dtype` (GRAFP_F32 / GRAFP_BF16),
 * R = B * N; statistics, weight, bias and their gradients are always float32.  A thread owns 16 bytes of channels:
 * C % V == 0 and C / V a power of two with V = 4 (fp32) / 8 (bf16), else GRAFP_EUNSUPPORTED.
 *
 *  forward : mean / biased variance over the R rows per channel (saved as save_mean, save_invstd =
 *            1 / sqrt(var + eps)); running_mean / running_var (may be NULL) are updated with `momentum`
 *            and the unbiased variance, like torch.nn.functional.batch_norm(training=True);
 *            out = (x - mean) * invstd * weight + bias  [+ residual]  [ReLU when relu != 0]
 *            (relu together with a residual is not implemented).
 *            conv_bias (C floats, may be NULL): bias of a convolution in front of the BatchNorm that was run WITHOUT it
 *            (a per-channel constant cancels in x - mean): it is added to the mean that enters running_mean.
 *            num_batches_tracked (device int64, may be NULL): incremented by one, like nn.BatchNorm2d does.
 *  backward: dz = dy masked by the ReLU (recomputed from x, no output is kept); dbias = sum dz,
 *            dweight = sum dz * xhat, dx = weight * invstd * (dz - dbias / R - xhat * dweight / R).
 *            The gradient of the residual input is dy itself and is not written here.
 *            dx_colsum (C floats, may be NULL): per-channel sum of dx over the rows - the bias gradient of the 1x1
 *            convolution that produced x (Conv2d(bias=True) + BatchNorm2d in Grapher.fc1 / fc2 and BasicConv), so
 *            its backward needs no separate reduction pass over dx.  (Zero in real arithmetic; what is returned is
 *            the rounding residue of the mean and of dbias / R, evaluated in double from the reduction sums.)
 *  Two launches each way (no finalize kernels: block partials are folded with red.f64 into the workspace).
 *  workspace: grafp_bn_workspace_bytes(C) bytes of caller-owned scratch, zeroed by the call itself.
 */
size_t grafp_bn_workspace_bytes(int C);
int grafp_bn_train_fwd(const void* x, const void* residual, const float* weight, const float* bias, float* running_mean,
                       float* running_var, const float* conv_bias, long long* num_batches_tracked, void* out, float* save_mean,
                       float* save_invstd, long long R, int C, float eps, float momentum, int relu, int dtype, void* workspace,
                       size_t workspace_bytes, void* stream);
int grafp_bn_train_bwd(const void* dy, const void* x, const float* weight, const float* bias, const float* save_mean,
                       const float* save_invstd, void* dx, float* dweight, float* dbias, float* dx_colsum, long long R, int C,
                       int relu, int dtype, void* workspace, size_t workspace_bytes, void* stream);

/*
 * 1x1 convolution with the BatchNorm statistics in its epilogue (SURVEY 8f row 2: "Conv2d(1x1) + BatchNorm [+ act]
 * fusion").  Replaces the Conv2d(Cin, Cout, 1) of torch_nn.py:52-64 (BasicConv), torch_vertex.py:152-162,183-194
 * (Grapher.fc1 / fc2) and graph_encoder.py:45-67 (FFN) together with the statistics pass of the train-mode BatchNorm2d
 * behind it: y = x w^T as one tcgen05 GEMM over the node rows, and per output channel sum y and sum y^2 (taken of the
 * values as stored, accumulated in double) left in the BatchNorm workspace.
 *   x (R, Cin), w (Cout, Cin / groups), y (R, Cout): rows of `dtype`; groups > 1 is Conv2d(groups=...) - output channels
 *   [g Cout/groups, (g+1) Cout/groups) see input channels [g Cin/groups, (g+1) Cin/groups) (BasicConv's groups = 4); GRAFP_F32 runs as TF32 with fp32 accumulation (what cuDNN
 *   does for this layer under torch.backends.cudnn.allow_tf32, PyTorch's default - callers that need full fp32 keep
 *   cuDNN), GRAFP_BF16 as bf16 with fp32 accumulation.  No bias: a per-channel constant cancels in the BatchNorm
 *   (conv_bias of grafp_bn_train_fwd* puts it back where it is visible, the running mean).
 *   Cin, Cout and Cin / groups must be multiples of 16 bytes of elements, Cout / groups a multiple of 16 channels that
 *   tiles 64 / 128 / 256 columns (GRAFP_EUNSUPPORTED otherwise; _supported() tells).
 * grafp_bn_train_fwd_from_moments is grafp_bn_train_fwd without its statistics pass: `workspace` must be the one the
 * convolution call wrote (same C = Cout); everything else - outputs, running statistics, saved mean / invstd - as there.
 */
int grafp_conv1x1_bn_stats_supported(long long R, int Cin, int Cout, int groups, int dtype);
int grafp_conv1x1_bn_stats_fwd(const void* x, const void* w, void* y, long long R, int Cin, int Cout, int groups, int dtype,
                               void* workspace, size_t workspace_bytes, void* stream);
int grafp_bn_train_fwd_from_moments(const void* x, const void* residual, const float* weight, const float* bias,
                                    float* running_mean, float* running_var, const float* conv_bias,
                                    long long* num_batches_tracked, void* out, float* save_mean, float* save_invstd, long long R,
                                    int C, float eps, float momentum, int relu, int dtype, void* workspace,
                                    size_t workspace_bytes, void* stream);

/*
 * Tap rows of the Downsample block (graph_encoder.py:16-28: Conv2d(3x3, stride 2, padding 1) over (B, C, N, 1): the image
 * is one pixel wide, so only the middle kernel column meets data and the layer is a 3-tap stride-2 convolution along
 * the node axis, i.e. a 1x1 convolution over taps[b][n'] = (x[b][2n'-1], x[b][2n'], x[b][2n'+1]), x[b][-1] = 0).
 *   x (B, N, C) rows -> taps (B, N/2, 3C) rows; backward: dtaps (B, N/2, 3C) -> dx (B, N, C), the overlapping thirds
 *   summed.  N even, C a multiple of 16 bytes of `dtype` elements (GRAFP_EUNSUPPORTED otherwise).
 */
int grafp_downsample_taps_fwd(const void* x, void* taps, int B, int N, int C, int dtype, void* stream);
int grafp_downsample_taps_bwd(const void* dtaps, void* dx, int B, int N, int C, int dtype, void* stream);

/*
 * NT-Xent contrastive loss (SURVEY 8f row 1).  Replaces simclr/ntxent.py:17-29 - a Python loop over the 2B rows of
 * z z^T / tau (log-softmax of each row without its diagonal entry, partner's entry picked) - and its autograd, without
 * materialising the (2B, 2B) similarity matrix.
 *   z        (n2, d) float32, the two views interleaved: rows 2m and 2m + 1 are partners (ntxent.py:18)
 *   lse      (n2) out: log sum_{j != i} exp(z_i . z_j / tau), kept for the backward
 *   row_loss (n2) scratch, loss (1) out: mean_i [lse_i - z_i . z_{i^1} / tau]
 *   backward: dz (n2, d) = grad_loss * dloss/dz, grad_loss a DEVICE scalar (the upstream gradient)
 * n2 even, d % 4 == 0, d <= 256 (else GRAFP_EUNSUPPORTED).
 */
int grafp_ntxent_fwd(const float* z, float* lse, float* row_loss, float* loss, int n2, int d, float inv_tau, void* stream);
int grafp_ntxent_bwd(const float* z, const float* lse, const float* grad_loss, float* dz, int n2, int d, float inv_tau,
                     void* stream);

/*
 * The same loss sharded by anchor rows, for data-parallel training (one process per GPU): z holds the embeddings of ALL
 * ranks (all-gathered), a rank evaluates only its own anchors [row_lo, row_hi) against every row - 1 / world of the work
 * instead of the whole (n2 x n2) problem on every rank.
 *   forward:  lse[i], row_loss[i] for i in [row_lo, row_hi) (arrays indexed by the global row), loss_part =
 *             sum of those row losses / n2; the loss is the sum of loss_part over the ranks.
 *   backward: needs lse of ALL rows (all-gather the slices).  dz_rows (row_hi - row_lo, d) = grad_scale * grad_loss *
 *             d loss / d z_i for the rank's own rows - complete, the P_ji terms of the other ranks' anchors included, so no
 *             gradient exchange for z is needed.  grad_scale: e.g. the world size when the parameter gradients are averaged
 *             over the ranks afterwards.
 * row_lo, row_hi even (partners stay together).
 */
int grafp_ntxent_rows_fwd(const float* z, float* lse, float* row_loss, float* loss_part, int n2, int d, int row_lo, int row_hi,
                          float inv_tau, void* stream);
int grafp_ntxent_rows_bwd(const float* z, const float* lse, const float* grad_loss, float* dz_rows, int n2, int d, int row_lo,
                          int row_hi, float inv_tau, float grad_scale, void* stream);

/*
 * Peak point-cloud front end (SURVEY 8f row 4).  Replaces GPUPeakExtractorv2.forward (peak_extractor.py:56-82): min-max
 * normalisation of the (H, W) log-mel segment, the time / frequency position ramps (torch.linspace(0, 1, W / H)),
 * Conv2d(3 -> F, kh x kw, stride (stride_h, 1), padding (kh / 2, kw / 2)) + ReLU and the reshape to a point cloud,
 * written directly as node rows out[b][n][f], n = oh * W + ow - the layout the encoder's stem consumes.
 *   spec (B, H, W) float32, weight (F, 3, kh, kw), bias (F), out (B, Ho * W, F), Ho = (H + 2 (kh / 2) - kh) / stride_h + 1.
 *   backward: gradients of weight and bias only (the spectrogram has none): `partial` is
 *   grafp_peak_extract_workspace_bytes(B, kh, kw) bytes of scratch (per-segment sums, reduced in a fixed order).
 * F must be 8 (config n_filters), kh and kw odd; else GRAFP_EUNSUPPORTED (the caller then runs the PyTorch modules).
 */
size_t grafp_peak_extract_workspace_bytes(int B, int kh, int kw);
int grafp_peak_extract_fwd(const float* spec, const float* weight, const float* bias, float* out, int B, int H, int W, int F,
                           int kh, int kw, int stride_h, void* stream);
int grafp_peak_extract_bwd(const float* spec, const float* out, const float* grad_out, void* partial, size_t partial_bytes,
                           float* dweight, float* dbias, int B, int H, int W, int F, int kh, int kw, int stride_h, void* stream);

/*
 * Exact flat search: the k nearest database rows of every query in squared L2 distance (faiss IndexFlatL2.search).
 *   grafp_search_prepare: fp16 planes hi / lo (n, d) of rows * 2^12 and sq (n) = |row|^2 (fp32) for the caller's rows
 *     (n, d) float32; called on appended rows through pointer offsets, so a database is prepared once.
 *   grafp_search_fwd: q (n_q, d) float32 against the n_db prepared rows; ids (n_q, k) int64 and dist (n_q, k) float32,
 *     ascending by (dist, id) - equal distances keep the lower id.  dist = (|q|^2 + (-2 q.x)) + |x|^2 in fp32.
 *     The database is cut into key slices searched in parallel and their lists merged; the result does not depend on
 *     the slicing or on the other queries of the batch - for k <= 3 on unit-norm rows up to near-ties: keys whose
 *     distances differ by less than the spread of the rows' |x|^2 (<= 1e-6) may be ordered or picked either way.
 *   Precondition: every database and query row has L2 norm <= 1 + 1e-4 (the fp16 plane split and the selection
 *   thresholds assume it; unit-norm fingerprints satisfy it).  Not checked here.
 *   Envelope: d % 8 == 0 and 64 <= d <= 256, 1 <= k <= 128, k <= n_db, n_q >= 1 (else GRAFP_EUNSUPPORTED / GRAFP_EINVAL).
 *   workspace: grafp_search_workspace_bytes(n_q, n_db, d, k) bytes (0 outside the envelope).  Nothing is allocated and
 *   nothing synchronises; the kernels run on `stream` of the current device.
 */
int grafp_search_prepare(const float* rows, long long n, int d, void* hi, void* lo, float* sq, void* stream);
size_t grafp_search_workspace_bytes(int n_q, int n_db, int d, int k);
int grafp_search_fwd(const float* q, int n_q, const void* hi, const void* lo, const float* sq, int n_db, int d, int k,
                     int64_t* ids, float* dist, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GRAFP_B200_H_ */
