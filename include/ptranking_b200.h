/* ptranking_b200.h -- C ABI of the B200-native PTRanking hot path (libptranking_b200.so).
 *
 * PTRanking has no FFI of its own: its plugin API is a Python class contract
 * (SURVEY.md 8b).  This header is the boundary a maintainer binds from that
 * contract (ctypes stub in INTEGRATION.md): every entry point replaces the
 * PyTorch-eager body of one reference function, cited per declaration
 * (paths relative to the wildltr/ptranking checkout, commit f1d366c).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *     marked "host"; tensors are dense row-major fp32 ([B,n] scores/labels,
 *     [B,n,F] features), int32 for index data.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - no allocation inside the library: the caller passes every output and
 *     workspace buffer; ptrb200_*_workspace_bytes() says how much.  (The one
 *     exception is ptrb200_peer_alloc: memory exported to the other processes
 *     of a node through CUDA IPC has to be a cudaMalloc base.)
 *   - return 0 on success or a negative PTRB200_ERR_* code; nothing throws
 *     across the boundary.  ptrb200_last_error() returns a host string
 *     describing the last failure on the calling thread.
 *   - every launch is asynchronous on `stream`; results are ordered after it.
 */
#ifndef PTRANKING_B200_H
#define PTRANKING_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* every entry point below is exported with default visibility; the rest of the library is hidden */
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define PTRB200_OK               0
#define PTRB200_ERR_INVALID     -1   /* bad argument (null pointer, non-positive size, unknown enum) */
#define PTRB200_ERR_UNSUPPORTED -2   /* size outside what the kernels are built for (see limits below) */
#define PTRB200_ERR_CUDA        -3   /* CUDA runtime / launch failure */
#define PTRB200_ERR_WORKSPACE   -4   /* workspace too small */

#define PTRB200_MAX_LIST_LEN  4096   /* docs per query handled by the per-list kernels */
#define PTRB200_MAX_FF_LAYERS   16   /* linear layers in one stacked feed-forward net */
#define PTRB200_MAX_CUTOFFS     32   /* nDCG cutoffs per call */

typedef void* ptrb200_stream_t;

/* ---- library bookkeeping -------------------------------------------------- */
int                ptrb200_version(void);
const char*        ptrb200_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
unsigned long long ptrb200_launch_count(void);
/* 1 if the current device is compute capability 10.x (the only target built) */
int                ptrb200_device_ok(void);
/* Per-launch CUDA-event timing on the launching stream (bench.py's roofline pass; off by default).
 * ptrb200_timing_report synchronises the recorded events and writes one line per kernel,
 * "name<TAB>launches<TAB>total_ms", into the host buffer, then clears the record. */
int                ptrb200_timing_enable(int on);
int                ptrb200_timing_report(char* buf_host, int buflen);

/* ---- ranking losses: loss value per query + d(sum loss)/d(scores) ---------- */
/* Each call writes loss_per_query[B] (the reference returns their sum) and
 * grad[B,n] = d(sum_b loss_b)/d scores -- the tensor autograd would hand back
 * to the scorer after the reference's `batch_loss.backward()`.
 *
 * `offsets`: NULL for the reference's dense batches (every query has n documents, scores/labels/grad are [B,n]:
 * data_utils.py:683-718).  Non-NULL (device, B+1 int32 prefix offsets) makes the batch RAGGED (SURVEY 8f-2): scores /
 * labels / grad are flat [offsets[B]] arrays, query b owns [offsets[b], offsets[b+1]) and `n` is the longest list of the
 * batch (it sizes the CTA and its shared memory).  Empty lists are allowed and contribute a zero loss. */

/* RankNet.custom_loss_function, ptranking/ltr_adhoc/pairwise/ranknet.py:25-36
 * (+ get_pairwise_comp_probs, ltr_adhoc/util/lambda_utils.py:5-23). */
int ptrb200_ranknet_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                            int B, int n, float sigma, ptrb200_stream_t stream);

/* LambdaRank.custom_loss_function, ptranking/ltr_adhoc/listwise/lambdarank.py:27-56
 * (+ get_delta_ndcg, metric/metric_utils.py:19-45).  Labels must be presorted
 * descending (lambdarank.py:36). */
int ptrb200_lambdarank_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                               int B, int n, float sigma, ptrb200_stream_t stream);

#define PTRB200_NDCG_LOSS1    0
#define PTRB200_NDCG_LOSS2    1
#define PTRB200_NDCG_LOSS2PP  2
/* LambdaLoss.custom_loss_function, ptranking/ltr_adhoc/listwise/lambdaloss.py:73-132.
 * NDCG_Loss1 is evaluated per query (the reference's broadcast only works for B==1). */
int ptrb200_lambdaloss_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                               int B, int n, int k, float sigma, float mu, int loss_type, int presort,
                               ptrb200_stream_t stream);

/* ListNet.custom_loss_function, ptranking/ltr_adhoc/listwise/listnet.py:39. */
int ptrb200_listnet_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                            int B, int n, ptrb200_stream_t stream);

/* ListMLE.custom_loss_function, ptranking/ltr_adhoc/listwise/listmle.py:83-97, with the
 * tie-shuffled ordering `perm[B,n]` (int32 doc positions within each query's own list, labels descending) supplied. */
int ptrb200_listmle_fwd_bwd(const float* scores, const int32_t* perm, const int32_t* offsets, float* grad, float* loss_per_query,
                            int B, int n, ptrb200_stream_t stream);

/* arg_shuffle_ties, ptranking/ltr_adhoc/util/sampling_utils.py:13-28: perm[B,n] orders each
 * row's labels descending with ties broken uniformly at random (Philox4x32-10 keyed by
 * (seed, offset, b, doc); not the torch RNG stream). */
int ptrb200_shuffle_ties_perm(const float* labels, const int32_t* offsets, int32_t* perm, int B, int n,
                              uint64_t seed, uint64_t offset, ptrb200_stream_t stream);

/* ApproxNDCG.custom_loss_function, ptranking/ltr_adhoc/listwise/approxNDCG.py:83-101
 * (+ get_approx_ranks :19-28, approxNDCG_loss :45-62, Robust_Sigmoid base/utils.py:57-92).
 * batch_coupled != 0 keeps the reference's [B]/[B,1] broadcast (every query scaled by
 * sum_a 1/iDCG_a, :58-61).  scratch: B+1 floats. */
int ptrb200_approxndcg_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                               float* scratch, int B, int n, float alpha, int presort, int batch_coupled,
                               ptrb200_stream_t stream);

/* ---- sibling losses (SURVEY 8f-4): same contract as above, `offsets` included ---------------- */

/* RankMSE.custom_loss_function, ptranking/ltr_adhoc/pointwise/rank_mse.py:13-22: the MEAN over queries of the per-query
 * summed squared error; loss_per_query[b] already carries the 1/B so that their sum is the reference's value. */
int ptrb200_rankmse_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                            int B, int n, ptrb200_stream_t stream);
/* RankCosine.custom_loss_function, ptranking/ltr_adhoc/listwise/rank_cosine.py:33 (nn.CosineSimilarity(dim=1), eps 1e-8). */
int ptrb200_rankcosine_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                               int B, int n, ptrb200_stream_t stream);
/* STListNet.custom_loss_function, ptranking/ltr_adhoc/listwise/st_listnet.py:41-49.  unif (optional, same layout as
 * scores) supplies the U[0,1) draw behind the Gumbel noise; NULL draws it from Philox4x32-10 keyed by (seed, offset, doc). */
int ptrb200_stlistnet_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, const float* unif,
                              float* grad, float* loss_per_query, int B, int n, float temperature,
                              uint64_t seed, uint64_t offset, ptrb200_stream_t stream);
/* SoftRank.custom_loss_function (metric nDCG), ptranking/ltr_adhoc/listwise/softrank.py:46-72; labels presorted
 * descending (:40).  top_k <= 0 means the whole list (the reference's top_k=None). */
int ptrb200_softrank_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                             int B, int n, float delta, int top_k, ptrb200_stream_t stream);
/* sinkstep, ptranking/ltr_adhoc/listwise/wassrank/pytorch_wasserstein.py:132-224 (the reference's one CUDA kernel,
 * CPU form :277-291): log_v[b][j] = log_nu[b][j] - logsumexp_i(-dist[i][j]/lambda + log_u[b][i]).
 * dist[d1,d2], log_nu[B,d2], log_u[B,d1], log_v[B,d2]. */
int ptrb200_sinkstep(const float* dist, const float* log_nu, const float* log_u, float* log_v,
                     int B, int d1, int d2, float lambda, ptrb200_stream_t stream);

/* WassRank.custom_loss_function, mode 'SinkhornOT': ptranking/ltr_adhoc/listwise/wassrank/wassRank.py:43-86 with
 * OldSinkhornOT (pytorch_wasserstein.py:323-394), the cost matrices of get_explicit_cost_mat and the histograms of
 * get_normalized_histograms (wasserstein_cost_mat.py:47-244).  One CTA per query; the [n,n] cost matrix is rebuilt in
 * registers from the labels and never stored.  The Sinkhorn updates run as row-wise log-sum-exps (finite in fp32 where
 * the reference's per-vector stabilisation underflows).  loss_per_query[b] and the gradient carry 1/B_total (the
 * reference's .mean(0) over the batch); B_total is the whole batch's query count, which a launch over one length bucket
 * (B queries) needs passed in.  grad is the reference's envelope gradient (lam * log_u centred twice) chained through
 * the histogram map.  gain_base, non_rele_gap, var_penalty: the 'eg' cost's parameters. */
#define PTRB200_WASS_COST_EG   0   /* 'eg'  explicit grouping of the labels (torch_cost_mat_group) */
#define PTRB200_WASS_COST_P1   1   /* 'p1'  |i - j| over positions */
#define PTRB200_WASS_COST_P2   2   /* 'p2'  (i - j)^2 */
#define PTRB200_WASS_COST_DG   3   /* 'dg'  |delta (2^y - 1)| */
#define PTRB200_WASS_COST_DDG  4   /* 'ddg' |delta (2^y - 1)| * |delta 1/log2(rank + 2)| */
#define PTRB200_WASS_SMOOTH_ST 0   /* 'ST' (norm_type 'BothST'): softmax of labels and of scores */
#define PTRB200_WASS_SMOOTH_NG 1   /* 'NG': normalised gains 2^y - 1; scores over their sum, shifted by the min if <= 0 */
int ptrb200_wassrank_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                             int B, int n, int B_total, int cost_type, int smooth_type, float lam, int sh_itr,
                             float gain_base, float non_rele_gap, float var_penalty, ptrb200_stream_t stream);

/* deterministic (fixed-order) sum of n floats into out[0] -- the `torch.sum` over queries
 * that ends every reference loss (e.g. lambdarank.py:56). */
int ptrb200_sum_f32(const float* x, float* out, int n, ptrb200_stream_t stream);

/* ---- evaluation metric ------------------------------------------------------ */
/* Evaluator.ndcg_at_ks ranking + torch_ndcg_at_ks, ptranking/base/ranker.py:67-95 and
 * metric/adhoc/adhoc_metric.py:219-260.  out[B,nks]; cutoffs > n yield 0 (the reference's
 * zero padding).  order[B,n] (optional, may be NULL) receives the doc indices in predicted
 * rank order (score descending, index ascending among equal scores).  ks: host pointer.  offsets: as for the losses. */
int ptrb200_ndcg_at_ks(const float* scores, const float* labels, const int32_t* offsets, const int32_t* ks_host, int nks,
                       float* out, int32_t* order, int B, int n, int presort, ptrb200_stream_t stream);

/* adhoc_performance_at_ks, ptranking/base/ranker.py:202-263 with torch_ndcg_at_ks / torch_nerr_at_ks / torch_ap_at_ks /
 * torch_precision_at_ks (metric/adhoc/adhoc_metric.py:36-64, 95-128, 132-193, 243-260): out[B][4][nks] in the order
 * nDCG, nERR, AP, P from one in-CTA sort per query; cutoffs > n yield 0; max_label as the evaluator passes it. */
int ptrb200_adhoc_metrics_at_ks(const float* scores, const float* labels, const int32_t* offsets, const int32_t* ks_host, int nks,
                                float* out, int B, int n, int presort, float max_label, ptrb200_stream_t stream);

/* ---- input side: per-query feature scaling -------------------------------------------------- */
/* sklearn StandardScaler().fit_transform applied per query as the loader does for MSLR-WEB / Istella
 * (ptranking/data/data_utils.py:482-487; selection :205-218): out = (x - mean_q) / std_q per feature column with the
 * population standard deviation, statistics in float64, constant columns divided by 1.  X/out: [B,n,F] dense, or flat
 * [offsets[B], F] with per-query offsets (ragged).  clip != 0 first clamps features at clip_max (the ISTELLA_MAX clip,
 * :484-485).  In-place (out == X) is allowed. */
int ptrb200_standard_scale(const float* X, const int32_t* offsets, float* out, int B, int n, int F,
                           int clip, float clip_max, ptrb200_stream_t stream);

/* ---- stacked feed-forward scorer (pointwise MLP; also the head/tail nets of listsf) ---- */
/* get_stacked_FFNet, ptranking/base/utils.py:288-356; PointNeuralRanker.forward,
 * base/point_ranker.py:45-55; LTRBatchNorm / LTRBatchNorm2, base/utils.py:201-282;
 * get_AF, base/utils.py:101-143. */
#define PTRB200_AF_NONE   0
#define PTRB200_AF_RELU   1   /* 'R'  */
#define PTRB200_AF_GELU   2   /* 'GE' exact erf */
#define PTRB200_AF_SIGM   3   /* 'S'  */
#define PTRB200_AF_TANH   4   /* 'T'  */
#define PTRB200_AF_CELU   5   /* 'CE' alpha=1 */
#define PTRB200_AF_ELU    6   /* 'E'  alpha=1 */
#define PTRB200_AF_LRELU  7   /* 'LR' slope 0.01 */
#define PTRB200_AF_SELU   8   /* 'SE' */

#define PTRB200_NORM_NONE 0
#define PTRB200_NORM_BN   1   /* LTRBatchNorm: statistics over all B*n rows, train and eval */
#define PTRB200_NORM_BN2  2   /* LTRBatchNorm2: statistics per query */

#define PTRB200_MATH_SIMT   0   /* fp32 FMA on the SIMT pipes (any shape)                              */
#define PTRB200_MATH_3XTF32 1   /* tcgen05 kind::tf32, error-compensated 3-pass split: fp32-equivalent */
#define PTRB200_MATH_TF32   2   /* tcgen05 kind::tf32, single pass (10-bit mantissa operands)           */
#define PTRB200_MATH_BF16   3   /* every GEMM operand (features, activations, weights, gradients) rounded to bf16
                                   (round-to-nearest-even), products exact, fp32 accumulation: the numerics of a bf16
                                   tensor-core GEMM, issued as one kind::tf32 pass (bf16 values are tf32 values);
                                   tensors stay fp32 in memory.  Needs tensor-core-eligible widths (no SIMT fallback) */

typedef struct ptrb200_ffnet {
    int num_linear;                        /* linear layers, output layer included            */
    int dims[PTRB200_MAX_FF_LAYERS + 1];   /* dims[0]=in features ... dims[num_linear]=out    */
    int act_hidden;                        /* PTRB200_AF_* after every hidden layer           */
    int act_tail;                          /* PTRB200_AF_* after the last layer, AF_NONE when apply_tl_af is false */
    int norm;                              /* PTRB200_NORM_* on every layer that has an activation */
    int norm_affine;                       /* bn_affine                                       */
    float dropout_p;                       /* Dropout before every hidden Linear; 0 disables  */
    int math_mode;                         /* PTRB200_MATH_*: the TF32 modes fall back to SIMT when a width is not a multiple of 4 */
    int sync_bn;                           /* != 0 with PTRB200_NORM_BN: the batch statistics (forward moments and the two backward
                                              sums) span every data-parallel rank -- the library folds its partial sums into
                                              2*C+1 doubles per layer and asks the hook below to all-reduce them (SUM) */
    /* parameters, one pointer per linear layer l = 0..num_linear-1 (nn.Linear layout [out,in]) */
    const float* weight[PTRB200_MAX_FF_LAYERS];
    const float* bias[PTRB200_MAX_FF_LAYERS];
    /* norm parameters per layer (NULL where absent): BN: gamma/beta = bn.weight/bn.bias when affine;
     * BN2: gamma/beta always, plus aff_w/aff_b when affine */
    const float* gamma[PTRB200_MAX_FF_LAYERS];
    const float* beta[PTRB200_MAX_FF_LAYERS];
    const float* aff_w[PTRB200_MAX_FF_LAYERS];
    const float* aff_b[PTRB200_MAX_FF_LAYERS];
} ptrb200_ffnet;

typedef struct ptrb200_ffnet_grads {       /* same layout as the parameter pointers; written (not accumulated) */
    float* weight[PTRB200_MAX_FF_LAYERS];
    float* bias[PTRB200_MAX_FF_LAYERS];
    float* gamma[PTRB200_MAX_FF_LAYERS];
    float* beta[PTRB200_MAX_FF_LAYERS];
    float* aff_w[PTRB200_MAX_FF_LAYERS];
    float* aff_b[PTRB200_MAX_FF_LAYERS];
} ptrb200_ffnet_grads;

/* Host hook for the two things a data-parallel caller has to do in the middle of a forward / backward call; the library
 * itself holds no communicator.  Called on the launching host thread, between kernel launches on `stream`:
 *   PTRB200_HOOK_ALLREDUCE_F64      all-reduce (SUM) `count` doubles at device pointer `ptr`, ordered on `stream`
 *                                   (sync_bn statistics of layer `layer`: 2*C sums + the row count)
 *   PTRB200_HOOK_LAYER_GRADS_READY  every parameter gradient of layer `layer` has been enqueued on `stream`
 *                                   (ptr NULL, count 0): the caller may start its gradient all-reduce for that layer
 * Return 0; anything else aborts the call with PTRB200_ERR_INVALID.  fn == NULL removes the hook. */
#define PTRB200_HOOK_ALLREDUCE_F64      1
#define PTRB200_HOOK_LAYER_GRADS_READY  2
typedef int (*ptrb200_hook_fn)(int what, int layer, void* ptr, int64_t count, void* stream, void* user);
int ptrb200_set_hook(ptrb200_hook_fn fn, void* user);

/* Batch shape of the three calls below.  Dense (the reference's contract): B queries of n documents, X is [B,n,dims[0]],
 * offsets = NULL, total_rows = 0.  Ragged (SURVEY 8f-2): B queries cut out of total_rows documents by the device prefix
 * offsets[B+1], n = the longest list, X is [total_rows, dims[0]].  Batch-level BN and norm-free nets treat a ragged batch as
 * one long list; per-query BN2 (LTRBatchNorm2) normalises every query over its own documents. */

/* bytes of activation workspace the forward pass fills for the backward pass */
int64_t ptrb200_ffnet_workspace_bytes(const ptrb200_ffnet* net, int B, int n, int total_rows);

/* `training` argument of the two calls below: bit 0 = training mode (dropout active); bit 1 (forward only) tells
 * ptrb200_ffnet_forward that no backward call will follow, so the by-products the backward pass reads are not written. */
#define PTRB200_FFNET_TRAINING 1
#define PTRB200_FFNET_FORWARD_ONLY 2
/* forward: X[B,n,dims[0]] -> out[B,n,dims[last]].  `workspace` keeps pre-activations and
 * statistics for ptrb200_ffnet_backward.  dropout uses Philox keyed by (seed, offset). */
int ptrb200_ffnet_forward(const ptrb200_ffnet* net, const float* X, float* out, void* workspace,
                          int64_t workspace_bytes, int B, int n, const int32_t* offsets, int total_rows, int training,
                          uint64_t seed, uint64_t offset, ptrb200_stream_t stream);

/* backward: dOut[B,n,dims[last]] -> parameter grads (+ dX[B,n,dims[0]] when dX != NULL).
 * Must follow a forward call with the same net/X/workspace/seed/offset. */
int ptrb200_ffnet_backward(const ptrb200_ffnet* net, const ptrb200_ffnet_grads* grads, const float* X,
                           const float* dOut, float* dX, void* workspace, int64_t workspace_bytes,
                           int B, int n, const int32_t* offsets, int total_rows, int training, uint64_t seed, uint64_t offset,
                           ptrb200_stream_t stream);

/* ---- optimizer step ---------------------------------------------------------------------- */
/* torch.optim.Adam.step() (ranker.py:512-525 -> config_optimizer; defaults betas=(0.9,0.999), eps=1e-8) over flat fp32
 * buffers of `count` elements with identical layouts: parameters, gradients, first and second moments.  `step` is the
 * 1-based step count (bias correction).  weight_decay is added to the gradient (torch's L2 form).  16-byte aligned. */
int ptrb200_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t count,
                      double lr, double beta1, double beta2, double eps, double weight_decay, int step,
                      ptrb200_stream_t stream);

/* torch.optim.Adagrad.step() (the list scorer's default optimizer, ltr_adhoc/eval/parameter.py:157-162; PyTorch defaults
 * lr_decay=0, eps=1e-10, initial_accumulator_value=0) and torch.optim.RMSprop.step() (alpha=0.99, eps=1e-8, momentum=0,
 * centered=False) as configured at ranker.py:517-520, over the same flat fp32 layout with one state buffer. */
int ptrb200_adagrad_step(float* param, const float* grad, float* state_sum, int64_t count,
                         double lr, double lr_decay, double eps, double weight_decay, int step,
                         ptrb200_stream_t stream);
int ptrb200_rmsprop_step(float* param, const float* grad, float* square_avg, int64_t count,
                         double lr, double alpha, double eps, double weight_decay,
                         ptrb200_stream_t stream);

/* Ragged <-> padded layout change for the list scorer (no counterpart: the reference batches equal-length lists only,
 * data_utils.py:683-742): padded[b, r, :] = flat[offsets[b] + r, :] for r < len_b, else 0; unpad is the inverse gather.
 * offsets: int32[B+1] prefix offsets, n_max: padded list length, F: row width (1 for score vectors). */
int ptrb200_pad_lists(const float* flat, const int32_t* offsets, float* padded, int B, int n_max, int F,
                      ptrb200_stream_t stream);
int ptrb200_unpad_lists(const float* padded, const int32_t* offsets, float* flat, int B, int n_max, int F,
                        ptrb200_stream_t stream);

/* ---- data-parallel gradient exchange over NVLink peer memory ------------------------------ */
/* The reference has no distributed code.  One process per GPU (torchrun); the sum of the ranks' flat gradient buffers
 * that precedes optimizer.step() in a data-parallel run is folded INTO the step kernel: every rank maps the other ranks'
 * buffers (CUDA IPC), the kernel synchronises through system-scope flags and reads the W buffers directly over NVLink
 * (see csrc/optim.cu).  The library exports / maps the memory; exchanging the 64-byte handles between the processes is
 * the caller's business (ptranking_b200.dist does it through torch.distributed).
 * ptrb200_peer_alloc is the ONE place where the library allocates device memory (CUDA IPC needs a cudaMalloc base). */
#define PTRB200_MAX_PEERS 16
typedef struct ptrb200_peer_group {
    int world, rank;
    const float* grads[PTRB200_MAX_PEERS];   /* rank r's gradient buffer of this step, as mapped into THIS process (own included) */
    uint32_t* flags[PTRB200_MAX_PEERS];      /* rank r's flag pad: `world` uint32, zero at allocation, never reset */
    uint32_t epoch;                          /* 1, 2, 3, ... : one value per exchange, the same on every rank */
    int* error;                              /* optional device int (own memory): 1 + r if rank r never arrived within 4 s */
} ptrb200_peer_group;
int ptrb200_peer_alloc(int64_t bytes, void** dev_ptr, unsigned char* handle64);   /* cudaMalloc + zero + export */
int ptrb200_peer_open(const unsigned char* handle64, void** dev_ptr);             /* map another process's export */
int ptrb200_peer_close(void* dev_ptr);
int ptrb200_peer_free(void* dev_ptr);
/* out[count] = sum over ranks of grads[r][0..count) -- the bare exchange (rank order 0..W-1 on every rank) */
int ptrb200_peer_allreduce_sum(const ptrb200_peer_group* grp, float* out, int64_t count, ptrb200_stream_t stream);
/* ptrb200_adam_step / adagrad_step / rmsprop_step with grad = that sum, in one launch */
int ptrb200_adam_step_peer(const ptrb200_peer_group* grp, float* param, float* exp_avg, float* exp_avg_sq, int64_t count,
                           double lr, double beta1, double beta2, double eps, double weight_decay, int step,
                           ptrb200_stream_t stream);
int ptrb200_adagrad_step_peer(const ptrb200_peer_group* grp, float* param, float* state_sum, int64_t count,
                              double lr, double lr_decay, double eps, double weight_decay, int step,
                              ptrb200_stream_t stream);
int ptrb200_rmsprop_step_peer(const ptrb200_peer_group* grp, float* param, float* square_avg, int64_t count,
                              double lr, double alpha, double eps, double weight_decay,
                              ptrb200_stream_t stream);

/* ---- multi-head self-attention list scorer ------------------------------------------------ */
/* MultiheadAttention.forward, ptranking/base/list_ranker.py:226-248: for every (query b, head h)
 * O = dropout(softmax(Q K^T / sqrt(D))) V, flash-style (no [n,n] tensor in HBM).  Q,K,V,O: [B,n,H*D] with head h
 * in columns [h*D,(h+1)*D) (the reference's view/permute, :222-224, :251).  LSE[B,H,n] is kept for backward. */
int ptrb200_attention_fwd(const float* Q, const float* K, const float* V, float* O, float* LSE,
                          int B, int n, int H, int D, float dropout_p, uint64_t seed, uint64_t offset,
                          ptrb200_stream_t stream);
/* autograd of the above; scratch: B*H*n floats. */
int ptrb200_attention_bwd(const float* Q, const float* K, const float* V, const float* O, const float* dO, const float* LSE,
                          float* dQ, float* dK, float* dV, float* scratch,
                          int B, int n, int H, int D, float dropout_p, uint64_t seed, uint64_t offset,
                          ptrb200_stream_t stream);
/* Tensor-core variant of the two calls above (same maths, same dropout stream): every contraction is a batched
 * tcgen05 kind::tf32 GEMM (passes = 3: 3xTF32 split, fp32-grade; 1: plain TF32); the attention matrix
 * P[B*H,n,n] is materialised in HBM and kept for the backward pass.
 * scratch: ptrb200_attention_tc_workspace_floats(B,n,H,D,backward) floats. */
int64_t ptrb200_attention_tc_workspace_floats(int B, int n, int H, int D, int backward);
int ptrb200_attention_tc_fwd(const float* Q, const float* K, const float* V, float* O, float* P_out, float* scratch,
                             int B, int n, int H, int D, float dropout_p, uint64_t seed, uint64_t offset, int passes,
                             ptrb200_stream_t stream);
int ptrb200_attention_tc_bwd(const float* Q, const float* K, const float* V, const float* P, const float* dO,
                             float* dQ, float* dK, float* dV, float* scratch,
                             int B, int n, int H, int D, float dropout_p, uint64_t seed, uint64_t offset, int passes,
                             ptrb200_stream_t stream);
/* The same two calls over row-pitched operands: ld_qkv = floats between consecutive documents of Q, K and V (and of dQ,
 * dK, dV), ld_o = the same for O and dO; 0 = packed (H*D).  With Q|K|V side by side in one [B,n,3*H*D] tensor -- the
 * output of ONE 136->408 projection instead of the reference's three (list_ranker.py:233-235) -- the call takes
 * Q = qkv, K = qkv + H*D, V = qkv + 2*H*D, ld_qkv = 3*H*D, and the backward call fills the matching gradient tensor.
 * key_lens (forward; NULL = every list has n documents): int32[B], query b attends to its first key_lens[b] documents only
 * -- a ragged batch padded to n (ptrb200_pad_lists); masked probabilities are exactly 0, so the backward call needs nothing. */
int ptrb200_attention_tc_fwd_ld(const float* Q, const float* K, const float* V, float* O, float* P_out, float* scratch,
                                int B, int n, int H, int D, int ld_qkv, int ld_o, const int32_t* key_lens, float dropout_p,
                                uint64_t seed, uint64_t offset, int passes, ptrb200_stream_t stream);
int ptrb200_attention_tc_bwd_ld(const float* Q, const float* K, const float* V, const float* P, const float* dO,
                                float* dQ, float* dK, float* dV, float* scratch,
                                int B, int n, int H, int D, int ld_qkv, int ld_o, float dropout_p, uint64_t seed,
                                uint64_t offset, int passes, ptrb200_stream_t stream);
/* LayerNorm.forward, ptranking/base/list_ranker.py:165-174: y = a_2 (x - mean) / (std_unbiased + eps) + b_2 per row;
 * mean/std[rows] are kept for backward. */
int ptrb200_layernorm_fwd(const float* x, const float* a2, const float* b2, float* y, float* mean, float* stdv,
                          int rows, int F, float eps, ptrb200_stream_t stream);
/* scratch: 297*2*F floats. */
int ptrb200_layernorm_bwd(const float* x, const float* a2, const float* dy, const float* mean, const float* stdv,
                          float* dx, float* da2, float* db2, float* scratch,
                          int rows, int F, float eps, ptrb200_stream_t stream);
/* elementwise glue of the encoder variants (list_ranker.py:138-149, 357-373) and of PositionwiseFeedForward (:269-277):
 * op 0: a+b   1: (a+1)*b (DASALC latent cross)   2: a*b   3: relu(a)   4: b>0 ? a : 0   5: dropout(a)   6: a*(b+1)
 * 7: a*b[0] (b = one device scalar: the incoming gradient of the summed batch loss, e.g. lambdarank.py:56-59)
 * 8 / 9: act(a) / act'(a) of get_AF (base/utils.py:101-143) with the PTRB200_AF_* code passed in `seed` -- the scorer's
 *        own activation routine, exposed so its accuracy can be tested element by element */
#define PTRB200_EW_ADD 0
#define PTRB200_EW_LATENT_CROSS 1
#define PTRB200_EW_MUL 2
#define PTRB200_EW_RELU 3
#define PTRB200_EW_RELU_BWD 4
#define PTRB200_EW_DROPOUT 5
#define PTRB200_EW_SCALE_ADD1 6
#define PTRB200_EW_MUL_SCALAR 7
#define PTRB200_EW_ACT 8
#define PTRB200_EW_ACT_GRAD 9
int ptrb200_elementwise(int op, const float* a, const float* b, float* out, int64_t count,
                        float dropout_p, uint64_t seed, uint64_t offset, ptrb200_stream_t stream);

/* ---- tensor-core GEMM building block ---------------------------------------------------- */
/* C[M,N] = A[M,K] * B[N,K]^T in fp32 through tcgen05.mma kind::tf32 with TMEM accumulation
 * (the contraction of nn.Linear: torch.nn.functional.linear as called by every ff_* layer of
 * get_stacked_FFNet, ptranking/base/utils.py:302,320).  passes = 1: plain TF32 operands;
 * passes = 3: error-compensated 3xTF32 (fp32-equivalent accuracy).  N <= 256. */
int ptrb200_tc_gemm_nt(const float* A, const float* B, float* C, int M, int N, int K, int passes,
                       ptrb200_stream_t stream);

/* dW[N,K] = dZ[rows,N]^T * P[rows,K] (the weight gradient autograd forms for nn.Linear) with both operands
 * consumed MN-major by tcgen05.mma; partials: 296*N*K floats of scratch.  N <= 128, K <= 256, K % 4 == 0. */
int ptrb200_tc_wgrad(const float* dZ, const float* P, float* dW, float* partials, int rows, int N, int K, int passes,
                     ptrb200_stream_t stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* PTRANKING_B200_H */
