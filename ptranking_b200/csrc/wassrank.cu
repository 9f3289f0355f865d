// wassrank.cu -- WassRank's SinkhornOT loss (entropic optimal transport between the score and label histograms of a query)
// and the gradient the reference's backward hands the scores, one CTA per query.
//
// Reference functions replaced (wildltr/ptranking @ f1d366c):
//   WassRank.custom_loss_function  ptranking/ltr_adhoc/listwise/wassrank/wassRank.py:43-86 (mode 'SinkhornOT')
//   OldSinkhornOT                  ptranking/ltr_adhoc/listwise/wassrank/pytorch_wasserstein.py:323-394
//   get_explicit_cost_mat, get_normalized_histograms
//                                  ptranking/ltr_adhoc/listwise/wassrank/wasserstein_cost_mat.py:47-244
//
// The cost matrix C[n,n] is never stored: every C_ij is rebuilt in registers from per-document values in shared memory
// (gain-derived value, rank discount, position).  The Sinkhorn updates are the reference's, written as row-wise
// log-sum-exps with each row's own maximum:
//     log_v_j = log nu_j - LSE_i(-C_ij/lam + log_u_i),    log_u_i = log mu_i - LSE_j(-C_ij/lam + log_v_j).
// The reference stabilises with one maximum per vector instead (pytorch_wasserstein.py:344-349); in fp32 most of
// exp(-C/lam) underflows at its default lam = 0.1, whole columns of K^T u vanish and log 0 turns into inf - inf = NaN.
// Every cost type is symmetric (C_ij and C_ji are the same fp32 value), so both half-steps walk one row per thread.
#include "losses_common.cuh"

namespace ptrb200 {

// cost types (PTRB200_WASS_COST_*)
enum { WC_EG = 0, WC_P1 = 1, WC_P2 = 2, WC_DG = 3, WC_DDG = 4 };

// C_ij from the per-document values a (gain-derived) and d (rank discount, 'ddg' only):
//   eg  (torch_cost_mat_group, :84-111): a = gain_base^y - 1, or -non_rele_gap where that is < 1; |a_i - a_j|, values
//        below 1 become var_penalty; the diagonal is var_penalty - var_penalty = 0
//   p1 / p2 (torch_cost_mat_dist, :47-60): |i - j| and |i - j|^2 over 1-based positions (exact integers in fp32)
//   dg  (get_delta_gains, :63-81): |a_i - a_j| with a = 2^y - 1
//   ddg: |a_i - a_j| * |d_i - d_j| with d = 1 / log2(rank + 2), rank 0-based
template <int COST>
static __device__ __forceinline__ float wass_cost(int i, int j, float ai, float aj, float di, float dj, float var_penalty) {
    if (COST == WC_EG) {
        const float c = fabsf(ai - aj);
        return i == j ? 0.0f : (c < 1.0f ? var_penalty : c);
    } else if (COST == WC_P1) {
        return fabsf((float)(i + 1) - (float)(j + 1));
    } else if (COST == WC_P2) {
        const float c = fabsf((float)(i + 1) - (float)(j + 1));
        return c * c;
    } else if (COST == WC_DG) {
        return fabsf(ai - aj);
    } else {
        return fabsf(ai - aj) * fabsf(di - dj);
    }
}

// online log-sum-exp: -inf terms are skipped, a NaN term makes the result NaN (as the reference's matrix products do)
static __device__ __forceinline__ void lse_add(float& m, float& s, float v) {
    if (!(v <= m)) { s = s * expf(m - v) + 1.0f; m = v; }
    else if (v > -INFINITY) s += expf(v - m);
}
static __device__ __forceinline__ float lse_final(float m, float s) { return m == -INFINITY ? -INFINITY : m + logf(s); }

// One Sinkhorn half-step over the rows this thread owns: out_i = log_h_i - LSE_j(-C_ij/lam + in_j).
template <int COST>
static __device__ __forceinline__ void sinkhorn_half(const float* a, const float* dsc, const float* in, const float* log_h,
                                                     float* out, int n, float lam, float var_penalty) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float ai = a[i], di = dsc[i];
        float m = -INFINITY, s = 0.0f;
        for (int j = 0; j < n; ++j) {
            const float c = wass_cost<COST>(i, j, ai, a[j], di, dsc[j], var_penalty);
            lse_add(m, s, __fdiv_rn(-c, lam) + in[j]);       // -cost / lam (pytorch_wasserstein.py:334), then the potential
        }
        out[i] = log_h[i] - lse_final(m, s);
    }
}

template <int COST>
__global__ void wassrank_kernel(const float* __restrict__ scores, const float* __restrict__ labels, const int32_t* __restrict__ offsets,
                                float* __restrict__ grad, float* __restrict__ loss_q, int n_uniform, int smooth_ng,
                                float lam, int sh_itr, float gain_base, float non_rele_gap, float var_penalty, float B_total) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* a = reinterpret_cast<float*>(smem_raw);
    float* dsc = a + n_uniform;
    float* lmu = dsc + n_uniform;      // log mu (prediction histogram)
    float* lnu = lmu + n_uniform;      // log nu (label histogram)
    float* lu = lnu + n_uniform;
    float* lv = lu + n_uniform;
    float* red = lv + n_uniform;
    const int b = blockIdx.x;
    const ListSpan sp = list_span(offsets, b, n_uniform);
    const int n = sp.n;
    if (n == 0) { if (threadIdx.x == 0) loss_q[b] = 0.0f; return; }
    const float* s = scores + sp.base;
    const float* y = labels + sp.base;

    // ---- per-document cost values ----
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float av = 0.0f, dv = 0.0f;
        if (COST == WC_EG) {
            const float g = powf(gain_base, y[i]) - 1.0f;
            av = g < 1.0f ? -non_rele_gap : g;
        } else if (COST == WC_DG || COST == WC_DDG) {
            av = powf(2.0f, y[i]) - 1.0f;
        }
        if (COST == WC_DDG) dv = __fdiv_rn(1.0f, (float)log2((double)i + 2.0));    // fp32 log2, correctly rounded
        a[i] = av; dsc[i] = dv;
    }

    // ---- histograms (wasserstein_cost_mat.py:142-246; the 'S' tail rescaling of :196-199 never runs, TL_AF is None) ----
    float smin = 0.0f, tsum = 0.0f, ms = -INFINITY, ss = 0.0f;
    if (!smooth_ng) {
        // nu = softmax(labels), mu = softmax(scores), both kept as log-softmax
        float my = -INFINITY;
        for (int i = threadIdx.x; i < n; i += blockDim.x) { my = fmaxf(my, y[i]); ms = fmaxf(ms, s[i]); }
        my = block_max(my, red);
        ms = block_max(ms, red);
        float sy = 0.0f;
        for (int i = threadIdx.x; i < n; i += blockDim.x) { sy += expf(y[i] - my); ss += expf(s[i] - ms); }
        sy = block_sum(sy, red);
        ss = block_sum(ss, red);
        const float ly = logf(sy), ls = logf(ss);
        for (int i = threadIdx.x; i < n; i += blockDim.x) { lnu[i] = (y[i] - my) - ly; lmu[i] = (s[i] - ms) - ls; }
    } else {
        // nu = (2^y - 1) / sum (the _GN form with its default base 2); mu = s / sum(s) if min(s) > 0 else
        // (s - min) / sum(s - min), min over the query
        float gy = 0.0f, mn = INFINITY;
        for (int i = threadIdx.x; i < n; i += blockDim.x) { gy += powf(2.0f, y[i]) - 1.0f; mn = fminf(mn, s[i]); }
        gy = block_sum(gy, red);
        smin = -block_max(-mn, red);
        const bool shift = !(smin > 0.0f);
        float ts = 0.0f;
        for (int i = threadIdx.x; i < n; i += blockDim.x) ts += shift ? s[i] - smin : s[i];
        tsum = block_sum(ts, red);
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            lnu[i] = logf(__fdiv_rn(powf(2.0f, y[i]) - 1.0f, gy));
            lmu[i] = logf(__fdiv_rn(shift ? s[i] - smin : s[i], tsum));
        }
    }
    const float init = (float)-log((double)n);              // -np.log(n) stored into fp32 (pytorch_wasserstein.py:340-341)
    for (int i = threadIdx.x; i < n; i += blockDim.x) { lu[i] = init; lv[i] = init; }
    __syncthreads();

    // ---- Sinkhorn ----
    for (int it = 0; it < sh_itr; ++it) {
        sinkhorn_half<COST>(a, dsc, lu, lnu, lv, n, lam, var_penalty);
        __syncthreads();
        sinkhorn_half<COST>(a, dsc, lv, lmu, lu, n, lam, var_penalty);
        __syncthreads();
    }

    // ---- loss: sum_i exp(log_u_i + LSE_{j: C_ij > 0}(log C_ij - C_ij/lam + log_v_j)), the reference's log(KM v) ----
    float part = 0.0f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float ai = a[i], di = dsc[i];
        float m = -INFINITY, sm = 0.0f;
        for (int j = 0; j < n; ++j) {
            const float c = wass_cost<COST>(i, j, ai, a[j], di, dsc[j], var_penalty);
            if (c > 0.0f) lse_add(m, sm, logf(c) + __fdiv_rn(-c, lam) + lv[j]);
            else if (c != c) lse_add(m, sm, c);
        }
        part += expf(lu[i] + lse_final(m, sm));
    }
    part = block_sum(part, red);
    if (threadIdx.x == 0) loss_q[b] = __fdiv_rn(part, B_total);

    // ---- gradient: d/d mu = lam * log_u centred twice, over the batch size (:371-380); then through the histogram map ----
    const float nf = (float)n;
    const bool shift = smooth_ng && !(smin > 0.0f);
    float acc = 0.0f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) acc += lu[i] * lam;
    const float mean1 = __fdiv_rn(block_sum(acc, red), nf);
    acc = 0.0f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) acc += lu[i] * lam - mean1;
    const float mean2 = __fdiv_rn(block_sum(acc, red), nf);
    float dot = 0.0f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float g = __fdiv_rn((lu[i] * lam - mean1) - mean2, B_total);
        const float mu = smooth_ng ? __fdiv_rn(shift ? s[i] - smin : s[i], tsum) : __fdiv_rn(expf(s[i] - ms), ss);
        lv[i] = g;                                            // lv is free now: it holds d loss / d mu
        lmu[i] = mu;                                          // and lmu mu itself
        dot += mu * g;
    }
    dot = block_sum(dot, red);
    if (!smooth_ng) {
        // softmax backward: mu * (g - <mu, g>)
        for (int i = threadIdx.x; i < n; i += blockDim.x) grad[sp.base + i] = lmu[i] * (lv[i] - dot);
        return;
    }
    // t / sum(t) backward: (g - <mu, g>) / sum(t); with t = s - min, the min's share -sum_k d/dt_k goes to the tied
    // minima in equal parts (ATen's full min reduction)
    float gsum = 0.0f, cnt = 0.0f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float gt = __fdiv_rn(lv[i] - dot, tsum);
        lv[i] = gt;
        gsum += gt;
        cnt += s[i] == smin ? 1.0f : 0.0f;
    }
    if (shift) { gsum = block_sum(gsum, red); cnt = block_sum(cnt, red); }
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        grad[sp.base + i] = (shift && s[i] == smin) ? lv[i] - __fdiv_rn(gsum, cnt) : lv[i];
}

template <int COST>
static int launch_wassrank(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_q,
                           int B, int n, int smooth_ng, float lam, int sh_itr, float gain_base, float non_rele_gap,
                           float var_penalty, float B_total, ptrb200_stream_t stream) {
    const size_t smem = (size_t)n * 4 * 6 + 33 * 4;
    int rc = allow_smem(wassrank_kernel<COST>, smem);
    if (rc) return rc;
    PTRB200_LAUNCH_TAG("wassrank_kernel", wassrank_kernel<COST>, B, block_threads(n), smem, stream, scores, labels, offsets,
                       grad, loss_q, n, smooth_ng, lam, sh_itr, gain_base, non_rele_gap, var_penalty, B_total);
    return check_launch("wassrank");
}

}  // namespace ptrb200

using namespace ptrb200;

extern "C" {

int ptrb200_wassrank_fwd_bwd(const float* scores, const float* labels, const int32_t* offsets, float* grad, float* loss_per_query,
                             int B, int n, int B_total, int cost_type, int smooth_type, float lam, int sh_itr,
                             float gain_base, float non_rele_gap, float var_penalty, ptrb200_stream_t stream) {
    int rc = check_list_args(scores, labels, grad, loss_per_query, B, n);
    if (rc) return rc;
    if (B_total < B) { set_error("wassrank: B_total=%d is smaller than the launch's B=%d", B_total, B); return PTRB200_ERR_INVALID; }
    if (!(lam != 0.0f) || sh_itr < 0) { set_error("wassrank: lam must be non-zero and sh_itr >= 0"); return PTRB200_ERR_INVALID; }
    if (smooth_type != PTRB200_WASS_SMOOTH_ST && smooth_type != PTRB200_WASS_SMOOTH_NG) {
        set_error("wassrank: unknown smooth_type %d", smooth_type);
        return PTRB200_ERR_INVALID;
    }
    const int ng = smooth_type == PTRB200_WASS_SMOOTH_NG;
    const float Bt = (float)B_total;
    switch (cost_type) {
        case PTRB200_WASS_COST_EG:  return launch_wassrank<WC_EG>(scores, labels, offsets, grad, loss_per_query, B, n, ng, lam, sh_itr, gain_base, non_rele_gap, var_penalty, Bt, stream);
        case PTRB200_WASS_COST_P1:  return launch_wassrank<WC_P1>(scores, labels, offsets, grad, loss_per_query, B, n, ng, lam, sh_itr, gain_base, non_rele_gap, var_penalty, Bt, stream);
        case PTRB200_WASS_COST_P2:  return launch_wassrank<WC_P2>(scores, labels, offsets, grad, loss_per_query, B, n, ng, lam, sh_itr, gain_base, non_rele_gap, var_penalty, Bt, stream);
        case PTRB200_WASS_COST_DG:  return launch_wassrank<WC_DG>(scores, labels, offsets, grad, loss_per_query, B, n, ng, lam, sh_itr, gain_base, non_rele_gap, var_penalty, Bt, stream);
        case PTRB200_WASS_COST_DDG: return launch_wassrank<WC_DDG>(scores, labels, offsets, grad, loss_per_query, B, n, ng, lam, sh_itr, gain_base, non_rele_gap, var_penalty, Bt, stream);
        default:
            set_error("wassrank: unknown cost_type %d", cost_type);
            return PTRB200_ERR_INVALID;
    }
}

}  // extern "C"
