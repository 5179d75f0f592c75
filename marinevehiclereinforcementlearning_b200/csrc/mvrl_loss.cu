// C ABI of the TQC / QR-DQN critic loss (K11): sb3_contrib's quantile_huber_loss and its gradient with respect to the
// current quantiles, fused.  PyTorch builds the pairwise [B, C, Nq, T] delta and half a dozen tensors of that shape forward
// and backward; here each thread owns one current quantile and keeps its T pairs in registers.  Two launches on the
// caller's stream: the pair kernel (one fp64 loss partial per block) and a one-block reduction of the partials in a fixed
// order, so the same inputs give the same bits, eager or replayed in a CUDA graph.
//
// Compiled with -fmad=false (Makefile): each term w * h takes sb3_contrib's fp32 operations one by one, each correctly
// rounded, with tau = (i + 0.5) / Nq the correctly rounded quotient (as torch computes it on the CPU; torch on the GPU
// multiplies by the fp32 reciprocal of Nq instead, which can move tau by one ulp).  So against sb3_contrib's fp32 result
// only the order of the sums differs, and tau where that ulp moves.  The gradient's accumulation is an explicit fmaf.
#include "mvrl_host.h"

namespace mvrl {

constexpr int kLossThreads = 256;          // current quantiles per block of quantile_huber_kernel
constexpr int kLossReduceThreads = 1024;
constexpr int kLossStageFloats = 2048;     // shared-memory floats for the staged target rows of one block (8 KB)

// The rows b of the target that the kLossThreads consecutive quantiles of one block can touch: at most
// (kLossThreads - 1) / (C * Nq) + 2 of them, never more than kLossThreads.
static inline int stage_rows(int64_t per_row) {
    return (int)std::min<int64_t>(kLossThreads, (kLossThreads - 1) / per_row + 2);
}

// One thread per current quantile r = (b * C + c) * Nq + i.  The block stages its target rows [b_lo, b_hi] in chunks of
// `chunk` columns (a multiple of 4, row stride chunk + 4 floats so that two rows read in one float4 load fall in different
// banks) and each thread walks its row's chunk in order.  Per pair, in sb3_contrib's fp32 operations and order:
//   d = t - q;  a = |d|;  h = a > 1 ? a - 0.5 : (d * d) * 0.5;  w = |tau_i - [d < 0]|;  term = w * h
// and the derivative of h, h' = a > 1 ? sign(d) : d, accumulated as sum_g = fmaf(w, h', sum_g).
__global__ void __launch_bounds__(kLossThreads) quantile_huber_kernel(
        int64_t rows, int per_row, int nq, int64_t T, int chunk, const float* __restrict__ current,
        const float* __restrict__ target, float neg_inv_n, float* __restrict__ grad, double* __restrict__ partials) {
    extern __shared__ float4 s_t4[];
    float* s_t = reinterpret_cast<float*>(s_t4);
    const int stride = chunk + 4;
    const int64_t r0 = (int64_t)blockIdx.x * kLossThreads;
    const int64_t r = r0 + threadIdx.x;
    const bool live = r < rows;
    const int64_t b_lo = r0 / per_row;
    const int64_t b_hi = (min(r0 + kLossThreads, rows) - 1) / per_row;
    const int nb = (int)(b_hi - b_lo + 1);
    const int64_t b = live ? r / per_row : b_hi;
    const float q = live ? current[r] : 0.0f;
    const int i = (int)(live ? r % nq : 0);
    const float tau = __fdiv_rn((float)i + 0.5f, (float)nq);   // (arange(nq) + 0.5) / nq, correctly rounded
    const float w_pos = tau;                                    // |tau - 0|
    const float w_neg = fabsf(__fsub_rn(tau, 1.0f));            // |tau - 1|
    const float* row = s_t + (b - b_lo) * stride;
    float sum_h = 0.0f, sum_g = 0.0f;
    for (int64_t j0 = 0; j0 < T; j0 += chunk) {
        const int len = (int)min((int64_t)chunk, T - j0);
        __syncthreads();
        for (int k = threadIdx.x; k < nb * len; k += kLossThreads) {
            const int rb = k / len, j = k - rb * len;
            s_t[rb * stride + j] = target[(b_lo + rb) * T + j0 + j];
        }
        __syncthreads();
        if (!live) continue;
        auto pair = [&](float t) {
            const float d = __fsub_rn(t, q);
            const float a = fabsf(d);
            const bool outer = a > 1.0f;
            const float h = outer ? __fsub_rn(a, 0.5f) : __fmul_rn(__fmul_rn(d, d), 0.5f);
            const float hp = outer ? copysignf(1.0f, d) : d;
            const float w = d < 0.0f ? w_neg : w_pos;
            sum_h = __fadd_rn(sum_h, __fmul_rn(w, h));
            sum_g = __fmaf_rn(w, hp, sum_g);
        };
        int j = 0;
        for (; j + 4 <= len; j += 4) {
            const float4 t4 = *reinterpret_cast<const float4*>(row + j);
            pair(t4.x); pair(t4.y); pair(t4.z); pair(t4.w);
        }
        for (; j < len; ++j) pair(row[j]);
    }
    if (live && grad != nullptr) grad[r] = __fmul_rn(sum_g, neg_inv_n);
    // block partial of the loss in fp64, in a fixed order: warp tree, then the warps in index order
    __shared__ double s_warp[kLossThreads / 32];
    double v = (double)sum_h;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int k = 0; k < kLossThreads / 32; ++k) s += s_warp[k];
        partials[blockIdx.x] = s;
    }
}

// One block: each thread sums a strided subset of the partials in index order, then a fixed tree; loss = sum / n_pairs.
__global__ void __launch_bounds__(kLossReduceThreads) quantile_huber_reduce_kernel(
        const double* __restrict__ partials, int64_t count, double n_div, float* __restrict__ loss) {
    __shared__ double s[kLossReduceThreads];
    double v = 0.0;
    for (int64_t k = threadIdx.x; k < count; k += kLossReduceThreads) v += partials[k];
    s[threadIdx.x] = v;
    __syncthreads();
    for (int o = kLossReduceThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) loss[0] = (float)(s[0] / n_div);
}

// rows = B * C * Nq, or -1 with mvrl_last_error() set
static int64_t loss_rows(int64_t B, int n_critics, int n_quantiles, int64_t n_target, const char* who) {
    if (B < 1 || n_critics < 1 || n_quantiles < 1 || n_target < 1) {
        mvrl_fail(MVRL_EINVAL, "%s: B %lld, n_critics %d, n_quantiles %d, n_target %lld must all be >= 1", who, (long long)B,
                  n_critics, n_quantiles, (long long)n_target);
        return -1;
    }
    int64_t per_row, rows, pairs, tgt;
    if (__builtin_mul_overflow((int64_t)n_critics, (int64_t)n_quantiles, &per_row) || per_row > INT32_MAX ||
        __builtin_mul_overflow(B, per_row, &rows) || __builtin_mul_overflow(rows, n_target, &pairs) ||
        __builtin_mul_overflow(B, n_target, &tgt) || (rows + kLossThreads - 1) / kLossThreads > INT32_MAX) {
        mvrl_fail(MVRL_EINVAL, "%s: B %lld x %d x %d x %lld overflows the index range", who, (long long)B, n_critics, n_quantiles,
                  (long long)n_target);
        return -1;
    }
    return rows;
}

}  // namespace mvrl

using namespace mvrl;

extern "C" MVRL_API int64_t mvrl_quantile_huber_scratch(int64_t rows) {
    if (rows < 1) return 0;
    return ((rows + kLossThreads - 1) / kLossThreads) * (int64_t)sizeof(double);
}

extern "C" MVRL_API int mvrl_quantile_huber_loss(int64_t B, int n_critics, int n_quantiles, int64_t n_target, const float* current,
                                                 const float* target, int sum_over_quantiles, float* loss, float* grad_current,
                                                 void* scratch, mvrl_stream_t stream) {
    const char* who = "mvrl_quantile_huber_loss";
    if (!current || !target || !loss || !scratch) return mvrl_fail(MVRL_EINVAL, "%s: null argument", who);
    const int64_t rows = loss_rows(B, n_critics, n_quantiles, n_target, who);
    if (rows < 0) return MVRL_EINVAL;
    MVRL_ON_DEVICE_OF(loss, current, who);
    const void* ptrs[] = {current, target, scratch, grad_current};
    static const char* const names[] = {"current", "target", "scratch", "grad_current"};
    if (int rc = mvrl_check_device_ptrs(mvrl_dev_out_, ptrs, names, 4, who)) return rc;
    const int per_row = n_critics * n_quantiles;
    const int nb = stage_rows(per_row);
    const int chunk = (int)std::min<int64_t>((kLossStageFloats / nb - 4) / 4 * 4, (n_target + 3) / 4 * 4);
    const size_t smem = (size_t)nb * (chunk + 4) * sizeof(float);
    // N: pairs averaged over (sb3: loss.mean()), or B * C * T when the sum over the current quantiles comes first
    const double n_div = sum_over_quantiles ? (double)B * n_critics * (double)n_target : (double)rows * (double)n_target;
    const unsigned g = mvrl_grid_for(rows, kLossThreads);
    cudaStream_t st = (cudaStream_t)stream;
    double* partials = (double*)scratch;
    quantile_huber_kernel<<<g, kLossThreads, smem, st>>>(rows, per_row, n_quantiles, n_target, chunk, current, target,
                                                        (float)(-1.0 / n_div), grad_current, partials);
    if (int rc = mvrl_check_launch("quantile_huber")) return rc;
    quantile_huber_reduce_kernel<<<1, kLossReduceThreads, 0, st>>>(partials, (int64_t)g, n_div, loss);
    return mvrl_check_launch("quantile_huber_reduce");
}
