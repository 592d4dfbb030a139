// Steps either side of the lag builder (SURVEY.md §8f-3): z-scoring, n-th differences and the rolling
// 5-95 % quantile min-max detrending of the reference's preprocessing module, for data that already live on the
// device (backend/sglm_pp.py:105-118 zscore, :120-190 diff, :488-545 detrend_data / lambda_min_max).
// All HBM-bound streaming kernels except the detrending, which sorts one window per output position in shared
// memory (bitonic network; the reference calls a Python lambda with two pandas quantiles per position).
#include <algorithm>

#include "common.cuh"

namespace sglm {

constexpr int PP_CHUNK = 4096;     // rows per partial sum (fixed: deterministic results)

// partial[chunk][c] = sum over the chunk's rows of f(X[t][c]); cnt likewise for the non-NaN count.
// pass 0: f = x; pass 1: f = (x - mean[c])^2.  skipna != 0: NaN entries are left out (pandas), else they propagate (numpy).
__global__ void __launch_bounds__(256)
pp_col_partial_kernel(const double *__restrict__ X, long long ldx, long long T, int C, const double *__restrict__ mean,
                      int pass, int skipna, double *__restrict__ part, double *__restrict__ cnt) {
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= C) return;
    const long long t0 = (long long)blockIdx.y * PP_CHUNK, t1 = min(T, t0 + PP_CHUNK);
    const double mu = pass ? mean[c] : 0.0;
    double s = 0.0, n = 0.0;
    for (long long t = t0; t < t1; ++t) {
        const double x = X[t * ldx + c];
        if (skipna && x != x) continue;
        const double d = x - mu;
        s += pass ? d * d : x;
        n += 1.0;
    }
    part[(long long)blockIdx.y * C + c] = s;
    if (!pass) cnt[(long long)blockIdx.y * C + c] = n;
}
// pass 0: mean[c] = sum / n, n_out[c] = n;  pass 1: std[c] = sqrt(sum / (n - ddof)), NaN when n <= ddof
__global__ void __launch_bounds__(256)
pp_col_finish_kernel(const double *__restrict__ part, const double *__restrict__ cnt, int n_chunks, int C, int pass,
                     int ddof, double *__restrict__ out, double *__restrict__ n_io) {
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= C) return;
    double s = 0.0, n = 0.0;
    for (int k = 0; k < n_chunks; ++k) { s += part[(long long)k * C + c]; if (!pass) n += cnt[(long long)k * C + c]; }
    if (!pass) { out[c] = s / n; n_io[c] = n; }
    else out[c] = n_io[c] > (double)ddof ? sqrt(s / (n_io[c] - (double)ddof))
                                         : __longlong_as_double(0x7ff8000000000000LL);   // pandas: NaN, not sqrt(-0.0)
}
__global__ void __launch_bounds__(256)
pp_zscore_kernel(const double *__restrict__ X, long long ldx, long long T, int C, const double *__restrict__ mean,
                 const double *__restrict__ sd, double *__restrict__ out, long long ldo) {
    const long long total = T * (long long)C;
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < total; e += (long long)gridDim.x * 256) {
        const long long t = e / C;
        const int c = (int)(e - t * C);
        out[t * ldo + c] = (X[t * ldx + c] - mean[c]) / sd[c];
    }
}
// out[t][j] = X[t + 1][cols[j]] - X[t][cols[j]]   (one first difference; the n-th is n launches, as np.diff does it)
__global__ void __launch_bounds__(256)
pp_diff_kernel(const double *__restrict__ X, long long ldx, long long T_out, const int *__restrict__ cols, int n_cols,
               double *__restrict__ out, long long ldo) {
    const long long total = T_out * (long long)n_cols;
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < total; e += (long long)gridDim.x * 256) {
        const long long t = e / n_cols;
        const int j = (int)(e - t * n_cols);
        const int c = cols ? cols[j] : j;
        out[t * ldo + j] = X[(t + 1) * ldx + c] - X[t * ldx + c];
    }
}

// Rolling min-max detrending (backend/sglm_pp.py:504-545): pandas `rolling(window=W, center=True).apply(f)` with
//   f(win) = (win[(W+1)//2 - 1] - q05) / (q95 - q05),  q = linear-interpolated quantiles of the W window values.
// The window of output position i is x[i - W/2 .. i + (W-1)/2 ... ] = the W values starting at i - (W - 1 - (W-1)/2)
// (pandas centring: offset (W-1)//2 to the right), it must lie inside the row's segment [seg_lo, seg_hi) and hold
// only finite values, else the result is NaN (min_periods = W; pandas' rolling counts +-inf as missing).  One CTA per
// output position: the window is sorted by a bitonic network in shared memory (padded with +inf to a power of two).
__global__ void __launch_bounds__(256)
pp_rolling_minmax_kernel(const double *__restrict__ x, long long n, const long long *__restrict__ seg_lo,
                         const long long *__restrict__ seg_hi, int W, int Wpad, double *__restrict__ out) {
    extern __shared__ double win[];
    __shared__ int bad;
    const int off_r = (W - 1) / 2;                   // values to the right of the labelled position
    for (long long i = blockIdx.x; i < n; i += gridDim.x) {
        const long long lo = i + off_r - (W - 1), hi = i + off_r;       // inclusive window [lo, hi]
        const long long s0 = seg_lo ? seg_lo[i] : 0, s1 = seg_hi ? seg_hi[i] : n;
        __syncthreads();
        if (lo < s0 || hi >= s1) {
            if (threadIdx.x == 0) out[i] = __longlong_as_double(0x7ff8000000000000LL);
            continue;                                 // uniform per CTA
        }
        if (threadIdx.x == 0) bad = 0;
        __syncthreads();
        for (int k = threadIdx.x; k < Wpad; k += 256) {
            double v = __longlong_as_double(0x7ff0000000000000LL);      // +inf padding
            if (k < W) { v = x[lo + k]; if (!isfinite(v)) bad = 1; }
            win[k] = v;
        }
        __syncthreads();
        const double centre = x[lo + (W + 1) / 2 - 1];
        if (bad) {
            if (threadIdx.x == 0) out[i] = __longlong_as_double(0x7ff8000000000000LL);
            continue;
        }
        for (int size = 2; size <= Wpad; size <<= 1)
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                for (int k = threadIdx.x; k < (Wpad >> 1); k += 256) {
                    const int a = 2 * k - (k & (stride - 1));           // index with bit `stride` cleared
                    const int b = a + stride;
                    const bool up = ((a & size) == 0);
                    const double va = win[a], vb = win[b];
                    if ((va > vb) == up) { win[a] = vb; win[b] = va; }
                }
                __syncthreads();
            }
        if (threadIdx.x == 0) {
            // numpy / pandas linear interpolation: position q (W - 1); lerp written as numpy's _lerp does it, every
            // product rounded before the sum (explicit _rn intrinsics: a contracted FMA rounds once and can differ
            // from numpy in the last bit)
            auto quant = [&](double q) {
                const double pos = __dmul_rn(q, (double)(W - 1));
                const int k = (int)floor(pos);
                const double g = __dsub_rn(pos, (double)k);
                const double a = win[k], b2 = win[min(k + 1, W - 1)];
                const double d = __dsub_rn(b2, a);
                double r = __dadd_rn(a, __dmul_rn(d, g));                                // a + (b - a) t ...
                if (g >= 0.5) r = __dsub_rn(b2, __dmul_rn(d, __dsub_rn(1.0, g)));       // ... from b for t >= 0.5
                return r;
            };
            const double q05 = quant(0.05), q95 = quant(0.95);
            out[i] = (centre - q05) / (q95 - q05);
        }
    }
}

}  // namespace sglm

using namespace sglm;

extern "C" size_t sglm_col_moments_workspace_bytes(int64_t T, int32_t C) {
    const long long n_chunks = std::max<long long>(1, ceil_div<long long>(std::max<long long>(T, 1), PP_CHUNK));
    return (size_t)(2 * n_chunks + 1) * (size_t)std::max(C, 1) * sizeof(double);
}

// mean[c], sd[c] of every column (two passes: mean, then centred squares; fixed chunking -> deterministic).
// ddof: 0 = numpy `std`, 1 = pandas `DataFrame.std`; skipna != 0 leaves NaN entries out (pandas).
extern "C" int sglm_col_moments_f64(const double *X, int64_t ldx, int64_t T, int32_t C, int32_t ddof, int32_t skipna,
                                    double *mean, double *sd, void *workspace, size_t workspace_bytes, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C >= 0 && ldx >= C, SGLM_E_SHAPE, "col_moments: bad shape");
    if (C == 0) return SGLM_OK;
    SGLM_CHECK_ARG(X && mean && sd && workspace, SGLM_E_INVALID_ARG, "col_moments: null pointer");
    SGLM_CHECK_ARG(workspace_bytes >= sglm_col_moments_workspace_bytes(T, C), SGLM_E_WORKSPACE, "col_moments: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int n_chunks = (int)std::max<long long>(1, ceil_div<long long>(std::max<long long>(T, 1), PP_CHUNK));
    double *part = (double *)workspace, *cnt = part + (size_t)n_chunks * C, *n_col = cnt + (size_t)n_chunks * C;
    dim3 grid((unsigned)ceil_div(C, 256), (unsigned)n_chunks);
    for (int pass = 0; pass < 2; ++pass) {
        pp_col_partial_kernel<<<grid, 256, 0, st>>>(X, ldx, T, C, mean, pass, skipna, part, cnt);
        SGLM_LAUNCH_OK("pp_col_partial_kernel");
        pp_col_finish_kernel<<<ceil_div(C, 256), 256, 0, st>>>(part, cnt, n_chunks, C, pass, ddof, pass ? sd : mean, n_col);
        SGLM_LAUNCH_OK("pp_col_finish_kernel");
    }
    return SGLM_OK;
}

extern "C" int sglm_zscore_apply_f64(const double *X, int64_t ldx, int64_t T, int32_t C, const double *mean,
                                     const double *sd, double *out, int64_t ldo, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C >= 0 && ldx >= C && ldo >= C, SGLM_E_SHAPE, "zscore_apply: bad shape");
    if (T == 0 || C == 0) return SGLM_OK;
    SGLM_CHECK_ARG(X && mean && sd && out, SGLM_E_INVALID_ARG, "zscore_apply: null pointer");
    const long long total = T * (long long)C;
    const int grid = (int)std::min<long long>(ceil_div<long long>(total, 256), (long long)sm_count() * 32);
    pp_zscore_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(X, ldx, T, C, mean, sd, out, ldo);
    SGLM_LAUNCH_OK("pp_zscore_kernel");
    return SGLM_OK;
}

// One first difference of the listed columns (cols NULL = all): out [T - 1][n_cols]
extern "C" int sglm_diff1_f64(const double *X, int64_t ldx, int64_t T, const int32_t *cols, int32_t n_cols, double *out,
                              int64_t ldo, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && n_cols >= 0 && ldo >= n_cols, SGLM_E_SHAPE, "diff1: bad shape");
    if (T <= 1 || n_cols == 0) return SGLM_OK;
    SGLM_CHECK_ARG(X && out, SGLM_E_INVALID_ARG, "diff1: null pointer");
    const long long total = (T - 1) * (long long)n_cols;
    const int grid = (int)std::min<long long>(ceil_div<long long>(total, 256), (long long)sm_count() * 32);
    pp_diff_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(X, ldx, T - 1, cols, n_cols, out, ldo);
    SGLM_LAUNCH_OK("pp_diff_kernel");
    return SGLM_OK;
}

// out[i] = rolling 5-95 % min-max of x (window W, centred as pandas centres it); seg_lo / seg_hi (may be NULL):
// bounds [seg_lo[i], seg_hi[i]) of the group row i belongs to (windows never cross a group).
extern "C" int sglm_rolling_minmax_f64(const double *x, int64_t n, const int64_t *seg_lo, const int64_t *seg_hi,
                                       int32_t window, double *out, void *stream) {
    SGLM_CHECK_ARG(n >= 0 && window >= 2 && window <= 16384, SGLM_E_SHAPE, "rolling_minmax: window must be in [2, 16384]");
    if (n == 0) return SGLM_OK;
    SGLM_CHECK_ARG(x && out && ((seg_lo == nullptr) == (seg_hi == nullptr)), SGLM_E_INVALID_ARG, "rolling_minmax: null pointer");
    int Wpad = 2;
    while (Wpad < window) Wpad <<= 1;
    const size_t smem = (size_t)Wpad * sizeof(double);
    SGLM_CUDA_OK(cudaFuncSetAttribute(pp_rolling_minmax_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = (int)std::min<long long>(n, (long long)sm_count() * 8);
    pp_rolling_minmax_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(x, n, (const long long *)seg_lo,
                                                                     (const long long *)seg_hi, window, Wpad, out);
    SGLM_LAUNCH_OK("pp_rolling_minmax_kernel");
    return SGLM_OK;
}
