// Explicit-matrix passes: predict, fused residual/score sums, IRLS preparation (Poisson, Gamma, Tweedie power > 1).
// Replaces GLM.predict / neg_mse_score / r2_score / get_residuals (reference
// backend/sglm.py:150-184, :314-347) and one evaluation of the TweedieRegressor(power=1)
// loss/gradient/Hessian weights (sklearn/linear_model/_glm/glm.py:276-316).
//
// Roofline: HBM — one streaming read of X (8*T*C bytes); everything else (link, residual,
// deviance terms, reductions) is fused into the same pass.  One warp per row, 16-byte
// loads, coefficient vector staged in shared memory, per-CTA partial sums reduced by a
// second single-CTA kernel in fixed order (deterministic).
#include <algorithm>

#include "common.cuh"

namespace sglm {

constexpr int PR_THREADS = 256;
constexpr int PR_WARPS = PR_THREADS / 32;
constexpr int PR_MAX_GRID = 4096;
constexpr int PR_NSUM = 8;

enum { MODE_PREDICT = 0, MODE_SCORE = 1, MODE_IRLS = 2 };

__device__ __forceinline__ double row_dot(const double *__restrict__ row, const double *ws, int C, bool vec2, int lane) {
    double s = 0.0;
    if (vec2) {
        const double2 *r2 = reinterpret_cast<const double2 *>(row);
        const double2 *w2 = reinterpret_cast<const double2 *>(ws);
        const int C2 = C >> 1;
#pragma unroll 4
        for (int k = lane; k < C2; k += 32) {
            const double2 a = __ldcs(r2 + k);
            const double2 b = w2[k];
            s += a.x * b.x + a.y * b.y;
        }
        if ((C & 1) && lane == 0) s += row[C - 1] * ws[C - 1];
    } else {
#pragma unroll 4
        for (int k = lane; k < C; k += 32) s += row[k] * ws[k];
    }
    return warp_sum(s);
}

// MODE_SCORE / MODE_IRLS: FAM selects the family terms (common.cuh); the power is read by FAM_TWEEDIE only
template <int MODE, int FAM = FAM_POISSON>
__global__ void __launch_bounds__(PR_THREADS)
row_pass_kernel(const double *__restrict__ X, long long ldx, const double *__restrict__ y,
                const double *__restrict__ rw, long long T, int C, const double *__restrict__ w,
                const double *__restrict__ b_dev, int link, double power, double *__restrict__ out0,
                double *__restrict__ out1, double *__restrict__ partials) {
    extern __shared__ __align__(16) double ws[];
    for (int j = threadIdx.x; j < C; j += PR_THREADS) ws[j] = w[j];
    __syncthreads();
    const double b = b_dev ? *b_dev : 0.0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool vec2 = ((ldx & 1) == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
    double acc[PR_NSUM];
#pragma unroll
    for (int i = 0; i < PR_NSUM; ++i) acc[i] = 0.0;

    for (long long t = (long long)blockIdx.x * PR_WARPS + warp; t < T; t += (long long)gridDim.x * PR_WARPS) {
        const double eta = row_dot(X + t * ldx, ws, C, vec2, lane) + b;
        if (lane == 0) {
            if (MODE == MODE_PREDICT) {
                out0[t] = link ? exp(eta) : eta;
            } else if (MODE == MODE_SCORE) {
                const double mu = link ? exp(eta) : eta;
                const double yt = y[t];
                const double r = yt - mu;
                const double m = rw ? rw[t] : 1.0;
                if (out0) out0[t] = r;
                if (m != 0.0) {
                    acc[0] += m;
                    acc[1] += m * r * r;
                    acc[2] += m * yt;
                    acc[3] += m * yt * yt;
                    if (FAM == FAM_POISSON) {
                        acc[4] += m * yt * eta;
                        acc[5] += m * mu;
                        acc[6] += (yt > 0.0) ? m * yt * log(yt) : 0.0;
                    } else if (FAM == FAM_GAMMA) {             // deviance terms, see pb_epilogue_kernel
                        acc[4] += m * eta;
                        acc[5] += m * (yt / mu);
                        acc[6] += m * log(yt);
                    } else {
                        const double mu1 = exp((1.0 - power) * eta);
                        acc[4] += m * (yt * mu1);
                        acc[5] += m * (mu * mu1);
                        acc[6] += m * pow(yt, 2.0 - power);
                    }
                    acc[7] += m * r;
                }
            } else {
                const double m = rw ? rw[t] : 1.0;
                if (m != 0.0) {
                    const double mu = exp(eta);
                    const double yt = y[t];
                    if (FAM == FAM_POISSON) {
                        out0[t] = m * mu;                   // IRLS weight
                        acc[0] += m * (mu - yt * eta);
                        acc[1] += m * mu;
                    } else if (FAM == FAM_GAMMA) {
                        out0[t] = m;                        // Fisher weight mu^(2-p) = 1
                        acc[0] += m * (eta + yt / mu);
                        acc[1] += m;
                    } else {
                        const double mu1 = exp((1.0 - power) * eta), mu2 = mu * mu1;
                        out0[t] = m * mu2;
                        acc[0] += m * (mu2 / (2.0 - power) - yt * mu1 / (1.0 - power));
                        acc[1] += m * mu2;
                    }
                    out1[t] = eta + (yt - mu) / mu;         // working response
                    acc[2] += m;
                    acc[3] += m * yt;
                } else {                                    // row not in this fold
                    out0[t] = 0.0;
                    out1[t] = 0.0;
                }
            }
        }
    }
    if (MODE != MODE_PREDICT) {
        __shared__ double red[PR_WARPS][PR_NSUM];
        if (lane == 0)
            for (int i = 0; i < PR_NSUM; ++i) red[warp][i] = acc[i];
        __syncthreads();
        if (threadIdx.x < PR_NSUM) {
            double s = 0.0;
            for (int wv = 0; wv < PR_WARPS; ++wv) s += red[wv][threadIdx.x];
            partials[(long long)blockIdx.x * PR_NSUM + threadIdx.x] = s;
        }
    }
}

__global__ void __launch_bounds__(256)
finish_sums_kernel(const double *__restrict__ partials, int n_part, double *__restrict__ sums) {
    // fixed-order tree: thread i owns partials i, i+256, ...; then a fixed smem tree.
    __shared__ double sh[256];
    for (int k = 0; k < PR_NSUM; ++k) {
        double s = 0.0;
        for (int i = threadIdx.x; i < n_part; i += 256) s += partials[(long long)i * PR_NSUM + k];
        sh[threadIdx.x] = s;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) sums[k] = sh[0];
        __syncthreads();
    }
}

// out[c] = sum_t X[t][c] * r[t]  (the exact gradient X'r of the Poisson Newton iteration): every CTA owns a
// contiguous range of rows, a thread owns columns tid, tid + 256, ... (coalesced row reads, r[t] broadcast),
// per-CTA partial sums are added by xt_finish_kernel in fixed order (deterministic).
constexpr int XT_COLS = 4;
__global__ void __launch_bounds__(PR_THREADS)
xt_vec_kernel(const double *__restrict__ X, long long ldx, const double *__restrict__ r, long long T, int C,
              double *__restrict__ partials) {
    const long long rows_per = (T + gridDim.x - 1) / gridDim.x;
    const long long t0 = (long long)blockIdx.x * rows_per, t1 = min(T, t0 + rows_per);
    for (int c0 = 0; c0 < C; c0 += PR_THREADS * XT_COLS) {
        double acc[XT_COLS];
#pragma unroll
        for (int j = 0; j < XT_COLS; ++j) acc[j] = 0.0;
        for (long long t = t0; t < t1; ++t) {
            const double rv = r[t];
            if (rv == 0.0) continue;                       // rows outside the fold (uniform per CTA row)
            const double *row = X + t * ldx + c0 + threadIdx.x;
#pragma unroll
            for (int j = 0; j < XT_COLS; ++j)
                if (c0 + threadIdx.x + j * PR_THREADS < C) acc[j] = fma(__ldcs(row + j * PR_THREADS), rv, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < XT_COLS; ++j) {
            const int c = c0 + threadIdx.x + j * PR_THREADS;
            if (c < C) partials[(long long)blockIdx.x * C + c] = acc[j];
        }
    }
}

__global__ void __launch_bounds__(256)
xt_finish_kernel(const double *__restrict__ partials, int n_part, int C, double *__restrict__ out) {
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= C) return;
    double s = 0.0;
    for (int i = 0; i < n_part; ++i) s += partials[(long long)i * C + c];
    out[c] = s;
}

static int pass_grid(long long T) {
    long long want = ceil_div<long long>(std::max<long long>(T, 1), PR_WARPS);
    return (int)std::min<long long>(want, std::min<long long>(PR_MAX_GRID, (long long)sm_count() * 8));
}

}  // namespace sglm

using namespace sglm;

extern "C" size_t sglm_score_workspace_bytes(void) { return (size_t)PR_MAX_GRID * PR_NSUM * sizeof(double); }

extern "C" int sglm_predict_f64(const double *X, int64_t ldx, int64_t T, int32_t C, const double *w,
                                const double *b_dev, int32_t link, double *out, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C > 0 && ldx >= C, SGLM_E_SHAPE, "predict: bad shape");
    if (T == 0) return SGLM_OK;
    SGLM_CHECK_ARG(X && w && out, SGLM_E_INVALID_ARG, "predict: null pointer");
    const size_t smem = (size_t)((C + 1) & ~1) * sizeof(double);
    SGLM_CHECK_ARG(smem <= 200 * 1024, SGLM_E_UNSUPPORTED, "predict: C=%d too large", C);
    SGLM_CUDA_OK(cudaFuncSetAttribute(row_pass_kernel<MODE_PREDICT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    row_pass_kernel<MODE_PREDICT><<<pass_grid(T), PR_THREADS, smem, (cudaStream_t)stream>>>(
        X, ldx, nullptr, nullptr, T, C, w, b_dev, link, 1.0, out, nullptr, nullptr);
    SGLM_LAUNCH_OK("row_pass_kernel<predict>");
    return SGLM_OK;
}

// one fused pass (MODE_SCORE or MODE_IRLS) of the family of `power` + the fixed-order reduction of its sums
template <int MODE, int FAM>
static int row_pass_sums(const double *X, int64_t ldx, const double *y, const double *rw, int64_t T, int32_t C,
                         const double *w, const double *b_dev, int32_t link, double power, double *out0, double *out1,
                         double *sums, void *workspace, void *stream) {
    const size_t smem = (size_t)((C + 1) & ~1) * sizeof(double);
    const int grid = pass_grid(T);
    cudaStream_t st = (cudaStream_t)stream;
    SGLM_CUDA_OK(cudaFuncSetAttribute(row_pass_kernel<MODE, FAM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    row_pass_kernel<MODE, FAM><<<grid, PR_THREADS, smem, st>>>(X, ldx, y, rw, T, C, w, b_dev, link, power, out0, out1,
                                                               (double *)workspace);
    SGLM_LAUNCH_OK(MODE == MODE_SCORE ? "row_pass_kernel<score>" : "row_pass_kernel<irls>");
    finish_sums_kernel<<<1, 256, 0, st>>>((const double *)workspace, grid, sums);
    SGLM_LAUNCH_OK("finish_sums_kernel");
    return SGLM_OK;
}

template <int MODE>
static int row_pass_sums_family(const double *X, int64_t ldx, const double *y, const double *rw, int64_t T, int32_t C,
                                const double *w, const double *b_dev, int32_t link, double power, double *out0,
                                double *out1, double *sums, void *workspace, void *stream) {
    switch (glm_family(power)) {
    case FAM_POISSON:
        return row_pass_sums<MODE, FAM_POISSON>(X, ldx, y, rw, T, C, w, b_dev, link, power, out0, out1, sums, workspace, stream);
    case FAM_GAMMA:
        return row_pass_sums<MODE, FAM_GAMMA>(X, ldx, y, rw, T, C, w, b_dev, link, power, out0, out1, sums, workspace, stream);
    default:
        return row_pass_sums<MODE, FAM_TWEEDIE>(X, ldx, y, rw, T, C, w, b_dev, link, power, out0, out1, sums, workspace, stream);
    }
}

extern "C" int sglm_score_f64(const double *X, int64_t ldx, const double *y, const double *rw, int64_t T,
                              int32_t C, const double *w, const double *b_dev, int32_t link, double *resid,
                              double *sums, void *workspace, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C > 0 && ldx >= C, SGLM_E_SHAPE, "score: bad shape");
    SGLM_CHECK_ARG(X && y && w && sums && workspace, SGLM_E_INVALID_ARG, "score: null pointer");
    SGLM_CHECK_ARG((size_t)((C + 1) & ~1) * sizeof(double) <= 200 * 1024, SGLM_E_UNSUPPORTED, "score: C=%d too large", C);
    return row_pass_sums<MODE_SCORE, FAM_POISSON>(X, ldx, y, rw, T, C, w, b_dev, link, 1.0, resid, nullptr, sums,
                                                  workspace, stream);
}

// The Tweedie family of `power` (sglm_b200.h).  T = 0 (an empty row slice): X, y and the row outputs may be null, the
// sums are 0.
extern "C" int sglm_score_glm_f64(const double *X, int64_t ldx, const double *y, const double *rw, int64_t T,
                                  int32_t C, const double *w, const double *b_dev, double power, double *resid,
                                  double *sums, void *workspace, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C > 0 && ldx >= C, SGLM_E_SHAPE, "score_glm: bad shape");
    SGLM_CHECK_ARG((T == 0 || (X && y)) && w && sums && workspace, SGLM_E_INVALID_ARG, "score_glm: null pointer");
    SGLM_CHECK_ARG(glm_power_ok(power), SGLM_E_UNSUPPORTED, "score_glm: power %g (supported: 1 and > 1, log link)", power);
    SGLM_CHECK_ARG((size_t)((C + 1) & ~1) * sizeof(double) <= 200 * 1024, SGLM_E_UNSUPPORTED, "score_glm: C=%d too large", C);
    return row_pass_sums_family<MODE_SCORE>(X, ldx, y, rw, T, C, w, b_dev, 1, power, resid, nullptr, sums, workspace,
                                            stream);
}

extern "C" int sglm_poisson_irls_prepare_f64(const double *X, int64_t ldx, const double *y, const double *rw,
                                             int64_t T, int32_t C, const double *w, const double *b_dev,
                                             double *weight, double *z, double *sums, void *workspace,
                                             void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C > 0 && ldx >= C, SGLM_E_SHAPE, "irls_prepare: bad shape");
    SGLM_CHECK_ARG(X && y && w && weight && z && sums && workspace, SGLM_E_INVALID_ARG, "irls_prepare: null pointer");
    SGLM_CHECK_ARG((size_t)((C + 1) & ~1) * sizeof(double) <= 200 * 1024, SGLM_E_UNSUPPORTED, "irls_prepare: C=%d too large", C);
    return row_pass_sums<MODE_IRLS, FAM_POISSON>(X, ldx, y, rw, T, C, w, b_dev, 1, 1.0, weight, z, sums, workspace,
                                                 stream);
}

extern "C" int sglm_glm_irls_prepare_f64(const double *X, int64_t ldx, const double *y, const double *rw,
                                         int64_t T, int32_t C, const double *w, const double *b_dev, double power,
                                         double *weight, double *z, double *sums, void *workspace, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C > 0 && ldx >= C, SGLM_E_SHAPE, "glm_irls_prepare: bad shape");
    SGLM_CHECK_ARG((T == 0 || (X && y && weight && z)) && w && sums && workspace, SGLM_E_INVALID_ARG,
                   "glm_irls_prepare: null pointer");
    SGLM_CHECK_ARG(glm_power_ok(power), SGLM_E_UNSUPPORTED, "glm_irls_prepare: power %g (supported: 1 and > 1, log link)",
                   power);
    SGLM_CHECK_ARG((size_t)((C + 1) & ~1) * sizeof(double) <= 200 * 1024, SGLM_E_UNSUPPORTED,
                   "glm_irls_prepare: C=%d too large", C);
    return row_pass_sums_family<MODE_IRLS>(X, ldx, y, rw, T, C, w, b_dev, 1, power, weight, z, sums, workspace, stream);
}

extern "C" size_t sglm_xt_vec_workspace_bytes(int32_t C) { return (size_t)sm_count() * 8 * (size_t)std::max(C, 1) * sizeof(double); }

// out[c] = sum_t X[t][c] r[t]: one streaming pass over X (8*T*C bytes), deterministic.  T = 0 (an empty row slice):
// X and r may be null, out = 0.
extern "C" int sglm_xt_vec_f64(const double *X, int64_t ldx, const double *r, int64_t T, int32_t C, double *out,
                               void *workspace, size_t workspace_bytes, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C > 0 && ldx >= C, SGLM_E_SHAPE, "xt_vec: bad shape");
    SGLM_CHECK_ARG((T == 0 || (X && r)) && out && workspace, SGLM_E_INVALID_ARG, "xt_vec: null pointer");
    SGLM_CHECK_ARG(workspace_bytes >= sglm_xt_vec_workspace_bytes(C), SGLM_E_WORKSPACE, "xt_vec: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (int)std::max<long long>(1, std::min<long long>((long long)sm_count() * 8, (T + 63) / 64));
    xt_vec_kernel<<<grid, PR_THREADS, 0, st>>>(X, ldx, r, T, C, (double *)workspace);
    SGLM_LAUNCH_OK("xt_vec_kernel");
    xt_finish_kernel<<<ceil_div(C, 256), 256, 0, st>>>((const double *)workspace, grid, C, out);
    SGLM_LAUNCH_OK("xt_finish_kernel");
    return SGLM_OK;
}
