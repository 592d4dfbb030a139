// Batched Poisson GLM grid (BASELINE configs[3]; north-star piece 4): every (fold, alpha) fit of a sweep advances
// together.  Replaces the per-(fold, alpha) TweedieRegressor(power=1).fit calls of the reference
// (backend/sglm.py:112-115, :241; sklearn/linear_model/_glm/glm.py:185-339) — each of which makes two passes over X
// per loss / gradient evaluation — by one Newton-type iteration over the whole batch of B models:
//
//   eta  = X Wt + b          one fp64 GEMM  [T x C] x [C x B]: X is read ONCE per iteration for all B models
//   R    = rw dl/deta        fused elementwise epilogue + per-model sums (objective, sum of weights, sum R), deterministic;
//                            templated on the family: Poisson rw (mu - y), Gamma rw (1 - y/mu), power p rw mu^(1-p) (mu - y)
//   Gw   = X' R              one fp64 GEMM  [C x T] x [T x B] (split over T, partials added in fixed order)
//   step                     per-model kernels: objective check / step halving, right-hand side H~ w - g, batched
//                            triangular solves with the cached factor of (H~ + alpha n I), intercept, convergence
//
// H~ = X' diag(rw mu_ref^(2-p)) X (Fisher weights; Gamma: 1, so H~ = X' diag(rw) X for every iterate) is the weighted
// Gram of ONE reference model per fold (tcgen05 digit-plane Gram, gram_tc.cu) shared by all alphas of the fold: exact gradient + approximate Hessian = the same fixed point as
// Newton's iteration, reached at a linear rate; the host refreshes H~ when the steps stop contracting fast.
// No host synchronisation inside an iteration (one small status read-back per iteration decides about refreshes).
//
// Rooflines: the two GEMMs are FP64-pipe bound (2 T C B flops each; B200: ~40 TFLOP/s), the epilogue is HBM bound
// (16 T B bytes).
#include <algorithm>

#include "common.cuh"

namespace sglm {

constexpr int PB_BM = 128, PB_BN = 64, PB_BK = 16, PB_THREADS = 256;
constexpr int PB_LDA = PB_BM + 4;      // padded k-major tiles (16-byte aligned rows)
constexpr int PB_LDB = PB_BN + 4;
constexpr size_t PB_GEMM_SMEM = (size_t)2 * PB_BK * (PB_LDA + PB_LDB) * sizeof(double);

// 8 x 4 register tile per thread from k-major shared tiles
__device__ __forceinline__ void pb_tile_fma(const double *As, const double *Bs, int ty, int tx, double (&acc)[8][4]) {
#pragma unroll
    for (int k = 0; k < PB_BK; ++k) {
        double a[8], b[4];
        const double2 *ap = reinterpret_cast<const double2 *>(As + k * PB_LDA + ty * 8);
        const double2 *bp = reinterpret_cast<const double2 *>(Bs + k * PB_LDB + tx * 4);
#pragma unroll
        for (int i = 0; i < 4; ++i) { const double2 v = ap[i]; a[2 * i] = v.x; a[2 * i + 1] = v.y; }
#pragma unroll
        for (int j = 0; j < 2; ++j) { const double2 v = bp[j]; b[2 * j] = v.x; b[2 * j + 1] = v.y; }
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
}

// Eta[M x N] = A[M x K] * B[K x N]   (A = X row-major, rows of the design; B = Wt row-major [C][ldb]; N % 64 == 0)
__global__ void __launch_bounds__(PB_THREADS, 2)
pb_gemm_nn_kernel(const double *__restrict__ A, long long lda, long long M, int K, const double *__restrict__ B,
                  long long ldb, double *__restrict__ Cc, long long ldc) {
    extern __shared__ __align__(16) double pb_smem[];
    double (*As)[PB_BK * PB_LDA] = reinterpret_cast<double (*)[PB_BK * PB_LDA]>(pb_smem);
    double (*Bs)[PB_BK * PB_LDB] = reinterpret_cast<double (*)[PB_BK * PB_LDB]>(pb_smem + 2 * PB_BK * PB_LDA);
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const long long m0 = (long long)blockIdx.x * PB_BM;
    const int n0 = blockIdx.y * PB_BN;
    double acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    // A tile: thread -> (row r = tid / 2, 8 consecutive k from (tid & 1) * 8), stored transposed (k-major)
    const int ar = tid >> 1, ak = (tid & 1) * 8;
    // B tile: thread -> (k = tid / 16, 4 consecutive n from (tid & 15) * 4)
    const int bk = tid >> 4, bn = (tid & 15) * 4;
    const bool a_vec = ((lda & 1) == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0);
    auto load = [&](int k0, double (&ra)[8], double (&rb)[4]) {
        const long long row = m0 + ar;
        if (row < M && a_vec && k0 + ak + 8 <= K) {
            const double2 *p = reinterpret_cast<const double2 *>(A + row * lda + k0 + ak);
#pragma unroll
            for (int i = 0; i < 4; ++i) { const double2 v = __ldg(p + i); ra[2 * i] = v.x; ra[2 * i + 1] = v.y; }
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) ra[i] = (row < M && k0 + ak + i < K) ? A[row * lda + k0 + ak + i] : 0.0;
        }
        if (k0 + bk < K) {
            const double2 *p = reinterpret_cast<const double2 *>(B + (long long)(k0 + bk) * ldb + n0 + bn);
            const double2 v0 = __ldg(p), v1 = __ldg(p + 1);
            rb[0] = v0.x; rb[1] = v0.y; rb[2] = v1.x; rb[3] = v1.y;
        } else { rb[0] = rb[1] = rb[2] = rb[3] = 0.0; }
    };
    auto store = [&](int buf, const double (&ra)[8], const double (&rb)[4]) {
#pragma unroll
        for (int i = 0; i < 8; ++i) As[buf][(ak + i) * PB_LDA + ar] = ra[i];
        double2 *q = reinterpret_cast<double2 *>(&Bs[buf][bk * PB_LDB + bn]);
        q[0] = make_double2(rb[0], rb[1]); q[1] = make_double2(rb[2], rb[3]);
    };
    double ra[8], rb[4];
    load(0, ra, rb);
    store(0, ra, rb);
    __syncthreads();
    int buf = 0;
    for (int k0 = 0; k0 < K; k0 += PB_BK) {
        const bool more = k0 + PB_BK < K;
        if (more) load(k0 + PB_BK, ra, rb);
        pb_tile_fma(As[buf], Bs[buf], ty, tx, acc);
        if (more) store(buf ^ 1, ra, rb);
        __syncthreads();
        buf ^= 1;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const long long row = m0 + ty * 8 + i;
        if (row < M) {
            double2 *q = reinterpret_cast<double2 *>(Cc + row * ldc + n0 + tx * 4);
            q[0] = make_double2(acc[i][0], acc[i][1]);
            q[1] = make_double2(acc[i][2], acc[i][3]);
        }
    }
}

// part[split][M x N] = A[k-range, M]' * B[k-range, N]   (A = X [T][lda], M = design columns; B = R [T][ldb])
__global__ void __launch_bounds__(PB_THREADS, 2)
pb_gemm_tn_kernel(const double *__restrict__ A, long long lda, long long Kt, int M, const double *__restrict__ B,
                  long long ldb, int N, long long rows_per_split, double *__restrict__ part, long long ldp) {
    extern __shared__ __align__(16) double pb_smem[];
    double (*As)[PB_BK * PB_LDA] = reinterpret_cast<double (*)[PB_BK * PB_LDA]>(pb_smem);
    double (*Bs)[PB_BK * PB_LDB] = reinterpret_cast<double (*)[PB_BK * PB_LDB]>(pb_smem + 2 * PB_BK * PB_LDA);
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const int m0 = blockIdx.x * PB_BM, n0 = blockIdx.y * PB_BN;
    const long long t_lo = (long long)blockIdx.z * rows_per_split, t_hi = min(Kt, t_lo + rows_per_split);
    double acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    const int ak = tid >> 4, am = (tid & 15) * 8;     // A tile [16 t][128 m]: 8 consecutive m per thread
    const int bk = tid >> 4, bn = (tid & 15) * 4;     // B tile [16 t][64 n]
    const bool a_vec = ((lda & 1) == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0) && ((m0 & 1) == 0);
    auto load = [&](long long t0, double (&ra)[8], double (&rb)[4]) {
        const long long t = t0 + ak;
        if (t < t_hi && a_vec && m0 + am + 8 <= M) {
            const double2 *p = reinterpret_cast<const double2 *>(A + t * lda + m0 + am);
#pragma unroll
            for (int i = 0; i < 4; ++i) { const double2 v = __ldg(p + i); ra[2 * i] = v.x; ra[2 * i + 1] = v.y; }
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) ra[i] = (t < t_hi && m0 + am + i < M) ? A[t * lda + m0 + am + i] : 0.0;
        }
        if (t < t_hi) {
            const double2 *p = reinterpret_cast<const double2 *>(B + t * ldb + n0 + bn);
            const double2 v0 = __ldg(p), v1 = __ldg(p + 1);
            rb[0] = v0.x; rb[1] = v0.y; rb[2] = v1.x; rb[3] = v1.y;
        } else { rb[0] = rb[1] = rb[2] = rb[3] = 0.0; }
    };
    auto store = [&](int buf, const double (&ra)[8], const double (&rb)[4]) {
        double2 *qa = reinterpret_cast<double2 *>(&As[buf][ak * PB_LDA + am]);
#pragma unroll
        for (int i = 0; i < 4; ++i) qa[i] = make_double2(ra[2 * i], ra[2 * i + 1]);
        double2 *q = reinterpret_cast<double2 *>(&Bs[buf][bk * PB_LDB + bn]);
        q[0] = make_double2(rb[0], rb[1]); q[1] = make_double2(rb[2], rb[3]);
    };
    double ra[8], rb[4];
    if (t_lo < t_hi) {
        load(t_lo, ra, rb);
        store(0, ra, rb);
        __syncthreads();
        int buf = 0;
        for (long long t0 = t_lo; t0 < t_hi; t0 += PB_BK) {
            const bool more = t0 + PB_BK < t_hi;
            if (more) load(t0 + PB_BK, ra, rb);
            pb_tile_fma(As[buf], Bs[buf], ty, tx, acc);
            if (more) store(buf ^ 1, ra, rb);
            __syncthreads();
            buf ^= 1;
        }
    }
    double *out = part + (long long)blockIdx.z * M * ldp;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int row = m0 + ty * 8 + i;
        if (row < M) {
            double2 *q = reinterpret_cast<double2 *>(out + (long long)row * ldp + n0 + tx * 4);
            q[0] = make_double2(acc[i][0], acc[i][1]);
            q[1] = make_double2(acc[i][2], acc[i][3]);
        }
    }
}

__global__ void __launch_bounds__(256)
pb_reduce_splits_kernel(const double *__restrict__ part, long long n_elem, int n_split, double *__restrict__ out) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < n_elem; e += (long long)gridDim.x * 256) {
        double s = 0.0;
        for (int k = 0; k < n_split; ++k) s += part[(long long)k * n_elem + e];      // fixed order
        out[e] = s;
    }
}

// Elementwise pass over Eta [T][ldb] (thread <-> model column, CTA <-> row range): eta += b, mu = exp(eta).
//   mode 0 (iteration): Eta <- R = rw dl/deta in place; partial sums {rw l, rw v, rw, R} with the loss l, its
//                       derivative and the Fisher weight v of the family (HalfTweedieLoss, log link):
//                         Poisson  l = mu - y eta                              dl/deta = mu - y            v = mu
//                         Gamma    l = eta + y / mu                            dl/deta = 1 - y / mu        v = 1
//                         power p  l = mu^(2-p)/(2-p) - y mu^(1-p)/(1-p)       dl/deta = mu^(1-p)(mu - y)  v = mu^(2-p)
//   mode 1 (scores)   : no write; 2 x 8 sums per model for the row weights rw_a / rw_b (train / test):
//                       {n, r^2, y, y^2, s4, s5, s6, r} with r = y - mu; the family terms s4..s6 give the deviance:
//                         Poisson {y eta, mu, y log y} (as sglm_score_f64), Gamma {eta, y / mu, log y},
//                         power p {y mu^(1-p), mu^(2-p), y^(2-p)}
// Y [T][ldy] holds the response columns (one per distinct `roll`), RW [n_w][ldrw] the row-weight vectors
// (rw id < 0: all rows).  Partial sums per CTA -> pb_finish_sums_kernel adds them in fixed order.
constexpr int PB_NS_IT = 4, PB_NS_SC = 16;
template <int MODE, int FAM>
__global__ void __launch_bounds__(128)
pb_epilogue_kernel(double *__restrict__ Eta, long long ldb, int n_models, long long T, const double *__restrict__ Y,
                   long long ldy, const int *__restrict__ ycol, const double *__restrict__ RW, long long ldrw,
                   const int *__restrict__ rw_a, const int *__restrict__ rw_b, const double *__restrict__ bvec,
                   const int *__restrict__ status, double power, double *__restrict__ partials) {
    constexpr int NS = MODE == 0 ? PB_NS_IT : PB_NS_SC;
    const double q1 = 1.0 - power, inv1 = 1.0 / (1.0 - power), inv2 = 1.0 / (2.0 - power);   // FAM_TWEEDIE only
    const int mdl = blockIdx.y * 128 + threadIdx.x;
    const bool live = mdl < n_models;
    const long long rows_per = (T + gridDim.x - 1) / gridDim.x;
    const long long t0 = (long long)blockIdx.x * rows_per, t1 = min(T, t0 + rows_per);
    double acc[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) acc[i] = 0.0;
    if (live && !(MODE == 0 && status && status[mdl] != 0)) {
        const double b = bvec[mdl];
        const double *y = Y + ycol[mdl];
        const double *wa = rw_a[mdl] >= 0 ? RW + (long long)rw_a[mdl] * ldrw : nullptr;
        const double *wb = (MODE == 1 && rw_b[mdl] >= 0) ? RW + (long long)rw_b[mdl] * ldrw : nullptr;
        for (long long t = t0; t < t1; ++t) {
            const double eta = Eta[t * ldb + mdl] + b;
            const double yt = y[t * ldy];
            if (MODE == 0) {
                const double m = wa ? wa[t] : 1.0;
                double r = 0.0;
                if (m != 0.0) {
                    if (FAM == FAM_POISSON) {
                        const double mu = exp(eta);
                        r = m * (mu - yt);
                        acc[0] += m * (mu - yt * eta);
                        acc[1] += m * mu;
                    } else if (FAM == FAM_GAMMA) {
                        const double y_mu = yt * exp(-eta);
                        r = m * (1.0 - y_mu);
                        acc[0] += m * (eta + y_mu);
                        acc[1] += m;
                    } else {
                        const double mu = exp(eta), mu1 = exp(q1 * eta), mu2 = mu * mu1;
                        r = m * (mu1 * (mu - yt));
                        acc[0] += m * (mu2 * inv2 - yt * mu1 * inv1);
                        acc[1] += m * mu2;
                    }
                    acc[2] += m;
                    acc[3] += r;
                }
                Eta[t * ldb + mdl] = r;
            } else {
                const double ma = wa ? wa[t] : 1.0, mb = (MODE == 1 && rw_b[mdl] < -1) ? 0.0 : (wb ? wb[t] : 1.0);
                if (ma != 0.0 || mb != 0.0) {
                    const double mu = exp(eta), r = yt - mu;
                    double s4, s5, s6;
                    if (FAM == FAM_POISSON) {
                        s4 = yt * eta; s5 = mu; s6 = (yt > 0.0) ? yt * log(yt) : 0.0;
                    } else if (FAM == FAM_GAMMA) {
                        s4 = eta; s5 = yt / mu; s6 = log(yt);
                    } else {
                        const double mu1 = exp(q1 * eta);
                        s4 = yt * mu1; s5 = mu * mu1; s6 = pow(yt, 2.0 - power);
                    }
                    const double v[8] = {1.0, r * r, yt, yt * yt, s4, s5, s6, r};
#pragma unroll
                    for (int i = 0; i < 8; ++i) { acc[i] += ma * v[i]; acc[8 + i] += mb * v[i]; }
                }
            }
        }
    }
    if (live) {
        double *dst = partials + ((long long)blockIdx.x * n_models + mdl) * NS;
#pragma unroll
        for (int i = 0; i < NS; ++i) dst[i] = acc[i];
    }
}

__global__ void __launch_bounds__(256)
pb_finish_sums_kernel(const double *__restrict__ partials, int n_part, long long n_vals, double *__restrict__ sums) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < n_vals; e += (long long)gridDim.x * 256) {
        double s = 0.0;
        for (int p = 0; p < n_part; ++p) s += partials[(long long)p * n_vals + e];
        sums[e] = s;
    }
}

// ---- per-model step logic (one CTA per model) -----------------------------------------------------------------
struct PbState {
    double *W, *Wprev, *Wnew, *rhs;          // [B][ldw]
    double *b, *bprev, *fprev, *fcur, *last_step, *step_out, *ratio_out;   // [B]
    int *halv, *n_iter, *status, *flag, *has_prev;                          // [B]
    const double *alpha, *n_tot, *tol;       // [B]
    const int *fit_icpt, *max_iter, *hess_id;
    const double *const *HQ;                 // [n_hess] centred weighted Gram Qc (C x ldq)
    const double *const *Hxbar;              // [n_hess] weighted column means
    const double *Hh11;                      // [n_hess] sum of the weights
    const double *sums;                      // [B][4] from the epilogue
    const double *Gw;                        // [C][ldb] gradient X'R
    const double *hscale;                    // [B] the model's Hessian = hscale * (the group's H~): a fold's first step
                                             // borrows the full-data Hessian scaled by its share of sum(y)
    long long ldw, ldq, ldb;
    int C, B;
};

__device__ __forceinline__ double pb_block_sum(double v, double *sh) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += sh[w];
    return s;
}
__device__ __forceinline__ double pb_block_max(double v, double *sh) {
    v = warp_max(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = sh[0];
    for (int w = 1; w < 8; ++w) s = fmax(s, sh[w]);
    return s;
}

// objective check / step halving, else the right-hand side of the chord step  (H~ + a n I) w_new = H~ w - g.
// l1_ratio [B] (null: all 0): the penalty is alpha r |w|_1 + alpha (1 - r)/2 |w|^2
__global__ void __launch_bounds__(256)
pb_rhs_kernel(PbState s, const double *__restrict__ l1_ratio) {
    __shared__ double sh[8];
    extern __shared__ __align__(16) double wsh[];          // [C] current w
    const int m = blockIdx.x, tid = threadIdx.x;
    if (s.status[m] != 0) { if (tid == 0) s.flag[m] = 0; return; }
    double *w = s.W + (long long)m * s.ldw;
    const double *wp = s.Wprev + (long long)m * s.ldw;
    double ww = 0.0, w1 = 0.0;
    for (int j = tid; j < s.C; j += 256) { const double v = w[j]; wsh[j] = v; ww = fma(v, v, ww); w1 += fabs(v); }
    ww = pb_block_sum(ww, sh);
    w1 = pb_block_sum(w1, sh);
    const double r1 = l1_ratio ? l1_ratio[m] : 0.0;
    // r = 0: alpha (1 - 0) = alpha and no L1 term, so f (and every halving decision) has the bits of the ridge path
    double f = s.sums[4 * m + 0] / s.n_tot[m] + 0.5 * (s.alpha[m] * (1.0 - r1)) * ww;
    if (r1 != 0.0) f += s.alpha[m] * r1 * w1;
    const double fp = s.fprev[m];
    const bool worse = s.has_prev[m] && !(f <= fp + 1e-12 * fmax(1.0, fabs(fp)));
    if (worse && s.halv[m] < 30) {
        for (int j = tid; j < s.C; j += 256) w[j] = 0.5 * (wsh[j] + wp[j]);
        if (tid == 0) { s.b[m] = 0.5 * (s.b[m] + s.bprev[m]); s.halv[m] += 1; s.flag[m] = 2; }
        return;
    }
    if (s.n_iter[m] >= s.max_iter[m]) { if (tid == 0) { s.status[m] = 2; s.flag[m] = 0; } return; }
    const int h = s.hess_id[m];
    const double *Q = s.HQ[h];
    const double *xbar = s.Hxbar[h];
    const double g_b = s.sums[4 * m + 3];
    const bool icpt = s.fit_icpt[m] != 0;
    const double inv_hs = 1.0 / s.hscale[m];
    double *rhs = s.rhs + (long long)m * s.ldw;
    const int warp = tid >> 5, lane = tid & 31;
    // (hs Q + a n I) w_new = hs Q w - g + xbar g_b   <=>   (Q + (a n / hs) I) w_new = Q w + (-g + xbar g_b) / hs ; the cached
    // factor belongs to Q + a n' I with a n' ~ a n / hs (exact for hs = 1)
    for (int j = warp; j < s.C; j += 8) {
        const double *row = Q + (long long)j * s.ldq;
        double d = 0.0;
        for (int k = lane; k < s.C; k += 32) d = fma(row[k], wsh[k], d);
        d = warp_sum(d);
        if (lane == 0) rhs[j] = d + (-s.Gw[(long long)j * s.ldb + m] + (icpt ? xbar[j] * g_b : 0.0)) * inv_hs;
    }
    if (tid == 0) { s.halv[m] = 0; s.fcur[m] = f; s.flag[m] = 1; }
}

// ---- elastic-net models (l1_ratio > 0): proximal-Newton step.  The quadratic model of the chord step keeps its
// Hessian and right-hand side; the triangular solves are replaced by a warm-started Gram coordinate-descent solve of
//   min_w 1/2 w'Qw - rhs'w + l1 |w|_1 + l2/2 |w|^2,   l1 = alpha r n / hs,  l2 = alpha (1 - r) n / hs
// (enet_cd_gram_kernel, solvers.cu).  Its duality gap needs a yy consistent with (Q, rhs): yy = rhs'(Q + l2 I)^-1 rhs,
// the ridge solution coming from the model's cached factor of (Q + alpha (1 - r) n I) (the chord solve that precedes
// this kernel), so that R^2 + l2 |w|^2 = (w - w_ridge)'(Q + l2 I)(w - w_ridge) >= 0.  A fold's first step borrows
// the full-data factor (hs != 1); there yy belongs to a nearby l2 and only makes that one step's stopping test
// approximate: the later steps use the fold's own Hessian (hs = 1).
//
// Inner tolerance: the kernel stops after a sweep that moved no coordinate by more than tol * max|w| and whose gap is
// <= tol * yy.  The sweep test is what resolves a small step: the gap is a difference of terms of size
// yy = |w_ridge|^2_(Q + l2 I) (rounding ~1e-16 yy), so it only bounds a step d through |d|_(Q + l2 I) <= sqrt(2 gap),
// i.e. to ~1e-8 relative.  Hence the solve is started with "at least one sweep" (a start whose gap is below tol * yy
// would otherwise be returned untouched and end the outer iteration up to ~1e-7 from its fixed point), and tol = 1e-13:
// the inner error (~1e-13 |w| times the CD contraction factor) stays far below what the outer rule
// (step * rho / (1 - rho) <= min(tol, 1e-8)) resolves, so inexact inner solves neither stall nor end the outer iteration,
// while the gap test at tol * yy = 1e-13 yy stays well above its rounding floor.
constexpr double PB_ENET_TOL = 1e-13;
// sweeps per inner solve: a cap, not a budget — a warm start near the optimum needs a few
constexpr int PB_ENET_SWEEPS = 1000;

// workspace of sglm_pb_step_enet_f64 (n_enet models): W [n][ldw], diag [n][ldw], yy / l1 / l2 / tol [n],
// Q / q / diag pointers [n], max_iter / problem ids [n] (int32)
struct PbEnetWork {
    double *W, *dg, *yy, *l1, *l2, *tol;
    const double **pQ, **pq, **pd;
    int *max_iter, *pid;
};
__host__ __device__ inline PbEnetWork pb_enet_carve(void *ws, long long ldw, int n) {
    PbEnetWork e;
    double *d = (double *)ws;
    e.W = d; d += (long long)n * ldw;
    e.dg = d; d += (long long)n * ldw;
    e.yy = d; d += n; e.l1 = d; d += n; e.l2 = d; d += n; e.tol = d; d += n;
    e.pQ = (const double **)d; d += n; e.pq = (const double **)d; d += n; e.pd = (const double **)d; d += n;
    e.max_iter = (int *)d; e.pid = e.max_iter + n;
    return e;
}

// one CTA per elastic-net model k (model m = idx[k]): the inner problem.  Models without a step this round (flag != 1:
// halving, converged, max_iter) get w = 0 and max_iter 0: the solve returns at once and its result is not used.
__global__ void __launch_bounds__(256)
pb_enet_prep_kernel(PbState s, const double *__restrict__ l1_ratio, const int *__restrict__ idx, PbEnetWork e) {
    __shared__ double sh[8];
    const int k = blockIdx.x, tid = threadIdx.x, m = idx[k];
    const bool step = s.flag[m] == 1;
    const int h = s.hess_id[m];
    const double *Q = s.HQ[h];
    const double *q = s.rhs + (long long)m * s.ldw, *wr = s.Wnew + (long long)m * s.ldw, *w = s.W + (long long)m * s.ldw;
    double *wk = e.W + (long long)k * s.ldw, *dk = e.dg + (long long)k * s.ldw;
    double yy = 0.0;
    for (int j = tid; j < s.C; j += 256) {
        dk[j] = Q[(long long)j * s.ldq + j];
        wk[j] = step ? w[j] : 0.0;
        yy = fma(q[j], wr[j], yy);
    }
    yy = pb_block_sum(yy, sh);
    if (tid == 0) {
        const double r1 = l1_ratio[m], an = s.alpha[m] * s.n_tot[m] / s.hscale[m];
        e.pQ[k] = Q; e.pq[k] = q; e.pd[k] = dk;
        e.yy[k] = yy;
        e.l1[k] = an * r1;
        e.l2[k] = an * (1.0 - r1);
        e.tol[k] = PB_ENET_TOL;
        e.max_iter[k] = step ? PB_ENET_SWEEPS : 0;
        e.pid[k] = k;
    }
}

// the inner solutions become the models' new iterates
__global__ void __launch_bounds__(256)
pb_enet_scatter_kernel(PbState s, const int *__restrict__ idx, PbEnetWork e) {
    const int k = blockIdx.x, m = idx[k];
    if (s.flag[m] != 1) return;
    for (int j = threadIdx.x; j < s.C; j += 256) s.Wnew[(long long)m * s.ldw + j] = e.W[(long long)k * s.ldw + j];
}

// intercept, step size, convergence
__global__ void __launch_bounds__(256)
pb_finish_kernel(PbState s) {
    __shared__ double sh[8];
    const int m = blockIdx.x, tid = threadIdx.x;
    if (s.flag[m] != 1) { if (tid == 0) s.step_out[m] = s.flag[m] == 2 ? -1.0 : 0.0; return; }
    double *w = s.W + (long long)m * s.ldw, *wp = s.Wprev + (long long)m * s.ldw;
    const double *wn = s.Wnew + (long long)m * s.ldw;
    const int h = s.hess_id[m];
    const double *xbar = s.Hxbar[h];
    const bool icpt = s.fit_icpt[m] != 0;
    double dot = 0.0, dw = 0.0, wmax = 0.0;
    for (int j = tid; j < s.C; j += 256) {
        const double a = wn[j], o = w[j];
        dot = fma(icpt ? xbar[j] : 0.0, a - o, dot);
        dw = fmax(dw, fabs(a - o));
        wmax = fmax(wmax, fabs(a));
    }
    dot = pb_block_sum(dot, sh);
    dw = pb_block_max(dw, sh);
    wmax = pb_block_max(wmax, sh);
    const double b_old = s.b[m];
    const double b_new = icpt ? b_old - s.sums[4 * m + 3] / (s.Hh11[h] * s.hscale[m]) - dot : 0.0;
    for (int j = tid; j < s.C; j += 256) { wp[j] = w[j]; w[j] = wn[j]; }
    if (tid == 0) {
        const double step = fmax(dw, fabs(b_new - b_old)) / fmax(1.0, wmax);
        const double last = s.last_step[m];
        const bool have = last > 0.0 && last < 1e300;
        const double ratio = have ? step / last : 1.0;
        // contraction estimate = the worse of the last two ratios (1.0 = not known yet: the first two steps after a
        // Hessian refresh cannot declare convergence unless the step itself is below the target)
        const double rho = fmin(fmax(ratio, s.ratio_out[m]), 0.9);
        s.bprev[m] = b_old; s.b[m] = b_new; s.fprev[m] = s.fcur[m]; s.has_prev[m] = 1;
        s.n_iter[m] += 1;
        // linear convergence (inexact Hessian): after a step that contracted by rho the iterate is within
        // step * rho / (1 - rho) of the optimum
        if (step * rho / (1.0 - rho) <= fmin(s.tol[m], 1e-8) || step <= 1e-12) s.status[m] = 1;
        s.step_out[m] = step;
        s.ratio_out[m] = ratio;
        s.last_step[m] = step;
    }
}

}  // namespace sglm

using namespace sglm;

extern "C" size_t sglm_pb_gemm_tn_workspace_bytes(int64_t T, int32_t C, int64_t ldb) {
    const long long rows_per = 8192;
    const long long n_split = std::max<long long>(1, ceil_div<long long>(std::max<long long>(T, 1), rows_per));
    return (size_t)n_split * (size_t)C * (size_t)ldb * sizeof(double);
}

// Eta [T][ldb] = X [T][C] * Wt [C][ldb]   (ldb a multiple of 64; the columns beyond the models are zero in Wt)
extern "C" int sglm_pb_eta_f64(const double *X, int64_t ldx, int64_t T, int32_t C, const double *Wt, int64_t ldb,
                               double *Eta, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C > 0 && ldx >= C && ldb >= 64 && ldb % 64 == 0, SGLM_E_SHAPE, "pb_eta: bad shape");
    if (T == 0) return SGLM_OK;
    SGLM_CHECK_ARG(X && Wt && Eta, SGLM_E_INVALID_ARG, "pb_eta: null pointer");
    SGLM_CHECK_ARG(((uintptr_t)Wt & 15) == 0 && ((uintptr_t)Eta & 15) == 0, SGLM_E_ALIGN, "pb_eta: 16-byte alignment");
    dim3 grid((unsigned)ceil_div<long long>(T, PB_BM), (unsigned)(ldb / PB_BN));
    SGLM_CUDA_OK(cudaFuncSetAttribute(pb_gemm_nn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PB_GEMM_SMEM));
    pb_gemm_nn_kernel<<<grid, PB_THREADS, PB_GEMM_SMEM, (cudaStream_t)stream>>>(X, ldx, T, C, Wt, ldb, Eta, ldb);
    SGLM_LAUNCH_OK("pb_gemm_nn_kernel");
    return SGLM_OK;
}

// ------------------------------------------------------------------ quadratic forms of many vectors: v_m' A v_m
// out[m] = sum_i Vt[i][m] (A Vt)[i][m]: one fp64 GEMM (A is read once per 64 vectors instead of once per 8 as in
// quadform_kernel) followed by column dots in fixed row chunks (deterministic).  Scores of a CV grid from the
// statistics: RSS(model, row set) = v' G[set] v (backend/sglm.py:305-312 computes them by three prediction passes).
constexpr int QG_PARTS = 16;
__global__ void __launch_bounds__(128)
coldot_kernel(const double *__restrict__ Vt, const double *__restrict__ Y, long long n, long long ldb, int n_models,
              double *__restrict__ part) {
    const int m = blockIdx.x * 128 + threadIdx.x;
    if (m >= n_models) return;
    const long long per = (n + QG_PARTS - 1) / QG_PARTS;
    const long long i0 = (long long)blockIdx.y * per, i1 = min(n, i0 + per);
    double acc = 0.0;
    for (long long i = i0; i < i1; ++i) acc = fma(Vt[i * ldb + m], Y[i * ldb + m], acc);
    part[(long long)blockIdx.y * n_models + m] = acc;
}
__global__ void __launch_bounds__(128)
coldot_finish_kernel(const double *__restrict__ part, int n_models, double *__restrict__ out) {
    const int m = blockIdx.x * 128 + threadIdx.x;
    if (m >= n_models) return;
    double s = 0.0;
    for (int p = 0; p < QG_PARTS; ++p) s += part[(long long)p * n_models + m];
    out[m] = s;
}

// Vt [n][ldb]: the vectors as COLUMNS (ldb % 64 == 0, columns >= n_models zero); work: 2 * n * ldb doubles is not needed —
// Y [n][ldb] and part [16][n_models] are caller buffers.
extern "C" int sglm_quadform_gemm_f64(const double *A, int64_t lda, int32_t n, const double *Vt, int64_t ldb,
                                      int32_t n_models, double *Y, double *part, double *out, void *stream) {
    SGLM_CHECK_ARG(n > 0 && lda >= n && n_models > 0 && ldb >= n_models && ldb % 64 == 0, SGLM_E_SHAPE, "quadform_gemm: bad shape");
    SGLM_CHECK_ARG(A && Vt && Y && part && out, SGLM_E_INVALID_ARG, "quadform_gemm: null pointer");
    SGLM_CHECK_ARG(((uintptr_t)Vt & 15) == 0 && ((uintptr_t)Y & 15) == 0, SGLM_E_ALIGN, "quadform_gemm: 16-byte alignment");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid((unsigned)ceil_div<long long>(n, PB_BM), (unsigned)(ldb / PB_BN));
    SGLM_CUDA_OK(cudaFuncSetAttribute(pb_gemm_nn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PB_GEMM_SMEM));
    pb_gemm_nn_kernel<<<grid, PB_THREADS, PB_GEMM_SMEM, st>>>(A, lda, n, n, Vt, ldb, Y, ldb);
    SGLM_LAUNCH_OK("pb_gemm_nn_kernel(quadform)");
    dim3 dgrid((unsigned)ceil_div(n_models, 128), QG_PARTS);
    coldot_kernel<<<dgrid, 128, 0, st>>>(Vt, Y, n, ldb, n_models, part);
    SGLM_LAUNCH_OK("coldot_kernel");
    coldot_finish_kernel<<<ceil_div(n_models, 128), 128, 0, st>>>(part, n_models, out);
    SGLM_LAUNCH_OK("coldot_finish_kernel");
    return SGLM_OK;
}

// Gw [C][ldb] = X' R   (R [T][ldb]); deterministic: fixed T chunks of 8192 rows, partials added in order.
// T = 0 (an empty row slice): X and R may be null, Gw = 0.
extern "C" int sglm_pb_xt_r_f64(const double *X, int64_t ldx, int64_t T, int32_t C, const double *R, int64_t ldb,
                                double *Gw, void *workspace, size_t workspace_bytes, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C > 0 && ldx >= C && ldb >= 64 && ldb % 64 == 0, SGLM_E_SHAPE, "pb_xt_r: bad shape");
    SGLM_CHECK_ARG((T == 0 || (X && R)) && Gw && workspace, SGLM_E_INVALID_ARG, "pb_xt_r: null pointer");
    SGLM_CHECK_ARG(((uintptr_t)R & 15) == 0 && ((uintptr_t)workspace & 15) == 0, SGLM_E_ALIGN, "pb_xt_r: 16-byte alignment");
    SGLM_CHECK_ARG(workspace_bytes >= sglm_pb_gemm_tn_workspace_bytes(T, C, ldb), SGLM_E_WORKSPACE, "pb_xt_r: workspace too small");
    const long long rows_per = 8192;
    const int n_split = (int)std::max<long long>(1, ceil_div<long long>(std::max<long long>(T, 1), rows_per));
    dim3 grid((unsigned)ceil_div(C, PB_BM), (unsigned)(ldb / PB_BN), (unsigned)n_split);
    SGLM_CUDA_OK(cudaFuncSetAttribute(pb_gemm_tn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PB_GEMM_SMEM));
    pb_gemm_tn_kernel<<<grid, PB_THREADS, PB_GEMM_SMEM, (cudaStream_t)stream>>>(X, ldx, T, C, R, ldb, (int)ldb, rows_per,
                                                                   (double *)workspace, ldb);
    SGLM_LAUNCH_OK("pb_gemm_tn_kernel");
    const long long n_elem = (long long)C * ldb;
    pb_reduce_splits_kernel<<<(unsigned)std::min<long long>(ceil_div<long long>(n_elem, 256), sm_count() * 8LL), 256, 0,
                              (cudaStream_t)stream>>>((const double *)workspace, n_elem, n_split, Gw);
    SGLM_LAUNCH_OK("pb_reduce_splits_kernel");
    return SGLM_OK;
}

// out[e] = sum over k = 0, 1, ... of parts[k][e], added in that order: the per-rank partial sums of a row-sharded
// batch, gathered in rank order, give the same bits on every rank.
extern "C" int sglm_reduce_parts_f64(const double *parts, int64_t n_elem, int32_t n_parts, double *out, void *stream) {
    SGLM_CHECK_ARG(n_elem >= 0 && n_parts >= 1, SGLM_E_SHAPE, "reduce_parts: bad shape");
    if (n_elem == 0) return SGLM_OK;
    SGLM_CHECK_ARG(parts && out, SGLM_E_INVALID_ARG, "reduce_parts: null pointer");
    pb_reduce_splits_kernel<<<(unsigned)std::min<long long>(ceil_div<long long>(n_elem, 256), sm_count() * 8LL), 256, 0,
                              (cudaStream_t)stream>>>(parts, n_elem, n_parts, out);
    SGLM_LAUNCH_OK("pb_reduce_splits_kernel");
    return SGLM_OK;
}

static int pb_epi_grid(long long T) { return (int)std::max<long long>(1, std::min<long long>(sm_count() * 8LL, ceil_div<long long>(T, 64))); }

extern "C" size_t sglm_pb_epilogue_workspace_bytes(int64_t T, int32_t n_models) {
    return (size_t)pb_epi_grid(T) * (size_t)std::max(n_models, 1) * PB_NS_SC * sizeof(double);
}

template <int MODE>
static void pb_epilogue_launch(int fam, dim3 grid, cudaStream_t st, double *Eta, int64_t ldb, int32_t n_models,
                               int64_t T, const double *Y, int64_t ldy, const int32_t *ycol, const double *RW,
                               int64_t ldrw, const int32_t *rw_a, const int32_t *rw_b, const double *b,
                               const int32_t *status, double power, double *part) {
    if (fam == FAM_POISSON)
        pb_epilogue_kernel<MODE, FAM_POISSON><<<grid, 128, 0, st>>>(Eta, ldb, n_models, T, Y, ldy, ycol, RW, ldrw, rw_a,
                                                                    rw_b, b, status, power, part);
    else if (fam == FAM_GAMMA)
        pb_epilogue_kernel<MODE, FAM_GAMMA><<<grid, 128, 0, st>>>(Eta, ldb, n_models, T, Y, ldy, ycol, RW, ldrw, rw_a,
                                                                  rw_b, b, status, power, part);
    else
        pb_epilogue_kernel<MODE, FAM_TWEEDIE><<<grid, 128, 0, st>>>(Eta, ldb, n_models, T, Y, ldy, ycol, RW, ldrw, rw_a,
                                                                    rw_b, b, status, power, part);
}

static int pb_epilogue(const char *name, double *Eta, int64_t ldb, int32_t n_models, int64_t T, const double *Y,
                       int64_t ldy, const int32_t *ycol, const double *RW, int64_t ldrw, const int32_t *rw_a,
                       const int32_t *rw_b, const double *b, const int32_t *status, double power, int32_t mode,
                       double *sums, void *workspace, size_t workspace_bytes, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && n_models > 0 && ldb >= n_models && ldy >= 1, SGLM_E_SHAPE, "%s: bad shape", name);
    // T = 0 (an empty row slice): no row is read or written, Eta, Y and RW may be null and the sums are 0.  RW is not
    // checked: with T > 0 it must hold every row-weight vector an rw id >= 0 names.
    SGLM_CHECK_ARG((T == 0 || (Eta && Y)) && ycol && rw_a && b && sums && workspace && (mode == 0 || rw_b),
                   SGLM_E_INVALID_ARG, "%s: null pointer", name);
    SGLM_CHECK_ARG(glm_power_ok(power), SGLM_E_UNSUPPORTED, "%s: power %g (supported: 1 and > 1, log link)", name, power);
    SGLM_CHECK_ARG(workspace_bytes >= sglm_pb_epilogue_workspace_bytes(T, n_models), SGLM_E_WORKSPACE,
                   "%s: workspace too small", name);
    cudaStream_t st = (cudaStream_t)stream;
    const int gx = pb_epi_grid(T);
    dim3 grid((unsigned)gx, (unsigned)ceil_div(n_models, 128));
    const int NS = mode == 0 ? PB_NS_IT : PB_NS_SC;
    const int fam = glm_family(power);
    if (mode == 0)
        pb_epilogue_launch<0>(fam, grid, st, Eta, ldb, n_models, T, Y, ldy, ycol, RW, ldrw, rw_a, rw_b, b, status, power,
                              (double *)workspace);
    else
        pb_epilogue_launch<1>(fam, grid, st, Eta, ldb, n_models, T, Y, ldy, ycol, RW, ldrw, rw_a, rw_b, b, status, power,
                              (double *)workspace);
    SGLM_LAUNCH_OK("pb_epilogue_kernel");
    const long long n_vals = (long long)n_models * NS;
    pb_finish_sums_kernel<<<(unsigned)ceil_div<long long>(n_vals, 256), 256, 0, st>>>((const double *)workspace, gx, n_vals, sums);
    SGLM_LAUNCH_OK("pb_finish_sums_kernel");
    return SGLM_OK;
}

// Poisson: mode 0: Eta <- rw (mu - y) in place, sums [B][4]; mode 1: scores, sums [B][16]  (see pb_epilogue_kernel)
extern "C" int sglm_pb_epilogue_f64(double *Eta, int64_t ldb, int32_t n_models, int64_t T, const double *Y,
                                    int64_t ldy, const int32_t *ycol, const double *RW, int64_t ldrw,
                                    const int32_t *rw_a, const int32_t *rw_b, const double *b,
                                    const int32_t *status, int32_t mode, double *sums, void *workspace,
                                    size_t workspace_bytes, void *stream) {
    return pb_epilogue("pb_epilogue", Eta, ldb, n_models, T, Y, ldy, ycol, RW, ldrw, rw_a, rw_b, b, status, 1.0, mode,
                       sums, workspace, workspace_bytes, stream);
}

// The same for the Tweedie family of `power` (1, or > 1; log link)
extern "C" int sglm_glm_epilogue_f64(double *Eta, int64_t ldb, int32_t n_models, int64_t T, const double *Y,
                                     int64_t ldy, const int32_t *ycol, const double *RW, int64_t ldrw,
                                     const int32_t *rw_a, const int32_t *rw_b, const double *b,
                                     const int32_t *status, double power, int32_t mode, double *sums, void *workspace,
                                     size_t workspace_bytes, void *stream) {
    return pb_epilogue("glm_epilogue", Eta, ldb, n_models, T, Y, ldy, ycol, RW, ldrw, rw_a, rw_b, b, status, power, mode,
                       sums, workspace, workspace_bytes, stream);
}

// One chord step of every active model: objective check / halving + right-hand sides, batched triangular solves with
// the cached factors L_of[m] of (H~ + alpha n I), intercepts + convergence.  `state_host` = the PbState fields as a
// host array of 64-bit words in declaration order (pointers, then ldw, ldq, ldb, then C | B << 32).
extern "C" int sglm_pb_step_f64(const uint64_t *state_host, const double *const *L_of, void *stream);

extern "C" int sglm_pb_state_words(void) { return (int)(sizeof(PbState) / 8); }

extern "C" int sglm_chol_solve_batched_f64(const double *const *L_of, int64_t ldq, int32_t C, const double *rhs,
                                           double *out, int64_t ld, const int32_t *flags, int32_t n_systems,
                                           void *stream);

extern "C" int sglm_enet_cd_gram_f64(const double *const *prob_Q, const double *const *prob_q,
                                     const double *const *prob_diag, const double *prob_yy, int64_t ldq, int32_t C,
                                     const int32_t *prob_of_model, const double *l1_reg, const double *l2_reg,
                                     const double *tol, const int32_t *max_iter, int32_t n_models, int32_t warm_start,
                                     int32_t do_screening, double *W, int64_t ldw, double *info, void *stream);
namespace sglm { size_t enet_cd_smem_bytes(int C); }

extern "C" int sglm_pb_step_f64(const uint64_t *state_host, const double *const *L_of, void *stream) {
    SGLM_CHECK_ARG(state_host && L_of, SGLM_E_INVALID_ARG, "pb_step: null pointer");
    static_assert(sizeof(PbState) % 8 == 0, "PbState is passed as 64-bit words");
    PbState s;
    memcpy(&s, state_host, sizeof(PbState));
    SGLM_CHECK_ARG(s.C > 0 && s.B > 0 && s.ldw >= s.C && s.ldq >= s.C && s.ldb >= s.B, SGLM_E_SHAPE, "pb_step: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)s.C * sizeof(double);
    SGLM_CHECK_ARG(smem <= 200 * 1024, SGLM_E_UNSUPPORTED, "pb_step: C=%d too large", s.C);
    SGLM_CUDA_OK(cudaFuncSetAttribute(pb_rhs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pb_rhs_kernel<<<s.B, 256, smem, st>>>(s, nullptr);
    SGLM_LAUNCH_OK("pb_rhs_kernel");
    const int rc = sglm_chol_solve_batched_f64(L_of, s.ldq, s.C, s.rhs, s.Wnew, s.ldw, s.flag, s.B, stream);
    if (rc != SGLM_OK) return rc;
    pb_finish_kernel<<<s.B, 256, 0, st>>>(s);
    SGLM_LAUNCH_OK("pb_finish_kernel");
    return SGLM_OK;
}

extern "C" size_t sglm_pb_enet_workspace_bytes(int32_t C, int64_t ldw, int32_t n_enet) {
    if (C <= 0 || ldw < C || n_enet <= 0) return 0;
    return (size_t)n_enet * (size_t)(2 * ldw + 8) * sizeof(double);
}

// sglm_pb_step_f64 for a batch with elastic-net models (l1_ratio [B]: r of every model, 0 for a ridge model): the
// models enet_models[0 .. n_enet) (those with r > 0, distinct) take a proximal-Newton step — the chord step's right-hand side, then a warm-started Gram CD solve of the
// quadratic model with the L1 term (enet_cd_gram_kernel) instead of the triangular solves; the others take the chord
// step.  L_of[m] of an elastic-net model is its factor of (H~ + alpha (1 - r) n I).  info [6 n_enet]: the inner
// solves' sglm_enet_cd_gram_f64 info (info[6k + 2] = sweeps).
extern "C" int sglm_pb_step_enet_f64(const uint64_t *state_host, const double *const *L_of, const double *l1_ratio,
                                     const int32_t *enet_models, int32_t n_enet, void *workspace,
                                     size_t workspace_bytes, double *info, void *stream) {
    SGLM_CHECK_ARG(state_host && L_of, SGLM_E_INVALID_ARG, "pb_step_enet: null pointer");
    PbState s;
    memcpy(&s, state_host, sizeof(PbState));
    SGLM_CHECK_ARG(s.C > 0 && s.B > 0 && s.ldw >= s.C && s.ldq >= s.C && s.ldb >= s.B, SGLM_E_SHAPE,
                   "pb_step_enet: bad shape");
    SGLM_CHECK_ARG(n_enet >= 1 && n_enet <= s.B, SGLM_E_SHAPE, "pb_step_enet: n_enet=%d outside [1, B=%d]", n_enet, s.B);
    SGLM_CHECK_ARG(l1_ratio && enet_models && workspace && info, SGLM_E_INVALID_ARG, "pb_step_enet: null pointer");
    SGLM_CHECK_ARG(((uintptr_t)workspace & 15) == 0, SGLM_E_ALIGN, "pb_step_enet: 16-byte alignment");
    SGLM_CHECK_ARG(workspace_bytes >= sglm_pb_enet_workspace_bytes(s.C, s.ldw, n_enet), SGLM_E_WORKSPACE,
                   "pb_step_enet: workspace too small");
    const size_t smem = (size_t)s.C * sizeof(double);
    SGLM_CHECK_ARG(smem <= 200 * 1024 && enet_cd_smem_bytes(s.C) <= 227 * 1024, SGLM_E_UNSUPPORTED,
                   "pb_step_enet: C=%d too large", s.C);
    cudaStream_t st = (cudaStream_t)stream;
    SGLM_CUDA_OK(cudaFuncSetAttribute(pb_rhs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pb_rhs_kernel<<<s.B, 256, smem, st>>>(s, l1_ratio);
    SGLM_LAUNCH_OK("pb_rhs_kernel");
    // every stepping model's chord solve: the new iterate of a ridge model, w_ridge (for yy) of an elastic-net model
    int rc = sglm_chol_solve_batched_f64(L_of, s.ldq, s.C, s.rhs, s.Wnew, s.ldw, s.flag, s.B, stream);
    if (rc != SGLM_OK) return rc;
    const PbEnetWork e = pb_enet_carve(workspace, s.ldw, n_enet);
    pb_enet_prep_kernel<<<n_enet, 256, 0, st>>>(s, l1_ratio, enet_models, e);
    SGLM_LAUNCH_OK("pb_enet_prep_kernel");
    // no screening: a yy from a borrowed factor (first step of a fold) is not a certified bound
    // warm start (bit 0) with at least one sweep (bit 1)
    rc = sglm_enet_cd_gram_f64(e.pQ, e.pq, e.pd, e.yy, s.ldq, s.C, e.pid, e.l1, e.l2, e.tol, e.max_iter, n_enet, 3, 0,
                               e.W, s.ldw, info, stream);
    if (rc != SGLM_OK) return rc;
    pb_enet_scatter_kernel<<<n_enet, 256, 0, st>>>(s, enet_models, e);
    SGLM_LAUNCH_OK("pb_enet_scatter_kernel");
    pb_finish_kernel<<<s.B, 256, 0, st>>>(s);
    SGLM_LAUNCH_OK("pb_finish_kernel");
    return SGLM_OK;
}
