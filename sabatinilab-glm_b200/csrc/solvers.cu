// Batched solvers on sufficient statistics: centring, Gram coordinate descent
// (ElasticNet / Lasso), Cholesky (Ridge / OLS), intercepts and scores-from-statistics.
//
// These replace the per-(fold, alpha, l1_ratio) scikit-learn fits that the reference
// launches one at a time from Python threads (backend/sglm_cv.py:106-170 -> backend/
// sglm.py:241 -> sklearn cd_fast / _ridge): every model of the CV grid becomes one CTA
// of a single launch, many models resident per SM.
//
// Roofline of the CD kernel: memory (rows of Q streamed from L2/HBM).  Algorithmic bytes
// per model = 8*C per coordinate update that changes w (one row of Q) — the kernel counts
// those updates (info[6m+3]) so bench.py can report sum(bytes)/time.
#include <algorithm>
#include <stdlib.h>

#include "common.cuh"

namespace sglm {

// --------------------------------------------------------------------------- centring
__global__ void __launch_bounds__(256)
center_stats_kernel(const double *__restrict__ Ap, const double *__restrict__ Am, long long ldg, int C,
                    int n_y, int y_col, int fit_intercept, double *__restrict__ Qc, long long ldq,
                    double *__restrict__ qc, double *__restrict__ xbar, double *__restrict__ diag,
                    double *__restrict__ scal) {
    const int one = C + n_y, yc = C + y_col;
    auto A = [&](int i, int j) {
        double v = Ap[(long long)i * ldg + j];
        if (Am) v -= Am[(long long)i * ldg + j];
        return v;
    };
    const double n = A(one, one);
    const double sy = A(yc, one);
    const double ybar = fit_intercept ? sy / n : 0.0;
    const int i = blockIdx.y;
    const double xi = fit_intercept ? A(i, one) / n : 0.0;
    for (int j = blockIdx.x * 256 + threadIdx.x; j < ldq; j += gridDim.x * 256) {
        double v = 0.0;
        if (j < C) {
            const double xj = fit_intercept ? A(j, one) / n : 0.0;
            v = A(i, j) - n * xi * xj;
        }
        Qc[(long long)i * ldq + j] = v;
        if (j == i) diag[i] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        qc[i] = A(i, yc) - n * xi * ybar;
        xbar[i] = xi;
        if (i == 0) {
            scal[0] = A(yc, yc) - n * ybar * ybar;
            scal[1] = n;
            scal[2] = ybar;
            scal[3] = sy;
        }
    }
}

// --------------------------------------------------------------------------- Gram CD
template <int NW>
__device__ __forceinline__ void cta_sync() {
    if (NW == 1) __syncwarp(); else __syncthreads();
}

// Reduce K partial values over the CTA.  Entries [0, K_SUM) are summed, the rest maxed.
template <int NW, int K, int K_SUM>
__device__ __forceinline__ void cta_reduce(double (&v)[K], double *scratch) {
#pragma unroll
    for (int i = 0; i < K; ++i) v[i] = (i < K_SUM) ? warp_sum(v[i]) : warp_max(v[i]);
    if (NW > 1) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < K; ++i) scratch[warp * K + i] = v[i];
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < K; ++i) {
            double a = scratch[i];
            for (int w = 1; w < NW; ++w) a = (i < K_SUM) ? a + scratch[w * K + i] : fmax(a, scratch[w * K + i]);
            v[i] = a;
        }
        __syncthreads();
    }
}

// Blocked coordinate descent, one CTA per model.
//
// Cyclic coordinate descent is sequential — coordinate j+1 needs the Qw produced by coordinate
// j — so a one-coordinate-at-a-time kernel is bound by the latency of its own instruction chain
// (measured ~2400 cycles per update, profiles/r1_cd_variants.txt).  The sweep is therefore
// blocked by 32 consecutive coordinates:
//
//   phase 1 (warp 0, registers + shuffles): lane l owns coordinate 32b+l and its Qw entry; the
//     diagonal 32x32 sub-block of Q sits in shared memory (fetched with cp.async while the
//     previous panel update runs).  The block's coordinates are visited in order, each delta is
//     broadcast with a shuffle and folded into the other lanes' Qw — the exact FMA sequence of
//     the unblocked algorithm;
//   phase 2 (panel warps): the rows of Q whose coefficient moved are streamed once
//     (RG*CH independent 16-byte loads in flight per thread) and applied to all of Qw,
//     Qw[k] = fma(delta_i, Q[i][k], Qw[k]) in coordinate order — again the same FMA sequence
//     per element, so the iterates are bit-identical to the sequential algorithm.
//
// ncu on the first blocked version showed every unit idle (L2 12 %, FP64 5 %, issue 12 %) with
// one 9-warp CTA per SM: the kernel is bound by latency x occupancy.  Hence the register diet
// (sub-block in shared memory, small panel tiles): several CTAs per SM so that one model's
// register phase overlaps other models' panel updates.
// Active sets are bit masks over the coordinate blocks (gap-safe screening only clears bits);
// the duality gap / screening / stopping rule run warp-locally in warp 0.
// Shared memory per model: w, Qw, two 32x32 sub-block buffers (no copy of Q).
__device__ __forceinline__ void cd_cp_async8(void *smem, const void *gmem) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cd_cp_async16(void *smem, const void *gmem) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cd_cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cd_cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

template <int NB, int CH, int RG, int MINB>
__global__ void __launch_bounds__((NB + 1) * 32, MINB)
enet_cd_gram_kernel(const double *const *__restrict__ prob_Q, const double *const *__restrict__ prob_q,
                    const double *const *__restrict__ prob_diag, const double *__restrict__ prob_yy,
                    long long ldq, int C, const int *__restrict__ prob_of_model,
                    const double *__restrict__ l1_reg, const double *__restrict__ l2_reg,
                    const double *__restrict__ tol_in, const int *__restrict__ max_iter_in, int warm_start,
                    int do_screening, double *__restrict__ W, long long ldw, double *__restrict__ info) {
    constexpr int NT = (NB + 1) * 32;
    constexpr int NTB = NB * 32;
    extern __shared__ __align__(16) double sm[];
    const int Cp = (C + 1) & ~1;
    const int NBLK = (C + 31) >> 5;
    double *w = sm;                                   // [Cp]
    double *Qw = w + Cp;                              // [Cp]  (element C, when C is odd, is a harmless pad)
    double *blk = Qw + Cp;                            // [2][32][32] diagonal sub-block, double buffered
    double *qd = blk + 2 * 1024;                      // [2][2][32]  q and diag of the block, double buffered
    double *dlt = qd + 128;                           // [32] deltas of the current block
    unsigned *act = reinterpret_cast<unsigned *>(dlt + 32);       // [NBLK] active-coordinate masks
    unsigned *drp = act + NBLK;                       // [NBLK] screened-out coordinates with w != 0
    unsigned *ctl = drp + NBLK;                       // [0] rows moved in the current block, [1] done
    unsigned char *pmv = reinterpret_cast<unsigned char *>(ctl + 2);     // [NBLK] coordinates moved in the last sweep

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int mdl = blockIdx.x;
    const int pid = prob_of_model[mdl];
    const double *__restrict__ Q = prob_Q[pid];
    const double *__restrict__ q = prob_q[pid];
    const double *__restrict__ dg = prob_diag[pid];
    const double yy = prob_yy[pid];
    const double l1 = l1_reg[mdl], l2 = l2_reg[mdl];
    const double d_w_tol = tol_in[mdl];
    const double tol = d_w_tol * yy;
    const int max_iter = max_iter_in[mdl];
    const bool vec2 = ((ldq & 1) == 0) && ((reinterpret_cast<uintptr_t>(Q) & 15) == 0) && (ldq >= Cp);
    const int Cp2 = Cp >> 1;
    const bool is_seq = warp == 0;
    const bool screening = do_screening && (l1 != 0.0);
    const int dbg_sel = warm_start >> 8;      // diagnostics: what info[6m+5] reports (6: start time, 7: duration, ns)
    // bit 1: at least one sweep — the start is not returned on its duality gap alone (the gap, a difference of terms of
    // size yy, cannot resolve a step below ~1e-8 |w|: a warm start at an outer iterate needs the sweep test to decide)
    const bool sweep_once = (warm_start & 2) != 0;
    warm_start &= 1;
    const unsigned long long gt_begin = global_timer_ns();

    for (int i = tid; i < Cp; i += NT) { w[i] = (warm_start && i < C) ? W[(long long)mdl * ldw + i] : 0.0; Qw[i] = 0.0; }
    if (tid == 0) { ctl[0] = 0u; ctl[1] = 0u; }
    for (int b = tid; b < NBLK; b += NT) {
        const int rem = C - (b << 5);
        act[b] = rem >= 32 ? 0xffffffffu : ((1u << rem) - 1u);
        drp[b] = 0u;
        pmv[b] = 0;
    }
    __syncthreads();

    double gap = 0.0, dual_norm = 0.0;
    int n_iter = 0;
    bool done = false;
    long long n_upd = 0, n_blk = 0, t_p1 = 0;
    const long long t_begin = clock64();

    // warp-local  Qw += a * Q[j, :]   (warm start, screening drops: rare)
    auto axpy_row_warp = [&](int j, double a) {
        const double *row = Q + (long long)j * ldq;
        for (int k = lane; k < C; k += 32) Qw[k] += a * __ldg(row + k);
        __syncwarp();
    };
    // duality gap (sklearn _cd_fast.pyx:1006-1092 gap_enet_gram), warp-local
    auto compute_gap = [&]() -> double {
        double v0 = 0, v1 = 0, v2 = 0, v3 = 0, v4 = 0, v5 = 0;   // ww, wq, wQw, |w|_1, sum xta^2, max |xta|
        for (int j = lane; j < C; j += 32) {
            const double wj = w[j], Qwj = Qw[j], qj = __ldg(q + j);
            v0 += wj * wj; v1 += wj * qj; v2 += wj * Qwj; v3 += fabs(wj);
            const double xta = (l1 == 0.0) ? (qj - Qwj) : (qj - Qwj - l2 * wj);
            v4 += xta * xta;
            v5 = fmax(v5, fabs(xta));
        }
        v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2); v3 = warp_sum(v3); v4 = warp_sum(v4);
        v5 = warp_max(v5);
        const double R2 = yy + v2 - 2.0 * v1;
        const double Ry = yy - v1;
        const double w22 = (l2 > 0.0) ? v0 : 0.0;
        if (l1 == 0.0) {
            dual_norm = v4;
            if (l2 == 0.0) return v4;
            return R2 + 0.5 * l2 * w22 - Ry + 1.0 / (2.0 * l2) * v4;
        }
        dual_norm = v5;
        const double primal = 0.5 * (R2 + l2 * w22) + l1 * v3;
        const double scale = (dual_norm > l1) ? l1 / dual_norm : 1.0;
        const double dual = -0.5 * scale * scale * (R2 + l2 * w22) + scale * Ry;
        return primal - dual;
    };
    // gap-safe screening (sklearn _cd_fast.pyx:1187-1208, :1259-1279), warp-local: clears mask
    // bits; dropped non-zero coordinates are applied afterwards in ascending order (XtA is taken
    // from the pre-drop Qw, as in sklearn).
    auto screen = [&](bool initial) {
        const double radius = sqrt(2.0 * fabs(gap)) / l1;
        const double denom = fmax(l1, dual_norm);
        bool any_drop = false;
        for (int b = 0; b < NBLK; ++b) {
            const int j = (b << 5) + lane;
            const bool in = (j < C) && ((act[b] >> lane) & 1u);
            bool keep = false, drop_nz = false;
            if (in) {
                const double djj = __ldg(dg + j);
                if (initial && djj == 0.0) {
                    w[j] = 0.0;
                } else {
                    const double xta = __ldg(q + j) - Qw[j] - l2 * w[j];
                    const double d_j = (1.0 - fabs(xta / denom)) / sqrt(djj + l2);
                    if (d_j <= radius) keep = true;
                    else if (w[j] != 0.0) drop_nz = true;
                }
            }
            const unsigned km = __ballot_sync(0xffffffffu, keep), dm = __ballot_sync(0xffffffffu, drop_nz);
            if (lane == 0) { act[b] = km; drp[b] = dm; }
            any_drop |= (dm != 0);
        }
        __syncwarp();
        if (any_drop) {
            for (int b = 0; b < NBLK; ++b) {
                unsigned dm = drp[b];
                while (dm) {
                    const int j = (b << 5) + __ffs(dm) - 1;
                    dm &= dm - 1;
                    const double wj = w[j];
                    __syncwarp();
                    axpy_row_warp(j, -wj);
                    if (lane == 0) w[j] = 0.0;
                    ++n_upd;
                    __syncwarp();
                }
            }
        }
    };

    if (is_seq) {
        if (warm_start) {
            for (int j = 0; j < C; ++j) {
                const double wj = w[j];
                if (wj != 0.0) { axpy_row_warp(j, wj); ++n_upd; }
            }
        }
        gap = compute_gap();
        done = (!sweep_once && gap >= 0.0 && gap <= tol) || max_iter <= 0;
        if (!done && screening) screen(true);
        if (lane == 0) ctl[1] = done ? 1u : 0u;
    }
    __syncthreads();

    // asynchronous fetch of block b's diagonal sub-block, q and diag into buffer `buf` (warp 0)
    auto fetch_block = [&](int b, int buf) {
        const int j_l = (b << 5) + lane;
        double *dst = blk + buf * 1024;
        if (j_l < C) {
#pragma unroll 8
            for (int i = 0; i < 32; ++i) {
                const int ji = (b << 5) + i;
                if (ji < C) cd_cp_async8(dst + i * 32 + lane, Q + (long long)ji * ldq + j_l);
            }
            cd_cp_async8(qd + buf * 64 + lane, q + j_l);
            cd_cp_async8(qd + buf * 64 + 32 + lane, dg + j_l);
        }
        cd_cp_async_commit();
    };

    while (ctl[1] == 0u) {
        double wmax_l = 0.0, dwmax_l = 0.0;
        int buf = 0;
        if (is_seq) {
            int b0 = 0;
            while (b0 < NBLK && act[b0] == 0u) ++b0;
            if (b0 < NBLK) fetch_block(b0, 0);
        }
        for (int b = 0; b < NBLK; ++b) {
            const unsigned mask = act[b];
            if (mask == 0u) continue;                                     // uniform: block screened out
            if (is_seq) {
                // ---------------- phase 1: the block's coordinates, in order
                const long long t_b = clock64();
                cd_cp_async_wait_all();
                __syncwarp();
                const int j_l = (b << 5) + lane;
                const bool inb = j_l < C;
                const double *S = blk + buf * 1024;
                const double q_l = inb ? qd[buf * 64 + lane] : 0.0;
                const double d_l = inb ? qd[buf * 64 + 32 + lane] : 0.0;
                const double inv_l = (d_l != 0.0) ? 1.0 / (d_l + l2) : 1.0;
                const bool ok_l = ((mask >> lane) & 1u) && d_l != 0.0;
                const double Qw_l = inb ? Qw[j_l] : 0.0;
                const double w_l = inb ? w[j_l] : 0.0;
                // Soft-threshold update written for a short dependent chain (the 32 steps are
                // serialised through Qw_l):  with r = (q + w d) - Qw,
                //   delta = r >  l1 ? (r - l1)/den - w : r < -l1 ? (r + l1)/den - w : -w
                // evaluated as one FMA per branch from per-lane constants; w_new = w + delta.
                const double a_l = fma(w_l, d_l, q_l);
                const double k_pos = fma(-l1, inv_l, -w_l), k_neg = fma(l1, inv_l, -w_l);
                double delta_l = 0.0;
                // Every lane's candidate step from the CURRENT state, all 32 at once.  Until some coordinate
                // moves the state does not change, so the lanes whose candidate is zero need no turn: the
                // sweep jumps to the first lane (in coordinate order) whose candidate is non-zero, applies it
                // exactly as the sequential algorithm would, and re-evaluates the lanes after it.  A sparse
                // model pays for the coordinates that move, not for 32 serial steps per block.
                // r = (q + w d) - Qw is carried directly: an update of Qw by +delta_i S_il is r -= delta_i S_il, one FMA
                // on the dependent chain instead of an FMA followed by a subtraction (the chain of 32 serial steps
                // per block is what bounds the heaviest models)
                double r_l = a_l - Qw_l;
                auto candidate = [&]() -> double {
                    const double r = r_l;
                    const double dpos = fma(r, inv_l, k_pos), dneg = fma(r, inv_l, k_neg);
                    const double dc = cd_soft_select(r, l1, dpos, dneg, -w_l);
                    return ok_l ? dc : 0.0;
                };
                if (pmv[b] >= 20) {
                    // dense block (20+ coordinates moved in the last sweep): the straight 32-step chain, no
                    // vote on the dependent path
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        if (!((mask >> i) & 1u)) continue;                // uniform: coordinate screened out
                        const double s_il = inb ? S[i * 32 + lane] : 0.0;
                        const double dc = candidate();
                        const double di = __shfl_sync(0xffffffffu, dc, i);
                        if (lane == i) delta_l = dc;
                        r_l = fma(-di, s_il, r_l);
                    }
                } else {
                    double dc = candidate();
                    unsigned todo = mask;
                    while (true) {
                        const unsigned mv = __ballot_sync(0xffffffffu, dc != 0.0) & todo;
                        if (!mv) break;
                        const int i = __ffs(mv) - 1;
                        const double di = __shfl_sync(0xffffffffu, dc, i);
                        if (lane == i) delta_l = dc;
                        r_l = fma(-di, inb ? S[i * 32 + lane] : 0.0, r_l);
                        todo &= ~((2u << i) - 1u);                        // coordinates up to i have had their turn
                        if (!todo) break;
                        dc = candidate();
                    }
                }
                const double w_new_l = w_l + delta_l;
                const unsigned nz = __ballot_sync(0xffffffffu, delta_l != 0.0);
                if (ok_l) {
                    dwmax_l = fmax(dwmax_l, fabs(delta_l));
                    wmax_l = fmax(wmax_l, fabs(w_new_l));
                }
                if (delta_l != 0.0) w[j_l] = w_new_l;
                dlt[lane] = delta_l;
                if (lane == 0) { ctl[0] = nz; pmv[b] = (unsigned char)__popc(nz); }
                n_upd += __popc(nz);
                ++n_blk;
                int bn = b + 1;
                while (bn < NBLK && act[bn] == 0u) ++bn;
                if (bn < NBLK) fetch_block(bn, buf ^ 1);                  // lands during phase 2
                buf ^= 1;
                t_p1 += clock64() - t_b;
            }
            __syncthreads();                                              // deltas and moved-row mask published
            // ---------------- phase 2: Qw += sum_i delta_i Q[32b+i, :]   (rows in coordinate order)
            const unsigned um = ctl[0];
            if (um && !is_seq) {
                const int bt = tid - 32;
                const long long row0 = (long long)(b << 5);
                if (vec2) {
                    const double2 *Q2 = reinterpret_cast<const double2 *>(Q) + row0 * (ldq >> 1);
                    const long long ld2 = ldq >> 1;
                    double2 *Qw2 = reinterpret_cast<double2 *>(Qw);
                    for (int c0 = bt; c0 < Cp2; c0 += NTB * CH) {
                        double2 acc[CH];
                        bool okc[CH];
#pragma unroll
                        for (int u = 0; u < CH; ++u) {
                            okc[u] = c0 + u * NTB < Cp2;
                            acc[u] = okc[u] ? Qw2[c0 + u * NTB] : make_double2(0.0, 0.0);
                        }
                        unsigned rem = um;
                        while (rem) {
                            double2 v[RG][CH];
                            double d[RG];
#pragma unroll
                            for (int r = 0; r < RG; ++r) {
                                const int i = rem ? (__ffs(rem) - 1) : 0;
                                d[r] = rem ? dlt[i] : 0.0;
                                rem &= rem - 1;                           // (0 & -1) stays 0
                                const double2 *row = Q2 + (long long)i * ld2 + c0;
#pragma unroll
                                for (int u = 0; u < CH; ++u)
                                    v[r][u] = okc[u] ? __ldg(row + u * NTB) : make_double2(0.0, 0.0);
                            }
#pragma unroll
                            for (int r = 0; r < RG; ++r)
#pragma unroll
                                for (int u = 0; u < CH; ++u) {
                                    acc[u].x = fma(d[r], v[r][u].x, acc[u].x);
                                    acc[u].y = fma(d[r], v[r][u].y, acc[u].y);
                                }
                        }
#pragma unroll
                        for (int u = 0; u < CH; ++u)
                            if (okc[u]) Qw2[c0 + u * NTB] = acc[u];
                    }
                } else {
                    for (int k = bt; k < C; k += NTB) {
                        double a = Qw[k];
                        unsigned rem = um;
                        while (rem) {
                            const int i = __ffs(rem) - 1;
                            rem &= rem - 1;
                            a = fma(dlt[i], __ldg(Q + (row0 + i) * ldq + k), a);
                        }
                        Qw[k] = a;
                    }
                }
            }
            __syncthreads();                                              // Qw updated
        }
        // ---------------- end of sweep: stopping rule / gap / screening
        if (is_seq) {
            const double w_max = warp_max(wmax_l), d_w_max = warp_max(dwmax_l);
            if (w_max == 0.0 || d_w_max / w_max <= d_w_tol || n_iter == max_iter - 1) {
                gap = compute_gap();
                if (gap <= tol) done = true;
                else if (screening) screen(false);
            }
            ++n_iter;
            if (n_iter >= max_iter) done = true;
            if (lane == 0) ctl[1] = done ? 1u : 0u;
        }
        __syncthreads();
    }
    if (is_seq) {
        for (int j = lane; j < C; j += 32) W[(long long)mdl * ldw + j] = w[j];
        if (lane == 0) {
            info[6 * mdl + 0] = gap;
            info[6 * mdl + 1] = tol;
            info[6 * mdl + 2] = (double)n_iter;
            info[6 * mdl + 3] = (double)n_upd;
            info[6 * mdl + 4] = (double)n_blk;
            info[6 * mdl + 5] = dbg_sel == 6 ? (double)gt_begin : dbg_sel == 7 ? (double)(global_timer_ns() - gt_begin)
                              : (double)t_p1 / (double)max(1LL, clock64() - t_begin);   // share of time in the register phase
        }
    }
}

// --------------------------------------------------------------------------- Cholesky (Ridge / OLS)
constexpr int RC_NB = 32;
constexpr int RC_THREADS = 256;

__global__ void __launch_bounds__(RC_THREADS)
ridge_cholesky_kernel(const double *__restrict__ Qc, long long ldq, const double *__restrict__ qc, int C,
                      const double *__restrict__ alpha, double *__restrict__ W, long long ldw,
                      int *__restrict__ status, double *__restrict__ work) {
    extern __shared__ __align__(16) double sh[];
    double *D = sh;                          // [32][33] diagonal block
    double *Pi = D + RC_NB * 33;             // [64][33]
    double *Pj = Pi + 64 * 33;               // [64][33]
    double *wv = Pj + 64 * 33;               // [C] solution vector
    __shared__ int bad;

    const int kq = blockIdx.x, tid = threadIdx.x;
    const double a = alpha[kq];
    double *M = work + (long long)kq * (C + 1) * ldq;
    if (tid == 0) bad = 0;
    // pivots at rounding-noise level (relative to the largest diagonal entry) mark a numerically rank-deficient
    // system: status bit 1 (the factorisation still completes); a non-positive pivot sets bit 0
    __shared__ double s_dmax[RC_THREADS / 32];
    {
        double dm = 0.0;
        for (int j = tid; j < C; j += RC_THREADS) dm = fmax(dm, fabs(Qc[(long long)j * ldq + j] + a));
        dm = warp_max(dm);
        if ((tid & 31) == 0) s_dmax[tid >> 5] = dm;
    }
    __syncthreads();
    double tiny_pivot = 0.0;
    for (int w_ = 0; w_ < RC_THREADS / 32; ++w_) tiny_pivot = fmax(tiny_pivot, s_dmax[w_]);
    tiny_pivot *= 1e-11;

    // M = lower(Qc) + a I ; row C = qc'
    for (long long e = tid; e < (long long)(C + 1) * C; e += RC_THREADS) {
        const int i = (int)(e / C), j = (int)(e - (long long)i * C);
        if (i == C) M[(long long)i * ldq + j] = qc[j];
        else if (j <= i) M[(long long)i * ldq + j] = Qc[(long long)i * ldq + j] + (i == j ? a : 0.0);
    }
    __syncthreads();

    for (int k0 = 0; k0 < C; k0 += RC_NB) {
        const int nb = min(RC_NB, C - k0);
        // 1. diagonal block -> smem, unblocked Cholesky by warp 0
        for (int e = tid; e < nb * nb; e += RC_THREADS) {
            const int r = e / nb, c = e - r * nb;
            D[r * 33 + c] = (c <= r) ? M[(long long)(k0 + r) * ldq + k0 + c] : 0.0;
        }
        __syncthreads();
        if (tid < 32) {
            for (int c = 0; c < nb; ++c) {
                double d = D[c * 33 + c];
                if (!(d > 0.0)) { if (tid == 0) bad |= 1; d = nan(""); }
                else if (d <= tiny_pivot) { if (tid == 0) bad |= 2; }
                const double l = sqrt(d);
                __syncwarp();
                if (tid == 0) D[c * 33 + c] = l;
                for (int r = c + 1 + tid; r < nb; r += 32) D[r * 33 + c] /= l;
                __syncwarp();
                // trailing update inside the block: D[r][cc] -= D[r][c]*D[cc][c] for c < cc <= r
                for (int e = tid; e < nb * nb; e += 32) {
                    const int r = e / nb, cc = e - r * nb;
                    if (cc > c && cc <= r) D[r * 33 + cc] -= D[r * 33 + c] * D[cc * 33 + c];
                }
                __syncwarp();
            }
        }
        __syncthreads();
        for (int e = tid; e < nb * nb; e += RC_THREADS) {
            const int r = e / nb, c = e - r * nb;
            if (c <= r) M[(long long)(k0 + r) * ldq + k0 + c] = D[r * 33 + c];
        }
        // 2. panel solve: rows below the block (incl. the rhs row C): x L_kk' = M[i, k0:k0+nb]
        for (int i = k0 + nb + tid; i <= C; i += RC_THREADS) {
            double x[RC_NB];
            double *row = M + (long long)i * ldq + k0;
#pragma unroll
            for (int c = 0; c < RC_NB; ++c) x[c] = (c < nb) ? row[c] : 0.0;
#pragma unroll
            for (int c = 0; c < RC_NB; ++c) {
                if (c < nb) {
                    double s = x[c];
#pragma unroll
                    for (int r = 0; r < RC_NB; ++r)
                        if (r < c) s -= x[r] * D[c * 33 + r];
                    x[c] = s / D[c * 33 + c];
                }
            }
#pragma unroll
            for (int c = 0; c < RC_NB; ++c)
                if (c < nb) row[c] = x[c];
        }
        __syncthreads();
        // 3. trailing update with 64x64 tiles: M[i][j] -= sum_c M[i][k0+c] M[j][k0+c]
        const int lo = k0 + nb;
        if (lo <= C) {
            const int ty = tid >> 4, tx = tid & 15;
            for (int i0 = lo; i0 <= C; i0 += 64) {
                for (int e = tid; e < 64 * RC_NB; e += RC_THREADS) {
                    const int r = e >> 5, c = e & 31;
                    Pi[r * 33 + c] = (i0 + r <= C && c < nb) ? M[(long long)(i0 + r) * ldq + k0 + c] : 0.0;
                }
                for (int j0 = lo; j0 <= i0 && j0 < C; j0 += 64) {
                    __syncthreads();
                    for (int e = tid; e < 64 * RC_NB; e += RC_THREADS) {
                        const int r = e >> 5, c = e & 31;
                        Pj[r * 33 + c] = (j0 + r < C && c < nb) ? M[(long long)(j0 + r) * ldq + k0 + c] : 0.0;
                    }
                    __syncthreads();
                    double acc[4][4];
#pragma unroll
                    for (int u = 0; u < 4; ++u)
#pragma unroll
                        for (int v = 0; v < 4; ++v) acc[u][v] = 0.0;
#pragma unroll 8
                    for (int c = 0; c < RC_NB; ++c) {
                        double pa[4], pb[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) pa[u] = Pi[(ty + 16 * u) * 33 + c];
#pragma unroll
                        for (int v = 0; v < 4; ++v) pb[v] = Pj[(tx + 16 * v) * 33 + c];
#pragma unroll
                        for (int u = 0; u < 4; ++u)
#pragma unroll
                            for (int v = 0; v < 4; ++v) acc[u][v] += pa[u] * pb[v];
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u)
#pragma unroll
                        for (int v = 0; v < 4; ++v) {
                            const int i = i0 + ty + 16 * u, j = j0 + tx + 16 * v;
                            if (i <= C && j < C && j <= i) M[(long long)i * ldq + j] -= acc[u][v];
                        }
                }
                __syncthreads();
            }
        }
        __syncthreads();
    }

    // row C now holds y with L y = qc.  Back substitution L' w = y, blocked from the end.
    for (int j = tid; j < C; j += RC_THREADS) wv[j] = M[(long long)C * ldq + j];
    __syncthreads();
    const int n_blk = (C + RC_NB - 1) / RC_NB;
    for (int b = n_blk - 1; b >= 0; --b) {
        const int k0 = b * RC_NB, nb = min(RC_NB, C - k0);
        for (int e = tid; e < nb * nb; e += RC_THREADS) {
            const int r = e / nb, c = e - r * nb;
            D[r * 33 + c] = (c <= r) ? M[(long long)(k0 + r) * ldq + k0 + c] : 0.0;
        }
        __syncthreads();
        if (tid == 0) {
            for (int c = nb - 1; c >= 0; --c) {
                double s = wv[k0 + c];
                for (int r = c + 1; r < nb; ++r) s -= D[r * 33 + c] * wv[k0 + r];
                wv[k0 + c] = s / D[c * 33 + c];
            }
        }
        __syncthreads();
        for (int i = tid; i < k0; i += RC_THREADS) {
            double s = wv[i];
            for (int r = 0; r < nb; ++r) s -= M[(long long)(k0 + r) * ldq + i] * wv[k0 + r];
            wv[i] = s;
        }
        __syncthreads();
    }
    for (int j = tid; j < C; j += RC_THREADS) W[(long long)kq * ldw + j] = wv[j];
    if (tid == 0) status[kq] = bad;
}

// --------------------------------------------------------------------------- Cholesky, left-looking form
// Same system and outputs as ridge_cholesky_kernel.  The right-looking form rewrites the whole trailing
// matrix after every 32-column panel (C^3/(3*32) * 16 bytes of global traffic per system: 0.9 GB at
// C = 1220, 35 ms with 120 systems in flight — scripts/c2_timeline.py); here a block column is brought up
// to date ONCE from the factor columns to its left (reads only: C^3/(6*32) * 8 bytes), factored and never
// touched again.  Row tiles of 256 rows x 32 columns, 8 x 4 accumulators per thread, the rhs travels as
// row C (forward substitution for free), back substitution as before.
constexpr int LL_RT = 256;      // rows per tile

constexpr int LL_LD = 34;       // padded row length of the staged factor tiles (16-byte aligned rows)

__global__ void __launch_bounds__(RC_THREADS)
ridge_cholesky_ll_kernel(const double *__restrict__ Qc, long long ldq, const double *__restrict__ qc, int C,
                         const double *__restrict__ alpha, double *__restrict__ W, long long ldw,
                         int *__restrict__ status, double *__restrict__ work) {
    extern __shared__ __align__(16) double sh[];
    double *D = sh;                                  // [32][33] diagonal block (steps 2, 3, back substitution)
    double *LJ = D + RC_NB * 33;                     // [2][32][34] factor rows of the block column, double buffered
    double *LI = LJ + 2 * RC_NB * LL_LD;             // [2][256][34] factor rows of the row tile, double buffered
    double *wv = LI + 2 * LL_RT * LL_LD;             // [C] solution vector
    __shared__ int bad;

    const int kq = blockIdx.x, tid = threadIdx.x;
    const double a = alpha[kq];
    double *M = work + (long long)kq * (C + 1) * ldq;
    if (tid == 0) bad = 0;
    // pivots at rounding-noise level (relative to the largest diagonal entry) mark a numerically rank-deficient
    // system: status bit 1 (the factorisation still completes); a non-positive pivot sets bit 0
    __shared__ double s_dmax[RC_THREADS / 32];
    {
        double dm = 0.0;
        for (int j = tid; j < C; j += RC_THREADS) dm = fmax(dm, fabs(Qc[(long long)j * ldq + j] + a));
        dm = warp_max(dm);
        if ((tid & 31) == 0) s_dmax[tid >> 5] = dm;
    }
    __syncthreads();
    double tiny_pivot = 0.0;
    for (int w_ = 0; w_ < RC_THREADS / 32; ++w_) tiny_pivot = fmax(tiny_pivot, s_dmax[w_]);
    tiny_pivot *= 1e-11;
    const int ty = tid >> 3, tx = tid & 7;      // rows ty + 32u (u < 8), columns tx + 8v (v < 4)
    const bool al16 = ((ldq & 1) == 0) && ((reinterpret_cast<uintptr_t>(M) & 15) == 0);

    for (int j0 = 0; j0 < C; j0 += RC_NB) {
        const int nb = min(RC_NB, C - j0);
        // 1. block column j0: A[i][c] = M0[i][j0+c] - sum_{k<j0} L[i][k] L[j0+c][k]  for rows i = j0..C (row C = rhs)
        for (int i0 = j0; i0 <= C; i0 += LL_RT) {
            double acc[8][4];
#pragma unroll
            for (int u = 0; u < 8; ++u)
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const int i = i0 + ty + 32 * u, c = tx + 8 * v, j = j0 + c;
                    double x = 0.0;
                    if (c < nb && i <= C) {
                        if (i == C) x = qc[j];
                        else if (j <= i) x = Qc[(long long)i * ldq + j] + (i == j ? a : 0.0);
                    }
                    acc[u][v] = x;
                }
            // asynchronous staging of the factor rows of chunk k0 (16-byte copies; rows past C are zero)
            auto stage = [&](int k0, int buf) {
                double *li = LI + buf * LL_RT * LL_LD, *lj = LJ + buf * RC_NB * LL_LD;
                for (int e = tid; e < (LL_RT + RC_NB) * 16; e += RC_THREADS) {
                    const int r = e >> 4, ch = (e & 15) * 2;
                    const bool isj = r >= LL_RT;
                    const int row = isj ? j0 + (r - LL_RT) : i0 + r;
                    double *dst = isj ? lj + (r - LL_RT) * LL_LD + ch : li + r * LL_LD + ch;
                    const bool ok = isj ? (r - LL_RT) < nb : row <= C;
                    if (ok && al16) {
                        cd_cp_async16(dst, M + (long long)row * ldq + k0 + ch);
                    } else if (ok) {
                        dst[0] = M[(long long)row * ldq + k0 + ch];
                        dst[1] = M[(long long)row * ldq + k0 + ch + 1];
                    } else {
                        dst[0] = 0.0; dst[1] = 0.0;
                    }
                }
                cd_cp_async_commit();
            };
            __syncthreads();                                   // previous tile / step done with the buffers
            int buf = 0;
            if (j0 > 0) stage(0, 0);
            for (int k0 = 0; k0 < j0; k0 += RC_NB) {
                const bool more = k0 + RC_NB < j0;
                if (more) stage(k0 + RC_NB, buf ^ 1);
                if (more) asm volatile("cp.async.wait_group 1;\n" ::: "memory");
                else cd_cp_async_wait_all();
                __syncthreads();
                const double *li = LI + buf * LL_RT * LL_LD, *lj = LJ + buf * RC_NB * LL_LD;
#pragma unroll 4
                for (int c = 0; c < RC_NB; ++c) {
                    double pa[8], pb[4];
#pragma unroll
                    for (int u = 0; u < 8; ++u) pa[u] = li[(ty + 32 * u) * LL_LD + c];
#pragma unroll
                    for (int v = 0; v < 4; ++v) pb[v] = lj[(tx + 8 * v) * LL_LD + c];
#pragma unroll
                    for (int u = 0; u < 8; ++u)
#pragma unroll
                        for (int v = 0; v < 4; ++v) acc[u][v] -= pa[u] * pb[v];
                }
                __syncthreads();                               // buffer `buf` may be refilled by the next stage()
                buf ^= 1;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u)
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const int i = i0 + ty + 32 * u, c = tx + 8 * v;
                    if (c < nb && i <= C && (i == C || j0 + c <= i)) M[(long long)i * ldq + j0 + c] = acc[u][v];
                }
        }
        __syncthreads();
        // 2. diagonal block -> smem, unblocked Cholesky by warp 0
        for (int e = tid; e < nb * nb; e += RC_THREADS) {
            const int r = e / nb, c = e - r * nb;
            D[r * 33 + c] = (c <= r) ? M[(long long)(j0 + r) * ldq + j0 + c] : 0.0;
        }
        __syncthreads();
        if (tid < 32) {
            for (int c = 0; c < nb; ++c) {
                double d = D[c * 33 + c];
                if (!(d > 0.0)) { if (tid == 0) bad |= 1; d = nan(""); }
                else if (d <= tiny_pivot) { if (tid == 0) bad |= 2; }
                const double l = sqrt(d);
                __syncwarp();
                if (tid == 0) D[c * 33 + c] = l;
                for (int r = c + 1 + tid; r < nb; r += 32) D[r * 33 + c] /= l;
                __syncwarp();
                for (int e = tid; e < nb * nb; e += 32) {
                    const int r = e / nb, cc = e - r * nb;
                    if (cc > c && cc <= r) D[r * 33 + cc] -= D[r * 33 + c] * D[cc * 33 + c];
                }
                __syncwarp();
            }
        }
        __syncthreads();
        for (int e = tid; e < nb * nb; e += RC_THREADS) {
            const int r = e / nb, c = e - r * nb;
            if (c <= r) M[(long long)(j0 + r) * ldq + j0 + c] = D[r * 33 + c];
        }
        // 3. panel solve: rows below the block (incl. the rhs row C): x L_jj' = A[i, :]
        for (int i = j0 + nb + tid; i <= C; i += RC_THREADS) {
            double x[RC_NB];
            double *row = M + (long long)i * ldq + j0;
#pragma unroll
            for (int c = 0; c < RC_NB; ++c) x[c] = (c < nb) ? row[c] : 0.0;
#pragma unroll
            for (int c = 0; c < RC_NB; ++c) {
                if (c < nb) {
                    double sv = x[c];
#pragma unroll
                    for (int r = 0; r < RC_NB; ++r)
                        if (r < c) sv -= x[r] * D[c * 33 + r];
                    x[c] = sv / D[c * 33 + c];
                }
            }
#pragma unroll
            for (int c = 0; c < RC_NB; ++c)
                if (c < nb) row[c] = x[c];
        }
        __syncthreads();
    }

    // row C now holds y with L y = qc.  Back substitution L' w = y, blocked from the end.
    for (int j = tid; j < C; j += RC_THREADS) wv[j] = M[(long long)C * ldq + j];
    __syncthreads();
    const int n_blk = (C + RC_NB - 1) / RC_NB;
    for (int b = n_blk - 1; b >= 0; --b) {
        const int k0 = b * RC_NB, nb = min(RC_NB, C - k0);
        for (int e = tid; e < nb * nb; e += RC_THREADS) {
            const int r = e / nb, c = e - r * nb;
            D[r * 33 + c] = (c <= r) ? M[(long long)(k0 + r) * ldq + k0 + c] : 0.0;
        }
        __syncthreads();
        if (tid == 0) {
            for (int c = nb - 1; c >= 0; --c) {
                double sv = wv[k0 + c];
                for (int r = c + 1; r < nb; ++r) sv -= D[r * 33 + c] * wv[k0 + r];
                wv[k0 + c] = sv / D[c * 33 + c];
            }
        }
        __syncthreads();
        for (int i = tid; i < k0; i += RC_THREADS) {
            double sv = wv[i];
            for (int r = 0; r < nb; ++r) sv -= M[(long long)(k0 + r) * ldq + i] * wv[k0 + r];
            wv[i] = sv;
        }
        __syncthreads();
    }
    for (int j = tid; j < C; j += RC_THREADS) W[(long long)kq * ldw + j] = wv[j];
    if (tid == 0) status[kq] = bad;
}

// --------------------------------------------------------------------------- solve with a stored Cholesky factor
// L L' x = rhs with the lower-triangular factor that ridge_cholesky_kernel leaves in its work buffer
// (row-major, L[i][j] for j <= i).  One CTA: blocked forward substitution (32 unknowns by one warp, then
// every thread corrects its rows with 32 contiguous factor entries) and blocked back substitution
// (column access of L is contiguous across threads).  Used by the Poisson Newton iteration to reuse a
// Hessian factor over several steps (chord iterations): 2 * C^2/2 * 8 bytes of factor traffic per solve.
__device__ __forceinline__ void chol_solve_body(const double *__restrict__ L, long long ldq, int C,
                                                const double *__restrict__ rhs, double *__restrict__ out, double *sh);

__global__ void __launch_bounds__(RC_THREADS)
chol_solve_kernel(const double *__restrict__ L, long long ldq, int C, const double *__restrict__ rhs,
                  double *__restrict__ out) {
    extern __shared__ __align__(16) double sh[];
    chol_solve_body(L, ldq, C, rhs, out, sh);
}

// One CTA per system: factor pointers L_of[s], right-hand sides / solutions as rows of [n][ld] matrices; systems whose
// flag is not 1 are skipped (the batched Poisson Newton iteration solves only the models that take a step).
__global__ void __launch_bounds__(RC_THREADS)
chol_solve_batched_kernel(const double *const *__restrict__ L_of, long long ldq, int C, const double *__restrict__ rhs,
                          double *__restrict__ out, long long ld, const int *__restrict__ flags) {
    extern __shared__ __align__(16) double sh[];
    const int s = blockIdx.x;
    if (flags && flags[s] != 1) return;
    chol_solve_body(L_of[s], ldq, C, rhs + (long long)s * ld, out + (long long)s * ld, sh);
}

__device__ __forceinline__ void chol_solve_body(const double *__restrict__ L, long long ldq, int C,
                                                const double *__restrict__ rhs, double *__restrict__ out, double *sh) {
    double *D = sh;                          // [32][33] diagonal block
    double *xv = D + RC_NB * 33;             // [C] running right-hand side / solution
    const int tid = threadIdx.x;
    for (int j = tid; j < C; j += RC_THREADS) xv[j] = rhs[j];
    __syncthreads();
    const int n_blk = (C + RC_NB - 1) / RC_NB;
    for (int b = 0; b < n_blk; ++b) {                       // forward: L y = rhs
        const int k0 = b * RC_NB, nb = min(RC_NB, C - k0);
        for (int e = tid; e < nb * nb; e += RC_THREADS) {
            const int r = e / nb, c = e - r * nb;
            D[r * 33 + c] = (c <= r) ? L[(long long)(k0 + r) * ldq + k0 + c] : 0.0;
        }
        __syncthreads();
        if (tid == 0) {
            for (int c = 0; c < nb; ++c) {
                double s = xv[k0 + c];
                for (int r = 0; r < c; ++r) s -= D[c * 33 + r] * xv[k0 + r];
                xv[k0 + c] = s / D[c * 33 + c];
            }
        }
        __syncthreads();
        for (int i = k0 + nb + tid; i < C; i += RC_THREADS) {
            const double *row = L + (long long)i * ldq + k0;
            double s = xv[i];
            for (int c = 0; c < nb; ++c) s -= row[c] * xv[k0 + c];
            xv[i] = s;
        }
        __syncthreads();
    }
    for (int b = n_blk - 1; b >= 0; --b) {                  // backward: L' x = y
        const int k0 = b * RC_NB, nb = min(RC_NB, C - k0);
        for (int e = tid; e < nb * nb; e += RC_THREADS) {
            const int r = e / nb, c = e - r * nb;
            D[r * 33 + c] = (c <= r) ? L[(long long)(k0 + r) * ldq + k0 + c] : 0.0;
        }
        __syncthreads();
        if (tid == 0) {
            for (int c = nb - 1; c >= 0; --c) {
                double s = xv[k0 + c];
                for (int r = c + 1; r < nb; ++r) s -= D[r * 33 + c] * xv[k0 + r];
                xv[k0 + c] = s / D[c * 33 + c];
            }
        }
        __syncthreads();
        for (int i = tid; i < k0; i += RC_THREADS) {
            double s = xv[i];
            for (int r = 0; r < nb; ++r) s -= L[(long long)(k0 + r) * ldq + i] * xv[k0 + r];
            xv[i] = s;
        }
        __syncthreads();
    }
    for (int j = tid; j < C; j += RC_THREADS) out[j] = xv[j];
}

// --------------------------------------------------------------------------- intercept + evaluation vectors
__global__ void __launch_bounds__(128)
finalize_models_kernel(const double *__restrict__ W, long long ldw, int C, int n_y,
                       const int *__restrict__ y_col_of_model, const double *const *__restrict__ xbar_of_model,
                       const double *__restrict__ ybar_of_model, double *__restrict__ intercept,
                       double *__restrict__ V, long long ldv) {
    const int m = blockIdx.x, tid = threadIdx.x;
    const double *w = W + (long long)m * ldw;
    const double *xb = xbar_of_model ? xbar_of_model[m] : nullptr;
    double s = 0.0;
    if (xb) for (int j = tid; j < C; j += 128) s += xb[j] * w[j];
    s = warp_sum(s);
    __shared__ double part[4];
    __shared__ double bsh;
    if ((tid & 31) == 0) part[tid >> 5] = s;
    __syncthreads();
    if (tid == 0) {
        const double b = xb ? (ybar_of_model[m] - (part[0] + part[1] + part[2] + part[3])) : 0.0;
        intercept[m] = b;
        bsh = b;
    }
    __syncthreads();
    if (V) {
        double *v = V + (long long)m * ldv;
        const int yc = y_col_of_model ? y_col_of_model[m] : 0;
        for (int j = tid; j < ldv; j += 128) {
            double x = 0.0;
            if (j < C) x = -w[j];
            else if (j < C + n_y) x = (j - C == yc) ? 1.0 : 0.0;
            else if (j == C + n_y) x = -bsh;
            v[j] = x;
        }
    }
}

// --------------------------------------------------------------------------- quadratic forms  v' A v
constexpr int QF_THREADS = 256;

template <int QF_MB>           // models per CTA: every row of A is streamed once for QF_MB quadratic forms
__global__ void __launch_bounds__(QF_THREADS)
quadform_kernel(const double *__restrict__ A, long long lda, int n, const double *__restrict__ V,
                long long ldv, int n_models, double *__restrict__ out) {
    extern __shared__ __align__(16) double vs[];   // [QF_MB][n]
    const int m0 = blockIdx.x * QF_MB, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nm = min(QF_MB, n_models - m0);
    for (int e = tid; e < QF_MB * n; e += QF_THREADS) {
        const int mm = e / n, j = e - mm * n;
        vs[e] = (mm < nm) ? V[(long long)(m0 + mm) * ldv + j] : 0.0;
    }
    __syncthreads();
    double acc[QF_MB];
#pragma unroll
    for (int mm = 0; mm < QF_MB; ++mm) acc[mm] = 0.0;
    // rows i = warp + 8 * (blockIdx.y + k * gridDim.y): the row splits of gridDim.y > 1 write partial sums
    for (int i = warp + (QF_THREADS / 32) * blockIdx.y; i < n; i += (QF_THREADS / 32) * gridDim.y) {
        const double *row = A + (long long)i * lda;
        double d[QF_MB];
#pragma unroll
        for (int mm = 0; mm < QF_MB; ++mm) d[mm] = 0.0;
        for (int j = lane; j < n; j += 32) {
            const double aij = __ldg(row + j);
#pragma unroll
            for (int mm = 0; mm < QF_MB; ++mm) d[mm] += aij * vs[mm * n + j];
        }
        // v' A v is linear in the lane partials of row i, so they are weighted by v_i here and reduced over
        // the warp once at the end (a shuffle reduction per row and model was most of this kernel's time)
#pragma unroll
        for (int mm = 0; mm < QF_MB; ++mm) acc[mm] += d[mm] * vs[mm * n + i];
    }
#pragma unroll
    for (int mm = 0; mm < QF_MB; ++mm) acc[mm] = warp_sum(acc[mm]);
    __shared__ double red[QF_THREADS / 32][QF_MB];
    if (lane == 0)
        for (int mm = 0; mm < QF_MB; ++mm) red[warp][mm] = acc[mm];
    __syncthreads();
    if (tid < nm) {
        double s = 0.0;
        for (int w = 0; w < QF_THREADS / 32; ++w) s += red[w][tid];
        out[(long long)blockIdx.y * n_models + m0 + tid] = s;
    }
}

}  // namespace sglm

using namespace sglm;

extern "C" int sglm_center_stats_f64(const double *A_plus, const double *A_minus, int64_t ldg, int32_t C,
                                     int32_t n_y, int32_t y_col, int32_t fit_intercept, double *Qc,
                                     int64_t ldq, double *qc, double *xbar, double *diag, double *scal,
                                     void *stream) {
    SGLM_CHECK_ARG(C > 0 && n_y > 0 && y_col >= 0 && y_col < n_y, SGLM_E_SHAPE, "center_stats: bad shape");
    SGLM_CHECK_ARG(A_plus && Qc && qc && xbar && diag && scal, SGLM_E_INVALID_ARG, "center_stats: null pointer");
    SGLM_CHECK_ARG(ldg >= C + n_y + 1 && ldq >= C, SGLM_E_SHAPE, "center_stats: leading dimension too small");
    dim3 grid((unsigned)std::min<long long>(ceil_div<long long>(ldq, 256), 64), (unsigned)C);
    center_stats_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A_plus, A_minus, ldg, C, n_y, y_col,
                                                                 fit_intercept, Qc, ldq, qc, xbar, diag, scal);
    SGLM_LAUNCH_OK("center_stats_kernel");
    return SGLM_OK;
}

namespace sglm { size_t enet_cd_smem_bytes(int C); }
size_t sglm::enet_cd_smem_bytes(int C) {
    const int Cp = (C + 1) & ~1, nblk = (C + 31) / 32;
    return (size_t)(2 * Cp + 2 * 1024 + 128 + 32) * sizeof(double) + (size_t)(2 * nblk + 2) * sizeof(unsigned) + (size_t)nblk + 64;
}

extern "C" int sglm_enet_cd_gram_f64(const double *const *prob_Q, const double *const *prob_q,
                                     const double *const *prob_diag, const double *prob_yy, int64_t ldq, int32_t C,
                                     const int32_t *prob_of_model, const double *l1_reg,
                                     const double *l2_reg, const double *tol, const int32_t *max_iter,
                                     int32_t n_models, int32_t warm_start, int32_t do_screening,
                                     double *W, int64_t ldw, double *info, void *stream) {
    SGLM_CHECK_ARG(C > 0 && n_models >= 0 && ldq >= C && ldw >= C, SGLM_E_SHAPE, "enet_cd: bad shape");
    if (n_models == 0) return SGLM_OK;
    SGLM_CHECK_ARG(prob_Q && prob_q && prob_diag && prob_yy && prob_of_model && l1_reg && l2_reg && tol && max_iter && W && info,
                   SGLM_E_INVALID_ARG, "enet_cd: null pointer");
    const size_t smem = enet_cd_smem_bytes(C);
    SGLM_CHECK_ARG(smem <= 227 * 1024, SGLM_E_UNSUPPORTED,
                   "enet_cd: C=%d needs %zu bytes of shared memory per model (> 227 KB)", C, smem);
    cudaStream_t st = (cudaStream_t)stream;
#define CD_LAUNCH(NBB, CHH, RGG, MB)                                                                       \
    do {                                                                                                   \
        SGLM_CUDA_OK(cudaFuncSetAttribute(enet_cd_gram_kernel<NBB, CHH, RGG, MB>,                          \
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));        \
        enet_cd_gram_kernel<NBB, CHH, RGG, MB><<<n_models, (NBB + 1) * 32, smem, st>>>(                    \
            prob_Q, prob_q, prob_diag, prob_yy, ldq, C, prob_of_model, l1_reg, l2_reg, tol, max_iter,      \
            warm_start, do_screening, W, ldw, info);                                                       \
    } while (0)
    // (panel warps, 16-byte chunks per thread, rows per load group, min CTAs per SM): chosen so that
    // several models are resident per SM (profiles/r1_cd_variants.txt); SGLM_CD_VARIANT is a tuning switch
    const char *var = tuning_env("SGLM_CD_VARIANT");
    const int variant = var ? atoi(var) : 0;
    if (C <= 256) CD_LAUNCH(1, 4, 4, 8);
    else if (C <= 512) CD_LAUNCH(2, 4, 4, 6);
    else if (C <= 1024) CD_LAUNCH(4, 4, 4, 4);
    else {
        switch (variant) {
            case 1: CD_LAUNCH(8, 4, 4, 1); break;
            case 2: CD_LAUNCH(8, 4, 2, 2); break;
            case 3: CD_LAUNCH(4, 8, 2, 2); break;
            case 4: CD_LAUNCH(4, 8, 1, 4); break;
            case 5: CD_LAUNCH(8, 4, 2, 3); break;
            case 6: CD_LAUNCH(16, 2, 4, 1); break;
            case 7: CD_LAUNCH(16, 2, 2, 2); break;
            case 8: CD_LAUNCH(8, 4, 3, 2); break;
            case 9: CD_LAUNCH(4, 8, 2, 3); break;
            default: CD_LAUNCH(8, 4, 2, 2); break;
        }
    }
#undef CD_LAUNCH
    SGLM_LAUNCH_OK("enet_cd_gram_kernel");
    return SGLM_OK;
}

extern "C" size_t sglm_ridge_workspace_bytes(int32_t C, int64_t ldq, int32_t n_alpha) {
    if (C <= 0 || ldq < C || n_alpha <= 0) return 0;
    return (size_t)n_alpha * (size_t)(C + 1) * (size_t)ldq * sizeof(double);
}

extern "C" int sglm_ridge_solve_f64(const double *Qc, int64_t ldq, const double *qc, int32_t C,
                                    const double *alpha, int32_t n_alpha, double *W, int64_t ldw,
                                    int32_t *status, void *work, size_t work_bytes, void *stream) {
    SGLM_CHECK_ARG(C > 0 && n_alpha >= 0 && ldq >= C && ldw >= C, SGLM_E_SHAPE, "ridge_solve: bad shape");
    if (n_alpha == 0) return SGLM_OK;
    SGLM_CHECK_ARG(Qc && qc && alpha && W && status && work, SGLM_E_INVALID_ARG, "ridge_solve: null pointer");
    SGLM_CHECK_ARG(work_bytes >= sglm_ridge_workspace_bytes(C, ldq, n_alpha), SGLM_E_WORKSPACE,
                   "ridge_solve: workspace too small");
    const char *form = tuning_env("SGLM_CHOLESKY");             // "right": the first right-looking kernel (A/B switch)
    if (form && form[0] == 'r') {
        const size_t smem = (size_t)(RC_NB * 33 + 2 * 64 * 33 + C) * sizeof(double);
        SGLM_CHECK_ARG(smem <= 227 * 1024, SGLM_E_UNSUPPORTED, "ridge_solve: C=%d too large for shared memory", C);
        SGLM_CUDA_OK(cudaFuncSetAttribute(ridge_cholesky_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ridge_cholesky_kernel<<<n_alpha, RC_THREADS, smem, (cudaStream_t)stream>>>(Qc, ldq, qc, C, alpha, W, ldw, status,
                                                                                  (double *)work);
        SGLM_LAUNCH_OK("ridge_cholesky_kernel");
        return SGLM_OK;
    }
    const size_t smem = (size_t)(RC_NB * 33 + 2 * RC_NB * LL_LD + 2 * LL_RT * LL_LD + C) * sizeof(double);
    SGLM_CHECK_ARG(smem <= 227 * 1024, SGLM_E_UNSUPPORTED, "ridge_solve: C=%d too large for shared memory", C);
    SGLM_CUDA_OK(cudaFuncSetAttribute(ridge_cholesky_ll_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ridge_cholesky_ll_kernel<<<n_alpha, RC_THREADS, smem, (cudaStream_t)stream>>>(Qc, ldq, qc, C, alpha, W, ldw, status,
                                                                                 (double *)work);
    SGLM_LAUNCH_OK("ridge_cholesky_ll_kernel");
    return SGLM_OK;
}

extern "C" int sglm_chol_solve_batched_f64(const double *const *L_of, int64_t ldq, int32_t C, const double *rhs,
                                           double *out, int64_t ld, const int32_t *flags, int32_t n_systems,
                                           void *stream) {
    SGLM_CHECK_ARG(C > 0 && ldq >= C && ld >= C && n_systems >= 0, SGLM_E_SHAPE, "chol_solve_batched: bad shape");
    if (n_systems == 0) return SGLM_OK;
    SGLM_CHECK_ARG(L_of && rhs && out, SGLM_E_INVALID_ARG, "chol_solve_batched: null pointer");
    const size_t smem = (size_t)(RC_NB * 33 + C) * sizeof(double);
    SGLM_CHECK_ARG(smem <= 227 * 1024, SGLM_E_UNSUPPORTED, "chol_solve_batched: C=%d too large for shared memory", C);
    SGLM_CUDA_OK(cudaFuncSetAttribute(chol_solve_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    chol_solve_batched_kernel<<<n_systems, RC_THREADS, smem, (cudaStream_t)stream>>>(L_of, ldq, C, rhs, out, ld, flags);
    SGLM_LAUNCH_OK("chol_solve_batched_kernel");
    return SGLM_OK;
}

extern "C" int sglm_finalize_models_f64(const double *W, int64_t ldw, int32_t C, int32_t n_y,
                                        const int32_t *y_col_of_model, const double *const *xbar_of_model,
                                        const double *ybar_of_model, int32_t n_models, double *intercept,
                                        double *V, int64_t ldv, void *stream) {
    SGLM_CHECK_ARG(C > 0 && n_models >= 0 && ldw >= C, SGLM_E_SHAPE, "finalize_models: bad shape");
    if (n_models == 0) return SGLM_OK;
    SGLM_CHECK_ARG(W && intercept, SGLM_E_INVALID_ARG, "finalize_models: null pointer");
    SGLM_CHECK_ARG(!V || ldv >= C + n_y + 1, SGLM_E_SHAPE, "finalize_models: ldv too small");
    SGLM_CHECK_ARG(!xbar_of_model || ybar_of_model, SGLM_E_INVALID_ARG, "finalize_models: xbar without ybar");
    finalize_models_kernel<<<n_models, 128, 0, (cudaStream_t)stream>>>(W, ldw, C, n_y, y_col_of_model, xbar_of_model,
                                                                       ybar_of_model, intercept, V, ldv);
    SGLM_LAUNCH_OK("finalize_models_kernel");
    return SGLM_OK;
}

static int quadform_launch(const double *A, int64_t lda, int32_t n, const double *V, int64_t ldv, int32_t n_models,
                           int32_t n_splits, double *out, void *stream);

extern "C" int sglm_quadform_f64(const double *A, int64_t lda, int32_t n, const double *V, int64_t ldv,
                                 int32_t n_models, double *out, void *stream) {
    return quadform_launch(A, lda, n, V, ldv, n_models, 1, out, stream);
}

// Row-split form: partial[s * n_models + m] = sum over the rows of split s of v_m[i] (A v_m)[i]; the caller adds
// the n_splits partial sums (fixed order: deterministic).  Few models (a fold's 250) otherwise leave most SMs idle.
extern "C" int sglm_quadform_split_f64(const double *A, int64_t lda, int32_t n, const double *V, int64_t ldv,
                                       int32_t n_models, int32_t n_splits, double *partial, void *stream) {
    SGLM_CHECK_ARG(n_splits >= 1 && n_splits <= 65535, SGLM_E_INVALID_ARG, "quadform_split: bad n_splits");
    return quadform_launch(A, lda, n, V, ldv, n_models, n_splits, partial, stream);
}

static int quadform_launch(const double *A, int64_t lda, int32_t n, const double *V, int64_t ldv, int32_t n_models,
                           int32_t n_splits, double *out, void *stream) {
    SGLM_CHECK_ARG(n > 0 && n_models >= 0 && lda >= n && ldv >= n, SGLM_E_SHAPE, "quadform: bad shape");
    if (n_models == 0) return SGLM_OK;
    SGLM_CHECK_ARG(A && V && out, SGLM_E_INVALID_ARG, "quadform: null pointer");
    const int mb = ((size_t)8 * n * sizeof(double) <= 200 * 1024 && n_models >= 8) ? 8 : 4;
    const size_t smem = (size_t)mb * n * sizeof(double);
    SGLM_CHECK_ARG(smem <= 227 * 1024, SGLM_E_UNSUPPORTED, "quadform: n=%d too large for shared memory", n);
    if (mb == 8) {
        SGLM_CUDA_OK(cudaFuncSetAttribute(quadform_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        quadform_kernel<8><<<dim3(ceil_div(n_models, 8), n_splits), QF_THREADS, smem, (cudaStream_t)stream>>>(A, lda, n, V, ldv, n_models, out);
    } else {
        SGLM_CUDA_OK(cudaFuncSetAttribute(quadform_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        quadform_kernel<4><<<dim3(ceil_div(n_models, 4), n_splits), QF_THREADS, smem, (cudaStream_t)stream>>>(A, lda, n, V, ldv, n_models, out);
    }
    SGLM_LAUNCH_OK("quadform_kernel");
    return SGLM_OK;
}

// x = (L L')^-1 rhs with the factor of system `k` that sglm_ridge_solve_f64 left in its work buffer
// (work + k * (C + 1) * ldq doubles).  Replaces a second factorisation when the matrix has not changed.
extern "C" int sglm_chol_solve_f64(const void *work, int64_t ldq, int32_t C, int32_t k, const double *rhs, double *out,
                                   void *stream) {
    SGLM_CHECK_ARG(C > 0 && ldq >= C && k >= 0, SGLM_E_SHAPE, "chol_solve: bad shape");
    SGLM_CHECK_ARG(work && rhs && out, SGLM_E_INVALID_ARG, "chol_solve: null pointer");
    const size_t smem = (size_t)(RC_NB * 33 + C) * sizeof(double);
    SGLM_CHECK_ARG(smem <= 227 * 1024, SGLM_E_UNSUPPORTED, "chol_solve: C=%d too large for shared memory", C);
    SGLM_CUDA_OK(cudaFuncSetAttribute(chol_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const double *L = (const double *)work + (size_t)k * (size_t)(C + 1) * (size_t)ldq;
    chol_solve_kernel<<<1, RC_THREADS, smem, (cudaStream_t)stream>>>(L, ldq, C, rhs, out);
    SGLM_LAUNCH_OK("chol_solve_kernel");
    return SGLM_OK;
}
