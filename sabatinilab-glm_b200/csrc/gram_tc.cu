// Tensor-core Gram builder: fp64-grade  G = Z' Z  (Z = [X | Y | 1], several row sets) on the
// 5th-generation tensor cores — tcgen05.mma kind::i8 with int32 accumulators in TMEM, operands
// staged by TMA into 128B-swizzled shared memory, mbarrier producer/consumer pipeline.
//
// tcgen05 has no f64 kind, so the fp64 Gram is computed EXACTLY in integers (split / Ozaki
// scheme): every column c of Z is scaled by 2^-E_c (E_c from the column's max |z|) and cut into
// signed radix-128 digits  z = 2^E_c (d_1 2^-6 + d_2 2^-13 + ... + d_s 2^-(6+7(s-1))),
// |d_k| <= 64, which int8 holds exactly.  The Gram of two digit planes is an int8 x int8 -> int32
// GEMM whose result is exact (|d d'| <= 2^12, drained from TMEM before 2^31 can be reached) and
// is accumulated in int64; the fp64 Gram is the power-of-two weighted sum of the digit-plane
// Grams.  With s = 8 planes the representation error is 2^-56 of the column scale — fp64 grade —
// and a column whose values are exactly representable in fewer digits (the 0/1 event indicators
// that make up most of a photometry design need ONE plane) is detected and only gets the planes
// it needs, so the integer work adapts to the data: ~4 dense int8 GEMM equivalents for the c3
// workload instead of 36.
//
// Replaces the same reference arithmetic as suffstats.cu (the X'X / X'y of every sklearn fit,
// backend/sglm.py:241) and produces the same output contract as sglm_suffstats_f64 for 0/1 row
// sets; the DMMA kernel remains the path for general row weights (Poisson IRLS) and the on-GPU
// cross-check of this one.
//
// Pipeline:  colscale -> digit count -> slice (digits, transposed to K-major, rows gathered per
// set) -> int8 tcgen05 GEMM over digit-plane tile pairs -> combine (fp64).
#include <cuda.h>

#include <algorithm>
#include <vector>

#include <stdlib.h>

#include "common.cuh"

namespace sglm {

constexpr int TC_SMAX = 8;       // digit planes for a general fp64 column
constexpr int TC_BK = 128;       // K bytes (= int8 elements = design rows) per pipeline stage
constexpr int TC_BM = 256;       // output tile rows: two UMMA M=128 accumulators
constexpr int TC_BN = 256;       // UMMA N
constexpr int TC_STAGES = 3;
constexpr int TC_THREADS = 192;  // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2-5: epilogue
constexpr int TC_MAX_KB_PER_SEG = 2048;   // 2048 * 128 rows * 2^12 < 2^31
constexpr uint32_t TC_STAGE_BYTES = (TC_BM + TC_BN) * TC_BK;
constexpr int TC_LEAD = 64;      // K blocks an item may run ahead of the slowest neighbouring item of its K part
constexpr int TC_FAR = 1024;     // items further behind than this belong to another wave

// ------------------------------------------------------------------ column scale and digit count
__device__ __forceinline__ double z_value(const double *X, long long ldx, const double *Y, long long ldy,
                                          int C, int n_y, long long t, int c) {
    if (c < C) return X[t * ldx + c];
    if (c < C + n_y) return Y[t * ldy + (c - C)];
    return 1.0;
}

// One pass over Z = [X | Y | 1]: per column the largest magnitude (-> scale exponent E) and the lowest set
// bit of any element (-> how many radix-128 digits represent the whole column exactly at that scale).
__global__ void __launch_bounds__(256)
tc_colmax_kernel(const double *__restrict__ X, long long ldx, const double *__restrict__ Y, long long ldy,
                 int C, int n_y, long long T, const double *__restrict__ rs,
                 unsigned long long *__restrict__ colmax_bits, int *__restrict__ col_lsb) {
    const int n_aug = C + n_y + 1;
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= n_aug) return;
    const long long rows_per = (T + gridDim.y - 1) / gridDim.y;
    const long long t0 = (long long)blockIdx.y * rows_per, t1 = min(T, t0 + rows_per);
    double m = 0.0;
    bool bad = false;
    int lsb = 0x7fffffff;
    for (long long t = t0; t < t1; ++t) {
        const double v = fabs(z_value(X, ldx, Y, ldy, C, n_y, t, c) * (rs ? rs[t] : 1.0));      // rs: optional row scale (sqrt of a row weight)
        bad |= !(v <= 1.7976931348623157e308);          // NaN or inf
        m = fmax(m, v);
        const long long bits = __double_as_longlong(v);
        const int e = (int)(bits >> 52);
        const long long frac = bits & 0xfffffffffffffLL;
        if (e > 0) lsb = min(lsb, e - 1075 + __ffsll(frac | (1LL << 52)) - 1);       // v = (2^52 + frac) * 2^(e-1075)
        else if (frac) lsb = min(lsb, -1074 + __ffsll(frac) - 1);                    // subnormal
    }
    if (bad) m = __longlong_as_double(0x7ff8000000000000LL);
    atomicMax(colmax_bits + c, (unsigned long long)__double_as_longlong(m));   // monotone for non-negative doubles; NaN pattern wins
    atomicMin(col_lsb + c, lsb);
}

// number of radix digits (1..TC_SMAX) a value needs to be represented exactly at scale 2^E
__device__ __forceinline__ int digits_needed(double z, int E) {
    double r = scalbn(z, -E);            // |r| < 1
    int need = 0;
    r *= 64.0;
#pragma unroll
    for (int k = 1; k <= TC_SMAX; ++k) {
        if (r == 0.0) break;
        const double d = rint(r);
        if (d != 0.0) need = k;
        r = (r - d) * 128.0;
    }
    if (r != 0.0) need = TC_SMAX;
    return need;
}

__global__ void __launch_bounds__(256)
tc_digits_kernel(const double *__restrict__ X, long long ldx, const double *__restrict__ Y, long long ldy,
                 int C, int n_y, long long T, const double *__restrict__ rs, const int *__restrict__ colE,
                 int *__restrict__ colS) {
    const int n_aug = C + n_y + 1;
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= n_aug) return;
    const long long rows_per = (T + gridDim.y - 1) / gridDim.y;
    const long long t0 = (long long)blockIdx.y * rows_per, t1 = min(T, t0 + rows_per);
    const int E = colE[c];
    int need = 1;
    for (long long t = t0; t < t1 && need < TC_SMAX; ++t)
        need = max(need, digits_needed(z_value(X, ldx, Y, ldy, C, n_y, t, c) * (rs ? rs[t] : 1.0), E));
    atomicMax(colS + c, need);
}

// colS holds the column's lowest set bit on entry (0x7f7f7f7f.. when the column is all zero) and the number
// of digit planes on exit: digit k carries the bits down to 2^(E - 6 - 7(k-1)), so the column is exact with
// k >= (E - 6 - lsb) / 7 + 1 planes (the same count the digit-by-digit expansion of every element gives).
__global__ void tc_exponent_kernel(const unsigned long long *__restrict__ colmax_bits, int n_aug, int max_planes,
                                   int *__restrict__ colE, int *__restrict__ colS, int *__restrict__ flag) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_aug) return;
    const double m = __longlong_as_double((long long)colmax_bits[c]);
    if (!(m <= 1.7976931348623157e308)) { atomicOr(flag, 1); colE[c] = 0; colS[c] = 1; return; }
    const int E = (m == 0.0) ? 0 : ilogb(m) + 1;      // |z| < 2^E
    colE[c] = E;
    const int lsb = colS[c];
    int need = 1;
    if (m != 0.0) {
        const int span = E - 6 - lsb;                 // bits below the first digit
        if (span > 0) need = 1 + (span + 6) / 7;
    }
    colS[c] = min(need, max_planes);      // fewer planes than needed = digits rounded at that plane (approximate Gram)
}

// ------------------------------------------------------------------ slicing (digits, transposed, gathered rows)
// At[(plane k of column c)][p] = digit k of Z[rows[p], c];  p runs over the concatenated, 128-padded
// row lists of all sets (rows[p] < 0 marks padding -> zeros, which the buffer already holds).
__global__ void __launch_bounds__(256)
tc_slice_kernel(const double *__restrict__ X, long long ldx, const double *__restrict__ Y, long long ldy,
                int C, int n_y, const double *__restrict__ rs, const long long *__restrict__ rows, long long n_pos,
                const int *__restrict__ colE, const int *__restrict__ colS, const int *__restrict__ plane_row,
                int8_t *__restrict__ At, long long ld_at, long long n_ident) {
    // plane_row[c * TC_SMAX + (k-1)] = row of At holding digit plane k of column c (or -1)
    // rows == nullptr: position p is row p for p < n_ident (the base signals of a lag design, sliced once)
    __shared__ __align__(16) double tile[32][130];        // [column][position], transposed on the way in
    const int n_aug = C + n_y + 1;
    const long long p0 = (long long)blockIdx.x * 128;
    const int c0 = blockIdx.y * 32;
    const int tid = threadIdx.x;
    // the 128 row indices first (one coalesced load), so that the 16 element loads of a thread below do not
    // each wait for their own index: 16 independent loads in flight per thread
    __shared__ long long srow[128];
    if (tid < 128) srow[tid] = (p0 + tid < n_pos) ? (rows ? rows[p0 + tid] : (p0 + tid < n_ident ? p0 + tid : -1)) : -1;
    __syncthreads();
    // load 128 positions x 32 columns, coalesced along the columns of the row-major source
    {
        const int cc = tid & 31, c = c0 + cc;
        double v[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const long long t = srow[(tid >> 5) + 8 * k];
            v[k] = (t >= 0 && c < n_aug) ? z_value(X, ldx, Y, ldy, C, n_y, t, c) * (rs ? rs[t] : 1.0) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) tile[cc][(tid >> 5) + 8 * k] = v[k];
    }
    __syncthreads();
    // thread <-> (4 consecutive positions, 4 columns): one packed 32-bit store per digit plane,
    // a warp writes 128 contiguous bytes of a plane row
    const int pq = tid & 31, cg = tid >> 5;
    const long long p = p0 + 4 * pq;
    if (p >= n_pos) return;
#pragma unroll 1
    for (int cc = cg * 4; cc < cg * 4 + 4; ++cc) {
        const int c = c0 + cc;
        if (c >= n_aug) break;
        const int S = colS[c], E = colE[c];
        const double2 v01 = *reinterpret_cast<const double2 *>(&tile[cc][4 * pq]);
        const double2 v23 = *reinterpret_cast<const double2 *>(&tile[cc][4 * pq + 2]);
        double r0, r1, r2, r3;
        if (E > -900 && E < 900) {
            // scaling by 2^(6-E) as ONE exact multiplication by a power of two built from its exponent bits
            // (scalbn is a multi-instruction routine and this pass is issue-bound: 44 % issue slots active, 2.2 TB/s, in its ncu capture)
            const double sc = __longlong_as_double((long long)(1023 + 6 - E) << 52);
            r0 = v01.x * sc; r1 = v01.y * sc; r2 = v23.x * sc; r3 = v23.y * sc;
        } else {
            r0 = scalbn(v01.x, -E) * 64.0; r1 = scalbn(v01.y, -E) * 64.0;
            r2 = scalbn(v23.x, -E) * 64.0; r3 = scalbn(v23.y, -E) * 64.0;
        }
        for (int k = 1; k <= S; ++k) {
            const double d0 = rint(r0), d1 = rint(r1), d2 = rint(r2), d3 = rint(r3);
            r0 = (r0 - d0) * 128.0; r1 = (r1 - d1) * 128.0; r2 = (r2 - d2) * 128.0; r3 = (r3 - d3) * 128.0;
            const unsigned pack = ((unsigned)(int)d0 & 0xffu) | (((unsigned)(int)d1 & 0xffu) << 8) |
                                  (((unsigned)(int)d2 & 0xffu) << 16) | (((unsigned)(int)d3 & 0xffu) << 24);
            *reinterpret_cast<unsigned *>(At + (long long)plane_row[c * TC_SMAX + (k - 1)] * ld_at + p) = pack;
        }
    }
}

// ------------------------------------------------------------------ lag designs: planes of the design from planes of the base
// A lag design column (base signal p, shift s) is the base signal read at another row:  Z[t, c] = base[t + off_c, p].
// Its digit planes are therefore the base signal's planes read at another position — the fp64 design is never
// built or read: the base signals (P columns instead of P*L) are sliced once into Bt, and the K-major operand
// At[(plane k of column c)][pos] = Bt[(plane k of p_c)][rows[pos] + off_c] is a byte gather (reads hit L1 / L2: the L
// shifts of a signal read the same bytes; HBM traffic = the write of At).  map[r] = (row of Bt, off) of At row r,
// (-1, .) for rows that are not lag columns (response / ones planes, padding between levels).
constexpr int TC_EXP_ROWS = 256;     // At rows per CTA (blockIdx.y)
constexpr int TC_EXP_POS = 512;      // positions per CTA: 32 chunks of 16 positions (one 16-byte store each)
__global__ void __launch_bounds__(256)
tc_expand_kernel(const int8_t *__restrict__ Bt, long long ld_bt, const long long *__restrict__ rows, long long n_pos,
                 const int2 *__restrict__ map, int n_at_rows, int8_t *__restrict__ At, long long ld_at) {
    __shared__ long long srow[TC_EXP_POS];
    const int tid = threadIdx.x;
    const long long p0 = (long long)blockIdx.x * TC_EXP_POS;
    for (int i = tid; i < TC_EXP_POS; i += 256) srow[i] = (p0 + i < n_pos) ? rows[p0 + i] : -1;
    __syncthreads();
    const int pq = tid & 31, rl = tid >> 5;
    const long long p = p0 + 16 * pq;
    if (p >= n_pos) return;                         // n_pos is a multiple of 128: whole chunks only
    const long long r0 = srow[16 * pq], r15 = srow[16 * pq + 15];
    // sorted, duplicate-free row lists: 16 positions are 16 consecutive rows iff last - first == 15 (padding is -1)
    const bool contig = r0 >= 0 && r15 == r0 + 15;
    const int r_end = min(n_at_rows, (int)(blockIdx.y + 1) * TC_EXP_ROWS);
    for (int r = blockIdx.y * TC_EXP_ROWS + rl; r < r_end; r += 8) {
        const int2 m = map[r];
        if (m.x < 0) continue;
        const int8_t *src = Bt + (long long)m.x * ld_bt + m.y;
        uint4 out;
        if (contig) {
            // 16 consecutive bytes at an arbitrary byte offset: five aligned words and four funnel shifts
            const unsigned long long a = (unsigned long long)(src + r0);
            const unsigned *w = reinterpret_cast<const unsigned *>(a & ~3ull);
            const unsigned sh = (unsigned)(a & 3ull) * 8u;
            const unsigned w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2), w3 = __ldg(w + 3);
            const unsigned w4 = sh ? __ldg(w + 4) : 0u;
            out = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                             __funnelshift_r(w3, w4, sh));
        } else {
            unsigned q[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                unsigned v = 0u;
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const long long rr = srow[16 * pq + 4 * j + b];
                    if (rr >= 0) v |= (unsigned)(unsigned char)__ldg(src + rr) << (8 * b);
                }
                q[j] = v;
            }
            out = make_uint4(q[0], q[1], q[2], q[3]);
        }
        *reinterpret_cast<uint4 *>(At + (long long)r * ld_at + p) = out;
    }
}

// ------------------------------------------------------------------ PTX helpers (mbarrier / TMA / tcgen05)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug must surface as a trapped kernel, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    const long long t_start = clock64();
    while (true) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.b32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) return;
        if (clock64() - t_start > 4000000000LL) { asm volatile("trap;"); }
    }
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *tmap, uint64_t *bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"((uint64_t)tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// multicast forms: the box lands at the same shared-memory offset of every CTA in `mask` and completes bytes on the mbarrier
// at the same offset there; the commit arrives on the mbarrier at the same offset of every CTA in `mask`
__device__ __forceinline__ void tma_load_2d_mc(void *dst, const CUtensorMap *tmap, uint64_t *bar, int c0, int c1, uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(dst)), "l"((uint64_t)tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
        : "memory");
}
__device__ __forceinline__ void tc_commit_mc(uint64_t *bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void tc_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// K-major, 128B-swizzled operand tile (rows of 128 bytes, 8-row groups 1024 bytes apart): the
// layout TMA writes for CU_TENSOR_MAP_SWIZZLE_128B with a 128-byte inner box.
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);          // start address
    d |= (uint64_t)1 << 16;                               // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                     // stride byte offset: next 8-row group
    d |= (uint64_t)1 << 46;                               // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                               // SWIZZLE_128B
    return d;
}
// instruction descriptor: dense, S32 accumulate, A/B signed int8, both K-major, M=128, N=256
__host__ __device__ constexpr uint32_t tc_idesc_i8() {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

struct TcSeg { int kb0, n_kb, set, first; };

// ------------------------------------------------------------------ the int8 tcgen05 GEMM
// One CTA per work item = (256 x 256 output tile of the digit-plane Gram, K part).  K runs over
// this part of the row segments of all sets; each segment's int32 accumulators (two UMMA M=128
// tiles, 512 TMEM columns) are drained into the int64 tile of its set with integer atomics —
// exact, hence independent of the order in which the K parts arrive (deterministic result).
// The kernel is bound by the L2 -> SM feed (~6 TB/s aggregate measured), so the tile is made as
// square as TMEM allows: 512 operand rows per 65536 outputs.
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_gram_i8_kernel(const __grid_constant__ CUtensorMap tmap, const int2 *__restrict__ tiles, int n_tiles,
                  int n_parts, const TcSeg *__restrict__ segs, int n_segs, long long *__restrict__ SG, long long S,
                  int *__restrict__ prog, const int2 *__restrict__ pairs, int n_pairs) {
    extern __shared__ __align__(1024) uint8_t tc_smem[];
    uint8_t *base = (uint8_t *)(((uintptr_t)tc_smem + 1023) & ~(uintptr_t)1023);
    uint8_t *sA = base;                                           // [STAGES][256][128]
    uint8_t *sB = base + TC_STAGES * TC_BM * TC_BK;               // [STAGES][256][128]
    uint64_t *bars = (uint64_t *)(base + TC_STAGES * TC_STAGE_BYTES);
    uint64_t *full = bars, *empty = bars + TC_STAGES, *tmem_full = bars + 2 * TC_STAGES, *tmem_empty = tmem_full + 1;
    uint32_t *tmem_slot = (uint32_t *)(tmem_empty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // a 2-CTA cluster per (pair of neighbouring tiles of one tile row, K part): CTA `rank` computes tile pr.x / pr.y; both
    // need the same A strip, each loads half of it and multicasts it to the other (half the A bytes through each SM's L2
    // port: the kernel is bound by the L2 -> SM ingest per SM, ~55 GB/s, not by DRAM or the tensor pipe)
    const int item = blockIdx.x;
    const int rank = item & 1;
    const int2 pr = pairs[(item >> 1) % n_pairs];
    const int part = (item >> 1) / n_pairs;
    const bool paired = pr.y >= 0;
    const int my_tile = rank == 0 ? pr.x : pr.y;
    const int2 tile = tiles[my_tile >= 0 ? my_tile : pr.x];
    const int m0 = tile.x * TC_BM, n0 = tile.y * TC_BN;
    (void)n_tiles;
    // This item's share of the K space: part p owns a CONTIGUOUS range of the concatenated K blocks of all
    // segments (so a tile is drained once per row set plus once per part boundary, however many row sets
    // there are).  seg_range gives its K blocks [lo, hi) inside segment sgi; `before` = K blocks of the
    // segments ahead of it.
    long long total_kb = 0;
    for (int sgi = 0; sgi < n_segs; ++sgi) total_kb += segs[sgi].n_kb;
    const long long part_lo = total_kb * part / n_parts, part_hi = total_kb * (part + 1) / n_parts;
    auto seg_range = [&](const TcSeg &sg, long long before, int &lo, int &hi) {
        const long long a = max(part_lo, before), b = min(part_hi, before + sg.n_kb);
        lo = sg.kb0 + (int)(a - before);
        hi = (b > a) ? sg.kb0 + (int)(b - before) : lo;
    };

    if (threadIdx.x == 0) {
        // a stage is free when the MMAs of BOTH CTAs have read it (the peer multicasts into it)
        for (int s = 0; s < TC_STAGES; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, paired ? 2 : 1); }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_cluster_sync();               // the peer's barriers exist before anything is multicast to them
    tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot;
    const uint16_t mc_mask = paired ? (uint16_t)3 : (uint16_t)(1u << rank);

    if (my_tile < 0) {
        // the idle half of a cluster whose tile has no neighbour
        if (prog != nullptr && threadIdx.x == 0)
            asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(prog + item), "r"(0x7fffffff) : "memory");
    } else if (warp == 0) {
        // ===== TMA producer (one elected lane issues the loads; the whole warp keeps the K schedule in step)
        // Optional K lock-step (prog != nullptr; measurement switch SGLM_TC_LOCKSTEP): the work items of one K part read the
        // same operand strips; while they walk K together every strip byte is fetched from DRAM once and served from L2 to
        // the ~13 CTAs that need it, left alone they drift apart by more than the ~175 K blocks L2 can hold and the strips
        // are re-fetched ~10x (ncu: 97 GB of DRAM reads for 9.6 GB of digit planes, L2 hit 51 %).  Every 32 K blocks an item
        // publishes its position and does not run more than TC_LEAD K blocks ahead of the slowest item of its part in its
        // neighbourhood (items further than TC_FAR behind belong to a later wave; finished / not yet started items are
        // ignored) — the slowest item never waits, so the scheme cannot deadlock.  It cuts the DRAM reads 4x and does NOT
        // make the kernel faster (it is bound by the L2 -> SM ingest per SM), so it is off by default.
        int it = 0;
        long long before = 0;
        for (int sgi = 0; sgi < n_segs; ++sgi) {
            int lo, hi;
            seg_range(segs[sgi], before, lo, hi);
            before += segs[sgi].n_kb;
            for (int kb = lo; kb < hi; ++kb, ++it) {
                if (prog != nullptr && (it & 31) == 0) {
                    __syncwarp();
                    if (lane == 0) asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(prog + item), "r"(it) : "memory");
                    const int *grp = prog + (long long)part * 2 * n_pairs;
                    const long long t_start = clock64();
                    while (true) {
                        int behind = 0;
                        for (int j = lane; j < 2 * n_pairs; j += 32) {
                            int v;
                            asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(grp + j) : "memory");
                            const int d = it - v;
                            if (v >= 0 && d > TC_LEAD && d <= TC_FAR) behind = 1;
                        }
                        if (!__any_sync(0xffffffffu, behind)) break;
                        __nanosleep(500);
                        if (clock64() - t_start > 4000000000LL) { asm volatile("trap;"); }
                    }
                }
                if (lane == 0) {
                    const int st = it % TC_STAGES;
                    const uint32_t ph = (it / TC_STAGES) & 1;
                    mbar_wait(empty + st, ph ^ 1);
                    mbar_expect_tx(full + st, TC_STAGE_BYTES);
                    const int kc = kb * TC_BK;
                    uint8_t *a = sA + st * TC_BM * TC_BK, *bq = sB + st * TC_BN * TC_BK;
                    if (paired) {
                        // my half of the shared A strip, to both CTAs; the other half arrives from the peer
                        tma_load_2d_mc(a + rank * 128 * TC_BK, &tmap, full + st, kc, m0 + 128 * rank, mc_mask);
                    } else {
                        tma_load_2d(a, &tmap, full + st, kc, m0);
                        tma_load_2d(a + 128 * TC_BK, &tmap, full + st, kc, m0 + 128);
                    }
                    tma_load_2d(bq, &tmap, full + st, kc, n0);
                    tma_load_2d(bq + 128 * TC_BK, &tmap, full + st, kc, n0 + 128);
                }
            }
        }
        __syncwarp();
        if (prog != nullptr && lane == 0)
            asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(prog + item), "r"(0x7fffffff) : "memory");
    } else if (warp == 1) {
        // ===== MMA issuer (one elected lane)
        if (lane == 0) {
            constexpr uint32_t idesc = tc_idesc_i8();
            int it = 0, drained = 0;
            long long before = 0;
            for (int sgi = 0; sgi < n_segs; ++sgi) {
                int lo, hi;
                seg_range(segs[sgi], before, lo, hi);
                before += segs[sgi].n_kb;
                if (hi <= lo) continue;
                if (drained > 0) { mbar_wait(tmem_empty, (drained - 1) & 1); tc_fence_after(); }
                for (int kb = lo; kb < hi; ++kb, ++it) {
                    const int st = it % TC_STAGES;
                    const uint32_t ph = (it / TC_STAGES) & 1;
                    mbar_wait(full + st, ph);
                    tc_fence_after();
                    const uint64_t da0 = umma_desc_k_sw128(smem_u32(sA + st * TC_BM * TC_BK));
                    const uint64_t da1 = umma_desc_k_sw128(smem_u32(sA + st * TC_BM * TC_BK + 128 * TC_BK));
                    const uint64_t db = umma_desc_k_sw128(smem_u32(sB + st * TC_BN * TC_BK));
#pragma unroll
                    for (int k = 0; k < TC_BK / 32; ++k) {        // UMMA K = 32 int8: +32 bytes inside the swizzle atom
                        const uint32_t accflag = ((kb - lo) | k) ? 1u : 0u;
                        tc_mma_i8(tmem_acc, da0 + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, accflag);
                        tc_mma_i8(tmem_acc + 256u, da1 + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, accflag);
                    }
                    if (paired) tc_commit_mc(empty + st, mc_mask);  // frees the stage in BOTH CTAs when these MMAs retire
                    else tc_commit(empty + st);
                }
                tc_commit(tmem_full);                              // accumulators of this segment complete
                ++drained;
            }
        }
    } else {
        // ===== epilogue: TMEM -> registers -> int64 atomics on the tile of the segment's set
        const int q = warp & 3;                                    // TMEM lane quarter this warp may access
        const int row = q * 32 + lane;
        int drained = 0;
        long long before = 0;
        for (int sgi = 0; sgi < n_segs; ++sgi) {
            const TcSeg sg = segs[sgi];
            int lo, hi;
            seg_range(sg, before, lo, hi);
            before += sg.n_kb;
            if (hi <= lo) continue;
            mbar_wait(tmem_full, drained & 1);
            tc_fence_after();
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                unsigned long long *out = reinterpret_cast<unsigned long long *>(
                    SG + ((long long)sg.set * S + (m0 + half * 128 + row)) * S + n0);
#pragma unroll 1
                for (int ch = 0; ch < TC_BN / 32; ++ch) {
                    uint32_t v[32];
                    const uint32_t taddr = tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * 256 + ch * 32);
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                        : "r"(taddr));
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const long long x = (long long)(int)v[j];
                        if (x != 0) atomicAdd(out + ch * 32 + j, (unsigned long long)x);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tmem_empty);
            ++drained;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_cluster_sync();               // no CTA leaves while its peer may still multicast into it or arrive on its barriers
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(512));
    }
}

// Measurement probe: the issue rate of tcgen05.mma kind::i8 with both operands resident in shared memory (no
// loads in the loop) — the denominator the Gram GEMM's tensor-pipe fraction is quoted against.  One CTA per SM,
// `iters` x (4 K-steps x 2 accumulators) UMMAs of M=128, N=256, K=32 on one stage of (arbitrary) operand bytes.
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_mma_probe_kernel(int iters) {
    extern __shared__ __align__(1024) uint8_t tc_smem[];
    uint8_t *base = (uint8_t *)(((uintptr_t)tc_smem + 1023) & ~(uintptr_t)1023);
    uint64_t *bars = (uint64_t *)(base + TC_STAGE_BYTES);
    uint32_t *tmem_slot = (uint32_t *)(bars + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < (int)(TC_STAGE_BYTES / 4); i += TC_THREADS) ((uint32_t *)base)[i] = 0x01010101u * (i & 3);
    if (threadIdx.x == 0) { mbar_init(bars, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot;
    if (warp == 1 && lane == 0) {
        constexpr uint32_t idesc = tc_idesc_i8();
        const uint64_t da0 = umma_desc_k_sw128(smem_u32(base));
        const uint64_t da1 = umma_desc_k_sw128(smem_u32(base + 128 * TC_BK));
        const uint64_t db = umma_desc_k_sw128(smem_u32(base + TC_BM * TC_BK));
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int k = 0; k < TC_BK / 32; ++k) {
                tc_mma_i8(tmem_acc, da0 + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (it | k) ? 1u : 0u);
                tc_mma_i8(tmem_acc + 256u, da1 + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (it | k) ? 1u : 0u);
            }
        }
        tc_commit(bars);
        mbar_wait(bars, 0);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(512));
    }
}

// Plain-CUDA-core version of the same tile computation (validation of the tcgen05 path on the
// GPU itself: the integer results must be identical).  One thread per output element.
__global__ void __launch_bounds__(256)
tc_gram_i8_check_kernel(const int8_t *__restrict__ At, long long ld_at, const int2 *__restrict__ tiles,
                        const TcSeg *__restrict__ segs, int n_segs, long long *__restrict__ SG, long long S) {
    const int2 tile = tiles[blockIdx.x];
    const int m0 = tile.x * TC_BM, n0 = tile.y * TC_BN;
    for (int e = threadIdx.x; e < TC_BM * TC_BN; e += 256) {
        const int m = m0 + e / TC_BN, n = n0 + e % TC_BN;
        const int *a = reinterpret_cast<const int *>(At + (long long)m * ld_at);
        const int *b = reinterpret_cast<const int *>(At + (long long)n * ld_at);
        for (int sgi = 0; sgi < n_segs; ++sgi) {
            const TcSeg sg = segs[sgi];
            long long acc = 0;
            const long long i0 = (long long)sg.kb0 * (TC_BK / 4), i1 = i0 + (long long)sg.n_kb * (TC_BK / 4);
            int part = 0;
            for (long long i = i0; i < i1; ++i) {
                part = __dp4a(a[i], b[i], part);
                if ((i & 1023) == 1023) { acc += part; part = 0; }
            }
            acc += part;
            SG[((long long)sg.set * S + m) * S + n] += acc;       // SG zeroed by the host; one thread per element
        }
    }
}

// ------------------------------------------------------------------ cells -> row sets (exact integer sums)
// SGout[o][e] = sum over the cells c with member[o * n_cells + c] != 0 of SG[c][e]: the row sets of a CV grid
// overlap (the full data contain every test fold, random folds intersect), so the GEMM runs once over the
// disjoint CELLS of the partition they induce and the Gram of each set is the sum of its cells' Grams.
constexpr int TC_SUM_OUT = 8;      // output sets accumulated per pass over the cells
constexpr int TC_SUM_CELLS = 256;  // cells whose membership masks are staged in shared memory
// Only the output tiles the GEMM computes (level pairs k <= l, upper triangle inside a level: 193 of 484 tiles at c3) are
// zeroed, summed and later read by the recombination; the rest of the S x S planes is never touched.
__global__ void __launch_bounds__(256)
tc_zero_tiles_kernel(long long *__restrict__ SG, long long S, const int2 *__restrict__ tiles) {
    const int2 tile = tiles[blockIdx.x];
    long long *base = SG + (long long)blockIdx.y * S * S + (long long)tile.x * TC_BM * S + (long long)tile.y * TC_BN;
    for (int e = threadIdx.x; e < TC_BM * TC_BN / 2; e += 256) {
        const int r = e / (TC_BN / 2), c2 = e % (TC_BN / 2);
        reinterpret_cast<longlong2 *>(base + (long long)r * S)[c2] = make_longlong2(0, 0);
    }
}

__global__ void __launch_bounds__(256)
tc_cell_sum_kernel(const long long *__restrict__ SG, long long S, const int2 *__restrict__ tiles, int n_tiles, int n_cells,
                   const int *__restrict__ member, int n_out, long long *__restrict__ SGout) {
    // every element of a computed tile is read once per group of TC_SUM_OUT output sets and added to the sets it belongs
    // to; membership of a cell = one bit mask per group (shared memory), two elements per thread, cells unrolled by 4
    __shared__ unsigned smask[TC_SUM_CELLS];
    const long long n_elem = S * S;
    const long long n_pairs = (long long)n_tiles * (TC_BM * TC_BN / 2);
    for (int o0 = 0; o0 < n_out; o0 += TC_SUM_OUT) {
        __syncthreads();
        for (int c = threadIdx.x; c < n_cells && c < TC_SUM_CELLS; c += 256) {
            unsigned m = 0;
            for (int k = 0; k < TC_SUM_OUT && o0 + k < n_out; ++k)
                if (member[(o0 + k) * n_cells + c]) m |= 1u << k;
            smask[c] = m;
        }
        __syncthreads();
        for (long long t = (long long)blockIdx.x * 256 + threadIdx.x; t < n_pairs; t += (long long)gridDim.x * 256) {
            const int2 tile = tiles[t / (TC_BM * TC_BN / 2)];
            const int w = (int)(t % (TC_BM * TC_BN / 2));
            const long long e = ((long long)tile.x * TC_BM + w / (TC_BN / 2)) * S + (long long)tile.y * TC_BN + 2 * (w % (TC_BN / 2));
            const bool two = true;
            long long a0[TC_SUM_OUT], a1[TC_SUM_OUT];
#pragma unroll
            for (int k = 0; k < TC_SUM_OUT; ++k) { a0[k] = 0; a1[k] = 0; }
#pragma unroll 4
            for (int c = 0; c < n_cells; ++c) {
                const long long *src = SG + (long long)c * n_elem + e;
                long long v0, v1 = 0;
                if (two) { const longlong2 v = *reinterpret_cast<const longlong2 *>(src); v0 = v.x; v1 = v.y; }
                else v0 = src[0];
                const unsigned m = smask[c];
#pragma unroll
                for (int k = 0; k < TC_SUM_OUT; ++k)
                    if ((m >> k) & 1u) { a0[k] += v0; a1[k] += v1; }
            }
#pragma unroll
            for (int k = 0; k < TC_SUM_OUT; ++k)
                if (o0 + k < n_out) {
                    long long *dst = SGout + (long long)(o0 + k) * n_elem + e;
                    dst[0] = a0[k];
                    if (two) dst[1] = a1[k];
                }
        }
    }
}

// ------------------------------------------------------------------ combine: digit-plane Grams -> fp64 Gram
// G[set][c1][c2] = 2^(E1+E2) * sum_{k<=S1, l<=S2, k+l<=SMAX+1} 2^-(p_k+p_l) SG[set][plane(c1,k)][plane(c2,l)],
// p_k = 6 + 7(k-1).  Only plane pairs with level(k) <= level(l) were computed; the others are read
// transposed.  Terms are added from the smallest weight to the largest (fixed order).
__global__ void __launch_bounds__(256)
tc_combine_kernel(const long long *__restrict__ SG, long long S, const int *__restrict__ colE,
                  const int *__restrict__ colS, const int *__restrict__ plane_row, int n_aug,
                  double *__restrict__ G, long long ldg) {
    const int set = blockIdx.z;
    const int c1 = blockIdx.y;
    const long long *SGs = SG + (long long)set * S * S;
    double *Gs = G + (long long)set * n_aug * ldg;
    for (int c2 = blockIdx.x * 256 + threadIdx.x; c2 < n_aug; c2 += gridDim.x * 256) {
        if (c2 < c1) continue;                                   // upper triangle, mirrored
        const int S1 = colS[c1], S2 = colS[c2];
        double acc = 0.0;
        for (int tot = TC_SMAX + 1; tot >= 2; --tot) {           // k + l = tot, smallest weights first
            double part = 0.0;
            for (int k = 1; k <= S1; ++k) {
                const int l = tot - k;
                if (l < 1 || l > S2) continue;
                const int r1 = plane_row[c1 * TC_SMAX + (k - 1)], r2 = plane_row[c2 * TC_SMAX + (l - 1)];
                const long long v = (k <= l) ? SGs[(long long)r1 * S + r2] : SGs[(long long)r2 * S + r1];
                part += (double)v;                               // exact: |v| < 2^53, few terms
            }
            acc += scalbn(part, -(12 + 7 * (tot - 2)));
        }
        const double g = scalbn(acc, colE[c1] + colE[c2]);
        Gs[(long long)c1 * ldg + c2] = g;
        Gs[(long long)c2 * ldg + c1] = g;
    }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

}  // namespace sglm

using namespace sglm;

// Plan layout exchanged with the caller (all int32, host memory):
//   colS_host[n_aug]            in : digit planes per column (from sglm_gram_tc_analyze_f64)
//   set_rows_host[n_sets]       in : rows of each set
// Derived inside (deterministic, so sizes can be queried first):
//   plane p of column c -> row of At:  planes are laid out level-major (all columns that have a
//   level-1 plane, then level 2, ...), each level padded to a multiple of 256 rows.
struct TcPlan {
    int n_aug, n_sets;
    long long S;                        // rows of At (digit planes incl. padding), multiple of 256
    long long n_pos;                    // columns of At (positions), multiple of 128
    std::vector<int> plane_row;         // [n_aug * TC_SMAX]
    std::vector<int> level_off, level_cnt;
    std::vector<int2> tiles;
    std::vector<int2> pairs;            // (tile, right-hand neighbour in the same tile row | -1): one 2-CTA cluster each
    int n_parts;                        // K parts per tile (work items = tiles * n_parts)
    std::vector<TcSeg> segs;
    std::vector<long long> set_pos0;    // first position of each set
};

static void tc_make_plan(int n_aug, const int *colS, int n_sets, const long long *set_rows, TcPlan &p) {
    p.n_aug = n_aug; p.n_sets = n_sets;
    p.plane_row.assign((size_t)n_aug * TC_SMAX, -1);
    p.level_off.assign(TC_SMAX + 1, 0); p.level_cnt.assign(TC_SMAX + 1, 0);
    long long off = 0;
    for (int k = 1; k <= TC_SMAX; ++k) {
        p.level_off[k] = (int)off;
        int cnt = 0;
        for (int c = 0; c < n_aug; ++c)
            if (colS[c] >= k) p.plane_row[(size_t)c * TC_SMAX + (k - 1)] = (int)off + cnt++;
        p.level_cnt[k] = cnt;
        off += ((long long)cnt + 255) / 256 * 256;
    }
    p.S = std::max<long long>(off, 256);
    // output tiles: level pairs (k <= l, k + l <= SMAX + 1)
    p.tiles.clear();
    for (int k = 1; k <= TC_SMAX; ++k)
        for (int l = k; l <= TC_SMAX && k + l <= TC_SMAX + 1; ++l) {
            if (!p.level_cnt[k] || !p.level_cnt[l]) continue;
            const int mt0 = p.level_off[k] / TC_BM, mt1 = (p.level_off[k] + p.level_cnt[k] + TC_BM - 1) / TC_BM;
            const int nt0 = p.level_off[l] / TC_BN, nt1 = (p.level_off[l] + p.level_cnt[l] + TC_BN - 1) / TC_BN;
            for (int mt = mt0; mt < mt1; ++mt)
                for (int nt = nt0; nt < nt1; ++nt) {
                    if (k == l && (long long)(nt + 1) * TC_BN <= (long long)mt * TC_BM) continue;  // strictly below the diagonal
                    p.tiles.push_back(make_int2(mt, nt));
                }
        }
    // pairs of neighbouring tiles of one tile row share their A strip: a 2-CTA cluster loads it once (TMA multicast)
    p.pairs.clear();
    for (size_t i = 0; i < p.tiles.size();) {
        if (i + 1 < p.tiles.size() && p.tiles[i + 1].x == p.tiles[i].x && p.tiles[i + 1].y == p.tiles[i].y + 1) {
            p.pairs.push_back(make_int2((int)i, (int)i + 1));
            i += 2;
        } else {
            p.pairs.push_back(make_int2((int)i, -1));
            i += 1;
        }
    }
    // K parts: fill the SMs evenly (>= 3 waves when the K extent allows it)
    {
        const int sms = sm_count();
        const int nt = std::max<int>(1, 2 * (int)p.pairs.size());
        long long total_kb = 0;
        for (int s = 0; s < n_sets; ++s) total_kb += (set_rows[s] + TC_BK - 1) / TC_BK;
        int best = 1;
        double best_eff = 0.0;
        for (int parts = 1; parts <= 16; ++parts) {
            if (parts > 1 && total_kb / parts < 64) break;
            const long long items = (long long)nt * parts;
            const double eff = (double)items / (double)(((items + sms - 1) / sms) * sms);
            const double score = eff - (items < 2LL * sms ? 0.5 : 0.0) - 0.002 * parts;
            if (score > best_eff) { best_eff = score; best = parts; }
        }
        p.n_parts = best;
        if (const char *v = tuning_env("SGLM_TC_PARTS")) p.n_parts = std::max(1, std::min(16, atoi(v)));      // measurement switch
    }
    // K segments: each set's rows padded to 128, cut into pieces that cannot overflow int32
    p.segs.clear(); p.set_pos0.assign(n_sets, 0);
    long long pos = 0;
    for (int s = 0; s < n_sets; ++s) {
        p.set_pos0[s] = pos;
        long long kb = (set_rows[s] + TC_BK - 1) / TC_BK;
        long long kb0 = pos / TC_BK;
        int first = 1;
        if (kb == 0) { p.segs.push_back(TcSeg{(int)kb0, 0, s, 1}); }
        while (kb > 0) {
            const int n = (int)std::min<long long>(kb, TC_MAX_KB_PER_SEG);
            p.segs.push_back(TcSeg{(int)kb0, n, s, first});
            first = 0; kb0 += n; kb -= n;
        }
        pos += (set_rows[s] + TC_BK - 1) / TC_BK * TC_BK;
    }
    p.n_pos = std::max<long long>(pos, TC_BK);
}

static inline size_t tc_align(size_t x) { return (x + 1023) & ~(size_t)1023; }

struct TcLayout { size_t off_at, off_sg, off_sgout, off_member, off_plane, off_tiles, off_segs, off_prog, off_pairs, total; };

// n_out > 0: the plan's sets are cells and n_out row sets are summed from them (extra int64 Grams + the
// membership table)
static TcLayout tc_layout(const TcPlan &p, int n_out = 0) {
    TcLayout L;
    size_t o = 0;
    L.off_at = o; o += tc_align((size_t)p.S * p.n_pos);
    L.off_sg = o; o += tc_align((size_t)p.n_sets * p.S * p.S * sizeof(long long));
    L.off_sgout = o; o += tc_align((size_t)n_out * p.S * p.S * sizeof(long long));
    L.off_member = o; o += tc_align((size_t)n_out * p.n_sets * sizeof(int));
    L.off_plane = o; o += tc_align(p.plane_row.size() * sizeof(int));
    L.off_tiles = o; o += tc_align(p.tiles.size() * sizeof(int2));
    L.off_segs = o; o += tc_align(p.segs.size() * sizeof(TcSeg));
    L.off_prog = o; o += tc_align(2 * p.pairs.size() * (size_t)std::max(p.n_parts, 1) * sizeof(int));
    L.off_pairs = o; o += tc_align(p.pairs.size() * sizeof(int2));
    L.total = o;
    return L;
}

// Lag designs (sglm_lag_design): digit planes of the base signals [base | 1] (consecutive rows of Bt, no level padding)
// and the extra workspace behind the ordinary layout: Bt, its plane table, the (row of Bt, offset) map of At's rows.
static void tc_lag_base_planes(int P, const int *baseS_host, std::vector<int> &bplane, int &nb) {
    bplane.assign((size_t)(P + 1) * TC_SMAX, -1);
    nb = 0;
    for (int q = 0; q <= P; ++q)
        for (int k = 0; k < std::min(std::max(baseS_host[q], 1), TC_SMAX); ++k) bplane[(size_t)q * TC_SMAX + k] = nb++;
}
struct TcLagLayout { size_t off_bt, off_bplane, off_map, total; long long ld_bt; };
static TcLagLayout tc_lag_layout(size_t base_total, int nb, int P, long long n_u, long long S) {
    TcLagLayout LL;
    LL.ld_bt = (std::max<long long>(n_u, 1) + 127) / 128 * 128;
    size_t o = tc_align(base_total);
    LL.off_bt = o; o += tc_align((size_t)nb * LL.ld_bt + 1024);
    LL.off_bplane = o; o += tc_align((size_t)(P + 1) * TC_SMAX * sizeof(int));
    LL.off_map = o; o += tc_align((size_t)S * sizeof(int2));
    LL.total = o;
    return LL;
}

// Pass 1: per-column exponent and number of digit planes (device arrays colE, colS of n_aug int32;
// colmax_scratch: n_aug uint64; flag: 1 int32, set when the data contain NaN/inf).
static int gram_tc_analyze(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                           int32_t C, const double *rs, int max_planes, int32_t *colE, int32_t *colS,
                           uint64_t *colmax_scratch, int32_t *flag, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C >= 0 && n_y >= 0 && ldx >= C && ldy >= n_y, SGLM_E_SHAPE, "gram_tc_analyze: bad shape");
    SGLM_CHECK_ARG(colE && colS && colmax_scratch && flag, SGLM_E_INVALID_ARG, "gram_tc_analyze: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int n_aug = C + n_y + 1;
    SGLM_CUDA_OK(cudaMemsetAsync(colmax_scratch, 0, (size_t)n_aug * sizeof(uint64_t), st));
    SGLM_CUDA_OK(cudaMemsetAsync(flag, 0, sizeof(int), st));
    SGLM_CUDA_OK(cudaMemsetAsync(colS, 0x7f, (size_t)n_aug * sizeof(int), st));       // running minimum of the lowest set bit
    const int gy = (int)std::max<long long>(1, std::min<long long>(T / 256, 64LL * sm_count() / std::max(1, ceil_div(n_aug, 256))));
    dim3 grid(ceil_div(n_aug, 256), gy);
    if (T > 0) {
        tc_colmax_kernel<<<grid, 256, 0, st>>>(X, ldx, Y, ldy, C, n_y, T, rs, (unsigned long long *)colmax_scratch, colS);
        SGLM_LAUNCH_OK("tc_colmax_kernel");
    }
    tc_exponent_kernel<<<ceil_div(n_aug, 256), 256, 0, st>>>((const unsigned long long *)colmax_scratch, n_aug, max_planes, colE, colS, flag);
    SGLM_LAUNCH_OK("tc_exponent_kernel");
    if (T > 0 && max_planes == TC_SMAX && tuning_env("SGLM_TC_DIGIT_PASS")) {
        // validation switch: the digit-by-digit second pass (atomicMax on colS) must not raise any count
        tc_digits_kernel<<<grid, 256, 0, st>>>(X, ldx, Y, ldy, C, n_y, T, rs, colE, colS);
        SGLM_LAUNCH_OK("tc_digits_kernel");
    }
    return SGLM_OK;
}

extern "C" int sglm_gram_tc_analyze_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                                        int64_t T, int32_t C, int32_t *colE, int32_t *colS,
                                        uint64_t *colmax_scratch, int32_t *flag, void *stream) {
    return gram_tc_analyze(X, ldx, Y, ldy, n_y, T, C, nullptr, TC_SMAX, colE, colS, colmax_scratch, flag, stream);
}

// The analysis in two steps, for designs whose ROWS are spread over several GPUs: every rank runs the column pass
// over its rows (colmax_bits = bits of max |z| per column, col_lsb = lowest set bit per column), the ranks combine
// them (max / min: an all-reduce of 2 * n_aug integers), and every rank derives the same exponents and digit-plane
// counts — so the integer digit planes, and the int64 plane Grams that are then summed over the ranks, are those of
// the one-GPU computation bit for bit.
static int gram_tc_colstats(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                            int32_t C, const double *rs, uint64_t *colmax_bits, int32_t *col_lsb, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int n_aug = C + n_y + 1;
    SGLM_CUDA_OK(cudaMemsetAsync(colmax_bits, 0, (size_t)n_aug * sizeof(uint64_t), st));
    SGLM_CUDA_OK(cudaMemsetAsync(col_lsb, 0x7f, (size_t)n_aug * sizeof(int), st));
    if (T > 0) {
        const int gy = (int)std::max<long long>(1, std::min<long long>(T / 256, 64LL * sm_count() / std::max(1, ceil_div(n_aug, 256))));
        dim3 grid(ceil_div(n_aug, 256), gy);
        tc_colmax_kernel<<<grid, 256, 0, st>>>(X, ldx, Y, ldy, C, n_y, T, rs, (unsigned long long *)colmax_bits, col_lsb);
        SGLM_LAUNCH_OK("tc_colmax_kernel");
    }
    return SGLM_OK;
}

extern "C" int sglm_gram_tc_colstats_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                                         int64_t T, int32_t C, uint64_t *colmax_bits, int32_t *col_lsb, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C >= 0 && n_y >= 0 && ldx >= C && ldy >= n_y, SGLM_E_SHAPE, "gram_tc_colstats: bad shape");
    SGLM_CHECK_ARG(colmax_bits && col_lsb, SGLM_E_INVALID_ARG, "gram_tc_colstats: null pointer");
    return gram_tc_colstats(X, ldx, Y, ldy, n_y, T, C, nullptr, colmax_bits, col_lsb, stream);
}

// The column pass of the weighted Gram (rows scaled by row_scale, as in sglm_gram_tc_analyze_scaled_f64) over THIS
// rank's rows; sglm_gram_tc_exponents with the Gram's max_planes finishes the analysis after the ranks' max / min.
extern "C" int sglm_gram_tc_colstats_scaled_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                                                int64_t T, int32_t C, const double *row_scale, uint64_t *colmax_bits,
                                                int32_t *col_lsb, void *stream) {
    SGLM_CHECK_ARG(T >= 0 && C >= 0 && n_y >= 0 && ldx >= C && ldy >= n_y, SGLM_E_SHAPE, "gram_tc_colstats_scaled: bad shape");
    SGLM_CHECK_ARG(colmax_bits && col_lsb && (row_scale || T == 0), SGLM_E_INVALID_ARG, "gram_tc_colstats_scaled: null pointer");
    return gram_tc_colstats(X, ldx, Y, ldy, n_y, T, C, row_scale, colmax_bits, col_lsb, stream);
}

// colS holds the (combined) lowest set bits on entry and the digit-plane counts on exit.
extern "C" int sglm_gram_tc_exponents(const uint64_t *colmax_bits, int32_t n_aug, int32_t max_planes, int32_t *colE,
                                      int32_t *colS, int32_t *flag, void *stream) {
    SGLM_CHECK_ARG(colmax_bits && colE && colS && flag && n_aug > 0, SGLM_E_INVALID_ARG, "gram_tc_exponents: bad argument");
    SGLM_CHECK_ARG(max_planes >= 1 && max_planes <= TC_SMAX, SGLM_E_INVALID_ARG, "gram_tc_exponents: max_planes out of range");
    cudaStream_t st = (cudaStream_t)stream;
    SGLM_CUDA_OK(cudaMemsetAsync(flag, 0, sizeof(int), st));
    tc_exponent_kernel<<<ceil_div(n_aug, 256), 256, 0, st>>>((const unsigned long long *)colmax_bits, n_aug, max_planes, colE, colS, flag);
    SGLM_LAUNCH_OK("tc_exponent_kernel");
    return SGLM_OK;
}

// Weighted form: every row t of Z = [X | Y | 1] is scaled by row_scale[t] (= sqrt of a row weight, so that the
// Gram is Z' diag(w) Z), and at most max_planes (1..8) digit planes are kept per column: with fewer planes than
// a column needs its digits are rounded at the last plane (relative error 2^-(7 max_planes)) — the approximate
// Hessian of the Poisson Newton iteration, whose gradient stays exact.
extern "C" int sglm_gram_tc_analyze_scaled_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy,
                                               int32_t n_y, int64_t T, int32_t C, const double *row_scale,
                                               int32_t max_planes, int32_t *colE, int32_t *colS,
                                               uint64_t *colmax_scratch, int32_t *flag, void *stream) {
    SGLM_CHECK_ARG(max_planes >= 1 && max_planes <= TC_SMAX, SGLM_E_INVALID_ARG, "gram_tc_analyze_scaled: max_planes out of range");
    return gram_tc_analyze(X, ldx, Y, ldy, n_y, T, C, row_scale, max_planes, colE, colS, colmax_scratch, flag, stream);
}

// int8 MACs issued = n_ctas * iters * 8 UMMAs * (128 * 256 * 32); the caller times the call with CUDA events.
extern "C" int sglm_probe_mma_i8(int32_t iters, int64_t *n_ctas_host, void *stream) {
    SGLM_CHECK_ARG(iters >= 1 && n_ctas_host, SGLM_E_INVALID_ARG, "probe_mma_i8: bad argument");
    const size_t smem = 1024 + (size_t)TC_STAGE_BYTES + 256;
    SGLM_CUDA_OK(cudaFuncSetAttribute(tc_mma_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int n = sm_count();
    *n_ctas_host = n;
    tc_mma_probe_kernel<<<n, TC_THREADS, smem, (cudaStream_t)stream>>>(iters);
    SGLM_LAUNCH_OK("tc_mma_probe_kernel");
    return SGLM_OK;
}

extern "C" size_t sglm_gram_tc_workspace_bytes(int32_t n_aug, const int32_t *colS_host, int32_t n_sets,
                                               const int64_t *set_rows_host) {
    if (n_aug <= 0 || n_sets <= 0 || !colS_host || !set_rows_host) return 0;
    TcPlan p;
    tc_make_plan(n_aug, colS_host, n_sets, (const long long *)set_rows_host, p);
    return tc_layout(p).total;
}

// Plan summary for reporting: out4 = {digit-plane rows S, positions n_pos, output tiles, K segments}.
extern "C" int sglm_gram_tc_plan_info(int32_t n_aug, const int32_t *colS_host, int32_t n_sets,
                                      const int64_t *set_rows_host, int64_t *out4) {
    SGLM_CHECK_ARG(n_aug > 0 && n_sets > 0 && colS_host && set_rows_host && out4, SGLM_E_INVALID_ARG,
                   "gram_tc_plan_info: bad argument");
    TcPlan p;
    tc_make_plan(n_aug, colS_host, n_sets, (const long long *)set_rows_host, p);
    out4[0] = p.S; out4[1] = p.n_pos; out4[2] = (int64_t)p.tiles.size(); out4[3] = (int64_t)p.n_parts;
    return SGLM_OK;
}

// Pass 2: slices, int8 tcgen05 GEMM, combine.  rows: device int64 [sum of 128-padded set sizes]
// (concatenated row lists of the sets, -1 = padding), built by the caller in set order.
// use_check_gemm != 0 runs the CUDA-core integer GEMM instead of tcgen05 (cross-check, small sizes).
static int gram_tc_run(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                       int32_t C, const int32_t *colE, const int32_t *colS, const int32_t *colS_host,
                       int32_t n_sets, const int64_t *set_rows_host, const int64_t *rows, int32_t n_out,
                       const int32_t *member_host, double *G, int64_t ldg, void *workspace, size_t workspace_bytes,
                       int32_t use_check_gemm, void *stream, const double *rs = nullptr, int stage = 0,
                       const sglm_lag_design *lag = nullptr);

extern "C" int sglm_gram_tc_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                                int32_t C, const int32_t *colE, const int32_t *colS, const int32_t *colS_host,
                                int32_t n_sets, const int64_t *set_rows_host, const int64_t *rows, double *G,
                                int64_t ldg, void *workspace, size_t workspace_bytes, int32_t use_check_gemm,
                                void *stream) {
    return gram_tc_run(X, ldx, Y, ldy, n_y, T, C, colE, colS, colS_host, n_sets, set_rows_host, rows, 0, nullptr, G, ldg,
                       workspace, workspace_bytes, use_check_gemm, stream);
}

// Weighted Gram Z' diag(row_scale^2) Z with the planes chosen by sglm_gram_tc_analyze_scaled_f64.
extern "C" int sglm_gram_tc_scaled_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                                       int64_t T, int32_t C, const double *row_scale, const int32_t *colE,
                                       const int32_t *colS, const int32_t *colS_host, int32_t n_sets,
                                       const int64_t *set_rows_host, const int64_t *rows, double *G, int64_t ldg,
                                       void *workspace, size_t workspace_bytes, void *stream) {
    return gram_tc_run(X, ldx, Y, ldy, n_y, T, C, colE, colS, colS_host, n_sets, set_rows_host, rows, 0, nullptr, G, ldg,
                       workspace, workspace_bytes, 0, stream, row_scale);
}

extern "C" size_t sglm_gram_tc_cells_workspace_bytes(int32_t n_aug, const int32_t *colS_host, int32_t n_cells,
                                                     const int64_t *cell_rows_host, int32_t n_out) {
    if (n_aug <= 0 || n_cells <= 0 || n_out <= 0 || !colS_host || !cell_rows_host) return 0;
    TcPlan p;
    tc_make_plan(n_aug, colS_host, n_cells, (const long long *)cell_rows_host, p);
    return tc_layout(p, n_out).total;
}

// Same statistics from DISJOINT cells: rows = concatenated (128-padded) row lists of the n_cells cells,
// member_host[o * n_cells + c] != 0 when cell c belongs to output row set o; G holds the n_out sets.
extern "C" int sglm_gram_tc_cells_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                                      int64_t T, int32_t C, const int32_t *colE, const int32_t *colS,
                                      const int32_t *colS_host, int32_t n_cells, const int64_t *cell_rows_host,
                                      const int64_t *rows, int32_t n_out, const int32_t *member_host, double *G,
                                      int64_t ldg, void *workspace, size_t workspace_bytes, int32_t use_check_gemm,
                                      void *stream) {
    SGLM_CHECK_ARG(n_out >= 1 && member_host, SGLM_E_INVALID_ARG, "gram_tc_cells: membership table missing");
    SGLM_CHECK_ARG(n_cells <= TC_SUM_CELLS, SGLM_E_UNSUPPORTED, "gram_tc_cells: at most %d cells", TC_SUM_CELLS);
    return gram_tc_run(X, ldx, Y, ldy, n_y, T, C, colE, colS, colS_host, n_cells, cell_rows_host, rows, n_out,
                       member_host, G, ldg, workspace, workspace_bytes, use_check_gemm, stream);
}

// Row-sharded form of sglm_gram_tc_cells_f64 (one process per GPU, each holding a slice of the rows):
//   partial : slicing + int8 GEMM + cell sums of THIS rank's rows; leaves the int64 plane Grams of the n_out row
//             sets at sglm_gram_tc_cells_sgout(...) inside the workspace (offset / byte count are the same on every
//             rank because the digit-plane layout depends only on the combined column analysis);
//   the caller adds them over the ranks (ncclAllReduce, int64 sum: exact, so the bits equal the one-GPU result);
//   combine : fp64 recombination of the summed plane Grams -> G.
extern "C" int sglm_gram_tc_cells_sgout(int32_t n_aug, const int32_t *colS_host, int32_t n_cells,
                                        const int64_t *cell_rows_host, int32_t n_out, uint64_t *offset_bytes,
                                        uint64_t *size_bytes) {
    SGLM_CHECK_ARG(n_aug > 0 && n_cells > 0 && n_out > 0 && colS_host && cell_rows_host && offset_bytes && size_bytes,
                   SGLM_E_INVALID_ARG, "gram_tc_cells_sgout: bad argument");
    TcPlan p;
    tc_make_plan(n_aug, colS_host, n_cells, (const long long *)cell_rows_host, p);
    const TcLayout L = tc_layout(p, n_out);
    *offset_bytes = L.off_sgout;
    *size_bytes = (uint64_t)n_out * p.S * p.S * sizeof(long long);
    return SGLM_OK;
}

extern "C" int sglm_gram_tc_cells_partial_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                                              int64_t T, int32_t C, const int32_t *colE, const int32_t *colS,
                                              const int32_t *colS_host, int32_t n_cells, const int64_t *cell_rows_host,
                                              const int64_t *rows, int32_t n_out, const int32_t *member_host,
                                              void *workspace, size_t workspace_bytes, void *stream) {
    SGLM_CHECK_ARG(n_out >= 1 && member_host, SGLM_E_INVALID_ARG, "gram_tc_cells_partial: membership table missing");
    SGLM_CHECK_ARG(n_cells <= TC_SUM_CELLS, SGLM_E_UNSUPPORTED, "gram_tc_cells_partial: at most %d cells", TC_SUM_CELLS);
    double dummy;
    return gram_tc_run(X, ldx, Y, ldy, n_y, T, C, colE, colS, colS_host, n_cells, cell_rows_host, rows, n_out,
                       member_host, &dummy, C + n_y + 1, workspace, workspace_bytes, 0, stream, nullptr, 1);
}

// Weighted form of sglm_gram_tc_cells_partial_f64 (rows of Z scaled by row_scale; colE / colS from
// sglm_gram_tc_colstats_scaled_f64 + sglm_gram_tc_exponents with the Gram's max_planes): a rank's share of
// Z' diag(row_scale^2) Z as int64 plane Grams.  The digits of a row depend only on that row and the combined analysis,
// so the partials summed over ANY partition of the rows and then combined are the bits of sglm_gram_tc_scaled_f64.
extern "C" int sglm_gram_tc_scaled_partial_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                                               int64_t T, int32_t C, const double *row_scale, const int32_t *colE,
                                               const int32_t *colS, const int32_t *colS_host, int32_t n_cells,
                                               const int64_t *cell_rows_host, const int64_t *rows, int32_t n_out,
                                               const int32_t *member_host, void *workspace, size_t workspace_bytes,
                                               void *stream) {
    SGLM_CHECK_ARG(n_out >= 1 && member_host, SGLM_E_INVALID_ARG, "gram_tc_scaled_partial: membership table missing");
    SGLM_CHECK_ARG(n_cells <= TC_SUM_CELLS, SGLM_E_UNSUPPORTED, "gram_tc_scaled_partial: at most %d cells", TC_SUM_CELLS);
    SGLM_CHECK_ARG(row_scale || T == 0, SGLM_E_INVALID_ARG, "gram_tc_scaled_partial: null row_scale");
    double dummy;
    return gram_tc_run(X, ldx, Y, ldy, n_y, T, C, colE, colS, colS_host, n_cells, cell_rows_host, rows, n_out,
                       member_host, &dummy, C + n_y + 1, workspace, workspace_bytes, 0, stream, row_scale, 1);
}

extern "C" int sglm_gram_tc_cells_combine_f64(int32_t C, int32_t n_y, const int32_t *colE, const int32_t *colS,
                                              const int32_t *colS_host, int32_t n_cells, const int64_t *cell_rows_host,
                                              int32_t n_out, double *G, int64_t ldg, void *workspace,
                                              size_t workspace_bytes, void *stream) {
    SGLM_CHECK_ARG(n_out >= 1, SGLM_E_INVALID_ARG, "gram_tc_cells_combine: n_out");
    static const int64_t no_rows = 0;
    return gram_tc_run(nullptr, C, nullptr, n_y, n_y, 0, C, colE, colS, colS_host, n_cells, cell_rows_host, &no_rows,
                       n_out, nullptr, G, ldg, workspace, workspace_bytes, 0, stream, nullptr, 2);
}

// Lag designs: the same statistics WITHOUT the design matrix (see tc_expand_kernel).  n_out == 0: the row lists are
// the sets themselves; n_out > 0: cells + membership as in sglm_gram_tc_cells_f64.  partial != 0: stop after the
// int64 plane Grams (row-sharded use; finish with sglm_gram_tc_cells_combine_f64 — the ordinary part of the
// workspace has the ordinary layout).
extern "C" size_t sglm_gram_tc_lag_workspace_bytes(int32_t n_aug, const int32_t *colS_host, int32_t n_cells,
                                                   const int64_t *cell_rows_host, int32_t n_out, int32_t P,
                                                   const int32_t *baseS_host, int64_t n_u) {
    if (n_aug <= 0 || n_cells <= 0 || n_out < 0 || !colS_host || !cell_rows_host || P <= 0 || !baseS_host || n_u < 0) return 0;
    TcPlan p;
    tc_make_plan(n_aug, colS_host, n_cells, (const long long *)cell_rows_host, p);
    std::vector<int> bplane;
    int nb = 0;
    tc_lag_base_planes(P, baseS_host, bplane, nb);
    return tc_lag_layout(tc_layout(p, n_out).total, nb, P, n_u, p.S).total;
}

extern "C" int sglm_gram_tc_lag_cells_f64(const sglm_lag_design *lag, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                                          int32_t C, const int32_t *colE, const int32_t *colS, const int32_t *colS_host,
                                          int32_t n_cells, const int64_t *cell_rows_host, const int64_t *rows,
                                          int32_t n_out, const int32_t *member_host, double *G, int64_t ldg,
                                          void *workspace, size_t workspace_bytes, int32_t partial, void *stream) {
    SGLM_CHECK_ARG(lag != nullptr, SGLM_E_INVALID_ARG, "gram_tc_lag_cells: null lag design");
    SGLM_CHECK_ARG(n_out == 0 || member_host, SGLM_E_INVALID_ARG, "gram_tc_lag_cells: membership table missing");
    SGLM_CHECK_ARG(n_out == 0 || n_cells <= TC_SUM_CELLS, SGLM_E_UNSUPPORTED, "gram_tc_lag_cells: at most %d cells", TC_SUM_CELLS);
    SGLM_CHECK_ARG(!partial || n_out > 0, SGLM_E_INVALID_ARG, "gram_tc_lag_cells: the partial form needs output sets");
    double dummy;
    return gram_tc_run(nullptr, C, Y, ldy, n_y, T, C, colE, colS, colS_host, n_cells, cell_rows_host, rows, n_out,
                       member_host, partial ? &dummy : G, partial ? (int64_t)(C + n_y + 1) : ldg, workspace, workspace_bytes, 0,
                       stream, nullptr, partial ? 1 : 0, lag);
}

static int gram_tc_run(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                       int32_t C, const int32_t *colE, const int32_t *colS, const int32_t *colS_host,
                       int32_t n_sets, const int64_t *set_rows_host, const int64_t *rows, int32_t n_out,
                       const int32_t *member_host, double *G, int64_t ldg, void *workspace, size_t workspace_bytes,
                       int32_t use_check_gemm, void *stream, const double *rs, int stage, const sglm_lag_design *lag) {
    const int n_aug = C + n_y + 1;
    SGLM_CHECK_ARG(T >= 0 && C >= 0 && n_y >= 0 && n_sets >= 1 && ldx >= C && ldy >= n_y && ldg >= n_aug, SGLM_E_SHAPE,
                   "gram_tc: bad shape");
    SGLM_CHECK_ARG(colE && colS && colS_host && set_rows_host && rows && G && workspace, SGLM_E_INVALID_ARG,
                   "gram_tc: null pointer");
    SGLM_CHECK_ARG(((uintptr_t)workspace & 1023) == 0, SGLM_E_ALIGN, "gram_tc: workspace must be 1024-byte aligned");
    TcPlan p;
    tc_make_plan(n_aug, colS_host, n_sets, (const long long *)set_rows_host, p);
    const TcLayout L = tc_layout(p, n_out);
    SGLM_CHECK_ARG(workspace_bytes >= L.total, SGLM_E_WORKSPACE, "gram_tc: workspace too small (%zu < %zu)",
                   workspace_bytes, L.total);
    SGLM_CHECK_ARG(p.n_pos < 0x7fffffffLL && p.S < 0x7fffffffLL, SGLM_E_SHAPE, "gram_tc: problem too large");
    cudaStream_t st = (cudaStream_t)stream;
    char *ws = (char *)workspace;
    int8_t *At = (int8_t *)(ws + L.off_at);
    long long *SG = (long long *)(ws + L.off_sg);
    int *d_plane = (int *)(ws + L.off_plane);
    int2 *d_tiles = (int2 *)(ws + L.off_tiles);
    TcSeg *d_segs = (TcSeg *)(ws + L.off_segs);
    // the slicing pass writes every position of every real digit-plane row; only the padding rows
    // between levels have to be cleared
    if (stage != 2) {
        long long covered = 0;
        for (int k = 1; k <= TC_SMAX; ++k) {
            const long long lo = (long long)p.level_off[k] + p.level_cnt[k];
            const long long hi = (long long)p.level_off[k] + ((long long)p.level_cnt[k] + 255) / 256 * 256;
            if (hi > lo) SGLM_CUDA_OK(cudaMemsetAsync(At + lo * p.n_pos, 0, (size_t)(hi - lo) * p.n_pos, st));
            covered = std::max(covered, hi);
        }
        if (p.S > covered) SGLM_CUDA_OK(cudaMemsetAsync(At + covered * p.n_pos, 0, (size_t)(p.S - covered) * p.n_pos, st));
    }
    if (stage != 2) {
        SGLM_CUDA_OK(cudaMemcpyAsync(d_plane, p.plane_row.data(), p.plane_row.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        SGLM_CUDA_OK(cudaMemcpyAsync(d_tiles, p.tiles.data(), p.tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
        SGLM_CUDA_OK(cudaMemcpyAsync(ws + L.off_pairs, p.pairs.data(), p.pairs.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
        SGLM_CUDA_OK(cudaMemcpyAsync(d_segs, p.segs.data(), p.segs.size() * sizeof(TcSeg), cudaMemcpyHostToDevice, st));
    }
    long long *SGout = (long long *)(ws + L.off_sgout);
    int *d_member = (int *)(ws + L.off_member);
    if (stage == 2) {
        // combine only: the int64 Grams of the output sets are already in the workspace (summed over the ranks)
        SGLM_CUDA_OK(cudaMemcpyAsync(d_plane, p.plane_row.data(), p.plane_row.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        SGLM_CUDA_OK(cudaStreamSynchronize(st));
        const long long *SGfin2 = n_out > 0 ? SGout : SG;
        const int n_fin2 = n_out > 0 ? n_out : n_sets;
        dim3 cgrid2((unsigned)std::min(ceil_div(n_aug, 256), 32), (unsigned)n_aug, (unsigned)n_fin2);
        tc_combine_kernel<<<cgrid2, 256, 0, st>>>(SGfin2, p.S, colE, colS, d_plane, n_aug, G, ldg);
        SGLM_LAUNCH_OK("tc_combine_kernel");
        return SGLM_OK;
    }
    if (n_out > 0)
        SGLM_CUDA_OK(cudaMemcpyAsync(d_member, member_host, (size_t)n_out * n_sets * sizeof(int), cudaMemcpyHostToDevice, st));
    TcLagLayout LL = {};
    std::vector<int> bplane;
    std::vector<int2> lag_map;
    if (lag) {
        // lag design: planes of the base signals + the map (row of Bt, row offset) of every plane row of At
        SGLM_CHECK_ARG(rs == nullptr, SGLM_E_UNSUPPORTED, "gram_tc: row scales are not supported for lag designs");
        SGLM_CHECK_ARG(lag->base && lag->src_host && lag->off_host && lag->baseE && lag->baseS && lag->baseS_host &&
                       lag->P > 0 && lag->ldb >= lag->P && lag->n_u >= T, SGLM_E_INVALID_ARG, "gram_tc: bad lag design");
        int nb = 0;
        tc_lag_base_planes(lag->P, lag->baseS_host, bplane, nb);
        LL = tc_lag_layout(L.total, nb, lag->P, lag->n_u, p.S);
        SGLM_CHECK_ARG(workspace_bytes >= LL.total, SGLM_E_WORKSPACE, "gram_tc: workspace too small for the lag design (%zu < %zu)",
                       workspace_bytes, LL.total);
        lag_map.assign((size_t)p.S, make_int2(-1, 0));
        for (int c = 0; c < C; ++c) {
            const int pc = lag->src_host[c], off = lag->off_host[c];
            SGLM_CHECK_ARG(pc >= 0 && pc < lag->P && off >= 0 && (long long)off + T <= lag->n_u, SGLM_E_INVALID_ARG,
                           "gram_tc: lag column %d reads outside the base window", c);
            for (int k = 0; k < colS_host[c]; ++k) {
                const int r = p.plane_row[(size_t)c * TC_SMAX + k], b = bplane[(size_t)pc * TC_SMAX + k];
                SGLM_CHECK_ARG(r >= 0 && b >= 0, SGLM_E_INVALID_ARG, "gram_tc: lag column %d has more planes than its base signal", c);
                lag_map[(size_t)r] = make_int2(b, off);
            }
        }
        SGLM_CUDA_OK(cudaMemcpyAsync(ws + LL.off_bplane, bplane.data(), bplane.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        SGLM_CUDA_OK(cudaMemcpyAsync(ws + LL.off_map, lag_map.data(), lag_map.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
    }
    SGLM_CUDA_OK(cudaStreamSynchronize(st));        // the pageable host vectors above die with this frame

    if (lag) {
        int8_t *Bt = (int8_t *)(ws + LL.off_bt);
        dim3 bgrid((unsigned)(LL.ld_bt / 128), (unsigned)ceil_div(lag->P + 1, 32));
        tc_slice_kernel<<<bgrid, 256, 0, st>>>(lag->base, lag->ldb, nullptr, 0, lag->P, 0, nullptr, nullptr, LL.ld_bt, lag->baseE,
                                               lag->baseS, (const int *)(ws + LL.off_bplane), Bt, LL.ld_bt, lag->n_u);
        SGLM_LAUNCH_OK("tc_slice_kernel(base)");
        dim3 egrid((unsigned)ceil_div<long long>(p.n_pos, TC_EXP_POS), (unsigned)ceil_div((int)p.S, TC_EXP_ROWS));
        tc_expand_kernel<<<egrid, 256, 0, st>>>(Bt, LL.ld_bt, (const long long *)rows, p.n_pos, (const int2 *)(ws + LL.off_map),
                                                (int)p.S, At, p.n_pos);
        SGLM_LAUNCH_OK("tc_expand_kernel");
        // response columns and the ones column: sliced from Y as before
        dim3 ygrid((unsigned)(p.n_pos / 128), (unsigned)ceil_div(n_y + 1, 32));
        tc_slice_kernel<<<ygrid, 256, 0, st>>>(nullptr, 0, Y, ldy, 0, n_y, nullptr, (const long long *)rows, p.n_pos, colE + C,
                                               colS + C, d_plane + (size_t)C * TC_SMAX, At, p.n_pos, 0);
        SGLM_LAUNCH_OK("tc_slice_kernel(y)");
    } else {
    dim3 sgrid((unsigned)(p.n_pos / 128), (unsigned)ceil_div(n_aug, 32));
    tc_slice_kernel<<<sgrid, 256, 0, st>>>(X, ldx, Y, ldy, C, n_y, rs, (const long long *)rows, p.n_pos, colE, colS,
                                           d_plane, At, p.n_pos, 0);
    SGLM_LAUNCH_OK("tc_slice_kernel");
    }

    const int n_tiles = (int)p.tiles.size();
    if (n_tiles > 0) {
        tc_zero_tiles_kernel<<<dim3((unsigned)n_tiles, (unsigned)p.n_sets), 256, 0, st>>>(SG, p.S, d_tiles);
        SGLM_LAUNCH_OK("tc_zero_tiles_kernel");
    }
    if (use_check_gemm) {
        tc_gram_i8_check_kernel<<<n_tiles, 256, 0, st>>>(At, p.n_pos, d_tiles, d_segs, (int)p.segs.size(), SG, p.S);
        SGLM_LAUNCH_OK("tc_gram_i8_check_kernel");
    } else {
        PFN_encodeTiled enc = get_encode_fn();
        SGLM_CHECK_ARG(enc != nullptr, SGLM_E_CUDA, "gram_tc: cuTensorMapEncodeTiled not available");
        CUtensorMap tmap;
        const cuuint64_t gdim[2] = {(cuuint64_t)p.n_pos, (cuuint64_t)p.S};
        const cuuint64_t gstride[1] = {(cuuint64_t)p.n_pos};
        const cuuint32_t box[2] = {(cuuint32_t)TC_BK, 128};
        const cuuint32_t estr[2] = {1, 1};
        CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, At, gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        SGLM_CHECK_ARG(r == CUDA_SUCCESS, SGLM_E_CUDA, "gram_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
        const size_t smem = 1024 + (size_t)TC_STAGES * TC_STAGE_BYTES + 256;
        SGLM_CUDA_OK(cudaFuncSetAttribute(tc_gram_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int *d_prog = (int *)(ws + L.off_prog);
        // measured (profiles/r2_cd_experiments.txt section 12): the K lock-step cuts the DRAM reads 97 -> 25 GB (L2 hit 51 -> 79 %)
        // but the kernel is bound by the L2 -> SM ingest per SM, not by DRAM; with the A strip multicast the throttling only
        // costs time (stage 33.7 ms against 28.6 ms) — off unless asked for
        const bool lockstep = tuning_env("SGLM_TC_LOCKSTEP") != nullptr;
        const int n_pairs = (int)p.pairs.size();
        if (lockstep) SGLM_CUDA_OK(cudaMemsetAsync(d_prog, 0xff, (size_t)2 * n_pairs * p.n_parts * sizeof(int), st));   // -1: not started
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(2 * n_pairs * p.n_parts));
        cfg.blockDim = dim3(TC_THREADS);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        SGLM_CUDA_OK(cudaLaunchKernelEx(&cfg, tc_gram_i8_kernel, tmap, (const int2 *)d_tiles, n_tiles, p.n_parts, (const TcSeg *)d_segs,
                                        (int)p.segs.size(), SG, (long long)p.S, lockstep ? d_prog : (int *)nullptr,
                                        (const int2 *)(ws + L.off_pairs), n_pairs));
        SGLM_LAUNCH_OK("tc_gram_i8_kernel");
    }
    const long long *SGfin = SG;
    int n_fin = n_sets;
    if (n_out > 0) {
        tc_cell_sum_kernel<<<sm_count() * 8, 256, 0, st>>>(SG, p.S, d_tiles, n_tiles, n_sets, d_member, n_out, SGout);
        SGLM_LAUNCH_OK("tc_cell_sum_kernel");
        SGfin = SGout;
        n_fin = n_out;
    }
    if (stage == 1) return SGLM_OK;                 // the caller sums the int64 set Grams over the ranks, then stage 2
    dim3 cgrid((unsigned)std::min(ceil_div(n_aug, 256), 32), (unsigned)n_aug, (unsigned)n_fin);
    tc_combine_kernel<<<cgrid, 256, 0, st>>>(SGfin, p.S, colE, colS, d_plane, n_aug, G, ldg);
    SGLM_LAUNCH_OK("tc_combine_kernel");
    return SGLM_OK;
}
