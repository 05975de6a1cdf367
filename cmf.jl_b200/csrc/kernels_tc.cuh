// tcgen05 (5th-gen tensor core) engine for the three big contractions of the fp32 CNMF path.
//
// Numerics: every fp32 operand x is split into two bf16 planes, hi = bf16(x), lo = bf16(x - hi),
// and each logical product is issued as three bf16 MMAs  hi*hi + hi*lo + lo*hi  with fp32
// accumulation in TMEM (~16-17 mantissa bits per operand; measured loss drift vs fp64 ~1e-7,
// DESIGN.md section 4).  Data movement: TMA (cp.async.bulk.tensor) into a 4-stage shared-memory ring,
// one elected thread issues tcgen05.mma, accumulators are double-buffered in TMEM (2 x 256
// columns) so the epilogue of one tile overlaps the main loop of the next; CTAs are persistent.
//
// One kernel template, three modes (shapes are per CTA tile, M = 128 TMEM lanes, N = 256 columns):
//   TC_CONV   D[n, t]      = sum_j Wc[n][j] * Hwin[t][j]          j = (L-1-l)*Kp + k   (K-major, SW64)
//             epilogue: sum (D - X[t][n])^2  -> loss partials        (src/common.jl:24-34,54-59)
//   TC_TRANS  D[(i,k), c]  = sum_{g} sum_n Wu[(gG+i)*Kp+k][n] * X[t0+c+gG][n]   (K-major, SW64; G = 128/Kp lags per tile)
//             epilogue: numH[t0+c-i][k] += D[(i,k), c]               (src/common.jl:71-81)
//   TC_CORR   D[j, n]      = sum_t Hwin[t][j] * X[t][n]             (both MN-major, SW128)
//             epilogue: every TC_FLUSH_T columns of t, part[(l,k)][n] (+)= D  in double
//                                                                      (src/algs/mult.jl:31-34)
//   TC_PLAIN  D[m, n]      = sum_k A[m][k] * B[n][k]                (K-major, SW64)  plain GEMM for the two small
//             epilogue: outp[m*ldo + n] = D                          T-independent products G*W and W*W'
// and the two per-frequency products of the frequency-domain engine (kernels_fd.cuh), one unit = (frequency f, column tile):
//   TC_FQT    D[m, b]      = sum_(c,n) Aw[f][m][(c,n)] * Xf[f][b][(c,n)]   (K-major, SW64)   numH^ -> Of[f][b][m]
//   TC_FQC    D[m, n]      = sum_(b,c) Ah[f][(b,c)][m] * Xf[f][(b,c)][n]   (MN-major, SW128) numW^ -> Df[f][m][n]
//   TC_FQX    D[n, b]      = sum_(c,k) Awm[f][co][(c,k)][n] * Hc[f][b][(c,k)]  (A MN-major SW128, B K-major SW64)
//             one unit = (f, co = re/im, tile of 128 units n, tile of 256 blocks): Xhat^ -> Yf[f][b][co][n]   (loss pass)
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cmf {
namespace tc {

constexpr int BM = 128, BN = 256, BK = 32;          // BK: K-elements per stage (K-major) / t rows (MN-major)
constexpr int STAGES = 4;
constexpr int A_PLANE = BM * BK * 2;                 // 8 KB  (one bf16 plane of the A tile)
constexpr int B_PLANE = BN * BK * 2;                 // 16 KB
constexpr int STAGE_BYTES = 2 * A_PLANE + 2 * B_PLANE;   // 48 KB
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024;  // + alignment slack
constexpr int EPI_WARPS = 8;                         // epilogue / promotion warps (2 per TMEM lane quarter)
constexpr int THREADS = 128 + 32 * EPI_WARPS;        // warpgroup 0: warp 0 TMA, warp 1 MMA + TMEM alloc (2,3 idle); warpgroups 1-2: epilogue
constexpr int PROMO = 8;                             // k-blocks accumulated in TMEM before promotion to registers
constexpr int FLUSH_T = 65536;                       // TC_CORR: columns of t accumulated in fp32 registers (RN) before the fp64 flush

enum Mode { TC_CONV = 0, TC_TRANS = 1, TC_CORR = 2, TC_PLAIN = 3, TC_FQT = 4, TC_FQC = 5, TC_FQX = 6 };

struct Params {
    // work decomposition
    int64_t units;          // number of CTA work units
    int64_t tiles_n;        // CONV: n tiles (fastest);  CORR: n tiles (fastest)
    int64_t tiles_m;        // CORR: j tiles
    int64_t nkb;            // CONV: k-blocks per tile
    // TRANS
    int64_t groups, nblocks;   // lag groups, n blocks of BK
    int G, Kp;                 // lags per 128-row group (128 / Kp, rounded down), K padded to a multiple of 8
    int64_t own;               // owned columns per t tile = BN - (G-1)
    // CORR
    int64_t split_len;         // t columns per split (multiple of BK)
    int *lockstep;             // CORR: per-CTA k-block counters (zeroed before the launch) or nullptr
    int lockstep_window;       // a CTA may run at most this many k-blocks ahead of the slowest CTA
    int64_t tau_hi;            // valid X columns [0, tau_hi)
    // dims
    int64_t N, K, L, Tl;
    // epilogue pointers
    const float *X;            // CONV: fp32 data [t][N]
    double *partial;           // CONV: EPI_WARPS partials per unit
    float *out;                // TRANS: numH [t][K];  PLAIN: output matrix
    int64_t Mrows, Ncols, ldo; // PLAIN: output bounds and row stride
    double *part;              // CORR: [split][L*K*N]
    int64_t fq_rows;           // FQT / FQC / FQX: rows of the B map per frequency (nblk resp. 2*nblk)
    int64_t b_off, nbc;        // FQX: first block and number of blocks of the chunk this launch covers
    int64_t MR;                // FQT / FQC / FQX: rows per frequency of the A operand / output (2 Kq = 128 or 256)
    int mtiles;                // FQT / FQC: 128-row tiles per frequency (MR / 128); the tiles of one column tile are adjacent units
    int sym;                   // PLAIN: the product is symmetric (A == B): tiles strictly above the diagonal are skipped, the caller mirrors
};

// Completes a symmetric product computed with Params::sym: the tiles strictly above the diagonal (column tile nt, row
// tile mt with nt*BN >= (mt+1)*BM) take their values from the mirrored entries.
__global__ void mirror_upper_kernel(float *__restrict__ S, int64_t rows, int64_t ld) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, a = blockIdx.y;
    if (b >= rows || a >= rows) return;
    if ((b / 256) * 256 >= (a / 128 + 1) * 128) S[a * ld + b] = S[b * ld + a];
}

// ---------------------------------------------------------------------------------- PTX wrappers
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
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, uint64_t *bar, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, uint64_t *bar, int32_t c0, int32_t c1, int32_t c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap *map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;           // descriptor version (Blackwell)
    d |= (uint64_t)(layout & 7) << 61; // 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
    return d;
}
// instruction descriptor: bf16 x bf16 -> f32, M = 128, N = 256
__host__ __device__ constexpr uint32_t make_idesc(int a_mn_major, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

// ---------------------------------------------------------------------------------- the kernel
// Accumulation is two-level: the tensor core accumulates at most PROMO k-blocks (PROMO*BK/16*3 MMAs)
// into one TMEM buffer -- its fp32 adder truncates, so long chains of same-sign terms pick up a
// systematic bias (measured -3e-8 relative per MMA) -- then the epilogue warps add that partial
// into fp32 registers with round-to-nearest ("promotion") while the other TMEM buffer is being filled.
template <int MODE>
__global__ void __launch_bounds__(THREADS, 1)
tc_kernel(const __grid_constant__ CUtensorMap mapA_hi, const __grid_constant__ CUtensorMap mapA_lo,
          const __grid_constant__ CUtensorMap mapB_hi, const __grid_constant__ CUtensorMap mapB_lo, const Params p) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES], tmem_full[2], tmem_empty[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ float stage_s[(MODE == TC_CORR || MODE == TC_PLAIN || MODE == TC_FQC) ? EPI_WARPS : 1][32][17];   // write-out staging

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        tma_prefetch_desc(&mapA_hi); tma_prefetch_desc(&mapA_lo); tma_prefetch_desc(&mapB_hi); tma_prefetch_desc(&mapB_lo);
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_s)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    // A unit is a sequence of segments (CORR: fp64 flush segments of FLUSH_T columns; others: one),
    // a segment is a range of k-blocks [kb0, kb0 + kbn), consumed in promotion chunks of PROMO k-blocks.
    auto n_segments = [&](int64_t unit) -> int64_t {
        if (MODE == TC_PLAIN && p.sym) {      // every role skips the same tiles: no segment, no pipeline traffic
            const int64_t nt = unit % p.tiles_n, mt = unit / p.tiles_n;
            return (nt * BN >= (mt + 1) * BM) ? 0 : 1;
        }
        if (MODE != TC_CORR) return 1;
        const int64_t sp = unit / (p.tiles_m * p.tiles_n);
        const int64_t ta = sp * p.split_len, tb = min(p.tau_hi, ta + p.split_len);
        const int64_t len = tb > ta ? tb - ta : 0;
        const int64_t c = (len + FLUSH_T - 1) / FLUSH_T;
        return c > 0 ? c : 1;
    };
    auto segment_kb = [&](int64_t unit, int64_t seg, int64_t &kb0, int64_t &kbn) {
        if (MODE == TC_CONV || MODE == TC_PLAIN || MODE == TC_FQT || MODE == TC_FQC || MODE == TC_FQX) { kb0 = 0; kbn = p.nkb; }
        else if (MODE == TC_TRANS) { kb0 = 0; kbn = p.groups * p.nblocks; }
        else {
            const int64_t sp = unit / (p.tiles_m * p.tiles_n);
            const int64_t ta = sp * p.split_len, tb = min(p.tau_hi, ta + p.split_len);
            const int64_t a = ta + seg * FLUSH_T, b = min(tb, a + FLUSH_T);
            kb0 = a / BK;
            kbn = b > a ? (b - a + BK - 1) / BK : 0;
        }
    };

    // register rebalancing (per warpgroup): the producer/MMA warpgroup gives registers to the
    // epilogue warpgroups, which keep 128 fp32 accumulators per thread in registers
    if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (warp == 0) {
        // ================================================================ TMA producer
        if (lane == 0) {
            int s = 0; uint32_t ph = 0;
            int kcount = 0;      // CORR lock-step: k-blocks issued by this CTA so far
            for (int64_t unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
                int64_t mt = 0, nt = 0;
                if (MODE == TC_CONV) { nt = unit % p.tiles_n; mt = unit / p.tiles_n; }          // nt: n tile, mt: t tile
                if (MODE == TC_PLAIN) { nt = unit % p.tiles_n; mt = unit / p.tiles_n; }         // nt: column tile, mt: row tile
                int64_t fq_m = 0;                                                                        // FQT / FQC: 128-row tile of the frequency
                if (MODE == TC_FQT || MODE == TC_FQC) { fq_m = unit % p.mtiles; const int64_t r = unit / p.mtiles; nt = r % p.tiles_n; mt = r / p.tiles_n; }   // nt: column tile, mt: frequency
                if (MODE == TC_CORR) { const int64_t r = unit % (p.tiles_m * p.tiles_n); mt = r % p.tiles_m; nt = r / p.tiles_m; }   // j tiles fastest: the CTAs that run together share the X tile
                const int64_t nseg = n_segments(unit);
                for (int64_t seg = 0; seg < nseg; ++seg) {
                    int64_t kb0, kbn;
                    segment_kb(unit, seg, kb0, kbn);
                    for (int64_t kb = kb0; kb < kb0 + kbn; ++kb) {
                        if (MODE == TC_CORR && p.lockstep != nullptr) {
                            // The ~50 CTAs that share an X tile must stay close in time or the tile falls out of L2 and is
                            // re-read from HBM (measured: 19x the algorithmic traffic without this).  Every 64 k-blocks each
                            // CTA publishes its progress and waits while it is more than lockstep_window ahead of the slowest.
                            if ((kcount & 63) == 0) {
                                atomicExch(p.lockstep + blockIdx.x, kcount);
                                for (;;) {
                                    int mn = 0x7fffffff;
                                    for (unsigned i = 0; i < gridDim.x; ++i) mn = min(mn, __ldcg(p.lockstep + i));
                                    if (kcount <= mn + p.lockstep_window) break;
                                    __nanosleep(200);
                                }
                            }
                            ++kcount;
                        }
                        mbar_wait(&empty_bar[s], ph ^ 1);
                        unsigned char *st = smem + (size_t)s * STAGE_BYTES;
                        mbar_expect_tx(&full_bar[s], STAGE_BYTES);
                        if (MODE == TC_CONV) {
                            const int32_t j0 = (int32_t)(kb * BK);
                            tma_load_2d(st, &mapA_hi, &full_bar[s], j0, (int32_t)(nt * BM));
                            tma_load_2d(st + A_PLANE, &mapA_lo, &full_bar[s], j0, (int32_t)(nt * BM));
                            tma_load_2d(st + 2 * A_PLANE, &mapB_hi, &full_bar[s], j0, (int32_t)(mt * BN));
                            tma_load_2d(st + 2 * A_PLANE + B_PLANE, &mapB_lo, &full_bar[s], j0, (int32_t)(mt * BN));
                        } else if (MODE == TC_PLAIN) {
                            const int32_t k0 = (int32_t)(kb * BK);
                            tma_load_2d(st, &mapA_hi, &full_bar[s], k0, (int32_t)(mt * BM));
                            tma_load_2d(st + A_PLANE, &mapA_lo, &full_bar[s], k0, (int32_t)(mt * BM));
                            tma_load_2d(st + 2 * A_PLANE, &mapB_hi, &full_bar[s], k0, (int32_t)(nt * BN));
                            tma_load_2d(st + 2 * A_PLANE + B_PLANE, &mapB_lo, &full_bar[s], k0, (int32_t)(nt * BN));
                        } else if (MODE == TC_TRANS) {
                            const int64_t nb = kb / p.groups, g = kb % p.groups;   // n-block outer, lag group inner: the X sub-window stays in L2
                            const int32_t c0 = (int32_t)(nb * BK);
                            const int32_t rowA = (int32_t)(g * p.G * p.Kp), rowB = (int32_t)(unit * p.own + g * p.G);   // G*Kp <= 128 rows per lag group
                            tma_load_2d(st, &mapA_hi, &full_bar[s], c0, rowA);
                            tma_load_2d(st + A_PLANE, &mapA_lo, &full_bar[s], c0, rowA);
                            tma_load_2d(st + 2 * A_PLANE, &mapB_hi, &full_bar[s], c0, rowB);
                            tma_load_2d(st + 2 * A_PLANE + B_PLANE, &mapB_lo, &full_bar[s], c0, rowB);
                        } else if (MODE == TC_FQT) {
                            const int32_t k0 = (int32_t)(kb * BK);
                            const int32_t rowB = (int32_t)(mt * p.fq_rows + nt * BN);
                            const int32_t rowA = (int32_t)(mt * p.MR + fq_m * BM);
                            tma_load_2d(st, &mapA_hi, &full_bar[s], k0, rowA);
                            tma_load_2d(st + A_PLANE, &mapA_lo, &full_bar[s], k0, rowA);
                            tma_load_2d(st + 2 * A_PLANE, &mapB_hi, &full_bar[s], k0, rowB);
                            tma_load_2d(st + 2 * A_PLANE + B_PLANE, &mapB_lo, &full_bar[s], k0, rowB);
                        } else if (MODE == TC_FQX) {
                            // unit = ((f*2 + co) * tiles_m + n tile) * tiles_n + block tile
                            const int64_t bt = unit % p.tiles_n, r1 = unit / p.tiles_n, ntile = r1 % p.tiles_m, fc = r1 / p.tiles_m;
                            const int32_t trow = (int32_t)(fc * p.MR + kb * BK);                     // Awm rows ((f*2+co)*MR + (c,k))
                            const int32_t rowB = (int32_t)((fc >> 1) * p.fq_rows + p.b_off + bt * BN);
                            tma_load_3d(st, &mapA_hi, &full_bar[s], 0, trow, (int32_t)(ntile * 2));
                            tma_load_3d(st + A_PLANE, &mapA_lo, &full_bar[s], 0, trow, (int32_t)(ntile * 2));
                            tma_load_2d(st + 2 * A_PLANE, &mapB_hi, &full_bar[s], (int32_t)(kb * BK), rowB);
                            tma_load_2d(st + 2 * A_PLANE + B_PLANE, &mapB_lo, &full_bar[s], (int32_t)(kb * BK), rowB);
                        } else if (MODE == TC_FQC) {
                            const int32_t trow = (int32_t)(mt * p.fq_rows + kb * BK);
                            tma_load_3d(st, &mapA_hi, &full_bar[s], 0, trow, (int32_t)(fq_m * 2));
                            tma_load_3d(st + A_PLANE, &mapA_lo, &full_bar[s], 0, trow, (int32_t)(fq_m * 2));
                            tma_load_3d(st + 2 * A_PLANE, &mapB_hi, &full_bar[s], 0, trow, (int32_t)(nt * 4));
                            tma_load_3d(st + 2 * A_PLANE + B_PLANE, &mapB_lo, &full_bar[s], 0, trow, (int32_t)(nt * 4));
                        } else {
                            // MN-major operands come through 3-D maps (64 contiguous elements, t rows, 64-element
                            // groups), so one TMA per plane fills all the 4 KB swizzle atoms of the tile
                            const int32_t trow = (int32_t)(kb * BK);
                            tma_load_3d(st, &mapA_hi, &full_bar[s], 0, trow, (int32_t)(mt * 2));
                            tma_load_3d(st + A_PLANE, &mapA_lo, &full_bar[s], 0, trow, (int32_t)(mt * 2));
                            tma_load_3d(st + 2 * A_PLANE, &mapB_hi, &full_bar[s], 0, trow, (int32_t)(nt * 4));
                            tma_load_3d(st + 2 * A_PLANE + B_PLANE, &mapB_lo, &full_bar[s], 0, trow, (int32_t)(nt * 4));
                        }
                        if (++s == STAGES) { s = 0; ph ^= 1; }
                    }
                }
            }
            if (MODE == TC_CORR && p.lockstep != nullptr) atomicExch(p.lockstep + blockIdx.x, 0x7fffffff);   // finished: never the slowest
        }
    } else if (warp == 1) {
        // ================================================================ MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = (MODE == TC_CORR || MODE == TC_FQC) ? make_idesc(1, 1) : (MODE == TC_FQX) ? make_idesc(1, 0) : make_idesc(0, 0);
            int s = 0; uint32_t ph = 0;
            int64_t q = 0;   // promotion-chunk counter (TMEM double buffer)
            for (int64_t unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
                const int64_t nseg = n_segments(unit);
                for (int64_t seg = 0; seg < nseg; ++seg) {
                    int64_t kb0, kbn;
                    segment_kb(unit, seg, kb0, kbn);
                    for (int64_t c0 = 0; c0 < kbn; c0 += PROMO, ++q) {
                        const int64_t cn = min((int64_t)PROMO, kbn - c0);
                        const int acc = (int)(q & 1);
                        mbar_wait(&tmem_empty[acc], (uint32_t)((q >> 1) & 1) ^ 1);
                        tc_fence_after();
                        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                        uint32_t accumulate = 0;
                        for (int64_t kb = 0; kb < cn; ++kb) {
                            mbar_wait(&full_bar[s], ph);
                            tc_fence_after();
                            const uint32_t sa = smem_u32(smem + (size_t)s * STAGE_BYTES);
                            const uint32_t a_hi = sa, a_lo = sa + A_PLANE, b_hi = sa + 2 * A_PLANE, b_lo = sa + 2 * A_PLANE + B_PLANE;
#pragma unroll
                            for (int ks = 0; ks < BK / 16; ++ks) {
                                uint64_t dah, dal, dbh, dbl;
                                if (MODE == TC_CORR || MODE == TC_FQC) {
                                    // MN-major SW128: LBO = 4096 B between 64-element MN groups, SBO = 1024 B between 8-row K groups
                                    const uint32_t off = (uint32_t)ks * 2048u;
                                    dah = make_desc(a_hi + off, 4096, 1024, 2); dal = make_desc(a_lo + off, 4096, 1024, 2);
                                    dbh = make_desc(b_hi + off, 4096, 1024, 2); dbl = make_desc(b_lo + off, 4096, 1024, 2);
                                } else if (MODE == TC_FQX) {
                                    // A MN-major SW128 (as above), B K-major SW64 (as below)
                                    const uint32_t offa = (uint32_t)ks * 2048u, offb = (uint32_t)ks * 32u;
                                    dah = make_desc(a_hi + offa, 4096, 1024, 2); dal = make_desc(a_lo + offa, 4096, 1024, 2);
                                    dbh = make_desc(b_hi + offb, 16, 512, 4); dbl = make_desc(b_lo + offb, 16, 512, 4);
                                } else {
                                    // K-major SW64: 64-byte rows, SBO = 512 B between 8-row groups, +32 B per 16-element K step
                                    const uint32_t off = (uint32_t)ks * 32u;
                                    dah = make_desc(a_hi + off, 16, 512, 4); dal = make_desc(a_lo + off, 16, 512, 4);
                                    dbh = make_desc(b_hi + off, 16, 512, 4); dbl = make_desc(b_lo + off, 16, 512, 4);
                                }
                                tc_mma(d_tmem, dal, dbh, idesc, accumulate);   // lo*hi
                                tc_mma(d_tmem, dah, dbl, idesc, 1u);           // hi*lo
                                tc_mma(d_tmem, dah, dbh, idesc, 1u);           // hi*hi
                                accumulate = 1u;
                            }
                            tc_commit(&empty_bar[s]);                          // frees the stage when these MMAs retire
                            if (++s == STAGES) { s = 0; ph ^= 1; }
                        }
                        tc_commit(&tmem_full[acc]);                            // partial ready for promotion
                    }
                }
            }
        }
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
        // ================================================================ epilogue / promotion (warps 4..11)
        const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
        const int half = (warp - 4) >> 2;             // which 128 columns of the tile this warp owns
        const int row = quarter * 32 + lane;          // TMEM lane = tile row
        const int col0 = half * (BN / 2);
        int64_t q = 0;
        float racc[BN / 2];
        for (int64_t unit = blockIdx.x; unit < p.units; unit += gridDim.x) {
            int64_t mt = 0, nt = 0, sp = 0;
            int64_t fq_m = 0;
            if (MODE == TC_CONV || MODE == TC_PLAIN) { nt = unit % p.tiles_n; mt = unit / p.tiles_n; }
            if (MODE == TC_FQT || MODE == TC_FQC) { fq_m = unit % p.mtiles; const int64_t r = unit / p.mtiles; nt = r % p.tiles_n; mt = r / p.tiles_n; }
            if (MODE == TC_CORR) { sp = unit / (p.tiles_m * p.tiles_n); const int64_t r = unit % (p.tiles_m * p.tiles_n); mt = r % p.tiles_m; nt = r / p.tiles_m; }
            const int64_t nseg = n_segments(unit);
            for (int64_t seg = 0; seg < nseg; ++seg) {
                int64_t kb0, kbn;
                segment_kb(unit, seg, kb0, kbn);
#pragma unroll
                for (int c = 0; c < BN / 2; ++c) racc[c] = 0.f;
                // ---- promotion: racc += TMEM partial, every PROMO k-blocks
                for (int64_t c0 = 0; c0 < kbn; c0 += PROMO, ++q) {
                    const int acc = (int)(q & 1);
                    mbar_wait(&tmem_full[acc], (uint32_t)((q >> 1) & 1));
                    tc_fence_after();
                    const uint32_t taddr0 = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + col0);
#pragma unroll
                    for (int cc = 0; cc < BN / 2; cc += 16) {
                        uint32_t v[16];
                        tmem_ld16(taddr0 + cc, v);
#pragma unroll
                        for (int c = 0; c < 16; ++c) racc[cc + c] += __uint_as_float(v[c]);
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tmem_empty[acc]);
                }
                // ---- write-out of the segment from registers
                if (MODE == TC_CONV) {
                    const int64_t n = nt * BM + row, t0 = mt * BN + col0;
                    float part = 0.f;
                    double sq = 0.0;
#pragma unroll
                    for (int c = 0; c < BN / 2; ++c) {
                        const int64_t t = t0 + c;
                        if (n < p.N && t < p.Tl) {
                            const float r = racc[c] - __ldg(p.X + t * p.N + n);
                            part = fmaf(r, r, part);
                        }
                        if ((c & 31) == 31) { sq += (double)part; part = 0.f; }
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
                    if (lane == 0) p.partial[unit * EPI_WARPS + (warp - 4)] = sq;
                } else if (MODE == TC_TRANS) {
                    const int i = row / p.Kp, k = row % p.Kp;       // lag index inside the group, component
                    const int64_t t0 = unit * p.own;
                    // one pass per lag of the group, ordered by a named barrier over the epilogue warps, so the
                    // additions into numH happen in a fixed order (deterministic)
                    for (int pass = 0; pass < p.G; ++pass) {
                        if (i == pass && k < p.K) {      // rows >= G*Kp (i >= G) belong to the next lag group: ignored
#pragma unroll
                            for (int c = 0; c < BN / 2; ++c) {
                                const int64_t cc = col0 + c - i;            // owned column index
                                const int64_t t = t0 + cc;
                                if (cc >= 0 && cc < p.own && t < p.Tl) {
                                    float *o = p.out + t * p.K + k;
                                    *o = (pass == 0) ? racc[c] : (*o + racc[c]);
                                }
                            }
                        }
                        if (p.G > 1) asm volatile("bar.sync 1, 256;" ::: "memory");
                    }
                } else if (MODE == TC_FQX) {
                    // Yf[f][b][co][n] (blocks numbered inside the chunk): lanes hold consecutive units n -> coalesced rows
                    const int64_t bt = unit % p.tiles_n, r1 = unit / p.tiles_n, ntile = r1 % p.tiles_m, fc = r1 / p.tiles_m;
                    const int64_t b0 = bt * BN + col0, n = ntile * BM + row;
                    float *o = p.out + (((fc >> 1) * p.nbc + b0) * 2 + (fc & 1)) * p.N + n;
                    if (n < p.N) {
#pragma unroll
                        for (int c = 0; c < BN / 2; ++c)
                            if (b0 + c < p.nbc) o[(int64_t)c * 2 * p.N] = racc[c];
                    }
                } else if (MODE == TC_FQT) {
                    // Of[f][b][m]: lanes hold consecutive rows m, so every column is one coalesced 128-byte store
                    const int64_t b0 = nt * BN + col0;
                    float *o = p.out + (mt * p.fq_rows + b0) * p.MR + fq_m * BM + row;
#pragma unroll
                    for (int c = 0; c < BN / 2; ++c)
                        if (b0 + c < p.fq_rows) o[(int64_t)c * p.MR] = racc[c];
                } else if (MODE == TC_PLAIN || MODE == TC_FQC) {
                    // fp32 store through the per-warp staging tile (coalesced 64-byte row segments);
                    // FQC: one 128-row output matrix per frequency, Df[f][m][n]
                    float(*stg)[17] = stage_s[warp - 4];
                    const int64_t mrow0 = (MODE == TC_FQC) ? fq_m * BM : mt * BM;
                    float *outp = p.out + ((MODE == TC_FQC) ? mt * p.MR * p.ldo : 0);
#pragma unroll
                    for (int cc = 0; cc < BN / 2; cc += 16) {
#pragma unroll
                        for (int c = 0; c < 16; ++c) stg[lane][c] = racc[cc + c];
                        __syncwarp();
#pragma unroll 1
                        for (int it = 0; it < 16; ++it) {
                            const int r = it * 2 + (lane >> 4), c = lane & 15;
                            const int64_t m = mrow0 + quarter * 32 + r;
                            const int64_t n = nt * BN + col0 + cc + c;
                            if (m < p.Mrows && n < p.Ncols) outp[m * p.ldo + n] = stg[r][c];
                        }
                        __syncwarp();
                    }
                } else {
                    // fp64 flush through a per-warp shared staging tile: registers -> smem with static
                    // indices, then a compact loop does the coalesced double read-modify-write
                    float(*stg)[17] = stage_s[warp - 4];
                    double *pbase = p.part + (size_t)sp * (size_t)(p.L * p.K * p.N);
#pragma unroll
                    for (int cc = 0; cc < BN / 2; cc += 16) {
#pragma unroll
                        for (int c = 0; c < 16; ++c) stg[lane][c] = racc[cc + c];
                        __syncwarp();
                        // 16 (row, column) pairs per lane, 8 at a time with all loads in flight before the adds
                        // (the partial buffer is not cache resident: a dependent load per element costs ~1 us each)
#pragma unroll 1
                        for (int it0 = 0; it0 < 16; it0 += 8) {
                            double *dp[8];
                            double old[8];
#pragma unroll
                            for (int u = 0; u < 8; ++u) {
                                const int r = (it0 + u) * 2 + (lane >> 4), c = lane & 15;
                                const int64_t j = mt * BM + quarter * 32 + r;
                                const int64_t lp = j / p.Kp, k = j - lp * p.Kp;
                                const int64_t n = nt * BN + col0 + cc + c;
                                dp[u] = (lp < p.L && k < p.K && n < p.N) ? pbase + ((p.L - 1 - lp) * p.K + k) * p.N + n : nullptr;
                            }
                            if (seg != 0) {
#pragma unroll
                                for (int u = 0; u < 8; ++u) old[u] = dp[u] ? __ldcg(dp[u]) : 0.0;
                            }
#pragma unroll
                            for (int u = 0; u < 8; ++u) {
                                const int r = (it0 + u) * 2 + (lane >> 4), c = lane & 15;
                                const double x = (double)stg[r][c];
                                if (dp[u]) *dp[u] = (seg == 0) ? x : (old[u] + x);
                            }
                        }
                        __syncwarp();
                    }
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// ---------------------------------------------------------------------------------- operand splitting
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16 &hi, __nv_bfloat16 &lo) {
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// X[t][N] fp32 -> hi/lo planes, same layout (elementwise)
__global__ void split_plain_kernel(const float *__restrict__ x, __nv_bfloat16 *__restrict__ hi,
                                   __nv_bfloat16 *__restrict__ lo, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    __nv_bfloat16 h, l;
    split_bf16(x[i], h, l);
    hi[i] = h; lo[i] = l;
}

// H[t][K] fp32 (local columns [-(L-1), Tl+L-1)) -> Hw[(t + L-1)][Kp] hi/lo with zero padding components;
// masked != 0 additionally zeroes the halo columns (owned-only copy for the W-side correlation).
__global__ void split_H_kernel(const float *__restrict__ Hbuf, __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo,
                               int64_t rows, int64_t K, int Kp, int64_t own_lo, int64_t own_hi, int masked) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * Kp) return;
    const int64_t r = i / Kp;
    const int k = (int)(i % Kp);
    float v = 0.f;
    if (k < K && (!masked || (r >= own_lo && r < own_hi))) v = Hbuf[r * K + k];
    __nv_bfloat16 h, l;
    split_bf16(v, h, l);
    hi[i] = h; lo[i] = l;
}

// Wi[(l*K+k)][N] fp32 ->  Wc[n][j], j = (L-1-l)*Kp + k  (row length KLp, zero padded)   [conv A operand]
//                    and  Wu[(l*Kp+k)][N]               (rows_u rows, zero padded)      [transconv A operand]
// One CTA per (32 units n, 32 components k, lag l): Wu is written as read (coalesced along n), Wc goes through a
// shared-memory transpose so that its rows are written 32 components (64 bytes) at a time.
// grid (ceil(N/32), ceil(Kp/32), L), block (32, 8).
__global__ void split_W_kernel(const float *__restrict__ Wi, __nv_bfloat16 *__restrict__ wc_hi, __nv_bfloat16 *__restrict__ wc_lo,
                               __nv_bfloat16 *__restrict__ wu_hi, __nv_bfloat16 *__restrict__ wu_lo, int64_t N, int64_t K,
                               int64_t L, int Kp, int64_t KLp) {
    __shared__ float tile[32][33];
    const int64_t l = blockIdx.z;
    const int64_t n0 = (int64_t)blockIdx.x * 32, k0 = (int64_t)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int64_t k = k0 + r, n = n0 + threadIdx.x;
        float v = 0.f;
        if (k < Kp && n < N) {
            if (k < K) v = Wi[(l * K + k) * N + n];
            __nv_bfloat16 h, lo_;
            split_bf16(v, h, lo_);
            const int64_t idx = (l * Kp + k) * N + n;
            wu_hi[idx] = h; wu_lo[idx] = lo_;
        }
        tile[r][threadIdx.x] = v;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int64_t n = n0 + r, k = k0 + threadIdx.x;
        if (n < N && k < Kp) {
            __nv_bfloat16 h, lo_;
            split_bf16(tile[threadIdx.x][r], h, lo_);
            const int64_t j = (L - 1 - l) * Kp + k;
            wc_hi[n * KLp + j] = h; wc_lo[n * KLp + j] = lo_;
        }
    }
}

// G = Htilde Htilde' (see build_G_kernel) written as bf16 hi/lo planes Gc[j][jj]: rows j = l*K + k (Wi order),
// columns jj = (L-1-l')*Kp + k' (the K-dim order of Wc), row length KLp, zero padded.      [G*W A operand]
// Written along the block diagonals (see s2_dot_G_diag_kernel): thread (d, k, k') walks (l, l') with the Toeplitz part
// constant and the tail updated by one product per step.  The zero padding of Gc is never touched.
__global__ void build_G_split_diag_kernel(const double *__restrict__ Rg, const double *__restrict__ Ht, __nv_bfloat16 *__restrict__ hi,
                                          __nv_bfloat16 *__restrict__ lo, int64_t K, int64_t L, int Kp, int64_t KLp) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (2 * L - 1) * K * K) return;
    const int64_t kp = e % K, k = (e / K) % K, d = e / (K * K) - (L - 1);
    const double r = (d >= 0) ? Rg[(d * K + k) * K + kp] : Rg[((-d) * K + kp) * K + k];
    const int64_t steps = L - (d >= 0 ? d : -d);
    int64_t l = d >= 0 ? d : 0, lp = d >= 0 ? 0 : -d;
    double tail = 0.0;
    for (int64_t s_ = 0; s_ < steps; ++s_, ++l, ++lp) {
        const int64_t idx = (l * K + k) * KLp + (L - 1 - lp) * Kp + kp;
        __nv_bfloat16 h, l_;
        split_bf16((float)(r - tail), h, l_);
        hi[idx] = h; lo[idx] = l_;
        if (s_ + 1 < steps) tail += Ht[(L - 2 - l) * K + k] * Ht[(L - 2 - lp) * K + kp];
    }
}

// Cf[(d')][k][k'] fp32 ((2L-1) x K x K) -> Cc[(d'*Kp + k)][Kp] hi/lo (rows_c rows, zero padded)  [denomH A operand]
__global__ void split_C_kernel(const float *__restrict__ Cf, __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo,
                               int64_t K, int64_t D, int Kp, int64_t rows_c) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows_c * Kp) return;
    const int kp = (int)(idx % Kp);
    const int64_t r = idx / Kp;
    const int64_t d = r / Kp;
    const int k = (int)(r % Kp);
    float v = 0.f;
    if (d < D && k < K && kp < K) v = Cf[(d * K + k) * K + kp];
    __nv_bfloat16 h, l;
    split_bf16(v, h, l);
    hi[idx] = h; lo[idx] = l;
}

}  // namespace tc
}  // namespace cmf
