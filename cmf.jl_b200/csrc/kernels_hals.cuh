// HALS H sweep (src/algs/hals.jl:121-154), second generation: one cooperative launch organised in ROUNDS with a grid-wide
// barrier between them (fp32, L <= 32).  Same arithmetic order as the reference's k-outer / t-inner sweep per component;
// the corrections that earlier components send to later ones are summed in a fixed order (deterministic).
//
// Recurrence form (oracle/restructured.py, SURVEY.md appendix B): with Q = transconv(W, conv(W,H) - X) at the start of the
// sweep, C[k',k,dd] the lag table and D = Delta H,
//     qeff[k,t]  = Q[k,t] + sum_{k'<k} sum_{|dd|<L} D[k',t-dd] C_w[k',k,dd]          ("pull", needs all earlier components)
//     h'[k,t]    = max((h c0 - qeff - pend(t) - l1) / (c0 + eps + l2), 0),   pend(t+s) += D[k,t] C[k,k,s], s = 1..L-1
//
// Why rounds.  The first-generation kernel gave one CTA per component and let each CTA stage, pull and run its recurrence
// one after the other; a cell took as long as the LAST component's pull (k-1 predecessors) and its one-lane recurrence.
// Here the three kinds of work are different CTAs that all run in every round:
//   * recurrence warps: one warp per 32 components, LANE = COMPONENT.  Every lane runs the sequential recurrence of its own
//     component over one chunk of CW columns per round; the pending window and the lag table of the component live in
//     registers, so a column costs ~L issue slots for 32 components at once (the old kernel spent the same slots on one).
//   * block items (g, g'), g' < g: the pull of the 8 targets of group g from the 8 sources of group g' for one chunk: an
//     8 x 8 block of component pairs on one staged window of Delta H, register tile 8 columns x 4 targets per thread.
//   * diagonal items (g): for every target of group g, the pull from the earlier components of its own group, the sum of
//     the block partials in the fixed order g' = 0, 1, ..., and the hand-over to the recurrence: a = (h c0 - qeff - l1) inv.
// Component k works on chunk c in round c + 4k + 1 (stagger of 4 chunks): the block items of (group g, chunk c) run in round
// c + 32g - 1 (their last source, component 8g-1, finished chunk c+1 in round c + 32g - 2), the diagonal item of (k, c) in
// round c + 4k (component k-1 finished chunk c+1 in round c + 4k - 2), the recurrence of (k, c) in round c + 4k + 1, and the
// truncated last L-1 columns of component k (tables C_w, w < L) in round nC + 4k + 1 by one thread.  Every read in a round is of
// data written in an EARLIER round, so a round is a bulk-synchronous step and one barrier per round is all the ordering
// there is; tests/test_oracle.py replays this schedule on the CPU and checks every read against the write rounds.
// For K = 128 that is 120 + 16 + 4 = 140 CTAs on 148 SMs, each with the same work in every round.
//
// Working layout: component-major (H_cm[k][t], AD_cm[k][t]) so that a lane / a staged source reads contiguous memory;
// the [t][K] arrays of the rest of the library are transposed on the way in (diagonal items) and out (hals2_finish_kernel).
#pragma once

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cmf {
namespace hals2 {

namespace cg = cooperative_groups;

constexpr int CW = 1024;        // columns per chunk
constexpr int NT = 256;         // threads of an item CTA
constexpr int GS = 8;           // components per group
constexpr int STAG = 4;         // chunks between consecutive components
constexpr int RING = 32;        // chunks a block partial stays alive: written in round c+32g-1, read no later than c+32g+28
constexpr int LMAX = 32;
static_assert(CW == 4 * NT, "the hand-over loop covers a chunk with one float4 per thread");
constexpr int KMAX = 128;        // components (the tail paths walk them in 4 passes of 32 lanes)
constexpr int WIN = CW + 2 * (LMAX - 1);      // staged window of Delta H (columns t0-(L-1) .. t0+CW+(L-1)-1), sized for L = 32
constexpr int QP = ((WIN + 7) >> 3) | 1;      // slots per plane of the 8-plane layout (odd: conflict-free)
constexpr int WINQ = 8 * QP;                  // words per staged source

struct Args {
    const float *Cf;      // [(dd+L-1)][k'][k]  interior lag table
    const float *Ct;      // [w-1][dd+L-1][k][k'] truncated tables (w = 1..L-1), nullptr when L == 1
    const float *S2;      // W W' (truncated self tables of the tail job)
    int64_t Ks, ld;       // addressing of S2
    float *H_cm;          // cells (see cell_at): H, old value until the recurrence overwrites it with the new one
    float *AD_cm;         // cells: Q (from hals2_prepare_kernel), then a (hand-over to the recurrence), then Delta H
    float *part;          // [RING][G][K][CW] block partials, indexed by ring slot and source group
    const float *coef;    // [K][64] self lag table of every component scaled by 1/(c0+eps+l2): 16 even-aligned pairs (cs[2m], cs[2m+1]), then
                          // 16 odd-aligned pairs (cs[2m+1], cs[2m+2]) (hals2_coef_kernel); cs[0] = cs[32] = 0
    int64_t K, L, T, nC;
    float l1, l2;
    int G;                // groups of 8 components
    int n_block_items, n_diag_items, n_rec;
    unsigned *barrier;    // grid barrier counter (zero before the launch)
};

__device__ __forceinline__ float ldcg(const float *p) { return __ldcg(p); }

// Working layout of H and of the Q / a / Delta H array: CELLS of CW columns of one component, ordered by the round that
// works on them: cell (k, c) lives at slice d = c + STAG*k, position k inside the slice.  What one round touches is then
// contiguous (the 32 cells of a recurrence warp are 128 KB, all the cells of a round 512 KB at K = 128), where a plain
// component-major array would spread a warp's lanes over rows 4*Tp bytes apart -- one 2 MB page per lane, all in the same
// TLB set (measured: every load of the kernel then took ~4000 cycles).
__host__ __device__ __forceinline__ int64_t cell_at(int64_t k, int64_t t, int64_t K) {
    const int64_t c = t / CW;
    return ((c + (int64_t)STAG * k) * K + k) * CW + (t - c * CW);
}
__host__ __device__ __forceinline__ int64_t cells_elems(int64_t K, int64_t nC) { return (nC + (int64_t)STAG * (K - 1)) * K * CW; }
__device__ __forceinline__ int64_t part_at(int64_t slot, int64_t gp, int64_t k, int64_t K, int G) { return ((slot * G + gp) * K + k) * CW; }

// FP32 on sm_100 runs at full rate only through the packed FFMA2 (two fp32 FMAs per instruction on a 64-bit register
// pair; a scalar FFMA occupies the same issue slots).  The pull therefore processes the staged sources two at a time: the
// window holds (source 2p, source 2p+1) pairs, the table (C[2p], C[2p+1]) pairs, and every accumulator is a pair
// (contribution of the even source, contribution of the odd source) that is added up at the end.
//
// Staging of Delta H of `nsrc` sources (components k0 .. k0+nsrc-1) over the window of chunk c, columns
// [c*CW - (L-1), (c+1)*CW + (L-1)), into the 8-plane pair layout (an odd last source is paired with zeros; columns outside
// [0, Tint) are zero: sources in the truncated tail go through the tail tables instead).  Split in two halves so that the
// loads (128-bit, from L2 / HBM: written by other SMs in earlier rounds, > 1000 cycles away) can be in flight while other
// work runs: stage_load fills registers, stage_store scatters them into shared memory.  Address arithmetic is per 4 columns.
constexpr int SCH = (WIN + 3 + 3) / 4;                   // aligned 4-column pieces covering a window
constexpr int SIT = (SCH + NT - 1) / NT;                 // pieces per thread and source
struct StageRegs { float4 va[GS / 2][SIT], vb[GS / 2][SIT]; };

__device__ __forceinline__ void stage_load(StageRegs &r, const Args &a, int64_t k0, int nsrc, int64_t c, int64_t Tint) {
    const int Lm = (int)a.L - 1, WW = CW + 2 * Lm;
    const int64_t tbase = c * CW - Lm, ta0 = tbase - (((tbase % 4) + 4) % 4);     // first aligned piece
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int p = 0; p < GS / 2; ++p) {
#pragma unroll
        for (int it = 0; it < SIT; ++it) {
            r.va[p][it] = z4; r.vb[p][it] = z4;
            const int64_t t = ta0 + 4 * (int64_t)(threadIdx.x + it * NT);
            if (2 * p < nsrc && t < tbase + WW && t >= 0 && t < Tint) {
                const int64_t cc = t >> 10, col = t & (CW - 1), ka = k0 + 2 * p;
                static_assert(CW == 1024, "shift / mask above");
                r.va[p][it] = __ldcg(reinterpret_cast<const float4 *>(a.AD_cm + ((cc + (int64_t)STAG * ka) * a.K + ka) * CW + col));
                if (2 * p + 1 < nsrc)
                    r.vb[p][it] = __ldcg(reinterpret_cast<const float4 *>(a.AD_cm + ((cc + (int64_t)STAG * (ka + 1)) * a.K + ka + 1) * CW + col));
            }
        }
    }
}

__device__ __forceinline__ void stage_store(float2 *Dwin2, const StageRegs &r, const Args &a, int nsrc, int64_t c, int64_t Tint) {
    const int Lm = (int)a.L - 1, WW = CW + 2 * Lm;
    const int64_t tbase = c * CW - Lm, ta0 = tbase - (((tbase % 4) + 4) % 4);
#pragma unroll
    for (int p = 0; p < GS / 2; ++p) {
        if (2 * p >= nsrc) break;
        float2 *dst = Dwin2 + p * WINQ;
#pragma unroll
        for (int it = 0; it < SIT; ++it) {
            const int64_t t = ta0 + 4 * (int64_t)(threadIdx.x + it * NT);
            const float xa[4] = {r.va[p][it].x, r.va[p][it].y, r.va[p][it].z, r.va[p][it].w};
            const float xb[4] = {r.vb[p][it].x, r.vb[p][it].y, r.vb[p][it].z, r.vb[p][it].w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int i = (int)(t + e - tbase);
                if (i >= 0 && i < WW) {
                    const bool ok = t + e >= 0 && t + e < Tint;      // the piece may straddle Tint: zero beyond it
                    dst[(i & 7) * QP + (i >> 3)] = make_float2(ok ? xa[e] : 0.f, ok ? xb[e] : 0.f);
                }
            }
        }
    }
}

// acc[r][q] (pair: even / odd source) += D[src][t'+(L-1)-j] * tab[src][j][q] over `npair` staged source pairs and all lags,
// t' = 8*cgp + r, q = 0..NTG-1.  tab2: [npair][NLP][8] pairs (lag rows padded with zeros to NLP = a multiple of 8), tq0 = first
// target column of the table.
template <int NTG>
__device__ __forceinline__ void pull_tile(float2 (&acc)[8][NTG], const float2 *Dwin2, const float2 *tab2, int npair, int L, int cgp, int tq0) {
    const int nl = 2 * L - 1, NLP = (nl + 7) & ~7;
    const int ib = 8 * cgp + 2 * (L - 1);
    for (int sp = 0; sp < npair; ++sp) {
        const float2 *dw = Dwin2 + sp * WINQ;
        const float2 *tb = tab2 + (size_t)sp * NLP * 8 + tq0;
        float2 w[8];
        w[0] = make_float2(0.f, 0.f);
#pragma unroll
        for (int o = 1; o < 8; ++o) { const int i = ib + o; w[o] = dw[(i & 7) * QP + (i >> 3)]; }
        for (int j0 = 0; j0 < nl; j0 += 8) {
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const int j = j0 + jj;
                const int in = max(ib - j, 0);              // window index entering at this step (column r = 0); padded lags multiply by zero
                w[(8 - jj) & 7] = dw[(in & 7) * QP + (in >> 3)];
                float2 cq[NTG];
#pragma unroll
                for (int q = 0; q < NTG; ++q) cq[q] = tb[j * 8 + q];
#pragma unroll
                for (int r = 0; r < 8; ++r)
#pragma unroll
                    for (int q = 0; q < NTG; ++q) acc[r][q] = __ffma2_rn(w[(r - jj + 8) & 7], cq[q], acc[r][q]);
            }
        }
    }
}

// table slice as source pairs: tab2[p][j][q] = (C[k0s+2p, k0t+q, j-(L-1)], C[k0s+2p+1, k0t+q, j-(L-1)]), zero where the pair is
// not a (source < target) pair or out of range
__device__ __forceinline__ void load_table(float2 *tab2, const Args &a, int64_t k0s, int64_t k0t, bool diagonal) {
    const int L = (int)a.L, nl = 2 * L - 1, NLP = (nl + 7) & ~7;
    float *tab = reinterpret_cast<float *>(tab2);
    for (int idx = threadIdx.x; idx < GS * NLP * 8; idx += NT) {
        const int q = idx & 7, j = (idx >> 3) % NLP, s = idx / (8 * NLP);
        const int64_t ks = k0s + s, kt = k0t + q;
        float v = 0.f;
        if (j < nl && ks < a.K && kt < a.K && (!diagonal || ks < kt)) v = a.Cf[((int64_t)j * a.K + ks) * a.K + kt];
        tab[2 * (((s >> 1) * NLP + j) * 8 + q) + (s & 1)] = v;
    }
}

// 64-bit register pairs for the recurrence: the coefficient pairs and the pending window stay packed for the whole kernel
// (as float2 the compiler splits them into scalars and rebuilds the aligned pairs FFMA2 needs with two moves per use)
typedef unsigned long long u64;
__device__ __forceinline__ u64 pack2(float x, float y) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y)); return r; }
__device__ __forceinline__ float lo_of(u64 v) { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v)); return x; }
__device__ __forceinline__ float hi_of(u64 v) { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v)); return y; }
__device__ __forceinline__ u64 ffma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }

// The recurrence warp streams a and h of its 32 cells through a shared-memory ring filled with cp.async (no registers held
// by loads in flight): RSTG stages of 16 columns, RPRE stages ahead of the one being consumed -- the cells were written by
// other SMs one round earlier and a load of such a line takes well over 1000 cycles (measured), one stage of compute ~700.
constexpr int RSTG = 8, RPRE = 6, RLS = 20;         // lane stride of a stage in floats (16 + 4: conflict-free 128-bit shared loads)
__device__ __forceinline__ void cp_async16(float *smem_dst, const float *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// issues the copies of half `h` (16 columns starting at column 16*h of the lane's cell) into its ring stage; always commits
__device__ __forceinline__ void rec_fetch(float *ring, const float *adp, const float *hp, int64_t t0, int h, int lane, bool on) {
    if (on && h < CW / 16) {
        float *st = ring + (h % RSTG) * (2 * 32 * RLS) + lane * RLS;
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            cp_async16(st + 4 * v, adp + t0 + 16 * h + 4 * v);
            cp_async16(st + 32 * RLS + 4 * v, hp + t0 + 16 * h + 4 * v);
        }
    }
    cp_async_commit();
}

// 16 columns of the lane's recurrence (HH = which half of the 32-slot pending window they occupy: static register indices).
// The pending window is kept as 16 register pairs (p[2m], p[2m+1]) and updated with FFMA2: for an even column u the pair of
// slots (u+2m, u+2m+1) takes d * (cs[2m], cs[2m+1]) (csE), for an odd one the pair (u+2m+1, u+2m+2) takes
// d * (cs[2m+1], cs[2m+2]) (csO); cs[0] = cs[32] = 0, so the freshly cleared slot u is touched with a zero coefficient only.
// FULL: every column of the half is an interior column of every active lane (no masks).
template <int HH, bool FULL>
__device__ __forceinline__ void rec_half(u64 (&p2)[16], const u64 (&csE)[16], const u64 (&csO)[16], float *ring, float *adp, float *hp,
                                         int64_t t0, int h, int lane, int nv, bool on) {
    float av[16], hv[16];
    cp_async_wait<RPRE - 1>();                          // the copies of half h (this lane's own) have landed
    {
        const float *st = ring + (h % RSTG) * (2 * 32 * RLS) + lane * RLS;
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const float4 x = *reinterpret_cast<const float4 *>(st + 4 * v), y = *reinterpret_cast<const float4 *>(st + 32 * RLS + 4 * v);
            av[4 * v] = x.x; av[4 * v + 1] = x.y; av[4 * v + 2] = x.z; av[4 * v + 3] = x.w;
            hv[4 * v] = y.x; hv[4 * v + 1] = y.y; hv[4 * v + 2] = y.z; hv[4 * v + 3] = y.w;
        }
    }
    rec_fetch(ring, adp, hp, t0, h + RPRE, lane, on);   // stage (h + RPRE) % RSTG was consumed RSTG - RPRE halves ago
    const int i0 = 16 * h;
#pragma unroll
    for (int uu = 0; uu < 16; ++uu) {
        constexpr int base = HH * 16;
        const int u = base + uu;
        const float plo = lo_of(p2[u >> 1]), phi = hi_of(p2[u >> 1]);
        const float pu = (u & 1) ? phi : plo;
        float vn = av[uu] - pu;
        vn = vn > 0.f ? vn : 0.f;
        float d = vn - hv[uu];
        if (FULL) {
            hv[uu] = vn;
            av[uu] = d;
        } else {
            const bool ok = i0 + uu < nv;
            d = ok ? d : 0.f;
            hv[uu] = ok ? vn : hv[uu];
            av[uu] = ok ? d : av[uu];                   // tail columns keep the raw qeff for the tail job
        }
        p2[u >> 1] = (u & 1) ? pack2(plo, 0.f) : pack2(0.f, phi);   // this slot now stands for column t + 32
        const u64 dd = pack2(d, d);
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            if (u & 1) { const int x = ((u + 2 * m + 1) & 31) >> 1; p2[x] = ffma2(dd, csO[m], p2[x]); }
            else       { const int x = ((u + 2 * m) & 31) >> 1;     p2[x] = ffma2(dd, csE[m], p2[x]); }
        }
    }
    if (on) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            reinterpret_cast<float4 *>(hp + t0 + i0)[v] = make_float4(hv[4 * v], hv[4 * v + 1], hv[4 * v + 2], hv[4 * v + 3]);
            reinterpret_cast<float4 *>(adp + t0 + i0)[v] = make_float4(av[4 * v], av[4 * v + 1], av[4 * v + 2], av[4 * v + 3]);
        }
    }
}

// Grid barrier between rounds: one release-add per CTA on a global counter and an acquire spin until the whole grid has arrived.
// (cooperative_groups' grid.sync() cost ~15 us per round in this kernel -- two fences and an atomic with return per CTA;
// the launch stays cooperative so that all CTAs are co-resident.)  The counter is zeroed by the host before the launch.
struct GridBarrier {
    unsigned *ctr;
    unsigned target;
    __device__ __forceinline__ void sync() {
        __syncthreads();
        if (threadIdx.x == 0) {
            target += gridDim.x;
            asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
            unsigned v;
            do {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
            } while ((int)(v - target) < 0);
        }
        __syncthreads();
    }
};

__global__ void __launch_bounds__(NT, 1) hals2_sweep_kernel(Args a) {
    GridBarrier grid{a.barrier, 0u};
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int L = (int)a.L, Lm = L - 1;
    const int64_t K = a.K, T = a.T, nC = a.nC;
    const int64_t Tint = T - Lm;                               // columns t < Tint use the full lag window
    const int64_t n_rounds = nC + (int64_t)STAG * (K - 1) + 3;
    const int b = blockIdx.x, tid = threadIdx.x;
    const float eps = 2.220446049250313e-16f;

    if (b < a.n_block_items) {
        // ============================================================ block item (g, g'), g' < g
        int g = 1, rem = b;
        while (rem >= g) { rem -= g; ++g; }                     // items enumerated as (1,0), (2,0), (2,1), (3,0), ...
        const int gp = rem;
        float2 *Dwin = reinterpret_cast<float2 *>(smem_raw);    // [4 source pairs][WINQ]
        float2 *tab = Dwin + (GS / 2) * WINQ;                   // [4][NLP][8]
        load_table(tab, a, (int64_t)gp * GS, (int64_t)g * GS, false);
        __syncthreads();
        const int cgp = tid & 127, th = tid >> 7;               // column group (8 columns), half of the targets
        const int64_t nleft = K - (int64_t)gp * GS;
        const int nsrc = (int)(nleft < GS ? nleft : GS);
        for (int64_t s = 0; s < n_rounds; ++s) {
            const int64_t c = s + 1 - (int64_t)STAG * GS * g;
            if (c >= 0 && c < nC) {
                {
                    StageRegs sr;
                    stage_load(sr, a, (int64_t)gp * GS, nsrc, c, Tint);
                    stage_store(Dwin, sr, a, nsrc, c, Tint);
                }
                __syncthreads();
                float2 acc[8][4];
#pragma unroll
                for (int r = 0; r < 8; ++r)
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[r][q] = make_float2(0.f, 0.f);
                pull_tile<4>(acc, Dwin, tab, (nsrc + 1) / 2, L, cgp, th * 4);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int64_t kt = (int64_t)g * GS + th * 4 + q;
                    if (kt < K) {
                        float *o = a.part + part_at(c % RING, gp, kt, K, a.G) + 8 * cgp;
                        *reinterpret_cast<float4 *>(o) = make_float4(acc[0][q].x + acc[0][q].y, acc[1][q].x + acc[1][q].y, acc[2][q].x + acc[2][q].y, acc[3][q].x + acc[3][q].y);
                        *reinterpret_cast<float4 *>(o + 4) = make_float4(acc[4][q].x + acc[4][q].y, acc[5][q].x + acc[5][q].y, acc[6][q].x + acc[6][q].y, acc[7][q].x + acc[7][q].y);
                    }
                }
                __syncthreads();
            }
            grid.sync();
        }
    } else if (b < a.n_block_items + a.n_diag_items) {
        // ============================================================ diagonal item (g): finalises qeff of its 8 targets
        const int g = b - a.n_block_items;
        float2 *Dwin0 = reinterpret_cast<float2 *>(smem_raw);   // 2 x [4 source pairs][WINQ]: the window of the next target loads
        float2 *tab = Dwin0 + 2 * (GS / 2) * WINQ;              // [4][NLP][8]                 while the current one is pulled
        float *qsum = reinterpret_cast<float *>(tab + (GS / 2) * (((2 * LMAX - 1) + 7) & ~7) * 8);   // [CW]
        load_table(tab, a, (int64_t)g * GS, (int64_t)g * GS, true);
        __syncthreads();
        const int cgp = tid & 127, th = tid >> 7;
        // target i of the group is active in round s when its chunk c = s - STAG*k exists
        auto active = [&](int i, int64_t s) -> bool {
            const int64_t k = (int64_t)g * GS + i, c = s - (int64_t)STAG * k;
            return i < GS && k < K && c >= 0 && c < nC;
        };
        for (int64_t s = 0; s < n_rounds; ++s) {
            int buf = 0;
            {
                // window of the first active target of the round (the later ones are loaded during the previous target's pull)
                int first = 0;
                while (first < GS && !active(first, s)) ++first;
                if (first > 0 && first < GS) {
                    StageRegs sr;
                    const int64_t cf = s - (int64_t)STAG * ((int64_t)g * GS + first);
                    stage_load(sr, a, (int64_t)g * GS, first, cf, Tint);
                    stage_store(Dwin0, sr, a, first, cf, Tint);
                }
            }
            for (int i = 0; i < GS; ++i) {
                const int64_t k = (int64_t)g * GS + i;
                const int64_t c = s - (int64_t)STAG * k;
                if (k >= K || c < 0 || c >= nC) continue;      // uniform over the CTA
                float2 *Dwin = Dwin0 + buf * (GS / 2) * WINQ;
                // loads of the NEXT active target's window go out now and are stored into the other buffer after this pull
                int nxt = i + 1;
                while (nxt < GS && !active(nxt, s)) ++nxt;
                const int64_t cn = s - (int64_t)STAG * ((int64_t)g * GS + nxt);
                StageRegs srn;
                if (nxt < GS) stage_load(srn, a, (int64_t)g * GS, nxt, cn, Tint);
                const int64_t t0 = c * CW;
                // the loads of the hand-over (Q, H and the block partials of this cell: L2 / HBM) are issued now and consumed
                // after the pull, so their latency hides behind it
                const int col = 4 * tid;
                const int64_t t = t0 + col;
                const float4 q4 = __ldcg(reinterpret_cast<const float4 *>(a.AD_cm + cell_at(k, t, K)));      // Q[k][t..t+3]
                const float4 h4 = __ldcg(reinterpret_cast<const float4 *>(a.H_cm + cell_at(k, t, K)));
                float4 pv[16];
#pragma unroll
                for (int gp = 0; gp < 16; ++gp)
                    pv[gp] = (gp < g) ? __ldcg(reinterpret_cast<const float4 *>(a.part + part_at(c % RING, gp, k, K, a.G) + col))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
                // ---- pull from the earlier components of the own group (sources g*8 .. k-1): the two thread halves split the sources
                float2 acc[8][1];
#pragma unroll
                for (int r = 0; r < 8; ++r) acc[r][0] = make_float2(0.f, 0.f);
                __syncthreads();                                // this target's window is complete in shared memory
                if (i > 0) {
                    const int npair = (i + 1) / 2;              // the two thread halves split the source pairs
                    const int p_lo = th == 0 ? 0 : (npair + 1) / 2, p_hi = th == 0 ? (npair + 1) / 2 : npair;
                    if (p_hi > p_lo) pull_tile<1>(acc, Dwin + p_lo * WINQ, tab + (size_t)p_lo * (((2 * L - 1) + 7) & ~7) * 8, p_hi - p_lo, L, cgp, i);
                }
                if (th == 1) {
#pragma unroll
                    for (int r = 0; r < 8; ++r) qsum[8 * cgp + r] = acc[r][0].x + acc[r][0].y;
                }
                __syncthreads();
                if (th == 0) {
#pragma unroll
                    for (int r = 0; r < 8; ++r) qsum[8 * cgp + r] += acc[r][0].x + acc[r][0].y;
                }
                if (nxt < GS) stage_store(Dwin0 + (buf ^ 1) * (GS / 2) * WINQ, srn, a, nxt, cn, Tint);
                buf ^= 1;
                __syncthreads();
                // ---- truncated tail: sources t >= Tint of ALL earlier components with the tables C_w (w = T - t); work item =
                //      (target column, block of earlier components), block sums added in a fixed order (deterministic)
                if (k > 0 && Lm > 0 && t0 + CW + Lm > Tint) {
                    const int64_t c_lo = (t0 > Tint - Lm) ? t0 : Tint - Lm;
                    const int64_t c_hi = (t0 + CW < T) ? t0 + CW : T;
                    const int ncol = (int)(c_hi - c_lo);          // <= 2 (L-1)
                    // Delta H of the tail columns of all earlier components -> shared memory (this target's window buffer: its pull
                    // is done), then one warp per target column: lanes over the earlier components (table rows are contiguous in
                    // k'), 4 source columns in flight, fixed shuffle tree
                    float *dt = reinterpret_cast<float *>(Dwin);  // [k][Lm]
                    const int ntl = (int)k * Lm;
                    for (int base = tid; base < ntl; base += NT * 8) {
                        float v[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int idx = base + u * NT;
                            v[u] = (idx < ntl) ? ldcg(a.AD_cm + cell_at(idx / Lm, Tint + idx % Lm, K)) : 0.f;
                        }
#pragma unroll
                        for (int u = 0; u < 8; ++u) { const int idx = base + u * NT; if (idx < ntl) dt[idx] = v[u]; }
                    }
                    __syncthreads();
                    const int wv = tid >> 5, ln = tid & 31;
                    for (int ci = wv; ci < ncol; ci += NT / 32) {
                        const int64_t tp = c_lo + ci;
                        const int64_t ta = (tp - Lm > Tint) ? tp - Lm : Tint;
                        const int64_t tb = tp + Lm < T - 1 ? tp + Lm : T - 1;
                        double accd = 0.0;
                        for (int64_t tq = ta; tq <= tb; tq += 4) {
                            float cv[4][4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int64_t t = tq + u, w = T - t;
                                const float *ct = a.Ct + ((((w - 1) * (2 * a.L - 1) + (tp - t + Lm)) * K + k) * K);
#pragma unroll
                                for (int e = 0; e < 4; ++e) { const int kp = ln + 32 * e; cv[u][e] = (t <= tb && kp < k) ? __ldg(ct + kp) : 0.f; }
                            }
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int64_t t = tq + u;
                                if (t > tb) break;
#pragma unroll
                                for (int e = 0; e < 4; ++e) { const int kp = ln + 32 * e; if (kp < k) accd += (double)dt[kp * Lm + (int)(t - Tint)] * (double)cv[u][e]; }
                            }
                        }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) accd += __shfl_xor_sync(0xffffffffu, accd, o);
                        if (ln == 0) qsum[(int)(c_lo - t0) + ci] += (float)accd;
                    }
                    __syncthreads();
                }
                // ---- Q + the block partials in the fixed order g' = 0 .. g-1 + the own-group pull, and the hand-over
                const float c0 = a.Cf[((int64_t)Lm * K + k) * K + k];
                const float inv = 1.f / (c0 + eps + a.l2);
                {
                    // 4 consecutive columns per thread (CW == 4 * NT)
                    float qv[4] = {q4.x, q4.y, q4.z, q4.w};
                    const float hv4[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
                    for (int gp = 0; gp < 16; ++gp) {
                        if (gp < g) { qv[0] += pv[gp].x; qv[1] += pv[gp].y; qv[2] += pv[gp].z; qv[3] += pv[gp].w; }
                    }
                    float ov[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float q = qv[e] + qsum[col + e];
                        ov[e] = (t + e < Tint) ? (hv4[e] * c0 - q - a.l1) * inv : q;          // tail columns keep the raw qeff
                    }
                    *reinterpret_cast<float4 *>(a.AD_cm + cell_at(k, t, K)) = make_float4(ov[0], ov[1], ov[2], ov[3]);
                }
                __syncthreads();
            }
            grid.sync();
        }
    } else {
        // ============================================================ recurrence warp: lane = component
        const int rb = b - a.n_block_items - a.n_diag_items;
        if (tid >= 32) {                                         // only warp 0 works; the others just keep the barrier count
            for (int64_t s = 0; s < n_rounds; ++s) grid.sync();
            return;
        }
        const int lane = tid;
        const int64_t k = (int64_t)rb * 32 + lane;
        const bool live = k < K;
        u64 csE[16], csO[16], p2[16];
        float c0 = 1.f, inv = 1.f;
        if (live) {
            c0 = a.Cf[((int64_t)Lm * K + k) * K + k];
            inv = 1.f / (c0 + eps + a.l2);
        }
        {
            // both alignments of the coefficient pairs come from memory as 64-bit loads: pairs built in registers from one set of
            // scalars are rebuilt by the compiler with two moves per FFMA2 instead of being kept
            const u64 *cp = reinterpret_cast<const u64 *>(a.coef + (live ? k : 0) * 64);
#pragma unroll
            for (int m = 0; m < 16; ++m) {
                csE[m] = live ? __ldg(cp + m) : 0ull;
                csO[m] = live ? __ldg(cp + 16 + m) : 0ull;
                p2[m] = pack2(0.f, 0.f);
            }
        }
        float *adp = a.AD_cm, *hp = a.H_cm;               // cell bases are added per round (t0 below is the offset of the cell)
        for (int64_t s = 0; s < n_rounds; ++s) {
            const int64_t c = s - 1 - (int64_t)STAG * k;
            const bool on = live && c >= 0 && c < nC;
            if (__any_sync(0xffffffffu, on)) {
                // interior columns of this chunk (the truncated tail is left to the tail job)
                int nv = 0;
                if (on) { const int64_t r = Tint - c * CW; nv = (int)(r < 0 ? 0 : (r > CW ? CW : r)); }
                const int64_t t0 = on ? cell_at(k, c * CW, K) : 0;      // offset of the cell inside the working arrays
                float *ring = reinterpret_cast<float *>(smem_raw);          // [RSTG][2][32][RLS]
                // a lane that is off (not started / finished) runs the same instructions on zeros and stores nothing; the
                // mask-free path needs every active lane to be on a full interior chunk (all but the last chunk of a component)
                const bool full = __all_sync(0xffffffffu, !on || nv == CW);
#pragma unroll 1
                for (int h = 0; h < RPRE; ++h) rec_fetch(ring, adp, hp, t0, h, lane, on);
                if (!on) {                                                  // zeros for the lanes that do not load
                    for (int h = 0; h < RSTG; ++h)
                        for (int v = 0; v < 16; ++v) { ring[h * (2 * 32 * RLS) + lane * RLS + v] = 0.f; ring[h * (2 * 32 * RLS) + 32 * RLS + lane * RLS + v] = 0.f; }
                }
                if (full) {
#pragma unroll 1
                    for (int h = 0; h < CW / 16; h += 2) {
                        rec_half<0, true>(p2, csE, csO, ring, adp, hp, t0, h, lane, nv, on);
                        rec_half<1, true>(p2, csE, csO, ring, adp, hp, t0, h + 1, lane, nv, on);
                    }
                } else {
#pragma unroll 1
                    for (int h = 0; h < CW / 16; h += 2) {
                        rec_half<0, false>(p2, csE, csO, ring, adp, hp, t0, h, lane, nv, on);
                        rec_half<1, false>(p2, csE, csO, ring, adp, hp, t0, h + 1, lane, nv, on);
                    }
                }
                cp_async_wait<0>();
            }
            // ---- tail job: the last L-1 columns of one component with the truncated tables, one round after its last chunk.  At most
            //      one lane of the warp has it in a given round; the whole warp works on it: lane = lag of the pending sum.
            {
                const unsigned jm = __ballot_sync(0xffffffffu, live && Lm > 0 && s == nC + (int64_t)STAG * k + 1);
                if (jm != 0) {
                    const int64_t kk = (int64_t)rb * 32 + (__ffs(jm) - 1);
                    __shared__ float tail_d[LMAX];
                    const int sft = lane + 1;                      // this lane's lag (1 .. L-1)
                    for (int64_t t = (Tint > 0 ? Tint : 0); t < T; ++t) {
                        const int64_t w = T - t;                     // 1 .. L-1 lags left; C_w[k,k,0] from the truncated tables
                        const float c0w = __ldg(a.Ct + ((((w - 1) * (2 * a.L - 1) + Lm) * K + kk) * K + kk));
                        double pe = 0.0;
                        const int64_t ts = t - sft;
                        if (sft <= Lm && ts >= 0) {
                            const int64_t ws = T - ts;
                            const float d = (ts >= Tint) ? tail_d[(int)(ts - Tint)] : ldcg(a.AD_cm + cell_at(kk, ts, K));
                            const float cw = (ws >= a.L) ? __ldg(a.Cf + ((int64_t)(sft + Lm) * K + kk) * K + kk)
                                                         : __ldg(a.Ct + ((((ws - 1) * (2 * a.L - 1) + (sft + Lm)) * K + kk) * K + kk));
                            pe = (double)d * (double)cw;
                        }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) pe += __shfl_xor_sync(0xffffffffu, pe, o);
                        if (lane == 0) {
                            const float h = ldcg(a.H_cm + cell_at(kk, t, K));
                            const float q = ldcg(a.AD_cm + cell_at(kk, t, K)) + (float)pe;
                            float vn = (h * c0w - q - a.l1) / (c0w + eps + a.l2);
                            vn = vn > 0.f ? vn : 0.f;
                            a.H_cm[cell_at(kk, t, K)] = vn;
                            a.AD_cm[cell_at(kk, t, K)] = vn - h;
                            tail_d[(int)(t - Tint)] = vn - h;
                        }
                        __syncwarp();
                    }
                }
            }
            grid.sync();
        }
    }
}

// coefficient pairs of the recurrence lanes: coef[k][0..31] = (cs[2m], cs[2m+1]), coef[k][32..63] = (cs[2m+1], cs[2m+2]), m = 0..15,
// cs[j] = C[k,k,j] / (C[k,k,0] + eps + l2) for 1 <= j < L, zero otherwise
__global__ void hals2_coef_kernel(const float *__restrict__ Cf, float *__restrict__ coef, int64_t K, int64_t L, float l2) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= K * 64) return;
    const int64_t k = e / 64;
    const int i = (int)(e % 64), m = (i & 31) >> 1, half = i & 1;
    const int j = (i < 32) ? 2 * m + half : 2 * m + 1 + half;
    const int64_t Lm = L - 1;
    const float c0 = Cf[(Lm * K + k) * K + k];
    const float inv = 1.f / (c0 + 2.220446049250313e-16f + l2);
    coef[e] = (j >= 1 && j < L) ? Cf[((j + Lm) * K + k) * K + k] * inv : 0.f;
}

// Q and H into the component-major working arrays (AD_cm <- Q', H_cm <- H')
__global__ void hals2_prepare_kernel(const float *__restrict__ Q, const float *__restrict__ H, float *__restrict__ AD_cm,
                                     float *__restrict__ H_cm, int64_t K, int64_t T, int64_t Tp) {      // Tp = nC * CW
    __shared__ float tq[32][33], thh[32][33];
    const int64_t t0 = (int64_t)blockIdx.x * 32, k0 = (int64_t)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t t = t0 + r, k = k0 + threadIdx.x;
        const bool ok = t < T && k < K;
        tq[r][threadIdx.x] = ok ? Q[t * K + k] : 0.f;
        thh[r][threadIdx.x] = ok ? H[t * K + k] : 0.f;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t k = k0 + r, t = t0 + threadIdx.x;
        if (k < K && t < Tp) { const int64_t o = cell_at(k, t, K); AD_cm[o] = tq[threadIdx.x][r]; H_cm[o] = thh[threadIdx.x][r]; }
    }
}

// new H back to the [t][K] layout
__global__ void hals2_finish_kernel(const float *__restrict__ H_cm, float *__restrict__ H, int64_t K, int64_t T, int64_t Tp) {
    __shared__ float tile[32][33];
    const int64_t t0 = (int64_t)blockIdx.x * 32, k0 = (int64_t)blockIdx.y * 32;
    {   // block (32, 8): four loads in flight per thread
        float v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t k = k0 + threadIdx.y + 8 * i, t = t0 + threadIdx.x;
            v[i] = (k < K && t < T) ? H_cm[cell_at(k, t, K)] : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) tile[threadIdx.y + 8 * i][threadIdx.x] = v[i];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t t = t0 + r, k = k0 + threadIdx.x;
        if (t < T && k < K) H[t * K + k] = tile[threadIdx.x][r];
    }
}

inline size_t smem_bytes() {
    // two window buffers (diagonal items double-buffer their staging), the table slice, the per-cell sums; the recurrence ring fits inside
    static_assert(RSTG * 2 * 32 * RLS <= 2 * GS * WINQ, "recurrence ring");
    return (size_t)(2 * GS * WINQ + GS * (((2 * LMAX - 1) + 7) & ~7) * 8 + CW) * sizeof(float);
}

}  // namespace hals2
}  // namespace cmf
