// SIMT (CUDA-core) kernels of the CNMF fit path, templated on the scalar type S (double/float).
// These are the fp64 engine and the fp32 fallback engine; the tcgen05 engine (kernels_tc.cuh)
// replaces the three big contractions for fp32 when K*L is large.
//
// Device layouts (DESIGN.md section 2), all t-major so that a time shift is a pointer offset:
//   X  [t][N]   (identical to Julia's column-major N x T), valid local columns [0, Tl + L-1)
//   H  [t][K]   (identical to Julia's column-major K x T), valid local columns [-(L-1), Tl + L-1)
//   Wi [j][N]   with j = l*K + k  (the unfolded row index of src/algs/hals.jl:102), n contiguous
//
// Reference semantics (file:line relative to /root/reference):
//   conv       src/common.jl:24-34     est[n,t]  = sum_{l,k} W[k,n,l] H[k,t-l]
//   transconv  src/common.jl:71-81     out[k,t]  = sum_{l,n} W[k,n,l] X[n,t+l]
//   corr       src/algs/mult.jl:31-34  num[k,n,l]= sum_u   H[k,u]   X[n,u+l]
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cmf {

#define CMF_EPS 2.220446049250313e-16 /* src/CMF.jl:20 */

// ------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum of one double per thread; result valid in thread 0.  `red` holds >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double *red) {
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    const int nthr = blockDim.x * blockDim.y;
    v = warp_sum(v);
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    double r = 0.0;
    if (tid < 32) {
        r = (tid < (nthr + 31) / 32) ? red[tid] : 0.0;
        r = warp_sum(r);
    }
    return r;
}

// Deterministic second stage: block b sums the `n` doubles in[b*n .. b*n+n) in a fixed order into out[b]
// (one block per restart of a batch handle; a single block otherwise).
__global__ void reduce_sum_kernel(const double *__restrict__ in, int64_t n, double *__restrict__ out) {
    __shared__ double red[32];
    in += (int64_t)blockIdx.x * n;
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += in[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[blockIdx.x] = s;
}

// Restart r of a batch handle: its rank K_r, the first of its components [off, off + K_r) on the stacked component axis
// (width C = sum K_r), and where its block starts in each per-restart buffer (elements).  Launches with a restart grid index
// read entry blockIdx.z (or .y); single handles pass no table and are restart 0 at offset 0.
struct BatchRest {
    int64_t K, off;
    int64_t gs;   // G_r / S2_r (K_r L x K_r L) in GS
    int64_t cf;   // lag table (2L-1) x K_r x K_r in Cf
    int64_t ex;   // Gram (L K_r^2) + H tail ((L-1) K_r) + 1 in exch1
    int64_t cp;   // the Gram's nsplit partials (nsplit L K_r^2) in corr_part
    int64_t tp;   // denomH tail partials (nb_r (L-1) K_r) in tail_part
};

// Restart of element i of an array whose component index is (i / inner) % C -- W in the internal layout (inner = N), H
// (inner = 1): col_rest[c] is the restart that owns stacked component c.
__device__ __forceinline__ int64_t restart_of(int64_t i, int64_t inner, const int *col_rest, int64_t C) { return col_rest[(i / inner) % C]; }

// ------------------------------------------------------------------------------------------
// conv (+ residual, + loss):   est[t][n] = sum_{l<L,k<K} Wi[l*K+k][n] * H[t-l][k]
//   block (16, TY) threads, micro-tile TN (n) x TT (t); tile BN = 16*TN, BT = TY*TT.
//   smem: H window of KC components  Hs[KC][BT + Lpad - 1], W chunk Ws[LC][BN] of one k.
//   flags: bit0 store est, bit1 store est - X, bit2 accumulate sum((est-X)^2) into partial[block],
//          bit3 synth epilogue out = max(0, est + noise*gauss(seed, n, t_global)),
//          bit4 partial[2b] = <est,X>, partial[2b+1] = ||est||^2 (init_rand rescale, src/model.jl:119-120),
//          bit5 store the loss gradient d D / d est of PGD's pluggable losses (src/algs/pgd.jl:28-70): 2 (est - X) for SquareLoss
//               (lossf 0), sign(est - X) for AbsoluteLoss (lossf 1), times mask[t][n] when a MaskedLoss wraps it,
//          bit6 accumulate the loss itself into partial[block]: sum (m (X - est))^2 resp. sum |m (X - est)| (pgd.jl:33-35,43-45,67-69).
// ------------------------------------------------------------------------------------------
template <typename S>
struct ConvArgs {
    const S *Wi;     // [L*K][N]
    const S *H;      // owned column 0; valid [-(hlo), Tl + hhi)
    const S *X;      // owned column 0 (flags 2|4)
    S *out;          // [t][N] local columns (flags 1|2|8)
    double *partial; // one per block (flag 4)
    int64_t N, K, L;
    int64_t t_lo, t_hi;   // local column range to produce [t_lo, t_hi)
    int64_t h_lo, h_hi;   // valid local column range of H: [h_lo, h_hi), zero outside
    int flags;
    uint64_t seed;        // synth
    int64_t t_global0;    // global index of local column 0 (synth)
    double noise;         // synth
    int KC;               // components staged per H window
    const S *mask;        // flags 32|64: optional mask [t][N] (nullptr = all ones)
    int lossf;            // flags 32|64: 0 SquareLoss, 1 AbsoluteLoss
    // restart z = blockIdx.z of a batch handle (tab != nullptr): K = tab[z].K, W rows (l*ldw + k) and H columns t*ldh + k from
    // Wi + tab[z].off*N and H + tab[z].off, partials from partial + z*part_rs (single handles: ldw = ldh = K, one z)
    int64_t ldw, ldh, part_rs;
    const BatchRest *tab;
};

__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z += 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
// counter-based uniform in (0,1): keyed on (seed, stream, index)
__device__ __forceinline__ double u01(uint64_t seed, uint64_t stream, uint64_t idx) {
    uint64_t h = mix64(mix64(seed ^ (stream * 0xd1342543de82ef95ull)) + idx);
    return ((double)(h >> 11) + 0.5) * (1.0 / 9007199254740992.0);
}
__device__ __forceinline__ double gauss01(uint64_t seed, uint64_t stream, uint64_t idx) {
    const double u1 = u01(seed, stream, 2 * idx), u2 = u01(seed, stream, 2 * idx + 1);
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

constexpr int CONV_LC = 32; // lags per staged W chunk

template <typename S, int TN, int TT, int TY>
__global__ void __launch_bounds__(16 * TY) conv_kernel(ConvArgs<S> a) {
    constexpr int BN = 16 * TN, BT = TY * TT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int64_t N = a.N, K = a.tab ? a.tab[blockIdx.z].K : a.K, L = a.L;
    const int64_t off = a.tab ? a.tab[blockIdx.z].off : 0;
    const int Lpad = (int)((L + 7) / 8 * 8);
    const int HW = BT + Lpad - 1;
    S *Hs = reinterpret_cast<S *>(smem_raw);            // [KC][HW]
    S *Ws = Hs + (size_t)a.KC * HW;                      // [CONV_LC][BN]
    __shared__ double red[32];

    const int tx = threadIdx.x, ty = threadIdx.y;
    const int tid = ty * 16 + tx, nthr = 16 * TY;
    const int64_t n0 = (int64_t)blockIdx.y * BN;          // grid.x runs over time tiles (can be > 65535)
    const int64_t t0 = a.t_lo + (int64_t)blockIdx.x * BT;
    const S *Wr = a.Wi + off * N, *Hr = a.H + off;
    double *partial = a.partial ? a.partial + (int64_t)blockIdx.z * a.part_rs : nullptr;

    S acc[TT][TN];
#pragma unroll
    for (int j = 0; j < TT; ++j)
#pragma unroll
        for (int i = 0; i < TN; ++i) acc[j][i] = S(0);

    for (int64_t kc0 = 0; kc0 < K; kc0 += a.KC) {
        const int kc = (int)min((int64_t)a.KC, K - kc0);
        __syncthreads();
        // stage the H window: Hs[k][i] = H[t0 - (Lpad-1) + i][kc0 + k]
        for (int idx = tid; idx < kc * HW; idx += nthr) {
            const int k = idx % kc, i = idx / kc;
            const int64_t t = t0 - (Lpad - 1) + i;
            S v = S(0);
            if (t >= a.h_lo && t < a.h_hi) v = Hr[t * a.ldh + kc0 + k];
            Hs[(size_t)k * HW + i] = v;
        }
        for (int k = 0; k < kc; ++k) {
            const S *hrow = Hs + (size_t)k * HW + ty * TT + (Lpad - 1) - 7;
            for (int lc0 = 0; lc0 < Lpad; lc0 += CONV_LC) {
                const int lcn = min(CONV_LC, Lpad - lc0);
                __syncthreads();
                for (int idx = tid; idx < lcn * BN; idx += nthr) {
                    const int n = idx % BN, dl = idx / BN;
                    const int64_t l = lc0 + dl;
                    S v = S(0);
                    if (l < L && n0 + n < N) v = Wr[((l * a.ldw) + kc0 + k) * N + n0 + n];
                    Ws[dl * BN + n] = v;
                }
                __syncthreads();
                for (int l8 = 0; l8 < lcn; l8 += 8) {
                    S hw[TT + 7];
#pragma unroll
                    for (int i = 0; i < TT + 7; ++i) hw[i] = hrow[i - (lc0 + l8)];
#pragma unroll
                    for (int dl = 0; dl < 8; ++dl) {
                        S wv[TN];
                        const S *wp = Ws + (l8 + dl) * BN + tx * TN;
#pragma unroll
                        for (int i = 0; i < TN; ++i) wv[i] = wp[i];
#pragma unroll
                        for (int j = 0; j < TT; ++j) {
                            const S h = hw[7 - dl + j];
#pragma unroll
                            for (int i = 0; i < TN; ++i) acc[j][i] = fma(wv[i], h, acc[j][i]);
                        }
                    }
                }
            }
        }
    }

    // epilogue
    double sq = 0.0, dxe = 0.0;
#pragma unroll
    for (int j = 0; j < TT; ++j) {
        const int64_t t = t0 + ty * TT + j;
        if (t >= a.t_hi) continue;
        S part = S(0), pdot = S(0);
#pragma unroll
        for (int i = 0; i < TN; ++i) {
            const int64_t n = n0 + tx * TN + i;
            if (n >= N) continue;
            const S e = acc[j][i];
            if (a.flags & 1) a.out[t * N + n] = e;
            if (a.flags & 16) {  // init_rand rescale partials: <est, X> and ||est||^2
                pdot = fma(e, a.X[t * N + n], pdot);
                part = fma(e, e, part);
            }
            if (a.flags & 8) {
                const double g = gauss01(a.seed, 3, (uint64_t)((a.t_global0 + t) * N + n));
                const double v = (double)e + a.noise * g;
                a.out[t * N + n] = (S)(v > 0.0 ? v : 0.0);
            }
            if (a.flags & 6) {
                const S r = e - a.X[t * N + n];
                if (a.flags & 2) a.out[t * N + n] = r;
                part = fma(r, r, part);
            }
            if (a.flags & 96) {
                const S r = e - a.X[t * N + n];
                const S m = a.mask ? a.mask[t * N + n] : S(1);
                if (a.flags & 32) a.out[t * N + n] = (a.lossf == 0 ? S(2) * r : (r > S(0) ? S(1) : (r < S(0) ? S(-1) : S(0)))) * m;
                if (a.flags & 64) { const S mr = m * r; part += (a.lossf == 0) ? mr * mr : (mr < S(0) ? -mr : mr); }
            }
        }
        sq += (double)part;
        dxe += (double)pdot;
    }
    if (a.flags & (4 | 64)) {
        sq = block_sum(sq, red);
        if (tid == 0) partial[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = sq;
    }
    if (a.flags & 16) {
        const size_t b = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
        dxe = block_sum(dxe, red);
        if (tid == 0) partial[2 * b] = dxe;
        sq = block_sum(sq, red);
        if (tid == 0) partial[2 * b + 1] = sq;
    }
}

// ------------------------------------------------------------------------------------------
// transconv (generic):  out[t][k] = sum_{l<Lin} sum_{n<Nin} Wg[(l*Kout + k)*Nin + n] * Xin[(t+l)*ldx + n]
//   used for numH (Wg = Wi, Xin = X) and for denomH (Wg = C table, Xin = H with halos).
//   block = kgroups x tgroups threads, micro-tile TK (k) x TT (t), lane index = kg fastest.
//   smem: Xs[NC][XWP] (t contiguous per n, one pad word every 8), Ws[8][NC][KP].
// ------------------------------------------------------------------------------------------
template <typename S>
struct TransArgs {
    const S *Wg;
    const S *Xin;   // column 0 of the window; valid columns [0, x_cols)
    S *out;         // [t][Kout], t in [0, t_out)
    int64_t Nin, Kout, Lin, ldx;
    int64_t t_out, x_cols;
    int kgroups, tgroups;
    int64_t n_chunk;      // units summed by one CTA (blockIdx.z % nsplit selects the chunk; a multiple of TR_NC); Nin rounded up = no split
    int64_t part_stride;  // elements between the partial outputs of consecutive chunks (0 = no split: `out` is the result)
    int nsplit;           // chunks per restart: blockIdx.z / nsplit is the restart (single handles: one restart)
    int64_t ldo;          // row stride of out (Kout, or C when restarts write their columns of a stacked array)
    // denomH of a batch handle (tab != nullptr): restart z has Nin = Kout = tab[z].K and reads Wg + tab[z].cf (its lag table)
    // and Xin + tab[z].off, writes out + tab[z].off; Nin / Kout above are the largest K_r (the grid's extent)
    const BatchRest *tab;
};

// out[i] = sum_z part[z * stride + i] in the fixed order z = 0, 1, ... (deterministic; the N-split of transconv_kernel)
template <typename S>
__global__ void sum_parts_kernel(const S *__restrict__ part, S *__restrict__ out, int64_t n, int64_t stride, int nparts) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    S v = part[i];
    for (int z = 1; z < nparts; ++z) v += part[(int64_t)z * stride + i];
    out[i] = v;
}

constexpr int TR_NC = 16;

template <typename S, int TK, int TT>
__global__ void __launch_bounds__(256) transconv_kernel(TransArgs<S> a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int kgroups = a.kgroups, tgroups = a.tgroups;
    const int BT = tgroups * TT;
    const int Lpad = (int)((a.Lin + 7) / 8 * 8);
    const int XW = BT + Lpad;               // logical window length (t0 .. t0 + BT + Lpad - 1)
    const int XWP = XW + XW / 8 + 1;        // padded: phys(i) = i + i/8
    const int KP = kgroups * TK;
    S *Xs = reinterpret_cast<S *>(smem_raw);        // [TR_NC][XWP]
    S *Ws = Xs + (size_t)TR_NC * XWP;               // [8][TR_NC][KP]

    const int tid = threadIdx.x, nthr = blockDim.x;
    const int kg = tid % kgroups, tg = tid / kgroups;
    const int64_t t0 = (int64_t)blockIdx.x * BT;
    const int64_t kb = (int64_t)blockIdx.y * KP;     // first k of this block
    const int64_t rs = blockIdx.z / a.nsplit, zs = blockIdx.z % a.nsplit;
    const S *Wg = a.Wg, *Xin = a.Xin;
    S *out = a.out;
    int64_t Nin = a.Nin, Kout = a.Kout;
    if (a.tab) {
        const BatchRest r = a.tab[rs];
        Nin = Kout = r.K;
        if (kb >= Kout) return;                      // past this restart's components
        Wg += r.cf; Xin += r.off; out += r.off;
    }

    S acc[TT][TK];
#pragma unroll
    for (int j = 0; j < TT; ++j)
#pragma unroll
        for (int i = 0; i < TK; ++i) acc[j][i] = S(0);

    const int64_t n_lo = zs * a.n_chunk, n_hi = min(Nin, n_lo + a.n_chunk);
    for (int64_t nc0 = n_lo; nc0 < n_hi; nc0 += TR_NC) {
        __syncthreads();
        // stage X window (transposed): Xs[n][phys(i)] = Xin[(t0+i)*ldx + nc0 + n]
        for (int idx = tid; idx < TR_NC * XW; idx += nthr) {
            const int n = idx % TR_NC, i = idx / TR_NC;
            const int64_t t = t0 + i;
            S v = S(0);
            if (t < a.x_cols && nc0 + n < n_hi) v = Xin[t * a.ldx + nc0 + n];
            Xs[(size_t)n * XWP + i + i / 8] = v;
        }
        for (int lc0 = 0; lc0 < Lpad; lc0 += 8) {
            __syncthreads();
            // stage W chunk: Ws[dl][n][k] = Wg[((lc0+dl)*Kout + kb + k)*Nin + nc0 + n]
            for (int idx = tid; idx < 8 * TR_NC * KP; idx += nthr) {
                const int n = idx % TR_NC, k = (idx / TR_NC) % KP, dl = idx / (TR_NC * KP);
                const int64_t l = lc0 + dl;
                S v = S(0);
                if (l < a.Lin && kb + k < Kout && nc0 + n < n_hi)
                    v = Wg[((l * Kout) + kb + k) * Nin + nc0 + n];
                Ws[((size_t)dl * TR_NC + n) * KP + k] = v;
            }
            __syncthreads();
            // thread's window base: logical index tg*TT + lc0 (a multiple of 8 when TT == 8)
            const int base = tg * TT + lc0;
#pragma unroll 2
            for (int n = 0; n < TR_NC; ++n) {
                S xw[TT + 7];
                const S *xr = Xs + (size_t)n * XWP;
#pragma unroll
                for (int i = 0; i < TT + 7; ++i) {
                    const int li = base + i;
                    xw[i] = xr[li + li / 8];
                }
#pragma unroll
                for (int dl = 0; dl < 8; ++dl) {
                    S wv[TK];
                    const S *wp = Ws + ((size_t)dl * TR_NC + n) * KP + kg * TK;
#pragma unroll
                    for (int i = 0; i < TK; ++i) wv[i] = wp[i];
#pragma unroll
                    for (int j = 0; j < TT; ++j) {
                        const S x = xw[j + dl];
#pragma unroll
                        for (int i = 0; i < TK; ++i) acc[j][i] = fma(wv[i], x, acc[j][i]);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < TT; ++j) {
        const int64_t t = t0 + tg * TT + j;
        if (t >= a.t_out) continue;
#pragma unroll
        for (int i = 0; i < TK; ++i) {
            const int64_t k = kb + kg * TK + i;
            if (k < Kout) out[zs * a.part_stride + t * a.ldo + k] = acc[j][i];
        }
    }
}

// ------------------------------------------------------------------------------------------
// corr (generic):  part[split][(l*K + k)*Nin + n] = sum_{tau in split} hm(tau - l)[k] * Xin[tau*ldx + n]
//   hm(u) = H[u*K + k] for u in [0, u_hi), zero outside (owned columns only).
//   block (16, 16): tx -> 8 consecutive n, ty -> pair p = (k, lag group of 8); reduction over tau.
//   fp32 accumulators are flushed into the double partial every CORR_FLUSH columns.
// ------------------------------------------------------------------------------------------
template <typename S>
struct CorrArgs {
    const S *H;      // owned column 0, [u][K]
    const S *Xin;    // column 0, [tau][ldx]
    double *part;    // [nsplit][L*K*Nin]
    int64_t Nin, K, L, ldx;
    int64_t u_hi;    // owned columns (H valid for u in [0,u_hi))
    int64_t tau_hi;  // Xin valid for tau in [0, tau_hi)
    int64_t split_len;
    int64_t ldh;     // row stride of H (K, or C for the per-restart Gram of a batch handle)
    int nsplit;      // splits per restart: blockIdx.z / nsplit is the restart (single handles: one restart)
    // the per-restart Gram of a batch handle (tab != nullptr): restart z has Nin = K = tab[z].K, reads H + tab[z].off and
    // Xin + tab[z].off and writes part + tab[z].cp; Nin / K above are the largest K_r (the grid's extent)
    const BatchRest *tab;
};

constexpr int CORR_BTAU = 32;
constexpr int CORR_PB = 16;
constexpr int CORR_FLUSH = 2048;

template <typename S>
__global__ void __launch_bounds__(256) corr_kernel(CorrArgs<S> a) {
    constexpr int TN = 8, BN = 16 * TN, HWN = CORR_BTAU + 7;
    __shared__ __align__(16) S Xs[CORR_BTAU][BN];
    __shared__ S Hs[CORR_PB][HWN + 1];
    const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * 16 + tx;
    const int64_t n0 = (int64_t)blockIdx.x * BN;
    const int64_t p = (int64_t)blockIdx.y * CORR_PB + ty;
    const int64_t ngrp = (a.L + 7) / 8;
    const int64_t rs = blockIdx.z / a.nsplit, zs = blockIdx.z % a.nsplit;
    const S *Hr = a.H, *Xr = a.Xin;
    double *part = a.part;
    int64_t K = a.K, Nin = a.Nin;
    if (a.tab) {
        const BatchRest r = a.tab[rs];
        K = Nin = r.K;
        if (n0 >= Nin || (int64_t)blockIdx.y * CORR_PB >= K * ngrp) return;   // past this restart's components
        Hr += r.off; Xr += r.off; part += r.cp;
    }
    const bool pvalid = p < K * ngrp;
    const int64_t k = pvalid ? p % K : 0, l0 = pvalid ? (p / K) * 8 : 0;
    const int64_t tau_a = zs * a.split_len;
    const int64_t tau_b = min(a.tau_hi, tau_a + a.split_len);
    part += (size_t)zs * (size_t)(a.L * K * Nin);

    S acc[8][TN];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = S(0);
    bool flushed_once = false;
    int since_flush = 0;

    auto flush = [&]() {
        if (!pvalid) return;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int64_t l = l0 + i;
            if (l >= a.L) continue;
#pragma unroll
            for (int j = 0; j < TN; ++j) {
                const int64_t n = n0 + tx * TN + j;
                if (n >= Nin) continue;
                double *d = part + (l * K + k) * Nin + n;
                *d = flushed_once ? (*d + (double)acc[i][j]) : (double)acc[i][j];
                acc[i][j] = S(0);
            }
        }
        flushed_once = true;
    };

    for (int64_t tau0 = tau_a; tau0 < tau_b; tau0 += CORR_BTAU) {
        __syncthreads();
        for (int idx = tid; idx < CORR_BTAU * BN; idx += 256) {
            const int n = idx % BN, dt = idx / BN;
            const int64_t tau = tau0 + dt;
            S v = S(0);
            if (tau < tau_b && n0 + n < Nin) v = Xr[tau * a.ldx + n0 + n];
            Xs[dt][n] = v;
        }
        for (int idx = tid; idx < CORR_PB * HWN; idx += 256) {
            const int i = idx % HWN, pp = idx / HWN;
            const int64_t q = (int64_t)blockIdx.y * CORR_PB + pp;
            S v = S(0);
            if (q < K * ngrp) {
                const int64_t kk = q % K, ll0 = (q / K) * 8;
                const int64_t u = tau0 - ll0 - 7 + i;
                if (u >= 0 && u < a.u_hi) v = Hr[u * a.ldh + kk];
            }
            Hs[pp][i] = v;
        }
        __syncthreads();
#pragma unroll
        for (int t8 = 0; t8 < CORR_BTAU; t8 += 8) {
            S hw[15];
#pragma unroll
            for (int i = 0; i < 15; ++i) hw[i] = Hs[ty][t8 + i];
#pragma unroll
            for (int dt = 0; dt < 8; ++dt) {
                S xv[TN];
#pragma unroll
                for (int j = 0; j < TN; ++j) xv[j] = Xs[t8 + dt][tx * TN + j];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const S h = hw[dt - i + 7];
#pragma unroll
                    for (int j = 0; j < TN; ++j) acc[i][j] = fma(h, xv[j], acc[i][j]);
                }
            }
        }
        since_flush += CORR_BTAU;
        if (sizeof(S) == 4 && since_flush >= CORR_FLUSH) {
            flush();
            since_flush = 0;
        }
    }
    flush();
}

// out[i] = (S) sum_s part[s][i]   (fixed order -> deterministic).  The per-restart Gram of a batch handle (tab != nullptr):
// restart blockIdx.y has n = L K_r^2, reads part + tab[y].cp and writes out_d + tab[y].ex
template <typename S>
__global__ void reduce_partials_kernel(const double *__restrict__ part, int nsplit, int64_t n,
                                       S *__restrict__ out, double *__restrict__ out_d, const BatchRest *tab = nullptr, int64_t L = 0) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tab) {
        const BatchRest r = tab[blockIdx.y];
        n = L * r.K * r.K;
        part += r.cp;
        if (out) out += r.ex;
        if (out_d) out_d += r.ex;
    }
    if (i >= n) return;
    double s = 0.0;
    for (int sp = 0; sp < nsplit; ++sp) s += part[(size_t)sp * n + i];
    if (out) out[i] = (S)s;
    if (out_d) out_d[i] = s;
}

// ------------------------------------------------------------------------------------------
// plain GEMM  C[M][Nn] = A[M][Kg] * B   (row-major; TRANSB: B is [Nn][Kg], else [Kg][Nn])
//   64x64 tile, BK 16, 256 threads, 4x4 micro-tile.  Used for G*Wi and Wi*Wi' (<1% of the FLOPs).
//   Each operand's rows are addressed through a GemmRows; blockIdx.z is the restart of a batch handle.
// ------------------------------------------------------------------------------------------
// Row j of a GEMM operand starts at (j / grp) * ldg + (j % grp) * ld.  Row-major with leading dimension ld: grp = INT64_MAX.
// Operands of a batch handle take restart z = blockIdx.z from the table (rank != RANK_NONE):
//   RANK_W  W_r, rows j = l*K_r + k at (l*C + off_r + k)*N: ld = N, ldg = C*N, grp = K_r, start off_r*N;
//   RANK_G  G_r / S2_r, a K_r L x K_r L row-major block at gs_r: ld = K_r L.
// Every extent an operand spans with K_r L rows or columns is K_r L for restart z; M, Nn, Kg passed in are the largest.
enum { RANK_NONE = 0, RANK_W = 1, RANK_G = 2 };
struct GemmRows {
    int64_t ld, grp, ldg;
    int rank;
    __device__ __forceinline__ int64_t at(int64_t j) const { return (j / grp) * ldg + (j % grp) * ld; }
    // this operand of restart r: sets its row layout and returns its start
    __device__ __forceinline__ int64_t of(const BatchRest &r, int64_t L) {
        if (rank == RANK_W) { grp = r.K; return r.off * ld; }
        ld = r.K * L;
        return r.gs;
    }
};

template <typename S, bool TRANSB>
__global__ void __launch_bounds__(256) gemm_kernel(const S *__restrict__ A, const S *__restrict__ B,
                                                   S *__restrict__ C, int64_t M, int64_t Nn,
                                                   int64_t Kg, GemmRows ra, GemmRows rb, GemmRows rc,
                                                   const BatchRest *tab = nullptr, int64_t L = 0) {
    constexpr int BM = 64, BNt = 64, BK = 16;
    __shared__ S As[BK][BM + 1];
    __shared__ S Bs[BK][BNt + 1];
    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
    const int64_t m0 = (int64_t)blockIdx.y * BM, c0 = (int64_t)blockIdx.x * BNt;
    if (tab) {
        const BatchRest r = tab[blockIdx.z];
        const int64_t kl = r.K * L;
        int64_t &Brows = TRANSB ? Nn : Kg, &Bcols = TRANSB ? Kg : Nn;
        if (ra.rank) { A += ra.of(r, L); M = kl; if (ra.rank == RANK_G) Kg = kl; }
        if (rb.rank) { B += rb.of(r, L); Brows = kl; if (rb.rank == RANK_G) Bcols = kl; }
        if (rc.rank) { C += rc.of(r, L); M = kl; if (rc.rank == RANK_G) Nn = kl; }
        if (m0 >= M || c0 >= Nn) return;                 // past this restart's block
    }
    S acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = S(0);
    for (int64_t k0 = 0; k0 < Kg; k0 += BK) {
        __syncthreads();
        for (int idx = tid; idx < BM * BK; idx += 256) {
            const int kk = idx % BK, mm = idx / BK;
            S v = S(0);
            if (m0 + mm < M && k0 + kk < Kg) v = A[ra.at(m0 + mm) + k0 + kk];
            As[kk][mm] = v;
        }
        for (int idx = tid; idx < BNt * BK; idx += 256) {
            S v = S(0);
            if (TRANSB) {
                const int kk = idx % BK, nn = idx / BK;
                if (c0 + nn < Nn && k0 + kk < Kg) v = B[rb.at(c0 + nn) + k0 + kk];
                Bs[kk][nn] = v;
            } else {
                const int nn = idx % BNt, kk = idx / BNt;
                if (c0 + nn < Nn && k0 + kk < Kg) v = B[rb.at(k0 + kk) + c0 + nn];
                Bs[kk][nn] = v;
            }
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            S av[4], bv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) av[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) bv[j] = Bs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t m = m0 + ty * 4 + i, c = c0 + tx * 4 + j;
            if (m < M && c < Nn) C[rc.at(m) + c] = acc[i][j];
        }
}

// ------------------------------------------------------------------------------------------
// G = Htilde Htilde'  from the Toeplitz part Rg[d][k][k'] and the tail Ht[c][k] = H[T-(L-1)+c][k]
//   G[(l,k)][(l',k')] = (l>=l' ? Rg[l-l'][k][k'] : Rg[l'-l][k'][k]) - sum_{i<min(l,l')} Ht[L-1-l+i][k] Ht[L-1-l'+i][k']
// ------------------------------------------------------------------------------------------
// Batch handles (tab != nullptr): Rg is the base of exch1; restart y = blockIdx.y has K = K_r, its Gram at Rg + ex_r, its tail
// right after it, and G_r at G + gs_r (Ht unused).
template <typename S>
__global__ void build_G_kernel(const double *__restrict__ Rg, const double *__restrict__ Ht,
                               S *__restrict__ G, int64_t K, int64_t L, const BatchRest *tab = nullptr) {
    if (tab) {
        const BatchRest r = tab[blockIdx.y];
        K = r.K; Rg += r.ex; Ht = Rg + L * K * K; G += r.gs;
    }
    const int64_t KL = K * L;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= KL * KL) return;
    const int64_t jp = idx % KL, j = idx / KL;
    const int64_t k = j % K, l = j / K, kp = jp % K, lp = jp / K;
    double g = (l >= lp) ? Rg[((l - lp) * K + k) * K + kp] : Rg[((lp - l) * K + kp) * K + k];
    const int64_t m = l < lp ? l : lp;
    double tail = 0.0;
    for (int64_t i = 0; i < m; ++i) tail += Ht[(L - 1 - l + i) * K + k] * Ht[(L - 1 - lp + i) * K + kp];
    G[idx] = (S)(g - tail);
}

// partial[block] = sum over a grid-stride slice of S2[j][j'] * G[j][j'], with G = Htilde Htilde' formed on the fly
// from Rg and the tail as in build_G_kernel:  ||conv(W,H)||^2 = <W W', Htilde Htilde'>.
// The sum walks the block diagonals of G: thread (d, k, k') visits (l, l') = (d+s, s) (d >= 0) or (s, s-d) (d < 0),
// where the Toeplitz part is constant and the tail grows by one product per step,
//   tail(l+1, l'+1) = tail(l, l') + Ht[L-2-l][k] Ht[L-2-l'][k'],
// so every element of S2 is read once and the (K L)^2 L tail work becomes (K L)^2.  grid-stride over (2L-1) K K diagonals.
// Restart y = blockIdx.y of a batch handle (tab != nullptr): K = Ks = K_r, ld = K_r L, S2 + gs_r, its Gram at Rg + ex_r with the
// tail right after it; its partials at partial + y * gridDim.x.
template <typename S>
__global__ void s2_dot_G_diag_kernel(const S *__restrict__ S2, int64_t Ks, int64_t ld, const double *__restrict__ Rg,
                                     const double *__restrict__ Ht, int64_t K, int64_t L, double *__restrict__ partial,
                                     const BatchRest *tab = nullptr) {
    __shared__ double red[32];
    if (tab) {
        const BatchRest r = tab[blockIdx.y];
        K = Ks = r.K; ld = r.K * L; S2 += r.gs; Rg += r.ex; Ht = Rg + L * K * K;
        partial += (int64_t)blockIdx.y * gridDim.x;
    }
    double acc = 0.0;
    const int64_t total = (2 * L - 1) * K * K;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t kp = e % K, k = (e / K) % K, d = e / (K * K) - (L - 1);
        const double r = (d >= 0) ? Rg[(d * K + k) * K + kp] : Rg[((-d) * K + kp) * K + k];
        const int64_t steps = L - (d >= 0 ? d : -d);
        int64_t l = d >= 0 ? d : 0, lp = d >= 0 ? 0 : -d;
        double tail = 0.0;
        for (int64_t s_ = 0; s_ < steps; ++s_, ++l, ++lp) {
            acc += (r - tail) * (double)S2[(l * Ks + k) * ld + lp * Ks + kp];
            if (s_ + 1 < steps) tail += Ht[(L - 2 - l) * K + k] * Ht[(L - 2 - lp) * K + kp];
        }
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}

// Cf[(d+L-1)][k][k'] = sum_{l, 0<=l-d<L} S2[(l,k)][(l-d,k')]      (S2 = W W' over the unfolded rows)
// S2 is addressed as S2[(l*Ks + k) * ld + (l'*Ks + k')]: (Ks, ld) = (K, K*L) for the SIMT product and
// (Kp, rows_u) for the tensor-core product over the padded rows.
// Restart y = blockIdx.y of a batch handle (tab != nullptr): K = Ks = K_r, ld = K_r L, S2 + gs_r, Cf + cf_r.
template <typename S>
__global__ void lag_table_kernel(const S *__restrict__ S2, S *__restrict__ Cf, int64_t K, int64_t L, int64_t Ks, int64_t ld,
                                 const BatchRest *tab = nullptr) {
    if (tab) {
        const BatchRest r = tab[blockIdx.y];
        K = Ks = r.K; ld = r.K * L; S2 += r.gs; Cf += r.cf;
    }
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (2 * L - 1) * K * K) return;
    const int64_t kp = idx % K, k = (idx / K) % K, d = idx / (K * K) - (L - 1);
    double s = 0.0;
    for (int64_t l = (d > 0 ? d : 0); l < L && l - d < L; ++l) s += (double)S2[(l * Ks + k) * ld + (l - d) * Ks + kp];
    Cf[idx] = (S)s;
}

// Truncated tail of denomH (columns with w = T - t < L):
//   den[t][k] = sum_{l<w} sum_{l'<L} sum_{k'} S2[(l,k)][(l',k')] * H[t + l - l'][k']
// one block per (tail column, k).
template <typename S>
__global__ void __launch_bounds__(256) denomH_tail_kernel(const S *__restrict__ S2, const S *__restrict__ H,
                                                           S *__restrict__ den, int64_t K, int64_t L,
                                                           int64_t Tl, int64_t h_lo, int64_t Ks, int64_t ld) {
    __shared__ double red[32];
    const int KL = (int)(K * L), Ki = (int)K;
    const int64_t c = blockIdx.x;                 // tail column index: t = Tl - (L-1) + c
    const int64_t k = blockIdx.y;
    const int64_t t = Tl - (L - 1) + c;
    if (t < 0) return;
    const int w = (int)(Tl - t);                  // 1 .. L-1
    double s = 0.0;
    // thread -> fixed set of (l', k') pairs (32-bit index math), loop over the w lags of row (l, k)
    for (int jp = threadIdx.x; jp < KL; jp += blockDim.x) {
        const int lp = jp / Ki, kp = jp - lp * Ki;
        const S *s2col = S2 + (int64_t)lp * Ks + kp;
        const S *hcol = H + kp;
        S acc = S(0);                                 // <= L terms per chain, accumulated in the handle's type
        for (int l = 0; l < w; ++l) {
            const int64_t u = t + l - lp;
            if (u < h_lo) continue;
            acc = fma(s2col[((int64_t)l * Ks + k) * ld], hcol[u * K], acc);
        }
        s += (double)acc;
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) den[t * K + k] = (S)s;
}

// The same tail in prefix form, each element of S2 read once: thread (d, k') keeps the truncated table entry
//   C_w[d][k][k'] = sum_{l<w, 0<=l-d<L} S2[(l,k)][(l-d,k')]        (w = 1 .. L-1, one more lag l = w-1 per step)
// in a register while w grows, and den[Tl-w][k] = sum_{d,k'} C_w[d][k][k'] H[Tl-w+d][k'].  Warp sums go to shared
// memory, block sums to part[block][c][k] (c = L-1-w, the tail column index); denomH_tail_reduce_kernel adds the blocks
// in order (deterministic).  grid (ceil((2L-1)K / 256), K, restarts), dynamic smem 8*(L-1) doubles.  Restart z of a batch
// handle (tab != nullptr) has K = Ks = K_r, ld = K_r L, reads S2 + gs_r and H + off_r (row stride ldh) and writes part + tp_r;
// the grid is sized for the largest K_r and the blocks past restart z's return at once.
template <typename S>
__global__ void __launch_bounds__(256) denomH_tail_prefix_kernel(const S *__restrict__ S2, const S *__restrict__ H,
                                                                  double *__restrict__ part, int64_t K, int64_t L, int64_t Tl,
                                                                  int64_t h_lo, int64_t Ks, int64_t ld, int64_t ldh,
                                                                  const BatchRest *tab = nullptr) {
    extern __shared__ double tail_sm[];                 // [8 warps][L-1]
    const int64_t k = blockIdx.y;
    if (tab) {
        const BatchRest r = tab[blockIdx.z];
        K = Ks = r.K; ld = r.K * L;
        if (k >= K || (int64_t)blockIdx.x * blockDim.x >= (2 * L - 1) * K) return;
        S2 += r.gs; H += r.off; part += r.tp;
    }
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = e < (2 * L - 1) * K;
    const int64_t dq = live ? e / K : 0, kp = live ? e - dq * K : 0;
    const int64_t d = dq - (L - 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int Lm = (int)(L - 1);
    S pre = S(0);
    // the S2 entries a thread walks (one per w) do not depend on one another: 8 loads in flight ahead of the running sum
    // (a dependent ~1 us load per step made this kernel latency-bound)
    S nxt[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int64_t l = q, lp = l - d;
        nxt[q] = (live && q < Lm && lp >= 0 && lp < L) ? S2[(l * Ks + k) * ld + lp * Ks + kp] : S(0);
    }
    for (int w0 = 1; w0 <= Lm; w0 += 8) {
        S cur[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) cur[q] = nxt[q];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int64_t l = w0 - 1 + 8 + q, lp = l - d;
            nxt[q] = (live && l < Lm && lp >= 0 && lp < L) ? S2[(l * Ks + k) * ld + lp * Ks + kp] : S(0);
        }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int w = w0 + q;
        if (w > Lm) break;
        pre += cur[q];
        const int64_t u = Tl - w + d;
        double v = 0.0;
        if (live && pre != S(0) && u >= h_lo) v = (double)(pre * H[u * ldh + kp]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) tail_sm[warp * Lm + (w - 1)] = v;
    }
    }
    __syncthreads();
    for (int w = threadIdx.x + 1; w <= Lm; w += blockDim.x) {
        double s = 0.0;
        for (int q = 0; q < 8; ++q) s += tail_sm[q * Lm + (w - 1)];
        part[((int64_t)blockIdx.x * Lm + (Lm - w)) * K + k] = s;
    }
}

// Restart y = blockIdx.y of a batch handle (tab != nullptr): K = K_r, part + tp_r with the ceil((2L-1) K_r / 256) blocks of
// its prefix launch, den + off_r with row stride ldd.
template <typename S>
__global__ void denomH_tail_reduce_kernel(const double *__restrict__ part, S *__restrict__ den, int64_t K, int64_t L, int64_t Tl,
                                          int nblocks, int64_t ldd, const BatchRest *tab = nullptr) {
    if (tab) {
        const BatchRest r = tab[blockIdx.y];
        K = r.K; nblocks = (int)(((2 * L - 1) * K + 255) / 256); part += r.tp; den += r.off;
    }
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;     // c * K + k
    if (i >= (L - 1) * K) return;
    const int64_t c = i / K, k = i - c * K, t = Tl - (L - 1) + c;
    if (t < 0) return;
    double s = 0.0;
    for (int b = 0; b < nblocks; ++b) s += part[(int64_t)b * (L - 1) * K + i];
    den[t * ldd + k] = (S)s;
}

// ------------------------------------------------------------------------------------------
// element-wise pieces
// ------------------------------------------------------------------------------------------
// src/algs/mult.jl:37-38 / :51-52   x <- max(eps, x * num / (den + l1 + 2*l2*x + eps))
// Batch handles pass reg != nullptr: restart r = restart_of(i, inner, col_rest, C) takes l1 = reg[4r], l2 = reg[4r+1] and
// is left alone while active[r] == 0 (a converged restart is frozen).
template <typename S>
__global__ void mu_update_kernel(S *__restrict__ x, const S *__restrict__ num, const S *__restrict__ den,
                                 S l1, S l2, int64_t n, const double *__restrict__ reg = nullptr,
                                 const int *__restrict__ active = nullptr, int64_t inner = 1, const int *__restrict__ col_rest = nullptr,
                                 int64_t C = 1) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (reg) {
        const int64_t r = restart_of(i, inner, col_rest, C);
        if (!active[r]) return;
        l1 = (S)reg[4 * r];
        l2 = (S)reg[4 * r + 1];
    }
    const S eps = (S)CMF_EPS;
    S v = x[i];
    v = v * (num[i] / (den[i] + l1 + S(2) * l2 * v + eps));
    x[i] = v > eps ? v : eps;
}

// The same update for fp32 arrays whose length is a multiple of 4 and whose pointers are 16-byte aligned: one float4 per thread
// and step (more bytes in flight per thread: the scalar kernel reaches ~55 % of the HBM peak), fixed grid, and -- for the H update
// of the expansion loss -- the inner product <num, x'> of the NEW x with the numerator, as one fp64 partial per CTA
// (partial == nullptr: no inner product).
__global__ void __launch_bounds__(256) mu_update_vec4_kernel(float4 *__restrict__ x, const float4 *__restrict__ num, const float4 *__restrict__ den,
                                                             float l1, float l2, int64_t n4, double *__restrict__ partial) {
    __shared__ double red[32];
    const float eps = (float)CMF_EPS;
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 v = x[i];
        const float4 a = __ldg(num + i), d = __ldg(den + i);
        v.x = v.x * (a.x / (d.x + l1 + 2.f * l2 * v.x + eps)); v.x = v.x > eps ? v.x : eps;
        v.y = v.y * (a.y / (d.y + l1 + 2.f * l2 * v.y + eps)); v.y = v.y > eps ? v.y : eps;
        v.z = v.z * (a.z / (d.z + l1 + 2.f * l2 * v.z + eps)); v.z = v.z > eps ? v.z : eps;
        v.w = v.w * (a.w / (d.w + l1 + 2.f * l2 * v.w + eps)); v.w = v.w > eps ? v.w : eps;
        x[i] = v;
        if (partial) acc += (double)a.x * (double)v.x + (double)a.y * (double)v.y + (double)a.z * (double)v.z + (double)a.w * (double)v.w;
    }
    if (partial) {
        acc = block_sum(acc, red);
        if (threadIdx.x == 0) partial[blockIdx.x] = acc;
    }
}

// s_r != nullptr (batch handles): restart restart_of(i, inner, col_rest, C) is scaled by s_r[r]
template <typename S>
__global__ void scale_kernel(S *__restrict__ x, S s, int64_t n, const double *__restrict__ s_r = nullptr, int64_t inner = 1,
                             const int *__restrict__ col_rest = nullptr, int64_t C = 1) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (s_r) s = (S)s_r[restart_of(i, inner, col_rest, C)];
    x[i] *= s;
}

// partial[block] = sum over a grid-stride slice of a[i]*b[i]  (b may alias a)
template <typename S>
__global__ void dot_partial_kernel(const S *__restrict__ a, const S *__restrict__ b, int64_t n,
                                   double *__restrict__ partial) {
    __shared__ double red[32];
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        s += (double)a[i] * (double)b[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

// Julia W[k + K*(n + N*l)]  <->  Wi[(l*ldk + k)*N + n]; ldk = K, or C for the stacked W of a batch handle (tab != nullptr),
// whose restart y = blockIdx.y has K = K_r, its Julia block at Wj + off_r*N*L and its rows at Wi + off_r*N
template <typename S>
__global__ void w_julia_to_internal(const S *__restrict__ Wj, S *__restrict__ Wi, int64_t K, int64_t N, int64_t L, int64_t ldk,
                                    const BatchRest *tab = nullptr) {
    if (tab) {
        const BatchRest r = tab[blockIdx.y];
        K = r.K; Wj += r.off * N * L; Wi += r.off * N;
    }
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= K * N * L) return;
    const int64_t n = idx % N, k = (idx / N) % K, l = idx / (N * K);
    Wi[(l * ldk + k) * N + n] = Wj[k + K * (n + N * l)];
}
template <typename S>
__global__ void w_internal_to_julia(const S *__restrict__ Wi, S *__restrict__ Wj, int64_t K, int64_t N, int64_t L, int64_t ldk,
                                    const BatchRest *tab = nullptr) {
    if (tab) {
        const BatchRest r = tab[blockIdx.y];
        K = r.K; Wj += r.off * N * L; Wi += r.off * N;
    }
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= K * N * L) return;
    const int64_t k = idx % K, n = (idx / K) % N, l = idx / (K * N);
    Wj[idx] = Wi[(l * ldk + k) * N + n];
}

// H of a batch handle: R host blocks K_r x T one after another (restart r's [t][k] at T*off_r + t*K_r + k) <-> the stacked
// device array st[t][off_r + k] of C = sum K_r columns
template <typename S>
__global__ void h_stack_kernel(const S *__restrict__ src, S *__restrict__ dst, int64_t C, int64_t T, const BatchRest *__restrict__ tab,
                               const int *__restrict__ col_rest, int to_stacked) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;     // index into the stacked array
    if (i >= C * T) return;
    const int64_t c = i % C, t = i / C;
    const BatchRest r = tab[col_rest[c]];
    const int64_t b = T * r.off + t * r.K + (c - r.off);
    if (to_stacked) dst[i] = src[b];
    else dst[b] = src[i];
}

// tail[c][k] (double) = H[Tl-(L-1)+c][k]; zeros when this shard is not the last one
// shift_and_stack (src/common.jl:133-142) on t-major storage: out[t][l*K + k] = H[t-l][k], zero for t < l
template <typename S>
__global__ void shift_stack_kernel(const S *__restrict__ H, S *__restrict__ out, int64_t K, int64_t L, int64_t T) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= K * L * T) return;
    const int64_t j = e % (K * L), t = e / (K * L), l = j / K, k = j % K;
    out[e] = (t >= l) ? H[(t - l) * K + k] : S(0);
}

// restart y = blockIdx.y of a batch handle (tab != nullptr): K = K_r, H + off_r with row stride ldh; tail is the base of
// exch1 and restart y's tail follows its Gram, at tail + ex_r + L K_r^2
template <typename S>
__global__ void h_tail_kernel(const S *__restrict__ H, double *__restrict__ tail, int64_t K, int64_t L,
                              int64_t Tl, int is_last, int64_t ldh, const BatchRest *tab = nullptr) {
    if (tab) {
        const BatchRest r = tab[blockIdx.y];
        K = r.K; H += r.off; tail += r.ex + L * K * K;
    }
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (L - 1) * K) return;
    const int64_t c = idx / K, k = idx % K;
    tail[idx] = is_last ? (double)H[(Tl - (L - 1) + c) * ldh + k] : 0.0;
}

// ------------------------------------------------------------------------------------------
// counter-based generators (synthetic data model of datasets/synthetic.jl:29-61, and init_rand)
// ------------------------------------------------------------------------------------------
template <typename S>
__global__ void uniform_kernel(S *__restrict__ x, int64_t n, uint64_t seed, uint64_t stream, int64_t idx0) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = (S)u01(seed, stream, (uint64_t)(idx0 + i));
}

// ground-truth H: Exponential(1) * Bernoulli(p_h), keyed on the global (t, k); zero for t < 0 or t >= T
template <typename S>
__global__ void synth_H_kernel(S *__restrict__ H, int64_t K, int64_t t_first, int64_t cols, int64_t T,
                               uint64_t seed, double p_h) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * cols) return;
    const int64_t k = i % K, t = t_first + i / K;
    S v = S(0);
    if (t >= 0 && t < T) {
        const uint64_t id = (uint64_t)(t * K + k);
        if (u01(seed, 1, id) < p_h) v = (S)(-log(u01(seed, 2, id)));
    }
    H[i] = v;
}

// Marsaglia-Tsang Gamma(alpha<1 via boost) with counter-based draws
__device__ inline double gamma_draw(double alpha, uint64_t seed, uint64_t stream, uint64_t id) {
    const double a = alpha + 1.0, d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    double g = d;
    for (uint64_t it = 0; it < 32; ++it) {
        const double x = gauss01(seed, stream, id * 64 + it);
        const double v0 = 1.0 + c * x;
        if (v0 <= 0.0) continue;
        const double v = v0 * v0 * v0, u = u01(seed, stream + 1, id * 64 + it);
        if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) { g = d * v; break; }
    }
    return g * pow(u01(seed, stream + 2, id), 1.0 / alpha);
}

// ground-truth W in the internal layout: Dirichlet(alpha) weights over k for each unit n, times a
// Gaussian bump over the lag axis linspace(-1,1,L) centred at U(-1,1)   (datasets/synthetic.jl:42-51)
template <typename S>
__global__ void synth_W_kernel(S *__restrict__ Wi, int64_t K, int64_t N, int64_t L, uint64_t seed,
                               double alpha, double sigma) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    double tot = 0.0;
    for (int64_t k = 0; k < K; ++k) tot += gamma_draw(alpha, seed, 10, (uint64_t)(n * K + k));
    for (int64_t k = 0; k < K; ++k) {
        const double wgt = gamma_draw(alpha, seed, 10, (uint64_t)(n * K + k)) / tot;
        const double cent = 2.0 * u01(seed, 20, (uint64_t)(n * K + k)) - 1.0;
        for (int64_t l = 0; l < L; ++l) {
            const double x = (L > 1) ? (-1.0 + 2.0 * (double)l / (double)(L - 1)) : -1.0;
            const double z = (x - cent) / sigma;
            Wi[(l * K + k) * N + n] = (S)(wgt * exp(-0.5 * z * z) / (sigma * 2.5066282746310002));
        }
    }
}

// ------------------------------------------------------------------------------------------
// HALS sweeps (src/algs/hals.jl:90-154) in the Gram / recurrence form of oracle/restructured.py
// ------------------------------------------------------------------------------------------
// W sweep: one block per unit n.  P row and W row live in shared memory.
//   for k, for l:  j = l*K+k;  g = G[j][j];  w' = max((w*g - P[j] - l1)/(g + eps + l2), 0);
//                  P[:] += (w'-w) * G[j][:]
template <typename S>
__global__ void __launch_bounds__(256) hals_w_sweep_kernel(const S *__restrict__ G, const S *__restrict__ P /*[KL][N]*/,
                                                            S *__restrict__ Wi /*[KL][N]*/, int64_t K, int64_t L,
                                                            int64_t N, S l1, S l2) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int64_t KL = K * L;
    S *Ps = reinterpret_cast<S *>(smem_raw);
    __shared__ S delta_s;
    const int64_t n = blockIdx.x;
    for (int64_t j = threadIdx.x; j < KL; j += blockDim.x) Ps[j] = P[j * N + n];
    __syncthreads();
    for (int64_t k = 0; k < K; ++k)
        for (int64_t l = 0; l < L; ++l) {
            const int64_t j = l * K + k;
            if (threadIdx.x == 0) {
                const S g = G[j * KL + j];
                const S w = Wi[j * N + n];
                S v = (w * g - Ps[j] - l1) / (g + (S)CMF_EPS + l2);
                v = v > S(0) ? v : S(0);
                Wi[j * N + n] = v;
                delta_s = v - w;
            }
            __syncthreads();
            const S d = delta_s;
            if (d != S(0)) {
                const S *grow = G + j * KL;
                for (int64_t jj = threadIdx.x; jj < KL; jj += blockDim.x) Ps[jj] = fma(d, grow[jj], Ps[jj]);
            }
            __syncthreads();
        }
}

// Sequential recurrence of one component over W = 32 interior columns (full lag window, no truncation) with the pending
// corrections of the next W columns held in registers: p[j] is the pending correction of column t + j.  The W steps
// are fully unrolled, so the rotation of the window is a compile-time renaming.  Lane u holds h and q of column i0 + u
// (one coalesced shared load per block) and receives that column's result; the per-column values are broadcast by
// shuffles that do not depend on the recurrence, so a step costs its dependent chain (add, 2 FMA/MUL, max, sub) plus W
// independent FMAs, with no shared-memory access inside the chain.  Every lane runs the same scalar code (the values
// are warp-uniform).  Requires L <= W.
template <typename S, int W, typename CT>
__device__ __forceinline__ void hals_recurrence_block(S *hch, S *qeff, S (&p)[W], const CT &c /*C[k,k,j], zero for j >= L*/, S c0,
                                                       S inv, S l1, int i0, int lane) {
    static_assert(W == 32, "one column per lane");
    const S hl = hch[i0 + lane], ql = qeff[i0 + lane];
    S vout = S(0), dout = S(0);
#pragma unroll
    for (int u = 0; u < W; ++u) {
        const S h = __shfl_sync(0xffffffffu, hl, u);
        const S q = __shfl_sync(0xffffffffu, ql, u) + p[u];
        S v = (h * c0 - q - l1) * inv;
        v = v > S(0) ? v : S(0);
        const S d = v - h;
        if (lane == u) { vout = v; dout = d; }
        p[u] = S(0);                                   // this slot now stands for column t + W
#pragma unroll
        for (int j = 1; j < W; ++j) p[(u + j) % W] = fma(d, c[j], p[(u + j) % W]);
    }
    hch[i0 + lane] = vout;
    qeff[i0 + lane] = dout;                            // Delta H of the block (qeff is dead now)
}

// Truncated lag tables of the H sweep for every pair of components (the sweep's pull over the last L-1 columns):
//   Ct[w-1][dd+L-1][k][k'] = C_w[k',k,dd] = sum_{l<w, 0<=l-dd<L} S2[(l,k')][(l-dd,k)],   w = 1..L-1
// one thread per (dd, k, k') walks w with a running sum (each element of S2 is read once per table it enters).  S2 = W W' is
// symmetric, so the element is read as S2[(l-dd,k)][(l,k')]: consecutive threads (k' fastest) then read consecutive addresses
// (the other orientation strides by a whole row: 40 ms instead of ~1 ms per sweep at config 5).
template <typename S>
__global__ void hals_tail_table_kernel(const S *__restrict__ S2, S *__restrict__ Ct, int64_t K, int64_t L, int64_t Ks, int64_t ld) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (2 * L - 1) * K * K) return;
    const int64_t kp = e % K, k = (e / K) % K, dq = e / (K * K), dd = dq - (L - 1);
    double pre = 0.0;
    for (int64_t w = 1; w < L; ++w) {
        const int64_t l = w - 1, lp = l - dd;
        if (lp >= 0 && lp < L) pre += (double)S2[(lp * Ks + k) * ld + l * Ks + kp];
        Ct[(((w - 1) * (2 * L - 1) + dq) * K + k) * K + kp] = (S)pre;
    }
}

// H sweep (hals.jl:121-154) as a wavefront over (component k, time chunk c) in ONE cooperative launch.
//   Q[t][k] = transconv(W, conv(W,H) - X)[k,t] at the start of the sweep (gradient of the H step),
//   Cf[(d+L-1)][k][k'] interior lag table, S2 = W W' for the truncated tail tables, D[t][k] = Delta H (output).
// Cell (k, c) = columns [c*HW_TC, (c+1)*HW_TC) of component k:
//   pull  : qeff[t'] = Q[t'][k] + sum_{k'<k} sum_{|t-t'|<L} D[t][k'] * C_{w(t)}[k',k,t'-t]      (all threads, no races)
//   sweep : for t: h' = max((h*c0 - qeff[t] - pend(t) - l1)/(c0 + eps + l2), 0);  D[t][k] = h'-h;
//           pend(t+s) += D[t][k] * C_w[k,k,s]                                                  (warp 0, sequential)
// Component k may run cell c once component k-1 has finished cell c+1 (its corrections reach L-1 columns back)
// and its own cell c-1; CTA b owns components b, b+grid, ...; progress[k] counts finished cells of k.
// Every Q element has exactly one reader/writer at a time, so the result is deterministic and identical to
// the sequential k-outer / t-inner sweep of the reference.
constexpr int HW_TC = 1024;  // columns per cell
constexpr int HW_NT = 512;   // threads per CTA (512 -> 128 registers per thread for the register-window recurrence)
// earlier components staged per pull step (sized so the transposed Delta window fits shared memory)
template <typename S> __host__ __device__ constexpr int hw_kb() { return sizeof(S) == 4 ? 32 : 16; }
// dynamic shared memory of hals_h_wave_kernel in elements of S
template <typename S>
inline size_t hals_wave_smem_elems(int64_t L) {
    const size_t WW = HW_TC + 2 * (L - 1);
    const size_t QP = ((WW + 7) >> 3) | 1;
    const size_t dwin = hw_kb<S>() * 8 * QP > (size_t)4 * HW_TC ? hw_kb<S>() * 8 * QP : (size_t)4 * HW_TC;
    return 2 * HW_TC + (2 * L + 32) + L + 32 + (2 * L + 6) * hw_kb<S>() + dwin;
}

template <typename S>
__global__ void __launch_bounds__(HW_NT) hals_h_wave_kernel(const S *__restrict__ Cf, const S *__restrict__ S2,
                                                             const S *__restrict__ Q, S *__restrict__ H, S *__restrict__ D,
                                                             S *__restrict__ tailC_all /*[grid][L*L]*/, int *progress /*[K]*/,
                                                             int64_t K, int64_t L, int64_t T, int64_t Ks, int64_t ld,
                                                             S l1, S l2, const S *__restrict__ Ct /*tail tables or nullptr*/) {
    constexpr int HW_KB = hw_kb<S>();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    S *qeff = reinterpret_cast<S *>(smem_raw);       // [HW_TC]
    S *pend = qeff + HW_TC;                          // ring of RB entries
    S *ckk = pend + (2 * L + 32);                    // Cf[k,k,s], s = 0..L-1
    S *ckk32 = ckk + L;                              // [32] C[k,k,j] zero padded (register-window recurrence, L <= 32)
    S *hch = ckk32 + 32;                             // [HW_TC] H of the current cell
    S *Cs = hch + HW_TC;                             // [(2L-1)][HW_KB] lag-table slice of the pull phase
    S *Dwin = Cs + (2 * L + 6) * HW_KB;              // [HW_KB][8 planes][QP] transposed Delta window of the pull phase (Cs: lag rows padded to a multiple of 8)
    const int RB = (int)(2 * L + 32);
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int64_t nC = (T + HW_TC - 1) / HW_TC;
    const int64_t Tint = T - (L - 1);                // columns t < Tint have the full lag window (w = L)
    S *tailC = tailC_all + (size_t)blockIdx.x * (size_t)(L * L);

    for (int64_t k = blockIdx.x; k < K; k += gridDim.x) {
        // per-component tables
        for (int64_t s = tid; s < L; s += nthr) ckk[s] = Cf[((s + L - 1) * K + k) * K + k];
        if (tid < 32) ckk32[tid] = (tid >= 1 && tid < L) ? Cf[((tid + L - 1) * K + k) * K + k] : S(0);
        // tailC[w][s] = C_w[k,k,s] = sum_{l<w, l-s>=0} S2[(l,k)][(l-s,k)],  w = 1..L-1, s = 0..L-1
        for (int64_t idx = tid; idx < L * L; idx += nthr) {
            const int64_t w = idx / L, s = idx % L;
            double acc = 0.0;
            for (int64_t l = s; l < w; ++l) acc += (double)S2[(l * Ks + k) * ld + (l - s) * Ks + k];
            tailC[idx] = (S)acc;
        }
        for (int i = tid; i < RB; i += nthr) pend[i] = S(0);
        __syncthreads();
        S Pw[32];                             // register window of pending corrections (warp 0, L <= 32)
        S creg[sizeof(S) == 4 ? 32 : 1];      // C[k,k,j] in registers (fp32; 128 registers per thread at 512 threads)
#pragma unroll
        for (int j = 0; j < 32; ++j) Pw[j] = S(0);
        if (sizeof(S) == 4) {
#pragma unroll
            for (int j = 0; j < 32; ++j) creg[j % (sizeof(S) == 4 ? 32 : 1)] = ckk32[j];
        }
        bool ring_mode = false;               // true once the window lives in the shared ring (tail / partial blocks / L > 32)

        for (int64_t c = 0; c < nC; ++c) {
            const int64_t t0 = c * HW_TC;
            // ---- wait: component k-1 must have finished cell min(c+1, nC-1)
            if (k > 0 && tid == 0) {
                const int need = (int)((c + 2 < nC) ? c + 2 : nC);
                volatile int *pr = progress + (k - 1);
                while (*pr < need) { __nanosleep(64); }
            }
            __syncthreads();
            __threadfence();
            // ---- pull: corrections from all earlier components, HW_KB components at a time through shared memory.
            //      Register tiling: thread (cg, kq) owns the 8 consecutive columns 8*cg .. 8*cg+7 and a quarter of the
            //      staged components; along the lag loop the 8 Delta values slide through registers, so each step costs
            //      one new Delta load + one (broadcast) table load for 8 FMAs.  The Delta window is stored transposed and
            //      split into 8 planes (index i -> plane i&7, slot i>>3) so that lanes read consecutive words.
            {
                const int WW = HW_TC + 2 * (int)(L - 1);
                const int QP = ((WW + 7) >> 3) | 1;            // slots per plane (odd)
                const int WWQ = 8 * QP;                        // words per staged component
                const int cg = tid & (HW_TC / 8 - 1), kq = tid >> 7;       // column group, component quarter
                constexpr int NKQ = HW_NT / (HW_TC / 8);                   // 4 groups of components per staged block
                constexpr int KQ = HW_KB / NKQ;
                S a8[8];
#pragma unroll
                for (int r = 0; r < 8; ++r) a8[r] = S(0);
                // counted in staged blocks: with kp0 < k as the loop condition, ptxas spills a fifth more in the fp64 instantiation
                const int nsb = (int)((k + HW_KB - 1) / HW_KB);
                for (int sb = 0; sb < nsb; ++sb) {
                    const int64_t kp0 = (int64_t)sb * HW_KB;
                    const int kb = (int)((k - kp0 < HW_KB) ? k - kp0 : HW_KB);
                    __syncthreads();
                    // 8 loads in flight per thread: Delta comes from L2 (written by other SMs), a dependent load per
                    // element would expose its latency 68 times per staged block
                    if (sizeof(S) == 4 && (K & 3) == 0) {
                        // 128-bit loads: 4 staged components per load (kp0 is a multiple of HW_KB, rows of Delta are K long)
                        constexpr int KB4 = HW_KB / 4;
                        for (int base = tid; base < WW * KB4; base += nthr * 4) {
                            float4 v4[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int idx = base + u * nthr;
                                const int k4 = (idx % KB4) * 4, i = idx / KB4;
                                const int64_t t = t0 - (L - 1) + i;
                                v4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                                if (idx < WW * KB4 && k4 < kb && t >= 0 && t < Tint)
                                    v4[u] = __ldcg(reinterpret_cast<const float4 *>(D + t * K + kp0 + k4));
                            }
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const int idx = base + u * nthr;
                                const int k4 = (idx % KB4) * 4, i = idx / KB4;
                                if (idx < WW * KB4) {
                                    const int ad = (i & 7) * QP + (i >> 3);
                                    Dwin[(k4 + 0) * WWQ + ad] = (S)((k4 + 0 < kb) ? v4[u].x : 0.f);
                                    Dwin[(k4 + 1) * WWQ + ad] = (S)((k4 + 1 < kb) ? v4[u].y : 0.f);
                                    Dwin[(k4 + 2) * WWQ + ad] = (S)((k4 + 2 < kb) ? v4[u].z : 0.f);
                                    Dwin[(k4 + 3) * WWQ + ad] = (S)((k4 + 3 < kb) ? v4[u].w : 0.f);
                                }
                            }
                        }
                    } else
                    for (int base = tid; base < WW * HW_KB; base += nthr * 8) {
                        S v8[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int idx = base + u * nthr;
                            const int kk = idx % HW_KB, i = idx / HW_KB;
                            const int64_t t = t0 - (L - 1) + i;
                            v8[u] = S(0);
                            if (idx < WW * HW_KB && kk < kb && t >= 0 && t < Tint) v8[u] = __ldcg(D + t * K + kp0 + kk);   // tail columns: slow path below
                        }
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int idx = base + u * nthr;
                            const int kk = idx % HW_KB, i = idx / HW_KB;
                            if (idx < WW * HW_KB) Dwin[kk * WWQ + (i & 7) * QP + (i >> 3)] = v8[u];
                        }
                    }
                    const int nlp = (2 * (int)L - 1 + 7) & ~7;                 // lag rows padded with zeros to a multiple of 8
                    for (int idx = tid; idx < nlp * HW_KB; idx += nthr) {
                        const int kk = idx % HW_KB;
                        const int64_t j = idx / HW_KB;
                        Cs[idx] = (kk < kb && j < 2 * L - 1) ? Cf[(j * K + kp0 + kk) * K + k] : S(0);
                    }
                    __syncthreads();
                    // two staged components per pass (they share the index arithmetic); the window of 8 Delta values per
                    // component is a circular register file whose rotation is compile-time: the lag loop is unrolled by 8,
                    // slot (r - jj) & 7 holds window index ib + r - j at step j = j0 + jj, and step jj refills slot -jj.
                    for (int kk = kq * KQ; kk < kq * KQ + KQ && kk < kb; kk += 2) {
                        const bool two = kk + 1 < kb;
                        const S *dwa = Dwin + kk * WWQ, *dwb = two ? dwa + WWQ : dwa;
                        const int ib = 8 * cg + 2 * (int)(L - 1);
                        const int nl = 2 * (int)L - 1;
                        S da[8], db[8];
                        da[0] = S(0); db[0] = S(0);
#pragma unroll
                        for (int o = 1; o < 8; ++o) {
                            const int ad = ((ib + o) & 7) * QP + ((ib + o) >> 3);
                            da[o] = dwa[ad]; db[o] = dwb[ad];
                        }
                        // the padded lag rows of Cs are zero, so whole groups of 8 steps run without a branch (window
                        // indices below 0 are clamped: their table entries are zero)
                        const int kkb = two ? kk + 1 : kk;
                        const S cbs = two ? S(1) : S(0);
                        for (int j0 = 0; j0 < nl; j0 += 8) {
#pragma unroll
                            for (int jj = 0; jj < 8; ++jj) {
                                const int j = j0 + jj;
                                const int in = max(ib - j, 0);         // window index entering at this step (column r = 0)
                                const int ad = (in & 7) * QP + (in >> 3);
                                da[(8 - jj) & 7] = dwa[ad]; db[(8 - jj) & 7] = dwb[ad];
                                const S ca = Cs[j * HW_KB + kk], cb = Cs[j * HW_KB + kkb] * cbs;
#pragma unroll
                                for (int r = 0; r < 8; ++r) {
                                    a8[r] = fma(da[(r - jj + 8) & 7], ca, a8[r]);
                                    a8[r] = fma(db[(r - jj + 8) & 7], cb, a8[r]);
                                }
                            }
                        }
                    }
                }
                // reduce the component groups: red[kq][column] (reuses the Delta window space), then add Q
                __syncthreads();
                S *red = Dwin;
#pragma unroll
                for (int r = 0; r < 8; ++r) red[kq * HW_TC + 8 * cg + r] = a8[r];
                __syncthreads();
                for (int col = tid; col < HW_TC; col += nthr) {
                    const int64_t tp = t0 + col;
                    S acc = (tp < T) ? Q[tp * K + k] : S(0);
#pragma unroll
                    for (int g = 0; g < NKQ; ++g) acc += red[g * HW_TC + col];
                    qeff[col] = acc;
                }
                __syncthreads();
                // truncated tail columns t >= Tint (only the last chunks see them): the tables C_w[k',k,dd] come precomputed
                // (hals_tail_table_kernel) as Ct[w-1][dd+L-1][k][k']; work item = (column, block of earlier components),
                // block sums go through shared memory and are added in a fixed order (deterministic)
                if (Ct != nullptr) {
                    if (k > 0 && t0 + HW_TC + (L - 1) > Tint) {
                        const int64_t c_lo = (t0 > Tint - (L - 1)) ? t0 : Tint - (L - 1);
                        const int64_t c_hi = (t0 + HW_TC < T) ? t0 + HW_TC : T;
                        const int ncol = (int)(c_hi - c_lo);
                        const int CH = (int)((k + 15) / 16 > 16 ? (k + 15) / 16 : 16);
                        const int nch = (int)((k + CH - 1) / CH);
                        S *part = Dwin;                            // [nch][HW_TC], nch <= 16
                        if (ncol > 0) {
                            for (int it = tid; it < ncol * nch; it += nthr) {
                                const int ci = it % ncol, ch = it / ncol;
                                const int64_t tp = c_lo + ci;
                                int64_t ta = (tp - (L - 1) > Tint) ? tp - (L - 1) : Tint;
                                if (ta < 0) ta = 0;
                                const int64_t tb = tp + (L - 1) < T - 1 ? tp + (L - 1) : T - 1;
                                const int64_t kp_lo = (int64_t)ch * CH, kp_hi = (kp_lo + CH < k) ? kp_lo + CH : k;
                                double accd = 0.0;
                                for (int64_t t = ta; t <= tb; ++t) {
                                    const int64_t dd = tp - t, w = T - t;
                                    const S *ct = Ct + ((((w - 1) * (2 * L - 1) + (dd + L - 1)) * K + k) * K);
                                    const S *dr = D + t * K;
                                    for (int64_t kp = kp_lo; kp < kp_hi; ++kp) accd += (double)__ldcg(dr + kp) * (double)ct[kp];
                                }
                                part[ch * HW_TC + ci] = (S)accd;
                            }
                            __syncthreads();
                            for (int ci = tid; ci < ncol; ci += nthr) {
                                double sacc = 0.0;
                                for (int ch = 0; ch < nch; ++ch) sacc += (double)part[ch * HW_TC + ci];
                                qeff[(int)(c_lo - t0) + ci] += (S)sacc;
                            }
                        }
                    }
                } else
                for (int col = tid; col < HW_TC; col += nthr) {
                    const int64_t tp = t0 + col;
                    if (tp < T && tp + (L - 1) >= Tint) {
                        double accd = 0.0;
                        const int64_t ta = (tp - (L - 1) > Tint) ? tp - (L - 1) : Tint;
                        const int64_t tb = tp + (L - 1) < T - 1 ? tp + (L - 1) : T - 1;
                        for (int64_t t = (ta > 0 ? ta : 0); t <= tb; ++t) {
                            const int64_t dd = tp - t;
                            const int64_t w = T - t;    // C_w[k',k,dd] = sum_{l<w, 0<=l-dd<L} S2[(l,k')][(l-dd,k)]
                            for (int64_t kp = 0; kp < k; ++kp) {
                                const S d = __ldcg(D + t * K + kp);
                                if (d == S(0)) continue;
                                double cw = 0.0;
                                for (int64_t l = (dd > 0 ? dd : 0); l < w && l - dd < L; ++l)
                                    cw += (double)S2[(l * Ks + kp) * ld + (l - dd) * Ks + k];
                                accd += (double)d * cw;
                            }
                        }
                        qeff[col] += (S)accd;
                    }
                }
            }
            __syncthreads();
            // ---- sweep: the sequential recurrence of component k over this chunk (warp 0), entirely in shared
            //      memory: H of the chunk is prefetched by all threads, results are written back by all threads
            for (int col = tid; col < HW_TC; col += nthr) {
                const int64_t tp = t0 + col;
                hch[col] = (tp < T) ? H[tp * K + k] : S(0);
            }
            __syncthreads();
            if (tid < 32) {
                const int lane = tid;
                const int n = (int)((t0 + HW_TC < T) ? HW_TC : T - t0);
                int i = 0;
                if (L <= 32 && !ring_mode) {
                    // register-window recurrence over whole blocks of 32 interior columns
                    const S c0i = ckk[0], inv_i = S(1) / (c0i + (S)CMF_EPS + l2);
                    while (i + 32 <= n && t0 + i + 32 <= Tint) {
                        if (sizeof(S) == 4) hals_recurrence_block<S, 32>(hch, qeff, Pw, creg, c0i, inv_i, l1, i, lane);   // table in registers
                        else hals_recurrence_block<S, 32>(hch, qeff, Pw, ckk32, c0i, inv_i, l1, i, lane);                  // fp64: table in shared memory
                        i += 32;
                    }
                    if (i < n) {
                        // the rest (truncated tail of the sequence / partial block) runs on the shared ring: hand the window over
                        int slot0 = (int)((t0 + i) % RB);
                        if (lane == 0) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) { int ps = slot0 + j; if (ps >= RB) ps -= RB; pend[ps] = Pw[j]; }
                        }
                        ring_mode = true;
                        __syncwarp();
                    }
                }
                {
                int slot = (int)((t0 + i) % RB);
                for (; i < n; ++i) {
                    const int64_t t = t0 + i;
                    const int w = (int)((T - t < L) ? (T - t) : L);
                    const S c0 = (w == (int)L) ? ckk[0] : tailC[w * L + 0];
                    const S h = hch[i];
                    const S q = qeff[i] + pend[slot];
                    S v = (h * c0 - q - l1) / (c0 + (S)CMF_EPS + l2);
                    v = v > S(0) ? v : S(0);
                    const S d = v - h;
                    __syncwarp();
                    if (lane == 0) {
                        hch[i] = v;
                        qeff[i] = d;            // Delta H of this column (qeff[i] is dead now)
                        pend[slot] = S(0);
                    }
                    if (d != S(0)) {
                        const S *ctab = (w == (int)L) ? ckk : tailC + (size_t)w * L;
                        for (int sft = 1 + lane; sft < w; sft += 32) {
                            int ps = slot + sft;
                            if (ps >= RB) ps -= RB;
                            pend[ps] += d * ctab[sft];
                        }
                    }
                    if (++slot == RB) slot = 0;
                    __syncwarp();
                }
                }
            }
            __syncthreads();
            for (int col = tid; col < HW_TC; col += nthr) {
                const int64_t tp = t0 + col;
                if (tp < T) {
                    H[tp * K + k] = hch[col];
                    D[tp * K + k] = qeff[col];
                }
            }
            __syncthreads();
            // ---- publish (every thread fences its own H / Delta stores, then one thread raises the counter)
            __threadfence();
            __syncthreads();
            if (tid == 0) atomicExch(progress + k, (int)(c + 1));
        }
        __syncthreads();
    }
}

// Projected gradient descent pieces (src/algs/pgd.jl:224-255, SquareLoss):
//   g = 2*(den - num) + 2*l2*x + l1*sign(x)      gradient of ||conv - X||^2 plus Square/Absolute penalties (:30-32,:77-88)
//   x = max(eps, x - step/(||g|| + eps) * g)      descent step and NonnegConstraint projection (:236-240,:93-95)
template <typename S>
__global__ void pgd_grad_kernel(S *g, const S *den, const S *num, const S *__restrict__ x, S l1, S l2, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const S xv = x[i];
    const S sg = xv > S(0) ? S(1) : (xv < S(0) ? S(-1) : S(0));
    g[i] = S(2) * (den[i] - num[i]) + S(2) * l2 * xv + l1 * sg;      // g may alias den
}
// g += 2*l2*x + l1*sign(x): the Square / Absolute penalties on top of a gradient that is already in g (pgd.jl:77-88)
template <typename S>
__global__ void pgd_penalty_kernel(S *g, const S *__restrict__ x, S l1, S l2, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const S v = x[i];
    g[i] += S(2) * l2 * v + l1 * (v > S(0) ? S(1) : (v < S(0) ? S(-1) : S(0)));
}

// pgd.jl:236-241: x -= step / (||g|| + eps) * g, then the projection: NonnegConstraint (x = max(eps, x), :93-95) here, or
// nothing here and unit_norm_* below for UnitNormConstraint (:98-110)
template <typename S>
__global__ void pgd_step_kernel(S *__restrict__ x, const S *__restrict__ g, double step, const double *__restrict__ nrm2, int64_t n,
                                int nonneg) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const S alpha = (S)(step / (sqrt(nrm2[0]) + CMF_EPS));
    const S v = x[i] - alpha * g[i];
    x[i] = (!nonneg || v > (S)CMF_EPS) ? v : (S)CMF_EPS;
}

// UnitNormConstraint (pgd.jl:98-110): every slice along the first Julia dimension (component k) with ||slice|| > 1 is divided by
// its norm.  Element e of component k lives at ((e / inner) * K + k) * inner + e % inner  (W: inner = N, rows (l, k); H: inner = 1).
// grid (UN_CHUNKS, K): fixed chunks and a fixed summation order -> deterministic.
constexpr int UN_CHUNKS = 64;
template <typename S>
__global__ void __launch_bounds__(256) unit_norm_partial_kernel(const S *__restrict__ x, double *__restrict__ part, int64_t K, int64_t inner,
                                                                 int64_t cnt) {
    __shared__ double red[256];
    const int64_t k = blockIdx.y, per = (cnt + UN_CHUNKS - 1) / UN_CHUNKS, e0 = (int64_t)blockIdx.x * per, e1 = min(cnt, e0 + per);
    double acc = 0.0;
    for (int64_t e = e0 + threadIdx.x; e < e1; e += 256) {
        const double v = (double)x[((e / inner) * K + k) * inner + e % inner];
        acc += v * v;
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) part[k * UN_CHUNKS + blockIdx.x] = red[0];
}
template <typename S>
__global__ void unit_norm_apply_kernel(S *__restrict__ x, const double *__restrict__ part, int64_t K, int64_t inner, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t k = (i / inner) % K;
    double ss = 0.0;
    for (int c = 0; c < UN_CHUNKS; ++c) ss += part[k * UN_CHUNKS + c];
    const double mag = sqrt(ss);
    if (mag > 1.0) x[i] = (S)((double)x[i] / mag);
}

// x[i] = a[i] - b[i]   (P = denomW - numW, Q = denomH - numH: the HALS gradients from the MU quantities)
template <typename S>
__global__ void sub_kernel(S *x, const S *a, const S *b, int64_t n) {   // x may alias a or b
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = a[i] - b[i];
}

}  // namespace cmf
