// Frequency-domain engine: the two data-sized contractions of the fit path,
//   numH[k,t]   = sum_l sum_n W[k,n,l] X[n,t+l]      (src/common.jl:71-81, called at src/algs/mult.jl:47)
//   numW[k,n,l] = sum_t H[k,t] X[n,t+l]              (src/algs/mult.jl:31-34)
// are correlations along t, so in overlap-save blocks of length B (hop V = B-L+1) they become, per frequency f, one
// small complex matrix product over the spectrum of X:
//   numH^[k,b,f] = sum_n conj(W^[k,n,f]) X^[n,b,f]          numW^[k,n,f] = sum_b conj(Hz^[k,b,f]) X^[n,b,f]
// (Hz = the V owned columns of block b, zero padded to B).  That cuts 2NKLT flops to ~8NKT(B/V) and makes the path
// HBM-bound on the spectrum of X, which is constant over the fit and computed once (the circular-convolution idea of
// src/common.jl:36-50, made exact by overlap-save).  The complex products run as real GEMMs on the tcgen05 kernel
// (kernels_tc.cuh, modes TC_FQT / TC_FQC) with split-bf16 operands; this file holds the SIMT FFT kernels around them.
//
// Layouts (bf16 hi/lo planes unless noted; c = 0 real part, 1 imaginary part; rows m = k real, m = Kq + k imaginary, Kq = 64 or 128):
//   Xf [f][b][c][n]          B operand of both products (K-major for TC_FQT, MN-major for TC_FQC)
//   Aw [f][m][c][n]          conj(W^) as the real 128 x 2N matrix [[Wr, Wi], [-Wi, Wr]]          (A of TC_FQT)
//   Ah [f][b][c][m]          conj(Hz^) as the real 2nblk x 128 matrix, rows (b,c): [Hr | -Hi], [Hi | Hr]  (A of TC_FQC)
//   Of [f][b][m]   fp32      numH^ (output of TC_FQT)
//   Df [f][m][n]   fp32      numW^ (output of TC_FQC)
// The Gram cross-correlation of H (Rg[d][k][k'] = sum_u H[k,u] H[k',u+d], the Toeplitz part of Htilde Htilde', mult.jl:28,33)
// is the same product with the spectrum of H itself as the B operand:
//   Hf [f][b][c][k']         full blocks of H (owned columns + right halo), 64 columns per row    (B of TC_FQC)
//   Gf [f][m][k']  fp32      Rg^ (output of TC_FQC)
// and denomH = C (*) H (mult.jl:44,48 in Gram form: 2L-1 lags of the K x K table C over H with both halos) is the numH
// product with N -> K: blocks of hop V2 = B-2L+2 starting L-1 columns early,
//   Ac [f][m][c][k']         conj(C^) as the real 128 x 128 matrix                                 (A of TC_FQT)
//   Hf [f][b][c][k']         full blocks of H (same layout as above, other blocking)               (B of TC_FQT)
// The direct loss ||conv(W,H) - X||^2 (mult.jl:55-57) goes the other way: Xhat^[n,b,f] = sum_k W^[k,n,f] H^[k,b,f] over full
// blocks of H that start L-1 columns early (hop V), inverse transform, the last V samples of a block are exact:
//   Awm[f][co][c][k][n]      W^ as the real matrices [Wr | -Wi] (co = re) and [Wi | Wr] (co = im), n contiguous (A of TC_FQX)
//   Yf [f][b][co][n] fp32    Xhat^ for a chunk of blocks (output of TC_FQX) -> ifft_resid_kernel subtracts X and sums squares
//
// FFT: in-place radix-2 decimation-in-frequency (two stages fused per pass) in shared memory over a tile d[B][C] of C
// independent complex columns (column index fastest: conflict-free), output in bit-reversed order.  Two real sequences ride in one complex transform
// (z = a + i b; A[f] = (Z[f] + conj(Z[B-f]))/2, B[f] = (Z[f] - conj(Z[B-f]))/(2i)), forward and inverse.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cmf {
namespace fd {

#ifndef CMF_FD_MINB
#define CMF_FD_MINB 3        // CTAs per SM the transforms are compiled for (3 x 512 threads: 40 registers per thread)
#endif
constexpr int LD_U = 8;      // global loads a thread keeps in flight while it fills / drains the shared-memory tile
constexpr int NT = 512;      // threads per CTA (A/B at c4: 256 -> 49, 512 -> 44, 1024 -> 50 ms per iteration)
constexpr int KQ_MAX = 128;  // components are padded to Kq = 64 or 128; the A operands / outputs have MROWS = 2 Kq rows per
                             // frequency (m = k real part, m = Kq + k imaginary part), i.e. one or two 128-row tensor-core tiles

// Every transform is a template on log2(B) and the tile width C (complex columns per CTA), so strides, pass count, the
// radix-4 / radix-2 tail and the bit reversals are constants.  The host instantiates B = 64 .. 1024 and C = 8, 16, 32
// (fd_dispatch in cmf_sm100.cu).
//
// Arithmetic runs on the packed fp32x2 pipe (FADD2 / FMUL2 / FFMA2).  Each lane does the same IEEE operation, in the same
// order and with the same fused multiply-adds, as the scalar code these kernels replaced, so the spectra are bit for bit
// what they were: a complex twiddle product rounds a.y*w.y and a.x*w.y and fuses a.x*w.x, a.y*w.x; the eighth-root
// products of the radix-8 stage 1 meet in stage 2 as (u5 * r) +- round(v7 * r); the residual of the loss pass is
// fma(z, 1/B, -x).
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 bcast(float x) { return make_float2(x, x); }

// full-circle table tw[m] = exp(-2 pi i m / B), m < B (the radix-8 passes index it up to 7B/8): computed once per handle
// (FdState::tw), copied into shared memory by every CTA of the transforms.  grid ceil(B / 256) x 256.
__global__ void twiddle_kernel(float2 *__restrict__ tw, int B) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m < B) {
        float s, c;
        sincospif(-2.0f * (float)m / (float)B, &s, &c);
        tw[m] = make_float2(c, s);
    }
}
template <int B>
__device__ __forceinline__ void load_twiddles(float2 *tw, const float2 *__restrict__ twg) {
#pragma unroll
    for (int m = threadIdx.x; m < B; m += NT) tw[m] = twg[m];
}

// 1-D grid over (block, tile): nbx = number of blocks when the block index runs fastest, 0 = the tile index runs fastest (ny
// tiles).  One 32-bit division for both indices.
__device__ __forceinline__ void grid_block_tile(int64_t nbx, int ny, int &blk, int &tile) {
    const unsigned dv = nbx ? (unsigned)nbx : (unsigned)ny, q = blockIdx.x / dv, r = blockIdx.x - q * dv;
    blk = (int)(nbx ? r : q);
    tile = (int)(nbx ? q : r);
}

template <int LOGB> __device__ __forceinline__ int rev(int x) { return (int)(__brev((unsigned)x) >> (32 - LOGB)); }

// a * w (INV: a * conj(w)), rounding a.y*w.y and a.x*w.y, fusing the other two products
template <bool INV> __device__ __forceinline__ float2 twmul(float2 a, float2 w) {
    const float2 t = mul2(make_float2(a.y, a.x), INV ? make_float2(w.y, -w.y) : make_float2(-w.y, w.y));
    return fma2(a, bcast(w.x), t);
}
// multiplication by -i (forward) / +i (inverse); the sums that the eighth roots w8 = exp(-+ i pi / 4), w8^3 scale by 1/sqrt(2)
template <bool INV> __device__ __forceinline__ float2 mul_mi(float2 a) { return INV ? make_float2(-a.y, a.x) : make_float2(a.y, -a.x); }
template <bool INV> __device__ __forceinline__ float2 w8_sum(float2 a) {
    return INV ? add2(make_float2(a.x, a.x), make_float2(-a.y, a.y)) : add2(a, make_float2(a.y, -a.x));
}
template <bool INV> __device__ __forceinline__ float2 w83_sum(float2 a) {
    return INV ? add2(make_float2(-a.x, a.x), make_float2(-a.y, -a.y)) : add2(make_float2(a.y, -a.x), make_float2(-a.x, -a.y));
}

// log2(B) radix-2 decimation-in-frequency stages over d[B][C], in place, output in bit-reversed order (X[f] ends up in row
// rev(f)), THREE stages fused per pass: a thread holds the 8 rows {pos + j n/8} of one block of size n in registers, runs the
// radix-8 butterfly with the constant eighth roots, and applies the position twiddles on the way out (row m of the butterfly
// carries w_n^(pos * bitrev3(m)): 7 table reads per 8 points).  B = 512 is three such passes; what is left of log2(B) after
// the radix-8 passes (blocks of 4 or 2 rows, all twiddles 1) is one radix-4 or radix-2 pass.  INV conjugates every root.
// The passes are unrolled (strides are immediates); a thread's butterflies within a pass are not: unrolled, they hold more
// rows in registers than 40 allow and spill.
template <bool INV, int LOGB, int C>
__device__ __forceinline__ void fft_passes(float2 *d, const float2 *tw) {
    constexpr int B = 1 << LOGB, JSTEP = NT / C;
    const float2 rr = bcast(0.70710678118654752f);
    const int c = threadIdx.x % C, j0 = threadIdx.x / C;
#pragma unroll
    for (int s = 0; s + 2 < LOGB; s += 3) {
        const int lq = LOGB - s - 3, q = 1 << lq, qC = q * C;             // eighth of the block size n = B >> s
#pragma unroll 1
        for (int jj = 0; jj < (B / 8 + JSTEP - 1) / JSTEP; ++jj) {
            const int j = j0 + jj * JSTEP;
            if ((B / 8) % JSTEP != 0 && j >= B / 8) break;
            const int pos = j & (q - 1), g = j >> lq;
            float2 *r = d + ((g << (lq + 3)) + pos) * C + c;
            float2 a0 = r[0], a1 = r[qC], a2 = r[2 * qC], a3 = r[3 * qC], a4 = r[4 * qC], a5 = r[5 * qC], a6 = r[6 * qC], a7 = r[7 * qC];
            // stage 1: rows j and j+4, constant root w8^j on the difference (rows 5 and 7 keep the unscaled sums u5, v7)
            float2 t, u5, v7;
            t = sub2(a0, a4); a0 = add2(a0, a4); a4 = t;
            t = sub2(a1, a5); a1 = add2(a1, a5); u5 = w8_sum<INV>(t);
            t = sub2(a2, a6); a2 = add2(a2, a6); a6 = mul_mi<INV>(t);
            t = sub2(a3, a7); a3 = add2(a3, a7); v7 = mul2(w83_sum<INV>(t), rr);
            // stage 2: rows j and j+2 inside each half, constant root w4^j
            t = sub2(a0, a2); a0 = add2(a0, a2); a2 = t;
            t = sub2(a1, a3); a1 = add2(a1, a3); a3 = mul_mi<INV>(t);
            t = sub2(a4, a6); a4 = add2(a4, a6); a6 = t;
            t = fma2(u5, rr, make_float2(-v7.x, -v7.y)); a5 = fma2(u5, rr, v7); a7 = mul_mi<INV>(t);
            // stage 3: neighbouring rows
            t = sub2(a0, a1); a0 = add2(a0, a1); a1 = t;
            t = sub2(a2, a3); a2 = add2(a2, a3); a3 = t;
            t = sub2(a4, a5); a4 = add2(a4, a5); a5 = t;
            t = sub2(a6, a7); a6 = add2(a6, a7); a7 = t;
            if (lq > 0) {                                                  // position twiddles (all 1 in the last radix-8 pass of 8^m)
                const int e = pos << s;
                a1 = twmul<INV>(a1, tw[4 * e]); a2 = twmul<INV>(a2, tw[2 * e]); a3 = twmul<INV>(a3, tw[6 * e]);
                a4 = twmul<INV>(a4, tw[e]);     a5 = twmul<INV>(a5, tw[5 * e]); a6 = twmul<INV>(a6, tw[3 * e]);
                a7 = twmul<INV>(a7, tw[7 * e]);
            }
            r[0] = a0; r[qC] = a1; r[2 * qC] = a2; r[3 * qC] = a3; r[4 * qC] = a4; r[5 * qC] = a5; r[6 * qC] = a6; r[7 * qC] = a7;
        }
        __syncthreads();
    }
    if constexpr (LOGB % 3 == 2) {                                        // blocks of 4 rows: pos = 0, twiddles 1
#pragma unroll
        for (int jj = 0; jj < (B / 4 + JSTEP - 1) / JSTEP; ++jj) {
            const int j = j0 + jj * JSTEP;
            if ((B / 4) % JSTEP != 0 && j >= B / 4) break;
            float2 *r = d + (4 * j) * C + c;
            float2 a0 = r[0], a1 = r[C], a2 = r[2 * C], a3 = r[3 * C], t;
            t = sub2(a0, a2); a0 = add2(a0, a2); a2 = t;
            t = sub2(a1, a3); a1 = add2(a1, a3); a3 = mul_mi<INV>(t);
            r[0] = add2(a0, a1); r[C] = sub2(a0, a1); r[2 * C] = add2(a2, a3); r[3 * C] = sub2(a2, a3);
        }
        __syncthreads();
    } else if constexpr (LOGB % 3 == 1) {                                 // blocks of 2 rows
#pragma unroll
        for (int jj = 0; jj < (B / 2 + JSTEP - 1) / JSTEP; ++jj) {
            const int j = j0 + jj * JSTEP;
            if ((B / 2) % JSTEP != 0 && j >= B / 2) break;
            float2 *r0 = d + (2 * j) * C + c, *r1 = r0 + C;
            const float2 a = *r0, b = *r1;
            *r0 = add2(a, b);
            *r1 = sub2(a, b);
        }
        __syncthreads();
    }
}

// spectra of the two real sequences packed in one complex transform at frequency f: A = (ar, ai), B = (br, bi), returned as
// the pairs (ar, br) and (ai, bi)
template <int LOGB, int C>
__device__ __forceinline__ void unpack_pair(const float2 *d, int f, int p, float2 &re, float2 &im) {
    constexpr int B = 1 << LOGB;
    const float2 z = d[rev<LOGB>(f) * C + p], y = d[rev<LOGB>((B - f) & (B - 1)) * C + p];
    const float2 sm = add2(z, y), df = sub2(z, y);
    re = mul2(sm, bcast(0.5f));                                          // (0.5 (z.x + y.x), 0.5 (z.y + y.y))
    im = mul2(make_float2(df.y, df.x), make_float2(0.5f, -0.5f));         // (0.5 (z.y - y.y), -0.5 (z.x - y.x))
}

// the inverse of unpack_pair: rows f and B-f of Z = A + iB from the half spectra A = (re.x, im.x), B = (re.y, im.y)
template <int LOGB, int C>
__device__ __forceinline__ void pack_pair(float2 *d, int f, int p, float2 re, float2 im) {
    constexpr int B = 1 << LOGB;
    if (f == 0 || f == B / 2) im = make_float2(0.f, 0.f);          // real sequences: these bins are real
    const float2 v = make_float2(im.y, im.x);
    const float2 sm = add2(re, v), df = sub2(re, v);                 // (re.x + im.y, re.y + im.x), (re.x - im.y, re.y - im.x)
    d[f * C + p] = make_float2(df.x, sm.y);
    if (f > 0 && f < B / 2) d[(B - f) * C + p] = make_float2(sm.x, df.y);
}

// (a, b) -> packed bf16 pairs hi = bf16(x), lo = bf16(x - hi) (round to nearest, as tc::split_bf16)
__device__ __forceinline__ void split2(float2 ab, uint32_t &h, uint32_t &l) {
    const __nv_bfloat162 hh = __floats2bfloat162_rn(ab.x, ab.y);
    const float2 lf = sub2(ab, __bfloat1622float2(hh));
    const __nv_bfloat162 ll = __floats2bfloat162_rn(lf.x, lf.y);
    h = *reinterpret_cast<const uint32_t *>(&hh);
    l = *reinterpret_cast<const uint32_t *>(&ll);
}
__device__ __forceinline__ void store_split2(__nv_bfloat16 *hi, __nv_bfloat16 *lo, int64_t idx, float2 ab) {
    uint32_t h, l;
    split2(ab, h, l);
    *reinterpret_cast<uint32_t *>(hi + idx) = h;
    *reinterpret_cast<uint32_t *>(lo + idx) = l;
}

// X[t][N] fp32 (xcols rows) -> Xf.  grid nblkp * ceil(N/32) (1-D); 16 complex columns = 32 units per CTA.
template <int LOGB>
__global__ void __launch_bounds__(NT, CMF_FD_MINB)
fft_x_kernel(const float *__restrict__ X, __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo, int64_t N, int64_t xcols,
             int V, int64_t nblkp, int64_t nbx, const float2 *__restrict__ twg) {
    constexpr int B = 1 << LOGB, C = 16, ISTEP = NT / C;
    extern __shared__ float2 fd_smem[];
    float2 *d = fd_smem, *tw = fd_smem + B * C;
    int b, tile;                                      // 1-D grid over (block, unit tile)
    grid_block_tile(nbx, (int)((N + 31) / 32), b, tile);
    const int p = threadIdx.x % C;
    const int n = tile * 32 + 2 * p;
    load_twiddles<B>(tw, twg);
    {
        // LD_U rows per thread are requested before any is stored: the transforms are bound by the latency of these loads, not by
        // bandwidth or issue slots (profiles/r2_ncu_fft_kernels.md), so memory-level parallelism is what counts
        const int i0 = threadIdx.x / C;
        const int64_t lim64 = xcols - (int64_t)b * V;
        const int lim = (n < N) ? (int)(lim64 < 0 ? 0 : (lim64 > B ? B : lim64)) : 0;
        const float *src = X + ((int64_t)b * V + i0) * N + n;
        float2 *dst = d + i0 * C + p;
#pragma unroll 1
        for (int i = i0; i < B; i += LD_U * ISTEP, src += (int64_t)LD_U * ISTEP * N, dst += LD_U * ISTEP * C) {
            float2 v[LD_U];
#pragma unroll
            for (int u = 0; u < LD_U; ++u) {
                v[u] = make_float2(0.f, 0.f);
                if (i + u * ISTEP < lim) v[u] = *reinterpret_cast<const float2 *>(src + (int64_t)u * ISTEP * N);
            }
#pragma unroll
            for (int u = 0; u < LD_U; ++u)
                if (B % (LD_U * ISTEP) == 0 || i + u * ISTEP < B) dst[u * ISTEP * C] = v[u];
        }
    }
    __syncthreads();
    fft_passes<false, LOGB, C>(d, tw);
    if (n >= N) return;
    for (int f = threadIdx.x / C; f <= B / 2; f += NT / C) {
        float2 re, im;
        unpack_pair<LOGB, C>(d, f, p, re, im);
        const int64_t r = ((int64_t)f * nblkp + b) * 2;
        store_split2(hi, lo, r * N + n, re);
        store_split2(hi, lo, (r + 1) * N + n, im);
    }
}

// H[t][K] fp32 (owned column 0 first; block b starts at column b*V + t_off, t_off <= 0 reaches into the left halo).
// full == 0: only the V owned columns of each block, zero padded -> Ah;
// full != 0: whole blocks over the columns present, t < hcols = Tl + L-1 (owned + right halo) -> Hf.
// grid nblkp * (kq / 2 / C) (1-D); C complex columns = 2C components per CTA.
template <int LOGB, int C>
__global__ void __launch_bounds__(NT, CMF_FD_MINB)
fft_h_kernel(const float *__restrict__ H, __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo, int64_t K, int64_t Tl,
             int64_t hcols, int V, int64_t nblkp, int full, int64_t t_off, int kq, int64_t nbx,
             const float2 *__restrict__ twg) {
    constexpr int B = 1 << LOGB, ISTEP = NT / C;
    const int64_t KQ = kq, MROWS = 2 * kq;
    extern __shared__ float2 fd_smem[];
    float2 *d = fd_smem, *tw = fd_smem + B * C;
    int bi, tile;                                     // 1-D grid over (block, component tile)
    grid_block_tile(nbx, (kq / 2) / C, bi, tile);
    const int64_t b = bi;
    const int p = threadIdx.x % C;
    const int k = 2 * (tile * C + p);
    load_twiddles<B>(tw, twg);
    {
        const int i0 = threadIdx.x / C;
        const int64_t tb = b * V + t_off;
        // rows of the block that hold data: [0, lim) (owned segment, or whatever of the block lies before hcols)
        const int64_t lim64 = full ? (hcols - tb) : ((Tl - tb < V) ? Tl - tb : V);
        const int lim = (int)(lim64 < 0 ? 0 : (lim64 > B ? B : lim64));
        const float *src = H + (tb + i0) * K + k;
        float2 *dst = d + i0 * C + p;
        const bool pair = ((K & 1) == 0) && (k + 1 < K);
#pragma unroll 1
        for (int i = i0; i < B; i += LD_U * ISTEP, src += (int64_t)LD_U * ISTEP * K, dst += LD_U * ISTEP * C) {
            float2 v[LD_U];
#pragma unroll
            for (int u = 0; u < LD_U; ++u) {
                v[u] = make_float2(0.f, 0.f);
                if (i + u * ISTEP < lim) {
                    const float *q = src + (int64_t)u * ISTEP * K;
                    if (pair) v[u] = *reinterpret_cast<const float2 *>(q);
                    else { if (k < K) v[u].x = q[0]; if (k + 1 < K) v[u].y = q[1]; }
                }
            }
#pragma unroll
            for (int u = 0; u < LD_U; ++u)
                if (B % (LD_U * ISTEP) == 0 || i + u * ISTEP < B) dst[u * ISTEP * C] = v[u];
        }
    }
    __syncthreads();
    fft_passes<false, LOGB, C>(d, tw);
    // row of frequency f: ((f * nblkp + b) * 2) * (full ? KQ : MROWS) + k; f advances by NT / C per step
    const int64_t rs = full ? 2 * KQ : 2 * MROWS;
    const int64_t rstep = (int64_t)(NT / C) * nblkp * rs;
    int64_t r = ((int64_t)(threadIdx.x / C) * nblkp + b) * rs + k;
    for (int f = threadIdx.x / C; f <= B / 2; f += NT / C, r += rstep) {
        float2 re, im;
        unpack_pair<LOGB, C>(d, f, p, re, im);
        uint32_t hr, lr, hi_, li_;
        split2(re, hr, lr);
        split2(im, hi_, li_);
        if (full) {
            *reinterpret_cast<uint32_t *>(hi + r) = hr; *reinterpret_cast<uint32_t *>(lo + r) = lr;
            *reinterpret_cast<uint32_t *>(hi + r + KQ) = hi_; *reinterpret_cast<uint32_t *>(lo + r + KQ) = li_;
            continue;
        }
        const uint32_t sg = 0x80008000u;                           // -x of a packed bf16 pair (hi and lo planes alike)
        *reinterpret_cast<uint32_t *>(hi + r) = hr; *reinterpret_cast<uint32_t *>(lo + r) = lr;                                 // row (b, re): [ Hr | -Hi ]
        *reinterpret_cast<uint32_t *>(hi + r + KQ) = hi_ ^ sg; *reinterpret_cast<uint32_t *>(lo + r + KQ) = li_ ^ sg;
        *reinterpret_cast<uint32_t *>(hi + r + MROWS) = hi_; *reinterpret_cast<uint32_t *>(lo + r + MROWS) = li_;               // row (b, im): [ Hi |  Hr ]
        *reinterpret_cast<uint32_t *>(hi + r + MROWS + KQ) = hr; *reinterpret_cast<uint32_t *>(lo + r + MROWS + KQ) = lr;
    }
}

// Wi[(l*K+k)][N] fp32 -> Aw (rows of ldw elements, imaginary block at column coff: 2N / N for W; 128 / 64 for the
// K x K lag table C with N = K and L = 2L-1 lags -> Ac).  grid (ceil(N / 2C), K): C complex columns = 2C units per CTA.
template <int LOGB, int C>
__global__ void __launch_bounds__(NT, CMF_FD_MINB)
fft_w_kernel(const float *__restrict__ Wi, __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo, int64_t N, int64_t K,
             int64_t L, int64_t ldw, int64_t coff, int xmode, int kq, const float2 *__restrict__ twg) {
    constexpr int B = 1 << LOGB, ISTEP = NT / C;
    const int64_t KQ = kq, MROWS = 2 * kq;
    extern __shared__ float2 fd_smem[];
    float2 *d = fd_smem, *tw = fd_smem + B * C;
    const int64_t k = blockIdx.y;
    const int p = threadIdx.x % C;
    const int64_t n = (int64_t)blockIdx.x * (2 * C) + 2 * p;
    load_twiddles<B>(tw, twg);
    {
        const int i0 = threadIdx.x / C;
        const float *src = Wi + ((int64_t)i0 * K + k) * N + n;
        float2 *dst = d + i0 * C + p;
#pragma unroll 1
        for (int i = i0; i < B; i += LD_U * ISTEP, src += (int64_t)LD_U * ISTEP * K * N, dst += LD_U * ISTEP * C) {
            float2 v[LD_U];
#pragma unroll
            for (int u = 0; u < LD_U; ++u) {
                const int ii = i + u * ISTEP;
                v[u] = make_float2(0.f, 0.f);
                if (ii < L && n < N) {
                    const float *q = src + (int64_t)u * ISTEP * K * N;
                    if ((N & 1) == 0) v[u] = *reinterpret_cast<const float2 *>(q);
                    else { v[u].x = q[0]; if (n + 1 < N) v[u].y = q[1]; }
                }
            }
#pragma unroll
            for (int u = 0; u < LD_U; ++u)
                if (B % (LD_U * ISTEP) == 0 || i + u * ISTEP < B) dst[u * ISTEP * C] = v[u];
        }
    }
    __syncthreads();
    fft_passes<false, LOGB, C>(d, tw);
    if (n >= N) return;
    for (int f = threadIdx.x / C; f <= B / 2; f += NT / C) {
        float2 re, im;
        unpack_pair<LOGB, C>(d, f, p, re, im);
        const float2 nim = make_float2(-im.x, -im.y);
        if (xmode) {                                               // Awm[f][co][c][k][n]: re = [Wr | -Wi], im = [Wi | Wr]
            const int64_t r0 = (((int64_t)f * 2 + 0) * MROWS + k) * N + n, r1 = r0 + MROWS * N;
            store_split2(hi, lo, r0, re);
            store_split2(hi, lo, r0 + KQ * N, nim);
            store_split2(hi, lo, r1, im);
            store_split2(hi, lo, r1 + KQ * N, re);
            continue;
        }
        const int64_t rw = ((int64_t)f * MROWS + k) * ldw + n, iw = rw + KQ * ldw;
        store_split2(hi, lo, rw, re);                              // row k:      [  Wr | Wi ]
        store_split2(hi, lo, rw + coff, im);
        store_split2(hi, lo, iw, nim);                             // row 64 + k: [ -Wi | Wr ]
        store_split2(hi, lo, iw + coff, re);
    }
}

// Of[f][b][m] fp32 -> numH[t][K] (owned columns; V valid outputs per block).  grid nblk * (kq / 2 / C) (1-D).
template <int LOGB, int C>
__global__ void __launch_bounds__(NT, CMF_FD_MINB)
ifft_numH_kernel(const float *__restrict__ Of, float *__restrict__ numH, int64_t K, int64_t Tl, int V, int64_t nblkp, int kq,
                 int64_t nbx, const float2 *__restrict__ twg) {
    constexpr int B = 1 << LOGB, FSTEP = NT / C;
    const int64_t KQ = kq, MROWS = 2 * kq;
    extern __shared__ float2 fd_smem[];
    float2 *d = fd_smem, *tw = fd_smem + B * C;
    int bi, tile;                                     // 1-D grid over (block, component tile)
    grid_block_tile(nbx, (kq / 2) / C, bi, tile);
    const int64_t b = bi;
    const int p = threadIdx.x % C;
    const int k = 2 * (tile * C + p);
    load_twiddles<B>(tw, twg);
    {
        const int f0 = threadIdx.x / C;
        const int64_t ustep = (int64_t)FSTEP * nblkp * MROWS;
        const float *o = Of + ((int64_t)f0 * nblkp + b) * MROWS + k;
#pragma unroll 1
        for (int f = f0; f <= B / 2; f += 4 * FSTEP, o += 4 * ustep) {
            float2 re[4], im[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (f + u * FSTEP <= B / 2) {
                    const float *q = o + u * ustep;
                    re[u] = *reinterpret_cast<const float2 *>(q); im[u] = *reinterpret_cast<const float2 *>(q + KQ);
                }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (f + u * FSTEP <= B / 2) pack_pair<LOGB, C>(d, f + u * FSTEP, p, re[u], im[u]);
        }
    }
    __syncthreads();
    fft_passes<true, LOGB, C>(d, tw);
    const float2 sc = bcast(1.0f / (float)B);
    const bool pair = ((K & 1) == 0) && (k + 1 < K);
    for (int i = threadIdx.x / C; i < V; i += NT / C) {
        const int64_t t = b * V + i;
        if (t >= Tl) break;
        const float2 z = mul2(d[rev<LOGB>(i) * C + p], sc);
        if (pair) *reinterpret_cast<float2 *>(numH + t * K + k) = z;
        else { if (k < K) numH[t * K + k] = z.x; if (k + 1 < K) numH[t * K + k + 1] = z.y; }
    }
}

// Yf[f][bc][co][n] fp32 (a chunk of nbc blocks starting at block b0) -> partial[bc * ceil(N/32) + unit tile] =
// sum over the V exact samples of the block and the CTA's 32 units of (Xhat - X)^2.  Block b covers the columns
// [b*V - (L-1), b*V - (L-1) + B) of H, so sample i >= L-1 of the inverse transform is Xhat at t = b*V + i - (L-1).
// grid nbc * ceil(N/32) (1-D).
template <int LOGB>
__global__ void __launch_bounds__(NT, CMF_FD_MINB)
ifft_resid_kernel(const float *__restrict__ Yf, const float *__restrict__ X, double *__restrict__ partial, int64_t N, int64_t Tl,
                  int64_t L, int V, int64_t nbc, int64_t b0, int64_t nbx, const float2 *__restrict__ twg) {
    constexpr int B = 1 << LOGB, C = 16, FSTEP = NT / C, ISTEP = NT / C;
    extern __shared__ float2 fd_smem[];
    __shared__ double red[NT / 32];
    float2 *d = fd_smem, *tw = fd_smem + B * C;
    const int ny = (int)((N + 31) / 32);
    int bc, by;                                       // 1-D grid over (block, unit tile)
    grid_block_tile(nbx, ny, bc, by);
    const int p = threadIdx.x % C;
    const int n = by * 32 + 2 * p;
    load_twiddles<B>(tw, twg);
    {
        const int f0 = threadIdx.x / C;
        const int64_t ustep = (int64_t)FSTEP * nbc * 2 * N;
        const float *y = Yf + (((int64_t)f0 * nbc + bc) * 2) * N + n;
#pragma unroll 1
        for (int f = f0; f <= B / 2; f += 4 * FSTEP, y += 4 * ustep) {
            float2 re[4], im[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                re[u] = make_float2(0.f, 0.f); im[u] = re[u];
                if (f + u * FSTEP <= B / 2 && n < N) {
                    const float *q = y + u * ustep;
                    re[u] = *reinterpret_cast<const float2 *>(q); im[u] = *reinterpret_cast<const float2 *>(q + N);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (f + u * FSTEP <= B / 2) pack_pair<LOGB, C>(d, f + u * FSTEP, p, re[u], im[u]);
        }
    }
    __syncthreads();
    fft_passes<true, LOGB, C>(d, tw);
    const float2 sc = bcast(1.0f / (float)B);
    double accd = 0.0;
    if (n < N) {
        // rows of this thread: i = L-1 + i0 + m*ISTEP; the X loads of 8 rows go out together, their squares are summed in fp32
        // and every group of 8 rows is added to the fp64 accumulator (same grouping as before)
        const int64_t tb = (b0 + bc) * (int64_t)V - (L - 1);
        const int lim = (int)(Tl - tb < B ? Tl - tb : B);                // rows of the block inside the shard
        const int i0 = (int)(L - 1) + threadIdx.x / C;
        const float *xs = X + (tb + i0) * N + n;
#pragma unroll 1
        for (int i = i0; i < B; i += LD_U * ISTEP, xs += (int64_t)LD_U * ISTEP * N) {
            float2 x[LD_U];
#pragma unroll
            for (int u = 0; u < LD_U; ++u) {
                x[u] = make_float2(0.f, 0.f);
                if (i + u * ISTEP < lim) x[u] = *reinterpret_cast<const float2 *>(xs + (int64_t)u * ISTEP * N);
            }
            float acc = 0.f;
#pragma unroll
            for (int u = 0; u < LD_U; ++u) {
                const int ii = i + u * ISTEP;
                if (ii < lim) {
                    const float2 r = fma2(d[rev<LOGB>(ii) * C + p], sc, make_float2(-x[u].x, -x[u].y));
                    acc = fmaf(r.x, r.x, acc);
                    acc = fmaf(r.y, r.y, acc);
                }
            }
            accd += (double)acc;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) accd += __shfl_xor_sync(0xffffffffu, accd, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = accd;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < NT / 32; ++w) s += red[w];
        partial[(int64_t)bc * ny + by] = s;
    }
}

// Df[f][m][n] fp32 (row stride ldi) -> out[(l*K+k)*N + n], l < L.  grid (ceil(N / 2C), K).
// OutT = float: numW (N even, paired stores);  OutT = double: the Gram partial Rg[d][k][k'] with N = K.
template <typename OutT, int LOGB, int C>
__global__ void __launch_bounds__(NT, CMF_FD_MINB)
ifft_numW_kernel(const float *__restrict__ Df, OutT *__restrict__ out, int64_t N, int64_t ldi, int64_t K, int64_t L, int kq,
                 const float2 *__restrict__ twg) {
    constexpr int B = 1 << LOGB, FSTEP = NT / C;
    const int64_t KQ = kq, MROWS = 2 * kq;
    extern __shared__ float2 fd_smem[];
    float2 *d = fd_smem, *tw = fd_smem + B * C;
    const int64_t k = blockIdx.y;
    const int p = threadIdx.x % C;
    const int64_t n = (int64_t)blockIdx.x * (2 * C) + 2 * p;
    load_twiddles<B>(tw, twg);
    {
        const int f0 = threadIdx.x / C;
        const int64_t ustep = (int64_t)FSTEP * MROWS * ldi;
        const float *src = Df + ((int64_t)f0 * MROWS + k) * ldi + n;
#pragma unroll 1
        for (int f = f0; f <= B / 2; f += 4 * FSTEP, src += 4 * ustep) {
            float2 re[4], im[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                re[u] = make_float2(0.f, 0.f); im[u] = re[u];
                if (f + u * FSTEP <= B / 2 && n < N) {
                    re[u] = *reinterpret_cast<const float2 *>(src + u * ustep);
                    im[u] = *reinterpret_cast<const float2 *>(src + u * ustep + KQ * ldi);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (f + u * FSTEP <= B / 2) pack_pair<LOGB, C>(d, f + u * FSTEP, p, re[u], im[u]);
        }
    }
    __syncthreads();
    fft_passes<true, LOGB, C>(d, tw);
    if (n >= N) return;
    const float2 sc = bcast(1.0f / (float)B);
    for (int l = threadIdx.x / C; l < L; l += NT / C) {
        const float2 z = mul2(d[rev<LOGB>(l) * C + p], sc);
        OutT *o = out + ((int64_t)l * K + k) * N + n;
        if (sizeof(OutT) == 4) {
            *reinterpret_cast<float2 *>(o) = z;
        } else {
            o[0] = (OutT)z.x;
            if (n + 1 < N) o[1] = (OutT)z.y;
        }
    }
}

}  // namespace fd
}  // namespace cmf
