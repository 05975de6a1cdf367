// Sparse-X contractions of the CNMF fit path (handles created with cmf_create_sparse), templated on the scalar type S.
//
// X is held twice on the device, both built once per data set by cmf_set_data_csc:
//   CSC  colptr[T+1] (int64), rowval[nnz] (int32), nzval[nnz]   -- column t = time bin t, rows increasing (numH)
//   CSR  rowptr[N+1] (int64), colidx[nnz] (int32), rval[nnz]    -- row n, times increasing               (numW)
// Every output element is written by exactly one thread and summed in double in a fixed order (no atomics), so the
// results are bit-identical from run to run.  The launch grids depend on N, T, C and L, never on nnz.
#pragma once
#include <cstdint>

namespace cmf {

constexpr int SP_WARPS = 8;        // warps per CTA of both contractions
constexpr int SP_A = 4;            // numW: (l, c) pairs per lane; a warp covers 32 * SP_A pairs of one row

// numW (mult.jl:32) on sparse X, split over time:
//   part[s][(l*C + c)*N + n] = sum over the nonzeros (n, t, x) of row n with t in [s*split_len, (s+1)*split_len), t >= l:
//                              x * H[(t-l)*ldh + c]
// One warp per (row n, chunk of 32*SP_A pairs q = l*C + c, split s): lane j owns the pairs q0 + 32a + j, the row's nonzeros
// of the split are walked in time order (warp-uniform loop) and the window H[t-l][c] is read by the 32 lanes together.
// reduce_partials_kernel adds the splits in order.  grid (ceil(N / SP_WARPS), ceil(L C / (32 SP_A)), nsplit).
template <typename S>
__global__ void __launch_bounds__(32 * SP_WARPS) sp_corr_kernel(const int64_t *__restrict__ rowptr, const int *__restrict__ colidx,
                                                                 const S *__restrict__ val, const S *__restrict__ H, int64_t ldh,
                                                                 int64_t C, int64_t L, int64_t N, int64_t split_len,
                                                                 double *__restrict__ part) {
    const int lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
    if (n >= N) return;
    const int64_t LC = L * C;
    const int64_t q0 = (int64_t)blockIdx.y * (32 * SP_A);
    int64_t lq[SP_A], cq[SP_A];
    double acc[SP_A];
#pragma unroll
    for (int a = 0; a < SP_A; ++a) {
        const int64_t q = q0 + 32 * a + lane;
        lq[a] = q < LC ? q / C : INT64_MAX;         // a pair past the end never contributes (t >= lq fails)
        cq[a] = q < LC ? q % C : 0;
        acc[a] = 0.0;
    }
    const int64_t t_lo = (int64_t)blockIdx.z * split_len, t_hi = t_lo + split_len;
    // first nonzero of the row at t >= t_lo (times increase along the row)
    int64_t lo = rowptr[n], hi = rowptr[n + 1];
    {
        int64_t a = lo, b = hi;
        while (a < b) {
            const int64_t m = (a + b) >> 1;
            if (colidx[m] < t_lo) a = m + 1; else b = m;
        }
        lo = a;
    }
    for (int64_t i = lo; i < hi; ++i) {
        const int64_t t = colidx[i];
        if (t >= t_hi) break;
        const double x = (double)val[i];
#pragma unroll
        for (int a = 0; a < SP_A; ++a)
            if (t >= lq[a]) acc[a] += x * (double)H[(t - lq[a]) * ldh + cq[a]];
    }
    double *p = part + (size_t)blockIdx.z * (size_t)(LC * N);
#pragma unroll
    for (int a = 0; a < SP_A; ++a) {
        const int64_t q = q0 + 32 * a + lane;
        if (q < LC) p[(size_t)q * N + n] = acc[a];
    }
}

// Wt[n][l*C + c] = Wi[(l*C + c)*N + n]: the K L weights of unit n contiguous, so the numH gather of one nonzero reads one
// row of Wt.  32 x 32 tiles through shared memory; grid (ceil(N / 32), ceil(L C / 32)), block (32, 8).
template <typename S>
__global__ void sp_w_transpose_kernel(const S *__restrict__ Wi, S *__restrict__ Wt, int64_t LC, int64_t N) {
    __shared__ S tile[32][33];
    const int64_t n0 = (int64_t)blockIdx.x * 32, j0 = (int64_t)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int64_t j = j0 + r, n = n0 + threadIdx.x;
        if (j < LC && n < N) tile[r][threadIdx.x] = Wi[j * N + n];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int64_t n = n0 + r, j = j0 + threadIdx.x;
        if (j < LC && n < N) Wt[n * LC + j] = tile[threadIdx.x][r];
    }
}

// numH (mult.jl:47) on sparse X:
//   out[t*ldo + c] = sum_{l < L, t+l < T} sum over the nonzeros (n, t+l, x) of column t+l:  x * Wt[n*LC + l*C + c]
// One warp per (column t, chunk of 32 components): lane = component, the CSC columns t .. t+L-1 (contiguous in colptr) are
// walked in order (warp-uniform loop), lag by lag.  grid (ceil(Tl / SP_WARPS), ceil(C / 32)).
template <typename S>
__global__ void __launch_bounds__(32 * SP_WARPS) sp_transconv_kernel(const int64_t *__restrict__ colptr, const int *__restrict__ rowval,
                                                                      const S *__restrict__ val, const S *__restrict__ Wt, int64_t C,
                                                                      int64_t L, int64_t Tl, int64_t T, S *__restrict__ out, int64_t ldo) {
    const int lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
    if (t >= Tl) return;
    const int64_t c = (int64_t)blockIdx.y * 32 + lane;
    const bool live = c < C;
    const int64_t LC = L * C;
    const int64_t l_hi = (T - t < L) ? T - t : L;
    double acc = 0.0;
    int64_t i = colptr[t];
    for (int64_t l = 0; l < l_hi; ++l) {
        const int64_t e = colptr[t + l + 1];
        const S *w = Wt + l * C + c;
        for (; i < e; ++i) {
            const double x = (double)val[i];
            if (live) acc += x * (double)w[(int64_t)rowval[i] * LC];
        }
    }
    if (live) out[t * ldo + c] = (S)acc;
}

// <numH_r, H_r> of every restart of a batch (the stacked [t][C] arrays, restart y = blockIdx.y owns the columns
// [off_r, off_r + K_r)): partial[y * gridDim.x + block] = a grid-stride slice of the sum, added in order by reduce_sum_kernel.
template <typename S>
__global__ void sp_seg_dot_partial_kernel(const S *__restrict__ a, const S *__restrict__ b, int64_t T, int64_t C,
                                          const BatchRest *__restrict__ tab, double *__restrict__ partial) {
    __shared__ double red[32];
    const BatchRest r = tab[blockIdx.y];
    const int64_t n = T * r.K;
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = (i / r.K) * C + r.off + i % r.K;
        acc += (double)a[j] * (double)b[j];
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) partial[(int64_t)blockIdx.y * gridDim.x + blockIdx.x] = acc;
}

}  // namespace cmf
