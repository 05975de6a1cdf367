// libcmf_sm100: C ABI + host orchestration of the B200 CNMF fit path (see include/cmf_sm100.h).
//
// One rank context (Ctx<S>) = one time-shard on one GPU; a handle holds one rank context, or one per device of a
// multi-GPU group.  All device memory is owned here; host arrays are copied during the call.  Errors never escape as C++ exceptions.
#include "../../include/cmf_sm100.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <numeric>
#include <mutex>
#include <tuple>
#include <stdexcept>
#include <string>
#include <vector>

#include <type_traits>
#include <variant>

#include "kernels_simt.cuh"
#include "kernels_tc.cuh"
#include "kernels_fd.cuh"
#include "kernels_hals.cuh"
#include "comm.h"

namespace {

thread_local std::string g_err;

struct CmfError : std::runtime_error {
    int code;
    CmfError(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            throw CmfError(CMF_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));     \
    } while (0)

#define REQUIRE(cond, msg)                                                                         \
    do {                                                                                           \
        if (!(cond)) throw CmfError(CMF_ERR_ARG, std::string(msg));                                \
    } while (0)

inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    void alloc(size_t count) {
        free();
        n = count;
        if (count) {
            CK(cudaMalloc(&p, count * sizeof(T)));
            // the zero-fill runs on the legacy default stream, which the handle's non-blocking stream is not ordered
            // against: wait for it here (allocation is never on the hot path)
            CK(cudaMemsetAsync(p, 0, count * sizeof(T), cudaStreamLegacy));
            CK(cudaStreamSynchronize(cudaStreamLegacy));
        }
    }
    void free() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
    ~DevBuf() { free(); }
};

// ------------------------------------------------------------------------------------------
// rank context: the state of one time-shard on one GPU that does not depend on the scalar type (Ctx<S> adds the rest)
// ------------------------------------------------------------------------------------------
struct RankState {
    int64_t N = 0, T = 0, t0 = 0, t1 = 0, Tl = 0, K = 0, L = 0;
    int alg = 0, device = 0, engine = 0;
    bool is_first = true, is_last = true;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int64_t launches = 0;
    double data_norm = 0.0;
    double data_sumsq_local = 0.0;   // ||X_owned||^2 of this shard
    double data_sumsq_global = 0.0;  // ||X||^2 over all shards (== local without a communicator)
    int loss_mode = 0;               // 0 = direct residual pass, 1 = algebraic expansion when its inputs are resident
    bool loss_mode_explicit = false; // set by cmf_set_loss_mode: engine changes then leave the mode alone
    // Calibrated expansion (loss_mode 1 at or below `loss_guard`): the expansion's error is a slowly varying bias (the
    // truncating fp32 adder of the tensor core shrinks numH and the Grams by ~1e-6), so it is measured against the direct
    // residual pass every `calib_interval` evaluations and subtracted in between; the interval doubles while the
    // prediction made with the previous bias agrees with the direct pass and halves when it does not.
    double loss_guard = 0.25;        // relative loss at or below which the expansion needs the calibration
    int calib_max_interval = 16;
    bool calib_have = false;
    double calib_bias = 0.0, calib_last_err = 0.0;
    int calib_left = 0, calib_interval = 1, calib_fail = 0;
    int64_t n_loss_direct = 0, n_loss_expansion = 0;
    void calib_reset() { calib_have = false; calib_left = 0; calib_interval = 1; calib_fail = 0; numH_dot_valid = false; }   // called wherever the factors or the data are replaced
    double pgd_stepW = 5.0, pgd_stepH = 5.0, pgd_cur_loss = 0.0;   // PGDUpdate state (pgd.jl:147-151)
    bool numH_valid = false;         // numH buffer == transconv(current W, X) and GS == W W' of the current W
    bool numH_dot_valid = false;     // scal[4] == <numH, H> of the current numH and H (left there by the MU update of H)
    bool gram_valid = false;         // exchange buffer 1 holds the local Gram/tail partial of the current H
    bool have_data = false, have_factors = false;
    int64_t R = 0;                   // restarts of a batch handle (cmf_create_batch[_ranks]); 0 = a handle of one factor set
    // optional per-kernel-class event timing (bench.py's roofline): class -> list of event pairs
    bool profiling = false;
    struct ProfEv { int which; cudaEvent_t a, b; };
    std::vector<ProfEv> prof_events;
    int prof_open = -1;
    void prof_begin(int which) {
        if (!profiling) return;
        ProfEv e; e.which = which;
        cudaEventCreate(&e.a); cudaEventCreate(&e.b);
        cudaEventRecord(e.a, stream);
        prof_events.push_back(e);
        prof_open = (int)prof_events.size() - 1;
    }
    void prof_end() {
        if (!profiling || prof_open < 0) return;
        cudaEventRecord(prof_events[prof_open].b, stream);
        prof_open = -1;
    }
    void prof_clear() {
        for (auto &e : prof_events) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
        prof_events.clear();
    }
    ~RankState() {
        prof_clear();
        if (ev_a) cudaEventDestroy(ev_a);
        if (ev_b) cudaEventDestroy(ev_b);
        if (comm_stream) cudaStreamDestroy(comm_stream);
    }
    // ---- multi-GPU (the reference is single-process: no counterpart; SURVEY.md section 8e)
    cmf::Comm comm;                  // NCCL communicator of this rank (world == 1: collectives are no-ops)
    cudaStream_t comm_stream = nullptr;  // side stream for collectives that overlap with kernels of the main stream
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;
    int world() const { return comm.world; }
    int rank() const { return comm.rank; }
};

enum { PROF_CONV = 0, PROF_TRANSCONV = 1, PROF_CORR = 2, PROF_SWEEP = 3, PROF_NCLASS = 4 };

using namespace cmf;


// ------------------------------------------------------------------------------------------
// tcgen05 engine state (fp32 handles only): bf16 hi/lo operand copies and their TMA tensor maps
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !ptr) throw CmfError(CMF_ERR_CUDA, "cuTensorMapEncodeTiled not available");
        fn = (EncodeTiledFn)ptr;
    }
    return fn;
}

// 2-D bf16 tensor map: dim0 (contiguous) x dim1 with row stride `stride1` bytes (rows may overlap)
CUtensorMap make_map_2d(void *base, uint64_t dim0, uint64_t dim1, uint64_t stride1, uint32_t box0, uint32_t box1,
                        CUtensorMapSwizzle swz) {
    CUtensorMap m;
    cuuint64_t gdim[2] = {dim0, dim1};
    cuuint64_t gstr[1] = {stride1};
    cuuint32_t box[2] = {box0, box1};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode_tiled_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, gdim, gstr, box, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw CmfError(CMF_ERR_CUDA, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
    return m;
}

// 3-D bf16 map for MN-major operands: (64 contiguous elements, rows with stride `row_stride` bytes,
// groups of 64 elements 128 bytes apart); box = (64, box_rows, box_groups), SWIZZLE_128B.
CUtensorMap make_map_mn(void *base, uint64_t rows, uint64_t row_stride, uint64_t groups, uint32_t box_rows, uint32_t box_groups) {
    CUtensorMap m;
    cuuint64_t gdim[3] = {64, rows, groups};
    cuuint64_t gstr[2] = {row_stride, 128};
    cuuint32_t box[3] = {64, box_rows, box_groups};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = encode_tiled_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, gdim, gstr, box, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw CmfError(CMF_ERR_CUDA, "cuTensorMapEncodeTiled (3-D) failed with code " + std::to_string((int)r));
    return m;
}

struct TcState {
    bool ok = false, tried = false;
    int Kp = 0, G = 0, num_sms = 148;
    int64_t KLp = 0, rows_u = 0, groups = 0, hrows = 0;
    DevBuf<__nv_bfloat16> X_hi, X_lo, Hw_hi, Hw_lo, Hm_hi, Hm_lo, Wc_hi, Wc_lo, Wu_hi, Wu_lo, Cc_hi, Cc_lo;
    CUtensorMap mWc[2], mHw[2], mHm[2], mWu[2], mXk[2], mXmn[2];
    CUtensorMap mHmn[2];   // H (owned + right halo) as the MN-major "X" operand of the Gram correlation
    CUtensorMap mCu[2];    // C table as the A operand of denomH
    CUtensorMap mHk[2];    // H (both halos) as the K-major "X" operand of denomH
    CUtensorMap mGc[2];    // G = Htilde Htilde' as the A operand of G*W
    CUtensorMap mWuB[2], mWcB[2];   // Wu / Wc with 256-row boxes (B operands of the plain GEMMs)
    DevBuf<__nv_bfloat16> Gc_hi, Gc_lo;
    int nsplit = 1, nsplit_g = 1;
    int64_t split_len = 0, split_len_g = 0, tiles_m = 0, tiles_n = 0, groups_c = 0, rows_c = 0;
    bool x_dirty = true, w_dirty = true;
};

// frequency-domain engine state (kernels_fd.cuh): spectrum of X (built once per data set) and the per-iteration spectra
struct FdState {
    bool ok = false, tried = false;
    int B = 0, logB = 0, V = 0, F = 0;
    int64_t nblk = 0, nblkp = 0;          // overlap-save blocks covering the owned columns; padded to a multiple of 16
    int Kq = 64, MR = 128;                // components padded to Kq = 64 or 128; MR = 2 Kq rows (real | imaginary) per frequency
    int V2 = 0;                           // hop of the denomH blocking (2L-1 lags): B - 2L + 2
    int64_t nblk2 = 0;
    DevBuf<__nv_bfloat16> Xf_hi, Xf_lo, Ah_hi, Ah_lo, Aw_hi, Aw_lo, Hf_hi, Hf_lo, Ac_hi, Ac_lo;
    DevBuf<float> Of, Df, Gf, Yf;
    DevBuf<float2> tw;                    // twiddle table of the transforms (fd::twiddle_kernel)
    DevBuf<__nv_bfloat16> Awm_hi, Awm_lo; // direct loss pass: spectrum of W as the A operand of TC_FQX (allocated on first use)
    int64_t nbc = 0;                      // blocks per chunk of the direct loss pass (Yf holds F x nbc x 2 x N floats)
    bool wx_dirty = true;
    CUtensorMap mXfK[2], mXfMN[2], mAw[2], mAh[2], mHfMN[2], mAc[2], mHf2K[2], mAwm[2], mHcK[2];
    bool x_dirty = true, w_dirty = true, h_dirty = true;   // h_dirty: Ah does not hold the spectrum of the current H
    bool hf2_valid = false;               // Hf holds the denomH blocking (hop V2) of the current H (prefetched while W is all-gathered)
    std::string why;                      // reason the engine is unavailable
    void release() {
        Xf_hi.free(); Xf_lo.free(); Ah_hi.free(); Ah_lo.free(); Aw_hi.free(); Aw_lo.free(); Of.free(); Df.free();
        Hf_hi.free(); Hf_lo.free(); Gf.free(); Ac_hi.free(); Ac_lo.free(); tw.free();
        Yf.free(); Awm_hi.free(); Awm_lo.free(); nbc = 0; wx_dirty = true;
        ok = tried = false;
        x_dirty = w_dirty = h_dirty = true; hf2_valid = false;
    }
};

// The transforms are compiled per block length (log2 B = 6 .. 10) and tile width C: fd_with_b calls fn(LOGB) and fd_with_bc
// calls fn(LOGB, C) with std::integral_constant arguments for the plan's values.  fd_cols_h never picks C = 32 at B = 1024
// (the tile would not fit in shared memory).
template <typename Fn>
void fd_with_b(int logB, Fn &&fn) {
    switch (logB) {
    case 6: fn(std::integral_constant<int, 6>{}); break;
    case 7: fn(std::integral_constant<int, 7>{}); break;
    case 8: fn(std::integral_constant<int, 8>{}); break;
    case 9: fn(std::integral_constant<int, 9>{}); break;
    case 10: fn(std::integral_constant<int, 10>{}); break;
    default: REQUIRE(false, "frequency-domain transforms: block length must be a power of two in [64, 1024]");
    }
}
template <typename Fn>
void fd_with_bc(int logB, int C, Fn &&fn) {
    fd_with_b(logB, [&](auto lb) {
        switch (C) {
        case 8: fn(lb, std::integral_constant<int, 8>{}); break;
        case 16: fn(lb, std::integral_constant<int, 16>{}); break;
        case 32: fn(lb, std::integral_constant<int, 32>{}); break;
        default: REQUIRE(false, "frequency-domain transforms: unsupported tile width");
        }
    });
}

template <typename S>
struct Ctx : RankState {
    static constexpr int dtype = std::is_same<S, double>::value ? CMF_F64 : CMF_F32;
    TcState tcs;
    FdState fds;
    DevBuf<S> X, Hbuf, Wi, Wtmp, numW, denW, GS, Cf, numH, denH, tailC;
    DevBuf<int> progress, lockstep;
    DevBuf<S> tailCt;                  // HALS H sweep: truncated lag tables of all component pairs
    int hals_grid = 0;
    DevBuf<double> exch1, corr_part, loss_part, scal;
    S *H = nullptr;  // owned column 0 inside Hbuf
    int nsplit_w = 1, nsplit_g = 1;
    int64_t split_w = 0, split_g = 0;
    int conv_blocks_max = 0;

    // conv tiling per dtype
    static constexpr int TN = sizeof(S) == 4 ? 8 : 4;
    static constexpr int TT = 8, TY = 16;
    static constexpr int BN = 16 * TN, BT = TY * TT;

    int64_t KL() const { return K * L; }

    void hals_setup() {
        // wavefront H sweep: one cooperative launch, CTA b owns components b, b+grid, ...
        REQUIRE(L - 1 <= HW_TC, "HALS: L-1 must not exceed the sweep chunk (1024 columns)");
        const size_t smem = hals_wave_smem_elems<S>(L) * sizeof(S);
        int per_sm = 0, sms = 0, coop = 0;
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
        REQUIRE(coop != 0, "HALS needs cooperative launch support");
        CK(cudaFuncSetAttribute(hals_h_wave_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hals_h_wave_kernel<S>, HW_NT, smem));
        hals_grid = (int)std::min<int64_t>(K, (int64_t)per_sm * sms);
        REQUIRE(hals_grid >= 1, "HALS: H sweep kernel does not fit on the device");
        tailC.alloc((size_t)hals_grid * (size_t)(L * L));
        progress.alloc((size_t)K);
    }

    void init() {
        if (R > 0) { init_batch(); return; }
        CK(cudaSetDevice(device));
        CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        own_stream = true;
        const int64_t hal = L - 1;
        X.alloc((size_t)((Tl + hal) * N));
        Hbuf.alloc((size_t)((Tl + 2 * hal) * K));
        H = Hbuf.p + hal * K;
        Wi.alloc((size_t)(KL() * N));
        Wtmp.alloc((size_t)(KL() * N));
        numW.alloc((size_t)(KL() * N));
        denW.alloc((size_t)(KL() * N));
        GS.alloc((size_t)(KL() * KL()));
        Cf.alloc((size_t)((2 * L - 1) * K * K));
        numH.alloc((size_t)(Tl * K));
        denH.alloc((size_t)(std::max<int64_t>(Tl * K, Tl)));
        exch1.alloc((size_t)(L * K * K + hal * K + 1));
        scal.alloc(8);
        if (alg == CMF_HALS) hals_setup();
        // corr splits: numW (Nin = N) and Gram (Nin = K)
        plan_split(N, Tl + hal, nsplit_w, split_w);
        plan_split(K, Tl + hal, nsplit_g, split_g);
        corr_part.alloc((size_t)std::max<int64_t>((int64_t)nsplit_w * KL() * N, (int64_t)nsplit_g * KL() * K));
        conv_blocks_max = (int)(cdiv(N, BN) * cdiv(Tl + hal, BT));
        loss_part.alloc((size_t)std::max(2 * conv_blocks_max, 4096));
        // the tensor-core engine is set up right away only where it is the default (big contractions); small problems
        // build it lazily on cmf_set_engine(h, 1)
        if constexpr (is_f32) {
            if (N >= 256 && Tl >= 4096 && K * L >= 256) {
                tc_setup();
                // frequency-domain engine by default where it wins: enough lags that 2*L direct flops per element exceed the
                // ~8.5 of the per-frequency products, and room for the spectrum of X (CMF_ENGINE_DEFAULT=1 keeps engine 1)
                const char *e = getenv("CMF_ENGINE_DEFAULT");
                if (tcs.ok && engine == 1 && L >= 8 && K <= fd::KQ_MAX && !(e && atoi(e) == 1)) {
                    fd_setup();
                    // with this engine the expansion loss is the default too: the direct pass would cost 10x the iteration
                    if (fds.ok) { engine = 2; loss_mode = 1; }
                }
            }
        }
        CK(cudaStreamSynchronize(stream));
    }

    // ---------------------------------------------------------------- tcgen05 engine (fp32 only)
    // Engines 1 and 2 exist for fp32 handles only.  The contraction dispatchers (section "contractions"), the direct loss
    // pass and the runtime entries (init, tc_available, fd_available, fd_denomH_prefetch) test this; the tc_* / fd_* methods
    // are reached only through them.  fd_active() implies tc_active().
    static constexpr bool is_f32 = std::is_same<S, float>::value;
    bool tc_active() const { return engine >= 1 && tcs.ok; }
    bool fd_active() const { return engine == 2 && tcs.ok && fds.ok; }
    bool fd_available() {
        if constexpr (is_f32) {
            if (!tc_available()) return false;
            if (!fds.ok && !fds.tried) fd_setup();
            if (fds.ok) { tcs.X_hi.free(); tcs.X_lo.free(); tcs.x_dirty = true; }   // the two engines never hold both copies of X
        }
        return fds.ok;
    }
    void fd_release() { fds.release(); }
    void fd_layout(int *B, int *V, int64_t *nblk) {
        *B = fd_active() ? fds.B : 0; *V = fd_active() ? fds.V : 0; *nblk = fd_active() ? fds.nblkp : 0;
    }

    // ---------------------------------------------------------------- frequency-domain engine (fp32, K <= 128, L <= 256)
    void fd_setup() {
        FdState &f = fds;
        f.tried = true;
        if (!tcs.ok) { f.why = "needs the tcgen05 engine"; return; }
        if (K > fd::KQ_MAX || L > 256 || N < 16) { f.why = "needs K <= 128, L <= 256, N >= 16"; return; }
        f.Kq = (K <= 64) ? 64 : 128;
        f.MR = 2 * f.Kq;
        // block length: the smallest power of two >= 8L, at most 1024 (>= 4L always: L <= 256).  A/B on B200 with the round-2
        // transforms, same box: c4 (L = 100) 512 -> 45.9 ms, 1024 -> 43.2 ms per iteration; c3 (L = 50) 256 -> 3.86, 512 -> 3.48,
        // 1024 -> 3.92 ms: the products move and multiply (B / V)(F / (B/2)) ~ 1.24 / 1.11 / 1.05 times the size of X at
        // B = 4L.. / 8L.. / 16L.., the transforms get longer
        int B0 = 64;
        while (B0 < 8 * L && B0 < 1024) B0 *= 2;
        while (B0 < 4 * L) B0 *= 2;
        // ... unless this shard is so short that the longer block only adds padding: the numH product works on tiles of 256
        // blocks, so its work goes like F * 256 * ceil(blocks / 256), the numW product's like F * blocks.  A rank of an
        // 8-GPU c4 fit (524288 columns) has 1270 blocks of 512 (5 tiles, 1 % padding) or 567 blocks of 1024 (3 tiles, 26 %
        // padding): the shorter block is kept when the longer one does not win at least 3 % on that count.
        if (B0 / 2 >= 4 * L && B0 / 2 >= 64) {
            auto work = [&](int B) {
                const int64_t nb = cdiv(Tl, (int64_t)(B - (int)L + 1));
                return (double)(B / 2 + 1) * (double)(cdiv(nb, tc::BN) * tc::BN + cdiv(nb, 16) * 16);
            };
            if (work(B0) > 0.97 * work(B0 / 2)) B0 /= 2;
        }
        int forced = 0;
        if (const char *e = getenv("CMF_FD_B")) {
            const int want = atoi(e);
            if (want >= 4 * L && want >= 64 && want <= 1024 && (want & (want - 1)) == 0) forced = want;
        }
        tcs.X_hi.free(); tcs.X_lo.free(); tcs.x_dirty = true;
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        // what this handle allocates later, beside the spectra: the HALS round kernel's component-major copies of H and
        // Delta H and its ring of block partials; the direct loss pass's spectrum of W and a minimal chunk buffer
        size_t later = (size_t)1 << 30;
        if (alg == CMF_HALS) later += (size_t)2 * (size_t)(Tl + 2048) * (size_t)K * 4 + (size_t)hals2::RING * (size_t)cdiv(K, hals2::GS) * (size_t)K * hals2::CW * 4;
        size_t xf = 0, ah = 0, aw = 0, of = 0, df = 0, hf = 0, gf = 0, ac = 0;
        bool fits = false;
        // the next power of two moves fewer bytes still (hop / length grows), so it is the fallback when the first choice does
        // not fit beside the data
        for (int B = forced ? forced : B0; B <= (forced ? forced : std::min(2 * B0, 1024)); B *= 2) {
            int logB = 0;
            while ((1 << logB) < B) ++logB;
            f.B = B; f.logB = logB; f.V = B - (int)L + 1; f.F = B / 2 + 1;
            f.nblk = cdiv(Tl, f.V);
            f.nblkp = cdiv(f.nblk, 16) * 16;
            xf = (size_t)f.F * (size_t)f.nblkp * 2 * (size_t)N + 64;
            ah = (size_t)f.F * (size_t)f.nblkp * 2 * f.MR + 64;
            aw = (size_t)f.F * f.MR * 2 * (size_t)N + 64;
            f.V2 = B - 2 * (int)L + 2;
            f.nblk2 = cdiv(Tl, f.V2);
            of = (size_t)f.F * (size_t)std::max(f.nblkp, f.nblk2) * f.MR; df = (size_t)f.F * f.MR * (size_t)N;
            // Hf serves the Gram partial (nblkp blocks) and, later on the same stream, denomH (nblk2 blocks)
            hf = (size_t)f.F * (size_t)std::max(f.nblkp, f.nblk2) * 2 * f.Kq + 256; gf = (size_t)f.F * f.MR * f.Kq;
            ac = (size_t)f.F * f.MR * f.MR;
            const size_t need = 4 * (xf + ah + aw + hf + ac) + 4 * (of + df + gf);
            const size_t loss_pass = 4 * aw + (size_t)256 * (size_t)f.F * 2 * (size_t)N * sizeof(float);
            if (need + later + loss_pass <= free_b) { fits = true; break; }
        }
        if (!fits) { f.why = "not enough device memory for the spectrum of X"; return; }
        f.Xf_hi.alloc(xf); f.Xf_lo.alloc(xf);
        f.Ah_hi.alloc(ah); f.Ah_lo.alloc(ah);
        f.Aw_hi.alloc(aw); f.Aw_lo.alloc(aw);
        f.Of.alloc(of); f.Df.alloc(df);
        f.Hf_hi.alloc(hf); f.Hf_lo.alloc(hf); f.Gf.alloc(gf);
        f.Ac_hi.alloc(ac); f.Ac_lo.alloc(ac);
        f.tw.alloc((size_t)f.B);
        fd::twiddle_kernel<<<(unsigned)cdiv(f.B, 256), 256, 0, stream>>>(f.tw.p, f.B);
        post_launch();
        __nv_bfloat16 *xs[2] = {f.Xf_hi.p, f.Xf_lo.p}, *as[2] = {f.Ah_hi.p, f.Ah_lo.p}, *ws[2] = {f.Aw_hi.p, f.Aw_lo.p};
        const uint64_t rows = (uint64_t)f.F * (uint64_t)f.nblkp;
        for (int i = 0; i < 2; ++i) {
            f.mXfK[i] = make_map_2d(xs[i], (uint64_t)(2 * N), rows, (uint64_t)N * 4, tc::BK, tc::BN, CU_TENSOR_MAP_SWIZZLE_64B);
            f.mXfMN[i] = make_map_mn(xs[i], rows * 2, (uint64_t)N * 2, (uint64_t)cdiv(N, 64), tc::BK, 4);
            f.mAw[i] = make_map_2d(ws[i], (uint64_t)(2 * N), (uint64_t)f.F * f.MR, (uint64_t)N * 4, tc::BK, tc::BM, CU_TENSOR_MAP_SWIZZLE_64B);
            f.mAh[i] = make_map_mn(as[i], rows * 2, (uint64_t)f.MR * 2, (uint64_t)(f.MR / 64), tc::BK, 2);
            f.mHfMN[i] = make_map_mn(i == 0 ? f.Hf_hi.p : f.Hf_lo.p, rows * 2, (uint64_t)f.Kq * 2, (uint64_t)(f.Kq / 64), tc::BK, 4);
            f.mAc[i] = make_map_2d(i == 0 ? f.Ac_hi.p : f.Ac_lo.p, f.MR, (uint64_t)f.F * f.MR, (uint64_t)f.MR * 2, tc::BK, tc::BM, CU_TENSOR_MAP_SWIZZLE_64B);
            f.mHf2K[i] = make_map_2d(i == 0 ? f.Hf_hi.p : f.Hf_lo.p, f.MR, (uint64_t)f.F * (uint64_t)f.nblk2, (uint64_t)f.MR * 2, tc::BK, tc::BN, CU_TENSOR_MAP_SWIZZLE_64B);
        }
        CK(cudaFuncSetAttribute(tc::tc_kernel<tc::TC_FQT>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
        CK(cudaFuncSetAttribute(tc::tc_kernel<tc::TC_FQC>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
        CK(cudaFuncSetAttribute(tc::tc_kernel<tc::TC_FQX>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));

        // shared memory of every transform instantiation of this block length (each C the H side may pick)
        fd_with_b(f.logB, [&](auto lb) {
            constexpr int LB = decltype(lb)::value;
            const int x16 = (int)fd_smem(16), w = (int)fd_smem(fd_cols_w());
            CK(cudaFuncSetAttribute(fd::fft_x_kernel<LB>, cudaFuncAttributeMaxDynamicSharedMemorySize, x16));
            CK(cudaFuncSetAttribute(fd::ifft_resid_kernel<LB>, cudaFuncAttributeMaxDynamicSharedMemorySize, x16));
            fd_with_bc(f.logB, fd_cols_w(), [&](auto, auto c) {
                constexpr int CW = decltype(c)::value;
                CK(cudaFuncSetAttribute(fd::fft_w_kernel<LB, CW>, cudaFuncAttributeMaxDynamicSharedMemorySize, w));
                CK(cudaFuncSetAttribute(fd::ifft_numW_kernel<float, LB, CW>, cudaFuncAttributeMaxDynamicSharedMemorySize, w));
                CK(cudaFuncSetAttribute(fd::ifft_numW_kernel<double, LB, CW>, cudaFuncAttributeMaxDynamicSharedMemorySize, w));
            });
            for (int ch : {8, 16, 32}) {
                if (LB == 10 && ch == 32) continue;
                const int h = (int)fd_smem(ch);
                fd_with_bc(f.logB, ch, [&](auto, auto c) {
                    constexpr int CH = decltype(c)::value;
                    CK(cudaFuncSetAttribute(fd::fft_h_kernel<LB, CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, h));
                    CK(cudaFuncSetAttribute(fd::ifft_numH_kernel<LB, CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, h));
                });
            }
        });
        f.x_dirty = f.w_dirty = f.h_dirty = true;
        f.ok = true;
    }
    // component pairs per CTA of the H-side transforms: 32 (all 64 rows) while the tile fits in shared memory
    int fd_cols_h() const {
        if (const char *e = getenv("CMF_FD_COLS")) {
            const int c = atoi(e);
            if ((c == 8 || c == 16 || c == 32) && (size_t)fds.B * (size_t)c * sizeof(float2) <= 160 * 1024) return c;
        }
        return fds.B >= 1024 ? 8 : 16;          // tiles of <= 64 KB + twiddles: three CTAs per SM (c4 at B = 1024: 44.96 -> 43.23 ms)
    }
    // scheduling order of the 1-D grids of the transforms: 0 = tile index fastest, block count = block index fastest (CMF_FD_ORDER=1)
    int64_t fd_order(int64_t nblocks) const { static const int o = getenv("CMF_FD_ORDER") ? atoi(getenv("CMF_FD_ORDER")) : 0; return o ? nblocks : 0; }
    // complex columns per CTA of the W-side transforms (fft_w / ifft_numW): as for the H side, 8 at B = 1024 keeps three CTAs per SM
    int fd_cols_w() const { return fds.B >= 1024 ? 8 : 16; }
    size_t fd_smem(int C) const { return ((size_t)fds.B * (size_t)C + (size_t)fds.B) * sizeof(float2); }   // tile + full-circle twiddle table
    // launches of the transforms whose tile width the host picks (fd_cols_h / fd_cols_w)
    // spectrum of nb blocks of H (hop V, first column t_off) -> hi / lo; full: see fft_h_kernel
    void fd_fft_h(__nv_bfloat16 *hi, __nv_bfloat16 *lo, int64_t nb, int V, int full, int64_t t_off) {
        const int C = fd_cols_h();
        fd_with_bc(fds.logB, C, [&](auto lb, auto c) {
            fd::fft_h_kernel<decltype(lb)::value, decltype(c)::value><<<(unsigned)(nb * (fds.Kq / 2 / C)), fd::NT, fd_smem(C), stream>>>(
                H, hi, lo, K, Tl, Tl + (L - 1), V, nb, full, t_off, fds.Kq, fd_order(nb), fds.tw.p);
        });
    }
    // Of (blocks of row stride nblkp_) -> the owned columns of out, nb blocks of hop V
    void fd_ifft_numH(const float *Of, float *out, int64_t nb, int V, int64_t nblkp_) {
        const int C = fd_cols_h();
        fd_with_bc(fds.logB, C, [&](auto lb, auto c) {
            fd::ifft_numH_kernel<decltype(lb)::value, decltype(c)::value><<<(unsigned)(nb * (fds.Kq / 2 / C)), fd::NT, fd_smem(C), stream>>>(
                Of, out, K, Tl, V, nblkp_, fds.Kq, fd_order(nb), fds.tw.p);
        });
    }
    // spectrum of the Lw lags of src[(l*K+k)][Nw] -> hi / lo (see fft_w_kernel)
    void fd_fft_w(const float *src, __nv_bfloat16 *hi, __nv_bfloat16 *lo, int64_t Nw, int64_t Lw, int64_t ldw, int64_t coff, int xmode) {
        const int C = fd_cols_w();
        fd_with_bc(fds.logB, C, [&](auto lb, auto c) {
            fd::fft_w_kernel<decltype(lb)::value, decltype(c)::value><<<dim3((unsigned)cdiv(Nw, 2 * C), (unsigned)K), fd::NT, fd_smem(C), stream>>>(
                src, hi, lo, Nw, K, Lw, ldw, coff, xmode, fds.Kq, fds.tw.p);
        });
    }
    // Df (rows of ldi) -> the first L lags of out[(l*K+k)][Nw]
    template <typename OutT>
    void fd_ifft_numW(const float *Df, OutT *out, int64_t Nw, int64_t ldi) {
        const int C = fd_cols_w();
        fd_with_bc(fds.logB, C, [&](auto lb, auto c) {
            fd::ifft_numW_kernel<OutT, decltype(lb)::value, decltype(c)::value><<<dim3((unsigned)cdiv(Nw, 2 * C), (unsigned)K), fd::NT, fd_smem(C), stream>>>(
                Df, out, Nw, ldi, K, L, fds.Kq, fds.tw.p);
        });
    }

    void fd_build_X() {
        FdState &f = fds;
        if (!f.x_dirty) return;
        dim3 grid((unsigned)(f.nblkp * cdiv(N, 32)));
        fd_with_b(f.logB, [&](auto lb) {
            fd::fft_x_kernel<decltype(lb)::value><<<grid, fd::NT, fd_smem(16), stream>>>(X.p, f.Xf_hi.p, f.Xf_lo.p, N, Tl + (L - 1), f.V, f.nblkp,
                                                                                        fd_order(f.nblkp), f.tw.p);
        });
        post_launch();
        f.x_dirty = false;
    }
    // numW through the spectrum of X (mult.jl:32)
    void fd_corr() {
        FdState &f = fds;
        fd_build_X();
        fd_spectrum_H();
        tc::Params q = tc_base_params();
        q.nprod = 3;
        q.tiles_n = cdiv(N, tc::BN);
        q.nkb = f.nblkp * 2 / tc::BK;
        q.MR = f.MR; q.mtiles = f.MR / tc::BM; q.units = (int64_t)f.F * q.tiles_n * q.mtiles;
        q.fq_rows = f.nblkp * 2;
        q.out = f.Df.p; q.Mrows = f.MR; q.Ncols = N; q.ldo = N;
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        prof_begin(PROF_CORR);
        tc::tc_kernel<tc::TC_FQC><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(f.mAh[0], f.mAh[1], f.mXfMN[0], f.mXfMN[1], q);
        prof_end();
        post_launch();
        fd_ifft_numW(f.Df.p, numW.p, N, N);
        post_launch();
    }
    // denomH = C (*) H through the spectrum of H (mult.jl:44,48): the numH product with the lag table in place of W and
    // H (both halos) in place of X; needs lag_tables() done.  The last L-1 columns are overwritten by the truncated tail.
    void fd_denomH() {
        FdState &f = fds;
        fd_fft_w(Cf.p, f.Ac_hi.p, f.Ac_lo.p, K, 2 * L - 1, f.MR, f.Kq, 0);
        post_launch();
        fd_denomH_prefetch();
        f.hf2_valid = false;                                   // consumed below; Hf is shared with the Gram / loss passes
        tc::Params q = tc_base_params();
        q.nprod = 3;
        q.tiles_n = cdiv(f.nblk2, tc::BN);
        q.nkb = f.MR / tc::BK;
        q.MR = f.MR; q.mtiles = f.MR / tc::BM; q.units = (int64_t)f.F * q.tiles_n * q.mtiles;
        q.fq_rows = f.nblk2;
        q.out = f.Of.p;
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        tc::tc_kernel<tc::TC_FQT><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(f.mAc[0], f.mAc[1], f.mHf2K[0], f.mHf2K[1], q);
        post_launch();
        fd_ifft_numH(f.Of.p, denH.p, f.nblk2, f.V2, f.nblk2);
        post_launch();
    }
    // the H-only part of fd_denomH: spectrum of the blocks of H (hop V2, both halos).  Depends on H alone, so a sharded fit runs it
    // while the all-gather of the new W is in flight (r_update_motifs).
    void fd_denomH_prefetch() {
        if constexpr (is_f32) {
            FdState &f = fds;
            if (!fd_active() || f.hf2_valid) return;
            fd_fft_h(f.Hf_hi.p, f.Hf_lo.p, f.nblk2, f.V2, 1, -(L - 1));
            post_launch();
            f.hf2_valid = true;
        }
    }
    // sum of squared residuals (mult.jl:55-57) through the frequency domain: Xhat^ = W^ H^ per frequency for a chunk of
    // blocks (TC_FQX), inverse transform, subtract X, sum of squares (ifft_resid_kernel); returns the number of partials.
    // ~5x cheaper than the time-domain TC_CONV pass at c4, and free of the cancellation of the expansion.
    int64_t fd_conv_loss() {
        FdState &f = fds;
        f.hf2_valid = false;
        const int64_t ntile32 = cdiv(N, 32);
        if (f.Awm_hi.n == 0) {
            const size_t aw = (size_t)f.F * 2 * f.MR * (size_t)N + 64;
            size_t free_b = 0, total_b = 0;
            CK(cudaMemGetInfo(&free_b, &total_b));
            const size_t per_block = (size_t)f.F * 2 * (size_t)N * sizeof(float);          // Yf bytes per block
            REQUIRE(free_b > 4 * aw + 256 * per_block + ((size_t)1 << 29), "not enough device memory for the frequency-domain loss pass");
            size_t budget = std::min<size_t>((free_b - 4 * aw - ((size_t)1 << 29)) / 2, (size_t)12 << 30);
            int64_t nbc = (int64_t)(budget / per_block) / tc::BN * tc::BN;
            nbc = std::max<int64_t>(tc::BN, std::min<int64_t>(nbc, cdiv(f.nblk, tc::BN) * tc::BN));
            if (const char *e = getenv("CMF_FD_NBC")) { const int64_t v = atoll(e); if (v >= tc::BN && v % tc::BN == 0 && v < nbc) nbc = v; }   // tests: force several chunks
            f.nbc = nbc;
            f.Awm_hi.alloc(aw); f.Awm_lo.alloc(aw);
            f.Yf.alloc((size_t)f.F * (size_t)nbc * 2 * (size_t)N);
            for (int i = 0; i < 2; ++i) {
                f.mAwm[i] = make_map_mn(i == 0 ? f.Awm_hi.p : f.Awm_lo.p, (uint64_t)f.F * 2 * f.MR, (uint64_t)N * 2, (uint64_t)cdiv(N, 64), tc::BK, 2);
                f.mHcK[i] = make_map_2d(i == 0 ? f.Hf_hi.p : f.Hf_lo.p, f.MR, (uint64_t)f.F * (uint64_t)f.nblk, (uint64_t)f.MR * 2, tc::BK, tc::BN, CU_TENSOR_MAP_SWIZZLE_64B);
            }
            f.wx_dirty = true;
        }
        const size_t need_lp = (size_t)(f.nblk * ntile32);
        if (loss_part.n < need_lp) loss_part.alloc(std::max<size_t>(need_lp, 4096));
        if (f.wx_dirty) {
            fd_fft_w(Wi.p, f.Awm_hi.p, f.Awm_lo.p, N, L, 2 * N, N, 1);
            post_launch();
            f.wx_dirty = false;
        }
        fd_fft_h(f.Hf_hi.p, f.Hf_lo.p, f.nblk, f.V, 1, -(L - 1));
        post_launch();
        prof_begin(PROF_CONV);
        for (int64_t b0 = 0; b0 < f.nblk; b0 += f.nbc) {
            const int64_t cur = std::min(f.nbc, f.nblk - b0);
            tc::Params q = tc_base_params();
            q.nprod = 3;
            q.tiles_n = cdiv(cur, tc::BN);
            q.tiles_m = cdiv(N, tc::BM);
            q.nkb = f.MR / tc::BK;
            q.MR = f.MR; q.mtiles = 1; q.units = (int64_t)f.F * 2 * q.tiles_m * q.tiles_n;
            q.fq_rows = f.nblk; q.b_off = b0; q.nbc = cur;
            q.out = f.Yf.p;
            const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
            tc::tc_kernel<tc::TC_FQX><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(f.mAwm[0], f.mAwm[1], f.mHcK[0], f.mHcK[1], q);
            post_launch();
            fd_with_b(f.logB, [&](auto lb) {
                fd::ifft_resid_kernel<decltype(lb)::value><<<(unsigned)(cur * ntile32), fd::NT, fd_smem(16), stream>>>(
                    f.Yf.p, X.p, loss_part.p + b0 * ntile32, N, Tl, L, f.V, cur, b0, fd_order(cur), f.tw.p);
            });
            post_launch();
        }
        prof_end();
        return f.nblk * ntile32;
    }
    // Ah = spectrum of the owned columns of the current H, block by block (shared by numW and the Gram partial)
    void fd_spectrum_H() {
        FdState &f = fds;
        if (!f.h_dirty) return;
        fd_fft_h(f.Ah_hi.p, f.Ah_lo.p, f.nblkp, f.V, 0, 0);
        post_launch();
        f.h_dirty = false;
    }
    // Gram partial Rg[d][k][k'] = sum_u H[u][k] H[u+d][k'] through the spectrum of H (u owned, u+d into the right halo)
    void fd_gram() {
        FdState &f = fds;
        f.hf2_valid = false;
        fd_spectrum_H();
        fd_fft_h(f.Hf_hi.p, f.Hf_lo.p, f.nblkp, f.V, 1, 0);
        post_launch();
        tc::Params q = tc_base_params();
        q.nprod = 3;
        q.tiles_n = 1;
        q.nkb = f.nblkp * 2 / tc::BK;
        q.MR = f.MR; q.mtiles = f.MR / tc::BM; q.units = (int64_t)f.F * q.mtiles;
        q.fq_rows = f.nblkp * 2;
        q.out = f.Gf.p; q.Mrows = f.MR; q.Ncols = K; q.ldo = f.Kq;
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        tc::tc_kernel<tc::TC_FQC><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(f.mAh[0], f.mAh[1], f.mHfMN[0], f.mHfMN[1], q);
        post_launch();
        fd_ifft_numW(f.Gf.p, exch1.p, K, f.Kq);
        post_launch();
    }
    // numH through the spectrum of X (mult.jl:47)
    void fd_transconv() {
        FdState &f = fds;
        fd_build_X();
        if (f.w_dirty) {
            fd_fft_w(Wi.p, f.Aw_hi.p, f.Aw_lo.p, N, L, 2 * N, N, 0);
            post_launch();
            f.w_dirty = false;
        }
        tc::Params q = tc_base_params();
        q.nprod = 3;
        q.tiles_n = cdiv(f.nblkp, tc::BN);
        q.nkb = cdiv(2 * N, tc::BK);
        q.MR = f.MR; q.mtiles = f.MR / tc::BM; q.units = (int64_t)f.F * q.tiles_n * q.mtiles;
        q.fq_rows = f.nblkp;
        q.out = f.Of.p;
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        prof_begin(PROF_TRANSCONV);
        tc::tc_kernel<tc::TC_FQT><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(f.mAw[0], f.mAw[1], f.mXfK[0], f.mXfK[1], q);
        prof_end();
        post_launch();
        fd_ifft_numH(f.Of.p, numH.p, f.nblk, f.V, f.nblkp);
        post_launch();
    }
    bool tc_available() {
        if constexpr (is_f32) {
            if (!tcs.ok && !tcs.tried) tc_setup();
        }
        return tcs.ok;
    }

    void tc_setup() {
        TcState &t = tcs;
        t.tried = true;
        if (K > 128 || N % 8 != 0) return;
        t.Kp = (int)(cdiv(K, 8) * 8);                          // TMA row strides must be multiples of 16 bytes
        t.G = 128 / t.Kp;                                      // lags per 128-row tile of the transposed conv
        t.KLp = cdiv(L * t.Kp, 64) * 64;
        t.groups = cdiv(L, t.G);
        t.rows_u = cdiv(L * t.Kp + 128, 128) * 128;             // dense rows l*Kp + k, padded so every 128-row box is in bounds
        const int64_t hal = L - 1;
        t.hrows = Tl + hal;                                   // window rows addressed (X columns incl. right halo)
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10) return;                         // tcgen05 needs sm_100
        t.num_sms = prop.multiProcessorCount;
        // the bf16 planes of H (4 x the size of H in bf16) are allocated on first use (tc_h_planes): a handle that runs on
        // the frequency-domain engine never touches them
        t.Wc_hi.alloc((size_t)(N * t.KLp)); t.Wc_lo.alloc((size_t)(N * t.KLp));
        t.Wu_hi.alloc((size_t)(t.rows_u * N)); t.Wu_lo.alloc((size_t)(t.rows_u * N));
        t.groups_c = cdiv(2 * L - 1, t.G);
        t.rows_c = cdiv((2 * L - 1) * t.Kp + 128, 128) * 128;
        t.Cc_hi.alloc((size_t)(t.rows_c * t.Kp)); t.Cc_lo.alloc((size_t)(t.rows_c * t.Kp));
        t.Gc_hi.alloc((size_t)(KL() * t.KLp)); t.Gc_lo.alloc((size_t)(KL() * t.KLp));
        if (GS.n < (size_t)(t.rows_u * t.rows_u)) GS.alloc((size_t)(t.rows_u * t.rows_u));
        // tensor maps (index 0 = hi plane, 1 = lo plane)
        __nv_bfloat16 *wc[2] = {t.Wc_hi.p, t.Wc_lo.p};
        __nv_bfloat16 *wu[2] = {t.Wu_hi.p, t.Wu_lo.p};
        for (int i = 0; i < 2; ++i) {
            t.mWc[i] = make_map_2d(wc[i], (uint64_t)t.KLp, (uint64_t)N, (uint64_t)t.KLp * 2, tc::BK, tc::BM, CU_TENSOR_MAP_SWIZZLE_64B);
            t.mWu[i] = make_map_2d(wu[i], (uint64_t)N, (uint64_t)t.rows_u, (uint64_t)N * 2, tc::BK, tc::BM, CU_TENSOR_MAP_SWIZZLE_64B);
            // denomH: A = C table rows (d'*Kp + k) x Kp
            __nv_bfloat16 *cc[2] = {t.Cc_hi.p, t.Cc_lo.p};
            t.mCu[i] = make_map_2d(cc[i], (uint64_t)t.Kp, (uint64_t)t.rows_c, (uint64_t)t.Kp * 2, tc::BK, tc::BM, CU_TENSOR_MAP_SWIZZLE_64B);
            __nv_bfloat16 *gc[2] = {t.Gc_hi.p, t.Gc_lo.p};
            t.mWuB[i] = make_map_2d(wu[i], (uint64_t)N, (uint64_t)t.rows_u, (uint64_t)N * 2, tc::BK, tc::BN, CU_TENSOR_MAP_SWIZZLE_64B);
            t.mWcB[i] = make_map_2d(wc[i], (uint64_t)t.KLp, (uint64_t)N, (uint64_t)t.KLp * 2, tc::BK, tc::BN, CU_TENSOR_MAP_SWIZZLE_64B);
            t.mGc[i] = make_map_2d(gc[i], (uint64_t)t.KLp, (uint64_t)KL(), (uint64_t)t.KLp * 2, tc::BK, tc::BM, CU_TENSOR_MAP_SWIZZLE_64B);
        }
        // correlation work split: balance persistent CTAs, keep splits >= FLUSH_T columns
        t.tiles_m = cdiv(t.KLp, tc::BM);
        t.tiles_n = cdiv(N, tc::BN);
        const int64_t tau = Tl + hal, base = t.tiles_m * t.tiles_n;
        double best = -1.0;
        for (int ns = 1; ns <= 16; ++ns) {
            const int64_t sl = cdiv(cdiv(tau, ns), tc::BK) * tc::BK;
            if (ns > 1 && sl < tc::FLUSH_T) break;
            const int64_t units = base * cdiv(tau, sl);
            const double eff = (double)units / (double)(cdiv(units, t.num_sms) * t.num_sms);
            if (eff > best + 1e-9) { best = eff; t.nsplit = (int)cdiv(tau, sl); t.split_len = sl; }
        }
        // Gram correlation (one n tile): enough splits to fill the machine
        {
            const int64_t want = std::max<int64_t>(1, cdiv(2 * t.num_sms, t.tiles_m));
            const int64_t maxs = std::max<int64_t>(1, tau / tc::FLUSH_T);
            const int64_t ns = std::min(want, maxs);
            t.split_len_g = cdiv(cdiv(tau, ns), tc::BK) * tc::BK;
            t.nsplit_g = (int)cdiv(tau, t.split_len_g);
        }
        const size_t need = std::max((size_t)t.nsplit * (size_t)(KL() * N), (size_t)t.nsplit_g * (size_t)(KL() * K));
        if (corr_part.n < need) corr_part.alloc(need);
        const size_t need_lp = (size_t)(tc::EPI_WARPS * cdiv(Tl, tc::BN) * cdiv(N, tc::BM));
        if (loss_part.n < need_lp) loss_part.alloc(std::max<size_t>(need_lp, 4096));
        CK(cudaFuncSetAttribute(tc::tc_kernel<tc::TC_CONV>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
        CK(cudaFuncSetAttribute(tc::tc_kernel<tc::TC_TRANS>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
        CK(cudaFuncSetAttribute(tc::tc_kernel<tc::TC_CORR>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
        CK(cudaFuncSetAttribute(tc::tc_kernel<tc::TC_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
        t.ok = true;
        t.x_dirty = t.w_dirty = true;
        // default engine: tensor cores when the contraction is big enough to fill 128x256 tiles
        if (N >= 256 && Tl >= 4096 && K * L >= 256) engine = 1;
    }

    tc::Params tc_base_params() {
        tc::Params q;
        memset(&q, 0, sizeof(q));
        q.N = N; q.K = K; q.L = L; q.Tl = Tl; q.G = tcs.G; q.Kp = tcs.Kp;
        { const char *e = getenv("CMF_PROMO"); q.promo = e ? std::max(1, atoi(e)) : tc::PROMO; }
        { const char *e = getenv("CMF_TC_PRODUCTS"); q.nprod = (e && atoi(e) == 2) ? 2 : 3; }   // experiment knob, default 3
        return q;
    }

    // the time-domain bf16 planes of X are allocated on first use: the frequency-domain engine never needs them
    void tc_split_X() {
        if (!tcs.ok || !tcs.x_dirty) return;
        TcState &t = tcs;
        if (t.X_hi.n == 0) {
            const int64_t hal = L - 1;
            t.X_hi.alloc(X.n + 64); t.X_lo.alloc(X.n + 64);      // +64: the 3-D maps may touch one atom past the last row
            __nv_bfloat16 *xs[2] = {t.X_hi.p, t.X_lo.p};
            for (int i = 0; i < 2; ++i) {
                t.mXk[i] = make_map_2d(xs[i], (uint64_t)N, (uint64_t)(Tl + hal), (uint64_t)N * 2, tc::BK, tc::BN, CU_TENSOR_MAP_SWIZZLE_64B);
                t.mXmn[i] = make_map_mn(xs[i], (uint64_t)(Tl + hal), (uint64_t)N * 2, (uint64_t)cdiv(N, 64), tc::BK, 4);
            }
        }
        tc::split_plain_kernel<<<(unsigned)cdiv((int64_t)X.n, 256), 256, 0, stream>>>(X.p, tcs.X_hi.p, tcs.X_lo.p, (int64_t)X.n);
        post_launch();
        tcs.x_dirty = false;
    }
    void tc_split_W() {
        if (!tcs.w_dirty) return;
        tc::split_W_kernel<<<dim3((unsigned)cdiv(N, 32), (unsigned)cdiv(tcs.Kp, 32), (unsigned)L), dim3(32, 8), 0, stream>>>(
            Wi.p, tcs.Wc_hi.p, tcs.Wc_lo.p, tcs.Wu_hi.p, tcs.Wu_lo.p, N, K, L, tcs.Kp, tcs.KLp);
        post_launch();
        tcs.w_dirty = false;
    }
    // bf16 hi/lo planes of H for the time-domain tensor-core kernels and the maps over them, on first use
    void tc_h_planes() {
        TcState &t = tcs;
        if (t.Hw_hi.n != 0) return;
        const int64_t hal = L - 1;
        const size_t hw_elems = (size_t)((Tl + 2 * hal) * t.Kp + t.KLp + 64);
        t.Hw_hi.alloc(hw_elems); t.Hw_lo.alloc(hw_elems);
        t.Hm_hi.alloc(hw_elems); t.Hm_lo.alloc(hw_elems);
        __nv_bfloat16 *hw[2] = {t.Hw_hi.p, t.Hw_lo.p}, *hm[2] = {t.Hm_hi.p, t.Hm_lo.p};
        for (int i = 0; i < 2; ++i) {
            // overlapping-row "window" map: row t starts at element t*Kp and is KLp long
            t.mHw[i] = make_map_2d(hw[i], (uint64_t)t.KLp, (uint64_t)t.hrows, (uint64_t)t.Kp * 2, tc::BK, tc::BN, CU_TENSOR_MAP_SWIZZLE_64B);
            t.mHm[i] = make_map_mn(hm[i], (uint64_t)t.hrows, (uint64_t)t.Kp * 2, (uint64_t)(t.KLp / 64), tc::BK, 2);
            // Gram: "X" = H rows from owned column 0 (owned + right halo), [t][Kp] MN-major
            t.mHmn[i] = make_map_mn(hw[i] + hal * t.Kp, (uint64_t)(Tl + hal), (uint64_t)t.Kp * 2, (uint64_t)cdiv(t.Kp, 64), tc::BK, 4);
            // denomH: "X" = H rows from the left halo on, K-major
            t.mHk[i] = make_map_2d(hw[i], (uint64_t)t.Kp, (uint64_t)(Tl + 2 * hal), (uint64_t)t.Kp * 2, tc::BK, tc::BN, CU_TENSOR_MAP_SWIZZLE_64B);
        }
    }
    void tc_split_H(bool masked) {
        tc_h_planes();
        const int64_t rows = Tl + 2 * (L - 1);
        tc::split_H_kernel<<<(unsigned)cdiv(rows * tcs.Kp, 256), 256, 0, stream>>>(
            Hbuf.p, masked ? tcs.Hm_hi.p : tcs.Hw_hi.p, masked ? tcs.Hm_lo.p : tcs.Hw_lo.p, rows, K, tcs.Kp,
            L - 1, L - 1 + Tl, masked ? 1 : 0);
        post_launch();
    }

    // numW via tensor cores (mult.jl:32)
    void tc_corr() {
        tc_split_X();
        tc_split_H(true);
        tc::Params q = tc_base_params();
        q.tiles_m = tcs.tiles_m; q.tiles_n = tcs.tiles_n; q.split_len = tcs.split_len; q.tau_hi = Tl + (L - 1);
        q.units = tcs.tiles_m * tcs.tiles_n * tcs.nsplit;
        q.part = corr_part.p;
        q.corr_order = 0;   // j tiles fastest: the CTAs that run together share the X tile (A/B: 124 vs 148 ms at T=1M)
        {
            const char *e = getenv("CMF_LOCKSTEP");            // k-block window; 0 disables (diagnostics)
            const int w = e ? atoi(e) : 256;
            if (w > 0) {
                if (lockstep.n == 0) lockstep.alloc(1024);
                CK(cudaMemsetAsync(lockstep.p, 0, lockstep.n * sizeof(int), stream));
                q.lockstep = lockstep.p; q.lockstep_window = w;
            }
        }
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        prof_begin(PROF_CORR);
        if (q.lockstep != nullptr) {
            // CTAs wait on one another inside this launch: co-residency must be guaranteed
            void *args[] = {&tcs.mHm[0], &tcs.mHm[1], &tcs.mXmn[0], &tcs.mXmn[1], &q};
            CK(cudaLaunchCooperativeKernel((void *)tc::tc_kernel<tc::TC_CORR>, dim3(grid), dim3(tc::THREADS), args, tc::SMEM_BYTES, stream));
        } else {
            tc::tc_kernel<tc::TC_CORR><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(tcs.mHm[0], tcs.mHm[1], tcs.mXmn[0], tcs.mXmn[1], q);
        }
        prof_end();
        post_launch();
        const int64_t n = KL() * N;
        reduce_partials_kernel<S><<<(unsigned)cdiv(n, 256), 256, 0, stream>>>(corr_part.p, tcs.nsplit, n, numW.p, nullptr);
        post_launch();
    }
    // plain GEMM out[m*ldo + n] = sum_k A[m][k] B[n][k] on tensor cores (operands given as hi/lo tensor maps)
    void tc_plain(const CUtensorMap *mA, const CUtensorMap *mB, S *out, int64_t Mrows, int64_t Ncols, int64_t Kdim, int64_t ldo, bool sym = false) {
        tc::Params q = tc_base_params();
        q.sym = (sym && !getenv("CMF_S2_FULL")) ? 1 : 0;
        q.tiles_n = cdiv(Ncols, tc::BN);
        q.nkb = cdiv(Kdim, tc::BK);
        q.units = q.tiles_n * cdiv(Mrows, tc::BM);
        q.out = out; q.Mrows = Mrows; q.Ncols = Ncols; q.ldo = ldo;
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        tc::tc_kernel<tc::TC_PLAIN><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(mA[0], mA[1], mB[0], mB[1], q);
        post_launch();
        if (q.sym) {
            tc::mirror_upper_kernel<<<dim3((unsigned)cdiv(Mrows, 256), (unsigned)Mrows), 256, 0, stream>>>(out, Mrows, ldo);
            post_launch();
        }
    }
    // denomW = G * Wi (mult.jl:28,33): G is built straight into bf16 planes in the K-dim order of Wc
    void tc_denomW(int64_t j0, int64_t j1) {
        if (getenv("CMF_G_DIRECT"))          // element-wise form (kept for A/B)
            tc::build_G_split_kernel<<<(unsigned)cdiv(KL() * tcs.KLp, 256), 256, 0, stream>>>(
                exch1.p, exch1.p + L * K * K, tcs.Gc_hi.p, tcs.Gc_lo.p, K, L, tcs.Kp, tcs.KLp);
        else
            tc::build_G_split_diag_kernel<<<(unsigned)cdiv((2 * L - 1) * K * K, 256), 256, 0, stream>>>(
                exch1.p, exch1.p + L * K * K, tcs.Gc_hi.p, tcs.Gc_lo.p, K, L, tcs.Kp, tcs.KLp);
        post_launch();
        tc_split_W();
        if (j0 == 0 && j1 == KL()) {
            tc_plain(tcs.mGc, tcs.mWcB, denW.p, KL(), N, tcs.KLp, N);
        } else {
            // rows [j0, j1) of G only (the W update is sharded by rows over the ranks): A maps over that row block
            CUtensorMap mg[2];
            __nv_bfloat16 *gc[2] = {tcs.Gc_hi.p, tcs.Gc_lo.p};
            for (int i = 0; i < 2; ++i)
                mg[i] = make_map_2d(gc[i] + j0 * tcs.KLp, (uint64_t)tcs.KLp, (uint64_t)(j1 - j0), (uint64_t)tcs.KLp * 2, tc::BK, tc::BM, CU_TENSOR_MAP_SWIZZLE_64B);
            tc_plain(mg, tcs.mWcB, denW.p + j0 * N, j1 - j0, N, tcs.KLp, N);
        }
    }
    // Gram partial Rg[d][k][k'] = sum_u H[u][k] H[u+d][k'] via tensor cores (needs tc_split_H(true) and (false) done)
    void tc_gram() {
        tc::Params q = tc_base_params();
        q.N = K;                                   // output row stride / column bound: Rg is [L][K][K]
        q.tiles_m = tcs.tiles_m; q.tiles_n = 1; q.split_len = tcs.split_len_g; q.tau_hi = Tl + (L - 1);
        q.units = tcs.tiles_m * tcs.nsplit_g;
        q.part = corr_part.p;
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        tc::tc_kernel<tc::TC_CORR><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(tcs.mHm[0], tcs.mHm[1], tcs.mHmn[0], tcs.mHmn[1], q);
        post_launch();
        const int64_t n = L * K * K;
        reduce_partials_kernel<S><<<(unsigned)cdiv(n, 256), 256, 0, stream>>>(corr_part.p, tcs.nsplit_g, n, nullptr, exch1.p);
        post_launch();
    }
    // denomH = C (*) H via tensor cores (mult.jl:44,48); needs lag_tables() and tc_split_H(false) done
    void tc_denomH(bool resplit_C = true) {
        if (resplit_C) {
            tc::split_C_kernel<<<(unsigned)cdiv(tcs.rows_c * tcs.Kp, 256), 256, 0, stream>>>(Cf.p, tcs.Cc_hi.p, tcs.Cc_lo.p, K, 2 * L - 1, tcs.Kp, tcs.rows_c);
            post_launch();
        }
        tc::Params q = tc_base_params();
        q.groups = tcs.groups_c; q.nblocks = cdiv(tcs.Kp, tc::BK); q.own = tc::BN - (tcs.G - 1);
        q.units = cdiv(Tl, q.own);
        q.out = denH.p;
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        tc::tc_kernel<tc::TC_TRANS><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(tcs.mCu[0], tcs.mCu[1], tcs.mHk[0], tcs.mHk[1], q);
        post_launch();
    }
    // numH via tensor cores (mult.jl:47)
    void tc_transconv() {
        tc_split_X();
        tc_split_W();
        tc::Params q = tc_base_params();
        q.groups = tcs.groups; q.nblocks = cdiv(N, tc::BK); q.own = tc::BN - (tcs.G - 1);
        q.units = cdiv(Tl, q.own);
        q.out = numH.p;
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        {
            const char *e = getenv("CMF_LOCKSTEP_TRANS");      // k-block window; 0 (default) disables
            const int w = e ? atoi(e) : 0;
            if (w > 0 && q.units >= (int64_t)grid) {
                if (lockstep.n == 0) lockstep.alloc(1024);
                CK(cudaMemsetAsync(lockstep.p, 0, lockstep.n * sizeof(int), stream));
                q.lockstep = lockstep.p; q.lockstep_window = w;
            }
        }
        prof_begin(PROF_TRANSCONV);
        if (q.lockstep != nullptr) {
            void *args[] = {&tcs.mWu[0], &tcs.mWu[1], &tcs.mXk[0], &tcs.mXk[1], &q};
            CK(cudaLaunchCooperativeKernel((void *)tc::tc_kernel<tc::TC_TRANS>, dim3(grid), dim3(tc::THREADS), args, tc::SMEM_BYTES, stream));
        } else {
            tc::tc_kernel<tc::TC_TRANS><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(tcs.mWu[0], tcs.mWu[1], tcs.mXk[0], tcs.mXk[1], q);
        }
        prof_end();
        post_launch();
    }
    // sum of squared residuals via tensor cores (mult.jl:55-57); returns the number of partials written
    int64_t tc_conv_loss() {
        tc_split_W();
        tc_split_H(false);
        tc::Params q = tc_base_params();
        q.tiles_n = cdiv(N, tc::BM);
        q.nkb = tcs.KLp / tc::BK;
        q.units = q.tiles_n * cdiv(Tl, tc::BN);
        q.X = X.p; q.partial = loss_part.p;
        const unsigned grid = (unsigned)std::min<int64_t>(q.units, tcs.num_sms);
        prof_begin(PROF_CONV);
        tc::tc_kernel<tc::TC_CONV><<<grid, tc::THREADS, tc::SMEM_BYTES, stream>>>(tcs.mWc[0], tcs.mWc[1], tcs.mHw[0], tcs.mHw[1], q);
        prof_end();
        post_launch();
        return tc::EPI_WARPS * q.units;
    }

    ~Ctx() {
        if (tracing) trace_dump();
        if (own_stream && stream) cudaStreamDestroy(stream);
    }

    // splits of the tau sum of corr_kernel so that the grid has ~592 CTAs; Kc components (default K), nrest restarts
    void plan_split(int64_t Nin, int64_t tau_hi, int &nsplit, int64_t &split_len, int64_t Kc = 0, int64_t nrest = 1) {
        const int64_t ngrp = cdiv(L, 8);
        const int64_t bxy = cdiv(Nin, 128) * cdiv((Kc ? Kc : K) * ngrp, CORR_PB) * nrest;
        int64_t ns = std::min<int64_t>(std::max<int64_t>(cdiv(592, bxy), 1), 64);
        split_len = cdiv(cdiv(tau_hi, ns), CORR_BTAU) * CORR_BTAU;
        if (split_len < CORR_BTAU) split_len = CORR_BTAU;
        nsplit = (int)cdiv(tau_hi, split_len);
    }

    // CMF_TRACE=1: an event after every launch; the destructor prints, per call site, the live stream time between consecutive
    // events (= the kernel plus whatever gap preceded it, at the clocks of the real run -- ncu's per-kernel times are not)
    struct TraceEv { cudaEvent_t e; const char *fn; int line; };
    std::vector<TraceEv> trace;
    const bool tracing = getenv("CMF_TRACE") && atoi(getenv("CMF_TRACE")) > 0;
    void post_launch(const char *fn = __builtin_FUNCTION(), int line = __builtin_LINE()) {
        ++launches;
        CK(cudaGetLastError());
        if (tracing) {
            TraceEv t; t.fn = fn; t.line = line;
            cudaEventCreate(&t.e);
            cudaEventRecord(t.e, stream);
            trace.push_back(t);
        }
    }
    void trace_dump() {
        if (trace.size() < 2) return;
        cudaStreamSynchronize(stream);
        struct Agg { double ms = 0.0; int64_t n = 0; };
        std::map<std::pair<std::string, int>, Agg> agg;
        const size_t skip = getenv("CMF_TRACE_SKIP") ? (size_t)atoll(getenv("CMF_TRACE_SKIP")) : 0;
        double total = 0.0;
        for (size_t i = std::max<size_t>(1, skip); i < trace.size(); ++i) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, trace[i - 1].e, trace[i].e) != cudaSuccess) continue;
            Agg &g = agg[{trace[i].fn, trace[i].line}];
            g.ms += ms; ++g.n; total += ms;
        }
        fprintf(stderr, "CMF_TRACE: %zu launches, %.3f ms between the first and last traced event (launches before #%zu skipped)\n", trace.size(), total, skip);
        for (auto &kv : agg)
            fprintf(stderr, "CMF_TRACE %-28s:%-5d n=%-6lld total %10.3f ms  mean %9.4f ms  %5.1f%%\n", kv.first.first.c_str(), kv.first.second,
                    (long long)kv.second.n, kv.second.ms, kv.second.ms / (double)kv.second.n, 100.0 * kv.second.ms / total);
        for (auto &t : trace) cudaEventDestroy(t.e);
        trace.clear();
    }

    // ---------------------------------------------------------------- kernel launch helpers
    // est over local columns [t_lo, t_hi) from (Wsrc, Hsrc) with dims (Kc, Lc).
    // per_restart: one grid slice z per restart of a batch handle (rank K_r, W rows l*C + off_r + k, H columns t*C + off_r + k,
    // Kc = the largest K_r), writing its partials at partial + z*part_rs
    void launch_conv(const S *Wsrc, const S *Hsrc, int64_t Kc, int64_t Lc, int64_t h_lo, int64_t h_hi,
                     int64_t t_lo, int64_t t_hi, int flags, S *out, double *partial, uint64_t seed = 0,
                     double noise = 0.0, bool per_restart = false, int64_t part_rs = 0) {
        if (t_hi <= t_lo) return;
        ConvArgs<S> a;
        a.Wi = Wsrc; a.H = Hsrc; a.X = X.p; a.out = out; a.partial = partial;
        a.N = N; a.K = Kc; a.L = Lc; a.t_lo = t_lo; a.t_hi = t_hi; a.h_lo = h_lo; a.h_hi = h_hi;
        a.flags = flags; a.seed = seed; a.t_global0 = t0; a.noise = noise;
        a.mask = pgd_mask.n ? pgd_mask.p : nullptr; a.lossf = pgd_loss;
        a.ldw = a.ldh = per_restart ? b_C : Kc; a.part_rs = part_rs; a.tab = per_restart ? b_tab.p : nullptr;
        const int Lpad = (int)(cdiv(Lc, 8) * 8);
        const int HW = BT + Lpad - 1;
        const size_t ws_bytes = (size_t)CONV_LC * BN * sizeof(S);
        const size_t budget = 160 * 1024 - ws_bytes;
        int KC = (int)std::min<int64_t>(Kc, (int64_t)(budget / ((size_t)HW * sizeof(S))));
        REQUIRE(KC >= 1, "conv: L too large for the shared-memory H window");
        a.KC = KC;
        const size_t smem = (size_t)KC * HW * sizeof(S) + ws_bytes;
        auto kern = conv_kernel<S, TN, TT, TY>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dim3 grid((unsigned)cdiv(t_hi - t_lo, BT), (unsigned)cdiv(N, BN), (unsigned)(per_restart ? R : 1));
        prof_begin(PROF_CONV);
        kern<<<grid, dim3(16, TY), smem, stream>>>(a);
        prof_end();
        post_launch();
    }
    int conv_nblocks(int64_t t_lo, int64_t t_hi) const { return (int)(cdiv(N, BN) * cdiv(t_hi - t_lo, BT)); }

    // nrest > 1: dst[r] = sum of part[r*n .. r*n+n)
    void reduce_scalar(const double *part, int64_t n, double *dst, int nrest = 1) {
        reduce_sum_kernel<<<(unsigned)nrest, 1024, 0, stream>>>(part, n, dst);
        post_launch();
    }
    double fetch_scalar(const double *dst) {
        double v;
        CK(cudaMemcpyAsync(&v, dst, sizeof(double), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        return v;
    }

    // out[t][k] for t in [0, t_out).  per_restart: denomH of a batch handle, one grid slice per restart (TransArgs::tab), with
    // Nin = Kout = the largest K_r and row stride ldo (no split over units unless R = 1).  split_need != nullptr: launch
    // nothing, return the elements of tr_part the call needs.
    void launch_transconv(const S *Wg, const S *Xin, S *out, int64_t Nin, int64_t Kout, int64_t Lin,
                          int64_t ldx, int64_t t_out, int64_t x_cols, bool per_restart = false, int64_t ldo = 0,
                          size_t *split_need = nullptr) {
        const int nrest = per_restart ? (int)R : 1;
        if (t_out <= 0) return;
        // choose TK / kgroups minimising padding
        int best_tk = 8, best_kg = 1;
        double best_waste = 1e30;
        const int tks[3] = {8, 5, 4};
        for (int tk : tks) {
            int kg = 1;
            while (kg < 16 && kg * tk < Kout) kg *= 2;
            const int64_t kp = (int64_t)kg * tk;
            const double waste = (double)(cdiv(Kout, kp) * kp - Kout) / (double)Kout;
            if (waste < best_waste - 1e-9) { best_waste = waste; best_tk = tk; best_kg = kg; }
        }
        int tg = std::max(128 / best_kg, 8);
        while (tg * best_kg > 32 && cdiv(t_out, (int64_t)tg * 8) < 296) tg /= 2;
        TransArgs<S> a;
        a.Wg = Wg; a.Xin = Xin; a.out = out; a.Nin = Nin; a.Kout = Kout; a.Lin = Lin; a.ldx = ldx;
        a.t_out = t_out; a.x_cols = x_cols; a.kgroups = best_kg; a.tgroups = tg;
        a.ldo = ldo ? ldo : Kout; a.tab = per_restart ? b_tab.p : nullptr;
        const int BTt = tg * 8, Lpad = (int)(cdiv(Lin, 8) * 8);
        const int XW = BTt + Lpad, XWP = XW + XW / 8 + 1, KP = best_kg * best_tk;
        const size_t smem = ((size_t)TR_NC * XWP + (size_t)8 * TR_NC * KP) * sizeof(S);
        REQUIRE(smem <= 200 * 1024, "transconv: L too large for the shared-memory window");
        dim3 grid((unsigned)cdiv(t_out, BTt), (unsigned)cdiv(Kout, KP), (unsigned)nrest);
        const int nthr = best_kg * tg;
        // small problems (configs 1-2: T = 2000 gives 8 CTAs) do not fill the device over (t, k) tiles alone: split the sum over
        // units across blockIdx.z into partial outputs and add them in a fixed order (deterministic)
        int nsplit = 1;
        a.n_chunk = cdiv(Nin, TR_NC) * TR_NC; a.part_stride = 0;
        const int64_t ctas = (int64_t)grid.x * grid.y;
        if (nrest == 1 && ctas < 296 && Nin >= 64) {
            const int64_t want = std::min<int64_t>(std::min<int64_t>(cdiv(Nin, 32), cdiv(296, ctas)), 32);
            a.n_chunk = cdiv(cdiv(Nin, want), TR_NC) * TR_NC;
            nsplit = (int)cdiv(Nin, a.n_chunk);
            if (nsplit > 1) {
                a.part_stride = t_out * Kout;
                const size_t need = (size_t)nsplit * (size_t)a.part_stride;
                if (split_need) { *split_need = need; return; }
                if (tr_part.n < need) tr_part.alloc(need);
                a.out = tr_part.p;
                a.ldo = Kout;
                grid.z = (unsigned)nsplit;
            }
        }
        if (split_need) { *split_need = 0; return; }
        a.nsplit = nsplit;
#define LAUNCH_TR(TKV)                                                                             \
    {                                                                                              \
        auto kern = transconv_kernel<S, TKV, 8>;                                                   \
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));    \
        kern<<<grid, nthr, smem, stream>>>(a);                                                     \
    }
        if (Nin == N) prof_begin(PROF_TRANSCONV);
        if (best_tk == 8) LAUNCH_TR(8) else if (best_tk == 5) LAUNCH_TR(5) else LAUNCH_TR(4)
#undef LAUNCH_TR
        prof_end();
        post_launch();
        if (nsplit > 1) {
            sum_parts_kernel<S><<<(unsigned)cdiv(a.part_stride, 256), 256, 0, stream>>>(tr_part.p, out, a.part_stride, a.part_stride, nsplit);
            post_launch();
        }
    }
    DevBuf<S> tr_part;     // partial outputs of the N-split transposed convolution

    // out_S / out_D [(l*K+k)*Nin + n] = sum_tau hm(tau-l)[k] Xin[tau][n].  hm = Hs (default: this handle's H) with Kc
    // components (default K) and row stride ldh (default Kc).  per_restart is the per-restart Gram of a batch handle: Xin and
    // Hs are both the stacked H, Nin = Kc = the largest K_r, and restart z reads its K_r columns at off_r and writes
    // out_d + ex_r (CorrArgs::tab).
    void launch_corr(const S *Xin, int64_t Nin, int64_t ldx, int64_t tau_hi, int nsplit, int64_t split_len,
                     S *out_s, double *out_d, const S *Hs = nullptr, int64_t Kc = 0, int64_t ldh = 0, bool per_restart = false) {
        if (!Hs) Hs = H;
        if (!Kc) Kc = K;
        CorrArgs<S> a;
        a.H = Hs; a.Xin = Xin; a.part = corr_part.p; a.Nin = Nin; a.K = Kc; a.L = L; a.ldx = ldx;
        a.u_hi = Tl; a.tau_hi = tau_hi; a.split_len = split_len;
        a.ldh = ldh ? ldh : Kc; a.nsplit = nsplit;
        const int64_t n = L * Kc * Nin;
        const BatchRest *tab = per_restart ? b_tab.p : nullptr;
        const int nrest = per_restart ? (int)R : 1;
        a.tab = tab;
        const int64_t ngrp = cdiv(L, 8);
        dim3 grid((unsigned)cdiv(Nin, 128), (unsigned)cdiv(Kc * ngrp, CORR_PB), (unsigned)(nsplit * nrest));
        if (Nin == N) prof_begin(PROF_CORR);
        corr_kernel<S><<<grid, dim3(16, 16), 0, stream>>>(a);
        prof_end();
        post_launch();
        reduce_partials_kernel<S><<<dim3((unsigned)cdiv(n, 256), (unsigned)nrest), 256, 0, stream>>>(corr_part.p, nsplit, n, out_s, out_d, tab, L);
        post_launch();
    }

    static GemmRows rows(int64_t ld) { return GemmRows{ld, INT64_MAX, 0, RANK_NONE}; }
    template <bool TB>
    void launch_gemm(const S *A, const S *B, S *C, int64_t M, int64_t Nn, int64_t Kg, int64_t lda, int64_t ldb,
                     int64_t ldc) {
        launch_gemm_rows<TB>(A, B, C, M, Nn, Kg, rows(lda), rows(ldb), rows(ldc), false);
    }
    // per_restart: one grid slice per restart of a batch handle, extents for the largest K_r (GemmRows::rank)
    template <bool TB>
    void launch_gemm_rows(const S *A, const S *B, S *C, int64_t M, int64_t Nn, int64_t Kg, GemmRows ra, GemmRows rb, GemmRows rc,
                          bool per_restart) {
        dim3 grid((unsigned)cdiv(Nn, 64), (unsigned)cdiv(M, 64), (unsigned)(per_restart ? R : 1));
        gemm_kernel<S, TB><<<grid, 256, 0, stream>>>(A, B, C, M, Nn, Kg, ra, rb, rc, per_restart ? b_tab.p : nullptr, L);
        post_launch();
    }

    // mult.jl:37-38 / 51-52.  dot_dst != nullptr additionally leaves <num, x'> (new x) there: the expansion loss's <numH, H'>
    // comes out of the H update for free.  Returns whether the inner product was produced.
    DevBuf<double> mu_part;
    bool launch_mu(S *x, const S *num, const S *den, double l1, double l2, int64_t n, double *dot_dst = nullptr) {
        if constexpr (is_f32) {
            const bool aligned = (((uintptr_t)x | (uintptr_t)num | (uintptr_t)den) & 15) == 0;
            if (aligned && n % 4 == 0 && n >= 4096) {
                const unsigned grid = (unsigned)std::min<int64_t>(cdiv(n / 4, 256), 148 * 8);
                if (dot_dst && mu_part.n == 0) mu_part.alloc(148 * 8);
                mu_update_vec4_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<float4 *>(x), reinterpret_cast<const float4 *>(num),
                                                                reinterpret_cast<const float4 *>(den), (float)l1, (float)l2, n / 4,
                                                                dot_dst ? mu_part.p : nullptr);
                post_launch();
                if (dot_dst) reduce_scalar(mu_part.p, grid, dot_dst);
                return dot_dst != nullptr;
            }
        }
        mu_update_kernel<S><<<(unsigned)cdiv(n, 256), 256, 0, stream>>>(x, num, den, (S)l1, (S)l2, n);
        post_launch();
        return false;
    }

    // ---------------------------------------------------------------- what a change of X, W or H makes stale
    // Every change of X, W or H goes through these.  Elsewhere a cache flag is written only by engine setup and by the code
    // that recomputes or consumes the cached operand.
    void x_changed() {                    // planes / spectrum of X, numH
        tcs.x_dirty = fds.x_dirty = true;
        numH_valid = numH_dot_valid = false;
        calib_reset();
    }
    void w_changed() {                    // planes / spectra of W, numH and W W'
        tcs.w_dirty = fds.w_dirty = fds.wx_dirty = true;
        numH_valid = numH_dot_valid = false;
    }
    void h_changed() {           // Gram partial, spectra of H; numH too (the HALS sweep leaves Q there)
        gram_valid = false; fds.h_dirty = true; fds.hf2_valid = false;
        numH_valid = numH_dot_valid = false;
    }
    void factors_replaced() { w_changed(); h_changed(); calib_reset(); }

    // ---------------------------------------------------------------- data
    void set_data(const void *Xh, int64_t first_col) {
        REQUIRE(Xh != nullptr, "set_data: null pointer");
        REQUIRE(first_col <= t0, "set_data: host array starts after the shard's first column");
        const int64_t hi = std::min(t1 + (L - 1), T);
        CK(cudaMemsetAsync(X.p, 0, X.n * sizeof(S), stream));
        const S *src = static_cast<const S *>(Xh) + (t0 - first_col) * N;
        CK(cudaMemcpyAsync(X.p, src, (size_t)((hi - t0) * N) * sizeof(S), cudaMemcpyHostToDevice, stream));
        finish_data();
    }
    void get_data(void *X_out, int with_halo) {
        const int64_t cols = with_halo ? std::min(t1 + (L - 1), T) - t0 : Tl;
        CK(cudaMemcpyAsync(X_out, X.p, (size_t)(cols * N) * sizeof(S), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    }
    void finish_data() {
        x_changed();
        data_sumsq_local = data_sumsq();
        data_norm = std::sqrt(data_sumsq_local);
        pgd_cur_loss = data_norm;
        have_data = true;
    }
    double data_sumsq() {
        dot_partial_kernel<S><<<1024, 256, 0, stream>>>(X.p, X.p, Tl * N, loss_part.p);
        post_launch();
        reduce_scalar(loss_part.p, 1024, scal.p);
        return fetch_scalar(scal.p);
    }

    void synth_data(uint64_t seed, int64_t Kt, int64_t Lt, double p_h, double noise) {
        REQUIRE(Kt >= 1 && Lt >= 1, "synth_data: bad ground-truth dims");
        DevBuf<S> Wt, Ht;
        Wt.alloc((size_t)(Kt * Lt * N));
        const int64_t cols_out = std::min(Tl + (L - 1), T - t0);   // local columns to produce
        const int64_t hcols = cols_out + (Lt - 1);
        Ht.alloc((size_t)(hcols * Kt));
        synth_W_kernel<S><<<(unsigned)cdiv(N, 128), 128, 0, stream>>>(Wt.p, Kt, N, Lt, seed, 0.1, 0.2);
        post_launch();
        synth_H_kernel<S><<<(unsigned)cdiv(hcols * Kt, 256), 256, 0, stream>>>(Ht.p, Kt, t0 - (Lt - 1), hcols, T, seed, p_h);
        post_launch();
        CK(cudaMemsetAsync(X.p, 0, X.n * sizeof(S), stream));
        launch_conv(Wt.p, Ht.p + (Lt - 1) * Kt, Kt, Lt, -(Lt - 1), cols_out, 0, cols_out, 8, X.p, nullptr, seed, noise);
        CK(cudaStreamSynchronize(stream));
        finish_data();
    }

    // ---------------------------------------------------------------- factors
    void set_factors(const void *Wh, const void *Hh, int64_t first_col) {
        REQUIRE(Wh && Hh, "set_factors: null pointer");
        const int64_t lo = std::max<int64_t>(t0 - (L - 1), 0), hi = std::min(t1 + (L - 1), T);
        REQUIRE(first_col <= lo, "set_factors: host H starts after the shard's left halo");
        CK(cudaMemcpyAsync(Wtmp.p, Wh, Wi.n * sizeof(S), cudaMemcpyHostToDevice, stream));
        w_julia_to_internal<S><<<(unsigned)cdiv(KL() * N, 256), 256, 0, stream>>>(Wtmp.p, Wi.p, K, N, L, K);
        post_launch();
        CK(cudaMemsetAsync(Hbuf.p, 0, Hbuf.n * sizeof(S), stream));
        const S *src = static_cast<const S *>(Hh) + (lo - first_col) * K;
        CK(cudaMemcpyAsync(H + (lo - t0) * K, src, (size_t)((hi - lo) * K) * sizeof(S), cudaMemcpyHostToDevice, stream));
        CK(cudaStreamSynchronize(stream));
        have_factors = true;
        factors_replaced();
        pgd_stepW = pgd_stepH = 5.0;            // a new rule instance (pgd.jl:147-149)
        pgd_cur_loss = data_norm;
    }

    void init_rand(uint64_t seed) {
        // W in Julia order (k + K*(n + N*l)) so the draw for element (k,n,l) does not depend on layout
        uniform_kernel<S><<<(unsigned)cdiv(KL() * N, 256), 256, 0, stream>>>(Wtmp.p, KL() * N, seed, 100, 0);
        post_launch();
        w_julia_to_internal<S><<<(unsigned)cdiv(KL() * N, 256), 256, 0, stream>>>(Wtmp.p, Wi.p, K, N, L, K);
        post_launch();
        const int64_t lo = std::max<int64_t>(t0 - (L - 1), 0), hi = std::min(t1 + (L - 1), T);
        CK(cudaMemsetAsync(Hbuf.p, 0, Hbuf.n * sizeof(S), stream));
        uniform_kernel<S><<<(unsigned)cdiv((hi - lo) * K, 256), 256, 0, stream>>>(H + (lo - t0) * K, (hi - lo) * K, seed, 101, lo * K);
        post_launch();
        CK(cudaStreamSynchronize(stream));
        have_factors = true;
        factors_replaced();
    }

    void init_scale_partials(double out[2]) {
        REQUIRE(have_data && have_factors, "init_scale_partials: data and factors must be set");
        const int nb = conv_nblocks(0, Tl);
        launch_conv(Wi.p, H, K, L, -(L - 1), Tl + (L - 1), 0, Tl, 16, nullptr, loss_part.p);
        // partial layout: [2*b] = <est, X>, [2*b+1] = ||est||^2  -> de-interleave by strided sums
        std::vector<double> hp((size_t)2 * nb);
        CK(cudaMemcpyAsync(hp.data(), loss_part.p, hp.size() * sizeof(double), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        double a = 0.0, b = 0.0;
        for (int i = 0; i < nb; ++i) { a += hp[2 * i]; b += hp[2 * i + 1]; }
        out[0] = a; out[1] = b;
    }

    void scale_factors(double s) {
        scale_kernel<S><<<(unsigned)cdiv(KL() * N, 256), 256, 0, stream>>>(Wi.p, (S)s, KL() * N);
        post_launch();
        scale_kernel<S><<<(unsigned)cdiv((int64_t)Hbuf.n, 256), 256, 0, stream>>>(Hbuf.p, (S)s, (int64_t)Hbuf.n);
        post_launch();
        factors_replaced();
    }

    void get_factors(void *Wo, void *Ho) {
        if (Wo) {
            w_internal_to_julia<S><<<(unsigned)cdiv(KL() * N, 256), 256, 0, stream>>>(Wi.p, Wtmp.p, K, N, L, K);
            post_launch();
            CK(cudaMemcpyAsync(Wo, Wtmp.p, Wi.n * sizeof(S), cudaMemcpyDeviceToHost, stream));
        }
        if (Ho) CK(cudaMemcpyAsync(Ho, H, (size_t)(Tl * K) * sizeof(S), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    }

    // ---------------------------------------------------------------- batch of R MultUpdate restarts (cmf_create_batch[_ranks])
    // Restart-stacked layout: restart r has rank K_r and owns components [off_r, off_r + K_r) of a stacked component axis of
    // width C = sum K_r (off_r = sum_{q<r} K_q): H is [t][C] with column off_r + k, Wi has rows j' = l*C + off_r + k.  numW
    // (mult.jl:32) and numH (mult.jl:47) are linear in the factor they contract with X, so ONE correlation and ONE transposed
    // convolution with C components serve every restart and X is read once per step.  Everything else is block-diagonal per
    // restart and runs as one launch with a restart grid index, sized for K = max K_r: each block reads its restart's rank and
    // offsets from the table b_tab, so the launches of an iteration depend neither on R nor on the ranks.  Equal ranks give
    // off_r = r*K and the offsets of the uniform layout.
    std::vector<int64_t> b_K;        // K_r of every restart
    std::vector<BatchRest> b_rest;   // host copy of b_tab (filled by batch_buffers)
    int64_t b_C = 0;                 // C = sum K_r
    DevBuf<BatchRest> b_tab;
    DevBuf<int> b_col;               // [C]: the restart that owns each stacked component
    DevBuf<double> b_reg, b_vals;    // [R][4] = (l1W, l2W, l1H, l2H) per restart; R per-restart scalars
    DevBuf<int> b_active;            // 0 = the restart has converged: the updates leave its factors alone
    int64_t b_exch(int64_t Kr) const { return L * Kr * Kr + (L - 1) * Kr + 1; }   // doubles of one restart's Gram + H tail block in exch1
    int64_t b_tail_blocks(int64_t Kr) const { return cdiv((2 * L - 1) * Kr, 256); }
    GemmRows b_wrows() const { return GemmRows{N, INT64_MAX, b_C * N, RANK_W}; }   // W_r: rows l*K_r + k of restart r
    GemmRows b_grows() const { return GemmRows{0, INT64_MAX, 0, RANK_G}; }         // G_r / S2_r: K_r L x K_r L blocks

    // Walks every device buffer of a batch handle: returns the bytes, and allocates them when `alloc` is set (so the footprint
    // checked before allocating is what is allocated).  Lays out the per-restart blocks in b_rest.
    size_t batch_buffers(bool alloc) {
        size_t bytes = 0;
        auto take = [&](auto &buf, int64_t count) {
            bytes += (size_t)count * sizeof(*buf.p);
            if (alloc) buf.alloc((size_t)count);
        };
        const int64_t hal = L - 1, KLR = L * b_C;
        plan_split(N, Tl + hal, nsplit_w, split_w, b_C, 1);
        plan_split(K, Tl + hal, nsplit_g, split_g, K, R);
        b_rest.assign((size_t)R, BatchRest{});
        BatchRest e{};                                    // running offsets; the totals after the last restart
        for (int64_t r = 0; r < R; ++r) {
            const int64_t Kr = b_K[(size_t)r];
            e.K = Kr;
            b_rest[(size_t)r] = e;
            e.off += Kr; e.gs += (Kr * L) * (Kr * L); e.cf += (2 * L - 1) * Kr * Kr; e.ex += b_exch(Kr);
            e.cp += (int64_t)nsplit_g * L * Kr * Kr; e.tp += b_tail_blocks(Kr) * hal * Kr;
        }
        size_t tr_need = 0;
        launch_transconv(nullptr, nullptr, nullptr, N, b_C, L, N, Tl, Tl + hal, false, 0, &tr_need);
        const int nb = conv_nblocks(0, Tl);
        take(X, (Tl + hal) * N);
        take(Hbuf, (Tl + 2 * hal) * b_C);
        take(Wi, KLR * N); take(Wtmp, KLR * N); take(numW, KLR * N); take(denW, KLR * N);
        take(GS, e.gs);
        take(Cf, e.cf);
        take(numH, Tl * b_C); take(denH, Tl * b_C);
        take(exch1, e.ex);
        take(corr_part, std::max<int64_t>((int64_t)nsplit_w * KLR * N, e.cp));
        take(loss_part, std::max<int64_t>(2 * nb * R, 4096));
        take(tail_part, e.tp);
        take(tr_part, (int64_t)tr_need);
        take(scal, 8);
        take(b_reg, 4 * R); take(b_vals, R); take(b_active, R);
        take(b_tab, R); take(b_col, b_C);
        return bytes;
    }

    void init_batch() {
        CK(cudaSetDevice(device));
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        const size_t need = batch_buffers(false);
        if (need > free_b)
            throw CmfError(CMF_ERR_ARG, "batch handle: " + std::to_string(R) + " restarts need " + std::to_string(need) +
                                            " bytes of device memory (" + std::to_string(b_C) + " stacked components); " +
                                            std::to_string(free_b) + " bytes are free");
        CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        own_stream = true;
        H = nullptr;
        batch_buffers(true);
        H = Hbuf.p + (L - 1) * b_C;
        conv_blocks_max = conv_nblocks(0, Tl);
        std::vector<int> col((size_t)b_C);
        for (int64_t r = 0; r < R; ++r)
            for (int64_t k = 0; k < b_K[(size_t)r]; ++k) col[(size_t)(b_rest[(size_t)r].off + k)] = (int)r;
        CK(cudaMemcpyAsync(b_tab.p, b_rest.data(), (size_t)R * sizeof(BatchRest), cudaMemcpyHostToDevice, stream));
        CK(cudaMemcpyAsync(b_col.p, col.data(), col.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
        CK(cudaStreamSynchronize(stream));
    }

    // host: R Julia blocks W (K_r x N x L) and H (K_r x T), one after another; numH stages H (it is recomputed before every use)
    void batch_set_factors(const void *Wh, const void *Hh) {
        REQUIRE(Wh && Hh, "cmf_set_factors_batch: null pointer");
        CK(cudaMemcpyAsync(Wtmp.p, Wh, Wtmp.n * sizeof(S), cudaMemcpyHostToDevice, stream));
        w_julia_to_internal<S><<<dim3((unsigned)cdiv(KL() * N, 256), (unsigned)R), 256, 0, stream>>>(Wtmp.p, Wi.p, K, N, L, b_C, b_tab.p);
        post_launch();
        CK(cudaMemsetAsync(Hbuf.p, 0, Hbuf.n * sizeof(S), stream));
        CK(cudaMemcpyAsync(numH.p, Hh, numH.n * sizeof(S), cudaMemcpyHostToDevice, stream));
        h_stack_kernel<S><<<(unsigned)cdiv(b_C * Tl, 256), 256, 0, stream>>>(numH.p, H, b_C, Tl, b_tab.p, b_col.p, 1);
        post_launch();
        CK(cudaStreamSynchronize(stream));
        have_factors = true;
    }
    void batch_get_factors(void *Wo, void *Ho) {
        REQUIRE(have_factors, "no factors");
        if (Wo) {
            w_internal_to_julia<S><<<dim3((unsigned)cdiv(KL() * N, 256), (unsigned)R), 256, 0, stream>>>(Wi.p, Wtmp.p, K, N, L, b_C, b_tab.p);
            post_launch();
            CK(cudaMemcpyAsync(Wo, Wtmp.p, Wtmp.n * sizeof(S), cudaMemcpyDeviceToHost, stream));
        }
        if (Ho) {
            h_stack_kernel<S><<<(unsigned)cdiv(b_C * Tl, 256), 256, 0, stream>>>(H, numH.p, b_C, Tl, b_tab.p, b_col.p, 0);
            post_launch();
            CK(cudaMemcpyAsync(Ho, numH.p, numH.n * sizeof(S), cudaMemcpyDeviceToHost, stream));
        }
        CK(cudaStreamSynchronize(stream));
    }

    // out[2r] = <X, est_r>, out[2r+1] = ||est_r||^2 (model.jl:119-120), each summed over the conv blocks in the order of
    // init_scale_partials
    void batch_scale_partials(double *out) {
        REQUIRE(have_data && have_factors, "cmf_init_scale_partials_batch: data and factors must be set");
        const int nb = conv_nblocks(0, Tl);
        launch_conv(Wi.p, H, K, L, -(L - 1), Tl + (L - 1), 0, Tl, 16, nullptr, loss_part.p, 0, 0.0, true, 2 * nb);
        std::vector<double> hp((size_t)(2 * nb * R));
        CK(cudaMemcpyAsync(hp.data(), loss_part.p, hp.size() * sizeof(double), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        for (int64_t r = 0; r < R; ++r) {
            const double *p = hp.data() + 2 * nb * r;
            double a = 0.0, b = 0.0;
            for (int i = 0; i < nb; ++i) { a += p[2 * i]; b += p[2 * i + 1]; }
            out[2 * r] = a; out[2 * r + 1] = b;
        }
    }
    void batch_scale(const double *s) {
        CK(cudaMemcpyAsync(b_vals.p, s, (size_t)R * sizeof(double), cudaMemcpyHostToDevice, stream));
        scale_kernel<S><<<(unsigned)cdiv((int64_t)Wi.n, 256), 256, 0, stream>>>(Wi.p, S(1), (int64_t)Wi.n, b_vals.p, N, b_col.p, b_C);
        post_launch();
        scale_kernel<S><<<(unsigned)cdiv((int64_t)Hbuf.n, 256), 256, 0, stream>>>(Hbuf.p, S(1), (int64_t)Hbuf.n, b_vals.p, 1, b_col.p, b_C);
        post_launch();
        CK(cudaStreamSynchronize(stream));
    }

    // relative loss of every restart (mult.jl:55-57): one direct conv + residual pass with a restart index, one deterministic
    // reduction per restart, one copy of R doubles
    void batch_loss(double *out) {
        REQUIRE(have_data && have_factors, "loss: data and factors must be set first");
        const int nb = conv_nblocks(0, Tl);
        launch_conv(Wi.p, H, K, L, -(L - 1), Tl + (L - 1), 0, Tl, 4, nullptr, loss_part.p, 0, 0.0, true, nb);
        reduce_scalar(loss_part.p, nb, b_vals.p, (int)R);
        CK(cudaMemcpyAsync(out, b_vals.p, (size_t)R * sizeof(double), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        for (int64_t r = 0; r < R; ++r) out[r] = std::sqrt(std::max(out[r], 0.0)) / data_norm;
    }

    // reg = R x (l1W, l2W, l1H, l2H) and / or the R active flags (either may be NULL)
    void batch_set_state(const double *reg, const int *active) {
        if (reg) CK(cudaMemcpyAsync(b_reg.p, reg, (size_t)(4 * R) * sizeof(double), cudaMemcpyHostToDevice, stream));
        if (active) CK(cudaMemcpyAsync(b_active.p, active, (size_t)R * sizeof(int), cudaMemcpyHostToDevice, stream));
        CK(cudaStreamSynchronize(stream));
    }

    // update_motifs! (mult.jl:23-39) of every active restart
    void batch_update_motifs() {
        REQUIRE(have_data && have_factors, "update: data and factors must be set first");
        launch_corr(X.p, N, N, Tl + (L - 1), nsplit_w, split_w, numW.p, nullptr, H, b_C, b_C);          // numW, all restarts
        launch_corr(H, K, b_C, Tl + (L - 1), nsplit_g, split_g, nullptr, exch1.p, H, K, b_C, true);   // Gram_r
        if (L > 1) {
            h_tail_kernel<S><<<dim3((unsigned)cdiv((L - 1) * K, 256), (unsigned)R), 256, 0, stream>>>(H, exch1.p, K, L, Tl, 1, b_C,
                                                                                                   b_tab.p);
            post_launch();
        }
        build_G_kernel<S><<<dim3((unsigned)cdiv(KL() * KL(), 256), (unsigned)R), 256, 0, stream>>>(exch1.p, nullptr, GS.p, K, L,
                                                                                                    b_tab.p);
        post_launch();
        launch_gemm_rows<false>(GS.p, Wi.p, denW.p, KL(), N, KL(), b_grows(), b_wrows(), b_wrows(), true);     // denomW_r = G_r W_r
        mu_update_kernel<S><<<(unsigned)cdiv((int64_t)Wi.n, 256), 256, 0, stream>>>(Wi.p, numW.p, denW.p, S(0), S(0), (int64_t)Wi.n,
                                                                                     b_reg.p, b_active.p, N, b_col.p, b_C);
        post_launch();
    }

    // update_feature_maps! (mult.jl:42-58, without the loss) of every active restart
    void batch_update_feature_maps() {
        REQUIRE(have_data && have_factors, "update: data and factors must be set first");
        launch_transconv(Wi.p, X.p, numH.p, N, b_C, L, N, Tl, Tl + (L - 1));                                // numH, all restarts
        launch_gemm_rows<true>(Wi.p, Wi.p, GS.p, KL(), KL(), N, b_wrows(), b_wrows(), b_grows(), true);       // S2_r = W_r W_r'
        lag_table_kernel<S><<<dim3((unsigned)cdiv((2 * L - 1) * K * K, 256), (unsigned)R), 256, 0, stream>>>(GS.p, Cf.p, K, L, K, KL(),
                                                                                                          b_tab.p);
        post_launch();
        launch_transconv(Cf.p, Hbuf.p, denH.p, K, K, 2 * L - 1, b_C, Tl, Tl + 2 * (L - 1), true, b_C);
        if (L > 1) {                                                                                          // truncated tail
            denomH_tail_prefix_kernel<S><<<dim3((unsigned)b_tail_blocks(K), (unsigned)K, (unsigned)R), 256,
                                           (size_t)8 * (size_t)(L - 1) * sizeof(double), stream>>>(GS.p, H, tail_part.p, K, L, Tl,
                                                                                                    -(L - 1), K, KL(), b_C, b_tab.p);
            post_launch();
            denomH_tail_reduce_kernel<S><<<dim3((unsigned)cdiv((L - 1) * K, 256), (unsigned)R), 256, 0, stream>>>(tail_part.p, denH.p, K, L,
                                                                                                                Tl, 0, b_C, b_tab.p);
            post_launch();
        }
        mu_update_kernel<S><<<(unsigned)cdiv(Tl * b_C, 256), 256, 0, stream>>>(H, numH.p, denH.p, S(0), S(0), Tl * b_C, b_reg.p + 2,
                                                                                 b_active.p, 1, b_col.p, b_C);
        post_launch();
    }

    // ---------------------------------------------------------------- contractions
    // Each contraction picks its engine here and nowhere else: SIMT unless the tensor cores are on (never on fp64 handles),
    // then the frequency-domain engine where it is active, the time-domain one otherwise.

    // numW partial over the owned u (mult.jl:32): Xin = X incl. right halo
    void compute_numW() {
        if (!tc_active()) launch_corr(X.p, N, N, Tl + (L - 1), nsplit_w, split_w, numW.p, nullptr);
        else if constexpr (is_f32) { if (fd_active()) fd_corr(); else tc_corr(); }
    }
    // numH (mult.jl:47)
    void compute_numH() {
        if (!tc_active()) launch_transconv(Wi.p, X.p, numH.p, N, K, L, N, Tl, Tl + (L - 1));
        else if constexpr (is_f32) { if (fd_active()) fd_transconv(); else tc_transconv(); }
    }
    // denomW = G * Wi (mult.jl:28,33) for the unfolded rows [j0, j1); the frequency-domain engine runs it in the time domain
    void compute_denomW(int64_t j0, int64_t j1) {
        if (!tc_active()) {
            build_G();
            launch_gemm<false>(GS.p + j0 * KL(), Wi.p, denW.p + j0 * N, j1 - j0, N, KL(), KL(), N, N);
        } else if constexpr (is_f32) {
            tc_denomW(j0, j1);
        }
    }
    // W W' and its lag tables, then denomH = C (*) H on all owned columns (mult.jl:44,48), then the truncated tail
    void compute_denomH() {
        lag_tables();
        if (!tc_active()) launch_transconv(Cf.p, Hbuf.p, denH.p, K, K, 2 * L - 1, K, Tl, Tl + 2 * (L - 1));
        else if constexpr (is_f32) {
            if (fd_active()) fd_denomH();
            else { tc_split_H(false); tc_denomH(); }
        }
        if (is_last && L > 1) launch_denomH_tail();
    }
    // Gram partial Rg[d][k][k'] = sum_u H[u][k] H[u+d][k'] (owned u, right halo for u+d) and the H tail block
    void gram_partial() {
        if (!tc_active()) launch_corr(H, K, K, Tl + (L - 1), nsplit_g, split_g, nullptr, exch1.p);
        else if constexpr (is_f32) {
            if (fd_active()) fd_gram();
            else { tc_split_H(true); tc_split_H(false); tc_gram(); }
        }
        if (L > 1) {
            h_tail_kernel<S><<<(unsigned)cdiv((L - 1) * K, 256), 256, 0, stream>>>(H, exch1.p + L * K * K, K, L, Tl, is_last ? 1 : 0, K);
            post_launch();
        }
    }

    void build_G() {
        build_G_kernel<S><<<(unsigned)cdiv(KL() * KL(), 256), 256, 0, stream>>>(exch1.p, exch1.p + L * K * K, GS.p, K, L);
        post_launch();
    }

    // ---------------------------------------------------------------- MU (src/algs/mult.jl)
    void w_partials() {
        REQUIRE(have_data && have_factors, "update: data and factors must be set first");
        compute_numW();
        // the Gram partial is already resident when the expansion loss of the previous iteration computed it for the same H
        if (!gram_valid) gram_partial();
        gram_valid = false;     // the host all-reduces the buffer in place: it is consumed by this step
    }

    void w_apply(double l1W, double l2W) {
        if (alg == CMF_HALS) { hals_w_apply(l1W, l2W); return; }
        REQUIRE(alg == CMF_MULT, "the split-phase W update serves MultUpdate and HALSUpdate");
        w_denom_rows(0, KL());
        w_update_rows(l1W, l2W, 0, KL());
    }
    void w_denom_rows(int64_t j0, int64_t j1) { compute_denomW(j0, j1); }
    // mult.jl:37-38 on the rows [j0, j1) (the whole update when the range is everything)
    void w_update_rows(double l1W, double l2W, int64_t j0, int64_t j1) {
        launch_mu(Wi.p + j0 * N, numW.p + j0 * N, denW.p + j0 * N, l1W, l2W, (j1 - j0) * N);
        w_changed();
    }
    void w_rows_buffers(void **numw, void **w, int64_t *row_elems) { *numw = numW.p; *w = Wi.p; *row_elems = N; }

    // layout of the W W' product held in GS: S2[(l*s2_ks + k)*s2_ld + l'*s2_ks + k']
    int64_t s2_ks = 0, s2_ld = 0;

    void lag_tables() {
        if (!tc_active()) {
            launch_gemm<true>(Wi.p, Wi.p, GS.p, KL(), KL(), N, N, N, KL());              // S2 = Wi Wi'
            s2_ks = K; s2_ld = KL();
        } else if constexpr (is_f32) {
            tc_split_W();
            tc_plain(tcs.mWu, tcs.mWuB, GS.p, tcs.rows_u, tcs.rows_u, N, tcs.rows_u, true);   // S2 = Wu Wu' on tensor cores (lower tiles + mirror)
            s2_ks = tcs.Kp; s2_ld = tcs.rows_u;
        }
        lag_table_kernel<S><<<(unsigned)cdiv((2 * L - 1) * K * K, 256), 256, 0, stream>>>(GS.p, Cf.p, K, L, s2_ks, s2_ld);
        post_launch();
    }

    // truncated tail of denomH (the last L-1 columns, mult.jl:44,48 with the conv cut at T) from S2 = W W' in GS
    DevBuf<double> tail_part;
    void launch_denomH_tail() {
        const int nb = (int)cdiv((2 * L - 1) * K, 256);
        const size_t smem = (size_t)8 * (size_t)(L - 1) * sizeof(double);
        if (getenv("CMF_TAIL_DIRECT") || smem > 48 * 1024) {          // literal form (kept for A/B and very long lags)
            dim3 grid((unsigned)(L - 1), (unsigned)K);
            denomH_tail_kernel<S><<<grid, 256, 0, stream>>>(GS.p, H, denH.p, K, L, Tl, -(L - 1), s2_ks, s2_ld);
            post_launch();
            return;
        }
        const size_t need = (size_t)nb * (size_t)(L - 1) * (size_t)K;
        if (tail_part.n < need) tail_part.alloc(need);
        denomH_tail_prefix_kernel<S><<<dim3((unsigned)nb, (unsigned)K), 256, smem, stream>>>(GS.p, H, tail_part.p, K, L, Tl, -(L - 1), s2_ks, s2_ld,
                                                                                            K);
        post_launch();
        denomH_tail_reduce_kernel<S><<<(unsigned)cdiv((L - 1) * K, 256), 256, 0, stream>>>(tail_part.p, denH.p, K, L, Tl, nb, K);
        post_launch();
    }

    void h_update(double l1H, double l2H) {
        REQUIRE(have_data && have_factors, "update: data and factors must be set first");
        compute_numH();
        compute_denomH();
        // mult.jl:51-52; with the expansion loss in force the update also leaves <numH, H'> in scal[4]
        const bool dot = launch_mu(H, numH.p, denH.p, l1H, l2H, Tl * K, (loss_mode == 1 && alg == CMF_MULT) ? scal.p + 4 : nullptr);
        h_changed();
        numH_valid = (alg == CMF_MULT);     // numH and W W' are still those of the current W
        numH_dot_valid = dot;
    }

    double *scalars() { return scal.p; }   // device buffer of 8 doubles

    // Leaves the local loss scalars in scal.p without a host synchronisation and returns how many there are:
    //   1 (direct pass):  scal[0] = sum of squared residuals over the owned columns (mult.jl:55-57)
    //   2 (expansion):    scal[0] = <numH, H>, scal[1] = <W W', Htilde Htilde'> over the owned columns
    // scal[1] is zeroed in the direct case so that a fixed-size all-reduce of two doubles serves both.
    int loss_partial_dev() {
        REQUIRE(have_data && have_factors, "loss: data and factors must be set first");
        if (loss_mode == 1 && tc_active()) {
            // frequency-domain engine: numH and W W' are cheap, so the expansion also serves calls that find them stale
            // (the loss at the initial factors, after a W-only step, after the HALS sweep overwrote numH)
            if (!numH_valid && fd_active()) { compute_numH(); lag_tables(); numH_valid = true; numH_dot_valid = false; }
            if (numH_valid) { loss_partial_expansion_dev(); return 2; }
        }
        int64_t nb = conv_nblocks(0, Tl);
        if (!tc_active()) launch_conv(Wi.p, H, K, L, -(L - 1), Tl + (L - 1), 0, Tl, 4, nullptr, loss_part.p);  // mult.jl:55-57
        else if constexpr (is_f32) nb = (fd_active() && !getenv("CMF_FD_LOSS_TC")) ? fd_conv_loss() : tc_conv_loss();
        reduce_scalar(loss_part.p, nb, scal.p);
        CK(cudaMemsetAsync(scal.p + 1, 0, sizeof(double), stream));
        return 1;
    }

    // local sum of squared residuals (for the expansion: this shard's share of the global identity)
    double loss_partial() {
        const int n = loss_partial_dev();
        double bc[2];
        CK(cudaMemcpyAsync(bc, scal.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        return n == 2 ? data_sumsq_local - 2.0 * bc[0] + bc[1] : bc[0];
    }

    // ||conv(W,H) - X||^2 = ||X||^2 - 2 <transconv(W,X), H> + <W W', Htilde Htilde'>, summed over the owned columns
    // (the global sum over shards is exact; a single shard's value is not its own residual).  numH and W W' are
    // resident from the H update with the current W; the Gram of the new H is computed here and reused by the
    // next cmf_w_partials (the halos must not change in between).
    void loss_partial_expansion_dev() {
        gram_partial();
        gram_valid = true;
        if (getenv("CMF_G_DIRECT"))
            s2_dot_G_kernel<S><<<1024, 256, 0, stream>>>(GS.p, s2_ks, s2_ld, exch1.p, exch1.p + L * K * K, K, L, loss_part.p + 1024);
        else
            s2_dot_G_diag_kernel<S><<<1024, 256, 0, stream>>>(GS.p, s2_ks, s2_ld, exch1.p, exch1.p + L * K * K, K, L, loss_part.p + 1024);
        post_launch();
        reduce_scalar(loss_part.p + 1024, 1024, scal.p + 1);
        if (numH_dot_valid) {             // produced by the H update itself (consumed once: anything may happen before the next call)
            CK(cudaMemcpyAsync(scal.p, scal.p + 4, sizeof(double), cudaMemcpyDeviceToDevice, stream));
            numH_dot_valid = false;
            return;
        }
        dot_partial_kernel<S><<<1024, 256, 0, stream>>>(numH.p, H, Tl * K, loss_part.p);
        post_launch();
        reduce_scalar(loss_part.p, 1024, scal.p);
    }

    // ---------------------------------------------------------------- HALS (src/algs/hals.jl)
    // The HALS gradients come from the same four quantities as MU (no residual matrix is kept):
    //   P = R Htilde' = denomW - numW   (hals.jl:111 projections for every column at once)
    //   Q = transconv(W, R) = denomH - numH
    // with R = conv(W,H) - X (hals.jl:22).  w_partials() / the Gram all-reduce are shared with MU.
    void hals_w_apply(double l1W, double l2W) {
        compute_denomW(0, KL());
        if (tc_active()) build_G();                                           // G as a matrix for the sweep (GS; SIMT built it above)
        sub_kernel<S><<<(unsigned)cdiv(KL() * N, 256), 256, 0, stream>>>(numW.p, denW.p, numW.p, KL() * N);   // P
        post_launch();
        const size_t smem = (size_t)KL() * sizeof(S);
        REQUIRE(smem <= 200 * 1024, "HALS W sweep: K*L too large for shared memory");
        auto kern = hals_w_sweep_kernel<S>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)N, 256, smem, stream>>>(GS.p, numW.p, Wi.p, K, L, N, (S)l1W, (S)l2W);   // hals.jl:90-112
        post_launch();
        w_changed();
    }

    // Q = transconv(W, R) = denomH - numH on the owned columns (left in numH)
    void hals_h_prepare() {
        REQUIRE(have_data && have_factors, "update: data and factors must be set first");
        compute_numH();
        compute_denomH();
        sub_kernel<S><<<(unsigned)cdiv(Tl * K, 256), 256, 0, stream>>>(numH.p, denH.p, numH.p, Tl * K);        // Q
        post_launch();
    }
    // device pointers of the local Q and H (owned columns), element count
    void hals_h_local(void **q, void **h, int64_t *count) { *q = numH.p; *h = H; *count = Tl * K; }
    // rank 0 of a T-sharded HALS fit holds Q, H and Delta H of ALL columns during the sweep: the sweep is a chain of T
    // dependent steps per component (hals.jl:124-128) that more GPUs cannot shorten, so the shards' Q are gathered here,
    // swept once in the reference's order, and the new H is scattered back (DESIGN.md section 6)
    DevBuf<S> Qfull, Hfull, Dfull;
    void hals_h_full(void **q, void **h) {
        const size_t n = (size_t)(T * K);
        if (Qfull.n < n) { Qfull.alloc(n); Hfull.alloc(n); Dfull.alloc(n); }
        *q = Qfull.p; *h = Hfull.p;
    }

    // second-generation sweep (kernels_hals.cuh): rounds with a grid barrier, lane = component recurrences, 8 x 8 pull blocks.
    // Returns false when the handle / shape is outside its envelope (the wavefront kernel below then runs).
    DevBuf<float> h2_Hcm, h2_AD, h2_part, h2_coef;
    DevBuf<unsigned> h2_bar;
    int h2_max_ctas = -1;
    bool hals2_sweep(const S *Qp, S *Hp, int64_t Tt, const S *ct, double l1H, double l2H) {
        if constexpr (!is_f32) { return false; } else {
            if (L > hals2::LMAX || K > 128 || (L > 1 && ct == nullptr)) return false;
            if (const char *e = getenv("CMF_HALS_SWEEP")) { if (atoi(e) == 1) return false; }      // 1: first-generation wavefront kernel
            const int G = (int)cdiv(K, hals2::GS);
            const int n_block = G * (G - 1) / 2, n_diag = G, n_rec = (int)cdiv(K, 32);
            const int grid = n_block + n_diag + n_rec;
            const size_t smem = hals2::smem_bytes();
            if (h2_max_ctas < 0) {
                int per_sm = 0, sms = 0;
                CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
                cudaError_t e1 = cudaFuncSetAttribute(hals2::hals2_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                cudaError_t e2 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hals2::hals2_sweep_kernel, hals2::NT, smem);
                h2_max_ctas = (e1 == cudaSuccess && e2 == cudaSuccess) ? per_sm * sms : 0;
                if (e1 != cudaSuccess || e2 != cudaSuccess) cudaGetLastError();
            }
            if (grid > h2_max_ctas) return false;
            const int64_t nC = cdiv(Tt, hals2::CW), Tp = nC * hals2::CW;
            const size_t ncm = (size_t)hals2::cells_elems(K, nC), npart = (size_t)G * (size_t)K * hals2::RING * hals2::CW;
            if (h2_Hcm.n < ncm) { h2_Hcm.alloc(ncm); h2_AD.alloc(ncm); }
            if (h2_part.n < npart) h2_part.alloc(npart);
            dim3 tb(32, 8), tg((unsigned)cdiv(Tp, 32), (unsigned)cdiv(K, 32));
            hals2::hals2_prepare_kernel<<<tg, tb, 0, stream>>>(Qp, Hp, h2_AD.p, h2_Hcm.p, K, Tt, Tp);
            post_launch();
            if (h2_coef.n < (size_t)(K * 64)) h2_coef.alloc((size_t)(K * 64));
            hals2::hals2_coef_kernel<<<(unsigned)cdiv(K * 64, 256), 256, 0, stream>>>(Cf.p, h2_coef.p, K, L, (float)l2H);
            post_launch();
            if (h2_bar.n == 0) h2_bar.alloc(32);
            CK(cudaMemsetAsync(h2_bar.p, 0, sizeof(unsigned), stream));
            hals2::Args a;
            a.barrier = h2_bar.p;
            a.coef = h2_coef.p;
            a.Cf = Cf.p; a.Ct = ct; a.S2 = GS.p; a.Ks = s2_ks; a.ld = s2_ld;
            a.H_cm = h2_Hcm.p; a.AD_cm = h2_AD.p; a.part = h2_part.p;
            a.K = K; a.L = L; a.T = Tt; a.nC = nC;
            a.l1 = (float)l1H; a.l2 = (float)l2H;
            a.G = G; a.n_block_items = n_block; a.n_diag_items = n_diag; a.n_rec = n_rec;
            DevBuf<long long> dbgbuf;
            const bool dbg2 = getenv("CMF_HALS_DEBUG") && atoi(getenv("CMF_HALS_DEBUG")) == 1;
            if (dbg2) dbgbuf.alloc((size_t)12 * grid);
            a.dbg = dbg2 ? dbgbuf.p : nullptr;
            a.dbg_mode = getenv("CMF_HALS_DBGMODE") ? atoi(getenv("CMF_HALS_DBGMODE")) : 0;
            void *args[] = {&a};
            prof_begin(PROF_SWEEP);
            CK(cudaLaunchCooperativeKernel((void *)hals2::hals2_sweep_kernel, dim3((unsigned)grid), dim3(hals2::NT), args, smem, stream));
            prof_end();
            post_launch();
            hals2::hals2_finish_kernel<<<dim3((unsigned)cdiv(Tt, 32), (unsigned)cdiv(K, 32)), tb, 0, stream>>>(h2_Hcm.p, Hp, K, Tt, Tp);
            post_launch();
            if (dbg2) {      // kcycles of work per active round (barrier waits excluded): worst and mean CTA of every role
                std::vector<long long> hv((size_t)12 * grid);
                CK(cudaMemcpyAsync(hv.data(), dbgbuf.p, hv.size() * sizeof(long long), cudaMemcpyDeviceToHost, stream));
                CK(cudaStreamSynchronize(stream));
                fprintf(stderr, "hals2: SM clock over the launch %lld MHz (clock64 / globaltimer, CTA 0)\n", hv[7]);
                const char *names[3] = {"block items", "diagonal items", "recurrence warps"};
                const int lo[4] = {0, n_block, n_block + n_diag, grid};
                for (int r = 0; r < 3; ++r) {
                    double worst = 0.0, mean = 0.0; int cnt = 0, wi = -1;
                    double phw[5] = {0, 0, 0, 0, 0};
                    long long mx = 0, slow = 0, rds = 0;
                    for (int i = lo[r]; i < lo[r + 1]; ++i) {
                        if (hv[12 * i + 1] == 0) continue;
                        const double v = (double)hv[12 * i] / (double)hv[12 * i + 1] / 1e3;
                        if (v > worst) { worst = v; wi = i - lo[r]; for (int q = 0; q < 5; ++q) phw[q] = (double)hv[12 * i + 2 + q] / (double)hv[12 * i + 1] / 1e3; }
                        mean += v; ++cnt;
                        mx = std::max(mx, hv[12 * i + 8]); slow += hv[12 * i + 9]; rds += hv[12 * i + 1];
                    }
                    fprintf(stderr, "hals2 %s: slowest single round %.1f kcycles, %.2f%% of the (CTA, round) pairs above 90 kcycles\n", names[r], mx / 1e3, rds ? 100.0 * slow / rds : 0.0);
                    fprintf(stderr, "hals2 %s: %d CTAs, kcycles of work per active round: mean %.1f, worst %.1f (item %d; phases stage %.1f pull %.1f tail/store %.1f final %.1f, barrier wait %.1f); rounds %lld, chunks %lld\n",
                            names[r], lo[r + 1] - lo[r], cnt ? mean / cnt : 0.0, worst, wi, phw[0], phw[1], phw[2], phw[3], phw[4], (long long)(nC + 4 * (K - 1) + 3), (long long)nC);
                }
            }
            return true;
        }
    }

    // wavefront sweep (hals.jl:121-154) over the local shard (single-shard handles) or over the gathered full-T buffers
    void hals_h_sweep(int full, double l1H, double l2H) {
        REQUIRE(full || (is_first && is_last), "the local HALS H sweep needs a single-shard handle");
        if (progress.n == 0) hals_setup();
        CK(cudaMemsetAsync(progress.p, 0, progress.n * sizeof(int), stream));
        const size_t smem = hals_wave_smem_elems<S>(L) * sizeof(S);
        const S *cf = Cf.p, *s2 = GS.p, *q = full ? Qfull.p : numH.p;
        S *hh = full ? Hfull.p : H, *dd = full ? Dfull.p : denH.p, *tc_ = tailC.p;
        int *pr = progress.p;
        int64_t Kk = K, Ll = L, Tt = full ? T : Tl, ks = s2_ks, ldv = s2_ld;
        S a1 = (S)l1H, a2 = (S)l2H;
        int dbg = getenv("CMF_HALS_DEBUG") ? atoi(getenv("CMF_HALS_DEBUG")) : 0;   // 1: phase clocks of the last component; 2 / 4: timing runs without the pull / recurrence
        // truncated lag tables of all component pairs for the pull over the last L-1 columns (skipped when they would not fit: the
        // kernel then forms them on the fly)
        const S *ct = nullptr;
        {
            const size_t need = (size_t)(L - 1) * (size_t)(2 * L - 1) * (size_t)(K * K);
            if (L > 1 && need * sizeof(S) <= ((size_t)1 << 30) && !getenv("CMF_HALS_TAIL_DIRECT")) {
                if (tailCt.n < need) tailCt.alloc(need);
                hals_tail_table_kernel<S><<<(unsigned)cdiv((2 * L - 1) * K * K, 256), 256, 0, stream>>>(GS.p, tailCt.p, K, L, s2_ks, s2_ld);
                post_launch();
                ct = tailCt.p;
            }
        }
        if (hals2_sweep(q, hh, Tt, ct, l1H, l2H)) return;     // round-based kernel (fp32, L <= 32, K <= 128)
        void *args[] = {&cf, &s2, &q, &hh, &dd, &tc_, &pr, &Kk, &Ll, &Tt, &ks, &ldv, &a1, &a2, &dbg, &ct};
        prof_begin(PROF_SWEEP);
        CK(cudaLaunchCooperativeKernel((void *)hals_h_wave_kernel<S>, dim3((unsigned)hals_grid), dim3(HW_NT), args, smem, stream));
        prof_end();
        post_launch();
    }

    // ---------------------------------------------------------------- PGD (src/algs/pgd.jl, SquareLoss)
    // The gradients are the MU quantities again: dW = 2 (denomW - numW), dH = 2 (denomH - numH) (pgd.jl:206-221).
    int pgd_constrW = 0, pgd_constrH = 0;     // 0 NonnegConstraint (pgd.jl:91-95), 1 UnitNormConstraint (:98-110)
    DevBuf<double> un_part;
    // `inner` = elements between consecutive components in memory (N for Wi rows (l, k), 1 for H[t][K])
    void pgd_step(S *x, S *g, int64_t n, double &step, int constr, int64_t inner) {
        dot_partial_kernel<S><<<1024, 256, 0, stream>>>(g, g, n, loss_part.p);
        post_launch();
        reduce_scalar(loss_part.p, 1024, scal.p + 2);                                   // ||grad||^2 stays on the device
        pgd_step_kernel<S><<<(unsigned)cdiv(n, 256), 256, 0, stream>>>(x, g, step, scal.p + 2, n, constr == 0 ? 1 : 0);   // pgd.jl:236-241
        post_launch();
        if (constr == 1) {
            if (un_part.n == 0) un_part.alloc((size_t)K * UN_CHUNKS);
            unit_norm_partial_kernel<S><<<dim3(UN_CHUNKS, (unsigned)K), 256, 0, stream>>>(x, un_part.p, K, inner, n / K);
            post_launch();
            unit_norm_apply_kernel<S><<<(unsigned)cdiv(n, 256), 256, 0, stream>>>(x, un_part.p, K, inner, n);
            post_launch();
        }
    }
    void pgd_adapt(double loss, double &step) {
        step *= (loss < pgd_cur_loss) ? 1.05 : 0.70;                                    // pgd.jl:247-251
        pgd_cur_loss = loss;
    }

    // ---- PGD with the pluggable losses of pgd.jl:28-70 (AbsoluteLoss, MaskedLoss): the loss gradient d D / d est is not
    // linear in (X, est) any more (sign) or carries a mask, so the Gram forms do not apply and the path follows pgd.jl:224-255
    // literally: conv + loss-gradient epilogue into an N x T scratch, then the W-side correlation (pgd.jl:206-214) resp. the
    // transposed conv (:218-221) of that scratch, on the SIMT kernels in the handle's type.
    int pgd_loss = 0;                 // 0 SquareLoss, 1 AbsoluteLoss
    DevBuf<S> pgd_mask, pgd_ge;       // mask [t][N] (empty = none), loss-gradient scratch [t][N] incl. a zero right halo
    bool pgd_general() const { return pgd_loss != 0 || pgd_mask.n != 0; }
    void set_pgd_constraints(int cw, int ch) {
        REQUIRE(alg == CMF_PGD, "cmf_set_pgd_constraints: PGD handles only");
        REQUIRE((cw == 0 || cw == 1) && (ch == 0 || ch == 1), "constraint must be 0 (NonnegConstraint) or 1 (UnitNormConstraint)");
        pgd_constrW = cw; pgd_constrH = ch;
    }
    void set_pgd_loss(int lossf, const void *mask_host) {
        REQUIRE(alg == CMF_PGD, "the pluggable loss belongs to PGDUpdate handles");
        REQUIRE(lossf == 0 || lossf == 1, "loss_func must be 0 (SquareLoss) or 1 (AbsoluteLoss)");
        pgd_loss = lossf;
        if (mask_host) {
            pgd_mask.alloc((size_t)(N * Tl));
            CK(cudaMemcpyAsync(pgd_mask.p, mask_host, pgd_mask.n * sizeof(S), cudaMemcpyHostToDevice, stream));
            CK(cudaStreamSynchronize(stream));
        } else pgd_mask.free();
        if (pgd_general() && pgd_ge.n == 0) pgd_ge.alloc((size_t)((Tl + (L - 1)) * N));
    }
    void pgd_loss_gradient() {       // pgd.jl:231: grad!(loss_func, est, est, data)
        launch_conv(Wi.p, H, K, L, -(L - 1), Tl + (L - 1), 0, Tl, 32, pgd_ge.p, nullptr);
    }
    double pgd_loss_eval() {         // pgd.jl:244-245: tensor_conv!(est, W, H); eval(loss_func, data, est)
        const int nb = conv_nblocks(0, Tl);
        launch_conv(Wi.p, H, K, L, -(L - 1), Tl + (L - 1), 0, Tl, 64, nullptr, loss_part.p);
        reduce_scalar(loss_part.p, nb, scal.p);
        return fetch_scalar(scal.p);
    }

    void pgd_update_motifs(double l1W, double l2W) {
        REQUIRE(is_first && is_last, "PGD is single-shard");
        if (pgd_general()) {
            pgd_loss_gradient();
            launch_corr(pgd_ge.p, N, N, Tl + (L - 1), nsplit_w, split_w, denW.p, nullptr);          // gradW (pgd.jl:206-214)
            pgd_penalty_kernel<S><<<(unsigned)cdiv(KL() * N, 256), 256, 0, stream>>>(denW.p, Wi.p, (S)l1W, (S)l2W, KL() * N);
            post_launch();
            pgd_step(Wi.p, denW.p, KL() * N, pgd_stepW, pgd_constrW, N);
            w_changed();
            pgd_adapt(pgd_loss_eval(), pgd_stepW);
            return;
        }
        w_partials();
        compute_denomW(0, KL());
        pgd_grad_kernel<S><<<(unsigned)cdiv(KL() * N, 256), 256, 0, stream>>>(denW.p, denW.p, numW.p, Wi.p, (S)l1W, (S)l2W, KL() * N);
        post_launch();
        pgd_step(Wi.p, denW.p, KL() * N, pgd_stepW, pgd_constrW, N);
        w_changed();
        pgd_adapt(loss_partial(), pgd_stepW);                                           // pgd.jl:244-252
    }

    double pgd_update_feature_maps(double l1H, double l2H) {
        REQUIRE(is_first && is_last, "PGD is single-shard");
        if (pgd_general()) {
            pgd_loss_gradient();
            launch_transconv(Wi.p, pgd_ge.p, denH.p, N, K, L, N, Tl, Tl + (L - 1));                   // gradH (pgd.jl:218-221)
            pgd_penalty_kernel<S><<<(unsigned)cdiv(Tl * K, 256), 256, 0, stream>>>(denH.p, H, (S)l1H, (S)l2H, Tl * K);
            post_launch();
            pgd_step(H, denH.p, Tl * K, pgd_stepH, pgd_constrH, 1);
            h_changed();
            pgd_adapt(pgd_loss_eval(), pgd_stepH);
            return pgd_cur_loss;
        }
        compute_numH();
        compute_denomH();                                                               // is_last: PGD is single-shard
        pgd_grad_kernel<S><<<(unsigned)cdiv(Tl * K, 256), 256, 0, stream>>>(denH.p, denH.p, numH.p, H, (S)l1H, (S)l2H, Tl * K);
        post_launch();
        pgd_step(H, denH.p, Tl * K, pgd_stepH, pgd_constrH, 1);
        h_changed();
        numH_valid = true;                                                              // W unchanged: the expansion loss may reuse numH / W W'
        pgd_adapt(loss_partial(), pgd_stepH);
        return pgd_cur_loss;                                                            // caller: sqrt(cur_loss / datanorm^2), pgd.jl:202
    }

    // ---------------------------------------------------------------- exchange
    void exchange_buffer(int which, void **p, int64_t *count, int *dt) {
        if (which == 0) { *p = numW.p; *count = KL() * N; *dt = dtype; }
        else if (which == 1) { *p = exch1.p; *count = L * K * K + (L - 1) * K; *dt = CMF_F64; }
        else if (which == 2) { *p = numH.p; *count = Tl * K; *dt = dtype; }   // diagnostics: numH [t][K]
        else if (which == 3) { *p = denH.p; *count = Tl * K; *dt = dtype; }   // diagnostics: denomH [t][K]
        else throw CmfError(CMF_ERR_ARG, "exchange_buffer: which must be 0..3");
    }
    void halo_buffers(void **sl, void **sr, void **rl, void **rr, int64_t *count) {
        *sl = H; *sr = H + (Tl - (L - 1)) * K; *rl = Hbuf.p; *rr = H + Tl * K; *count = (L - 1) * K;
    }

    // ---------------------------------------------------------------- primitives
    void prim_conv(void *out_host) {
        DevBuf<S> out;
        out.alloc((size_t)(N * Tl));
        launch_conv(Wi.p, H, K, L, -(L - 1), Tl + (L - 1), 0, Tl, 1, out.p, nullptr);
        CK(cudaMemcpyAsync(out_host, out.p, out.n * sizeof(S), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    }
    void prim_transconv(const void *X_host, void *out_host) {
        set_data(X_host, 0);
        launch_transconv(Wi.p, X.p, numH.p, N, K, L, N, Tl, Tl + (L - 1));
        CK(cudaMemcpyAsync(out_host, numH.p, numH.n * sizeof(S), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    }
    void prim_corr(const void *X_host, void *out_host) {
        set_data(X_host, 0);
        launch_corr(X.p, N, N, Tl + (L - 1), nsplit_w, split_w, numW.p, nullptr);
        w_internal_to_julia<S><<<(unsigned)cdiv(KL() * N, 256), 256, 0, stream>>>(numW.p, Wtmp.p, K, N, L, K);
        post_launch();
        CK(cudaMemcpyAsync(out_host, Wtmp.p, Wtmp.n * sizeof(S), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    }
    // compute_resids (src/common.jl:58-59): conv(W,H) - X through the conv kernel's residual epilogue
    void prim_resids(void *out_host) {
        REQUIRE(have_data && have_factors, "compute_resids: data and factors must be set");
        DevBuf<S> out;
        out.alloc((size_t)(N * Tl));
        launch_conv(Wi.p, H, K, L, -(L - 1), Tl + (L - 1), 0, Tl, 2, out.p, nullptr);
        CK(cudaMemcpyAsync(out_host, out.p, out.n * sizeof(S), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    }
    // shift_and_stack (src/common.jl:133-142): Htilde[(l*K+k), t] = H[k, t-l], zero for t < l (materialised only here, for tests
    // and small problems: the fit itself addresses the same rows through overlapping windows of H)
    void prim_shift_and_stack(void *out_host) {
        REQUIRE(have_factors, "shift_and_stack: factors must be set");
        DevBuf<S> out;
        out.alloc((size_t)(KL() * Tl));
        shift_stack_kernel<S><<<(unsigned)cdiv(KL() * Tl, 256), 256, 0, stream>>>(H, out.p, K, L, Tl);
        post_launch();
        CK(cudaMemcpyAsync(out_host, out.p, out.n * sizeof(S), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    }
};

// One rank context, initialised on `device`.  S is chosen by the caller from dtype (with_dtype); the dtype check stays here
// so that the checks run, and fail, in the same order for every create call.  A batch handle passes the rank of every restart
// (`ranks`, non-empty) and K = their maximum.
template <typename S>
std::unique_ptr<Ctx<S>> make_ctx(int64_t N, int64_t T, int64_t t0, int64_t t1, int64_t K, int64_t L, int dtype, int alg,
                                 int device, const std::vector<int64_t> &ranks = {}) {
    REQUIRE(N >= 1 && K >= 1 && L >= 1 && T >= 1, "dimensions must be positive");
    REQUIRE(L <= T, "need L <= T (src/common.jl:28-31)");
    REQUIRE(0 <= t0 && t0 < t1 && t1 <= T, "bad shard range");
    REQUIRE(dtype == CMF_F64 || dtype == CMF_F32, "dtype must be 0 (f64) or 1 (f32)");
    REQUIRE(alg == CMF_MULT || alg == CMF_HALS || alg == CMF_PGD, "alg must be 0 (mult), 1 (hals) or 2 (pgd)");
    const bool sharded = !(t0 == 0 && t1 == T);
    if (sharded) {
        REQUIRE(t1 - t0 >= L - 1, "each shard needs at least L-1 columns");
        if (alg == CMF_PGD) throw CmfError(CMF_ERR_UNSUPPORTED, "PGD is single-shard only in this version");
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        throw CmfError(CMF_ERR_CUDA, std::string("no CUDA device available (") + cudaGetErrorString(e) + "); libcmf_sm100 has no CPU fallback");
    REQUIRE(device >= 0 && device < ndev, "bad device ordinal");
    std::unique_ptr<Ctx<S>> c(new Ctx<S>());
    c->N = N; c->T = T; c->t0 = t0; c->t1 = t1; c->Tl = t1 - t0; c->K = K; c->L = L;
    c->alg = alg; c->device = device;
    c->is_first = (t0 == 0); c->is_last = (t1 == T);
    c->R = (int64_t)ranks.size();
    c->b_K = ranks;
    c->b_C = std::accumulate(ranks.begin(), ranks.end(), (int64_t)0);
    c->init();
    return c;
}

// f(S()) with S = double for CMF_F64 and float otherwise (make_ctx rejects any other dtype)
template <typename F>
decltype(auto) with_dtype(int dtype, F &&f) {
    if (dtype == CMF_F64) return f(double());
    return f(float());
}

template <typename F>
int guarded(F &&f) {
    try {
        f();
        return CMF_OK;
    } catch (const CmfError &e) {
        g_err = e.what();
        return e.code;
    } catch (const std::exception &e) {
        g_err = e.what();
        return CMF_ERR_ARG;
    } catch (...) {
        g_err = "unknown error";
        return CMF_ERR_ARG;
    }
}

// Every ABI call runs on the handle's device and leaves the caller's current device as it found it.
struct DevGuard {
    int prev = -1;
    explicit DevGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        CK(cudaSetDevice(dev));
    }
    ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
    DevGuard(const DevGuard &) = delete;
    DevGuard &operator=(const DevGuard &) = delete;
};
// only restores the caller's current device on exit (constructors: the argument checks come before any CUDA call)
struct DevRestore {
    int prev = -1;
    DevRestore() { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); } }
    ~DevRestore() { if (prev >= 0) cudaSetDevice(prev); }
};

// src/model.jl:91-107
bool converged(const double *loss_hist, int64_t n, int patience, double tol) {
    if (n <= patience) return false;
    for (int64_t i = n - patience; i < n; ++i)
        if (!(std::fabs(loss_hist[i] - loss_hist[i - 1]) < tol)) return false;
    return true;
}

// ------------------------------------------------------------------------------------------
// multi-GPU: T-sharding with NCCL inside the library (SURVEY.md section 8e; the reference is single-process)
// ------------------------------------------------------------------------------------------
#define NK(call)                                                                                   \
    do {                                                                                           \
        ncclResult_t r__ = (call);                                                                 \
        if (r__ != ncclSuccess)                                                                    \
            throw CmfError(CMF_ERR_NCCL, std::string(#call) + ": " + NcclApi::get().GetErrorString(r__)); \
    } while (0)

NcclApi &nccl() {
    NcclApi &a = NcclApi::get();
    if (!a.ok()) throw CmfError(CMF_ERR_NCCL, "NCCL is not available: " + a.why);
    return a;
}

// balanced contiguous partition of the time axis (the same rule as cmf.jl_b200/sharded.py ShardPlan)
void shard_range(int64_t T, int world, int rank, int64_t *t0, int64_t *t1) {
    const int64_t base = T / world, rem = T % world;
    *t0 = rank * base + std::min<int64_t>(rank, rem);
    *t1 = *t0 + base + (rank < rem ? 1 : 0);
}

template <typename S>
ncclDataType_t nccl_dt(const Ctx<S> &) { return std::is_same<S, double>::value ? ncclFloat64 : ncclFloat32; }
template <typename S>
constexpr size_t elem_size(const Ctx<S> &) { return sizeof(S); }

template <typename S>
void c_allreduce(Ctx<S> &ctx, void *buf, size_t count, ncclDataType_t dt, ncclRedOp_t op = ncclSum) {
    if (ctx.world() == 1) return;
    NK(nccl().AllReduce(buf, buf, count, dt, op, ctx.comm.comm, ctx.stream));
}

// all-reduce of a few host doubles through the handle's scalar buffer (slots 4..7); synchronises the stream
template <typename S>
void c_allreduce_host(Ctx<S> &ctx, double *vals, int n, ncclRedOp_t op = ncclSum) {
    if (ctx.world() == 1) return;
    REQUIRE(n <= 4, "at most 4 scalars");
    double *d = ctx.scalars() + 4;
    CK(cudaMemcpyAsync(d, vals, n * sizeof(double), cudaMemcpyHostToDevice, ctx.stream));
    c_allreduce(ctx, d, (size_t)n, ncclFloat64, op);
    CK(cudaMemcpyAsync(vals, d, n * sizeof(double), cudaMemcpyDeviceToHost, ctx.stream));
    CK(cudaStreamSynchronize(ctx.stream));
}

// L-1 columns of H each way (left neighbour's right halo <- my first L-1 columns; right neighbour's left halo <- my last)
template <typename S>
void c_halo_exchange(Ctx<S> &ctx) {
    if (ctx.world() == 1 || ctx.L <= 1) return;
    void *sl, *sr, *rl, *rr;
    int64_t cnt;
    ctx.halo_buffers(&sl, &sr, &rl, &rr, &cnt);
    NcclApi &a = nccl();
    const ncclDataType_t dt = nccl_dt(ctx);
    const int r = ctx.rank(), w = ctx.world();
    NK(a.GroupStart());
    if (r + 1 < w) {
        NK(a.Send(sr, (size_t)cnt, dt, r + 1, ctx.comm.comm, ctx.stream));
        NK(a.Recv(rr, (size_t)cnt, dt, r + 1, ctx.comm.comm, ctx.stream));
    }
    if (r > 0) {
        NK(a.Send(sl, (size_t)cnt, dt, r - 1, ctx.comm.comm, ctx.stream));
        NK(a.Recv(rl, (size_t)cnt, dt, r - 1, ctx.comm.comm, ctx.stream));
    }
    NK(a.GroupEnd());
}

// ||X||_F over all shards (mult.jl:13, hals.jl:23)
template <typename S>
void r_data_norm(Ctx<S> &ctx) {
    double ss = ctx.data_sumsq_local;
    c_allreduce_host(ctx, &ss, 1);
    ctx.data_sumsq_global = ss;
    ctx.data_norm = std::sqrt(ss);
    ctx.pgd_cur_loss = ctx.data_norm;
}

// <X, est> and ||est||^2 of the alpha rescale (src/model.jl:119-120), summed over shards
template <typename S>
void r_init_scale_partials(Ctx<S> &ctx, double out[2]) {
    ctx.init_scale_partials(out);
    c_allreduce_host(ctx, out, 2);
}

// sum of squared residuals over ALL shards: one fixed-size all-reduce of the two loss scalars, one read-back
template <typename S>
double r_loss_sumsq(Ctx<S> &ctx, bool force_direct = false, bool *expansion_used = nullptr) {
    const int saved = ctx.loss_mode;
    if (force_direct) ctx.loss_mode = 0;
    int n;
    try { n = ctx.loss_partial_dev(); } catch (...) { ctx.loss_mode = saved; throw; }
    ctx.loss_mode = saved;
    double *d = ctx.scalars();
    c_allreduce(ctx, d, 2, ncclFloat64);
    double v[2];
    CK(cudaMemcpyAsync(v, d, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx.stream));
    CK(cudaStreamSynchronize(ctx.stream));
    if (expansion_used) *expansion_used = (n == 2);
    ++(n == 2 ? ctx.n_loss_expansion : ctx.n_loss_direct);
    return n == 2 ? ctx.data_sumsq_global - 2.0 * v[0] + v[1] : v[0];
}

// Loss of the current factors, mult.jl:55-57.  With loss_mode 1 the algebraic expansion serves while the relative loss is
// above `loss_guard` (25 %): its error is ~2e-6/loss^2 relative.  At or below the guard the expansion is CALIBRATED: its
// error is a bias that moves slowly with the factors, so the direct residual pass is run every `calib_interval`
// evaluations, the difference is kept and subtracted in between, and at each direct pass the value the previous bias would
// have predicted is checked against it -- agreement to 5e-6 (relative, on the loss) doubles the interval (up to 16), more
// than 2e-5 halves it, more than 1e-4 three times in a row returns the handle to the direct pass for good.  Values returned
// at calibration points are the direct pass itself.  Every rank sees the same all-reduced numbers and takes the same branch.
template <typename S>
double r_guarded_loss(Ctx<S> &ctx) {
    if (ctx.loss_mode != 1) return std::sqrt(std::max(r_loss_sumsq(ctx), 0.0)) / ctx.data_norm;
    bool exp_used = false;
    const double se = r_loss_sumsq(ctx, false, &exp_used);
    if (!exp_used) return std::sqrt(std::max(se, 0.0)) / ctx.data_norm;
    const double g2 = ctx.loss_guard * ctx.loss_guard * ctx.data_sumsq_global;
    if (!ctx.calib_have && se > g2) return std::sqrt(se) / ctx.data_norm;
    if (ctx.calib_have && ctx.calib_left > 0 && se - ctx.calib_bias > 0.0) {
        --ctx.calib_left;
        return std::sqrt(se - ctx.calib_bias) / ctx.data_norm;
    }
    const double sd = r_loss_sumsq(ctx, true);
    if (ctx.calib_have && sd > 0.0) {
        const double err = std::fabs((se - ctx.calib_bias) - sd) / (2.0 * sd);
        ctx.calib_last_err = err;
        if (err > 1e-4) { ctx.calib_interval = 1; ++ctx.calib_fail; }
        else {
            ctx.calib_fail = 0;
            if (err > 2e-5) ctx.calib_interval = std::max(1, ctx.calib_interval / 2);
            else if (err < 5e-6) ctx.calib_interval = std::min(ctx.calib_max_interval, ctx.calib_interval * 2);
        }
        if (ctx.calib_fail >= 3) { ctx.loss_mode = 0; ctx.calib_reset(); }      // the expansion is not reliable on this problem
    }
    ctx.calib_bias = se - sd;
    ctx.calib_have = true;
    ctx.calib_left = ctx.calib_interval - 1;
    return std::sqrt(std::max(sd, 0.0)) / ctx.data_norm;
}

// update_motifs! (mult.jl:23-39 / hals.jl:31-34 / pgd.jl:158-178) on this rank's shard
template <typename S>
void r_update_motifs(Ctx<S> &ctx, double l1W, double l2W) {
    if (ctx.alg == CMF_PGD) { ctx.pgd_update_motifs(l1W, l2W); return; }
    ctx.w_partials();
    const int64_t KL = ctx.K * ctx.L;
    if (ctx.world() > 1 && ctx.alg == CMF_MULT && KL % ctx.world() == 0 && !getenv("CMF_W_REPLICATED")) {
        // MultUpdate: the W update is sharded by unfolded rows j = l*K + k (contiguous row blocks of numW / W):
        // reduce-scatter of numW on the side stream while this rank forms its rows of denomW = G W, update of those
        // rows, all-gather of W.  Same bytes on the wire as an all-reduce; G W, the ratio update and the eps floor cost 1/world.
        NcclApi &a = nccl();
        void *p; int64_t cnt; int dt;
        ctx.exchange_buffer(1, &p, &cnt, &dt);
        c_allreduce(ctx, p, (size_t)cnt, ncclFloat64);                                   // Gram + H tail (small, needed by G)
        void *nw, *w; int64_t row;
        ctx.w_rows_buffers(&nw, &w, &row);
        const int64_t rows = KL / ctx.world(), j0 = rows * ctx.rank(), chunk = rows * row;
        const size_t es = elem_size(ctx);
        CK(cudaEventRecord(ctx.ev_a, ctx.stream));
        CK(cudaStreamWaitEvent(ctx.comm_stream, ctx.ev_a, 0));
        NK(a.ReduceScatter(nw, (char *)nw + (size_t)(j0 * row) * es, (size_t)chunk, nccl_dt(ctx), ncclSum, ctx.comm.comm, ctx.comm_stream));
        CK(cudaEventRecord(ctx.ev_b, ctx.comm_stream));
        ctx.w_denom_rows(j0, j0 + rows);
        CK(cudaStreamWaitEvent(ctx.stream, ctx.ev_b, 0));
        ctx.w_update_rows(l1W, l2W, j0, j0 + rows);
        // all-gather of W on the side stream; the one piece of the H half-step that does not need W (the spectrum of H for
        // denomH) runs meanwhile
        CK(cudaEventRecord(ctx.ev_a, ctx.stream));
        CK(cudaStreamWaitEvent(ctx.comm_stream, ctx.ev_a, 0));
        NK(a.AllGather((char *)w + (size_t)(j0 * row) * es, w, (size_t)chunk, nccl_dt(ctx), ctx.comm.comm, ctx.comm_stream));
        CK(cudaEventRecord(ctx.ev_b, ctx.comm_stream));
        if (ctx.alg == CMF_MULT) ctx.fd_denomH_prefetch();
        CK(cudaStreamWaitEvent(ctx.stream, ctx.ev_b, 0));
        return;
    }
    if (ctx.world() > 1) {
        void *p; int64_t cnt; int dt;
        ctx.exchange_buffer(0, &p, &cnt, &dt);
        c_allreduce(ctx, p, (size_t)cnt, dt == CMF_F64 ? ncclFloat64 : ncclFloat32);     // numW            (K*N*L)
        ctx.exchange_buffer(1, &p, &cnt, &dt);
        c_allreduce(ctx, p, (size_t)cnt, ncclFloat64);                                   // Gram + H tail   (K*K*L + (L-1)*K doubles)
    }
    ctx.w_apply(l1W, l2W);                                                              // identical update on every rank
}

// HALS H sweep of a T-sharded fit: gather Q and H on rank 0, sweep once in the reference's order, scatter H
template <typename S>
void r_hals_sweep_sharded(Ctx<S> &ctx, double l1H, double l2H) {
    NcclApi &a = nccl();
    const ncclDataType_t dt = nccl_dt(ctx);
    const size_t es = elem_size(ctx);
    const int w = ctx.world(), r = ctx.rank();
    void *ql, *hl, *qf = nullptr, *hf = nullptr;
    int64_t cnt;
    ctx.hals_h_local(&ql, &hl, &cnt);
    if (r == 0) ctx.hals_h_full(&qf, &hf);
    for (int pass = 0; pass < 2; ++pass) {          // 0: gather Q and H, 1: scatter H
        if (pass == 1 && r == 0) ctx.hals_h_sweep(1, l1H, l2H);
        NK(a.GroupStart());
        if (r == 0) {
            for (int p = 1; p < w; ++p) {
                int64_t a0, a1;
                shard_range(ctx.T, w, p, &a0, &a1);
                const size_t off = (size_t)(a0 * ctx.K) * es, c = (size_t)((a1 - a0) * ctx.K);
                if (pass == 0) {
                    NK(a.Recv((char *)qf + off, c, dt, p, ctx.comm.comm, ctx.stream));
                    NK(a.Recv((char *)hf + off, c, dt, p, ctx.comm.comm, ctx.stream));
                } else {
                    NK(a.Send((char *)hf + off, c, dt, p, ctx.comm.comm, ctx.stream));
                }
            }
        } else if (pass == 0) {
            NK(a.Send(ql, (size_t)cnt, dt, 0, ctx.comm.comm, ctx.stream));
            NK(a.Send(hl, (size_t)cnt, dt, 0, ctx.comm.comm, ctx.stream));
        } else {
            NK(a.Recv(hl, (size_t)cnt, dt, 0, ctx.comm.comm, ctx.stream));
        }
        NK(a.GroupEnd());
        if (r == 0) {
            if (pass == 0) {
                CK(cudaMemcpyAsync(qf, ql, (size_t)cnt * es, cudaMemcpyDeviceToDevice, ctx.stream));
                CK(cudaMemcpyAsync(hf, hl, (size_t)cnt * es, cudaMemcpyDeviceToDevice, ctx.stream));
            } else {
                CK(cudaMemcpyAsync(hl, hf, (size_t)cnt * es, cudaMemcpyDeviceToDevice, ctx.stream));
            }
        }
    }
}

// loss = update_feature_maps! (mult.jl:42-58 / hals.jl:37-42 / pgd.jl:181-203)
template <typename S>
double r_update_feature_maps(Ctx<S> &ctx, double l1H, double l2H) {
    if (ctx.alg == CMF_PGD) {
        const double loss = std::sqrt(ctx.pgd_update_feature_maps(l1H, l2H)) / ctx.data_norm;
        if (ctx.loss_mode == 1 && !(loss > 0.25)) ctx.loss_mode = 0;   // PGD adapts its step on this value: no re-evaluation
        return loss;
    }
    if (ctx.alg == CMF_HALS) {
        ctx.hals_h_prepare();
        if (ctx.world() == 1) ctx.hals_h_sweep(0, l1H, l2H);
        else r_hals_sweep_sharded(ctx, l1H, l2H);
        ctx.h_changed();
    } else {
        ctx.h_update(l1H, l2H);
    }
    c_halo_exchange(ctx);
    return r_guarded_loss(ctx);
}

// src/algs/alternating.jl:16-71 on one rank (every rank runs the same loop: the loss is all-reduced, and the elapsed
// time that decides `max_time` is rank 0's, so all ranks take the same branches)
template <typename S>
void r_fit(Ctx<S> &ctx, int64_t max_itr, double max_time, int eval_mode, int check_convergence, int patience, double tol,
           double l1W, double l2W, double l1H, double l2H, std::vector<double> &loss_hist, std::vector<double> &time_hist,
           int64_t cap, int *converged_early) {
    *converged_early = 0;
    loss_hist.clear(); time_hist.clear();
    loss_hist.push_back(r_guarded_loss(ctx));   // alternating.jl:37
    time_hist.push_back(0.0);
    int64_t itr = 1;
    const bool timed = max_time < 1e300;
    while ((max_itr < 0 || itr <= max_itr) && time_hist.back() <= max_time) {   // alternating.jl:45
        ++itr;
        REQUIRE((int64_t)loss_hist.size() < cap, "history capacity exhausted");
        auto t_start = std::chrono::steady_clock::now();
        if (!eval_mode) r_update_motifs(ctx, l1W, l2W);
        const double loss = r_update_feature_maps(ctx, l1H, l2H);
        double dur = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
        if (timed && ctx.world() > 1) {          // rank 0's clock decides for everyone
            if (ctx.rank() != 0) dur = 0.0;
            c_allreduce_host(ctx, &dur, 1);
        }
        time_hist.push_back(time_hist.back() + dur);
        loss_hist.push_back(loss);
        if (check_convergence && converged(loss_hist.data(), (int64_t)loss_hist.size(), patience, tol)) {   // alternating.jl:63-66
            *converged_early = 1;
            break;
        }
    }
}

template <typename S>
void r_set_engine(Ctx<S> &ctx, int engine) {
    REQUIRE(engine >= 0 && engine <= 2, "engine must be 0 (SIMT), 1 (tcgen05, time domain) or 2 (tcgen05, frequency domain)");
    if (ctx.R > 0 && engine != 0) throw CmfError(CMF_ERR_UNSUPPORTED, "batch handles run the SIMT engine (0) only");
    if (engine == 2 && !ctx.fd_available())
        throw CmfError(CMF_ERR_UNSUPPORTED, "the frequency-domain engine needs an fp32 handle with K <= 128, L <= 256, N % 8 == 0 on sm_100 and room for the spectrum of X");
    if (engine < 2) ctx.fd_release();               // the spectrum of X and the time-domain planes never coexist
    if (engine >= 1 && !ctx.tc_available())
        throw CmfError(CMF_ERR_UNSUPPORTED, "tcgen05 engine needs an fp32 MultUpdate handle with K <= 128 and N % 8 == 0 on sm_100");
    ctx.engine = engine;
    if (!ctx.loss_mode_explicit) ctx.loss_mode = (engine == 2) ? 1 : 0;   // the expansion is the default of engine 2 only
}

// every rank must run the same engine (the collectives are matched by program order): take the minimum of what the
// ranks selected by themselves (shard lengths and free memory may differ by a little)
template <typename S>
void r_agree_engine(Ctx<S> &ctx) {
    if (ctx.world() == 1) return;
    double e = (double)ctx.engine;
    c_allreduce_host(ctx, &e, 1, ncclMin);
    if ((int)e != ctx.engine) r_set_engine(ctx, (int)e);
}

template <typename S>
void attach_comm(Ctx<S> &ctx, ncclComm_t comm, int rank, int world) {
    int64_t a0, a1;
    shard_range(ctx.T, world, rank, &a0, &a1);
    REQUIRE(a0 == ctx.t0 && a1 == ctx.t1, "the handle's column range is not the balanced shard of this rank (use cmf_shard_range)");
    ctx.comm.comm = comm; ctx.comm.rank = rank; ctx.comm.world = world;
    if (world > 1 && !ctx.comm_stream) {
        CK(cudaStreamCreateWithFlags(&ctx.comm_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx.ev_a, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx.ev_b, cudaEventDisableTiming));
    }
    r_agree_engine(ctx);
}

// src/algs/alternating.jl:16-71 for R restarts at once.  Restart r keeps its own history and early stop; once it has
// converged its factors are frozen (active flag 0) while the others go on.  The loop ends when every restart has stopped or
// max_itr / max_time is reached; the elapsed time is the batch's own, shared by all restarts.
template <typename S>
void b_fit(Ctx<S> &ctx, int64_t max_itr, double max_time, int eval_mode, int check_convergence, int patience, double tol,
           const double *l1W, const double *l2W, const double *l1H, const double *l2H, double *loss_hist,
           std::vector<double> &time_hist, int64_t cap, int64_t *n_hist, int *converged_early) {
    const int64_t R = ctx.R;
    std::vector<double> reg((size_t)(4 * R));
    for (int64_t r = 0; r < R; ++r) { reg[4 * r] = l1W[r]; reg[4 * r + 1] = l2W[r]; reg[4 * r + 2] = l1H[r]; reg[4 * r + 3] = l2H[r]; }
    std::vector<int> active((size_t)R, 1);
    ctx.batch_set_state(reg.data(), active.data());
    std::vector<double> loss((size_t)R);
    ctx.batch_loss(loss.data());                                     // alternating.jl:37
    for (int64_t r = 0; r < R; ++r) { loss_hist[r * cap] = loss[r]; n_hist[r] = 1; converged_early[r] = 0; }
    time_hist.assign(1, 0.0);
    int64_t itr = 1, n_active = R;
    while (n_active > 0 && (max_itr < 0 || itr <= max_itr) && time_hist.back() <= max_time) {   // alternating.jl:45
        ++itr;
        REQUIRE((int64_t)time_hist.size() < cap, "history capacity exhausted");
        auto t_start = std::chrono::steady_clock::now();
        if (!eval_mode) ctx.batch_update_motifs();
        ctx.batch_update_feature_maps();
        ctx.batch_loss(loss.data());
        time_hist.push_back(time_hist.back() + std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count());
        bool stopped = false;
        for (int64_t r = 0; r < R; ++r) {
            if (!active[r]) continue;
            double *lh = loss_hist + r * cap;
            lh[n_hist[r]++] = loss[r];
            if (check_convergence && converged(lh, n_hist[r], patience, tol)) {   // alternating.jl:63-66
                converged_early[r] = 1;
                active[r] = 0;
                --n_active;
                stopped = true;
            }
        }
        if (stopped && n_active > 0) ctx.batch_set_state(nullptr, active.data());
    }
}

template <typename S>
using Ranks = std::vector<std::unique_ptr<Ctx<S>>>;

}  // namespace

// A handle is the list of its rank contexts, all of one dtype.  cmf_create, cmf_create_shard, cmf_create_rank and
// cmf_create_batch make one rank context; cmf_create_multi with ngpu > 1 makes one per device, each driven by its own worker
// thread, over NCCL communicators the handle owns.
struct cmf_ctx {
    std::variant<Ranks<float>, Ranks<double>> ranks;
    std::vector<ncclComm_t> comms;             // several rank contexts: one communicator per rank context
    std::unique_ptr<cmf::Workers> workers;     // several rank contexts: worker i drives rank context i
    size_t size() const { return std::visit([](auto &v) { return v.size(); }, ranks); }
    ~cmf_ctx() {
        if (!workers) return;   // one rank context: cmf_destroy frees it on its device
        // every rank context and its communicator are freed by the worker that drives them (a failed create leaves gaps)
        try {
            std::visit([&](auto &v) {
                workers->run_all([&](int i) {
                    auto &r = v[(size_t)i];
                    if (!r) return;
                    cudaSetDevice(r->device);
                    r.reset();
                    if (comms[(size_t)i]) NcclApi::get().CommDestroy(comms[(size_t)i]);
                });
            }, ranks);
        } catch (...) {}
    }
};

namespace {

template <typename S>
cmf_ctx *handle_of(std::unique_ptr<Ctx<S>> r) {
    Ranks<S> v;
    v.push_back(std::move(r));
    return new cmf_ctx{std::move(v)};
}

// A handle with several rank contexts follows two rules: its first rank context speaks for it (it alone writes the loss,
// the histories, W, the scale partials and the early-stop flag), and a host H or X array starts at that context's first
// column, so rank context r reads and writes it at column r.t0 - first(h).t0 (0 on every handle of one rank context).
RankState &first(cmf_handle h) { return std::visit([](auto &v) -> RankState & { return *v.front(); }, h->ranks); }
RankState &last(cmf_handle h) { return std::visit([](auto &v) -> RankState & { return *v.back(); }, h->ranks); }

// f(Ctx<S> &) on every rank context of the handle: inline on the calling thread for one, concurrently on the workers for
// several (the ranks meet in NCCL collectives); each under its device
template <typename F>
void on_ranks(cmf_handle h, F &&f) {
    REQUIRE(h != nullptr, "null handle");
    std::visit([&](auto &v) {
        if (v.size() == 1) {
            DevGuard g(v[0]->device);
            f(*v[0]);
            return;
        }
        h->workers->run_all([&](int i) {
            auto &r = *v[(size_t)i];
            DevGuard g(r.device);
            f(r);
        });
    }, h->ranks);
}
// f(Ctx<S> &) on the first rank context, on the calling thread and its current device
template <typename F>
void on_first(cmf_handle h, F &&f) {
    std::visit([&](auto &v) { f(*v.front()); }, h->ranks);
}

// The split-phase, stream and PGD-setup calls drive one rank context.
void single_rank(cmf_handle h) { REQUIRE(h && h->size() == 1, "single-rank call"); }
// Every call that takes or returns ONE factor set refuses a batch handle and names the call to use instead.
void single_set(cmf_handle h, const char *use) {
    if (h && first(h).R > 0) throw CmfError(CMF_ERR_ARG, std::string("this is a batch handle (cmf_create_batch): use ") + use);
}
void no_batch_split(cmf_handle h) {
    if (h && first(h).R > 0) throw CmfError(CMF_ERR_UNSUPPORTED, "batch handles have no split-phase calls: use cmf_fit_batch");
}
void batch_handle(cmf_handle h) { REQUIRE(h && first(h).R > 0, "not a batch handle (cmf_create_batch)"); }

// a handle of one rank context (make_ctx's checks)
cmf_ctx *make_handle(int64_t N, int64_t T, int64_t t0, int64_t t1, int64_t K, int64_t L, int dtype, int alg, int device,
                     const std::vector<int64_t> &ranks = {}) {
    return with_dtype(dtype, [&](auto s) { return handle_of(make_ctx<decltype(s)>(N, T, t0, t1, K, L, dtype, alg, device, ranks)); });
}

// cmf_create_batch and cmf_create_batch_ranks (after their checks of R): restart r has rank ranks[r].  Every check runs
// before any device query.
cmf_ctx *make_batch(int64_t N, int64_t T, const std::vector<int64_t> &ranks, int64_t L, int dtype, int alg, int device) {
    REQUIRE(alg == CMF_MULT || alg == CMF_HALS || alg == CMF_PGD, "alg must be 0 (mult), 1 (hals) or 2 (pgd)");
    if (alg != CMF_MULT)
        throw CmfError(CMF_ERR_UNSUPPORTED, "batched restarts serve MultUpdate only (HALS sweeps run sequentially per restart; PGD is not batched)");
    REQUIRE(N >= 1 && L >= 1 && T >= 1, "dimensions must be positive");
    for (size_t r = 0; r < ranks.size(); ++r) {
        REQUIRE(ranks[r] >= 1, "dimensions must be positive: K[" + std::to_string(r) + "] = " + std::to_string(ranks[r]));
        REQUIRE(ranks[r] <= 4 * 65535, "R*K too large for one launch grid: K[" + std::to_string(r) + "] = " + std::to_string(ranks[r]));
    }
    const int64_t C = std::accumulate(ranks.begin(), ranks.end(), (int64_t)0), Kmax = *std::max_element(ranks.begin(), ranks.end());
    REQUIRE(C * cdiv(L, 8) <= (int64_t)CORR_PB * 65535 && C <= 4 * 65535, "R*K too large for one launch grid (the ranks of all restarts add up to " + std::to_string(C) + ")");
    if (L > 769) throw CmfError(CMF_ERR_UNSUPPORTED, "batched restarts need L <= 769");
    return make_handle(N, T, 0, T, Kmax, L, dtype, alg, device, ranks);
}

}  // namespace

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

const char *cmf_last_error(void) { return g_err.c_str(); }

int cmf_create(cmf_handle *out, int64_t N, int64_t T, int64_t K, int64_t L, int dtype, int alg, int device) {
    return guarded([&] {
        REQUIRE(out != nullptr, "null output pointer");
        DevRestore g;
        *out = make_handle(N, T, 0, T, K, L, dtype, alg, device);
    });
}

int cmf_create_shard(cmf_handle *out, int64_t N, int64_t T_global, int64_t t_begin, int64_t t_end, int64_t K,
                     int64_t L, int dtype, int alg, int device) {
    return guarded([&] {
        REQUIRE(out != nullptr, "null output pointer");
        DevRestore g;
        *out = make_handle(N, T_global, t_begin, t_end, K, L, dtype, alg, device);
    });
}

int cmf_shard_range(int64_t T, int world, int rank, int64_t *t_begin, int64_t *t_end) {
    return guarded([&] {
        REQUIRE(t_begin && t_end, "null output");
        REQUIRE(world >= 1 && rank >= 0 && rank < world && T >= world, "need 0 <= rank < world <= T");
        shard_range(T, world, rank, t_begin, t_end);
    });
}

int cmf_comm_unique_id(void *id_out) {
    return guarded([&] {
        REQUIRE(id_out, "null output");
        ncclUniqueId id;
        NK(nccl().GetUniqueId(&id));
        memcpy(id_out, &id, sizeof(id));
    });
}

// One communicator per (device, rank, world) of this process is kept alive and reused by later handles created with
// unique_id == NULL (building one costs ~0.5 s; a fit does not need a new one).  Communicators in the cache live until exit.
struct CommKey { int device, rank, world; bool operator<(const CommKey &o) const { return std::tie(device, rank, world) < std::tie(o.device, o.rank, o.world); } };
static std::map<CommKey, ncclComm_t> g_comm_cache;
static std::mutex g_comm_mu;

int cmf_create_rank(cmf_handle *out, int64_t N, int64_t T, int64_t K, int64_t L, int dtype, int alg, int device,
                    const void *unique_id, int rank, int world) {
    return guarded([&] {
        REQUIRE(out != nullptr, "null pointer");
        REQUIRE(world >= 1 && rank >= 0 && rank < world, "need 0 <= rank < world");
        DevRestore g;
        int64_t a0, a1;
        shard_range(T, world, rank, &a0, &a1);
        *out = with_dtype(dtype, [&](auto s) {
            auto c = make_ctx<decltype(s)>(N, T, a0, a1, K, L, dtype, alg, device);
            ncclComm_t comm = nullptr;
            if (world > 1) {
                std::lock_guard<std::mutex> lk(g_comm_mu);
                const CommKey key{device, rank, world};
                if (unique_id == nullptr) {
                    auto it = g_comm_cache.find(key);
                    REQUIRE(it != g_comm_cache.end(), "unique_id == NULL reuses this process's communicator for (device, rank, world), but none exists yet");
                    comm = it->second;
                } else {
                    ncclUniqueId id;
                    memcpy(&id, unique_id, sizeof(id));
                    CK(cudaSetDevice(device));
                    NK(nccl().CommInitRank(&comm, world, id, rank));
                    g_comm_cache[key] = comm;            // replaces (and leaks until exit) an older one: it may still serve a live handle
                }
            }
            attach_comm(*c, comm, rank, world);
            return handle_of(std::move(c));
        });
    });
}

int cmf_create_multi(cmf_handle *out, int64_t N, int64_t T, int64_t K, int64_t L, int dtype, int alg, int ngpu,
                     const int *devices) {
    return guarded([&] {
        REQUIRE(out != nullptr, "null output pointer");
        REQUIRE(ngpu >= 1 && ngpu <= 64, "ngpu must be in 1..64");
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0)
            throw CmfError(CMF_ERR_CUDA, std::string("no CUDA device available (") + cudaGetErrorString(e) + "); libcmf_sm100 has no CPU fallback");
        std::vector<int> devs((size_t)ngpu);
        for (int i = 0; i < ngpu; ++i) {
            devs[(size_t)i] = devices ? devices[i] : i;
            REQUIRE(devs[(size_t)i] >= 0 && devs[(size_t)i] < ndev, "bad device ordinal in the device list");
        }
        if (ngpu == 1) {
            DevRestore g;
            *out = make_handle(N, T, 0, T, K, L, dtype, alg, devs[0]);
            return;
        }
        int prev = 0;
        cudaGetDevice(&prev);
        with_dtype(dtype, [&](auto s) {
            using S = decltype(s);
            auto *mc = new cmf_ctx{Ranks<S>((size_t)ngpu)};
            Ranks<S> &ranks = std::get<Ranks<S>>(mc->ranks);
            try {
                mc->comms.assign((size_t)ngpu, nullptr);
                mc->workers.reset(new Workers(ngpu));
                NK(nccl().CommInitAll(mc->comms.data(), ngpu, devs.data()));
                cudaSetDevice(prev);
                mc->workers->run_all([&](int i) {
                    DevGuard g(devs[(size_t)i]);
                    int64_t a0, a1;
                    shard_range(T, ngpu, i, &a0, &a1);
                    ranks[(size_t)i] = make_ctx<S>(N, T, a0, a1, K, L, dtype, alg, devs[(size_t)i]);
                });
                mc->workers->run_all([&](int i) {
                    Ctx<S> &r = *ranks[(size_t)i];
                    DevGuard g(r.device);
                    attach_comm(r, mc->comms[(size_t)i], i, ngpu);
                });
            } catch (...) {
                cudaSetDevice(prev);
                delete mc;
                throw;
            }
            *out = mc;
        });
    });
}

int cmf_comm_info(cmf_handle h, int *rank_out, int *world_out, int64_t *t_begin, int64_t *t_end) {
    return guarded([&] {
        REQUIRE(h, "null handle");
        if (rank_out) *rank_out = first(h).rank();
        if (world_out) *world_out = first(h).world();
        if (t_begin) *t_begin = first(h).t0;
        if (t_end) *t_end = last(h).t1;
    });
}

int cmf_destroy(cmf_handle h) {
    return guarded([&] {
        if (!h) return;
        if (h->workers) { delete h; return; }   // ~cmf_ctx frees every rank context on its worker
        DevGuard g(first(h).device);
        delete h;
    });
}

int cmf_set_data(cmf_handle h, const void *X, int64_t first_col) {
    return guarded([&] { on_ranks(h, [&](auto &r) { r.set_data(X, first_col); r_data_norm(r); }); });
}
int cmf_synth_data(cmf_handle h, uint64_t seed, int64_t K_true, int64_t L_true, double p_h, double noise) {
    return guarded([&] { on_ranks(h, [&](auto &r) { r.synth_data(seed, K_true, L_true, p_h, noise); r_data_norm(r); }); });
}
int cmf_data_sumsq(cmf_handle h, double *out) {
    return guarded([&] {
        REQUIRE(out, "null output");
        const RankState &r = first(h);
        REQUIRE(r.have_data, "no data");
        *out = r.world() > 1 ? r.data_sumsq_global : r.data_sumsq_local;
    });
}
int cmf_set_data_norm(cmf_handle h, double norm) {
    return guarded([&] { on_ranks(h, [&](auto &r) { r.data_norm = norm; r.data_sumsq_global = norm * norm; }); });
}
int cmf_set_factors(cmf_handle h, const void *W, const void *H, int64_t first_col) {
    return guarded([&] { single_set(h, "cmf_set_factors_batch"); on_ranks(h, [&](auto &r) { r.set_factors(W, H, first_col); }); });
}
int cmf_exchange_halos(cmf_handle h) {
    return guarded([&] { no_batch_split(h); on_ranks(h, [&](auto &r) { c_halo_exchange(r); r.h_changed(); }); });
}
int cmf_init_rand(cmf_handle h, uint64_t seed) {
    return guarded([&] { single_set(h, "cmf_set_factors_batch with drawn factors"); on_ranks(h, [&](auto &r) { r.init_rand(seed); }); });
}
int cmf_init_scale_partials(cmf_handle h, double out[2]) {
    return guarded([&] { single_set(h, "cmf_init_scale_partials_batch");
        REQUIRE(out, "null output");
        on_ranks(h, [&](auto &r) {
            double v[2];
            r_init_scale_partials(r, v);
            if (&r == &first(h)) { out[0] = v[0]; out[1] = v[1]; }
        });
    });
}
int cmf_scale_factors(cmf_handle h, double s) {
    return guarded([&] { single_set(h, "cmf_scale_factors_batch"); on_ranks(h, [&](auto &r) { r.scale_factors(s); }); });
}
int cmf_get_factors(cmf_handle h, void *W_out, void *H_out) {
    return guarded([&] { single_set(h, "cmf_get_factors_batch");
        on_ranks(h, [&](auto &r) {
            REQUIRE(r.have_factors, "no factors");
            void *Hp = H_out ? (char *)H_out + (size_t)((r.t0 - first(h).t0) * r.K) * elem_size(r) : nullptr;
            r.get_factors(&r == &first(h) ? W_out : nullptr, Hp);
        });
    });
}

int cmf_update_motifs(cmf_handle h, double l1W, double l2W) {
    return guarded([&] { single_set(h, "cmf_fit_batch"); on_ranks(h, [&](auto &r) { r_update_motifs(r, l1W, l2W); }); });
}

int cmf_update_feature_maps(cmf_handle h, double l1H, double l2H, double *loss_out) {
    return guarded([&] { single_set(h, "cmf_fit_batch");
        on_ranks(h, [&](auto &r) {
            const double loss = r_update_feature_maps(r, l1H, l2H);
            if (loss_out && &r == &first(h)) *loss_out = loss;
        });
    });
}

int cmf_loss(cmf_handle h, double *loss_out) {
    return guarded([&] { single_set(h, "cmf_loss_batch");
        REQUIRE(loss_out, "null output");
        on_ranks(h, [&](auto &r) {
            REQUIRE(r.world() > 1 || (r.is_first && r.is_last), "shards without a communicator use cmf_loss_partial");
            const double loss = r_guarded_loss(r);
            if (&r == &first(h)) *loss_out = loss;
        });
    });
}

int cmf_fit(cmf_handle h, int64_t max_itr, double max_time, int eval_mode, int check_convergence, int patience,
            double tol, double l1W, double l2W, double l1H, double l2H, double *loss_hist, double *time_hist,
            int64_t cap, int64_t *n_hist, int *converged_early) {
    return guarded([&] { single_set(h, "cmf_fit_batch");
        REQUIRE(loss_hist && time_hist && n_hist, "null history pointers");
        REQUIRE(patience >= 1, "patience must be >= 1 (src/algs/alternating.jl:30)");
        REQUIRE(cap >= 1, "history capacity must be >= 1");
        if (converged_early) *converged_early = 0;
        on_ranks(h, [&](auto &r) {
            REQUIRE(r.world() > 1 || (r.is_first && r.is_last), "shards without a communicator use the split-phase calls");
            std::vector<double> lh, th;
            int early = 0;
            r_fit(r, max_itr, max_time, eval_mode, check_convergence, patience, tol, l1W, l2W, l1H, l2H, lh, th, cap, &early);
            if (&r == &first(h)) {
                std::copy(lh.begin(), lh.end(), loss_hist);
                std::copy(th.begin(), th.end(), time_hist);
                *n_hist = (int64_t)lh.size();
                if (converged_early) *converged_early = early;
            }
        });
    });
}

int cmf_w_partials(cmf_handle h) {
    return guarded([&] { no_batch_split(h); single_rank(h); on_ranks(h, [&](auto &r) { r.w_partials(); }); });
}
int cmf_w_apply(cmf_handle h, double l1W, double l2W) {
    return guarded([&] { no_batch_split(h); single_rank(h); on_ranks(h, [&](auto &r) { r.w_apply(l1W, l2W); }); });
}
int cmf_h_update(cmf_handle h, double l1H, double l2H) {
    return guarded([&] { no_batch_split(h);
        single_rank(h);
        on_ranks(h, [&](auto &r) {
            REQUIRE(r.alg == CMF_MULT, "the split-phase H update is MultUpdate only");
            r.h_update(l1H, l2H);
        });
    });
}
int cmf_loss_partial(cmf_handle h, double *sumsq_out) {
    return guarded([&] { no_batch_split(h); single_rank(h); REQUIRE(sumsq_out, "null output"); on_ranks(h, [&](auto &r) { *sumsq_out = r.loss_partial(); }); });
}
int cmf_exchange_buffer(cmf_handle h, int which, void **dev_ptr, int64_t *count, int *dtype) {
    return guarded([&] { no_batch_split(h); single_rank(h); REQUIRE(dev_ptr && count && dtype, "null output"); on_first(h, [&](auto &r) { r.exchange_buffer(which, dev_ptr, count, dtype); }); });
}
int cmf_halo_buffers(cmf_handle h, void **sl, void **sr, void **rl, void **rr, int64_t *count) {
    return guarded([&] { no_batch_split(h); single_rank(h); REQUIRE(sl && sr && rl && rr && count, "null output"); on_first(h, [&](auto &r) { r.halo_buffers(sl, sr, rl, rr, count); }); });
}
int cmf_sync(cmf_handle h) {
    return guarded([&] { on_ranks(h, [&](auto &r) { CK(cudaStreamSynchronize(r.stream)); }); });
}
int cmf_launch_count(cmf_handle h, int64_t *out) {
    return guarded([&] {
        REQUIRE(h && out, "null argument");
        *out = std::visit([](auto &v) { int64_t n = 0; for (auto &r : v) n += r->launches; return n; }, h->ranks);
    });
}
int cmf_stream(cmf_handle h, void **stream_out) {
    return guarded([&] { REQUIRE(h && stream_out, "null argument"); *stream_out = (void *)first(h).stream; });
}
int cmf_get_data(cmf_handle h, void *X_out, int with_halo) {
    return guarded([&] {
        REQUIRE(X_out, "null output");
        on_ranks(h, [&](auto &r) {
            REQUIRE(r.have_data, "no data");
            // several rank contexts fill one N x T array: no halos
            r.get_data((char *)X_out + (size_t)((r.t0 - first(h).t0) * r.N) * elem_size(r), h->size() > 1 ? 0 : with_halo);
        });
    });
}
int cmf_profile(cmf_handle h, int enable) {
    return guarded([&] {
        on_ranks(h, [&](auto &r) {
            CK(cudaStreamSynchronize(r.stream));
            r.prof_clear();
            r.profiling = enable != 0;
        });
    });
}
int cmf_profile_read(cmf_handle h, int which, double *ms_total, int64_t *count) {
    return guarded([&] {
        REQUIRE(h && ms_total && count, "null output");
        REQUIRE(which >= 0 && which < PROF_NCLASS, "which must be 0 (conv), 1 (transconv), 2 (corr) or 3 (HALS H sweep)");
        RankState &r = first(h);
        DevGuard g(r.device);
        CK(cudaStreamSynchronize(r.stream));
        double tot = 0.0;
        int64_t n = 0;
        for (auto &e : r.prof_events) {
            if (e.which != which) continue;
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, e.a, e.b));
            tot += ms;
            ++n;
        }
        *ms_total = tot;
        *count = n;
    });
}
int cmf_set_stream(cmf_handle h, void *stream) {
    return guarded([&] {
        single_rank(h);
        RankState &r = first(h);
        DevGuard g(r.device);
        CK(cudaStreamSynchronize(r.stream));
        if (r.own_stream && r.stream) cudaStreamDestroy(r.stream);
        r.own_stream = false;
        r.stream = (cudaStream_t)stream;
    });
}
int cmf_set_engine(cmf_handle h, int engine) {
    return guarded([&] { on_ranks(h, [&](auto &r) { r_set_engine(r, engine); }); });
}

int cmf_set_loss_mode(cmf_handle h, int mode) {
    return guarded([&] {
        REQUIRE(mode == 0 || mode == 1, "loss mode must be 0 (direct) or 1 (expansion)");
        if (h && first(h).R > 0 && mode != 0) throw CmfError(CMF_ERR_UNSUPPORTED, "batch handles evaluate the loss by the direct pass (mode 0) only");
        on_ranks(h, [&](auto &r) { r.loss_mode = mode; r.loss_mode_explicit = true; r.calib_reset(); });
    });
}
int cmf_set_loss_guard(cmf_handle h, double guard, int max_interval) {
    return guarded([&] {
        REQUIRE(guard >= 0.0, "loss guard must be >= 0");
        REQUIRE(max_interval >= 1 && max_interval <= 1024, "calibration interval must be in [1, 1024]");
        on_ranks(h, [&](auto &r) { r.loss_guard = guard; r.calib_max_interval = max_interval; r.calib_reset(); });
    });
}
int cmf_get_loss_stats(cmf_handle h, int64_t *n_direct, int64_t *n_expansion, int *interval, double *last_err) {
    return guarded([&] {
        REQUIRE(h, "null handle");
        const RankState &r = first(h);
        if (n_direct) *n_direct = r.n_loss_direct;
        if (n_expansion) *n_expansion = r.n_loss_expansion;
        if (interval) *interval = r.calib_have ? r.calib_interval : 0;
        if (last_err) *last_err = r.calib_last_err;
    });
}
int cmf_get_loss_mode(cmf_handle h, int *mode_out) {
    return guarded([&] { REQUIRE(h && mode_out, "null argument"); *mode_out = first(h).loss_mode; });
}
int cmf_get_fd_layout(cmf_handle h, int *block_len, int *hop, int64_t *nblocks) {
    return guarded([&] {
        REQUIRE(h && block_len && hop && nblocks, "null argument");
        on_first(h, [&](auto &r) { r.fd_layout(block_len, hop, nblocks); });
    });
}
int cmf_get_engine(cmf_handle h, int *engine_out) {
    return guarded([&] { REQUIRE(h && engine_out, "null argument"); *engine_out = first(h).engine; });
}

static int current_device() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) d = 0;
    return d;
}

int cmf_set_pgd_constraints(cmf_handle h, int constrW, int constrH) {
    return guarded([&] { single_rank(h); on_first(h, [&](auto &r) { r.set_pgd_constraints(constrW, constrH); }); });
}
int cmf_set_pgd_loss(cmf_handle h, int loss_func, const void *mask) {
    return guarded([&] { single_rank(h); on_ranks(h, [&](auto &r) { r.set_pgd_loss(loss_func, mask); }); });
}

int cmf_tensor_conv(int64_t N, int64_t T, int64_t K, int64_t L, int dtype, const void *W, const void *H, void *out) {
    return guarded([&] {
        REQUIRE(W && H && out, "null pointer");
        with_dtype(dtype, [&](auto s) {
            auto c = make_ctx<decltype(s)>(N, T, 0, T, K, L, dtype, CMF_MULT, current_device());
            c->set_factors(W, H, 0);
            c->prim_conv(out);
        });
    });
}
int cmf_tensor_transconv(int64_t N, int64_t T, int64_t K, int64_t L, int dtype, const void *W, const void *X, void *out) {
    return guarded([&] {
        REQUIRE(W && X && out, "null pointer");
        with_dtype(dtype, [&](auto s) {
            auto c = make_ctx<decltype(s)>(N, T, 0, T, K, L, dtype, CMF_MULT, current_device());
            std::vector<decltype(s)> Hz((size_t)(K * T), 0);
            c->set_factors(W, Hz.data(), 0);
            c->prim_transconv(X, out);
        });
    });
}
int cmf_corr_w(int64_t N, int64_t T, int64_t K, int64_t L, int dtype, const void *H, const void *X, void *out) {
    return guarded([&] {
        REQUIRE(H && X && out, "null pointer");
        with_dtype(dtype, [&](auto s) {
            auto c = make_ctx<decltype(s)>(N, T, 0, T, K, L, dtype, CMF_MULT, current_device());
            std::vector<decltype(s)> Wz((size_t)(K * N * L), 0);
            c->set_factors(Wz.data(), H, 0);
            c->prim_corr(X, out);
        });
    });
}
int cmf_compute_resids(int64_t N, int64_t T, int64_t K, int64_t L, int dtype, const void *X, const void *W, const void *H, void *out) {
    return guarded([&] {
        REQUIRE(X && W && H && out, "null pointer");
        with_dtype(dtype, [&](auto s) {
            auto c = make_ctx<decltype(s)>(N, T, 0, T, K, L, dtype, CMF_MULT, current_device());
            c->set_data(X, 0);
            c->set_factors(W, H, 0);
            c->prim_resids(out);
        });
    });
}
int cmf_shift_and_stack(int64_t K, int64_t T, int64_t L, int dtype, const void *H, void *out) {
    return guarded([&] {
        REQUIRE(H && out, "null pointer");
        with_dtype(dtype, [&](auto s) {
            auto c = make_ctx<decltype(s)>(8, T, 0, T, K, L, dtype, CMF_MULT, current_device());
            std::vector<decltype(s)> Wz((size_t)(K * 8 * L), 0);
            c->set_factors(Wz.data(), H, 0);
            c->prim_shift_and_stack(out);
        });
    });
}

int cmf_create_batch(cmf_handle *out, int64_t N, int64_t T, int64_t K, int64_t L, int dtype, int alg, int64_t R, int device) {
    return guarded([&] {
        REQUIRE(out != nullptr, "null output pointer");
        REQUIRE(R >= 1 && R <= 32768, "R (restarts) must be in 1..32768");
        DevRestore g;
        *out = make_batch(N, T, std::vector<int64_t>((size_t)R, K), L, dtype, alg, device);
    });
}
int cmf_create_batch_ranks(cmf_handle *out, int64_t N, int64_t T, const int64_t *K, int64_t L, int dtype, int alg, int64_t R,
                           int device) {
    return guarded([&] {
        REQUIRE(out != nullptr, "null output pointer");
        REQUIRE(K != nullptr, "null rank array K");
        REQUIRE(R >= 1 && R <= 32768, "R (restarts) must be in 1..32768");
        DevRestore g;
        *out = make_batch(N, T, std::vector<int64_t>(K, K + R), L, dtype, alg, device);
    });
}
int cmf_set_factors_batch(cmf_handle h, const void *W, const void *H) {
    return guarded([&] { batch_handle(h); on_ranks(h, [&](auto &r) { r.batch_set_factors(W, H); }); });
}
int cmf_get_factors_batch(cmf_handle h, void *W_out, void *H_out) {
    return guarded([&] { batch_handle(h); on_ranks(h, [&](auto &r) { r.batch_get_factors(W_out, H_out); }); });
}
int cmf_init_scale_partials_batch(cmf_handle h, double *out) {
    return guarded([&] { REQUIRE(out, "null output"); batch_handle(h); on_ranks(h, [&](auto &r) { r.batch_scale_partials(out); }); });
}
int cmf_scale_factors_batch(cmf_handle h, const double *s) {
    return guarded([&] { REQUIRE(s, "null scale factors"); batch_handle(h); on_ranks(h, [&](auto &r) { r.batch_scale(s); }); });
}
int cmf_loss_batch(cmf_handle h, double *loss_out) {
    return guarded([&] { REQUIRE(loss_out, "null output"); batch_handle(h); on_ranks(h, [&](auto &r) { r.batch_loss(loss_out); }); });
}
int cmf_fit_batch(cmf_handle h, int64_t max_itr, double max_time, int eval_mode, int check_convergence, int patience, double tol,
                  const double *l1W, const double *l2W, const double *l1H, const double *l2H, double *loss_hist, double *time_hist,
                  int64_t cap, int64_t *n_hist, int *converged_early) {
    return guarded([&] {
        batch_handle(h);
        REQUIRE(l1W && l2W && l1H && l2H, "null regulariser arrays");
        REQUIRE(loss_hist && time_hist && n_hist && converged_early, "null history pointers");
        REQUIRE(patience >= 1, "patience must be >= 1 (src/algs/alternating.jl:30)");
        REQUIRE(cap >= 1, "history capacity must be >= 1");
        on_ranks(h, [&](auto &r) {
            std::vector<double> th;
            b_fit(r, max_itr, max_time, eval_mode, check_convergence, patience, tol, l1W, l2W, l1H, l2H, loss_hist, th, cap, n_hist,
                  converged_early);
            std::copy(th.begin(), th.end(), time_hist);
        });
    });
}

}  // extern "C"
