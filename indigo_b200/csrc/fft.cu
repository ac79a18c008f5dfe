// Batched 1-D/2-D/3-D complex64 FFT (unscaled forward, unscaled inverse).
//
// Interface replaced: Backend.fftn / ifftn (indigo/backends/backend.py:497-509),
// semantics of the numpy backend (np.py:102-115); the reference GPU path is a
// cuFFT plan cache (cuda.py:470-498).  Hand-written instead:
//   * one pass per axis, each a shared-memory Stockham auto-sort over a tile of
//     L lines x n points; on strided axes the first radix stage reads global
//     memory directly and the last one writes it directly, so a pass moves every
//     element through HBM exactly once in each direction (16 B per point);
//   * strided axes (1, 2) take tiles of L=16 neighbouring lines so that every
//     global access is a 128-byte segment; axis 0 takes L consecutive lines
//     (one contiguous chunk) and transposes through shared memory;
//   * mixed radix 2,3,4,5,7,8,11,13,16 in registers (416 = 13*8*4), generic
//     butterfly for other primes; the inverse reuses the forward butterflies by
//     swapping re/im on load and store; optional diagonal multiply fused into
//     the first load / last store (coil maps, apodisation, centring phase).
// Tile logic lives in fft_core.cuh, planning in fft_plan.hpp (both shared with
// the CPU emulation harness used by the GPU-less tests).
#include "fft_plan.hpp"
#include "fft_il.cuh"
#include "fft_pk.cuh"

#include <cstdlib>
#include <new>

namespace ib200 {

static const int kFftThreads = 256;

template <bool AXIS0>
__global__ void __launch_bounds__(kFftThreads) fft_pass_kernel(const FftKernelArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    fft_pass_body<AXIS0>(a, reinterpret_cast<c64 *>(smem_raw), (int64_t)blockIdx.x, (int)threadIdx.x, (int)blockDim.x);
}

template <int N, int R0, int R1, int R2, bool AXIS0, int THREADS>
__global__ void __launch_bounds__(THREADS, (THREADS > 256 ? 2 : 2)) fft_spec_kernel(const FftKernelArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    fft_pass_body_spec<N, R0, R1, R2, AXIS0>(a, reinterpret_cast<c64 *>(smem_raw), (int64_t)blockIdx.x,
                                             (int)threadIdx.x, (int)blockDim.x);
}

template <int N, int R0, int R1, int R2, bool AXIS0, int THREADS>
static int launch_spec_t(cudaStream_t s, const FftKernelArgs &k) {
    static bool attr_done[64] = {false};
    const size_t smem = (size_t)(R2 > 1 ? 2 : 1) * N * kSpecLP * sizeof(c64);
    int dev = 0;
    IB200_TRY(cudaGetDevice(&dev));
    if (!attr_done[dev & 63]) {
        IB200_TRY(cudaFuncSetAttribute(fft_spec_kernel<N, R0, R1, R2, AXIS0, THREADS>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev & 63] = true;
    }
    const int64_t blocks = AXIS0 ? ceil_div(k.outer, kSpecL) : ceil_div(k.inner, kSpecL) * k.outer;
    IB200_REQUIRE(blocks < (1LL << 31), "fft: too many tiles for one launch");
    fft_spec_kernel<N, R0, R1, R2, AXIS0, THREADS><<<(unsigned)blocks, THREADS, smem, s>>>(k);
    IB200_LAUNCH_CHECK();
    return 0;
}

template <int N, int R0, int R1, int R2, bool AXIS0>
static int launch_spec(cudaStream_t s, const FftKernelArgs &k) {
    // 512 threads (two CTAs of 16 warps per SM) measured 15-20 % faster than 256 on the 416-point
    // passes of cfg3 (profiles/r01_s4_*): the passes are issue/latency bound, not DRAM bound.
    static const int threads = getenv("IB200_FFT_THREADS") ? atoi(getenv("IB200_FFT_THREADS")) : (N >= 128 ? 512 : 256);
    if (threads == 512) return launch_spec_t<N, R0, R1, R2, AXIS0, 512>(s, k);
    if (threads == 128) return launch_spec_t<N, R0, R1, R2, AXIS0, 128>(s, k);
    return launch_spec_t<N, R0, R1, R2, AXIS0, 256>(s, k);
}

static int try_pk_pass(cudaStream_t s, const IlPassArgs &a, int n, const FftStages &st, bool swap_in, bool swap_out);

// returns 1 if a specialised kernel was launched, 0 if none applies, <0 / >0 on error (offset by 1000)
static int try_spec(cudaStream_t s, bool axis0, const FftKernelArgs &k) {
    if (!axis0 && k.inner < kSpecL) return 0;
    if (axis0 && k.outer < kSpecL) return 0;
    // strided axes transformed in place, no fused diagonal, whole 16-line tiles: the packed two-lines-per-thread
    // passes of the fused recipe (fft_pk.cuh) serve Backend.fftn / ifftn too
    if (!axis0 && k.x == k.y && !k.din && !k.dout && k.inner % kSpecL == 0 && k.inner < (1LL << 32) &&
        !(k.swap_in && k.swap_out) && k.in0 == 0 && k.in1 == k.n && k.out0 == 0 && k.out1 == k.n) {
        IlPassArgs a;
        a.x = k.y; a.tw = k.tw; a.inner = k.inner; a.outer = k.outer; a.outer_stride = k.outer_stride;
        a.pstride = (unsigned)k.inner; a.in0 = 0; a.in1 = k.n; a.out0 = 0; a.out1 = k.n;
        const int r = try_pk_pass(s, a, k.n, k.st, k.swap_in != 0, k.swap_out != 0);
        if (r != 0) return r;
    }
#define IB200_TRY_SPEC(n, r0, r1, r2)                                                        \
    if (fft_spec_matches(k, n, r0, r1, r2)) {                                                \
        const int rc = axis0 ? launch_spec<n, r0, r1, r2, true>(s, k) : launch_spec<n, r0, r1, r2, false>(s, k); \
        return rc == 0 ? 1 : (rc > 0 ? rc + 1000 : rc);                                      \
    }
    IB200_FFT_SPEC_LIST(IB200_TRY_SPEC)
#undef IB200_TRY_SPEC
    return 0;
}

// ---- fused SENSE x passes on the interleaved grid (fft_il.cuh) ---------------------------------
static constexpr int sense_x_threads(int n) { return n >= 128 ? 512 : 256; }

template <int N, int R0, int R1, int R2>
__global__ void __launch_bounds__(sense_x_threads(N), 2) sense_expand_kernel(const SenseFftArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    sense_expand_body<N, R0, R1, R2>(a, reinterpret_cast<c64 *>(smem_raw), (int64_t)blockIdx.x, (int)threadIdx.x,
                                     (int)blockDim.x);
}

template <int N, int R0, int R1, int R2>
__global__ void __launch_bounds__(sense_x_threads(N), 2) sense_combine_kernel(const SenseFftArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    c64 *buf = reinterpret_cast<c64 *>(smem_raw);
    sense_combine_body<N, R0, R1, R2>(a, buf, buf + (size_t)2 * N * kSpecLP, (int64_t)blockIdx.x, (int)threadIdx.x,
                                      (int)blockDim.x);
}

template <int N, int R0, int R1, int R2>
static int launch_sense_x(cudaStream_t s, bool combine, const SenseFftArgs &a) {
    static bool attr_done[2][64] = {{false}};
    const size_t smem = (size_t)2 * N * kSpecLP * sizeof(c64) + (combine ? (size_t)a.N0 * sense_x_tile(a.C).YY * sizeof(c64) : 0);
    IB200_REQUIRE((int64_t)smem <= smem_optin(), "sense x pass: tile does not fit shared memory");
    int dev = 0;
    IB200_TRY(cudaGetDevice(&dev));
    if (!attr_done[combine ? 1 : 0][dev & 63]) {
        if (combine) IB200_TRY(cudaFuncSetAttribute(sense_combine_kernel<N, R0, R1, R2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin()));
        else         IB200_TRY(cudaFuncSetAttribute(sense_expand_kernel<N, R0, R1, R2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin()));
        attr_done[combine ? 1 : 0][dev & 63] = true;
    }
    const int64_t blocks = sense_x_blocks(a.N1, a.N2, a.C);
    IB200_REQUIRE(blocks < (1LL << 31), "sense x pass: too many rows for one launch");
    if (combine) sense_combine_kernel<N, R0, R1, R2><<<(unsigned)blocks, sense_x_threads(N), smem, s>>>(a);
    else         sense_expand_kernel<N, R0, R1, R2><<<(unsigned)blocks, sense_x_threads(N), smem, s>>>(a);
    IB200_LAUNCH_CHECK();
    return 0;
}

template <int N, int R0, int R1, int R2, bool SI, bool SO>
__global__ void __launch_bounds__(sense_x_threads(N), 2) fft_il_pass_kernel(const IlPassArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    fft_il_pass_body<N, R0, R1, R2, SI, SO>(a, reinterpret_cast<c64 *>(smem_raw), (int64_t)blockIdx.x, (int)threadIdx.x,
                                            (int)blockDim.x);
}

template <int N, int R0, int R1, int R2, bool SI, bool SO>
static int launch_il_pass(cudaStream_t s, const IlPassArgs &a) {
    static bool attr_done[64] = {false};
    const size_t smem = (size_t)(R2 > 1 ? 2 : 1) * N * kSpecLP * sizeof(c64);
    int dev = 0;
    IB200_TRY(cudaGetDevice(&dev));
    if (!attr_done[dev & 63]) {
        IB200_TRY(cudaFuncSetAttribute(fft_il_pass_kernel<N, R0, R1, R2, SI, SO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev & 63] = true;
    }
    const int64_t blocks = (a.inner / kSpecL) * a.outer;
    IB200_REQUIRE(blocks < (1LL << 31), "fft: too many tiles for one launch");
    fft_il_pass_kernel<N, R0, R1, R2, SI, SO><<<(unsigned)blocks, sense_x_threads(N), smem, s>>>(a);
    IB200_LAUNCH_CHECK();
    return 0;
}

// returns 1 when launched, 0 when no specialised size matches, else an error code (+1000 when positive)
static int try_il_pass(cudaStream_t s, const IlPassArgs &a, int n, const FftStages &st, bool swap_in, bool swap_out) {
    FftKernelArgs k;
    k.n = n; k.st = st;
#define IB200_IL_PASS(nn, r0, r1, r2)                                                            \
    if (fft_spec_matches(k, nn, r0, r1, r2)) {                                                   \
        int rc;                                                                                  \
        if (swap_in)       rc = launch_il_pass<nn, r0, r1, r2, true, false>(s, a);               \
        else if (swap_out) rc = launch_il_pass<nn, r0, r1, r2, false, true>(s, a);               \
        else               rc = launch_il_pass<nn, r0, r1, r2, false, false>(s, a);              \
        return rc == 0 ? 1 : (rc > 0 ? rc + 1000 : rc);                                          \
    }
    IB200_FFT_SPEC_LIST(IB200_IL_PASS)
#undef IB200_IL_PASS
    return 0;
}

// ---- packed two-lines-per-thread variants (fft_pk.cuh): 256 threads, split-plane tiles ----------------
static const int kPkThreads = 256;
static bool pk_enabled() { static const bool on = getenv("IB200_FFT_NOPK") == nullptr; return on; }

template <int N, int R0, int R1, int R2, bool SI, bool SO>
__global__ void __launch_bounds__(kPkThreads, 2) fft_pk_pass_kernel(const IlPassArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    fft_pk_pass_body<N, R0, R1, R2, SI, SO, kPkThreads>(a, reinterpret_cast<float *>(smem_raw), (int64_t)blockIdx.x, (int)threadIdx.x,
                                            (int)blockDim.x);
}

template <int N, int R0, int R1, int R2, bool SI, bool SO>
static int launch_pk_pass(cudaStream_t s, const IlPassArgs &a) {
    static bool attr_done[64] = {false};
    const size_t smem = pk_smem_floats(N, R2 > 1, false) * sizeof(float);
    if ((int64_t)smem > smem_optin()) return -100;                  // caller falls back to the one-line kernels
    int dev = 0;
    IB200_TRY(cudaGetDevice(&dev));
    if (!attr_done[dev & 63]) {
        IB200_TRY(cudaFuncSetAttribute(fft_pk_pass_kernel<N, R0, R1, R2, SI, SO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev & 63] = true;
    }
    const int64_t blocks = (a.inner / kSpecL) * a.outer;
    IB200_REQUIRE(blocks < (1LL << 31), "fft: too many tiles for one launch");
    fft_pk_pass_kernel<N, R0, R1, R2, SI, SO><<<(unsigned)blocks, kPkThreads, smem, s>>>(a);
    IB200_LAUNCH_CHECK();
    return 0;
}

// persistent prefetching form (fft_pk.cuh): one CTA pair per SM walks the tiles
template <int N, int R0, int R1, int R2, bool SI, bool SO>
__global__ void __launch_bounds__(kPkThreads, 2) fft_pkp_pass_kernel(const IlPassArgs a, int64_t ntiles) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *bufA = reinterpret_cast<float *>(smem_raw);
    c64 *raw = reinterpret_cast<c64 *>(bufA + pk_buf_floats(N));
    // twiddle table in shared memory: every butterfly of every tile reads R-1 entries; as cached global loads
    // they were 15 % of the pass (long-scoreboard stalls on top of the L1 traffic), as shared-memory reads 0
    c64 *stw = raw + (size_t)N * kSpecL;
    const int tid = (int)threadIdx.x;
    int64_t tile = pkp_next_active(a, blockIdx.x, gridDim.x, ntiles, tid, kPkThreads);
    if (tile < 0) return;
    pkp_prefetch(a, tile, raw, tid, kPkThreads);
    for (int i = tid; i < N; i += kPkThreads) stw[i] = a.tw[i];
    while (tile >= 0) {
        const int64_t next = pkp_next_active(a, tile + gridDim.x, gridDim.x, ntiles, tid, kPkThreads);
        pkp_wait();
        __syncthreads();                                             // raw[] of this tile visible; bufA of the last tile consumed
        fft_pkp_tile_body<N, R0, R1, R2, SI, SO, kPkThreads>(a, tile, next, bufA, raw, tid, kPkThreads, stw);
        tile = next;
    }
}

template <int N, int R0, int R1, int R2, bool SI, bool SO>
static int launch_pkp_pass(cudaStream_t s, const IlPassArgs &a) {
    static bool attr_done[64] = {false};
    const size_t smem = pk_buf_floats(N) * sizeof(float) + (size_t)N * kSpecL * sizeof(c64) + (size_t)N * sizeof(c64);
    if ((int64_t)smem > smem_optin()) return -100;
    int dev = 0;
    IB200_TRY(cudaGetDevice(&dev));
    if (!attr_done[dev & 63]) {
        IB200_TRY(cudaFuncSetAttribute(fft_pkp_pass_kernel<N, R0, R1, R2, SI, SO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev & 63] = true;
    }
    const int64_t ntiles = (a.inner / kSpecL) * a.outer;
    static const int per_sm = getenv("IB200_FFT_PKP_CTAS") ? atoi(getenv("IB200_FFT_PKP_CTAS")) : 2;
    int64_t blocks = (int64_t)sm_count() * per_sm;
    if (blocks > ntiles) blocks = ntiles;
    fft_pkp_pass_kernel<N, R0, R1, R2, SI, SO><<<(unsigned)blocks, kPkThreads, smem, s>>>(a, ntiles);
    IB200_LAUNCH_CHECK();
    return 0;
}

template <int N, int R0, int R1, int R2, bool SI, bool SO>
static int launch_pk_or_pkp(cudaStream_t s, const IlPassArgs &a) {
    static const bool persistent = getenv("IB200_FFT_NOPKP") == nullptr;
    if (persistent && pkp_mid_pairs(N, R1, R2, kPkThreads) <= 16) {
        const int rc = launch_pkp_pass<N, R0, R1, R2, SI, SO>(s, a);
        if (rc != -100) return rc;
    }
    return launch_pk_pass<N, R0, R1, R2, SI, SO>(s, a);
}

// returns 1 when launched, 0 when not applicable, else an error code (+1000 when positive)
static int try_pk_pass(cudaStream_t s, const IlPassArgs &a, int n, const FftStages &st, bool swap_in, bool swap_out) {
    if (!pk_enabled() || (a.outer_stride & 1) || ((uintptr_t)a.x & 15)) return 0;
    FftKernelArgs k;
    k.n = n; k.st = st;
#define IB200_PK_PASS(nn, r0, r1, r2)                                                            \
    if (fft_spec_matches(k, nn, r0, r1, r2)) {                                                   \
        int rc;                                                                                  \
        if (swap_in)       rc = launch_pk_or_pkp<nn, r0, r1, r2, true, false>(s, a);             \
        else if (swap_out) rc = launch_pk_or_pkp<nn, r0, r1, r2, false, true>(s, a);             \
        else               rc = launch_pk_or_pkp<nn, r0, r1, r2, false, false>(s, a);            \
        if (rc == -100) return 0;                                                                \
        return rc == 0 ? 1 : (rc > 0 ? rc + 1000 : rc);                                          \
    }
    IB200_FFT_SPEC_LIST(IB200_PK_PASS)
#undef IB200_PK_PASS
    return 0;
}

// Toeplitz convolution pass (fft_pkt_tile_body): persistent like fft_pkp_pass_kernel, same shared memory
template <int N, int R0, int R1, int R2>
__global__ void __launch_bounds__(kPkThreads, 2) fft_pkt_pass_kernel(const IlPassArgs a, int64_t ntiles,
                                                                     const float *__restrict__ kern, int64_t kplane, int C) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *bufA = reinterpret_cast<float *>(smem_raw);
    c64 *raw = reinterpret_cast<c64 *>(bufA + pk_buf_floats(N));
    c64 *stw = raw + (size_t)N * kSpecL;
    const int tid = (int)threadIdx.x;
    int64_t tile = blockIdx.x;
    if (tile >= ntiles) return;
    pkp_prefetch(a, tile, raw, tid, kPkThreads);
    for (int i = tid; i < N; i += kPkThreads) stw[i] = a.tw[i];
    while (tile >= 0) {
        const int64_t next = tile + gridDim.x < ntiles ? tile + gridDim.x : -1;
        pkp_wait();
        __syncthreads();
        fft_pkt_tile_body<N, R0, R1, R2, kPkThreads>(a, tile, next, bufA, raw, tid, kPkThreads, stw, kern, kplane, C);
        tile = next;
    }
}

// every stage of the Toeplitz pass runs in place at least once: all of them must stay within the 16 register pairs
// per thread of the persistent pass (every length up to 512; the longer ones are never a Toeplitz grid)
static constexpr int pk_inplace_pairs(int n, int r) { return ((kSpecL / 2 * (n / r) + kPkThreads - 1) / kPkThreads) * r; }
static constexpr bool pkt_fits(int n, int r0, int r1, int r2) {
    return pk_inplace_pairs(n, r0) <= 16 && pk_inplace_pairs(n, r1) <= 16 && (r2 <= 1 || pk_inplace_pairs(n, r2) <= 16);
}

template <int N, int R0, int R1, int R2>
static int launch_pkt_pass(cudaStream_t s, const IlPassArgs &a, const float *kern, int64_t kplane, int C) {
    const size_t smem = pk_buf_floats(N) * sizeof(float) + (size_t)N * kSpecL * sizeof(c64) + (size_t)N * sizeof(c64);
    if constexpr (!pkt_fits(N, R0, R1, R2)) {
        (void)s; (void)a; (void)kern; (void)kplane; (void)C; (void)smem;
        set_error("Toeplitz pass: length %d does not fit the persistent packed pass", N);
        return IB200_E_UNSUPPORTED;
    } else {
    static bool attr_done[64] = {false};
    if ((int64_t)smem > smem_optin()) {
        set_error("Toeplitz pass: length %d does not fit shared memory", N);
        return IB200_E_UNSUPPORTED;
    }
    int dev = 0;
    IB200_TRY(cudaGetDevice(&dev));
    if (!attr_done[dev & 63]) {
        IB200_TRY(cudaFuncSetAttribute(fft_pkt_pass_kernel<N, R0, R1, R2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev & 63] = true;
    }
    const int64_t ntiles = (a.inner / kSpecL) * a.outer;
    int64_t blocks = (int64_t)sm_count() * 2;
    if (blocks > ntiles) blocks = ntiles;
    fft_pkt_pass_kernel<N, R0, R1, R2><<<(unsigned)blocks, kPkThreads, smem, s>>>(a, ntiles, kern, kplane, C);
    IB200_LAUNCH_CHECK();
    return 0;
    }
}

static int run_pkt_pass(cudaStream_t s, const IlPassArgs &a, int n, const FftStages &st, const float *kern, int64_t kplane,
                        int C) {
    FftKernelArgs k;
    k.n = n; k.st = st;
#define IB200_PKT_PASS(nn, r0, r1, r2) \
    if (fft_spec_matches(k, nn, r0, r1, r2)) return launch_pkt_pass<nn, r0, r1, r2>(s, a, kern, kplane, C);
    IB200_FFT_SPEC_LIST(IB200_PKT_PASS)
#undef IB200_PKT_PASS
    set_error("Toeplitz pass needs an axis length with a specialised FFT (got %d)", n);
    return IB200_E_UNSUPPORTED;
}

template <int N, int R0, int R1, int R2>
__global__ void __launch_bounds__(kPkThreads, 2) sense_expand_pk_kernel(const SenseFftArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    sense_expand_pk_body<N, R0, R1, R2, kPkThreads>(a, reinterpret_cast<float *>(smem_raw), (int64_t)blockIdx.x, (int)threadIdx.x,
                                                    (int)blockDim.x);
}

template <int N, int R0, int R1, int R2>
__global__ void __launch_bounds__(kPkThreads, 2) sense_combine_pk_kernel(const SenseFftArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *buf = reinterpret_cast<float *>(smem_raw);
    c64 *acc = reinterpret_cast<c64 *>(buf + pk_smem_floats(N, R2 > 1, true));
    // (a shared-memory twiddle table, which pays in the persistent strided passes, costs these one-shot kernels
    // registers they do not have: measured slower)
    sense_combine_pk_body<N, R0, R1, R2, kPkThreads>(a, buf, acc, (int64_t)blockIdx.x, (int)threadIdx.x, (int)blockDim.x);
}

// returns 0 when launched, -100 when the packed kernels do not apply
template <int N, int R0, int R1, int R2>
static int launch_sense_x_pk(cudaStream_t s, bool combine, const SenseFftArgs &a) {
    static bool attr_done[2][64] = {{false}};
    if (!pk_enabled() || (a.C & 1)) return -100;
    if (((uintptr_t)a.grid & 15) || ((uintptr_t)a.pf & 15)) return -100;
    // the cross-chunk accumulators of the coil fold are only needed with more than one 16-coil chunk; without them a
    // 2-coil operator (8 image rows per tile) keeps two CTAs per SM (r02: 12.5 % occupancy, 0.52 ms with them)
    const size_t accb = a.C > kSpecL ? (size_t)a.N0 * sense_x_tile(a.C).YY * sizeof(c64) : 0;
    const size_t smem = combine ? pk_smem_floats(N, R2 > 1, true) * sizeof(float) + accb
                                : pk_smem_floats(N, R2 > 1, false) * sizeof(float);
    if ((int64_t)smem > smem_optin()) return -100;
    int dev = 0;
    IB200_TRY(cudaGetDevice(&dev));
    if (!attr_done[combine ? 1 : 0][dev & 63]) {
        if (combine) IB200_TRY(cudaFuncSetAttribute(sense_combine_pk_kernel<N, R0, R1, R2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin()));
        else         IB200_TRY(cudaFuncSetAttribute(sense_expand_pk_kernel<N, R0, R1, R2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin()));
        attr_done[combine ? 1 : 0][dev & 63] = true;
    }
    const int64_t blocks = sense_x_blocks(a.N1, a.N2, a.C);
    IB200_REQUIRE(blocks < (1LL << 31), "sense x pass: too many rows for one launch");
    if (combine) sense_combine_pk_kernel<N, R0, R1, R2><<<(unsigned)blocks, kPkThreads, smem, s>>>(a);
    else         sense_expand_pk_kernel<N, R0, R1, R2><<<(unsigned)blocks, kPkThreads, smem, s>>>(a);
    IB200_LAUNCH_CHECK();
    return 0;
}

static int run_sense_x(cudaStream_t s, bool combine, const SenseFftArgs &a, const FftStages &st) {
    FftKernelArgs k;
    k.n = a.n0; k.st = st;
#define IB200_SENSE_X(n, r0, r1, r2)                                       \
    if (fft_spec_matches(k, n, r0, r1, r2)) {                              \
        const int rc = launch_sense_x_pk<n, r0, r1, r2>(s, combine, a);    \
        if (rc != -100) return rc;                                         \
        return launch_sense_x<n, r0, r1, r2>(s, combine, a);               \
    }
    IB200_FFT_SPEC_LIST(IB200_SENSE_X)
#undef IB200_SENSE_X
    set_error("fused SENSE passes need a grid extent with a specialised FFT (got %d)", a.n0);
    return IB200_E_UNSUPPORTED;
}

}  // namespace ib200

struct ib200_fft_plan_s {
    ib200::FftPlanData d;
};

namespace ib200 {

static int ensure_device_state(FftPlanData *pl) {
    int dev = 0;
    IB200_TRY(cudaGetDevice(&dev));
    if (pl->dev == dev) return 0;
    IB200_REQUIRE(pl->dev == -1, "fft plan used on a different device than it was first executed on");
    for (int a = 0; a < pl->ndim; ++a) {
        AxisPlan &ax = pl->ax[a];
        if (ax.n <= 1) continue;
        std::vector<c64> tw;
        fft_make_twiddles(ax.n, tw);
        IB200_TRY(cudaMalloc(&ax.tw_dev, sizeof(c64) * (size_t)ax.n));
        IB200_TRY(cudaMemcpy(ax.tw_dev, tw.data(), sizeof(c64) * (size_t)ax.n, cudaMemcpyHostToDevice));
    }
    IB200_TRY(cudaFuncSetAttribute(fft_pass_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin()));
    IB200_TRY(cudaFuncSetAttribute(fft_pass_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_optin()));
    pl->dev = dev;
    return 0;
}

static int exec_impl(FftPlanData *pl, cudaStream_t s, c64 *y, const c64 *x, int direction, const c64 *din,
                     int conj_in, const c64 *dout, int conj_out) {
    int64_t total = pl->batch;
    for (int a = 0; a < pl->ndim; ++a) total *= pl->dims[a];
    if (total == 0) return 0;
    int rc = ensure_device_state(pl);
    if (rc) return rc;
    bool copy_only = false;
    static const bool use_spec = getenv("IB200_FFT_GENERIC") == nullptr;
    auto launch = [&](bool axis0, int64_t blocks, size_t smem, const FftKernelArgs &k) -> int {
        if (use_spec) {
            const int sp = try_spec(s, axis0, k);
            if (sp == 1) return 0;
            if (sp != 0) return sp > 1000 ? sp - 1000 : sp;
        }
        if (axis0) fft_pass_kernel<true><<<(unsigned)blocks, kFftThreads, smem, s>>>(k);
        else       fft_pass_kernel<false><<<(unsigned)blocks, kFftThreads, smem, s>>>(k);
        IB200_LAUNCH_CHECK();
        return 0;
    };
    rc = fft_exec_passes(pl, y, x, direction, din, conj_in, dout, conj_out, smem_optin(), launch, &copy_only);
    if (rc) return rc;
    if (copy_only && x != y)
        IB200_TRY(cudaMemcpyAsync(y, x, (size_t)total * sizeof(c64), cudaMemcpyDeviceToDevice, s));
    return 0;
}

}  // namespace ib200

using namespace ib200;

// z axis of at most kTinyAxis points (2-D problems carried as N0 x N1 x 1 images: cfg1's grid is 512 x 512 x 2):
// the "transform" is a handful of complex adds per (y, x, coil) line, done directly by one thread per line, in
// place.  Forward: out[k] = sum_{j in window} in[j] e^{-2 pi i jk/n}.  Inverse: this is the FIRST pass of the
// inverse chain, whose later passes run forward transforms on (im, re)-swapped data (conjugation trick), so it
// stores swap(sum_k in[k] e^{+2 pi i jk/n}) for the output window j only.
static const int kTinyAxis = 8;

template <bool INV>
__global__ void __launch_bounds__(256) sense_tiny_z_kernel(c64 *__restrict__ grid, int64_t plane, int n, int w0, int w1) {
    c64 tw[kTinyAxis];
    for (int m = 0; m < n; ++m) {
        double sn, cs;
        sincospi(2.0 * (double)m / (double)n, &sn, &cs);
        tw[m] = mk((float)cs, (float)(INV ? sn : -sn));
    }
    const int64_t nth = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < plane; i += nth) {
        c64 v[kTinyAxis];
        if (!INV) {
            for (int j = w0; j < w1; ++j) v[j - w0] = grid[(int64_t)j * plane + i];
            for (int k = 0; k < n; ++k) {
                c64 acc = mk(0.f, 0.f);
                for (int j = w0; j < w1; ++j) acc = cfma(v[j - w0], tw[(j * k) % n], acc);
                grid[(int64_t)k * plane + i] = acc;
            }
        } else {
            for (int k = 0; k < n; ++k) v[k] = grid[(int64_t)k * plane + i];
            for (int j = w0; j < w1; ++j) {
                c64 acc = mk(0.f, 0.f);
                for (int k = 0; k < n; ++k) acc = cfma(v[k], tw[(j * k) % n], acc);
                grid[(int64_t)j * plane + i] = cswap(acc);
            }
        }
    }
}

extern "C" {

int ib200_fft_plan_create(ib200_fft_plan *plan, int ndim, const int64_t *dims, int64_t batch) {
    IB200_REQUIRE(plan && dims, "null pointer");
    IB200_REQUIRE(ndim >= 1 && ndim <= 3, "ndim must be 1, 2 or 3");
    IB200_REQUIRE(batch >= 0, "negative batch");
    ib200_fft_plan_s *p = new (std::nothrow) ib200_fft_plan_s();
    if (!p) { set_error("out of host memory"); return IB200_E_NOMEM; }
    int rc = fft_plan_init(&p->d, ndim, dims, batch);
    if (rc) { delete p; return rc; }
    *plan = p;
    return 0;
}

int ib200_fft_plan_destroy(ib200_fft_plan plan) {
    if (!plan) return 0;
    for (int a = 0; a < 3; ++a)
        if (plan->d.ax[a].tw_dev) cudaFree(plan->d.ax[a].tw_dev);
    delete plan;
    return 0;
}

int ib200_fft_plan_describe(ib200_fft_plan plan, int axis, int *radices, int max) {
    IB200_REQUIRE(plan && axis >= 0 && axis < plan->d.ndim, "bad plan/axis");
    const FftStages &st = plan->d.ax[axis].st;
    if (plan->d.ax[axis].n <= 1) return 0;
    for (int i = 0; i < st.nst && i < max; ++i) radices[i] = st.radix[i];
    return st.nst;
}

int ib200_fft_exec(ib200_fft_plan plan, void *stream, void *y, const void *x, int direction) {
    IB200_RANGE("ib200_fft_exec");
    IB200_REQUIRE(plan, "null plan");
    return exec_impl(&plan->d, as_stream(stream), (c64 *)y, (const c64 *)x, direction, nullptr, 0, nullptr, 0);
}

int ib200_fft_exec_diag(ib200_fft_plan plan, void *stream, void *y, const void *x, int direction, const void *d_in,
                        int conj_in, const void *d_out, int conj_out) {
    IB200_REQUIRE(plan, "null plan");
    return exec_impl(&plan->d, as_stream(stream), (c64 *)y, (const c64 *)x, direction, (const c64 *)d_in, conj_in,
                     (const c64 *)d_out, conj_out);
}

/* ---- fused SENSE transforms (see include/indigo_b200.h) ---------------------------------------- */
struct ib200_sense_plan_s {
    ib200_fft_plan fft;
    int64_t N[3], oN[3], off[3];
    int64_t C;
    const int32_t *win = nullptr;          // k-space support windows of the z passes (ib200_sense_plan_set_support)
};

// does the z pass of this plan run on the persistent packed kernel (the only one that honours windows)?
static bool sense_z_pass_is_persistent(const ib200_sense_plan_s *p) {
    if (!pk_enabled() || getenv("IB200_FFT_NOPKP") || getenv("IB200_FFT_IL_GENERIC")) return false;
    const AxisPlan &ax = p->fft->d.ax[2];
    const int64_t sz = p->oN[0] * p->C * p->oN[1];
    if (sz % kSpecL || sz >= (1LL << 32) || ((sz * p->oN[2]) & 1)) return false;
    FftKernelArgs k;
    k.n = ax.n; k.st = ax.st;
    bool ok = false;
#define IB200_PKP_OK(n, r0, r1, r2)                                                                         \
    if (fft_spec_matches(k, n, r0, r1, r2))                                                                 \
        ok = pkp_mid_pairs(n, r1, r2, kPkThreads) <= 16 &&                                                  \
             (int64_t)(pk_buf_floats(n) * sizeof(float) + (size_t)n * kSpecL * sizeof(c64) + (size_t)n * sizeof(c64)) <= smem_optin();
    IB200_FFT_SPEC_LIST(IB200_PKP_OK)
#undef IB200_PKP_OK
    return ok;
}

static int sense_strided_pass(ib200_sense_plan_s *p, cudaStream_t s, c64 *grid, int axis, bool inverse, bool first,
                              bool last) {
    if (axis == 2 && p->oN[2] <= kTinyAxis) {
        const int64_t plane = p->oN[0] * p->C * p->oN[1];
        const int w0 = (int)p->off[2], w1 = (int)(p->off[2] + p->N[2]);
        int64_t blocks = ceil_div(plane, 256 * 4);
        const int64_t cap = (int64_t)sm_count() * 16;
        if (blocks > cap) blocks = cap;
        if (inverse) sense_tiny_z_kernel<true><<<(unsigned)blocks, 256, 0, s>>>(grid, plane, (int)p->oN[2], w0, w1);
        else         sense_tiny_z_kernel<false><<<(unsigned)blocks, 256, 0, s>>>(grid, plane, (int)p->oN[2], w0, w1);
        IB200_LAUNCH_CHECK();
        return 0;
    }
    // axis 1: lines are the (x, c) pairs of one y row, one slab per z of the image window;
    // axis 2: lines are all (y, x, c) triples, a single slab.
    const FftPlanData &pl = p->fft->d;
    const AxisPlan &ax = pl.ax[axis];
    const int64_t sy = p->oN[0] * p->C, sz = sy * p->oN[1];
    FftKernelArgs k;
    k.tw = ax.tw_dev; k.din = k.dout = nullptr; k.conj_in = k.conj_out = 0;
    k.plane = 0;
    k.n = ax.n; k.L = kSpecL; k.log2L = 4;
    k.swap_in = (inverse && first) ? 1 : 0; k.swap_out = (inverse && last) ? 1 : 0;
    k.load_first = 0; k.store_last = 0;
    k.st = ax.st;
    const int w0 = (int)p->off[axis], w1 = (int)(p->off[axis] + p->N[axis]);
    if (!inverse) { k.in0 = w0; k.in1 = w1; k.out0 = 0; k.out1 = ax.n; }
    else          { k.in0 = 0; k.in1 = ax.n; k.out0 = w0; k.out1 = w1; }
    c64 *base = grid;
    if (axis == 1) {
        k.inner = sy; k.outer = p->N[2]; k.outer_stride = sz;
        base = grid + p->off[2] * sz;
    } else {
        k.inner = sz; k.outer = 1; k.outer_stride = sz * p->oN[2];
    }
    k.x = base; k.y = base;
    if (k.inner % kSpecL == 0 && k.inner < (1LL << 32) && !(k.swap_in && k.swap_out) && getenv("IB200_FFT_IL_GENERIC") == nullptr) {
        IlPassArgs a;
        a.x = base; a.tw = ax.tw_dev; a.inner = k.inner; a.outer = k.outer; a.outer_stride = k.outer_stride;
        a.pstride = (unsigned)k.inner; a.in0 = k.in0; a.in1 = k.in1; a.out0 = k.out0; a.out1 = k.out1;
        if (axis == 2 && p->win) { a.win = p->win; a.win_mode = inverse ? 2 : 1; a.win_div = (int)p->C; }
        int r = try_pk_pass(s, a, ax.n, ax.st, k.swap_in != 0, k.swap_out != 0);
        if (r == 1) return 0;
        if (axis == 2 && p->win && r == 0) { set_error("support windows set but the persistent z pass is unavailable"); return IB200_E_UNSUPPORTED; }
        if (r != 0) return r > 1000 ? r - 1000 : r;
        r = try_il_pass(s, a, ax.n, ax.st, k.swap_in != 0, k.swap_out != 0);
        if (r == 1) return 0;
        if (r != 0) return r > 1000 ? r - 1000 : r;
    }
    const int rc = try_spec(s, false, k);
    if (rc == 1) return 0;
    if (rc == 0) { set_error("fused SENSE passes need a grid extent with a specialised FFT (axis %d: %d)", axis, ax.n); return IB200_E_UNSUPPORTED; }
    return rc > 1000 ? rc - 1000 : rc;
}

int ib200_sense_plan_create(ib200_sense_plan *plan, const int64_t N[3], const int64_t oN[3], int64_t ncoils) {
    IB200_REQUIRE(plan && N && oN, "null pointer");
    IB200_REQUIRE(ncoils >= 1, "need at least one coil");
    for (int d = 0; d < 3; ++d) IB200_REQUIRE(N[d] >= 1 && oN[d] >= N[d], "grid must be at least as large as the image");
    IB200_REQUIRE(oN[0] * ncoils >= kSpecL, "grid row too short");
    ib200_sense_plan_s *p = new (std::nothrow) ib200_sense_plan_s();
    if (!p) { set_error("out of host memory"); return IB200_E_NOMEM; }
    int rc = ib200_fft_plan_create(&p->fft, 3, oN, ncoils);
    if (rc) { delete p; return rc; }
    for (int d = 0; d < 3; ++d) {
        p->N[d] = N[d]; p->oN[d] = oN[d];
        p->off[d] = oN[d] / 2 - N[d] / 2;                       // Zpad 'center': oN//2 + ceil(-N/2), backend.py:379-381
        FftKernelArgs k; k.n = (int)oN[d]; k.st = p->fft->d.ax[d].st;
        bool ok = d == 2 && oN[d] <= kTinyAxis;                 // tiny z axis: direct pass (sense_tiny_z_kernel)
#define IB200_SENSE_OK(n, r0, r1, r2) ok = ok || fft_spec_matches(k, n, r0, r1, r2);
        IB200_FFT_SPEC_LIST(IB200_SENSE_OK)
#undef IB200_SENSE_OK
        if (!ok) {
            set_error("fused SENSE passes: grid extent %lld has no specialised FFT", (long long)oN[d]);
            ib200_fft_plan_destroy(p->fft); delete p;
            return IB200_E_UNSUPPORTED;
        }
    }
    p->C = ncoils;
    *plan = p;
    return 0;
}

int ib200_sense_plan_set_support(ib200_sense_plan plan, const int32_t *win, int block_x) {
    IB200_REQUIRE(plan, "null plan");
    if (!win) { plan->win = nullptr; return 0; }
    IB200_REQUIRE(block_x >= 1, "bad block extent");
    // all 16 lines of a tile must belong to grid points of one block
    const int64_t C = plan->C;
    bool ok = (C % kSpecL == 0) || (kSpecL % C == 0 && (block_x * C) % kSpecL == 0 && plan->oN[0] % block_x == 0);
    if ((uintptr_t)win & 7) ok = false;
    if (!ok || !sense_z_pass_is_persistent(plan)) {
        set_error("support windows need the persistent packed z pass and tiles that do not straddle blocks");
        return IB200_E_UNSUPPORTED;
    }
    plan->win = win;
    return 0;
}

int ib200_sense_plan_destroy(ib200_sense_plan plan) {
    if (!plan) return 0;
    ib200_fft_plan_destroy(plan->fft);
    delete plan;
    return 0;
}

static void sense_args(ib200_sense_plan_s *p, SenseFftArgs *a) {
    a->N0 = (int)p->N[0]; a->N1 = (int)p->N[1]; a->N2 = (int)p->N[2];
    a->n0 = (int)p->oN[0]; a->n1 = (int)p->oN[1]; a->n2 = (int)p->oN[2];
    a->off0 = (int)p->off[0]; a->off1 = (int)p->off[1]; a->off2 = (int)p->off[2];
    a->C = (int)p->C;
    a->tw = p->fft->d.ax[0].tw_dev;
    a->img = nullptr; a->img_out = nullptr; a->pf = nullptr; a->grid = nullptr;
    a->alpha = mk(1.f, 0.f); a->beta = mk(0.f, 0.f); a->beta_zero = 1;
}

int ib200_sense_expand_fft(ib200_sense_plan plan, void *stream, void *grid_il, const void *img, const void *pf) {
    IB200_RANGE("ib200_sense_expand_fft");
    IB200_REQUIRE(plan && grid_il && img && pf, "null pointer");
    int rc = ensure_device_state(&plan->fft->d);
    if (rc) return rc;
    cudaStream_t s = as_stream(stream);
    SenseFftArgs a;
    sense_args(plan, &a);
    a.img = (const c64 *)img; a.pf = (const c64 *)pf; a.grid = (c64 *)grid_il;
    rc = run_sense_x(s, false, a, plan->fft->d.ax[0].st);
    if (rc) return rc;
    rc = sense_strided_pass(plan, s, (c64 *)grid_il, 1, false, false, false);
    if (rc) return rc;
    return sense_strided_pass(plan, s, (c64 *)grid_il, 2, false, false, true);
}

int ib200_sense_ifft_combine(ib200_sense_plan plan, void *stream, void *img_out, void *grid_il, const void *pf,
                             float ar, float ai, float br, float bi) {
    IB200_RANGE("ib200_sense_ifft_combine");
    IB200_REQUIRE(plan && grid_il && img_out && pf, "null pointer");
    int rc = ensure_device_state(&plan->fft->d);
    if (rc) return rc;
    cudaStream_t s = as_stream(stream);
    rc = sense_strided_pass(plan, s, (c64 *)grid_il, 2, true, true, false);
    if (rc) return rc;
    rc = sense_strided_pass(plan, s, (c64 *)grid_il, 1, true, false, false);
    if (rc) return rc;
    SenseFftArgs a;
    sense_args(plan, &a);
    a.img_out = (c64 *)img_out; a.pf = (const c64 *)pf; a.grid = (c64 *)grid_il;
    a.alpha = mk(ar, ai); a.beta = mk(br, bi); a.beta_zero = (br == 0.f && bi == 0.f) ? 1 : 0;
    return run_sense_x(s, true, a, plan->fft->d.ax[0].st);
}

/* One pass of the two fused transforms on its own (same kernels, same arguments as inside
 * ib200_sense_expand_fft / ib200_sense_ifft_combine), so that a caller can bracket every kernel with events:
 * which = 0 expand + x pass, 1 forward y, 2 forward z, 3 inverse z, 4 inverse y, 5 x pass + combine. */
int ib200_sense_pass(ib200_sense_plan plan, void *stream, int which, void *grid_il, const void *img, void *img_out,
                     const void *pf, float ar, float ai, float br, float bi) {
    IB200_RANGE("ib200_sense_pass");
    IB200_REQUIRE(plan && grid_il, "null pointer");
    IB200_REQUIRE(which >= 0 && which <= 5, "pass index out of range");
    int rc = ensure_device_state(&plan->fft->d);
    if (rc) return rc;
    cudaStream_t s = as_stream(stream);
    if (which == 0 || which == 5) {
        SenseFftArgs a;
        sense_args(plan, &a);
        a.pf = (const c64 *)pf; a.grid = (c64 *)grid_il;
        IB200_REQUIRE(pf && (which == 0 ? img != nullptr : img_out != nullptr), "null pointer");
        if (which == 0) { a.img = (const c64 *)img; return run_sense_x(s, false, a, plan->fft->d.ax[0].st); }
        a.img_out = (c64 *)img_out;
        a.alpha = mk(ar, ai); a.beta = mk(br, bi); a.beta_zero = (br == 0.f && bi == 0.f) ? 1 : 0;
        return run_sense_x(s, true, a, plan->fft->d.ax[0].st);
    }
    const bool inverse = which >= 3;
    const int axis = (which == 1 || which == 4) ? 1 : 2;
    return sense_strided_pass(plan, s, (c64 *)grid_il, axis, inverse, inverse && axis == 2, !inverse && axis == 2);
}

/* Convolution pass of the Toeplitz normal operator on the last transformed axis (z, or y when oN[2] == 1): the
 * forward transform of the input window, times kernel, then the first inverse pass; see include/indigo_b200.h. */
int ib200_sense_toeplitz_pass(ib200_sense_plan plan, void *stream, void *grid_il, const float *kernel) {
    IB200_RANGE("ib200_sense_toeplitz_pass");
    IB200_REQUIRE(plan && grid_il && kernel, "null pointer");
    IB200_REQUIRE(((uintptr_t)grid_il & 15) == 0, "grid must be 16-byte aligned");
    IB200_REQUIRE(plan->win == nullptr, "the Toeplitz pass takes no support windows");
    int rc = ensure_device_state(&plan->fft->d);
    if (rc) return rc;
    const int axis = plan->oN[2] > 1 ? 2 : 1;
    IB200_REQUIRE(axis == 2 || plan->N[2] == 1, "2-D plans need a one-plane image");
    const AxisPlan &ax = plan->fft->d.ax[axis];
    const int64_t sy = plan->oN[0] * plan->C, sz = sy * plan->oN[1];
    IlPassArgs a;
    a.x = (c64 *)grid_il; a.tw = ax.tw_dev;
    a.inner = axis == 2 ? sz : sy; a.outer = 1; a.outer_stride = a.inner * plan->oN[axis];
    IB200_REQUIRE(a.inner % kSpecL == 0 && a.inner < (1LL << 32), "Toeplitz pass: grid slab must be a multiple of 16 lines");
    a.pstride = (unsigned)a.inner;
    a.in0 = a.out0 = (int)plan->off[axis];
    a.in1 = a.out1 = (int)(plan->off[axis] + plan->N[axis]);
    return run_pkt_pass(as_stream(stream), a, ax.n, ax.st, kernel, a.inner / plan->C, (int)plan->C);
}

}  // extern "C"
