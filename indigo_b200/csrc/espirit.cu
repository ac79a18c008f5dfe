// ESPIRiT coil sensitivity estimation (indigo_b200/espirit.py; DESIGN.md section 12, tests/espirit_ref.py).
//
// espirit_gram_kernel   G = A^H A of the calibration matrix A (one row per kernel position s inside the calibration
//                       region, one column per (coil c, tap p)), straight from the calibration k-space: A[s, (c, p)] =
//                       X_c(s + p) is gathered into shared memory stage by stage and never stored.  A CTA computes one
//                       64 x 64 tile of the upper triangle and writes it and its conjugate mirror.
// espirit_lag_pass_kernel  one axis of the separable evaluation of M(x) = sum_delta P(delta) e^{+2 pi i delta.(x-N/2)/N}:
//                       out[o][x][i] = sum_j in[o][j][i] tw[x][j].
// espirit_maps_kernel   per image line (y, z): the line's lag matrices P(delta_0) (delta_1, delta_2 already summed) in
//                       shared memory; per voxel a group of CP lanes (one row of M(x) per lane, in registers) runs the
//                       power iteration, phase-normalises to coil 0, crops and stores the map and the eigenvalue.
// Every output has one writer and every sum a fixed order: results are bit-identical from run to run.
#include <algorithm>

#include "common.cuh"

namespace ib200 {

static const int kGramTile = 64;          // G tile (rows and columns)
static const int kGramStage = 16;         // calibration rows per shared-memory stage
static const int kGramThreads = 256;      // 16 x 16 threads, 4 x 4 outputs each
static const int kMapsThreads = 256;

struct GramArgs {
    const c64 *calib;
    c64 *G;
    int w0, w1;                 // calibration extents of axes 0 and 1 (axis 2 via the coil stride)
    int64_t wvol;               // w0 * w1 * w2
    int k0, k1, kD;             // taps of axes 0, 1 and in all
    int r0, r1;                 // kernel positions along axes 0 and 1
    int64_t R;                  // kernel positions in all (rows of A)
    int n;                      // C * kD (columns of A)
    int nt;                     // tiles per side
};

__global__ void __launch_bounds__(kGramThreads) espirit_gram_kernel(const GramArgs a) {
    __shared__ c64 sa[kGramStage][kGramTile], sb[kGramStage][kGramTile];
    __shared__ int64_t offa[kGramTile], offb[kGramTile];
    // upper-triangle tile (bi <= bj) of this CTA
    int t = blockIdx.x, bi = 0;
    while (t >= a.nt - bi) { t -= a.nt - bi; ++bi; }
    const int bj = bi + t;
    const int i0 = bi * kGramTile, j0 = bj * kGramTile;
    if (threadIdx.x < 2 * kGramTile) {
        const int l = threadIdx.x & (kGramTile - 1);
        const int col = (threadIdx.x < kGramTile ? i0 : j0) + l;
        int64_t off = -1;
        if (col < a.n) {
            const int c = col / a.kD, p = col - c * a.kD;
            const int p0 = p % a.k0, p1 = (p / a.k0) % a.k1, p2 = p / (a.k0 * a.k1);
            off = p0 + (int64_t)a.w0 * (p1 + (int64_t)a.w1 * p2) + a.wvol * c;
        }
        (threadIdx.x < kGramTile ? offa : offb)[l] = off;
    }
    // thread (tx, ty) owns rows i0 + ty + 16 u and columns j0 + tx + 16 v: neighbouring lanes read neighbouring
    // shared-memory words
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    c64 acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = mk(0.f, 0.f);
    for (int64_t s0 = 0; s0 < a.R; s0 += kGramStage) {
        __syncthreads();
        for (int e = threadIdx.x; e < 2 * kGramStage * kGramTile; e += kGramThreads) {
            const int which = e / (kGramStage * kGramTile), r = e - which * (kGramStage * kGramTile);
            const int sl = r / kGramTile, l = r - sl * kGramTile;
            const int64_t s = s0 + sl, off = which ? offb[l] : offa[l];
            c64 v = mk(0.f, 0.f);
            if (s < a.R && off >= 0) {
                const int64_t q = s / a.r0;
                const int64_t s_0 = s - q * a.r0, s_1 = q % a.r1, s_2 = q / a.r1;
                v = __ldg(a.calib + off + s_0 + (int64_t)a.w0 * (s_1 + (int64_t)a.w1 * s_2));
            }
            (which ? sb : sa)[sl][l] = v;
        }
        __syncthreads();
        // one stage summed on its own, then added: partial sums of 16 rows keep the fp32 error of long sums small
        c64 part[4][4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int v = 0; v < 4; ++v) part[u][v] = mk(0.f, 0.f);
#pragma unroll
        for (int sl = 0; sl < kGramStage; ++sl) {
            c64 av[4], bv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) { av[u] = sa[sl][ty + 16 * u]; bv[u] = sb[sl][tx + 16 * u]; }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int v = 0; v < 4; ++v) part[u][v] = cfmac(av[u], bv[v], part[u][v]);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int v = 0; v < 4; ++v) acc[u][v] = cadd(acc[u][v], part[u][v]);
    }
    const int64_t n = a.n;
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const int i = i0 + ty + 16 * u, j = j0 + tx + 16 * v;
            if (i >= a.n || j >= a.n || i > j) continue;
            if (i == j) {
                a.G[i + n * i] = mk(acc[u][v].x, 0.f);
            } else {
                a.G[i + n * j] = acc[u][v];
                a.G[j + n * i] = cconj(acc[u][v]);
            }
        }
}

__global__ void espirit_lag_pass_kernel(const c64 *__restrict__ in, c64 *__restrict__ out, const c64 *__restrict__ tw,
                                        int64_t outer, int L, int N, int64_t inner) {
    const int64_t total = outer * N * inner;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t t = idx / inner, i = idx - t * inner;
        const int64_t o = t / N;
        const int x = (int)(t - o * N);
        const c64 *src = in + o * L * inner + i;
        const c64 *w = tw + (int64_t)x * L;
        c64 acc = mk(0.f, 0.f);
        for (int j = 0; j < L; ++j) acc = cfma(__ldg(src + j * inner), __ldg(w + j), acc);
        out[idx] = acc;
    }
}

struct MapsArgs {
    const c64 *coef;            // [z][y][j0][c'][c]
    const c64 *tw0;             // [x][j0]
    c64 *maps;                  // (nvox, C) column-major
    float *eig;                 // nvox
    int N0;
    int64_t lines, nvox;
    int L0, C, iters;
    float crop;
};

template <int CP>
__global__ void __launch_bounds__(kMapsThreads, 2) espirit_maps_kernel(const MapsArgs a) {
    extern __shared__ float4 smem_f4[];
    const int CC = a.C * a.C;
    c64 *q = reinterpret_cast<c64 *>(smem_f4);                           // L0 * C * C
    c64 *vs = q + ((a.L0 * CC + 1) & ~1);                                // kMapsThreads, 16-byte aligned
    const int64_t line = blockIdx.x;
    {
        const c64 *src = a.coef + line * (int64_t)(a.L0 * CC);
        for (int e = threadIdx.x; e < a.L0 * CC; e += kMapsThreads) q[e] = __ldg(src + e);
    }
    __syncthreads();
    const int r = threadIdx.x % CP, grp = threadIdx.x / CP;
    const int groups = kMapsThreads / CP;
    c64 *vg = vs + grp * CP;
    const bool row = r < a.C;
    for (int base = 0; base < a.N0; base += groups) {                   // uniform over the CTA: shuffles stay full-warp
        const int x = base + grp;
        const int xs = x < a.N0 ? x : a.N0 - 1;
        // row r of M(x)
        c64 m[CP];
#pragma unroll
        for (int c = 0; c < CP; ++c) m[c] = mk(0.f, 0.f);
        if (row) {
            for (int j = 0; j < a.L0; ++j) {
                const c64 w = __ldg(a.tw0 + (int64_t)xs * a.L0 + j);
                const c64 *qj = q + j * CC + r;
#pragma unroll
                for (int c = 0; c < CP; ++c)
                    if (c < a.C) m[c] = cfma(qj[c * a.C], w, m[c]);
            }
        }
        c64 v = mk(row ? 1.f : 0.f, 0.f);
        float nrm = 0.f;
        for (int it = 0; it < a.iters; ++it) {
            __syncwarp();
            vg[r] = v;
            __syncwarp();
            c64 w = mk(0.f, 0.f);
#pragma unroll
            for (int c = 0; c < CP; c += 2) {
                if constexpr (CP == 1) {
                    w = cfma(m[0], vg[0], w);
                } else {
                    const float4 p = reinterpret_cast<const float4 *>(vg)[c >> 1];
                    w = cfma(m[c], mk(p.x, p.y), w);
                    w = cfma(m[c + 1], mk(p.z, p.w), w);
                }
            }
            float n2 = fmaf(w.x, w.x, w.y * w.y);
#pragma unroll
            for (int o = 1; o < CP; o <<= 1) n2 += __shfl_xor_sync(0xffffffffu, n2, o);
            nrm = sqrtf(n2);
            v = n2 > 0.f ? mk(w.x / nrm, w.y / nrm) : mk(0.f, 0.f);
        }
        // phase of coil 0 real and non-negative (unchanged where coil 0 is 0); zero where eig <= crop
        const int lane0 = (threadIdx.x & 31) & ~(CP - 1);
        const c64 v0 = mk(__shfl_sync(0xffffffffu, v.x, lane0), __shfl_sync(0xffffffffu, v.y, lane0));
        const float a0 = sqrtf(fmaf(v0.x, v0.x, v0.y * v0.y));
        if (a0 > 0.f) v = cmulc(v, mk(v0.x / a0, v0.y / a0));
        if (!(nrm > a.crop)) v = mk(0.f, 0.f);
        if (x < a.N0) {
            const int64_t vox = x + line * a.N0;
            if (row) a.maps[vox + a.nvox * r] = v;
            if (r == 0) a.eig[vox] = nrm;
        }
    }
}

template <int CP>
static int launch_maps(cudaStream_t s, const MapsArgs &a, size_t smem) {
    if (smem > 48 * 1024)
        IB200_TRY(cudaFuncSetAttribute(espirit_maps_kernel<CP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    espirit_maps_kernel<CP><<<(unsigned)a.lines, kMapsThreads, smem, s>>>(a);
    IB200_LAUNCH_CHECK();
    return 0;
}

}  // namespace ib200

using namespace ib200;

extern "C" {

int ib200_espirit_calib_gram(void *stream, const int64_t w[3], const int64_t k[3], int ncoils, const void *calib,
                             void *gram) {
    IB200_RANGE("ib200_espirit_calib_gram");
    IB200_REQUIRE(w && k && calib && gram, "null pointer");
    IB200_REQUIRE(ncoils >= 1, "need at least one coil");
    for (int d = 0; d < 3; ++d) IB200_REQUIRE(k[d] >= 1 && k[d] <= w[d], "kernel must fit the calibration region");
    const int64_t kD = k[0] * k[1] * k[2], n = kD * ncoils;
    IB200_REQUIRE(n < (1LL << 20), "calibration matrix too wide");
    GramArgs a;
    a.calib = (const c64 *)calib;
    a.G = (c64 *)gram;
    a.w0 = (int)w[0]; a.w1 = (int)w[1];
    a.wvol = w[0] * w[1] * w[2];
    a.k0 = (int)k[0]; a.k1 = (int)k[1]; a.kD = (int)kD;
    a.r0 = (int)(w[0] - k[0] + 1); a.r1 = (int)(w[1] - k[1] + 1);
    a.R = (int64_t)a.r0 * a.r1 * (w[2] - k[2] + 1);
    a.n = (int)n;
    a.nt = (int)ceil_div(n, kGramTile);
    const int64_t tiles = (int64_t)a.nt * (a.nt + 1) / 2;
    espirit_gram_kernel<<<(unsigned)tiles, kGramThreads, 0, as_stream(stream)>>>(a);
    IB200_LAUNCH_CHECK();
    return 0;
}

int ib200_espirit_lag_pass(void *stream, int64_t outer, int lags, int n, int64_t inner, const void *twiddle,
                           const void *in, void *out) {
    IB200_RANGE("ib200_espirit_lag_pass");
    IB200_REQUIRE(twiddle && in && out, "null pointer");
    IB200_REQUIRE(outer >= 1 && lags >= 1 && n >= 1 && inner >= 1, "bad extents");
    const int64_t total = outer * n * inner;
    const int threads = 256;
    const int64_t blocks = std::min<int64_t>(ceil_div(total, threads), (int64_t)sm_count() * 16);
    espirit_lag_pass_kernel<<<(unsigned)blocks, threads, 0, as_stream(stream)>>>(
        (const c64 *)in, (c64 *)out, (const c64 *)twiddle, outer, lags, n, inner);
    IB200_LAUNCH_CHECK();
    return 0;
}

int ib200_espirit_maps(void *stream, const int64_t N[3], int lags0, int ncoils, int max_iter, float crop,
                       const void *twiddle0, const void *coef, void *maps, float *eig) {
    IB200_RANGE("ib200_espirit_maps");
    IB200_REQUIRE(N && twiddle0 && coef && maps && eig, "null pointer");
    IB200_REQUIRE(N[0] >= 1 && N[1] >= 1 && N[2] >= 1, "bad image shape");
    IB200_REQUIRE(ncoils >= 1 && ncoils <= 32, "1 to 32 coils");
    IB200_REQUIRE(lags0 >= 1 && max_iter >= 1, "bad lag count or iteration count");
    MapsArgs a;
    a.coef = (const c64 *)coef;
    a.tw0 = (const c64 *)twiddle0;
    a.maps = (c64 *)maps;
    a.eig = eig;
    a.N0 = (int)N[0];
    a.lines = N[1] * N[2];
    a.nvox = N[0] * a.lines;
    a.L0 = lags0;
    a.C = ncoils;
    a.iters = max_iter;
    a.crop = crop;
    IB200_REQUIRE(a.lines < (1LL << 31), "too many image lines");
    const size_t smem = (size_t)((lags0 * ncoils * ncoils + 1) & ~1) * sizeof(c64) + kMapsThreads * sizeof(c64);
    IB200_REQUIRE((int64_t)smem <= smem_optin(), "espirit maps: the lag matrices of one line do not fit shared memory");
    cudaStream_t s = as_stream(stream);
    if (ncoils <= 1) return launch_maps<1>(s, a, smem);
    if (ncoils <= 2) return launch_maps<2>(s, a, smem);
    if (ncoils <= 4) return launch_maps<4>(s, a, smem);
    if (ncoils <= 8) return launch_maps<8>(s, a, smem);
    if (ncoils <= 16) return launch_maps<16>(s, a, smem);
    return launch_maps<32>(s, a, smem);
}

}  // extern "C"
