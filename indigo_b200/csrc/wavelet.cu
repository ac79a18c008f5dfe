// Orthonormal separable wavelet transform and the FISTA prox step of l1-wavelet reconstruction
// (indigo_b200/wavelet.py; the transform is defined in DESIGN.md section 11 and restated in tests/wavelet_ref.py).
//
// One level on one axis of even length n, periodized, low-pass h and high-pass g[m] = (-1)^m h[Lf-1-m]:
//     a[k] = sum_m h[m] x[(2k+m) mod n] -> position k,   d[k] = sum_m g[m] x[(2k+m) mod n] -> position n/2 + k.
// Synthesis is the transpose: x[p] = sum over m of the parity of p of h[m] a[k] + g[m] d[k], k = ((p-m) mod n)/2.
// Level j acts on the sub-box of extent N_d / 2^(j-1) on each transformed axis (N_d > 1): an x pass, a y pass and
// (3-D) a z pass, in place; synthesis runs the passes in reverse order.
//
// wavelet_pass_kernel: a CTA loads a tile of whole lines of the sub-box into shared memory, then every thread
// computes output points of the tile from shared memory and stores them.  x lines are contiguous; a y or z tile is
// a run of consecutive x positions of `tx` lines, so that loads and stores move runs of tx complex values.  Every
// output point has exactly one writer and every sum a fixed order, so results are bit-identical from run to run.
// Options of a pass, all applied in the load or the store:
//   pre      (first analysis pass of a prox step)  loads u = src - step (g - b) instead of src;
//   thresh   (last axis pass of each analysis level) soft-thresholds the detail points of the level on store;
//   ab       (last pass of a plain transform) stores alpha v + beta dst, never reading dst when beta == 0;
//   fista    (last synthesis pass of a prox step)  dst is x: stores x_k, reads x_{k-1} from the same place and
//            stores z = x_k + mom (x_k - x_{k-1}) with mom = momentum[*counter]; optionally per-CTA partial sums of
//            |x_k - x_{k-1}|^2 and |x_k|^2, which wavelet_finish_kernel folds in a fixed order.
#include <algorithm>
#include <utility>

#include "common.cuh"

namespace ib200 {

static const int kWvThreads = 256;
static const int kWvTile = 4096;            // complex points per tile (32 KB of shared memory)
static const int kWvMaxTx = 32;             // x positions per y / z tile
static const int kWvMaxLine = 512;          // longest transformed axis
static const int kWvMaxGrid = 4096;         // per-CTA partial slots of the reduction (IB200_WAVELET_STATS)

struct WvFilter {
    float h[8], g[8];
};

struct WvArgs {
    const c64 *src;
    c64 *dst;
    // pre
    const c64 *g, *b;
    float step;
    // thresh
    float thresh;
    int thr;
    // ab
    c64 alpha, beta;
    int ab;
    // fista
    c64 *z;
    const double *mom;
    const int *counter;
    double *partial;
    int fista;
    // geometry: full image, active sub-box, transformed axes
    int N0, N1, N2, n0, n1, n2, tmask;
    WvFilter f;
};

__device__ __forceinline__ double wv_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// tile element e -> global index, shared index and sub-box coordinates
template <int AXIS>
__device__ __forceinline__ bool wv_locate(const WvArgs &a, int n, int tile, int per, int tx, int ntx, int e,
                                          int64_t &gi, int &si, int &p, int &c0, int &c1, int &c2) {
    const int64_t N0 = a.N0, N01 = (int64_t)a.N0 * a.N1;
    if (AXIS == 0) {
        const int l = e / n;
        p = e - l * n;
        const int line = tile * per + l;
        if (line >= a.n1 * a.n2) return false;
        c1 = line % a.n1; c2 = line / a.n1; c0 = p;
        gi = c1 * N0 + c2 * N01 + p;
        si = l * n + p;
    } else {
        const int xi = e % tx;
        p = e / tx;
        const int xt = tile % ntx, o = tile / ntx;
        c0 = xt * tx + xi;
        if (c0 >= a.n0) return false;
        if (AXIS == 1) { c1 = p; c2 = o; } else { c1 = o; c2 = p; }
        gi = c0 + c1 * N0 + c2 * N01;
        si = p * tx + xi;
    }
    return true;
}

template <int LF, int AXIS, bool INV>
__global__ void __launch_bounds__(kWvThreads) wavelet_pass_kernel(const WvArgs a) {
    __shared__ c64 s[kWvTile];
    __shared__ double red[2][kWvThreads / 32];
    const int n = AXIS == 0 ? a.n0 : AXIS == 1 ? a.n1 : a.n2;
    const int half = n >> 1;
    int per = 0, tx = 1, ntx = 1, ntiles;
    if (AXIS == 0) {
        per = kWvTile / n;
        ntiles = (a.n1 * a.n2 + per - 1) / per;
    } else {
        tx = min(kWvMaxTx, kWvTile / n);
        ntx = (a.n0 + tx - 1) / tx;
        ntiles = ntx * (AXIS == 1 ? a.n2 : a.n1);
    }
    const int cnt = AXIS == 0 ? per * n : tx * n;
    // the step of the tile: neighbouring points along the axis in shared memory
    const int sstep = AXIS == 0 ? 1 : tx;
    const float mom = a.fista ? (float)a.mom[*a.counter] : 0.f;
    double accd = 0.0, accn = 0.0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        __syncthreads();
        for (int e = threadIdx.x; e < cnt; e += kWvThreads) {
            int64_t gi; int si, p, c0, c1, c2;
            if (!wv_locate<AXIS>(a, n, tile, per, tx, ntx, e, gi, si, p, c0, c1, c2)) continue;
            c64 v = a.src[gi];
            if (a.g) {
                const c64 gv = __ldg(a.g + gi), bv = __ldg(a.b + gi);
                v = mk(fmaf(-a.step, gv.x - bv.x, v.x), fmaf(-a.step, gv.y - bv.y, v.y));
            }
            s[si] = v;
        }
        __syncthreads();
        for (int e = threadIdx.x; e < cnt; e += kWvThreads) {
            int64_t gi; int si, q, c0, c1, c2;
            if (!wv_locate<AXIS>(a, n, tile, per, tx, ntx, e, gi, si, q, c0, c1, c2)) continue;
            const c64 *line = s + (si - q * sstep);
            c64 v = mk(0.f, 0.f);
            if (!INV) {
                const int k = q < half ? q : q - half;
                if (q < half) {
#pragma unroll
                    for (int m = 0; m < LF; ++m) {
                        int p = 2 * k + m;
                        while (p >= n) p -= n;
                        const c64 x = line[p * sstep];
                        v.x = fmaf(a.f.h[m], x.x, v.x); v.y = fmaf(a.f.h[m], x.y, v.y);
                    }
                } else {
#pragma unroll
                    for (int m = 0; m < LF; ++m) {
                        int p = 2 * k + m;
                        while (p >= n) p -= n;
                        const c64 x = line[p * sstep];
                        v.x = fmaf(a.f.g[m], x.x, v.x); v.y = fmaf(a.f.g[m], x.y, v.y);
                    }
                }
            } else {
                // m runs over the parity of q: (q - m) is even, k = ((q - m) mod n) / 2
#define IB200_WV_SYN(M0)                                                                 \
    _Pragma("unroll") for (int j = 0; j < LF / 2; ++j) {                                 \
        const int m = 2 * j + (M0);                                                      \
        int t = q - m;                                                                   \
        while (t < 0) t += n;                                                            \
        const int k = t >> 1;                                                            \
        const c64 lo = line[k * sstep], hi = line[(half + k) * sstep];                   \
        v.x = fmaf(a.f.h[m], lo.x, v.x); v.y = fmaf(a.f.h[m], lo.y, v.y);                \
        v.x = fmaf(a.f.g[m], hi.x, v.x); v.y = fmaf(a.f.g[m], hi.y, v.y);                \
    }
                if (q & 1) { IB200_WV_SYN(1) } else { IB200_WV_SYN(0) }
#undef IB200_WV_SYN
            }
            if (a.thr) {
                const bool detail = ((a.tmask & 1) && c0 >= (a.n0 >> 1)) || ((a.tmask & 2) && c1 >= (a.n1 >> 1)) ||
                                    ((a.tmask & 4) && c2 >= (a.n2 >> 1));
                if (detail) {
                    const float r = sqrtf(v.x * v.x + v.y * v.y);
                    const float sc = r > a.thresh ? 1.f - a.thresh / r : 0.f;
                    v = mk(sc * v.x, sc * v.y);
                }
            }
            if (a.fista) {
                const c64 xo = a.dst[gi];
                const c64 dx = mk(v.x - xo.x, v.y - xo.y);
                a.dst[gi] = v;
                a.z[gi] = mk(fmaf(mom, dx.x, v.x), fmaf(mom, dx.y, v.y));
                accd += (double)dx.x * dx.x + (double)dx.y * dx.y;
                accn += (double)v.x * v.x + (double)v.y * v.y;
            } else if (a.ab) {
                c64 r = cmul(a.alpha, v);
                if (a.beta.x != 0.f || a.beta.y != 0.f) r = cfma(a.beta, a.dst[gi], r);
                a.dst[gi] = r;
            } else {
                a.dst[gi] = v;
            }
        }
    }
    if (!a.partial) return;
    accd = wv_warp_sum(accd); accn = wv_warp_sum(accn);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) { red[0][w] = accd; red[1][w] = accn; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double sd = 0.0, sn = 0.0;
        for (int i = 0; i < kWvThreads / 32; ++i) { sd += red[0][i]; sn += red[1][i]; }
        a.partial[2 + 2 * blockIdx.x] = sd;
        a.partial[3 + 2 * blockIdx.x] = sn;
    }
}

// y = alpha w + beta y over n points (beta == 0 never reads y): the store of a multi-level analysis, whose last
// pass covers only the coarse sub-box
__global__ void __launch_bounds__(kWvThreads) wavelet_axpby_kernel(int64_t n, c64 alpha, c64 beta,
                                                                   const c64 *__restrict__ w, c64 *__restrict__ y) {
    const bool rd = beta.x != 0.f || beta.y != 0.f;
    for (int64_t i = (int64_t)blockIdx.x * kWvThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kWvThreads) {
        c64 r = cmul(alpha, w[i]);
        if (rd) r = cfma(beta, y[i], r);
        y[i] = r;
    }
}

// stats[0..1] = the sums of the nblocks partials in index order (when stats != NULL); then *counter += 1
__global__ void __launch_bounds__(kWvThreads) wavelet_finish_kernel(int nblocks, double *stats, int *counter) {
    __shared__ double red[2][kWvThreads];
    if (stats) {
        double sd = 0.0, sn = 0.0;
        for (int i = threadIdx.x; i < nblocks; i += kWvThreads) { sd += stats[2 + 2 * i]; sn += stats[3 + 2 * i]; }
        red[0][threadIdx.x] = sd; red[1][threadIdx.x] = sn;
        __syncthreads();
#pragma unroll
        for (int k = kWvThreads / 2; k > 0; k >>= 1) {
            if ((int)threadIdx.x < k) {
                red[0][threadIdx.x] += red[0][threadIdx.x + k];
                red[1][threadIdx.x] += red[1][threadIdx.x + k];
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) { stats[0] = red[0][0]; stats[1] = red[1][0]; }
    }
    if (threadIdx.x == 0) *counter += 1;
}

struct WvGeom {
    int N[3];
    int tmask;
    int last_axis;   // the last transformed axis (the level's last pass)
};

static int wv_geometry(const int64_t dims[3], int lf, const double *h, int levels, WvGeom &G, WvFilter &F) {
    IB200_REQUIRE(dims && h, "null pointer");
    IB200_REQUIRE(lf == 2 || lf == 8, "filter length must be 2 or 8");
    IB200_REQUIRE(levels >= 1 && levels <= 30, "levels must be at least 1");
    IB200_REQUIRE(dims[0] > 0 && dims[1] > 0 && dims[2] > 0 && dims[0] * dims[1] * dims[2] < (1LL << 31), "bad shape");
    G.tmask = 0;
    G.last_axis = -1;
    for (int d = 0; d < 3; ++d) {
        G.N[d] = (int)dims[d];
        if (dims[d] == 1) continue;
        if (dims[d] > kWvMaxLine) {
            set_error("wavelet transform: axis %d has %lld points, more than the %d the pass supports", d,
                      (long long)dims[d], kWvMaxLine);
            return IB200_E_UNSUPPORTED;
        }
        IB200_REQUIRE(dims[d] % (1LL << levels) == 0, "every transformed axis must be divisible by 2^levels");
        G.tmask |= 1 << d;
        G.last_axis = d;
    }
    IB200_REQUIRE(G.tmask != 0, "no axis to transform");
    for (int m = 0; m < 8; ++m) {
        F.h[m] = m < lf ? (float)h[m] : 0.f;
        F.g[m] = m < lf ? (float)((m & 1 ? -1.0 : 1.0) * h[lf - 1 - m]) : 0.f;
    }
    return 0;
}

static int wv_grid(const WvGeom &G, int axis, const int n[3]) {
    int64_t tiles;
    if (axis == 0) {
        const int per = kWvTile / n[0];
        tiles = ceil_div((int64_t)n[1] * n[2], per);
    } else {
        const int tx = std::min(kWvMaxTx, kWvTile / n[axis]);
        tiles = ceil_div(n[0], tx) * (axis == 1 ? n[2] : n[1]);
    }
    int64_t cap = (int64_t)sm_count() * 8;
    if (cap > kWvMaxGrid) cap = kWvMaxGrid;
    return (int)std::max<int64_t>(1, std::min(tiles, cap));
}

template <int LF>
static void wv_launch_lf(cudaStream_t s, int axis, bool inv, int grid, const WvArgs &a) {
#define IB200_WV_GO(AX, INV) wavelet_pass_kernel<LF, AX, INV><<<grid, kWvThreads, 0, s>>>(a)
    if (!inv) {
        if (axis == 0) IB200_WV_GO(0, false); else if (axis == 1) IB200_WV_GO(1, false); else IB200_WV_GO(2, false);
    } else {
        if (axis == 0) IB200_WV_GO(0, true); else if (axis == 1) IB200_WV_GO(1, true); else IB200_WV_GO(2, true);
    }
#undef IB200_WV_GO
}

// one pass of level `level` on `axis`; returns the grid it ran with
static int wv_pass(cudaStream_t s, const WvGeom &G, int lf, int level, int axis, bool inv, WvArgs a, int *grid_out) {
    int n[3];
    for (int d = 0; d < 3; ++d) n[d] = (G.tmask >> d & 1) ? G.N[d] >> (level - 1) : 1;
    a.N0 = G.N[0]; a.N1 = G.N[1]; a.N2 = G.N[2];
    a.n0 = n[0]; a.n1 = n[1]; a.n2 = n[2];
    a.tmask = G.tmask;
    const int grid = wv_grid(G, axis, n);
    if (lf == 2) wv_launch_lf<2>(s, axis, inv, grid, a); else wv_launch_lf<8>(s, axis, inv, grid, a);
    IB200_LAUNCH_CHECK();
    if (grid_out) *grid_out = grid;
    return 0;
}

// the passes of a transform in execution order: (level, axis)
static int wv_schedule(const WvGeom &G, int levels, bool inv, int (*out)[2]) {
    int cnt = 0;
    for (int j = 1; j <= levels; ++j)
        for (int d = 0; d < 3; ++d)
            if (G.tmask >> d & 1) { out[cnt][0] = j; out[cnt][1] = d; ++cnt; }
    if (inv)
        for (int i = 0; i < cnt / 2; ++i) {
            std::swap(out[i][0], out[cnt - 1 - i][0]);
            std::swap(out[i][1], out[cnt - 1 - i][1]);
        }
    return cnt;
}

}  // namespace ib200

using namespace ib200;

extern "C" {

int ib200_wavelet(void *stream, const int64_t dims[3], int lf, const double *h, int levels, int inverse, float alpha_re,
                  float alpha_im, float beta_re, float beta_im, const void *x, void *y, void *work) {
    IB200_RANGE("ib200_wavelet");
    WvGeom G;
    WvFilter F;
    const int rc = wv_geometry(dims, lf, h, levels, G, F);
    if (rc) return rc;
    IB200_REQUIRE(x && y && work, "null pointer");
    cudaStream_t s = as_stream(stream);
    int sched[3 * 30][2];
    const int np = wv_schedule(G, levels, inverse != 0, sched);
    // With one level every pass covers the whole image.  Otherwise an analysis ends on the coarse sub-box, so it
    // stays in work and one elementwise pass stores y; and a synthesis starts on the coarse sub-box, so the detail
    // bands it reads later come from a copy of x in work.
    const bool last_is_full = inverse != 0 || levels == 1;
    const bool first_is_full = inverse == 0 || levels == 1;
    if (!first_is_full)
        IB200_TRY(cudaMemcpyAsync(work, x, (size_t)(dims[0] * dims[1] * dims[2]) * sizeof(c64), cudaMemcpyDeviceToDevice, s));
    for (int i = 0; i < np; ++i) {
        WvArgs a = {};
        a.f = F;
        a.src = i == 0 && first_is_full ? (const c64 *)x : (const c64 *)work;
        a.dst = (c64 *)work;
        if (i == np - 1 && last_is_full) {
            a.dst = (c64 *)y;
            a.ab = 1;
            a.alpha = mk(alpha_re, alpha_im);
            a.beta = mk(beta_re, beta_im);
        }
        const int r = wv_pass(s, G, lf, sched[i][0], sched[i][1], inverse != 0, a, nullptr);
        if (r) return r;
    }
    if (!last_is_full) {
        const int64_t n = dims[0] * dims[1] * dims[2];
        const int64_t grid = std::min<int64_t>(ceil_div(n, kWvThreads), (int64_t)sm_count() * 8);
        wavelet_axpby_kernel<<<(unsigned)grid, kWvThreads, 0, s>>>(n, mk(alpha_re, alpha_im), mk(beta_re, beta_im),
                                                                   (const c64 *)work, (c64 *)y);
        IB200_LAUNCH_CHECK();
    }
    return 0;
}

int ib200_wavelet_fista_step(void *stream, const int64_t dims[3], int lf, const double *h, int levels, float step,
                             float thresh, const void *g, const void *b, void *z, void *x, void *work,
                             const double *momentum, int *counter, double *stats) {
    IB200_RANGE("ib200_wavelet_fista_step");
    WvGeom G;
    WvFilter F;
    const int rc = wv_geometry(dims, lf, h, levels, G, F);
    if (rc) return rc;
    IB200_REQUIRE(g && b && z && x && work && momentum && counter, "null pointer");
    IB200_REQUIRE(thresh >= 0.f, "negative threshold");
    cudaStream_t s = as_stream(stream);
    int sched[3 * 30][2];
    int np = wv_schedule(G, levels, false, sched);
    for (int i = 0; i < np; ++i) {
        WvArgs a = {};
        a.f = F;
        a.src = i == 0 ? (const c64 *)z : (const c64 *)work;
        a.dst = (c64 *)work;
        if (i == 0) { a.g = (const c64 *)g; a.b = (const c64 *)b; a.step = step; }
        if (sched[i][1] == G.last_axis) { a.thr = 1; a.thresh = thresh; }
        const int r = wv_pass(s, G, lf, sched[i][0], sched[i][1], false, a, nullptr);
        if (r) return r;
    }
    np = wv_schedule(G, levels, true, sched);
    int grid = 0;
    for (int i = 0; i < np; ++i) {
        WvArgs a = {};
        a.f = F;
        a.src = (const c64 *)work;
        a.dst = i == np - 1 ? (c64 *)x : (c64 *)work;
        if (i == np - 1) {
            a.fista = 1; a.z = (c64 *)z; a.mom = momentum; a.counter = counter; a.partial = stats;
        }
        const int r = wv_pass(s, G, lf, sched[i][0], sched[i][1], true, a, i == np - 1 ? &grid : nullptr);
        if (r) return r;
    }
    wavelet_finish_kernel<<<1, kWvThreads, 0, s>>>(grid, stats, counter);
    IB200_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
