// Pipe-Menon density compensation on the matrix-free gridding structures (indigo_b200/sense.py: pipe_menon_dcf).
//
//     w_0 = 1,   w_{k+1} = w_k / (I I^T w_k)
//
// with I the Kaiser-Bessel interpolation matrix on the oversampled grid (oracle/sense.py: interp_matrix).  One
// iteration is a real, single-channel adjoint gridding followed by a real, single-channel forward gridding; the
// complex kernels move a coil line per tap (kb_gather) or C complex coils per entry (kb_blocks_apply), this needs
// one float per grid point and one per sample.
//   ib200_kb_density_spread   g = I^T w on the 4x4x4 tile entries of kbblocks.cu: the same work items, the same
//                             entries, the same fixed-order fold of split blocks.  Every grid point inside the
//                             rowmap is written on every call, nothing else: the grid is zeroed once by the caller.
//   ib200_kb_density_update   per sample q = sum_taps g[tap] wx wy wz from the separable records (4 bytes per tap),
//                             then w <- w / q in the same kernel, so q never goes to memory; optionally the sum of
//                             (q - 1)^2 over the samples, in a fixed summation tree.
// The records carry mod * scale: per-axis factors of +-1 (the fused path factors out the unit constant) and
// scale = 1/sqrt(prod oN) on z.  The signs cancel in I I^T, scale^2 does not: the update multiplies q by
// inv_scale2 = 1/scale^2.  Both kernels are deterministic: every sum has a fixed order and there are no atomics.
#include "kbblocks.cuh"
#include "kb.cuh"

namespace ib200 {

static const int kDcfLanes = 16;                                     // lanes per work item: one x-row of 4 points each
static const int kDcfBatch = 16 + 3 * 16 * kTB;                      // a 4x4x4 batch: ids | wx[4][4] | wy[4][4] | wz[4][4]
static_assert(kDcfBatch == 208, "4x4x4 batch layout");

// lane (y, z) of the work item's block accumulates the four points x = 0..3 of its row over the item's batches
__global__ void __launch_bounds__(256) kb_density_spread_kernel(int nwork, const int4 *__restrict__ work,
                                                                const unsigned char *__restrict__ ent,
                                                                const float *__restrict__ w, float *__restrict__ g,
                                                                const int32_t *__restrict__ rowmap,
                                                                float *__restrict__ scratch) {
    const int idx = (int)((blockIdx.x * blockDim.x + threadIdx.x) / kDcfLanes);
    const int gl = (int)(threadIdx.x % kDcfLanes);
    if (idx >= nwork) return;
    const int y = gl % kTE, z = gl / kTE, rr = z * kTE + y;
    const int4 d = __ldg(work + idx);
    float acc[kTE] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
    for (int b = d.y; b < d.z; ++b) {
        const unsigned char *base = ent + (int64_t)b * kDcfBatch;
        const int4 ids = __ldg(reinterpret_cast<const int4 *>(base));
        const int id[kTB] = {ids.x, ids.y, ids.z, ids.w};
#pragma unroll
        for (int u = 0; u < kTB; ++u) {
            const float wv = __ldg(w + id[u]);
            const float4 wx = __ldg(reinterpret_cast<const float4 *>(base + 16 + 16 * u));
            const float wy = __ldg(reinterpret_cast<const float *>(base + 16 + 16 * kTB) + kTE * u + y);
            const float wz = __ldg(reinterpret_cast<const float *>(base + 16 + 32 * kTB) + kTE * u + z);
            const float r = wv * wy * wz;
            acc[0] = fmaf(r, wx.x, acc[0]); acc[1] = fmaf(r, wx.y, acc[1]);
            acc[2] = fmaf(r, wx.z, acc[2]); acc[3] = fmaf(r, wx.w, acc[3]);
        }
    }
    if (d.w < 0) {
        const int4 rv4 = __ldg(reinterpret_cast<const int4 *>(rowmap + block_row(d.x, rr, kTE, kTE)));
        const int rv[kTE] = {rv4.x, rv4.y, rv4.z, rv4.w};
#pragma unroll
        for (int j = 0; j < kTE; ++j)
            if (rv[j] >= 0) g[rv[j]] = acc[j];
    } else {
        *reinterpret_cast<float4 *>(scratch + (int64_t)d.w * kTV + rr * kTE) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    }
}

// split blocks: thread (split, point) adds the item partial sums of its block in item order
__global__ void __launch_bounds__(256) kb_density_fold_kernel(int nsplit, const int4 *__restrict__ split,
                                                              const float *__restrict__ scratch, float *__restrict__ g,
                                                              const int32_t *__restrict__ rowmap) {
    const int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) / kTV);
    const int p = (int)(threadIdx.x % kTV);
    if (i >= nsplit) return;
    const int4 d = __ldg(split + i);
    float s = 0.f;
    for (int k = 0; k < d.z; ++k) s += __ldcs(scratch + (int64_t)(d.y + k) * kTV + p);
    const int out = __ldg(rowmap + block_row(d.x, p / kTE, kTE, kTE) + p % kTE);
    if (out >= 0) g[out] = s;
}

// one thread per record (records in tile-sorted order: the threads of a warp read neighbouring grid lines, from L1)
__global__ void __launch_bounds__(256) kb_density_update_kernel(int64_t m, const KbRecord *__restrict__ rec,
                                                                const float *__restrict__ g, int n0, int n1, int n2,
                                                                float inv_scale2, float *__restrict__ w,
                                                                double *__restrict__ partial) {
    constexpr unsigned FULL = 0xffffffffu;
    __shared__ double red[256];
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float wx[kKbTaps], wy[kKbTaps], wz[kKbTaps];
    int ix0 = 0, iy0 = 0, iz0 = 0, out = -1, nt = 0;
    if (r < m) {
        const float4 *p = reinterpret_cast<const float4 *>(rec + r);
        const float4 a = __ldcs(p), b = __ldcs(p + 1), c = __ldcs(p + 2), d = __ldcs(p + 3), e = __ldcs(p + 4);
        const int4 h = __ldcs(reinterpret_cast<const int4 *>(p + 5));
        wx[0] = a.x; wx[1] = a.y; wx[2] = a.z; wx[3] = a.w; wx[4] = b.x; wx[5] = b.y;
        wy[0] = b.z; wy[1] = b.w; wy[2] = c.x; wy[3] = c.y; wy[4] = c.z; wy[5] = c.w;
        wz[0] = d.x; wz[1] = d.y; wz[2] = d.z; wz[3] = d.w; wz[4] = e.x; wz[5] = e.y;
        ix0 = __float_as_int(e.z); iy0 = __float_as_int(e.w); iz0 = h.x; out = h.y; nt = h.z;
    } else {
#pragma unroll
        for (int t = 0; t < kKbTaps; ++t) { wx[t] = 0.f; wy[t] = 0.f; wz[t] = 0.f; }
    }
    // trip counts: the maximum over the warp (weights beyond a record's own count are zero, addresses stay in the grid)
    const int nxm = __reduce_max_sync(FULL, nt & 255), nym = __reduce_max_sync(FULL, (nt >> 8) & 255),
              nzm = __reduce_max_sync(FULL, (nt >> 16) & 255);
    int xo[kKbTaps];
    {
        int j = ix0;
#pragma unroll
        for (int t = 0; t < kKbTaps; ++t) { xo[t] = j; if (++j >= n0) j = 0; }
    }
    float q = 0.f;
    int iz = iz0;
#pragma unroll
    for (int k = 0; k < kKbTaps; ++k) {
        if (k < nzm) {
            int iy = iy0;
#pragma unroll
            for (int j = 0; j < kKbTaps; ++j) {
                if (j < nym) {
                    const float *row = g + ((int64_t)iz * n1 + iy) * n0;
                    float t = 0.f;
#pragma unroll
                    for (int i = 0; i < kKbTaps; ++i)
                        if (i < nxm) t = fmaf(wx[i], __ldg(row + xo[i]), t);
                    q = fmaf(wz[k] * wy[j], t, q);
                    if (++iy >= n1) iy = 0;
                }
            }
            if (++iz >= n2) iz = 0;
        }
    }
    q *= inv_scale2;
    double e2 = 0.0;
    if (r < m) {
        const float wv = w[out];
        w[out] = (q > 0.f && isfinite(q)) ? wv / q : 0.f;
        e2 = (double)(q - 1.f) * (double)(q - 1.f);
    }
    if (!partial) return;
    red[threadIdx.x] = e2;
    __syncthreads();
#pragma unroll
    for (int s = 128; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[1 + blockIdx.x] = red[0];
}

// partial[0] = sum of partial[1 .. n]: strided per-thread sums, then a fixed tree
__global__ void __launch_bounds__(256) kb_density_residual_kernel(int64_t n, double *partial) {
    __shared__ double red[256];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 256) s += partial[1 + i];
    red[threadIdx.x] = s;
    __syncthreads();
#pragma unroll
    for (int k = 128; k > 0; k >>= 1) {
        if ((int)threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[0] = red[0];
}

}  // namespace ib200

using namespace ib200;

extern "C" {

int ib200_kb_density_spread(void *stream, int nwork, const int32_t *work, const void *entries, const float *w, float *grid,
                            const int32_t *rowmap, int nsplit, const int32_t *split, float *scratch) {
    IB200_RANGE("ib200_kb_density_spread");
    IB200_REQUIRE(nwork >= 0 && nsplit >= 0, "bad arguments");
    if (nwork == 0) return 0;
    IB200_REQUIRE(work && entries && w && grid && rowmap, "null pointer");
    IB200_REQUIRE(((uintptr_t)entries & 15) == 0 && ((uintptr_t)work & 15) == 0 && ((uintptr_t)rowmap & 15) == 0,
                  "entries, work items and rowmap must be 16-byte aligned");
    IB200_REQUIRE(nsplit == 0 || (split && scratch && ((uintptr_t)scratch & 15) == 0 && ((uintptr_t)split & 15) == 0),
                  "split arrays missing");
    cudaStream_t s = as_stream(stream);
    const int64_t threads = (int64_t)nwork * kDcfLanes;
    IB200_REQUIRE(ceil_div(threads, 256) < (1LL << 31), "too many work items");
    kb_density_spread_kernel<<<(unsigned)ceil_div(threads, 256), 256, 0, s>>>(nwork, (const int4 *)work,
                                                                              (const unsigned char *)entries, w, grid,
                                                                              rowmap, scratch);
    IB200_LAUNCH_CHECK();
    if (nsplit > 0) {
        kb_density_fold_kernel<<<(unsigned)ceil_div((int64_t)nsplit * kTV, 256), 256, 0, s>>>(nsplit, (const int4 *)split,
                                                                                             scratch, grid, rowmap);
        IB200_LAUNCH_CHECK();
    }
    return 0;
}

int ib200_kb_density_update(void *stream, int64_t m, const void *records, const float *grid, const int64_t dims[3],
                            float inv_scale2, float *w, double *residual) {
    IB200_RANGE("ib200_kb_density_update");
    IB200_REQUIRE(m >= 0 && dims, "bad arguments");
    if (m == 0) return 0;
    IB200_REQUIRE(records && grid && w, "null pointer");
    IB200_REQUIRE(dims[0] > 0 && dims[1] > 0 && dims[2] > 0 && dims[0] * dims[1] * dims[2] < (1LL << 31), "bad grid");
    IB200_REQUIRE(((uintptr_t)records & 15) == 0, "records must be 16-byte aligned");
    const int64_t blocks = ceil_div(m, 256);
    IB200_REQUIRE(blocks < (1LL << 31), "too many samples");
    cudaStream_t s = as_stream(stream);
    kb_density_update_kernel<<<(unsigned)blocks, 256, 0, s>>>(m, (const KbRecord *)records, grid, (int)dims[0], (int)dims[1],
                                                              (int)dims[2], inv_scale2, w, residual);
    IB200_LAUNCH_CHECK();
    if (residual) {
        kb_density_residual_kernel<<<1, 256, 0, s>>>(blocks, residual);
        IB200_LAUNCH_CHECK();
    }
    return 0;
}

}  // extern "C"
