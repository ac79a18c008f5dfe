// Setup of the Toeplitz-embedded normal operator (indigo_b200/fused.py: toeplitz_normal).
//
// The normal operator of a non-uniform DFT is a convolution with the point-spread function
// p(d) = sum_m w_m^2 exp(+2 pi i kappa_m . d).  Its kernel on the zero-padded grid of L points per axis is
// K = Re FFT_L(p_sym) / prod(L), where p_sym(d) = (p(d) + conj p(-d)) / 2 is the Hermitian part of p: K is
// then exactly real and the operator exactly self-adjoint.  p comes from a gridded adjoint on an image of L
// points per axis (PSF centred at index L/2); these two kernels re-lay it into circular order and turn its
// spectrum into the real kernel the convolution pass (ib200_sense_toeplitz_pass) reads.  The FFT between them
// is ib200_fft_exec.
#include "common.cuh"

namespace ib200 {

// out[circular index of d] = (p(d) + conj p(-d)) / 2, p(d) = img[d + L/2], one thread per output point
__global__ void __launch_bounds__(256) toeplitz_psf_kernel(int64_t L0, int64_t L1, int64_t L2, const c64 *__restrict__ img,
                                                           c64 *__restrict__ out) {
    const int64_t n = L0 * L1 * L2;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j0 = j % L0, j1 = (j / L0) % L1, j2 = j / (L0 * L1);
        // circular position j holds lag d = j (mod L) in [-L/2, L/2): image index d + L/2, mirror index L/2 - d
        const int64_t i0 = (j0 + L0 / 2) % L0, i1 = (j1 + L1 / 2) % L1, i2 = (j2 + L2 / 2) % L2;
        const int64_t m0 = (L0 - i0) % L0, m1 = (L1 - i1) % L1, m2 = (L2 - i2) % L2;
        const c64 a = img[(i2 * L1 + i1) * L0 + i0], b = img[(m2 * L1 + m1) * L0 + m0];
        out[j] = mk(0.5f * (a.x + b.x), 0.5f * (a.y - b.y));
    }
}

__global__ void __launch_bounds__(256) toeplitz_kernel_kernel(int64_t n, const c64 *__restrict__ spec, float scale,
                                                              float *__restrict__ kern) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        kern[i] = scale * spec[i].x;
}

static unsigned grid_blocks(int64_t n) {
    int64_t b = ceil_div(n, (int64_t)256);
    const int64_t cap = (int64_t)sm_count() * 16;
    return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace ib200

using namespace ib200;

extern "C" {

int ib200_toeplitz_psf(void *stream, const int64_t L[3], const void *img, void *psf) {
    IB200_RANGE("ib200_toeplitz_psf");
    IB200_REQUIRE(L && img && psf && img != psf, "null or aliased pointer");
    for (int d = 0; d < 3; ++d) IB200_REQUIRE(L[d] >= 1, "bad grid extent");
    const int64_t n = L[0] * L[1] * L[2];
    toeplitz_psf_kernel<<<grid_blocks(n), 256, 0, as_stream(stream)>>>(L[0], L[1], L[2], (const c64 *)img, (c64 *)psf);
    IB200_LAUNCH_CHECK();
    return 0;
}

int ib200_toeplitz_kernel(void *stream, int64_t n, const void *spectrum, float scale, float *kernel) {
    IB200_RANGE("ib200_toeplitz_kernel");
    IB200_REQUIRE(spectrum && kernel && n >= 1, "null pointer or empty kernel");
    toeplitz_kernel_kernel<<<grid_blocks(n), 256, 0, as_stream(stream)>>>(n, (const c64 *)spectrum, scale, kernel);
    IB200_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
