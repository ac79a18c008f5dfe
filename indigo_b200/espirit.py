"""
ESPIRiT coil sensitivity estimation (DESIGN.md section 12), following sigpy's EspiritCalib with one map set.

    calib = calibration_kspace(B, N, coord, y)        # non-Cartesian (M, C) data -> Cartesian centre (w, w, w, C)
    maps  = espirit_maps(B, calib, N)                 # (N0, N1, N2, C), what sense_operator_fused & co. take

The calibration matrix has one row per position of a k^D patch inside the calibration region and C k^D columns.  Its
Gram matrix G = A^H A is formed on the device (ib200_espirit_calib_gram); the eigenvectors of G whose singular
values exceed thresh * sigma_max are found on the host in float64 (the project has no device eigensolver); their
per-voxel image-domain matrix M(x) is evaluated in lag form, M(x) = sum_delta P(delta) e^{+2 pi i delta.(x-N/2)/N},
one axis at a time (ib200_espirit_lag_pass for z and y, ib200_espirit_maps for x), and ib200_espirit_maps runs the
power iteration per voxel.  No FFT of the image size is needed, so any extent works, odd ones included.
"""
import ctypes

import numpy as np

_C64 = np.dtype('complex64')
MAX_COILS = 32


def calib_shape(N, width):
    """(w0, w1, w2): `width` on every axis with N_d > 1, 1 elsewhere."""
    return tuple(int(width) if int(n) > 1 else 1 for n in N)


def _check_N(N):
    N = tuple(int(v) for v in N)
    if len(N) != 3 or min(N) < 1 or max(N) < 2:
        raise ValueError("N must be three positive extents with at least one above 1, got %r" % (N,))
    return N


def calibration_kspace(B, N, coord, y, width=24, oversamp=2.0, dcf_iters=30):
    """Cartesian calibration k-space (w0, w1, w2, C) complex64, column-major, DC at index w_d // 2, from multi-coil
    non-Cartesian data: y is (M, C) column-major complex64 (the layout A.H * y takes), M = prod(coord.shape[1:]),
    coord (3, ...) in cycles/FOV for an image of shape N.

    The samples with |N_d coord_d| < w_d / 2 on every axis with N_d > 1 are kept and rescaled to the calibration
    image, coord_cal = N coord / w.  Each coil is gridded with Pipe-Menon weights (pipe_menon_dcf, `dcf_iters`
    iterations): the adjoint of a one-coil SENSE operator on the w image (map 1, row weights sqrt(dcf)) applied to
    sqrt(dcf) * y_c.  The centred forward FFT of the coil images, with the SENSE operator's sign, gives calib.
    ValueError for inconsistent shapes, a width outside [2, N_d] or no sample inside the calibration region."""
    from .sense import pipe_menon_dcf, sense_operator_device
    from .fused import sense_operator_fused
    N = _check_N(N)
    width = int(width)
    w = calib_shape(N, width)
    if width < 2 or any(wd > n for wd, n in zip(w, N)):
        raise ValueError("calibration width %d must lie in [2, N_d] on every axis of N = %r" % (width, N))
    coord = np.asarray(coord, dtype=np.float64)
    if coord.ndim < 2 or coord.shape[0] != 3:
        raise ValueError("coord must be (3, ...), got shape %r" % (coord.shape,))
    pts = coord.reshape((3, -1), order='F')
    M = pts.shape[1]
    y = np.asarray(y)
    if M == 0 or y.size == 0 or y.size % M != 0 or (y.ndim == 2 and y.shape[0] != M) or y.ndim > 2:
        raise ValueError("y must be (M, C) with M = %d samples, got shape %r" % (M, y.shape))
    C = y.size // M
    y = y.reshape((M, C), order='F')
    kappa = pts * np.array(N, dtype=np.float64)[:, None]
    keep = np.ones(M, dtype=bool)
    for d in range(3):
        if N[d] > 1:
            keep &= np.abs(kappa[d]) < w[d] / 2.0
    if not keep.any():
        raise ValueError("no sample falls inside the %r calibration region" % (w,))
    ccal = kappa[:, keep] / np.array(w, dtype=np.float64)[:, None]
    dcf = pipe_menon_dcf(B, w, ccal, oversamp=oversamp, maxiter=dcf_iters)
    sw = np.sqrt(dcf).astype(np.float32).reshape(-1)
    ones = np.ones(w + (1,), dtype=_C64, order='F')
    try:
        A = sense_operator_fused(B, w, ccal, ones, oversamp, weights=sw)
    except RuntimeError:                                   # grid without specialised passes (2w = 48 has none)
        A = sense_operator_device(B, w, ccal, ones, oversamp, weights=sw)
    ysel = y[keep]
    nw = int(np.prod(w))
    img = np.empty((nw, C), dtype=_C64, order='F')
    for c in range(C):
        img[:, c] = (A.H * np.asfortranarray((sw * ysel[:, c]).astype(_C64).reshape(-1, 1))).reshape(-1)
    del A
    img = np.fft.ifftshift(img.reshape(w + (C,), order='F'), axes=(0, 1, 2))
    src = B.copy_array(np.asfortranarray(img))
    dst = B.empty_array(src.shape, _C64, name='espirit.calib')
    B.fftn(dst, src)
    return np.asfortranarray(np.fft.fftshift(dst.to_host(), axes=(0, 1, 2)))


def kept_vectors(G, thresh):
    """Eigenvectors of the Hermitian Gram matrix G (float64) whose singular values sqrt(lambda) exceed
    thresh * sigma_max, as the columns of V (n x r), largest first.  RuntimeError when none survives."""
    lam, V = np.linalg.eigh(np.asarray(G, dtype=np.complex128))
    sig = np.sqrt(np.maximum(lam, 0.0))
    smax = sig.max() if sig.size else 0.0
    keep = sig > thresh * smax
    if not smax > 0 or not keep.any():
        raise RuntimeError("ESPIRiT: no singular value of the calibration matrix survives the threshold %g" % thresh)
    return V[:, keep][:, ::-1]


def lag_coefficients(V, C, k):
    """Lag form of the per-voxel matrix: P (L2, L1, L0, C, C) complex128 with L_d = 2 k_d - 1, index j_d the lag
    j_d - (k_d - 1), P[j][c, c'] = prod(k)^-1 sum_kernels sum_{p - p' = delta} kern[c, p] conj(kern[c', p']) with
    kern = conj(v) reshaped (C, k2, k1, k0).  Computed as a correlation by FFTs of length L_d (no wrap-around)."""
    k0, k1, k2 = (int(v) for v in k)
    L = (2 * k2 - 1, 2 * k1 - 1, 2 * k0 - 1)
    r = V.shape[1]
    kern = np.conj(V).reshape(C, k2, k1, k0, r)
    F = np.fft.fftn(kern, s=L, axes=(1, 2, 3))                         # (C, L2, L1, L0, r)
    F = np.moveaxis(F.reshape(C, -1, r), 1, 0)                         # (L, C, r)
    Pf = np.matmul(F, np.conj(np.swapaxes(F, 1, 2)))                   # (L, C, C)
    P = np.fft.ifftn(Pf.reshape(L + (C, C)), axes=(0, 1, 2)) / (k0 * k1 * k2)
    return np.fft.fftshift(P, axes=(0, 1, 2))


def lag_twiddles(n, k):
    """(n, 2k - 1) table e^{+2 pi i (j - (k - 1)) (x - n//2) / n}, phases reduced exactly in integers."""
    lag = np.arange(2 * k - 1, dtype=np.int64) - (k - 1)
    m = np.mod(np.outer(np.arange(n, dtype=np.int64) - n // 2, lag), n)
    return np.exp(2j * np.pi * m / n).astype(_C64)


probe = None          # label -> context manager around each step of espirit_maps (tools/bench_espirit.py times them)


def _step(label):
    import contextlib
    return probe(label) if probe is not None else contextlib.nullcontext()


def calib_gram(B, calib, k):
    """G = A^H A (n x n, complex64, on the host) of the calibration matrix of calib (w0, w1, w2, C) for kernel taps
    k = (k0, k1, k2), formed on the device by ib200_espirit_calib_gram."""
    w, C = tuple(int(v) for v in calib.shape[:3]), int(calib.shape[3])
    n = C * int(np.prod(k))
    X = B.copy_array(np.asfortranarray(np.asarray(calib, dtype=_C64)))
    G = B.empty_array((n, n), _C64, name='espirit.gram')
    with _step("espirit_calib_gram"):
        B._lib.espirit_calib_gram(B._stream, (ctypes.c_int64 * 3)(*w), (ctypes.c_int64 * 3)(*k), C, X.ptr, G.ptr)
    return G.to_host()


def espirit_maps(B, calib, N, kernel=6, thresh=0.02, crop=0.95, max_iter=100, return_eig=False):
    """ESPIRiT sensitivity maps (N0, N1, N2, C) complex64, column-major, from Cartesian calibration k-space calib
    (w0, w1, w2, C), DC at w_d // 2, w_d = 1 on the axes with N_d = 1 (as calibration_kspace returns it).

    kernel: taps per transformed axis; thresh: singular values above thresh * sigma_max span the kept subspace;
    crop: the map is zero where the largest eigenvalue is <= crop; max_iter: power iterations per voxel.  With
    return_eig, returns (maps, eig), eig (N0, N1, N2) float32.  The result is bit-identical from run to run.
    ValueError for a shape mismatch, kernel > width, more than 32 coils or a bad thresh, crop or max_iter;
    RuntimeError when no singular value survives the threshold."""
    N = _check_N(N)
    calib = np.asarray(calib)
    if calib.ndim != 4:
        raise ValueError("calib must be (w0, w1, w2, C), got shape %r" % (calib.shape,))
    w, C = tuple(int(v) for v in calib.shape[:3]), int(calib.shape[3])
    kernel = int(kernel)
    if any((n == 1) != (wd == 1) for n, wd in zip(N, w)):
        raise ValueError("calib shape %r does not match N = %r: w_d must be 1 exactly where N_d is 1" % (calib.shape, N))
    if kernel < 1 or any(kernel > wd for wd, n in zip(w, N) if n > 1):
        raise ValueError("kernel %d must lie in [1, calibration width %r]" % (kernel, w))
    if not 1 <= C <= MAX_COILS:
        raise ValueError("ESPIRiT takes 1 to %d coils, got %d" % (MAX_COILS, C))
    if not 0.0 <= float(thresh) < 1.0:
        raise ValueError("thresh must lie in [0, 1), got %r" % (thresh,))
    if not 0.0 <= float(crop) <= 1.0:
        raise ValueError("crop must lie in [0, 1], got %r" % (crop,))
    if int(max_iter) < 1 or int(max_iter) != max_iter:
        raise ValueError("max_iter must be a positive integer, got %r" % (max_iter,))
    k = tuple(kernel if n > 1 else 1 for n in N)
    lags = tuple(2 * kd - 1 for kd in k)
    lib, s = B._lib, B._stream

    # 1. Gram matrix of the calibration matrix on the device; 2. kept subspace and lag form on the host, float64
    Gh = calib_gram(B, calib, k)
    with _step("host_eigh_lag"):
        V = kept_vectors(Gh, float(thresh))
        P = lag_coefficients(V, C, k)                                   # (L2, L1, L0, C, C)
        coef = np.ascontiguousarray(np.swapaxes(P, 3, 4)).astype(_C64)  # [j2][j1][j0][c'][c]
    del Gh, V, P

    # 3. z and y passes, then x, the power iteration, phase and crop per voxel
    CC = C * C
    P_d = B.copy_array(coef.reshape(-1))
    tw = [B.copy_array(lag_twiddles(N[d], k[d]).reshape(-1)) for d in range(3)]
    Q1 = B.empty_array((N[2] * lags[1] * lags[0] * CC,), _C64, name='espirit.lag_z')
    with _step("espirit_lag_pass[z]"):
        lib.espirit_lag_pass(s, 1, lags[2], N[2], lags[1] * lags[0] * CC, tw[2].ptr, P_d.ptr, Q1.ptr)
    del P_d
    Q2 = B.empty_array((N[2] * N[1] * lags[0] * CC,), _C64, name='espirit.lag_zy')
    with _step("espirit_lag_pass[y]"):
        lib.espirit_lag_pass(s, N[2], lags[1], N[1], lags[0] * CC, tw[1].ptr, Q1.ptr, Q2.ptr)
    del Q1
    nvox = int(np.prod(N))
    maps_d = B.empty_array((nvox, C), _C64, name='espirit.maps')
    eig_d = B.empty_array((nvox,), np.dtype('float32'), name='espirit.eig')
    with _step("espirit_maps"):
        lib.espirit_maps(s, (ctypes.c_int64 * 3)(*N), lags[0], C, int(max_iter), float(crop), tw[0].ptr, Q2.ptr,
                         maps_d.ptr, eig_d.ptr)
    maps = np.asfortranarray(maps_d.to_host().reshape(N + (C,), order='F'))
    eig = eig_d.to_host().reshape(N, order='F')
    del Q2, maps_d, eig_d
    return (maps, eig) if return_eig else maps
