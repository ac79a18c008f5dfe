"""
ESPIRiT as defined in DESIGN.md section 12, checked on the CPU: the float64 restatement (tests/espirit_ref.py)
recovers birdcage maps from Cartesian and from gridded non-Cartesian calibration data, the lag form equals the
direct sum over kernels (and indigo_b200.espirit's FFT construction of it), synth.birdcage_maps matches the model,
and the public functions reject bad input before touching a device.
"""
import numpy as np
import pytest

from indigo_b200 import synth
from indigo_b200 import espirit as E
from oracle import sense as osense
import dcf_ref as D
import espirit_ref as R


def _cartesian(N, C, width):
    true = R.birdcage(N, C)
    ph = synth.phantom(N).astype(np.complex128)
    return true, np.abs(ph) > 0, R.cartesian_calib(true * ph[..., None], width)


@pytest.mark.parametrize("N,C,width", [((64, 64, 1), 8, 24), ((24, 24, 24), 8, 16)])
def test_cartesian_maps_align(N, C, width):
    true, mask, calib = _cartesian(N, C, width)
    maps, eig, kept = R.espirit(calib, N)
    assert R.alignment(maps, true, mask).mean() >= 0.999
    assert eig[mask].min() > 0.95
    if N == (64, 64, 1):
        assert kept == 49
        # the sign convention is visible: conjugated maps align far worse
        assert R.alignment(np.conj(maps), true, mask).mean() < 0.9


def test_power_iteration_matches_eigh():
    N, C = (64, 64, 1), 8
    _, mask, calib = _cartesian(N, C, 24)
    m1, e1, _ = R.espirit(calib, N, form='lag')
    m2, e2, _ = R.espirit(calib, N, form='eigh')
    sel = mask                            # outside the object lambda_2 / lambda_1 may be near 1
    np.testing.assert_allclose(e1[sel], e2[sel], atol=1e-6)
    assert np.abs(m1[sel] - m2[sel]).max() < 1e-3


@pytest.mark.parametrize("N,C,width,kernel", [((20, 16, 1), 4, 12, 5), ((12, 10, 9), 3, 8, 4)])
def test_lag_form_equals_direct_sum(N, C, width, kernel):
    _, _, calib = _cartesian(N, C, width)
    k = R.kernel_taps(N, kernel)
    A = R.calib_matrix(calib, k)
    V = R.kept(A.conj().T @ A, 0.02)
    P = R.lag_form(V, C, k)
    np.testing.assert_allclose(E.lag_coefficients(V, C, k), P, atol=1e-13 * np.abs(P).max())
    Md, Ml = R.matrices_direct(V, C, k, N), R.matrices_lag(P, N, k)
    assert np.abs(Md - Ml).max() <= 1e-12 * np.abs(Md).max()
    # the twiddle table of the device passes is the same phase
    tw = E.lag_twiddles(N[0], k[0])
    lag = np.arange(2 * k[0] - 1) - (k[0] - 1)
    want = np.exp(2j * np.pi * np.outer(np.arange(N[0]) - N[0] // 2, lag) / N[0])
    assert np.abs(tw - want).max() < 1e-6


def test_birdcage_maps_model():
    for N, C in [((16, 12, 10), 12), ((32, 32, 1), 8), ((8, 8, 8), 20)]:
        m = synth.birdcage_maps(N, C)
        assert m.shape == N + (C,) and m.dtype == np.complex64 and m.flags.f_contiguous
        np.testing.assert_allclose(m, R.birdcage(N, C), atol=1e-6)
        np.testing.assert_allclose((np.abs(m) ** 2).sum(axis=3), 1.0, atol=1e-5)
    assert np.array_equal(synth.birdcage_maps((8, 8, 8), 8), synth.birdcage_maps((8, 8, 8), 8))


def gridded_calibration(N, coord, y, width, dcf_iters=30):
    """calibration_kspace restated with the oracle's NUFFT and the float64 Pipe-Menon restatement."""
    pts = coord.reshape(3, -1, order='F')
    kappa = pts * np.array(N, dtype=np.float64)[:, None]
    w = tuple(width if n > 1 else 1 for n in N)
    keep = np.ones(pts.shape[1], dtype=bool)
    for d in range(3):
        if N[d] > 1:
            keep &= np.abs(kappa[d]) < w[d] / 2.0
    ccal = kappa[:, keep] / np.array(w, dtype=np.float64)[:, None]
    dcf = D.dcf(w, ccal, maxiter=dcf_iters)
    sw = np.sqrt(dcf).astype(np.float32).reshape(-1)
    op = osense.SenseOperator(w, ccal, np.ones(w + (1,), dtype=np.complex64, order='F'), 2.0, weights=sw)
    C = y.shape[1]
    img = np.stack([op.adjoint((sw * y[keep, c]).reshape(-1, 1)).reshape(w, order='F') for c in range(C)], axis=3)
    return np.fft.fftshift(np.fft.fftn(np.fft.ifftshift(img, axes=(0, 1, 2)), axes=(0, 1, 2)), axes=(0, 1, 2))


def test_gridded_calibration_maps_align():
    """Small kooshball: y = A_true phantom with the oracle's SENSE operator, then the calibration path restated.
    Measured: mean alignment 0.99986 (minimum 0.935) in the support (20^3 image, 8 coils, width 12, kernel 5)."""
    N, C = (20, 20, 20), 8
    coord = synth.kooshball_3d(nspokes=800, nread=40)
    true = synth.birdcage_maps(N, C)
    ph = synth.phantom(N)
    y = osense.SenseOperator(N, coord, true, 2.0).forward(ph.reshape(-1, 1, order='F'))
    calib = gridded_calibration(N, coord, y, 12)
    maps, eig, _ = R.espirit(calib, N, kernel=5)
    mask = np.abs(ph) > 0
    assert R.alignment(maps, true, mask).mean() >= 0.99


def test_error_paths():
    N = (16, 16, 1)
    calib = np.zeros((12, 12, 1, 4), dtype=np.complex64)
    with pytest.raises(ValueError):
        E.espirit_maps(None, calib[:, :, :, :, None], N)              # not (w0, w1, w2, C)
    with pytest.raises(ValueError):
        E.espirit_maps(None, np.zeros((12, 12, 3, 4), np.complex64), N)   # w2 != 1 for N2 == 1
    with pytest.raises(ValueError):
        E.espirit_maps(None, calib, N, kernel=13)                     # kernel > width
    with pytest.raises(ValueError):
        E.espirit_maps(None, np.zeros((12, 12, 1, 33), np.complex64), N)   # more than 32 coils
    for bad in (dict(thresh=-0.1), dict(thresh=1.0), dict(crop=1.5), dict(crop=-1), dict(max_iter=0),
                dict(max_iter=2.5)):
        with pytest.raises(ValueError):
            E.espirit_maps(None, calib, N, **bad)
    with pytest.raises(ValueError):
        E.espirit_maps(None, calib, (16, 16))                         # N not three extents
    coord = synth.radial_2d(nspokes=8, nread=16)
    y = np.zeros((coord.shape[1] * coord.shape[2], 4), np.complex64)
    with pytest.raises(ValueError):
        E.calibration_kspace(None, N, coord, y[:-1])                  # wrong sample count
    with pytest.raises(ValueError):
        E.calibration_kspace(None, N, coord, y, width=24)             # width above N
    with pytest.raises(ValueError):
        E.calibration_kspace(None, N, coord, y, width=1)
    with pytest.raises(ValueError):
        E.calibration_kspace(None, N, coord * 0 + 0.45, y, width=4)   # no sample in the calibration region
    with pytest.raises(RuntimeError):
        E.kept_vectors(np.zeros((8, 8)), 0.02)                        # nothing survives the threshold
