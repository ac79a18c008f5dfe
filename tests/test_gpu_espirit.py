"""
ESPIRiT on the device (indigo_b200.espirit, csrc/espirit.cu) against the float64 restatement (tests/espirit_ref.py):
the calibration Gram matrix, the kept subspace, eigenvalues and maps on 3-D, odd-extent and 2-D shapes with 8 and
32 coils, bit-identity, the non-Cartesian calibration path end to end with CG, the maps in the existing operators,
and the error paths.
"""
import numpy as np
import pytest

from indigo_b200 import synth, calibration_kspace, espirit_maps, l1wavelet_recon
from indigo_b200 import espirit as E
from indigo_b200.fused import sense_operator_fused, toeplitz_normal
from indigo_b200.sense import normal_operator
import espirit_ref as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    from indigo_b200 import B200Backend
    return B200Backend(0)


SHAPES = {  # name: (N, coils, calibration width)
    "cube16_c8": ((16, 16, 16), 8, 12),
    "box_c8": ((32, 24, 20), 8, 16),
    "odd2d_c8": ((33, 40, 1), 8, 24),
    "2d_c8": ((64, 64, 1), 8, 24),
    "2d_c32": ((64, 64, 1), 32, 24),
}


def _calib(N, C, width):
    true = synth.birdcage_maps(N, C)
    ph = synth.phantom(N)
    return true, np.abs(ph) > 0, R.cartesian_calib(true.astype(np.complex128) * ph[..., None], width).astype(np.complex64)


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_gram_and_kept(B, name):
    N, C, width = SHAPES[name]
    _, _, calib = _calib(N, C, width)
    k = R.kernel_taps(N, 6)
    G = E.calib_gram(B, calib, k)
    A = R.calib_matrix(calib.astype(np.complex128), k)
    G64 = A.conj().T @ A
    assert np.linalg.norm(G - G64) <= 1e-5 * np.linalg.norm(G64)
    assert np.array_equal(G, np.conj(G.T))
    assert E.kept_vectors(G, 0.02).shape[1] == R.kept(G64, 0.02).shape[1]


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_maps_against_restatement(B, name):
    N, C, width = SHAPES[name]
    true, mask, calib = _calib(N, C, width)
    maps, eig = espirit_maps(B, calib, N, return_eig=True)
    assert maps.shape == N + (C,) and maps.dtype == np.complex64 and maps.flags.f_contiguous
    assert eig.shape == N and eig.dtype == np.float32
    want, weig, _ = R.espirit(calib, N)
    assert np.abs(eig - weig).max() <= 1e-5
    sel = (weig > 0.95) & (eig > 0.95)
    assert sel.sum() >= mask.sum()
    assert np.abs(maps[sel] - want[sel]).max() <= 1e-4
    assert not np.any(maps[eig <= 0.95])
    assert R.alignment(maps, true, mask).mean() >= 0.999


def test_bit_identical(B):
    N, C, width = SHAPES["box_c8"]
    _, _, calib = _calib(N, C, width)
    m1, e1 = espirit_maps(B, calib, N, return_eig=True)
    m2, e2 = espirit_maps(B, calib, N, return_eig=True)
    assert np.array_equal(m1, m2) and np.array_equal(e1, e2)


def _operator(B, N, coord, maps):
    try:
        return sense_operator_fused(B, N, coord, maps)
    except RuntimeError:                                   # grid without specialised passes
        from indigo_b200.sense import sense_operator_device
        return sense_operator_device(B, N, coord, maps)


def _nrmse(x, ph, mask):
    a, b = np.abs(x.reshape(ph.shape, order='F'))[mask], np.abs(ph)[mask]
    return np.linalg.norm(a - b) / np.linalg.norm(b)


E2E = {  # name: (N, coils, trajectory)
    "koosh32": ((32, 32, 32), 8, lambda: synth.kooshball_3d(nspokes=2000, nread=64)),
    "radial2d": ((64, 64, 1), 8, lambda: synth.radial_2d(nspokes=100, nread=128)),
}


@pytest.mark.parametrize("name", sorted(E2E))
def test_end_to_end_cg(B, name):
    """y = A_true phantom, maps from calibration_kspace + espirit_maps, 30 CG iterations with either maps."""
    N, C, traj = E2E[name]
    coord = traj()
    true = synth.birdcage_maps(N, C)
    ph = synth.phantom(N)
    mask = np.abs(ph) > 0
    y = _operator(B, N, coord, true) * ph.reshape(-1, 1, order='F')
    calib = calibration_kspace(B, N, coord, y.reshape(-1, C, order='F'))
    assert calib.shape == tuple(24 if n > 1 else 1 for n in N) + (C,)
    maps = espirit_maps(B, calib, N)
    align = R.alignment(maps, true, mask)
    assert align.mean() >= 0.99
    err = {}
    for label, m in (("true", true), ("est", maps)):
        A = _operator(B, N, coord, m)
        b = A.H * y
        x = np.zeros_like(b, order='F')
        B.cg(normal_operator(A), b, x, lamda=0.0, maxiter=30, tol=0.0)
        err[label] = _nrmse(x, ph, mask)
    print("%s: alignment %.5f, NRMSE true maps %.4f, estimated maps %.4f" % (name, align.mean(), err["true"], err["est"]))
    assert err["est"] <= 1.1 * err["true"]


def test_maps_feed_operators(B):
    N, C = (32, 32, 32), 8
    coord = synth.kooshball_3d(nspokes=1500, nread=64)
    true, _, calib = _calib(N, C, 24)
    maps = espirit_maps(B, calib, N)
    A = sense_operator_fused(B, N, coord, maps)
    y = A * synth.phantom(N).reshape(-1, 1, order='F')
    b = A.H * y
    T = toeplitz_normal(A)
    t = T * b
    assert np.all(np.isfinite(t)) and np.linalg.norm(t) > 0
    x = np.zeros_like(b, order='F')
    l1wavelet_recon(B, T, b, x, N, lamda=1e-4 * np.abs(b).max(), maxiter=5)
    assert np.all(np.isfinite(x)) and np.linalg.norm(x) > 0


def test_error_paths(B):
    N = (16, 16, 1)
    with pytest.raises(RuntimeError):
        espirit_maps(B, np.zeros((12, 12, 1, 4), np.complex64), N)      # no singular value survives
    with pytest.raises(ValueError):
        espirit_maps(B, np.zeros((12, 12, 1, 40), np.complex64), N)
    with pytest.raises(ValueError):
        espirit_maps(B, np.ones((12, 12, 1, 4), np.complex64), N, kernel=13)
    coord = synth.radial_2d(nspokes=8, nread=16)
    with pytest.raises(ValueError):
        calibration_kspace(B, N, coord, np.zeros((7, 4), np.complex64))
