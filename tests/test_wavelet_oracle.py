"""
CPU tests of the l1-wavelet definition (tests/wavelet_ref.py, DESIGN.md section 11) and of the host-side pieces of
indigo_b200.wavelet: filters, levels, orthonormality, FISTA convergence and what l1-wavelet buys over Tikhonov CG.
"""
import numpy as np
import pytest

from indigo_b200 import synth
from indigo_b200 import wavelet as W
import wavelet_ref as R


def test_db4_derivation():
    h = R.db_filter(4)
    g = R.highpass(h)
    assert len(h) == 8
    assert abs(h.sum() - np.sqrt(2.0)) <= 1e-13
    assert abs((h * h).sum() - 1.0) <= 1e-13
    for s in (1, 2, 3):
        assert abs((h[:8 - 2 * s] * h[2 * s:]).sum()) <= 1e-13
    n = np.arange(8.0)
    for p in range(4):
        assert abs((g * n ** p).sum()) <= 1e-13 * max(1.0, (np.abs(g) * n ** p).sum())
    # the package's table is the derivation to the last digit or two
    assert np.abs(W.wavelet_filter('db4') - h).max() <= 1e-15
    assert np.abs(W.wavelet_filter('haar') - R.lowpass('haar')).max() <= 2e-16


@pytest.mark.parametrize("N,wave,J", [
    ((16, 16, 16), 'db4', 1), ((16, 16, 16), 'haar', 4), ((32, 16, 24), 'db4', 3), ((32, 16, 24), 'haar', 3),
    ((64, 64, 1), 'db4', 3), ((16, 16, 1), 'db4', 3),       # level 3 of 16 points: sub-box of 4 < 8 taps
    ((8, 2, 1), 'db4', 1), ((6, 1, 1), 'db4', 1),
])
def test_orthonormal(N, wave, J):
    rs = np.random.RandomState(0)
    nvox = int(np.prod(N))
    x = rs.randn(nvox, 1) + 1j * rs.randn(nvox, 1)
    c = R.dwt(x, N, wave, J)
    assert abs(np.linalg.norm(c) - np.linalg.norm(x)) <= 1e-12 * np.linalg.norm(x)
    assert np.linalg.norm(R.idwt(c, N, wave, J) - x) <= 1e-12 * np.linalg.norm(x)


def test_synthesis_is_the_transpose():
    N, wave, J = (8, 4, 4), "db4", 2
    n = int(np.prod(N))
    Wm = np.hstack([R.dwt(e.reshape(-1, 1), N, wave, J) for e in np.eye(n)])
    Hm = np.hstack([R.idwt(e.reshape(-1, 1), N, wave, J) for e in np.eye(n)])
    assert np.abs(Wm.T - Hm).max() <= 1e-13
    assert np.abs(Wm.T @ Wm - np.eye(n)).max() <= 1e-13


def test_levels():
    assert W.wavelet_levels((208, 208, 208), 'db4') == 4
    assert W.wavelet_levels((256, 256, 1), 'db4') == 5
    assert W.wavelet_levels((256, 256, 128), 'db4') == 4
    assert W.wavelet_levels((16, 16, 16), 'haar') == 4
    assert W.wavelet_levels((208, 208, 208), 'db4', levels=2) == 2
    assert W.wavelet_levels((16, 16, 1), 'db4', levels=4) == 4           # explicit: divisibility only
    for N, lv in (((16, 16, 16), 0), ((16, 16, 16), 5), ((16, 12, 16), 3), ((16, 16, 16), -1)):
        with pytest.raises(ValueError):
            W.wavelet_levels(N, 'db4', levels=lv)
    with pytest.raises(ValueError):
        W.wavelet_levels((6, 6, 1), 'db4')                                # log2(6/7) < 1
    with pytest.raises(ValueError):
        W.wavelet_levels((1, 1, 1), 'haar')
    with pytest.raises(ValueError):
        W.wavelet_levels((16, 16, 16), 'db8')


def test_soft_threshold_and_momentum():
    c = np.array([3 + 4j, 0j, 0.5 + 0j, -2j])
    np.testing.assert_allclose(R.soft(c, 1.0), [(3 + 4j) * 0.8, 0, 0, -1j], rtol=0, atol=1e-15)
    m = W.fista_momentum(4)
    t = [1.0]
    for _ in range(4):
        t.append((1 + np.sqrt(1 + 4 * t[-1] ** 2)) / 2)
    np.testing.assert_allclose(m, [(t[k] - 1) / t[k + 1] for k in range(4)], rtol=1e-15)
    assert m[0] == 0.0


def _small_problem():
    N = (8, 8, 1)
    rs = np.random.RandomState(4)
    coord = np.zeros((3, 48))
    coord[:2] = rs.rand(2, 48) - 0.5
    E = R.nudft_matrix(N, coord)
    x0 = synth.phantom(N).reshape(-1, 1, order='F').astype(np.complex128)
    y = E @ x0
    y = y + 0.05 * np.abs(y).max() * (rs.randn(48, 1) + 1j * rs.randn(48, 1))
    return N, E, y


def test_fista_converges_on_a_dense_nudft():
    """48 samples of an 8 x 8 image (underdetermined): after 200 iterations the objective is within 1e-6 of a
    5000-iteration run (measured: 3.5e-12)."""
    N, E, y = _small_problem()
    AHA, b = E.conj().T @ E, E.conj().T @ y
    L = np.linalg.norm(AHA, 2)
    lam, step, J = 0.02 * L, 0.9 / L, 2
    hist = []
    x200 = R.fista(lambda v: AHA @ v, b, np.zeros_like(b), N, lam, step, 'db4', J, 200, history=hist)
    x5000 = R.fista(lambda v: AHA @ v, b, np.zeros_like(b), N, lam, step, 'db4', J, 5000)
    f200, f5000 = (R.objective(E, y, x, N, 'db4', J, lam) for x in (x200, x5000))
    assert f5000 <= f200
    assert (f200 - f5000) / f5000 <= 1e-6
    assert len(hist) == 200 and hist[-1] < hist[0]


def test_l1_wavelet_beats_tikhonov_on_undersampled_radial():
    """2-D 32 x 32 phantom, 16 radial spokes of 64 samples (Nyquist is about pi/2 * 32 = 50 spokes), exact NUDFT,
    noiseless, 50 iterations each.  Measured: l1-wavelet (db4, 2 levels, lamda = 1e-3 ||A^H A||) NRMSE 0.413;
    Tikhonov CG at its best lamda of {1e-4, 1e-3, 1e-2, 1e-1} ||A^H A|| NRMSE 0.458."""
    N = (32, 32, 1)
    truth = synth.phantom(N).reshape(-1, 1, order='F').astype(np.complex128)
    E = R.nudft_matrix(N, synth.radial_2d(nspokes=16, nread=64))
    y = E @ truth
    AHA, b = E.conj().T @ E, E.conj().T @ y
    L = np.linalg.norm(AHA, 2)
    it = 50

    def cg(lam):
        x, r = np.zeros_like(b), b.copy()
        p, rr = r.copy(), np.vdot(r, r).real
        for _ in range(it):
            Ap = AHA @ p + lam * p
            a = rr / np.vdot(p, Ap).real
            x, r = x + a * p, r - a * Ap
            r2 = np.vdot(r, r).real
            p, rr = r + (r2 / rr) * p, r2
        return x

    best_cg = min(R.nrmse(cg(f * L), truth) for f in (1e-4, 1e-3, 1e-2, 1e-1))
    J = W.wavelet_levels(N, 'db4')
    x = R.fista(lambda v: AHA @ v, b, np.zeros_like(b), N, 1e-3 * L, 0.9 / L, 'db4', J, it)
    l1 = R.nrmse(x, truth)
    assert l1 < best_cg - 0.02, (l1, best_cg)


def test_phantom():
    p3 = synth.phantom((32, 24, 16))
    assert p3.dtype == np.complex64 and p3.flags['F_CONTIGUOUS'] and p3.shape == (32, 24, 16)
    assert np.array_equal(p3, synth.phantom((32, 24, 16)))
    vals = np.unique(np.round(p3.real, 6))
    assert 3 <= len(vals) <= 12 and np.all(p3.imag == 0)              # piecewise constant
    p2 = synth.phantom((64, 64, 1))
    assert p2.shape == (64, 64, 1) and p2.real.max() == pytest.approx(1.0) and p2[0, 0, 0] == 0
