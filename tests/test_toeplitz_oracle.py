"""
The Toeplitz embedding of the SENSE normal operator in numpy/float64 (tests/toeplitz_ref.py), no device:
the embedding is exact for the exact PSF, the gridded PSF gives an operator at least as close to the exact model
as the gridded normal operator itself, and the symmetrised kernel is real.
"""
import numpy as np
import pytest

from indigo_b200 import synth
from indigo_b200.fused import toeplitz_grid
from oracle import sense as osense
import toeplitz_ref as R


def _w2(coord, w):
    m = osense.flat_coord(coord).shape[1]
    return np.ones(m) if w is None else np.asarray(w, dtype=np.float64) ** 2


@pytest.mark.parametrize("N", [(8, 8, 8), (16, 16, 1), (9, 7, 5), (12, 8, 6), (20, 6, 4)])
def test_exact_psf_reproduces_normal_matrix(N):
    rs = np.random.RandomState(1)
    coord = synth.random_3d(rs, 300)
    if N[2] == 1:
        coord[2] = 0
    w2 = rs.rand(300) + 0.5
    L = toeplitz_grid(N)
    assert all(l >= 2 * n - 1 for l, n in zip(L, N) if n > 1)
    K = R.kernel(R.exact_psf(L, coord, w2))
    maps = synth.unit_rss_maps(rs, N, 2).astype(np.complex128)
    x = synth.rand64c(rs, int(np.prod(N)), 1).astype(np.complex128)
    want = sum(np.conj(maps[..., c]).reshape(-1, 1, order='F') *
               R.exact_normal(N, coord, w2, maps[..., c].reshape(-1, 1, order='F') * x) for c in range(2))
    assert R.rel(R.apply(K, N, maps, x), want) <= 1e-10


def test_grid_lengths():
    assert toeplitz_grid((208, 208, 208)) == (416, 416, 416)
    assert toeplitz_grid((64, 64, 1)) == (128, 128, 1)
    assert toeplitz_grid((20, 20, 20)) == (52, 52, 52)
    assert toeplitz_grid((100, 60, 30)) == (208, 128, 64)
    with pytest.raises(RuntimeError):
        toeplitz_grid((256, 256, 1))            # L = 512 would need 1024-point passes for the PSF


CASES = {
    "koosh": lambda rs: ((16, 16, 16), synth.kooshball_3d(nspokes=256, nread=32), False),
    "koosh_dcf": lambda rs: ((16, 16, 16), synth.kooshball_3d(nspokes=256, nread=32), True),
    "random": lambda rs: ((16, 16, 16), synth.random_3d(rs, 4000), False),
    "radial2d": lambda rs: ((32, 32, 1), synth.radial_2d(nspokes=64, nread=64), False),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_gridded_psf_closer_to_exact_than_gridded_normal(case):
    rs = np.random.RandomState(0)
    N, coord, dcf = CASES[case](rs)
    w = osense.sqrt_dcf(coord) if dcf else None
    C = 3
    maps = synth.unit_rss_maps(rs, N, C)
    K, s2, L = R.toeplitz_operator(N, coord, maps, w)
    x = synth.rand64c(rs, int(np.prod(N)), 1)
    grid = osense.SenseOperator(N, coord, maps, 2.0, weights=w).normal(x).astype(np.complex128)
    exact = sum(np.conj(maps[..., c]).reshape(-1, 1, order='F') *
                R.exact_normal(N, coord, _w2(coord, w), maps[..., c].reshape(-1, 1, order='F') * x) for c in range(C))
    exact = R.ls_scale(grid, exact) * exact
    t = R.apply(K, N, maps, x, s2)
    assert R.rel(t, exact) <= R.rel(grid, exact)
    assert R.rel(t, grid) <= 2e-2


def test_symmetrised_kernel_is_real():
    rs = np.random.RandomState(2)
    coord = synth.random_3d(rs, 500)
    L = (32, 32, 32)
    p = R.gridded_psf(L, coord, None)
    K = R.kernel(p)
    assert np.abs(K.imag).max() <= 1e-12 * np.abs(K.real).max()
    assert np.abs(np.fft.fftn(p).imag).max() > 1e-6 * np.abs(K.real).max() * p.size      # p itself is not Hermitian
