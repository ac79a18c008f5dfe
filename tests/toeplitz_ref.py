"""
TEST INFRASTRUCTURE ONLY -- numpy/float64 restatement of the Toeplitz embedding of the SENSE normal operator
(indigo_b200.fused.toeplitz_normal, DESIGN.md section 9), next to the -O3 oracle of oracle/sense.py:

    T x = s^2 * sum_c conj(S_c) * crop_N( IFFT_L( K * FFT_L( pad_L(S_c * x) ) ) ),   K = Re FFT_L(p_sym) / prod(L)

with the padded grid L of fused.toeplitz_grid, the image window at offset L//2 - N//2 (as the fused plan pads),
and p either the exact direct sum  p(d) = sum_m w_m^2 exp(+2 pi i kappa_m . d)  or the gridded adjoint of an
oracle operator on an image of L points applied to the k-space w (PSF read at image index d + L/2).
"""
import numpy as np

from oracle import sense as osense


def lags(L):
    """Per axis: the lag d of every circular grid index (d = j for j < L/2, j - L above)."""
    return [np.where(np.arange(l) < (l + 1) // 2, np.arange(l), np.arange(l) - l) for l in L]


def _axis_phases(kappa, pos, sign):
    """(M, len(pos)) exp(sign * 2 pi i kappa_m pos_j)."""
    return np.exp(sign * 2j * np.pi * np.outer(kappa, pos))


def exact_psf(L, coord, w2):
    """Direct-sum PSF in circular order, complex128 (L0, L1, L2)."""
    c = osense.flat_coord(coord).astype(np.float64)
    e = [_axis_phases(c[a], d, +1) for a, d in enumerate(lags(L))]
    X = (w2[:, None] * e[0])[:, :, None] * e[1][:, None, :]                  # (M, L0, L1)
    return np.tensordot(X, e[2], axes=([0], [0]))                            # (L0, L1, L2)


def gridded_psf(L, coord, weights, oversamp=2.0):
    """PSF from the oracle's gridded adjoint on an image of L points, centred at L/2, in circular order."""
    op = osense.SenseOperator(L, coord, np.ones(tuple(L) + (1,), dtype=np.complex64), oversamp, weights=weights)
    w = np.ones(op.M) if weights is None else np.asarray(weights, dtype=np.float64).reshape(-1, order='F')
    img = op.adjoint(w.astype(np.complex64).reshape(-1, 1)).reshape(tuple(L), order='F').astype(np.complex128)
    idx = [(j + l // 2) % l for j, l in zip(np.meshgrid(*[np.arange(l) for l in L], indexing='ij'), L)]
    return img[idx[0], idx[1], idx[2]]


def symmetrise(p):
    """(p(d) + conj p(-d)) / 2 in circular order."""
    m = p[np.ix_(*[(-np.arange(l)) % l for l in p.shape])]
    return 0.5 * (p + np.conj(m))


def kernel(p):
    """K = FFT_L(p_sym) / prod(L) (complex; its imaginary part vanishes for a Hermitian p)."""
    return np.fft.fftn(symmetrise(p)) / p.size


def apply(K, N, maps, x, s2=1.0):
    """T x for images x (prod(N),) or (prod(N), 1), column-major; K real or complex (L0, L1, L2)."""
    N, L = tuple(int(v) for v in N), K.shape
    off = [l // 2 - n // 2 for l, n in zip(L, N)]
    win = tuple(slice(o, o + n) for o, n in zip(off, N))
    X = np.asarray(x, dtype=np.complex128).reshape(N, order='F')
    out = np.zeros(N, dtype=np.complex128)
    for c in range(maps.shape[3]):
        S = maps[..., c].astype(np.complex128)
        g = np.zeros(L, dtype=np.complex128)
        g[win] = S * X
        g = np.fft.ifftn(K * np.fft.fftn(g)) * g.size
        out += np.conj(S) * g[win]
    return (s2 * out).reshape(-1, 1, order='F')


def exact_normal(N, coord, w2, x):
    """E^H W E x with E[m, r] = exp(-2 pi i kappa_m . r) (column-major voxels), complex128."""
    N = tuple(int(v) for v in N)
    c = osense.flat_coord(coord).astype(np.float64)
    e = [_axis_phases(c[a], np.arange(n), -1) for a, n in enumerate(N)]
    X = np.asarray(x, dtype=np.complex128).reshape(N, order='F')
    t = np.einsum('abc,mc->mab', X, e[2])
    t = np.einsum('mab,mb->ma', t, e[1])
    y = np.einsum('ma,ma->m', t, e[0]) * w2
    t = np.conj(e[0])[:, :, None] * y[:, None, None]                        # (M, N0, 1)
    t = t * np.conj(e[1])[:, None, :]                                       # (M, N0, N1)
    out = np.tensordot(t, np.conj(e[2]), axes=([0], [0]))                   # (N0, N1, N2)
    return out.reshape(-1, 1, order='F')


def probe(nvox, seed=20):
    rs = np.random.RandomState(seed)
    return (rs.rand(nvox, 1) + 1j * rs.rand(nvox, 1)).astype(np.complex64)


def fit_scale(K, N, coord, weights, oversamp=2.0, seed=20):
    """s^2 = Re<T1 v, N1 v> / ||T1 v||^2 with the unit map (one coil): T1 = T at s = 1, N1 the oracle's gridded
    normal operator -- the fit toeplitz_normal makes."""
    N = tuple(int(v) for v in N)
    ones = np.ones(N + (1,), dtype=np.complex64)
    v = probe(int(np.prod(N)), seed)
    t = apply(K, N, ones, v)
    a = osense.SenseOperator(N, coord, ones, oversamp, weights=weights).normal(v).astype(np.complex128)
    return float(np.vdot(t, a).real / np.vdot(t, t).real)


def toeplitz_operator(N, coord, maps, weights=None, oversamp=2.0):
    """(K real, s^2, L) of the recipe on the oracle's gridded PSF."""
    from indigo_b200.fused import toeplitz_grid
    L = toeplitz_grid(N, oversamp)
    K = kernel(gridded_psf(L, coord, weights, oversamp)).real
    return K, fit_scale(K, N, coord, weights, oversamp), L


def ls_scale(a, b):
    """c minimising ||a - c b||."""
    return float(np.vdot(b, a).real / np.vdot(b, b).real)


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))
