"""
float64 numpy restatement of the l1-wavelet reconstruction (DESIGN.md section 11): filters, the periodized
separable orthonormal wavelet transform, the complex soft threshold and FISTA against any `normal(x)` callable.
Written from the definition, not from the kernels; the tests compare indigo_b200.wavelet with it.
"""
from math import comb

import numpy as np
from numpy.polynomial import polynomial as P


def db_filter(p=4):
    """Daubechies low-pass filter with p vanishing moments (2p taps) by spectral factorisation in float64:
    Q(y) = sum_{k<p} C(p-1+k, k) y^k with y = (2 - z - 1/z)/4, the roots of z^(p-1) Q inside the unit circle,
    h ~ (1 + z)^p prod (z - z0), normalised to sum h = sqrt(2)."""
    poly = np.zeros(1)
    for k in range(p):
        t = np.array([1.0])
        for _ in range(k):
            t = P.polymul(t, np.array([-0.25, 0.5, -0.25]))
        t = np.concatenate([np.zeros(p - 1 - k), t, np.zeros(p - 1 - k)])
        poly = P.polyadd(poly, comb(p - 1 + k, k) * t)
    roots = np.roots(poly[::-1])
    h = np.array([1.0])
    for _ in range(p):
        h = P.polymul(h, [1.0, 1.0])
    for z0 in roots[np.abs(roots) < 1]:
        h = P.polymul(h, [-z0, 1.0])
    h = np.real(h)
    h = h / h.sum() * np.sqrt(2.0)
    return h[::-1] if abs(h[0]) < abs(h[-1]) else h


def lowpass(wave):
    if wave == 'haar':
        return np.array([1.0, 1.0]) / np.sqrt(2.0)
    if wave == 'db4':
        return db_filter(4)
    raise ValueError(wave)


def highpass(h):
    L = len(h)
    return np.array([(-1) ** n * h[L - 1 - n] for n in range(L)])


def _analysis(X, h, g):
    """One level along axis 0 of X (even length n): [a | d]."""
    n = X.shape[0]
    k = np.arange(n // 2)
    a = sum(h[m] * X[(2 * k + m) % n] for m in range(len(h)))
    d = sum(g[m] * X[(2 * k + m) % n] for m in range(len(h)))
    return np.concatenate([a, d], axis=0)


def _synthesis(C, h, g):
    """Transpose of _analysis."""
    n = C.shape[0]
    k = np.arange(n // 2)
    a, d = C[:n // 2], C[n // 2:]
    X = np.zeros_like(C)
    for m in range(len(h)):
        X[(2 * k + m) % n] += h[m] * a + g[m] * d
    return X


def _passes(N, J):
    """(level, axis, sub-box extents) of the analysis in execution order."""
    out = []
    for j in range(1, J + 1):
        ext = tuple(n >> (j - 1) if n > 1 else 1 for n in N)
        for ax in range(3):
            if N[ax] > 1:
                out.append((j, ax, ext))
    return out


def _apply(c, N, wave, J, inverse):
    N = tuple(int(v) for v in N)
    h = lowpass(wave)
    g = highpass(h)
    C = np.asarray(c, dtype=np.complex128).reshape(N, order='F').copy()
    passes = _passes(N, J)
    for j, ax, ext in (passes[::-1] if inverse else passes):
        box = tuple(slice(0, e) for e in ext)
        sub = np.moveaxis(C[box], ax, 0)
        sub = (_synthesis if inverse else _analysis)(sub, h, g)
        C[box] = np.moveaxis(sub, 0, ax)
    return C.reshape(-1, 1, order='F')


def dwt(x, N, wave, J):
    """W x for a column-major image of shape N; (nvox, 1) complex128."""
    return _apply(x, N, wave, J, False)


def idwt(c, N, wave, J):
    """W^H c = W^-1 c."""
    return _apply(c, N, wave, J, True)


def detail_mask(N, J):
    """True on the detail coefficients, False on the coarse band (extent N_d / 2^J); (nvox, 1)."""
    N = tuple(int(v) for v in N)
    m = np.ones(N, dtype=bool)
    m[tuple(slice(0, n >> J if n > 1 else 1) for n in N)] = False
    return m.reshape(-1, 1, order='F')


def soft(c, t):
    """c max(0, 1 - t / |c|), 0 where c == 0."""
    r = np.abs(c)
    with np.errstate(divide='ignore', invalid='ignore'):
        s = np.where(r > t, 1.0 - t / np.where(r > 0, r, 1.0), 0.0)
    return c * s


def prox(u, N, wave, J, t):
    c = dwt(u, N, wave, J)
    mask = detail_mask(N, J)
    c = np.where(mask, soft(c, t), c)
    return idwt(c, N, wave, J)


def fista(normal, b, x0, N, lamda, step, wave, J, maxiter, history=None):
    """FISTA (Beck-Teboulle) on 1/2 ||A x - y||^2 + lamda ||detail(W x)||_1 with normal(x) = A^H A x, b = A^H y."""
    b = np.asarray(b, dtype=np.complex128).reshape(-1, 1)
    x = np.asarray(x0, dtype=np.complex128).reshape(-1, 1).copy()
    z, t = x.copy(), 1.0
    for _ in range(maxiter):
        u = z - step * (np.asarray(normal(z), dtype=np.complex128).reshape(-1, 1) - b)
        xn = prox(u, N, wave, J, step * lamda)
        t1 = (1.0 + np.sqrt(1.0 + 4.0 * t * t)) / 2.0
        z = xn + ((t - 1.0) / t1) * (xn - x)
        if history is not None:
            history.append(np.linalg.norm(xn - x) / np.linalg.norm(xn))
        x, t = xn, t1
    return x


def objective(E, y, x, N, wave, J, lamda):
    """1/2 ||E x - y||^2 + lamda ||detail(W x)||_1 for a dense E."""
    r = E @ x - y
    c = dwt(x, N, wave, J)
    return 0.5 * float(np.vdot(r, r).real) + lamda * float(np.abs(c[detail_mask(N, J)]).sum())


def nudft_matrix(N, coord):
    """Dense E[m, r] = exp(-2 pi i kappa_m . r) on column-major voxels r (centred indices), complex128."""
    N = tuple(int(v) for v in N)
    c = np.asarray(coord, dtype=np.float64).reshape(3, -1)
    grids = np.meshgrid(*[np.arange(n) - n // 2 for n in N], indexing='ij')
    pos = np.stack([gg.reshape(-1, order='F') for gg in grids])           # (3, nvox)
    return np.exp(-2j * np.pi * (c.T @ pos))


def nrmse(x, truth):
    return float(np.linalg.norm(np.ravel(x) - np.ravel(truth)) / np.linalg.norm(np.ravel(truth)))
