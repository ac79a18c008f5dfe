"""
float64 numpy restatement of ESPIRiT as DESIGN.md section 12 defines it (indigo_b200/espirit.py, csrc/espirit.cu):
calibration matrix, kept subspace, the per-voxel matrix M(x) as a direct sum over kernels and in lag form, its
largest eigenvector by dense eigh and by the power iteration, and the birdcage maps of synth.birdcage_maps.
"""
import numpy as np


def birdcage(N, C, r=1.5):
    """sigpy.mri.birdcage_maps on the (x, y, z) = (axis 0, 1, 2) grid, complex128 (N0, N1, N2, C)."""
    x, y, z = np.meshgrid(*[(np.arange(n) - n / 2.0) / (n / 2.0) for n in N], indexing='ij')
    out = np.empty(tuple(N) + (C,), dtype=np.complex128)
    for c in range(C):
        three = N[2] > 1
        ang = c * 2 * np.pi / (8 if three else C)
        cz = np.floor(c / 8) - 0.5 * (np.ceil(C / 8) - 1) if three else 0.0
        phs = -(c + np.floor(c / 8)) * 2 * np.pi / 8 if three else -c * 2 * np.pi / C
        xc, yc, zc = x - r * np.cos(ang), y - r * np.sin(ang), (z - cz if three else 0.0)
        out[..., c] = np.exp(1j * (np.arctan2(xc, -yc) + phs)) / np.sqrt(xc ** 2 + yc ** 2 + zc ** 2)
    return out / np.sqrt((np.abs(out) ** 2).sum(axis=3, keepdims=True))


def kernel_taps(N, k):
    return tuple(k if n > 1 else 1 for n in N)


def cartesian_calib(img, width):
    """Centred forward DFT of img (N0, N1, N2, C) cropped to the centre: (w0, w1, w2, C), DC at w // 2."""
    N = img.shape[:3]
    X = np.fft.fftshift(np.fft.fftn(np.fft.ifftshift(img, axes=(0, 1, 2)), axes=(0, 1, 2)), axes=(0, 1, 2))
    sl = tuple(slice(n // 2 - width // 2, n // 2 - width // 2 + width) if n > 1 else slice(0, 1) for n in N)
    return X[sl]


def calib_matrix(calib, k):
    """A (R, C k0 k1 k2): row s = kernel position (s0 fastest), column p0 + k0 (p1 + k1 p2) + k0 k1 k2 c."""
    w, C = calib.shape[:3], calib.shape[3]
    r = [w[d] - k[d] + 1 for d in range(3)]
    rows = []
    for s2 in range(r[2]):
        for s1 in range(r[1]):
            for s0 in range(r[0]):
                patch = calib[s0:s0 + k[0], s1:s1 + k[1], s2:s2 + k[2], :]        # (k0, k1, k2, C)
                rows.append(patch.transpose(3, 2, 1, 0).reshape(-1))             # (c, p2, p1, p0)
    return np.array(rows, dtype=np.complex128)


def kept(G, thresh):
    lam, V = np.linalg.eigh(G)
    sig = np.sqrt(np.maximum(lam, 0.0))
    return V[:, sig > thresh * sig.max()]


def matrices_direct(V, C, k, N):
    """M(x) (nvox, C, C), x column-major, from the kernels kern_j = conj(v_j): k^-D sum_j vt_j vt_j^H."""
    kD = int(np.prod(k))
    kern = np.conj(V.T).reshape(-1, C, k[2], k[1], k[0])                    # (r, c, p2, p1, p0)
    E = [np.exp(2j * np.pi * np.outer(np.arange(k[d]), np.arange(N[d]) - N[d] // 2) / N[d]) for d in range(3)]
    vt = np.einsum('jczyx,xa,yb,zg->jcabg', kern, E[0], E[1], E[2])          # (r, C, N0, N1, N2)
    vt = vt.reshape(vt.shape[0], C, -1, order='F')                           # voxels column-major
    return np.einsum('jcv,jdv->vcd', vt, np.conj(vt)) / kD


def lag_form(V, C, k):
    """P (2k2-1, 2k1-1, 2k0-1, C, C) by the explicit double sum over taps."""
    kD = int(np.prod(k))
    kern = np.conj(V.T).reshape(-1, C, k[2], k[1], k[0])
    L = tuple(2 * kk - 1 for kk in (k[2], k[1], k[0]))
    P = np.zeros(L + (C, C), dtype=np.complex128)
    for p2 in range(k[2]):
        for p1 in range(k[1]):
            for p0 in range(k[0]):
                a = kern[:, :, p2, p1, p0]                                   # (r, C)
                for q2 in range(k[2]):
                    for q1 in range(k[1]):
                        for q0 in range(k[0]):
                            b = kern[:, :, q2, q1, q0]
                            P[p2 - q2 + k[2] - 1, p1 - q1 + k[1] - 1, p0 - q0 + k[0] - 1] += a.T @ np.conj(b)
    return P / kD


def matrices_lag(P, N, k):
    """M(x) (nvox, C, C) from the lag form: sum_delta P(delta) e^{+2 pi i delta.(x - N//2)/N}."""
    E = []
    for d in range(3):
        lag = np.arange(2 * k[d] - 1) - (k[d] - 1)
        E.append(np.exp(2j * np.pi * np.outer(np.arange(N[d]) - N[d] // 2, lag) / N[d]))   # (N_d, L_d)
    M = np.einsum('zyxcd,az,by,gx->gbacd', P, E[2], E[1], E[0])            # (N0, N1, N2, C, C)
    return M.reshape((-1,) + P.shape[3:], order='F')


def power_maps(M, iters, crop):
    """The power iteration from the all-ones vector, coil-0 phase, crop; returns (maps (nvox, C), eig (nvox,))."""
    v = np.ones(M.shape[:2], dtype=np.complex128)
    nrm = np.zeros(M.shape[0])
    for _ in range(iters):
        w = np.einsum('vcd,vd->vc', M, v)
        nrm = np.linalg.norm(w, axis=1)
        v = w / np.where(nrm > 0, nrm, 1.0)[:, None]
    return _finish(v, nrm, crop)


def eigh_maps(M, crop):
    """Largest eigenpair of every M(x) by dense eigh, same phase and crop."""
    lam, U = np.linalg.eigh(M)
    return _finish(U[:, :, -1], lam[:, -1], crop)


def _finish(v, eig, crop):
    a = np.abs(v[:, 0])
    ph = np.where(a > 0, np.conj(v[:, 0]) / np.where(a > 0, a, 1.0), 1.0)
    v = v * ph[:, None]
    v[eig <= crop] = 0
    return v, eig


def espirit(calib, N, kernel=6, thresh=0.02, crop=0.95, iters=100, form='lag'):
    """maps (N0, N1, N2, C), eig (N0, N1, N2), kept count; form 'lag' / 'direct' / 'eigh' (lag form, dense eigh)."""
    C = calib.shape[3]
    k = kernel_taps(N, kernel)
    A = calib_matrix(np.asarray(calib, dtype=np.complex128), k)
    V = kept(A.conj().T @ A, thresh)
    M = matrices_direct(V, C, k, N) if form == 'direct' else matrices_lag(lag_form(V, C, k), N, k)
    m, e = eigh_maps(M, crop) if form == 'eigh' else power_maps(M, iters, crop)
    return m.reshape(tuple(N) + (C,), order='F'), e.reshape(N, order='F'), V.shape[1]


def alignment(est, true, mask):
    """|<m_est(x), m_true(x)>| / (|m_est| |m_true|) averaged over the voxels of mask."""
    e, t = est[mask], true[mask]
    num = np.abs((np.conj(e) * t).sum(axis=1))
    den = np.linalg.norm(e, axis=1) * np.linalg.norm(t, axis=1)
    return num / np.where(den > 0, den, 1.0)
