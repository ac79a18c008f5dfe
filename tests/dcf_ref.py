"""
TEST INFRASTRUCTURE ONLY -- numpy/float64 restatement of the Pipe-Menon density compensation
(indigo_b200.sense.pipe_menon_dcf, DESIGN.md section 10) on the oracle's interpolation matrix:

    w_0 = 1,   w_{k+1} = w_k / (I I^T w_k),      I = oracle.sense.interp_matrix (the NUFFT's gridding matrix
                                                  without the centring phase and the scale)

where a sample whose q = (I I^T w)_m is not positive and finite gets the weight 0, as on the device.
"""
import numpy as np

from oracle import sense as osense


def interp(N, coord, oversamp=2.0, width=3, n=128):
    """I (M x prod(oN)) in float64 CSR, the float32 matrix of the reference's Backend.Interp promoted."""
    oN, omin = osense.oversampled_shape(tuple(int(v) for v in N), oversamp)
    beta, table = osense.kb_table(width, omin, n)
    return osense.interp_matrix(oN, coord, width, table).astype(np.float64).tocsr()


def residual(I, w):
    """Fixed-point residual ||I I^T w - 1|| / sqrt(M)."""
    return float(np.linalg.norm(I @ (I.T @ w) - 1.0) / np.sqrt(I.shape[0]))


def pipe_menon(I, maxiter=30, history=None):
    """Weights (M,) float64 in the sample order of I's rows; history (list): the residual of the weights each
    iteration starts from, as pipe_menon_dcf reports it."""
    w = np.ones(I.shape[0])
    for _ in range(maxiter):
        q = I @ (I.T @ w)
        if history is not None:
            history.append(float(np.linalg.norm(q - 1.0) / np.sqrt(q.size)))
        ok = np.isfinite(q) & (q > 0)
        w = np.where(ok, w / np.where(ok, q, 1.0), 0.0)
    return w


def dcf(N, coord, oversamp=2.0, width=3, n=128, maxiter=30, history=None):
    """The restatement with pipe_menon_dcf's arguments and result layout (shaped like coord.shape[1:], samples in
    column-major order), float64."""
    coord = np.asarray(coord)
    w = pipe_menon(interp(N, coord, oversamp, width, n), maxiter, history)
    return w.reshape(coord.shape[1:], order='F')


def kabs(coord):
    """|k| of every sample, in the same layout as dcf()."""
    coord = np.asarray(coord, dtype=np.float64)
    return np.sqrt((coord ** 2).sum(axis=0))


def rel(a, b):
    """||a - b|| / ||b|| in double precision (complex or real)."""
    a, b = (np.asarray(v).astype(np.complex128 if np.iscomplexobj(v) else np.float64) for v in (a, b))
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))
