"""
l1-wavelet compressed-sensing reconstruction on the device (DESIGN.md section 11).

    W = wavelet_operator(B, N, wave='db4')                        # orthonormal, W.H == W^-1
    x_h = np.zeros((nvox, 1), np.complex64, order='F')
    l1wavelet_recon(B, normal_operator(A), A.H * y, x_h, N, lamda=1e-3)

solves  min_x  1/2 ||A x - y||^2 + lamda ||detail bands of W x||_1  by FISTA (Beck and Teboulle), given any node
AHA ~ A^H A with .eval(out, inp) (normal_operator(A), toeplitz_normal(A) or the six-call tree) and b = A^H y.
The transform is the periodized, separable (Mallat) orthonormal wavelet transform of a column-major
N0 x N1 x N2 image; axes of one point are not transformed.  One FISTA iteration is one apply of AHA and one call of
ib200_wavelet_fista_step, whose passes fuse the gradient step, the soft threshold and the momentum update.
"""
import ctypes
import math

import numpy as np

_C64 = np.dtype('complex64')

# Orthonormal low-pass filters.  db4 (8 taps, 4 vanishing moments) is the spectral factorisation of
# Q(y) = sum_{k<4} C(3+k, k) y^k with y = (2 - z - 1/z)/4, minimum phase, in float64; tests/wavelet_ref.py derives it
# and checks these digits.
FILTERS = {
    'haar': (2 ** -0.5, 2 ** -0.5),
    'db4': (0.23037781330889615, 0.7148465705529148, 0.6308807679298586, -0.027983769416858723,
            -0.1870348117190923, 0.0308413818355607, 0.03288301166688511, -0.010597401785069),
}
MAX_AXIS = 512                      # longest transformed axis of the device passes
STATS_DOUBLES = 2 + 2 * 4096        # IB200_WAVELET_STATS


def wavelet_filter(wave):
    """Low-pass filter of `wave` ('haar' or 'db4') as a float64 array; ValueError for any other name."""
    if wave not in FILTERS:
        raise ValueError("unknown wavelet %r (known: %s)" % (wave, ", ".join(sorted(FILTERS))))
    return np.array(FILTERS[wave], dtype=np.float64)


def wavelet_levels(N, wave='db4', levels=None):
    """Number of levels J.  Default: the largest J such that every transformed axis (N_d > 1) is divisible by 2^J
    and J <= floor(log2(N_d / (Lf - 1))).  An explicit `levels` must satisfy the divisibility rule only.  J < 1, a
    violated rule or no axis to transform raise ValueError."""
    lf = len(wavelet_filter(wave))
    N = tuple(int(v) for v in N)
    if len(N) != 3 or min(N) < 1:
        raise ValueError("N must be three positive extents, got %r" % (N,))
    axes = [n for n in N if n > 1]
    if not axes:
        raise ValueError("no axis of N = %r has more than one point" % (N,))

    def divisible(j):
        return all(n % (1 << j) == 0 for n in axes)

    if levels is None:
        j = 0
        while divisible(j + 1) and all(j + 1 <= math.floor(math.log2(n / (lf - 1))) for n in axes):
            j += 1
        if j < 1:
            raise ValueError("N = %r admits no wavelet level for %s" % (N, wave))
        return j
    j = int(levels)
    if j < 1:
        raise ValueError("levels must be at least 1, got %d" % j)
    if not divisible(j):
        raise ValueError("every transformed axis of N = %r must be divisible by 2^%d" % (N, j))
    return j


class _Geometry(object):
    """Shape, filter and levels of one transform, in the form the C ABI takes them."""

    def __init__(self, N, wave, levels):
        self.N = tuple(int(v) for v in N)
        self.J = wavelet_levels(self.N, wave, levels)
        self.h = wavelet_filter(wave)
        self.wave = wave
        self.nvox = int(np.prod(self.N))
        self.dims = (ctypes.c_int64 * 3)(*self.N)
        self.hp = (ctypes.c_double * len(self.h))(*self.h)


def make_wavelet_class(ops):
    """The wavelet node on top of the operator family `ops` (indigo_b200.linop or the reference's operators)."""

    class Wavelet(ops.Operator):
        """W : image (nvox) -> coefficients (nvox), orthonormal; W.H is its inverse."""

        def __init__(self, backend, geom, name='W'):
            ops.Operator.__init__(self, backend, name=name)
            self._geom = geom
            self._work = None

        shape = property(lambda self: (self._geom.nvox, self._geom.nvox))
        dtype = property(lambda self: _C64)

        def _mem_usage(self, ncols=1):
            return 0

        def _eval(self, y, x, alpha=1, beta=0, forward=True, left=True):
            if not left:
                raise NotImplementedError("Right-multiplication not implemented for Wavelet.")
            if x.shape[1] != 1:
                raise ValueError("Wavelet takes one image at a time (got %d columns)" % x.shape[1])
            B, g = self._backend, self._geom
            if self._work is None:
                self._work = B.empty_array((g.nvox, 1), _C64, name='wavelet.work')
            a, b = complex(alpha), complex(beta)
            B._lib.wavelet(B._stream, g.dims, len(g.h), g.hp, g.J, 0 if forward else 1, a.real, a.imag, b.real, b.imag,
                           x.ptr, y.ptr, self._work.ptr)

    return Wavelet


_cache = {}


def wavelet_operator(B, N, wave='db4', levels=None):
    """Orthonormal wavelet transform W of N0 x N1 x N2 images (column-major, x fastest) as an operator of B's
    family: W * x, W.H * c and W.eval(y, x, alpha, beta) work.  Transformed axes (N_d > 1) must have at most 512
    points (RuntimeError otherwise); `levels` as in wavelet_levels (ValueError)."""
    from .sense import _ops_of
    geom = _Geometry(N, wave, levels)
    if any(n > MAX_AXIS for n in geom.N):
        raise RuntimeError("wavelet transform: axes of more than %d points are not supported, N = %r" % (MAX_AXIS, geom.N))
    ops = _ops_of(B)
    if ops not in _cache:
        _cache[ops] = make_wavelet_class(ops)
    return _cache[ops](B, geom, name='W.%s' % wave)


def _check_team(team):
    if team is not None and not hasattr(team, 'allreduce_array'):
        raise TypeError("team must provide allreduce_array (the image is summed over ranks after every apply), got %s"
                        % type(team).__name__)


def _check_square(AHA, nvox, N):
    if tuple(int(v) for v in AHA.shape) != (nvox, nvox):
        raise ValueError("AHA has shape %r, which does not match N = %r (%d voxels)" % (tuple(AHA.shape), tuple(N), nvox))


def spectral_norm(B, AHA, iters=15, seed=0, team=None):
    """||AHA||_2 by power iteration on the device: v <- AHA v / ||AHA v||, `iters` times, from the probe of
    oracle.sense.spectral_norm (RandomState(seed), rand + 1j*rand, complex64).  With a team, the image is summed
    over ranks after every apply (team.allreduce_array)."""
    _check_team(team)
    n = int(AHA.shape[1])
    rs = np.random.RandomState(seed)
    v = B.copy_array((rs.rand(n, 1) + 1j * rs.rand(n, 1)).astype(_C64, order='F'), name='power.v')
    w = B.empty_array((n, 1), _C64, name='power.w')
    nv = 1.0
    for _ in range(int(iters)):
        AHA.eval(w, v)
        if team is not None:
            team.allreduce_array(w)
        nv = math.sqrt(B.norm2(w))
        if nv == 0.0:
            return 0.0
        B.axpby(0, v, 1.0 / nv, w)
    return nv


def fista_momentum(maxiter):
    """(t_k - 1) / t_{k+1} for k = 1 .. maxiter with t_1 = 1, t_{k+1} = (1 + sqrt(1 + 4 t_k^2)) / 2, in float64."""
    t, out = 1.0, []
    for _ in range(int(maxiter)):
        t1 = (1.0 + math.sqrt(1.0 + 4.0 * t * t)) / 2.0
        out.append((t - 1.0) / t1)
        t = t1
    return np.array(out, dtype=np.float64)


def l1wavelet_recon(B, AHA, b_h, x_h, N, lamda, wave='db4', levels=None, step=None, maxiter=50, tol=0.0, team=None,
                    graph=False, history=None):
    """FISTA on  min_x 1/2 ||A x - y||^2 + lamda ||detail bands of W x||_1,  given AHA ~ A^H A and b = A^H y:

        x_k     = W^H soft_{step lamda}(W (z_k - step (AHA z_k - b)))      (detail bands only)
        z_{k+1} = x_k + ((t_k - 1) / t_{k+1}) (x_k - x_{k-1}),   z_1 = x_0,  t_1 = 1.

    Same contract as B.cg: b_h and x_h are host arrays, column-major (nvox, 1), complex64; x_h holds the initial
    guess and receives the result.  `lamda` is absolute.  step=None uses 0.9 / spectral_norm(B, AHA, team=team).
    With `team` (needs allreduce_array), the output of every apply is summed over ranks; the vectors stay
    replicated, so every rank computes the same iterates.  After iteration k, r_k = ||x_k - x_{k-1}|| / ||x_k|| is
    computed on the device when `history` (a list, r_k appended) or tol > 0 (stop once r_k < tol) asks for it;
    otherwise the loop never synchronises with the host.  graph=True (needs tol <= 0 and history None) runs one
    eager iteration, captures the next one (apply, all-reduce, prox step) in a CUDA graph and replays it; the
    result is bit-identical to the eager loop."""
    _check_team(team)
    _check_square(AHA, int(np.prod([int(v) for v in N])), N)
    geom = _Geometry(N, wave, levels)
    if any(n > MAX_AXIS for n in geom.N):
        raise RuntimeError("wavelet transform: axes of more than %d points are not supported, N = %r" % (MAX_AXIS, geom.N))
    nvox = geom.nvox
    lamda = float(lamda)
    if not lamda >= 0.0:
        raise ValueError("lamda must be >= 0, got %r" % lamda)
    if step is not None and not float(step) > 0.0:
        raise ValueError("step must be > 0, got %r" % step)
    if graph and (tol > 0 or history is not None):
        raise ValueError("graph=True needs tol <= 0 and history=None (a replayed graph cannot stop early or report)")
    maxiter = int(maxiter)
    if maxiter < 1:
        return
    if step is None:
        step = 0.9 / spectral_norm(B, AHA, team=team)
    step = float(step)
    torch, lib = B._torch, B._lib
    x = B.copy_array(x_h, name='fista.x')
    b = B.copy_array(b_h, name='fista.b')
    z = x.copy(name='fista.z')
    g = B.empty_array((nvox, 1), _C64, name='fista.g')
    work = B.empty_array((nvox, 1), _C64, name='fista.work')
    mom = torch.from_numpy(fista_momentum(maxiter)).to(B._device)
    counter = torch.zeros(1, dtype=torch.int32, device=B._device)
    report = tol > 0 or history is not None
    stats = torch.zeros(STATS_DOUBLES, dtype=torch.float64, device=B._device) if report else None
    thresh = step * lamda

    def iteration():
        AHA.eval(g, z)
        if team is not None:
            team.allreduce_array(g)
        lib.wavelet_fista_step(B._stream, geom.dims, len(geom.h), geom.hp, geom.J, step, thresh, g.ptr, b.ptr, z.ptr,
                               x.ptr, work.ptr, mom.data_ptr(), counter.data_ptr(),
                               stats.data_ptr() if report else None)

    if graph and maxiter >= 2:
        iteration()                                            # eager: first-use allocations and attributes
        side = torch.cuda.Stream(device=B._device)
        side.wait_stream(torch.cuda.current_stream(B._device))
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(cg, stream=side):
                iteration()
        torch.cuda.current_stream(B._device).wait_stream(side)
        for _ in range(maxiter - 1):                           # capturing records the iteration, it does not run it
            cg.replay()
        x.copy_to(x_h)
        return
    for _ in range(maxiter):
        iteration()
        if report:
            d2, n2 = (float(v) for v in stats[:2].cpu())
            r = math.sqrt(d2 / n2) if n2 > 0 else (0.0 if d2 == 0 else math.inf)
            if history is not None:
                history.append(r)
            if tol > 0 and r < tol:
                break
    x.copy_to(x_h)
