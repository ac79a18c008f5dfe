"""
l1-wavelet reconstruction on the device (indigo_b200.wavelet): the transform against the float64 restatement
(tests/wavelet_ref.py), spectral_norm against the oracle, and FISTA with the gridded and the Toeplitz normal
operators against the restatement's FISTA on the float64 operators.
"""
import ctypes

import numpy as np
import pytest

from indigo_b200 import synth
from indigo_b200.fused import sense_operator_fused, toeplitz_normal
from indigo_b200.sense import normal_operator, sqrt_dcf
from indigo_b200.wavelet import wavelet_operator, l1wavelet_recon, spectral_norm, wavelet_levels
from oracle import sense as osense
import toeplitz_ref as TR
import wavelet_ref as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    from indigo_b200 import B200Backend
    return B200Backend(0)


def _rel(a, b):
    return float(np.linalg.norm(np.ravel(a) - np.ravel(b)) / np.linalg.norm(np.ravel(b)))


def _max_levels(N):
    j = 1
    while all(n % (1 << (j + 1)) == 0 for n in N if n > 1):
        j += 1
    return j


SHAPES = [(16, 16, 16), (32, 16, 24), (64, 64, 1), (208, 208, 208)]
CASES = [(N, w, j) for N in SHAPES for w in ('haar', 'db4') for j in range(1, _max_levels(N) + 1)]


@pytest.fixture(scope="module")
def images():
    cache = {}

    def get(N):
        if N not in cache:
            rs = np.random.RandomState(7)
            cache[N] = synth.rand64c(rs, int(np.prod(N)), 1) - (0.5 + 0.5j)
        return cache[N]
    return get


@pytest.mark.parametrize("N,wave,J", CASES, ids=["%dx%dx%d-%s-J%d" % (N + (w, j)) for N, w, j in CASES])
def test_transform_against_restatement(B, images, N, wave, J):
    x = images(N)
    W = wavelet_operator(B, N, wave, levels=J)
    assert W.shape == (x.shape[0], x.shape[0])
    c = W * x
    c_ref = R.dwt(x, N, wave, J)
    assert _rel(c, c_ref) <= 1e-6
    # W^H against the restatement: W^H (W_ref x) = x, and W^H W x = x
    assert _rel(W.H * c_ref.astype(np.complex64), x) <= 1e-6
    assert _rel(W.H * c, x) <= 2e-6
    if int(np.prod(N)) <= 1 << 16:
        cr = synth.rand64c(np.random.RandomState(8), int(np.prod(N)), 1)
        assert _rel(W.H * cr, R.idwt(cr, N, wave, J)) <= 1e-6


def test_alpha_beta_and_determinism(B, images):
    N = (32, 16, 24)
    x = images(N)
    W = wavelet_operator(B, N, 'db4')
    n = x.shape[0]
    c = W * x
    assert np.array_equal(c, W * x)
    y = synth.rand64c(np.random.RandomState(9), n, 1)
    for fwd, want in ((True, c), (False, W.H * x)):
        xd, yd = B.copy_array(x), B.copy_array(y)
        W.eval(yd, xd, alpha=0.5 - 0.25j, beta=2.0, forward=fwd)
        np.testing.assert_allclose(yd.to_host(), (0.5 - 0.25j) * want + 2.0 * y, rtol=0, atol=1e-5 * np.abs(want).max())
        nan = B.copy_array(np.full((n, 1), np.nan, dtype=np.complex64, order='F'))
        W.eval(nan, xd, alpha=1.0, beta=0.0, forward=fwd)
        out = nan.to_host()
        assert np.isfinite(out).all() and np.array_equal(out, want)


def _koosh(B, C=4, dcf=True):
    N = (16, 16, 16)
    rs = np.random.RandomState(0)
    coord = synth.kooshball_3d(nspokes=256, nread=32)
    maps = synth.unit_rss_maps(rs, N, C)
    w = sqrt_dcf(coord) if dcf else None
    return N, coord, maps, w


def _radial(B, C=4):
    N = (64, 64, 1)
    rs = np.random.RandomState(1)
    coord = synth.radial_2d(nspokes=48, nread=128)
    maps = synth.unit_rss_maps(rs, N, C)
    return N, coord, maps, None


def _problem(N, coord, maps, w):
    """b = A^H A truth (oracle, complex64) for the phantom, and the float64 normal operator."""
    op = osense.SenseOperator(N, coord, maps, 2.0, weights=w)
    truth = synth.phantom(N).reshape(-1, 1, order='F')
    b = op.normal(truth).astype(np.complex64).reshape(-1, 1, order='F')
    return op, np.asfortranarray(b), osense.SenseTruth64(op).normal


def test_spectral_norm_against_oracle(B):
    N, coord, maps, w = _koosh(B)
    A = sense_operator_fused(B, N, coord, maps, 2.0, weights=w)
    op = osense.SenseOperator(N, coord, maps, 2.0, weights=w)
    got = spectral_norm(B, normal_operator(A))
    want = osense.spectral_norm(op)
    assert abs(got - want) <= 1e-4 * want


@pytest.mark.parametrize("geom", ["koosh", "radial"])
@pytest.mark.parametrize("lam_f,x0_kind", [(1e-2, "zero"), (0.0, "zero"), (1e-2, "rand")])
def test_fista_gridded_against_restatement(B, geom, lam_f, x0_kind):
    N, coord, maps, w = (_koosh if geom == "koosh" else _radial)(B)
    A = sense_operator_fused(B, N, coord, maps, 2.0, weights=w)
    op, b, normal64 = _problem(N, coord, maps, w)
    L = osense.spectral_norm(op)
    step, lam, J = 0.9 / L, lam_f * L, wavelet_levels(N, 'db4')
    nvox = int(np.prod(N))
    x0 = (np.zeros((nvox, 1), np.complex64, order='F') if x0_kind == "zero"
          else synth.rand64c(np.random.RandomState(3), nvox, 1))
    x = x0.copy(order='F')
    l1wavelet_recon(B, normal_operator(A), b, x, N, lam, step=step, maxiter=30)
    want = R.fista(normal64, b, x0, N, lam, step, 'db4', J, 30)
    assert _rel(x, want) <= 1e-4


def test_fista_toeplitz_against_restatement(B):
    N, coord, maps, w = _koosh(B)
    A = sense_operator_fused(B, N, coord, maps, 2.0, weights=w)
    T = toeplitz_normal(A)
    K, s2, _ = TR.toeplitz_operator(N, coord, maps, w)
    truth = synth.phantom(N).reshape(-1, 1, order='F')
    b = np.asfortranarray(TR.apply(K, N, maps, truth, s2).astype(np.complex64))
    L = spectral_norm(B, T)
    step, lam = 0.9 / L, 1e-2 * L
    x = np.zeros_like(b, order='F')
    l1wavelet_recon(B, T, b, x, N, lam, wave='haar', step=step, maxiter=30)
    want = R.fista(lambda v: TR.apply(K, N, maps, v, s2), b, np.zeros_like(b), N, lam, step, 'haar',
                   wavelet_levels(N, 'haar'), 30)
    assert _rel(x, want) <= 1e-4


def test_large_lamda_zeroes_the_detail_bands(B):
    N, coord, maps, w = _koosh(B)
    A = sense_operator_fused(B, N, coord, maps, 2.0, weights=w)
    _, b, _ = _problem(N, coord, maps, w)
    x = np.zeros_like(b, order='F')
    l1wavelet_recon(B, normal_operator(A), b, x, N, 1e6, maxiter=5)
    c = wavelet_operator(B, N, 'db4') * x
    mask = R.detail_mask(N, wavelet_levels(N, 'db4'))
    assert np.linalg.norm(c) > 0
    assert np.linalg.norm(c[mask]) <= 1e-6 * np.linalg.norm(c)


def test_graph_history_tol_and_determinism(B):
    N, coord, maps, w = _radial(B)
    A = sense_operator_fused(B, N, coord, maps, 2.0, weights=w)
    AHA = normal_operator(A)
    _, b, _ = _problem(N, coord, maps, w)
    L = spectral_norm(B, AHA)
    kw = dict(step=0.9 / L, maxiter=20)
    runs = []
    for graph in (False, False, True):
        x = np.zeros_like(b, order='F')
        l1wavelet_recon(B, AHA, b, x, N, 1e-2 * L, graph=graph, **kw)
        runs.append(x)
    assert np.array_equal(runs[0], runs[1])
    assert np.array_equal(runs[0], runs[2])
    hist = []
    x = np.zeros_like(b, order='F')
    l1wavelet_recon(B, AHA, b, x, N, 1e-2 * L, history=hist, **kw)
    assert len(hist) == 20 and np.array_equal(x, runs[0])
    assert all(np.isfinite(hist)) and hist[0] == 1.0 and hist[-1] < hist[0]
    tol = hist[9] * 1.0000001
    hist2 = []
    x = np.zeros_like(b, order='F')
    l1wavelet_recon(B, AHA, b, x, N, 1e-2 * L, tol=tol, history=hist2, **kw)
    stop = next(i for i, r in enumerate(hist) if r < tol)
    assert len(hist2) == stop + 1 < 20
    assert hist2 == hist[:stop + 1]


class _DoublingTeam(object):
    """Stands for the all-reduce over two identical coil shards: sums the image of both ranks (2 x its own)."""

    def __init__(self, B):
        self.B = B

    def allreduce_array(self, arr):
        self.B.scale(arr, 2.0)


def test_team_of_two_shards(B):
    N, coord, maps, w = _koosh(B)
    A = sense_operator_fused(B, N, coord, maps, 2.0, weights=w)
    _, b, _ = _problem(N, coord, maps, w)
    L = spectral_norm(B, normal_operator(A))
    x1 = np.zeros_like(b, order='F')
    l1wavelet_recon(B, normal_operator(A), b, x1, N, 1e-2 * L, maxiter=15)
    team = _DoublingTeam(B)
    shards = [sense_operator_fused(B, N, coord, np.asfortranarray((maps / np.sqrt(2)).astype(np.complex64)), 2.0,
                                   weights=w) for _ in range(2)]
    assert abs(spectral_norm(B, normal_operator(shards[0]), team=team) - L) <= 1e-5 * L
    outs = []
    for S in shards:
        x = np.zeros_like(b, order='F')
        l1wavelet_recon(B, normal_operator(S), b, x, N, 1e-2 * L, maxiter=15, team=team)
        outs.append(x)
    assert np.array_equal(outs[0], outs[1])
    assert _rel(outs[0], x1) <= 1e-6


def test_errors(B):
    N, coord, maps, w = _koosh(B, C=1)
    A = sense_operator_fused(B, N, coord, maps, 2.0, weights=w)
    AHA = normal_operator(A)
    b = np.zeros((4096, 1), np.complex64, order='F')
    x = np.zeros_like(b, order='F')
    bad = [dict(N=(16, 16, 8)), dict(N=(16, 16, 16), levels=5), dict(N=(16, 16, 16), wave='db8'),
           dict(N=(16, 16, 16), lamda=-1.0), dict(N=(16, 16, 16), step=0.0), dict(N=(16, 16, 16), step=-1.0),
           dict(N=(16, 16, 16), graph=True, tol=1e-3), dict(N=(16, 16, 16), graph=True, history=[])]
    for kw in bad:
        args = dict(lamda=1.0, maxiter=3)
        args.update(kw)
        with pytest.raises(ValueError):
            l1wavelet_recon(B, AHA, b, x, **args)
    with pytest.raises(ValueError):                        # an indivisible axis
        wavelet_operator(B, (16, 12, 16), 'haar', levels=3)
    with pytest.raises(ValueError):                        # too many levels
        wavelet_operator(B, (16, 16, 16), 'haar', levels=5)
    with pytest.raises(ValueError):
        wavelet_operator(B, (16, 16, 16), 'sym8')
    with pytest.raises(TypeError):
        l1wavelet_recon(B, AHA, b, x, (16, 16, 16), 1.0, maxiter=3, team=object())
    with pytest.raises(TypeError):
        spectral_norm(B, AHA, team=object())
    with pytest.raises(RuntimeError):
        wavelet_operator(B, (1024, 8, 1), 'haar')
    # the C entry point refuses long axes and bad filters by status, without launching
    h = (ctypes.c_double * 2)(2 ** -0.5, 2 ** -0.5)
    d = B.empty_array((1024 * 8, 1), np.dtype('complex64'))
    with pytest.raises(RuntimeError, match="512"):
        B._lib.wavelet(B._stream, (ctypes.c_int64 * 3)(1024, 8, 1), 2, h, 1, 0, 1.0, 0.0, 0.0, 0.0, d.ptr, d.ptr, d.ptr)
    with pytest.raises(RuntimeError, match="filter length"):
        B._lib.wavelet(B._stream, (ctypes.c_int64 * 3)(16, 8, 1), 4, h, 1, 0, 1.0, 0.0, 0.0, 0.0, d.ptr, d.ptr, d.ptr)
