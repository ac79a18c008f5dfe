"""
Toeplitz-embedded normal operator (indigo_b200.fused.toeplitz_normal) on the device, against the numpy/float64
restatement of the recipe (tests/toeplitz_ref.py) and against the gridded fused normal operator.
"""
import numpy as np
import pytest

from indigo_b200 import synth
from indigo_b200.sense import sense_operator_device, normal_operator, sqrt_dcf
from indigo_b200.fused import sense_operator_fused, toeplitz_normal
from oracle import np_oracle as Kn
import toeplitz_ref as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    from indigo_b200 import B200Backend
    return B200Backend(0)


def _traj(kind, N):
    rs = np.random.RandomState(3)
    if kind == "koosh":
        return synth.kooshball_3d(nspokes=256, nread=2 * max(N))
    if kind == "random":
        return synth.random_3d(rs, 4000)
    return synth.radial_2d(nspokes=96, nread=2 * N[0])


CASES = [  # (trajectory, N, coils, sqrt-DCF)
    ("koosh", (16, 16, 16), 1, False),
    ("koosh", (16, 16, 16), 2, True),
    ("koosh", (16, 16, 16), 3, False),
    ("random", (16, 16, 16), 8, False),
    ("random", (16, 16, 16), 2, True),
    ("koosh", (26, 26, 26), 16, False),             # L = 52 (the smallest image with L = 52 the fused operator serves)
    ("koosh", (32, 16, 26), 2, True),               # anisotropic: L = (64, 32, 52)
    ("radial", (64, 64, 1), 32, False),
    ("radial", (64, 64, 1), 2, True),
]


def _build(B, kind, N, C, dcf, seed=0):
    rs = np.random.RandomState(seed)
    coord = _traj(kind, N)
    w = sqrt_dcf(coord) if dcf else None
    maps = synth.unit_rss_maps(rs, N, C)
    A = sense_operator_fused(B, N, coord, maps, 2.0, weights=w)
    return A, coord, maps, w


@pytest.mark.parametrize("kind,N,C,dcf", CASES)
def test_toeplitz_against_oracle_and_gridded(B, kind, N, C, dcf):
    A, coord, maps, w = _build(B, kind, N, C, dcf)
    T = toeplitz_normal(A)
    assert T.shape == (int(np.prod(N)),) * 2
    K, s2, L = R.toeplitz_operator(N, coord, maps, w)
    assert T._tdev.L == L
    x = synth.rand64c(np.random.RandomState(1), int(np.prod(N)), 1)
    got = T * x
    want = R.apply(K, N, maps, x, s2)
    assert R.rel(got, want) <= 1e-5
    aha = normal_operator(A) * x
    # the gridded operator is itself ~1.7e-2 from the exact model on the random trajectory (test_toeplitz_oracle.py,
    # where T is the closer of the two); the two differ by about that much
    assert R.rel(got, aha) <= (3e-2 if kind == "random" else 2e-2)


def test_self_adjoint_alpha_beta_determinism(B):
    N = (16, 16, 16)
    A, coord, maps, w = _build(B, "koosh", N, 4, True)
    T = toeplitz_normal(A)
    rs = np.random.RandomState(2)
    x, y = synth.rand64c(rs, 4096, 1), synth.rand64c(rs, 4096, 1)
    tx, ty = T * x, T * y
    assert abs(np.vdot(y, tx) - np.vdot(ty, x)) <= 1e-6 * np.linalg.norm(tx) * np.linalg.norm(y)
    # bit-identical: two applies, and a second node built independently
    assert np.array_equal(tx, T * x)
    assert np.array_equal(tx, toeplitz_normal(A) * x)
    # alpha / beta; beta = 0 never reads y
    xd, yd = B.copy_array(x), B.copy_array(y)
    T.eval(yd, xd, alpha=0.5 - 0.25j, beta=2.0)
    np.testing.assert_allclose(yd.to_host(), (0.5 - 0.25j) * tx + 2.0 * y, rtol=0, atol=1e-5 * np.abs(tx).max())
    nan = B.copy_array(np.full((4096, 1), np.nan, dtype=np.complex64, order='F'))
    T.eval(nan, xd, alpha=1.0, beta=0.0)
    out = nan.to_host()
    assert np.isfinite(out).all() and np.array_equal(out, tx)


def test_cg_against_numpy_and_graph(B):
    N = (16, 16, 16)
    A, coord, maps, w = _build(B, "koosh", N, 4, True)
    T = toeplitz_normal(A)
    K, s2, L = R.toeplitz_operator(N, coord, maps, w)
    rs = np.random.RandomState(5)
    y = synth.rand64c(rs, A.shape[0], 1)
    b = A.H * y
    b = (b / np.abs(b).max()).astype(np.complex64)
    lam = 0.05 * float(np.linalg.norm(T * b) / np.linalg.norm(b))
    xs = np.zeros_like(b, order='F')
    B.cg(T, b, xs, lamda=lam, maxiter=50, tol=0.0)
    xg = np.zeros_like(b, order='F')
    B.cg(T, b, xg, lamda=lam, maxiter=50, tol=0.0, graph=True)
    assert np.array_equal(xs, xg)

    def op(out, inp):
        out[...] = R.apply(K, N, maps, inp, s2).reshape(out.shape)
    xo = Kn.cg(op, b.astype(np.complex128), np.zeros(b.shape, np.complex128), lamda=lam, tol=0.0, maxiter=50)
    assert R.rel(xs, xo) <= 1e-5


def test_coil_shards_sum_to_whole(B):
    N, C = (16, 16, 16), 4
    A, coord, maps, w = _build(B, "koosh", N, C, False)

    class StubTeam(object):
        def __init__(self):
            self.vals = []

        def allreduce(self, v):                    # both shards run in this process: the sum is twice the value
            return 2.0 * v

    x = synth.rand64c(np.random.RandomState(7), 4096, 1)
    whole = toeplitz_normal(A) * x
    parts = 0
    for sl in (slice(0, 2), slice(2, 4)):
        As = sense_operator_fused(B, N, coord, np.asfortranarray(maps[..., sl]), 2.0)
        parts = parts + toeplitz_normal(As, team=StubTeam()) * x
    assert R.rel(parts, whole) <= 1e-6


def test_errors(B):
    N = (16, 16, 16)
    A, coord, maps, w = _build(B, "koosh", N, 2, False)
    T = toeplitz_normal(A)
    with pytest.raises(TypeError):
        toeplitz_normal(normal_operator(sense_operator_device(B, N, coord, maps, 2.0)))
    with pytest.raises(TypeError):
        toeplitz_normal(object())
    with pytest.raises(NotImplementedError):
        T._eval(None, B.copy_array(np.zeros((4096, 1), np.complex64, order='F')), left=False)
    with pytest.raises(ValueError):
        T * np.zeros((4096, 2), np.complex64, order='F')
    # an image whose padded grid needs more than the passes serve (2N - 1 > 512)
    from indigo_b200.fused import toeplitz_grid
    with pytest.raises(RuntimeError):
        toeplitz_grid((300, 16, 16))
    with pytest.raises(RuntimeError):
        toeplitz_normal(sense_operator_fused(B, (256, 256, 1), synth.radial_2d(nspokes=16, nread=512),
                                             synth.unit_rss_maps(np.random.RandomState(0), (256, 256, 1), 2), 2.0))


def test_fuse_transform_tree():
    """The tree of examples/pics.py:92-95, fused by fuse_transform, then made Toeplitz."""
    from indigo_b200.fused import fuse_transform
    from indigo_b200.sense import sense_operator
    try:
        from refenv import b200_reference_backend
        Bref = b200_reference_backend(0)
    except ImportError as e:
        pytest.skip("reference package unavailable: %s" % e)
    rs = np.random.RandomState(0)
    N, C = (16, 16, 16), 4
    coord = synth.kooshball_3d(nspokes=256, nread=32)
    maps = synth.unit_rss_maps(rs, N, C)
    w = sqrt_dcf(coord)
    A = sense_operator(Bref, N, coord, maps, 2.0, weights=w, recipe=[fuse_transform(Bref)])
    assert type(A).__name__ == "FusedSenseNUFFT"
    T = toeplitz_normal(A)
    x = synth.rand64c(rs, 4096, 1)
    K, s2, L = R.toeplitz_operator(N, coord, maps, w)
    assert R.rel(T * x, R.apply(K, N, maps, x, s2)) <= 1e-5
    assert R.rel(T * x, normal_operator(A) * x) <= 2e-2
