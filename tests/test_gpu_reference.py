"""
The drop-in claim, tested on the reference itself (SURVEY.md section 8 row a9, BASELINE.json north_star:
"operator trees built in operators.py ... run unchanged").

Everything here runs the UNMODIFIED reference package (tests/refenv.py: /root/reference in the build
container, oracle/_ref/reference_pkg.zip on the GPU box) with `indigo_b200.register()` applied -- the
monkey-patch equivalent of the two-line upstream patch in INTEGRATION.md:

  * `indigo.backends.get_backend('b200')` / `available_backends()` (backends/__init__.py:6-64);
  * the SENSE tree of examples/pics.py:92-95 built by the reference's own B.NUFFT / KronI / VStack / Diag,
    rewritten by the script's own -O3 recipe (exec'd from the reference's text) and by
    indigo_b200.refcompat.reference_sense_recipe, walked by the reference's operators.py on the B200
    kernels: exactly six Backend calls per A^H A, A x / A^H y / A^H A x and 50 CG iterates against the oracle;
  * `apgd` + `max` (examples/mpi.py:63-79) and `HStack` (examples/phasespace.py) with value checks against
    the reference's NumpyBackend running the same code;
  * the reference's own test modules with INDIGO_TEST_BACKENDS=b200 (sub-sampled here; the full run is
    tools/run_reference_suites.py, result in profiles/).
"""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as spp

from indigo_b200 import synth
from indigo_b200.sense import sense_operator, normal_operator, sqrt_dcf
from oracle import sense as osense, np_oracle as K
from refenv import reference, b200_reference_backend, numpy_backend, pics_recipe

pytestmark = pytest.mark.gpu
C64 = np.dtype('complex64')
TOL = 1e-5


def relerr(a, b):
    a = np.asarray(a).ravel(order='F'); b = np.asarray(b).ravel(order='F')
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


@pytest.fixture(scope="module")
def B():
    return b200_reference_backend(0)


@pytest.fixture(scope="module")
def SB():
    """Standalone build (no reference package involved)."""
    from indigo_b200 import B200Backend
    return B200Backend(0)


def test_registered_with_the_reference_lookup(B, monkeypatch):
    indigo = reference()
    from indigo.backends import get_backend, available_backends
    from indigo.backends.backend import Backend
    assert isinstance(B, Backend) and type(B).__name__ == "B200Backend"
    assert isinstance(B.zero_array((4,), C64), Backend.dndarray)
    monkeypatch.setenv("INDIGO_TEST_BACKENDS", "b200")
    assert [c.__name__ for c in available_backends()] == ["B200Backend"]
    monkeypatch.setenv("INDIGO_TEST_BACKENDS", "np")
    assert "B200Backend" not in [c.__name__ for c in available_backends()]
    assert type(get_backend('numpy')).__name__ == "NumpyBackend"          # the original lookup still works
    with pytest.raises(ValueError):
        get_backend('quantumcomputer')


class CallCounter(object):
    """Counts the Backend calls an evaluation makes (instance-level wrappers, removed on exit)."""
    NAMES = ("ccsrmm", "ccsrmm_packed", "fftn", "ifftn", "axpby", "scale", "cgemm", "csymm", "onemm", "cdiamm")

    def __init__(self, B):
        self.B, self.calls = B, []

    def __enter__(self):
        self.NAMES = tuple(n for n in self.NAMES if hasattr(self.B, n))
        for n in self.NAMES:
            fn = getattr(self.B, n)
            setattr(self.B, n, (lambda f, nm: lambda *a, **k: (self.calls.append(nm), f(*a, **k))[1])(fn, n))
        return self

    def __exit__(self, *exc):
        for n in self.NAMES:
            delattr(self.B, n)


def _problem(seed=5, N=(16, 12, 8), C=4, nsamp=500, weighted=True):
    rs = np.random.RandomState(seed)
    coord = synth.random_3d(rs, nsamp)
    maps = synth.unit_rss_maps(rs, N, C)
    w = sqrt_dcf(coord) if weighted else None
    return rs, N, C, coord, maps, w


@pytest.mark.parametrize("recipe_from", ["examples/pics.py", "indigo_b200.refcompat"])
def test_pics_tree_runs_unchanged_on_b200(B, recipe_from):
    from indigo_b200.refcompat import reference_sense_recipe
    rs, N, C, coord, maps, w = _problem()
    recipe = pics_recipe(3) if recipe_from == "examples/pics.py" else reference_sense_recipe(3)
    A = sense_operator(B, N, coord, maps, 2.0, weights=w, recipe=recipe)
    import indigo.operators as iop
    assert isinstance(A, iop.Product)                                      # the reference's own node classes
    ref = osense.SenseOperator(N, coord, maps, 2.0, weights=w)
    nvox = int(np.prod(N))
    x = synth.rand64c(rs, nvox, 1)
    y = synth.rand64c(rs, ref.M * C, 1)
    assert relerr(A * x, ref.forward(x)) < TOL
    assert relerr(A.H * y, ref.adjoint(y)) < TOL
    AHA = normal_operator(A)
    xd, yd = B.copy_array(x), B.zero_array((nvox, 1), C64)
    with CallCounter(B) as cc:
        AHA.eval(yd, xd)
    assert relerr(yd.to_host(), ref.normal(x)) < TOL
    sparse = [c for c in cc.calls if c.startswith("ccsrmm")]
    assert len(sparse) == 4 and cc.calls.count("fftn") == 1 and cc.calls.count("ifftn") == 1, cc.calls
    assert len(cc.calls) == 6, cc.calls                                     # SURVEY.md section 3.1: six Backend calls
    # evaluated inside the arena reserved by Optimize (transforms.py:62-78): slices with huge leading dims
    assert getattr(B, '_scratch', None) is not None and B._scratch_pos == 0


def test_every_recipe_level_agrees(B):
    """-O1 .. -O3 of the same tree give the same operator (the reference's rewrites are semantics-preserving on
    this backend too: Kron batching, VStack/Adjoint scale-then-accumulate, beta=0 into the uninitialised arena).
    (-O0 through optimize() fails in the reference itself: its arena estimate for the unrewritten tree is 0 bytes.)"""
    rs, N, C, coord, maps, w = _problem(seed=8, weighted=False)
    ref = osense.SenseOperator(N, coord, maps, 2.0)
    x = synth.rand64c(rs, int(np.prod(N)), 1)
    y = synth.rand64c(rs, ref.M * C, 1)
    for level in (1, 2, 3):
        A = sense_operator(B, N, coord, maps, 2.0, recipe=pics_recipe(level))
        assert relerr(A * x, ref.forward(x)) < TOL, level
        assert relerr(A.H * y, ref.adjoint(y)) < TOL, level


def test_cg_50_iterates_through_the_reference_tree(B):
    rs, N, C, coord, maps, w = _problem(seed=12, N=(16, 16, 12), C=6, nsamp=900)
    A = sense_operator(B, N, coord, maps, 2.0, weights=w, recipe=pics_recipe(3))
    AHA = normal_operator(A)
    ref = osense.SenseOperator(N, coord, maps, 2.0, weights=w)
    x = synth.rand64c(rs, int(np.prod(N)), 1)
    want = ref.normal(x)
    b = (want / np.abs(want).max()).astype(C64)
    lam = 0.05 * osense.spectral_norm(ref)
    mine, theirs = [], []
    B.cg(AHA, b, np.zeros_like(b, order='F'), lamda=lam, maxiter=50, tol=0.0, iterates=mine)
    K.cg(ref.normal_into, b, np.zeros_like(b), lamda=lam, tol=0.0, maxiter=50, iterates=theirs)
    assert len(mine) == 50
    worst = max(relerr(m, t) for m, t in zip(mine, theirs))
    assert worst < TOL, worst
    # the reference's own solver (Backend.cg, host scalars through dot/norm2) on the same kernels
    x2 = np.zeros_like(b, order='F')
    super(type(B), B).cg(AHA, b, x2, lamda=lam, maxiter=50, tol=0.0)
    assert relerr(x2, theirs[-1]) < TOL


def test_apgd_values_match_the_numpy_backend(B):
    """examples/mpi.py:46-79 in miniature: apgd on min ||A x - y||^2 s.t. x >= 0 with A = D * S (KronI of Eye - One/pz,
    segment SpMatrix); the reference's apgd driver on the B200 primitives (axpby, max, ccsrmm) against the
    same driver on the reference's NumpyBackend after 1, 5 and 25 iterations."""
    rs = np.random.RandomState(2)
    npf, px, pz, nimg = 3, 4, 6, 40
    cols = rs.randint(0, nimg, npf * px * pz)
    Sm = spp.coo_matrix((np.ones(cols.size, dtype=C64), (np.arange(cols.size), cols)), shape=(cols.size, nimg))
    Y = synth.rand64c(rs, cols.size, 1)

    def solve(Bk, iters):
        S = Bk.SpMatrix(Sm.conjugate().transpose(), name='segment').H
        # DC removal per partial field of view (mpi.py:56 builds it from Eye - One/pz; realised here as one sparse
        # matrix because the reference NumpyBackend's onemm cannot evaluate that Kron, np.py:95-97)
        D = Bk.SpMatrix(spp.kron(spp.eye(npf * px), np.eye(pz) - np.ones((pz, pz)) / pz).astype(C64), name='dc')
        A = (D * S).optimize()
        AHA = A.H * A
        AHy_d = Bk.copy_array(A.H * Y)

        def proxg(x_d, alpha):
            Bk.max(0, x_d)

        def gradf(gf, x):
            AHA.eval(gf, x)
            Bk.axpby(1, gf, -1, AHy_d)

        X = np.zeros((nimg, 1), dtype=C64, order='F')
        Bk.apgd(gradf, proxg, 0.05, X, maxiter=iters)
        return X

    NB = numpy_backend()
    for iters in (1, 5, 25):
        got, want = solve(B, iters), solve(NB, iters)
        assert np.abs(want).max() > 0
        assert relerr(got, want) < TOL, (iters, relerr(got, want))
        assert got.real.min() >= 0 and got.imag.min() >= 0


@pytest.mark.parametrize("stack,K,alpha,beta", [(1, 1, 1, 0), (2, 8, 0.5, 1), (3, 9, 1, 0.5), (3, 17, 0.5, 0)])
def test_hstack_values(B, stack, K, alpha, beta):
    """operators.py:458-498 (HStack forward = scale(y, beta) then accumulate children with beta=1; adjoint slices x)."""
    rs = np.random.RandomState(stack * 10 + K)
    M, N = 6, 7
    mats = [(spp.random(M, N, density=0.5, random_state=rs) + 1j * spp.random(M, N, density=0.5, random_state=rs)).astype(C64)
            for _ in range(stack)]
    H = B.HStack([B.SpMatrix(m) for m in mats])
    Hm = spp.hstack(mats).toarray()
    x, y = synth.rand64c(rs, N * stack, K), synth.rand64c(rs, M, K)
    xd, yd = B.copy_array(x), B.copy_array(y)
    H.eval(yd, xd, alpha=alpha, beta=beta)
    np.testing.assert_allclose(yd.to_host(), alpha * (Hm @ x) + beta * y, atol=1e-5)
    u, v = synth.rand64c(rs, M, K), synth.rand64c(rs, N * stack, K)
    ud, vd = B.copy_array(u), B.copy_array(v)
    H.H.eval(vd, ud, alpha=alpha, beta=beta)
    np.testing.assert_allclose(vd.to_host(), alpha * (Hm.conj().T @ u) + beta * v, atol=1e-5)


def test_int64_indices_split_into_column_blocks(SB, monkeypatch):
    """backend.py:549-550 keeps scipy's index dtype; cfg4's P on one GPU has 2.3 G columns and arrives with int64
    indices.  Here the block width is forced down so that a small int64 matrix takes the same path."""
    B = SB
    rs = np.random.RandomState(4)
    M, N, K = 37, 101, 5
    A = (spp.random(M, N, density=0.2, random_state=rs, format='csr') +
         1j * spp.random(M, N, density=0.2, random_state=rs, format='csr')).astype(C64).tocsr()
    A.sort_indices()
    A64 = spp.csr_matrix(A.shape, dtype=C64)
    A64.data, A64.indices, A64.indptr = A.data, A.indices.astype(np.int64), A.indptr.astype(np.int64)
    monkeypatch.setattr(B.csr_matrix, "max_block_cols", 32)
    Ad = B.csr_matrix(B, A64)
    # (scipy narrows the indices of a matrix this small back to int32 inside astype(), exactly as it does for the
    # reference; above 2^31 columns they stay int64 and the same block path is taken)
    assert len(Ad._blocks) == 4
    np.testing.assert_array_equal(Ad.colInds.to_host(), A.indices)
    dense = A.toarray()
    x, y = synth.rand64c(rs, N, K), synth.rand64c(rs, M, K)
    xd, yd = B.copy_array(x), B.copy_array(y)
    Ad.forward(yd, xd, alpha=0.5, beta=1.5)
    np.testing.assert_allclose(yd.to_host(), 0.5 * (dense @ x) + 1.5 * y, atol=1e-5)
    yd = B.copy_array(np.full((M, K), np.nan, dtype=C64, order='F'))
    Ad.forward(yd, xd)
    np.testing.assert_allclose(yd.to_host(), dense @ x, atol=1e-5)
    u, v = synth.rand64c(rs, M, K), synth.rand64c(rs, N, K)
    ud, vd = B.copy_array(u), B.copy_array(v)
    Ad.adjoint(vd, ud, alpha=2.0, beta=0.5)
    np.testing.assert_allclose(vd.to_host(), 2.0 * (dense.conj().T @ u) + 0.5 * v, atol=1e-5)
    frac = np.count_nonzero(np.diff(A.indptr)) / M
    assert abs(Ad._row_frac - frac) < 1e-12 and abs(Ad._col_frac - np.count_nonzero(np.bincount(A.indices, minlength=N)) / N) < 1e-12


def test_dia_matrix_with_scipy_chosen_width(SB):
    """np.py:129-136 accepts whatever width scipy gives dia.data: todia() of a matrix with an empty last column is
    narrower than k, diags() with positive offsets on a wide matrix can be wider than the row count."""
    B = SB
    rs = np.random.RandomState(9)
    A1 = spp.csr_matrix(np.array([[1, 2, 0, 0], [0, 3, 4, 0], [0, 0, 5, 0], [0, 0, 0, 0]], dtype=C64)).todia()
    assert A1.data.shape[1] < A1.shape[1]
    A2 = spp.diags([synth.rand64c(rs, 5), synth.rand64c(rs, 7), synth.rand64c(rs, 3)], [0, 2, -2], shape=(5, 9)).todia()
    A3 = spp.dia_matrix((synth.rand64c(rs, 2, 12), np.array([1, -3])), shape=(6, 8))      # data wider than k
    for A in (A1, A2, A3):
        A = A.astype(C64)
        Ad = B.dia_matrix(B, A)
        m, k = A.shape
        dense = A.toarray()
        x, y = synth.rand64c(rs, k, 3), synth.rand64c(rs, m, 3)
        xd, yd = B.copy_array(x), B.copy_array(y)
        Ad.forward(yd, xd, alpha=0.5, beta=1.0)
        np.testing.assert_allclose(yd.to_host(), 0.5 * (dense @ x) + y, atol=1e-5)
        u, v = synth.rand64c(rs, m, 3), synth.rand64c(rs, k, 3)
        ud, vd = B.copy_array(u), B.copy_array(v)
        Ad.adjoint(vd, ud, alpha=1.0, beta=0.0)
        np.testing.assert_allclose(vd.to_host(), dense.conj().T @ u, atol=1e-5)


def test_two_dimensional_row_weights_follow_sample_order():
    """Weights given as an (nread, nspokes) array: B.Diag flattens them in column-major order (the sample order of
    coord.reshape((3, -1), order='F')); the fused and device-built operators must apply them to the same samples."""
    from indigo_b200 import B200Backend
    from indigo_b200.fused import sense_operator_fused
    from indigo_b200.sense import sense_operator_device
    SB = B200Backend(0)
    rs = np.random.RandomState(6)
    N, C = (16, 16, 16), 2
    coord = synth.kooshball_3d(nspokes=24, nread=32)
    maps = synth.unit_rss_maps(rs, N, C)
    w2 = np.ascontiguousarray(0.5 + rs.rand(*coord.shape[1:]).astype(np.float32))           # C-ordered 2-D weights
    ref = osense.SenseOperator(N, coord, maps, 2.0, weights=np.asfortranarray(w2).flatten(order='A'))
    x = synth.rand64c(rs, int(np.prod(N)), 1)
    for make in (sense_operator_fused, sense_operator_device):
        A = make(SB, N, coord, maps, 2.0, weights=w2)
        assert relerr(A * x, ref.forward(x)) < TOL, make.__name__
        assert relerr(normal_operator(A) * x, ref.normal(x)) < TOL, make.__name__


@pytest.mark.parametrize("suite,stride,minimum", [("indigo/backends/test_backends.py", 5, 850),
                                                  ("indigo/test_operators.py", 13, 850),
                                                  ("indigo/test_transforms.py", 1, 100)])
def test_reference_own_suites_on_b200(suite, stride, minimum):
    """The reference's own test modules with INDIGO_TEST_BACKENDS=b200, every `stride`-th test (all of them:
    tools/run_reference_suites.py; counts recorded in profiles/r02_reference_suites.json)."""
    reference()
    import refshim
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from run_reference_suites import run_suite
    forced = os.environ.get("IB200_REFSUITE_TEST_STRIDE")
    if forced:
        stride, minimum = int(forced), 1
    r = run_suite(refshim.reference_root(), suite, stride=stride, timeout=1500)
    assert r["rc"] == 0, (r["summary"], r["failures"], r["output_tail"])
    assert r["counts"].get("failed", 0) == 0 and r["counts"].get("passed", 0) >= minimum, r["summary"]
