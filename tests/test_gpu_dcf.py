"""
Pipe-Menon density compensation on the device (indigo_b200.sense.pipe_menon_dcf, csrc/dcf.cu) against the
numpy/float64 restatement (tests/dcf_ref.py), against one I I^T w through the complex gridding path of the fused
operator, and in use as row weights of the fused operator, its Toeplitz form and CG.
"""
import numpy as np
import pytest

from indigo_b200 import synth, pipe_menon_dcf
from indigo_b200.fused import sense_operator_fused, toeplitz_normal
from indigo_b200.sense import normal_operator
from oracle import sense as osense
import dcf_ref as D

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    from indigo_b200 import B200Backend
    return B200Backend(0)


CASES = {  # name: (N, trajectory)
    "koosh": ((16, 16, 16), lambda: synth.kooshball_3d(nspokes=256, nread=32)),
    "random": ((16, 16, 16), lambda: synth.random_3d(np.random.RandomState(3), 4000)),
    "spirals": ((16, 16, 8), lambda: synth.stack_of_spirals(nz=8, nleaves=8, nread=512, turns=4.0)),
    "anisotropic": ((32, 16, 26), lambda: synth.kooshball_3d(nspokes=512, nread=64)),
    "radial2d": ((64, 64, 1), lambda: synth.radial_2d(nspokes=96, nread=128)),          # grid 128 x 128 x 2
    "noplan": ((20, 12, 10), lambda: synth.random_3d(np.random.RandomState(5), 3000)),  # grid 40 x 24 x 20
    "noplan_odd": ((17, 12, 10), lambda: synth.random_3d(np.random.RandomState(6), 3000)),  # grid 34 x 24 x 20
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_against_restatement(B, case):
    N, traj = CASES[case]
    coord = traj()
    if case.startswith("noplan"):                        # the fused operator has no FFT passes for this grid
        maps = synth.unit_rss_maps(np.random.RandomState(0), N, 2)
        with pytest.raises(RuntimeError):
            sense_operator_fused(B, N, coord, maps, 2.0)
    w = pipe_menon_dcf(B, N, coord)
    assert w.dtype == np.float32 and w.shape == coord.shape[1:]
    want = D.dcf(N, coord)
    assert D.rel(w, want) <= 1e-4


def test_bit_identical_and_history(B):
    N, traj = CASES["koosh"]
    coord = traj()
    hist = []
    w1 = pipe_menon_dcf(B, N, coord, history=hist)
    w2 = pipe_menon_dcf(B, N, coord)
    assert np.array_equal(w1, w2)
    assert np.array_equal(w2, pipe_menon_dcf(B, N, coord))
    assert len(hist) == 30 and all(b < a for a, b in zip(hist, hist[1:]))
    want = []
    D.dcf(N, coord, history=want)
    np.testing.assert_allclose(hist, want, rtol=1e-3)


def test_user_sample_order(B):
    N, traj = CASES["koosh"]
    coord = traj()
    rs = np.random.RandomState(4)
    pr, ps = rs.permutation(coord.shape[1]), rs.permutation(coord.shape[2])
    w = pipe_menon_dcf(B, N, coord)
    wp = pipe_menon_dcf(B, N, coord[:, pr][:, :, ps])
    assert D.rel(wp, w[pr][:, ps]) <= 1e-5


def test_against_complex_gridding_path(B):
    """I I^T w through the fused operator's own gridding: a 2-coil operator without row weights, maps (1, 0),
    k-space [w, 0] -> samples_to_grid -> grid_to_samples (no FFT), divided by the scale^2 the records carry."""
    N, traj = CASES["koosh"]
    coord = traj()
    maps = np.zeros(N + (2,), dtype=np.complex64, order='F')
    maps[..., 0] = 1
    d = sense_operator_fused(B, N, coord, maps, 2.0)._dev
    assert d.tiles is not None and d.ksp_sorted
    lib, s, M = B._lib, B._stream, d.M
    scl = float(np.float32(np.complex64(1.0 / np.sqrt(np.prod(d.oN))).real))

    def iit(w):
        x = np.zeros((M, 2), dtype=np.complex64, order='F')
        x[:, 0] = w.reshape(-1, order='F')
        xd, yd = B.copy_array(x), B.empty_array((M, 2), np.complex64)
        lib.interleave_rows(s, M, 2, xd.ptr, M, d.ksp.ptr, 2, d.pos.ptr)
        d.samples_to_grid()
        d.grid_to_samples()
        lib.deinterleave_rows(s, M, 2, d.ksp.ptr, 2, 0.0, 0.0, yd.ptr, M, d.pos.ptr)
        y = yd.to_host()
        assert np.abs(y[:, 1]).max() == 0 and np.abs(y[:, 0].imag).max() <= 1e-6 * np.abs(y[:, 0].real).max()
        return y[:, 0].real.astype(np.float64) / (scl * scl)

    w1 = pipe_menon_dcf(B, N, coord, maxiter=1).reshape(-1, order='F').astype(np.float64)     # 1 / (I I^T 1)
    w2 = pipe_menon_dcf(B, N, coord, maxiter=2).reshape(-1, order='F').astype(np.float64)     # w1 / (I I^T w1)
    assert D.rel(1.0 / w1, iit(np.ones(M))) <= 1e-5
    assert D.rel(w1 / w2, iit(w1.astype(np.float32))) <= 1e-5


def test_weights_in_operators_and_cg(B):
    N, traj = CASES["koosh"]
    coord = traj()
    w = pipe_menon_dcf(B, N, coord)
    sw = np.sqrt(w)
    rs = np.random.RandomState(0)
    maps = synth.unit_rss_maps(rs, N, 4)
    A = sense_operator_fused(B, N, coord, maps, 2.0, weights=sw)
    ref = osense.SenseOperator(N, coord, maps, 2.0, weights=sw.reshape(-1, order='F'))
    x = synth.rand64c(rs, int(np.prod(N)), 1)
    AHA = normal_operator(A)
    assert D.rel(AHA * x, ref.normal(x)) <= 1e-5
    T = toeplitz_normal(A)
    assert D.rel(T * x, AHA * x) <= 2e-2
    b = A.H * synth.rand64c(rs, A.shape[0], 1)
    b = (b / np.abs(b).max()).astype(np.complex64)
    lam = 1e-2 * float(np.linalg.norm(AHA * b) / np.linalg.norm(b))
    for op in (AHA, T):
        xs = np.zeros_like(b, order='F')
        B.cg(op, b, xs, lamda=lam, maxiter=40, tol=0.0)
        r = (op * xs + lam * xs) - b
        assert np.linalg.norm(r) <= 1e-3 * np.linalg.norm(b)         # the oracle's CG: 2.3e-5 at 40 iterations


def test_errors(B):
    N, traj = CASES["koosh"]
    coord = traj()
    bad = coord.copy()
    bad[0, 3, 5] = np.nan
    with pytest.raises(ValueError):
        pipe_menon_dcf(B, N, bad)
    with pytest.raises(ValueError):
        pipe_menon_dcf(B, N, coord, maxiter=0)
    with pytest.raises(RuntimeError):
        pipe_menon_dcf(B, N, coord, width=4)             # 8 taps per axis: no separable records


def test_full_size_cfg3(B):
    """The cfg3 kooshball (6.8 M samples, grid 416^3): the kernels at the benchmarked size, 64-bit grid offsets."""
    coord = synth.kooshball_3d(16384, 416)
    hist = []
    w = pipe_menon_dcf(B, (208, 208, 208), coord, maxiter=10, history=hist)
    assert w.shape == (416, 16384) and np.isfinite(w).all() and (w >= 0).all()
    # measured on a B200: 1.07e4 for w = 1, 7.2e-3 after 9 iterations, 5.6e-3 after 30 (profiles/r04_dcf.md).  The
    # |k|^2 profile of the small case does not apply here: 16384 spokes sample a 416^3 grid below the Nyquist rate
    # away from the centre, where the weights flatten out
    assert hist[0] > 1e3 and all(b < a for a, b in zip(hist, hist[1:])) and hist[-1] < 1e-2
