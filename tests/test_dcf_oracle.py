"""
Pipe-Menon density compensation in numpy/float64 (tests/dcf_ref.py), no device: the iteration reaches its fixed
point I I^T w = 1 on the trajectories the package generates, the weights have the known radial profiles, and they
come back in the caller's sample order.
"""
import numpy as np
import pytest

from indigo_b200 import synth
import dcf_ref as D

TRAJ = {
    "koosh": lambda: synth.kooshball_3d(nspokes=256, nread=32),
    "spirals": lambda: synth.stack_of_spirals(nz=8, nleaves=8, nread=512, turns=4.0),
    "random": lambda: synth.random_3d(np.random.RandomState(3), 4000),
}


@pytest.mark.parametrize("kind", sorted(TRAJ))
def test_fixed_point_residual(kind):
    I = D.interp((16, 16, 8), TRAJ[kind]())
    hist = []
    w = D.pipe_menon(I, 30, hist)
    assert len(hist) == 30 and hist[0] > 10.0          # w = 1 is far from the fixed point on all three
    assert D.residual(I, w) < 2e-2                      # 1.2e-2 (spirals) to 1.7e-2 (random)
    assert (w > 0).all()


def _profile(N, coord, power):
    """Largest relative deviation of the spoke-averaged weights from c |k|^power over 0.1 < |k| < 0.4 (c the
    median ratio).  Single samples deviate more: Pipe-Menon weights ripple from spoke to spoke (about 10-20 %
    per sample on the 2-D case) while the average over the spokes at one radius follows |k|^power."""
    w = D.dcf(N, coord)
    nread = coord.shape[1]
    r = np.abs((np.arange(nread) - nread // 2) / nread)
    band = (r > 0.1) & (r < 0.4)
    ratio = w.mean(axis=1)[band] / r[band] ** power
    return float(np.abs(ratio / np.median(ratio) - 1).max())


def test_radial_2d_weights_follow_k():
    assert _profile((64, 64, 1), synth.radial_2d(nspokes=96, nread=128), 1) <= 0.10      # 3.2e-2


def test_kooshball_weights_follow_k_squared():
    assert _profile((16, 16, 16), synth.kooshball_3d(nspokes=256, nread=32), 2) <= 0.15  # 0.114


def test_weights_in_user_sample_order():
    coord = synth.kooshball_3d(nspokes=64, nread=32)
    rs = np.random.RandomState(4)
    pr, ps = rs.permutation(32), rs.permutation(64)
    w = D.dcf((16, 16, 16), coord, maxiter=10)
    assert w.shape == (32, 64)
    wp = D.dcf((16, 16, 16), coord[:, pr][:, :, ps], maxiter=10)
    np.testing.assert_allclose(wp, w[pr][:, ps], rtol=1e-10, atol=0)
