"""
Seeded synthetic inputs of BASELINE.json's configurations (SURVEY.md section 8d).
Pure numpy, no device code: shared by tests, bench.py (both arms) and smoke().

Values follow indigo.util.rand64c (indigo/util.py:9-19): U[0,1) + i*U[0,1),
real part drawn first, each cast to float32 -- but from an explicit
RandomState so every run is reproducible (the reference never seeds).
"""
import numpy as np

C64 = np.dtype("complex64")


def rand64c(rs, *shape, order="F"):
    re = rs.rand(*shape).astype(np.float32)
    im = rs.rand(*shape).astype(np.float32)
    arr = (re + 1j * im).astype(np.complex64)
    return np.asfortranarray(arr) if order == "F" else arr


def unit_rss_maps(rs, N, C):
    """Coil sensitivities (N0,N1,N2,C), rand64c normalised to unit root-sum-of-squares."""
    m = rand64c(rs, *N, C)
    rss = np.sqrt((np.abs(m) ** 2).sum(axis=3, keepdims=True))
    return np.asfortranarray((m / rss).astype(np.complex64))


def birdcage_maps(N, C, r=1.5):
    """Deterministic, smooth coil sensitivities (N0,N1,N2,C), complex64, column-major, unit root-sum-of-squares: the
    birdcage model of sigpy.mri.birdcage_maps.  Coil c sits on a ring of radius r (image half-widths) around the z
    axis with magnitude 1/distance and phase atan2(x', -y') - 2 pi c / C.  For 3-D images (N2 > 1) the coils form
    rings of 8, stacked in z: coil c at angle 2 pi c / 8, height floor(c/8) - (ceil(C/8) - 1)/2, phase offset
    -2 pi (c + floor(c/8)) / 8.  Voxel i of an axis of n points sits at (i - n/2) / (n/2)."""
    N = tuple(int(v) for v in N)
    C = int(C)
    x, y, z = np.meshgrid(*[(np.arange(n) - n / 2.0) / (n / 2.0) for n in N], indexing='ij')
    out = np.empty(N + (C,), dtype=np.complex128)
    for c in range(C):
        if N[2] > 1:
            ang, cz = c * 2.0 * np.pi / 8, np.floor(c / 8) - 0.5 * (np.ceil(C / 8) - 1)
            phs = -(c + np.floor(c / 8)) * 2.0 * np.pi / 8
        else:
            ang, cz, phs = c * 2.0 * np.pi / C, 0.0, -c * 2.0 * np.pi / C
        xc, yc = x - r * np.cos(ang), y - r * np.sin(ang)
        zc = z - cz if N[2] > 1 else 0.0
        rr = np.sqrt(xc ** 2 + yc ** 2 + zc ** 2)
        out[..., c] = np.exp(1j * (np.arctan2(xc, -yc) + phs)) / rr
    out /= np.sqrt((np.abs(out) ** 2).sum(axis=3, keepdims=True))
    return np.asfortranarray(out.astype(np.complex64))


def radial_2d(nspokes=402, nread=512):
    """cfg1: in-plane radial, k = r*(cos t, sin t, 0), r in [-1/2,1/2), t_j = pi*j/nspokes.
    Returns coord (3, nread, nspokes) float64 (BART layout: ksp dims (1, nread, nspokes))."""
    r = (np.arange(nread) - nread // 2) / nread
    t = np.pi * np.arange(nspokes) / nspokes
    c = np.zeros((3, nread, nspokes))
    c[0] = r[:, None] * np.cos(t)[None, :]
    c[1] = r[:, None] * np.sin(t)[None, :]
    return c


def kooshball_3d(nspokes=16384, nread=416):
    """cfg3/4: 3-D radial with Fibonacci (golden-angle) spoke directions.
    Returns coord (3, nread, nspokes) float64."""
    j = np.arange(nspokes) + 0.5
    z = 1.0 - 2.0 * j / nspokes
    phi = np.pi * (1.0 + 5.0 ** 0.5) * j
    s = np.sqrt(np.maximum(0.0, 1.0 - z * z))
    d = np.stack([s * np.cos(phi), s * np.sin(phi), z])          # (3, nspokes)
    r = (np.arange(nread) - nread // 2) / nread                   # [-1/2, 1/2)
    return r[None, :, None] * d[:, None, :]


def stack_of_spirals(nz=128, nleaves=48, nread=2048, turns=16.0):
    """cfg5: Archimedean spiral interleaves in-plane, one stack per kz plane.
    Returns coord (3, nread, nleaves*nz) float64."""
    t = np.arange(nread) / nread
    rad = 0.5 * t
    c = np.zeros((3, nread, nleaves, nz))
    for l in range(nleaves):
        ang = 2.0 * np.pi * (turns * t + l / nleaves)
        c[0, :, l, :] = (rad * np.cos(ang))[:, None]
        c[1, :, l, :] = (rad * np.sin(ang))[:, None]
    c[2] = ((np.arange(nz) - nz // 2) / nz)[None, None, :]
    return c.reshape(3, nread, nleaves * nz)


def random_3d(rs, npts):
    """Uniform random sample positions in [-1/2, 1/2)^3, (3, npts, 1)."""
    return (rs.rand(3, npts, 1) - 0.5)


# Modified 3-D Shepp-Logan ellipsoids (Kak and Slaney's table with Toft's contrasts), rotations about z only:
#   intensity, semi-axes (a, b, c), centre (x0, y0, z0), rotation phi in degrees, on [-1, 1]^3.
_PHANTOM = (
    (1.0, .6900, .920, .810, 0.0, 0.0, 0.0, 0.0),
    (-.8, .6624, .874, .780, 0.0, -.0184, 0.0, 0.0),
    (-.2, .1100, .310, .220, .22, 0.0, 0.0, -18.0),
    (-.2, .1600, .410, .280, -.22, 0.0, 0.0, 18.0),
    (.1, .2100, .250, .410, 0.0, .35, -.15, 0.0),
    (.1, .0460, .046, .050, 0.0, .1, .25, 0.0),
    (.1, .0460, .046, .050, 0.0, -.1, .25, 0.0),
    (.1, .0460, .023, .050, -.08, -.605, 0.0, 0.0),
    (.1, .0230, .023, .020, 0.0, -.606, 0.0, 0.0),
    (.1, .0230, .046, .020, .06, -.605, 0.0, 0.0),
)


def phantom(N):
    """Deterministic piecewise-constant Shepp-Logan-like phantom of shape N = (N0, N1, N2), complex64, column-major
    (x = axis 0 fastest).  Voxel i of an axis of n points sits at (2 i - n) / n in [-1, 1).  For N2 == 1 it is the
    2-D phantom: the ellipses (a, b, x0, y0, phi) of the same table, with no z extent."""
    N = tuple(int(v) for v in N)
    ax = [(2.0 * np.arange(n) - n) / n for n in N]
    X, Y, Z = np.meshgrid(ax[0], ax[1], ax[2], indexing='ij')
    img = np.zeros(N, dtype=np.float64)
    for amp, a, b, c, x0, y0, z0, phi in _PHANTOM:
        if N[2] == 1 and z0 != 0.0:
            continue
        t = np.deg2rad(phi)
        u = (X - x0) * np.cos(t) + (Y - y0) * np.sin(t)
        v = -(X - x0) * np.sin(t) + (Y - y0) * np.cos(t)
        r = (u / a) ** 2 + (v / b) ** 2
        if N[2] > 1:
            r = r + ((Z - z0) / c) ** 2
        img[r <= 1.0] += amp
    return np.asfortranarray(img.astype(np.complex64))


def random_csr(rs, rows, cols, nnz_per_row):
    """cfg2: `nnz_per_row` distinct uniformly-random sorted columns per row, rand64c values.
    Returns (indptr int32, indices int32, data complex64)."""
    r = int(nnz_per_row)
    # distinct columns per row: sample with a stride trick (jittered stratified draw)
    width = cols // r
    base = (np.arange(r, dtype=np.int64) * width)[None, :]
    idx = base + (rs.rand(rows, r) * width).astype(np.int64)
    indptr = (np.arange(rows + 1, dtype=np.int64) * r).astype(np.int32)
    data = rand64c(rs, rows * r, order="C")
    return indptr, idx.astype(np.int32).reshape(-1), data
