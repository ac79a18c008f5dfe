"""
Construction of the non-Cartesian SENSE operator exactly as examples/pics.py
does it (pics.py:92-95 and its -O1..-O3 recipe, pics.py:179-193), for any
backend object that offers the reference's builder interface (B200Backend, the
reference's own backends, or the test backends).

    A = KronI(C, NUFFT(M, N, coord)) * VStack_c Diag(maps_c)

After the -O3 recipe one `A.H * A` evaluation is the six backend calls of
SURVEY.md section 3.1:
    ccsrmm(P^H, adjoint) -> fftn -> ccsrmm(G') -> ccsrmm(G', adjoint) -> ifftn -> ccsrmm(P^H)
"""
import collections

import numpy as np

_C64 = np.dtype('complex64')

# Tiles of the gridding structures of the fused operator and of the density compensation.  The adjoint gather's
# kernels (block entries, x-runs) assume GRID_TILE = 4 x 4 x 4.
SAMPLE_TILE = (8, 8, 8)     # samples are sorted by the grid tile of this size they fall into,
SAMPLE_SUPER = (8, 8, 8)    # tiles grouped into super-tiles of this many tiles (64^3 points: L2-sized working set)
GRID_TILE = (4, 4, 4)       # tile-major grid order: rows of the stored adjoint, blocks of the adjoint gather


def _ops_of(B):
    """Operator module of B's family: indigo_b200.linop for the standalone build, the reference's
    indigo.operators when B was built on the reference's Backend (indigo_b200.register())."""
    ops = getattr(B, 'ops', None)
    if ops is None:
        import indigo.operators as ops
    return ops


def sense_operator(B, N, coord, maps, oversamp=2.0, level=3, weights=None, recipe=None, width=3, n=128):
    """Returns the optimised forward operator A (image -> multi-coil k-space), built by the
    REFERENCE's own builders and rewritten by its Transform machinery: B must be a backend
    built on `indigo.backends.backend.Backend` (indigo_b200.register() / make_backend_class).

    N      image shape (N0, N1, N2)
    coord  (3, nread, nspokes...) sample positions in cycles/FOV, [-1/2, 1/2)
    maps   (N0, N1, N2, C) coil sensitivities
    weights optional per-sample row weights (sqrt density compensation), applied as
            Diag(w) * NUFFT like test_compat.py:185
    recipe list of Transform classes; default = the -O`level` recipe of examples/pics.py."""
    if not hasattr(B, 'NUFFT'):
        raise RuntimeError("sense_operator builds the reference's operator tree and needs a backend created by "
                           "indigo_b200.register(); without the reference package use sense_operator_fused() "
                           "or sense_operator_device()")
    coord = np.asarray(coord)
    Mshape = (1,) + tuple(coord.shape[1:])           # BART layout: READ dim of k-space is 1 (pics.py:60-63)
    F1 = B.NUFFT(Mshape, tuple(N), coord, width=width, n=n, oversamp=oversamp, dtype=_C64)
    if weights is not None:
        F1 = B.Diag(np.asarray(weights), name='dcf') * F1
    C = maps.shape[3]
    F = B.KronI(C, F1)
    S = B.VStack([B.Diag(maps[:, :, :, c:c + 1]) for c in range(C)], name='maps')
    A = F * S
    A._name = 'SENSE1'
    if recipe is None:
        recipe = default_recipe(B, level)
    return A.optimize(recipe)


def default_recipe(B, level=3):
    """The -O`level` recipe (examples/pics.py:179-191) on the reference's Transform family."""
    from .refcompat import reference_sense_recipe
    return reference_sense_recipe(level)


def normal_operator(A):
    """A^H A (the north-star apply).  lamda is passed to cg(lamda=...), never folded
    in as a Sum: under coil sharding a Sum would add it once per rank (SURVEY 8e)."""
    if hasattr(A, 'normal'):              # fused node (indigo_b200.fused): k-space never leaves the interleaved layout
        return A.normal
    AHA = A.H * A
    AHA._name = 'SENSE'
    # Reference trees only: the arena reserved by A.optimize() is sized for A alone
    # (transforms.py:72-76); A^H A nests one more Product temporary (the k-space vector).  The
    # reference gets away with it because its estimate also counts the matrices' bytes; size the
    # arena for the tree that is evaluated.
    B = A._backend
    if getattr(B, '_scratch', None) is not None and hasattr(AHA, 'memusage'):
        need = int(AHA.memusage()) // _C64.itemsize
        if B._scratch.size < need and B._scratch_pos == 0:
            B._scratch = None
            B._scratch = B.empty_array((need,), _C64)
    return AHA


def sqrt_dcf(coord):
    """sqrt(|k|) row weights of the well-conditioned CG protocol (SURVEY 8d, cfg4)."""
    c = np.asarray(coord, dtype=np.float64)
    c = c.reshape((3, -1), order='F')
    return np.sqrt(np.sqrt((c ** 2).sum(axis=0))).astype(np.float32)


# ---------------------------------------------------------------------------
# Device-side construction (SURVEY.md section 8f rank 2)
# ---------------------------------------------------------------------------
def _fftc_mod_times_scale(oN):
    """Diagonal of mod*scale as the -O2 realisation produces it: mod = exp(2 pi i sum_d
    (i_d - c_d/2) c_d/n_d) in float64 (backend.py:357-363) cast to complex64, times the
    complex64 cast of 1/sqrt(prod(oN)) (backend.py:349-351).  Evaluated slab by slab so
    that a 416^3 grid never needs the full float64 mgrid."""
    terms = []
    for d in range(3):
        c = oN[d] // 2
        terms.append((np.arange(oN[d]) - c / 2.0) * (c / oN[d]))
    scl = np.complex64(_grid_scale(oN))
    out = np.empty(oN, dtype=_C64, order='F')
    txy = (0 + terms[0][:, None]) + terms[1][None, :]
    for z in range(oN[2]):
        ph = txy + terms[2][z]
        out[:, :, z] = np.exp(1j * 2.0 * np.pi * ph).astype(_C64) * scl
    return out.reshape(-1, order='F')


def _fftc_mod(oN):
    terms = []
    for d in range(3):
        c = oN[d] // 2
        terms.append((np.arange(oN[d]) - c / 2.0) * (c / oN[d]))
    ph = ((0 + terms[0][:, None, None]) + terms[1][None, :, None]) + terms[2][None, None, :]
    return np.exp(1j * 2.0 * np.pi * ph).astype(_C64)


def _sample_weights(weights, m):
    """Per-sample row weights in sample order.  Samples are ordered like coord.reshape((3, -1), order='F'),
    and B.Diag flattens its argument in memory order ('A'); an (nread, nspokes) array is therefore taken in
    column-major order, a 1-D array as it is."""
    w = np.asarray(weights, dtype=np.float32)
    if w.ndim > 1:
        w = np.asfortranarray(w).flatten(order='A')
    if w.size != m:
        raise ValueError("expected %d row weights, got %d" % (m, w.size))
    return np.ascontiguousarray(w)



def gridding_matrix_device(B, N, coord, oversamp=2.0, weights=None, width=3, n=128, unphase=None):
    """G' = interp * (mod * scale) built on the GPU straight into device CSR arrays
    (ib200_kb_count -> exclusive scan -> ib200_kb_fill).  Returns (csr, oN, omin, beta).
    unphase (a unit constant u in {1, -1, i, -i}): build conj(u) * G' instead -- exact, and real when u is
    gridding_geometry(...).u; the caller applies u through alpha."""
    import ctypes

    lib, s = B._lib, B._stream
    geo = gridding_geometry(N, oversamp, width, n)
    oN, table = geo.oN, geo.table
    on = int(np.prod(oN))
    c3 = _coords_f64(coord)
    m = c3.shape[1]
    grid = (ctypes.c_int64 * 3)(*oN)
    coord_d = B.copy_array(c3)
    table_d = B.copy_array(table)
    counts = B.empty_array((max(m, 1),), np.dtype('int32'))
    lib.kb_count(s, m, coord_d.ptr, grid, float(width), counts.ptr)
    g_ptr = B.empty_array((m + 1,), np.dtype('int32'), name='interp*mod*scale.rowPtrs')
    lib.exclusive_scan_i32(s, m, counts.ptr, g_ptr.ptr)
    nnz = int(g_ptr[m:m + 1].to_host()[0])
    g_ind = B.empty_array((max(nnz, 1),), np.dtype('int32'), name='interp*mod*scale.colInds')
    g_val = B.empty_array((max(nnz, 1),), _C64, name='interp*mod*scale.data')
    colscale = _fftc_mod_times_scale(oN)
    if unphase is not None and complex(unphase) != 1:
        colscale = (colscale * np.complex64(np.conj(unphase))).astype(_C64)
    colscale_d = B.copy_array(colscale)
    w_d = None
    if weights is not None:
        w_d = B.copy_array(_sample_weights(weights, m))
    lib.kb_fill(s, m, coord_d.ptr, grid, float(width), table_d.ptr, int(table.size),
                w_d.ptr if w_d is not None else None, colscale_d.ptr, g_ptr.ptr, g_ind.ptr, g_val.ptr)
    B.barrier()
    del colscale_d, coord_d, counts
    Gd = B.csr_matrix.from_device(B, (m, on), g_ptr, g_ind[0:nnz], g_val[0:nnz], name='interp*mod*scale')
    return Gd, oN, geo.omin, geo.beta


def sample_order_device(B, geo, coord):
    """Matrix-free part of the fused operator's construction: (perm, nnz) with perm[r] = the sample at position r of
    the tile-sorted order (ib200_kb_sample_order: SAMPLE_TILE tiles in SAMPLE_SUPER super-tiles) and nnz = entries
    the gridding matrix would have (ib200_kb_count)."""
    import ctypes
    lib, s = B._lib, B._stream
    c3 = _coords_f64(coord)
    m = c3.shape[1]
    coord_d = B.copy_array(c3)
    grid = (ctypes.c_int64 * 3)(*geo.oN)
    i32 = np.dtype('int32')
    counts = B.empty_array((max(m, 1),), i32)
    lib.kb_count(s, m, coord_d.ptr, grid, float(geo.width), counts.ptr)
    ptr = B.empty_array((m + 1,), i32)
    lib.exclusive_scan_i32(s, m, counts.ptr, ptr.ptr)
    nnz = int(ptr[m:m + 1].to_host()[0])
    perm = B.empty_array((max(m, 1),), i32, name='G.sorted.rowmap')
    lib.kb_sample_order(s, m, coord_d.ptr, grid, float(geo.width), (ctypes.c_int64 * 3)(*SAMPLE_TILE),
                        (ctypes.c_int64 * 3)(*SAMPLE_SUPER), perm.ptr)
    return perm, nnz


def _fftc_unit_phases(oN):
    """Per axis: (unit constant u_d in {1, -1, i, -i}, real factor array) with mod_d = u_d * factor_d, where
    mod = prod_d exp(2 pi i (i_d - c_d/2) c_d/n_d) (backend.py:349-364); None when an axis is not real up to such a
    constant.  Every even axis length gives u_d = 1 except n_d = 2 (mod 4 in general), whose factors are -i, +i:
    the two-point z axis of a 2-D problem."""
    out = []
    for d in range(3):
        c = oN[d] // 2
        m = np.exp(1j * 2.0 * np.pi * ((np.arange(oN[d]) - c / 2.0) * (c / oN[d])))
        u = min((1, -1, 1j, -1j), key=lambda v: abs(m[0] - v))
        r = m * np.conj(u)
        if np.abs(r.imag).max() > 1e-6:
            return None
        out.append((complex(u), r.real.astype(np.float32)))
    return out


def _grid_scale(oN):
    """The grid scale 1/sqrt(prod(oN)) as the -O2 realisation rounds it (complex64 cast, backend.py:349-351): a
    float32."""
    return np.float32(np.complex64(np.complex128(1.0) / np.sqrt(int(np.prod(oN)))).real)


GriddingGeometry = collections.namedtuple('GriddingGeometry', 'N oN omin width beta table u factors separable')


def gridding_geometry(N, oversamp=2.0, width=3, n=128):
    """Oversampled grid and Kaiser-Bessel kernel of the NUFFT of an N image (backend.py:403-442): N, oN, omin (smallest
    oversampling), width, beta, table (float64 right half of kaiser(2n + 1, beta)), u (unit constant of the centring
    phase: 1 for every 3-D grid the fused path serves, -i for 2-D problems), factors (per-axis real factors of
    conj(u) * mod * scale, float32, the scale folded into the last) and separable (whether ib200_kb_records can
    describe G': at most 6 taps per axis).  When mod is not real up to a unit constant: u = 1, factors None."""
    from scipy.signal.windows import kaiser
    N = tuple(int(v) for v in N)
    os3 = oversamp if isinstance(oversamp, tuple) else (oversamp,) * 3
    oN = tuple(int(a * o) for a, o in zip(N, os3))
    omin = min(os3)
    beta = np.pi * np.sqrt(((width * 2. / omin) * (omin - 0.5)) ** 2 - 0.8)
    table = np.ascontiguousarray(kaiser(2 * n + 1, beta)[n:], dtype=np.float64)
    ph = _fftc_unit_phases(oN)
    u, factors = 1.0, None
    if ph is not None:
        u = complex(np.prod([p[0] for p in ph]))
        u = complex(round(u.real), round(u.imag))
        factors = [p[1] for p in ph]
        factors[2] = (factors[2] * _grid_scale(oN)).astype(np.float32)
    return GriddingGeometry(N, oN, omin, width, beta, table, u, factors,
                            factors is not None and 2 * width <= 6)


def _coords_f64(coord):
    """Sample coordinates as the column-major float64 (3, M) array the construction kernels read; samples in the
    order of coord.reshape((3, -1), order='F')."""
    return np.asfortranarray(np.asarray(coord).reshape((3, -1), order='F').astype(np.float64))


def _mod_apod(geo):
    """(cut, q): the image's window in the oversampled grid (Zpad 'center', backend.py:379-381) and q = mod * apod at
    the image voxels, column-major complex64 (the diagonal factor of P, pics.py:111-126)."""
    from .kbmath import rolloff3
    cut = tuple(slice(a // 2 + int(np.ceil(-b / 2)), a // 2 + int(np.ceil(b / 2))) for a, b in zip(geo.oN, geo.N))
    mod_at = _fftc_mod(geo.oN)[cut].flatten(order='F')
    apod = rolloff3(geo.omin, geo.width, geo.beta, geo.N).flatten(order='F').astype(_C64)
    return cut, (mod_at * np.complex64(1)) * apod


def kb_records_device(B, geo, coord, weights=None, perm=None, out_sorted=False):
    """Separable-weight records of G' = interp*mod*scale (ib200_kb_records, csrc/kbgrid.cu): 96 bytes per
    sample instead of a stored row.  perm (device int32, optional): record r describes sample perm[r];
    out_sorted: results go to row r (sorted order) instead of row perm[r].
    Returns the device array of records, or None when this grid / kernel width is not served
    (not geo.separable, or the kernel refuses a sample)."""
    import ctypes

    if not geo.separable:
        return None
    lib, s = B._lib, B._stream
    c3 = _coords_f64(coord)
    m = c3.shape[1]
    coord_d, table_d = B.copy_array(c3), B.copy_array(geo.table)
    f_d = [B.copy_array(np.ascontiguousarray(f)) for f in geo.factors]
    w_d = None
    if weights is not None:
        w_d = B.copy_array(_sample_weights(weights, m))
    nb = int(lib.kb_record_bytes())
    rec = B.empty_array((max(m, 1) * nb // 8,), np.dtype('int64'), name='G.records')
    flag = ctypes.c_int()
    grid = (ctypes.c_int64 * 3)(*geo.oN)
    lib.kb_records(s, m, coord_d.ptr, grid, float(geo.width), table_d.ptr, int(geo.table.size),
                   w_d.ptr if w_d is not None else None, f_d[0].ptr, f_d[1].ptr, f_d[2].ptr,
                   perm.ptr if perm is not None else None, 1 if out_sorted else 0, rec.ptr, ctypes.byref(flag))
    return rec if flag.value == 0 else None


def tile_rowmap_device(B, oN):
    """Tile-major row order of the oversampled grid in GRID_TILE tiles (ib200_grid_tile_rank): (kp, colrank, rowmap)
    with kp the padded point count, colrank[point] its tile-major row and rowmap[row] the grid point of a row
    (< 0: padding)."""
    import ctypes
    lib, s = B._lib, B._stream
    grid3, tile3 = (ctypes.c_int64 * 3)(*oN), (ctypes.c_int64 * 3)(*GRID_TILE)
    padded = ctypes.c_int64()
    lib.grid_tile_rank(s, grid3, tile3, None, None, ctypes.byref(padded))
    kp = int(padded.value)
    i32 = np.dtype('int32')
    colrank = B.empty_array((int(np.prod(oN)),), i32)
    rowmap = B.empty_array((kp,), i32, name='G.H.rowmap')
    lib.grid_tile_rank(s, grid3, tile3, colrank.ptr, rowmap.ptr, ctypes.byref(padded))
    return kp, colrank, rowmap


def support_windows_device(B, m, records, oN, kp, rowmap, bx):
    """k-space support windows from the separable records of m samples (ib200_kb_support_windows): one z interval
    per column block of bx x GRID_TILE[1] grid points, the hull of the taps that fall into it.  Returns (win, rowmap_w,
    inside): the windows, the tile-major rowmap of kp rows with the rows outside set to -1, and the number of grid
    points inside."""
    import ctypes
    lib, s = B._lib, B._stream
    i32 = np.dtype('int32')
    win = B.empty_array((2 * oN[0] * oN[1],), i32, name='G.support')
    rowmap_w = B.empty_array((kp,), i32, name='G.H.rowmap.support')
    inside = ctypes.c_int64()
    lib.kb_support_windows(s, m, records.ptr, (ctypes.c_int64 * 3)(*oN), kp, rowmap.ptr,
                           (ctypes.c_int64 * 3)(bx, GRID_TILE[1], GRID_TILE[2]), win.ptr, rowmap_w.ptr,
                           ctypes.byref(inside))
    return win, rowmap_w, int(inside.value)


def block_entries_device(B, m, records, oN, rowmap, kp, shape, seg_batches):
    """Block entries of the matrix-free adjoint gridding (ib200_kb_blocks_count / _fill, csrc/kbblocks.cu) from the
    separable records of m samples, for blocks of 4 x by x bz grid points (shape = (by, bz)) and the tile-major
    rowmap of kp rows.  Returns dict(ent, work, nwork, split, nsplit, nslot, batches, bytes, shape); the caller
    allocates the partial sums of the nslot work items of split blocks."""
    import ctypes
    lib, s = B._lib, B._stream
    by, bz = shape
    i32 = np.dtype('int32')
    grid3 = (ctypes.c_int64 * 3)(*oN)
    segb = max(1, int(seg_batches))
    nblk = kp // 64 * (4 // by) * (4 // bz)
    bptr = B.empty_array((nblk + 1,), i32, name='G.H.blocks.batchptr')
    wptr = B.empty_array((nblk + 1,), i32, name='G.H.blocks.workptr')
    tot = (ctypes.c_int64 * 5)()
    lib.kb_blocks_count(s, m, records.ptr, grid3, by, bz, rowmap.ptr, segb, bptr.ptr, wptr.ptr, tot)
    nbat, nwork, nsplit, nslot = int(tot[1]), int(tot[2]), int(tot[3]), int(tot[4])
    bb = int(lib.kb_blocks_batch_bytes(by, bz))
    ent = B.empty_array((max(nbat, 1) * bb // 8,), np.dtype('int64'), name='G.H.blocks.entries')
    work = B.empty_array((4 * max(nwork, 1),), i32, name='G.H.blocks.work')
    split = B.empty_array((4 * max(nsplit, 1),), i32, name='G.H.blocks.split')
    lib.kb_blocks_fill(s, m, records.ptr, grid3, by, bz, segb, bptr.ptr, wptr.ptr, ent.ptr, work.ptr, split.ptr)
    return dict(ent=ent, work=work, nwork=nwork, split=split, nsplit=nsplit, nslot=nslot, batches=nbat,
                bytes=nbat * bb, shape=(by, bz))


class DensityDevice(object):
    """Device state of pipe_menon_dcf: the matrix-free construction of the fused operator without row weights
    (sample order, separable records in sorted order with out = position, tile-major rowmap, support windows, 4x4x4
    block entries), the real grid g = I^T w (prod(oN) float32, zeroed once) and the weights w in sorted order."""

    probe = None          # as SenseDevice.probe: label -> context manager around each kernel of an iteration

    def __init__(self, B, N, coord, oversamp=2.0, width=3, n=128):
        import ctypes
        coord = np.asarray(coord)
        if not np.isfinite(coord).all():
            raise ValueError("pipe_menon_dcf: the trajectory has non-finite coordinates")
        self.B = B
        geo = gridding_geometry(N, oversamp, width, n)
        oN = self.oN = geo.oN
        m = self.M = int(np.prod(coord.shape[1:]))
        self.shape = tuple(coord.shape[1:])
        self.grid3 = (ctypes.c_int64 * 3)(*oN)
        self.perm, _ = sample_order_device(B, geo, coord)
        self.rec = kb_records_device(B, geo, coord, perm=self.perm, out_sorted=True)
        if self.rec is None:
            raise RuntimeError("pipe_menon_dcf: no separable records for kernel width %g on the oversampled grid %s "
                               "(they serve at most 6 taps per axis and a centring phase that is real up to a constant)"
                               % (width, oN))
        kp, colrank, rowmap = tile_rowmap_device(B, oN)
        del colrank
        win, self.rowmap, self.inside = support_windows_device(B, m, self.rec, oN, kp, rowmap, GRID_TILE[0])
        del win, rowmap
        # whole 4x4x4 tiles (one channel), blocks of more than 256 batches cut into work items
        self.tiles = block_entries_device(B, m, self.rec, oN, self.rowmap, kp, (4, 4), 256)
        f32 = np.dtype('float32')
        self.scratch = B.empty_array((max(self.tiles['nslot'], 1) * 64,), f32, name='dcf.partial')
        self.g = B.zero_array((int(np.prod(oN)),), f32, name='dcf.grid')
        self.w = B.copy_array(np.ones(m, dtype=np.float32))
        self.resid = B.empty_array((1 + (m + 255) // 256,), np.dtype('float64'), name='dcf.residual')
        # the records carry scale = 1/sqrt(prod oN) (float32) on z: the update divides q = scale^2 (I I^T w) by it
        scl = float(_grid_scale(oN))
        self.inv_s2 = 1.0 / (scl * scl)

    def _step(self, label):
        import contextlib
        return self.probe(label) if self.probe is not None else contextlib.nullcontext()

    def iterate(self, residual=False):
        """One iteration w <- w / (I I^T w); residual: also the sum of (I I^T w - 1)^2 into resid[0] (device)."""
        lib, s, t = self.B._lib, self.B._stream, self.tiles
        with self._step("kb_density_spread"):
            lib.kb_density_spread(s, t['nwork'], t['work'].ptr, t['ent'].ptr, self.w.ptr, self.g.ptr, self.rowmap.ptr,
                                  t['nsplit'], t['split'].ptr, self.scratch.ptr)
        with self._step("kb_density_update"):
            lib.kb_density_update(s, self.M, self.rec.ptr, self.g.ptr, self.grid3, self.inv_s2, self.w.ptr,
                                  self.resid.ptr if residual else None)

    def residual(self):
        """||I I^T w - 1|| / sqrt(M) of the weights the last iterate(residual=True) started from (host read-back)."""
        return float(np.sqrt(self.resid[0:1].to_host()[0] / self.M))

    def weights(self):
        """w in the caller's sample order, shaped like coord.shape[1:] (column-major)."""
        out = np.empty(self.M, dtype=np.float32)
        out[self.perm.to_host()] = self.w.to_host()
        return out.reshape(self.shape, order='F')


def pipe_menon_dcf(B, N, coord, oversamp=2.0, width=3, n=128, maxiter=30, history=None):
    """Pipe-Menon density compensation of the trajectory `coord` (3, d1, d2, ...) for an image of shape N:
        w_0 = 1,   w_{k+1} = w_k / (I I^T w_k),
    I the Kaiser-Bessel interpolation matrix of the NUFFT on the oversampled grid (oversamp, width, n as for
    sense_operator), so that the fixed point satisfies I I^T w = 1.  Unlike sqrt_dcf's |k|^(1/2) it is right for any
    trajectory (stack of spirals, random, ...).  Both products run on the device with no matrix formed
    (csrc/dcf.cu): I^T w on the 4x4x4 block entries of the matrix-free adjoint gridding, I g on the separable
    records of the forward gridding, fused with the update.  No FFT plan is needed: grids the fused operator has no
    passes for are served as well.

    Returns float32 weights w shaped like coord.shape[1:] (samples in column-major order, as the operators take
    them): weights=np.sqrt(w) feeds sense_operator_fused, sense_operator and fuse_transform trees as they are.
    The result is bit-identical from run to run.  With `history` a list, the fixed-point residual
    ||I I^T w_k - 1|| / sqrt(M) of the weights each iteration starts from (w_0 = 1 first) is appended to it, one
    host read-back per iteration; without it the iterations issue no host synchronisation.
    Under coil sharding every rank computes the same weights from the same trajectory; no collective is needed.
    Raises ValueError for non-finite coordinates or maxiter < 1, RuntimeError when the separable records cannot be
    built (kernels of more than 6 taps per axis, grids whose centring phase is not real up to a constant)."""
    if int(maxiter) < 1:
        raise ValueError("pipe_menon_dcf: maxiter must be at least 1, got %r" % (maxiter,))
    coord = np.asarray(coord)
    if int(np.prod(coord.shape[1:])) == 0:
        return np.zeros(tuple(coord.shape[1:]), dtype=np.float32, order='F')
    d = DensityDevice(B, N, coord, oversamp, width, n)
    for _ in range(int(maxiter)):
        d.iterate(residual=history is not None)
        if history is not None:
            history.append(d.residual())
    w = d.weights()
    del d                                   # device temporaries go with it
    return w


class _SixCallSense(object):
    """Mixin with the evaluation of the -O3 tree's six Backend calls (SURVEY.md section 3.1) on
    device-built operands; combined with the Operator base of B's family by sense_operator_device."""

    def _setup(self, Gd, Pd, oN, C, nvox):
        self.G, self.P = Gd, Pd                          # device CSR holders (B.csr_matrix.from_device)
        self.oN, self.C, self.nvox = tuple(oN), int(C), int(nvox)
        self.M, self.on = int(Gd.shape[0]), int(Gd.shape[1])
        self._t = None

    shape = property(lambda self: (self.M * self.C, self.nvox))
    dtype = property(lambda self: _C64)

    def _mem_usage(self, ncols=1):
        return 0

    def _temps(self):
        if self._t is None:
            B = self._backend
            self._t = (B.empty_array((self.on * self.C, 1), _C64, name='SENSE1.grid.a'),
                       B.empty_array((self.on * self.C, 1), _C64, name='SENSE1.grid.b'))
        return self._t

    def _eval(self, y, x, alpha=1, beta=0, forward=True, left=True):
        if not left:
            raise NotImplementedError("Right-multiplication not implemented for the six-call SENSE operator.")
        assert x.shape[1] == 1, "one image / one multi-coil data set at a time"
        B, C = self._backend, self.C
        a, b = self._temps()
        a3, b3 = a.reshape(self.oN + (C,)), b.reshape(self.oN + (C,))
        a2, b2 = a.reshape((self.on, C)), b.reshape((self.on, C))
        if forward:
            self.P.adjoint(a, x)                                          # ccsrmm(P^H, adjoint): expand
            B.fftn(b3, a3)                                                # fftn
            self.G.forward(y.reshape((self.M, C)), b2, alpha=alpha, beta=beta)    # ccsrmm(G')
        else:
            self.G.adjoint(a2, x.reshape((self.M, C)))                    # ccsrmm(G', adjoint)
            B.ifftn(b3, a3)                                               # ifftn
            self.P.forward(y, b, alpha=alpha, beta=beta)                  # ccsrmm(P^H): combine


def sense_operator_device(B, N, coord, maps, oversamp=2.0, weights=None, width=3, n=128):
    """Same operator and the same six Backend calls per A^H A as the -O3 tree of
    sense_operator(), issued directly (no tree, works without the reference package); G' and P^H are built on the GPU (ib200_kb_* / ib200_sense_ph_*)
    straight into device CSR arrays: no COO triplets, no scipy products, no 10 GB upload.
    Needed at BASELINE.json's full sizes (416^3 grid, 6.8 M samples: 853 M stored entries).
    tests/test_gpu_sense.py checks structure (bit-identical) and values against the
    host-built matrices."""
    lib, s = B._lib, B._stream
    geo = gridding_geometry(N, oversamp, width, n)
    N, oN, C = geo.N, geo.oN, int(maps.shape[3])
    Gd = gridding_matrix_device(B, N, coord, oversamp, weights, width, n)[0]
    on, nvox = int(np.prod(oN)), int(np.prod(N))

    # ---- P^H, stored adjoint of kron(I_C, mod*zpad*apod) * vstack(maps) ----------------
    cut, q = _mod_apod(geo)                                                 # (mod @ zpad) @ apod
    lin = np.arange(on, dtype=np.int64).reshape(oN, order='F')
    zp = np.ascontiguousarray(lin[cut].flatten(order='F').astype(np.int32))
    del lin
    maps_f = np.asfortranarray(maps.reshape((nvox, C), order='F').astype(_C64))
    maps_d, q_d, zp_d = B.copy_array(maps_f), B.copy_array(q), B.copy_array(zp)
    counts = B.empty_array((nvox,), np.dtype('int32'))
    lib.sense_ph_count(s, nvox, C, maps_d.ptr, q_d.ptr, counts.ptr)
    p_ptr = B.empty_array((nvox + 1,), np.dtype('int32'), name='P.H.rowPtrs')
    lib.exclusive_scan_i32(s, nvox, counts.ptr, p_ptr.ptr)
    pnnz = int(p_ptr[nvox:nvox + 1].to_host()[0])
    p_ind = B.empty_array((max(pnnz, 1),), np.dtype('int32'), name='P.H.colInds')
    p_val = B.empty_array((max(pnnz, 1),), _C64, name='P.H.data')
    lib.sense_ph_fill(s, nvox, C, on, maps_d.ptr, q_d.ptr, zp_d.ptr, p_ptr.ptr, p_ind.ptr, p_val.ptr)
    B.barrier()
    del maps_d, q_d, zp_d, counts
    Pd = B.csr_matrix.from_device(B, (nvox, C * on), p_ptr, p_ind[0:pnnz], p_val[0:pnnz],
                                  name='((x)mod*zpad*apod)*+.H')

    # ---- the six calls around them (what the -O3 tree of examples/pics.py evaluates, SURVEY 3.1) ----
    ops = _ops_of(B)
    cls = _six_cache.get(ops)
    if cls is None:
        cls = _six_cache[ops] = type('SixCallSense', (_SixCallSense, ops.Operator), {})
    A = cls(B, name='SENSE1')
    A._setup(Gd, Pd, oN, C, nvox)
    return A


_six_cache = {}
