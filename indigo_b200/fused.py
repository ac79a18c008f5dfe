"""
Backend-specific fusion of the SENSE-NUFFT operator (SURVEY.md section 8f rank 1; the
north star's "fused elementwise" item).

The reference's -O3 tree evaluates A^H A as six Backend calls
    ccsrmm(P^H, adj) -> fftn -> ccsrmm(G') -> ccsrmm(G', adj) -> ifftn -> ccsrmm(P^H)
on column-major (grid, coil) arrays (SURVEY.md section 3.1).  On the B200 the same
arithmetic runs as

    ib200_sense_expand_fft      grid = FFT3(zpad(pf .* x))           coil-interleaved grid[z][y][x][c],
                                                                      zero rows never touched (pruned passes),
                                                                      last pass stores only inside the support
    ib200_kb_gather   (G')      k    = G' grid                        no stored matrix: separable 96-byte records,
                                                                      one 128-byte line per tap
    ib200_ccsrmm_runs (G'^H)    grid = G'^H k                         stored adjoint merged into x-runs of 4 points
    ib200_sense_ifft_combine    y    = sum_c conj(pf) .* crop(IFFT3(grid))

(fallbacks on stored entries: ib200_ccsrmm_ilr / ib200_ccsrmm_il; every stage has a switch on SenseDevice)
so the 9.2 GB zero-padded volume of cfg3 is never written by a scatter, read back by the FFT,
or transposed between the coil-slow layout of the interface and the coil-fast layout the
gather wants.  The node below is an ordinary operator of the family the backend uses (the reference's
`indigo.operators.Operator` when the backend was built on the reference, indigo_b200.linop.Operator
otherwise): `A * x`, `A.H * y`, `(A.H * A) * x`, `B.cg(A.H * A, ...)` work as for the
unfused tree, and tests/test_gpu_fused.py checks all of them against the same oracle.
"""
import ctypes

import numpy as np

_C64 = np.dtype('complex64')


class SenseDevice(object):
    """Device-resident pieces shared by the fused nodes of one SENSE operator."""

    tile = (4, 4, 4)
    allow_real = True          # use the real-weight packed kernels when the matrix values are real
    long_thresh = 512          # rows of G'^H with more entries than this get a whole CTA each
    sample_tile = (8, 8, 8)    # samples (rows of G') are sorted by the grid tile of this size they fall into,
    sample_super = (8, 8, 8)   # tiles grouped into super-tiles of this many tiles (64^3 points: L2-sized working set)
    # rows_per_group codes of ib200_ccsrmm_ilr (measured on cfg3, profiles/r01_s5_*): shared-memory staged
    # entries; one coil per lane for the long forward rows, two coils per lane for the short adjoint rows
    staged_fwd = -41
    staged_adj = -4
    allow_separable = True     # forward gridding from 96-byte separable-weight records instead of stored entries
    allow_sorted_ksp = True    # keep k-space in tile-sorted sample order between the two gridding steps
    allow_runs = True          # adjoint gridding on merged x-runs of the stored adjoint (csrc/csrmm_runs.cu)
    run_long_thresh = 1024     # runs with more entries than this are cut into segments of this length
    allow_tiles = True         # adjoint gridding on block entries built from the separable records (csrc/kbblocks.cu)
    tiles_max_coils = 4        # whole 4x4x4 tiles up to this many coils (coil-sharded operators) ...
    blocks_max_coils = 64      # ... 4x2x2 blocks up to this many; the x-runs of the stored adjoint above
                               # (measured at cfg3, profiles/r02_blocks.md: 2 coils 1.15 / 2.77 ms, 4: 2.0 / 3.0,
                               #  8: 2.95 / 3.6, 16: 4.9 / 5.4 for blocks / x-runs)
    block_shape = None         # (by, bz) forced for every coil count (tests, tools/)
    tiles_seg_batches = 256    # blocks with more batches (of 4 entries) than this are cut into work items of this length
    tiles_lanes = 0            # lanes sharing the rows of a block (0: kernel default)
    matrix_free_setup = True   # build the matrix-free operator without ever forming the CSR matrix or its stored adjoint
    keep_stored = False        # keep the CSR matrix and its stored adjoint after a matrix-free operator was built
    allow_windows = True       # k-space support windows: skip the grid outside the trajectory's support
    window_min_saving = 0.05   # ... when at least this fraction of the grid lies outside

    def __init__(self, B, N, coord, maps, oversamp=2.0, weights=None, width=3, n=128):
        import os
        from .sense import gridding_matrix_device, _fftc_mod, kb_records_device, _fftc_unit_phase
        if os.environ.get("IB200_SAMPLE_SUPER"):                    # tuning knob: super-tile edge in tiles
            self.sample_super = (int(os.environ["IB200_SAMPLE_SUPER"]),) * 3
        if os.environ.get("IB200_SAMPLE_TILE"):                     # tuning knob: sample tile edge in grid points
            self.sample_tile = (int(os.environ["IB200_SAMPLE_TILE"]),) * 3
        if os.environ.get("IB200_TILES_MAXC"):                      # tuning knobs (tools/): tile-block adjoint gather
            self.tiles_max_coils = int(os.environ["IB200_TILES_MAXC"])
        if os.environ.get("IB200_BLOCKS_MAXC"):
            self.blocks_max_coils = int(os.environ["IB200_BLOCKS_MAXC"])
        if os.environ.get("IB200_BLOCKS_SHAPE"):
            self.block_shape = tuple(int(v) for v in os.environ["IB200_BLOCKS_SHAPE"].split(","))
        if os.environ.get("IB200_TILES_SEG"):
            self.tiles_seg_batches = int(os.environ["IB200_TILES_SEG"])
        if os.environ.get("IB200_RUN_LONG"):                        # tuning knob (tools/): run-length threshold
            self.run_long_thresh = int(os.environ["IB200_RUN_LONG"])
        elif int(np.prod(np.asarray(coord).shape[1:])) < (1 << 20) and type(self).run_long_thresh == 1024:
            # small problems (cfg1: 0.2 M samples) are bound by the longest serial walk of one lane group, not by
            # throughput: cut dense runs into shorter segments (r02 session 3: adjoint step 0.17 ms of a 0.37 ms apply)
            self.run_long_thresh = 256
        if (int(np.prod(np.asarray(coord).shape[1:])) < (1 << 20) and type(self).tiles_seg_batches == 256
                and not os.environ.get("IB200_TILES_SEG")):
            self.tiles_seg_batches = 32                             # the same for the block gather (r02 session 18: cfg1
                                                                    # 0.141 -> 0.049 ms; 16 and 64 batches are slower)
        from .kbmath import rolloff3

        self.B = B
        lib, s = B._lib, B._stream
        N = tuple(int(v) for v in N)
        C = int(maps.shape[3])
        # the construction's arguments, for operators derived from this one (toeplitz_normal)
        self.coord, self.maps, self.weights = coord, maps, weights
        self.oversamp, self.width, self.n = oversamp, width, n
        if C > 32:
            raise RuntimeError("fused SENSE path serves at most 32 coils per operator; shard or split the coils")
        self._plan = None
        # centring phase of G' that is real only up to a unit constant (2-D problems: -i on the two-point z axis): the
        # fused path holds conj(u) G', a real matrix, and applies u through alpha in the two gridding steps
        os3 = oversamp if isinstance(oversamp, tuple) else (oversamp,) * 3
        oN = tuple(int(a * o) for a, o in zip(N, os3))
        omin = min(os3)
        beta = np.pi * np.sqrt(((width * 2. / omin) * (omin - 0.5)) ** 2 - 0.8)       # as gridding_matrix_device
        self.gphase = _fftc_unit_phase(oN) or 1.0
        self.N, self.oN, self.C = N, oN, C
        self.M = int(np.prod(np.asarray(coord).shape[1:]))
        self.nvox, self.on = int(np.prod(N)), int(np.prod(oN))
        # matrix-free construction: sample order from the coordinates, windows and block entries from the separable
        # records; the CSR matrix G' (10 GB at cfg3), its transposition and their sorts are never made.  Anything the
        # matrix-free kernels do not serve (odd coil counts, complex centring phase, wide kernels, switches off) takes the
        # construction on stored matrices below.
        mf = bool(self.matrix_free_setup and self.allow_real and self.allow_separable and self.allow_sorted_ksp
                  and self.allow_tiles and not self.keep_stored and self._want_tiles() is not None and self.M > 0)
        self.G = None
        if not mf:
            self.G, oN_, omin_, beta_ = gridding_matrix_device(B, N, coord, oversamp, weights, width, n, unphase=self.gphase)
            assert tuple(int(v) for v in oN_) == oN
            self.nnz = int(self.G.values.size)
        # fused plan first: raises RuntimeError (unsupported) for grids without specialised passes
        n3, on3 = (ctypes.c_int64 * 3)(*N), (ctypes.c_int64 * 3)(*self.oN)
        self._plan = ctypes.c_void_p()
        lib.sense_plan_create(ctypes.byref(self._plan), n3, on3, C)
        # pf[voxel][coil] = (mod[zp] * apod)[voxel] * maps[voxel, coil]  (the factor P of pics.py:111-126)
        cut = tuple(slice(a // 2 + int(np.ceil(-b / 2)), a // 2 + int(np.ceil(b / 2))) for a, b in zip(self.oN, N))
        mod_at = _fftc_mod(self.oN)[cut].flatten(order='F')
        apod = rolloff3(omin, width, beta, N).flatten(order='F').astype(_C64)
        q = (mod_at * np.complex64(1)) * apod
        self.q = q                                                     # (mod * apod) at the image voxels
        maps_f = maps.reshape((self.nvox, C), order='F').astype(_C64)
        self.pf = B.copy_array(np.ascontiguousarray(q[:, None] * maps_f).reshape(-1))
        # stored adjoint of G' with the grid points in (padded) tile-major order
        from .sense import tile_rowmap_device
        grid3 = (ctypes.c_int64 * 3)(*self.oN)
        padded = ctypes.c_int64()
        i32 = np.dtype('int32')
        kp, colrank, self.rowmap = tile_rowmap_device(B, self.oN, self.tile)
        self.kp = kp
        self.t_ptr = self.t_ind = self.t_val = self.t_pk = None
        if not mf:
            self.t_ptr = B.empty_array((kp + 1,), i32, name='G.H.rowPtrs')
            self.t_ind = B.empty_array((max(self.nnz, 1),), i32, name='G.H.colInds')
            self.t_val = B.empty_array((max(self.nnz, 1),), _C64, name='G.H.data')
            work = B.empty_array((kp + 1,), i32)
            lib.csr_transpose_conj(s, self.M, kp, self.nnz, self.G.values.ptr, self.G.colInds.ptr, self.G.rowPtrs.ptr,
                                   self.t_val.ptr, self.t_ind.ptr, self.t_ptr.ptr, work.ptr, colrank.ptr)
            del work
        del colrank
        # real-weight packed entries (8 B instead of 12 B per stored entry, half the multiplies) when
        # the centring phase folded into G' is real, i.e. on every grid the fused path serves
        self.real, self.kb, self.ksp_sorted, self.pos = False, None, False, None
        if mf:
            from .sense import sample_order_device
            self.g_map, self.nnz = sample_order_device(B, self.oN, coord, width, self.sample_tile, self.sample_super)
            self.kb = kb_records_device(B, self.oN, coord, beta, weights, width, n, perm=self.g_map, out_sorted=True)
            if self.kb is not None:
                self.real = self.ksp_sorted = True
                self.pos = B.empty_array((max(self.M, 1),), i32, name='G.sorted.position')
                lib.invert_perm(s, self.M, self.g_map.ptr, self.pos.ptr)
                self.g_pk = self.g_ptr = None
        elif self.nnz and self.allow_real:
            pk = np.dtype('int64')                                     # 8-byte (int32 column, float32 weight) records
            g_pk = B.zero_array((self.nnz + 2,), pk, name='G.packed')  # +2: the staged kernel copies 16-byte granules
            hmax = (ctypes.c_float * 2)()
            lib.csr_pack_real(s, self.nnz, self.G.values.ptr, self.G.colInds.ptr, g_pk.ptr, hmax)
            if hmax[1] <= 1e-8 * hmax[0]:
                t_pk = B.zero_array((self.nnz + 2,), pk, name='G.H.packed')
                lib.csr_pack_real(s, self.nnz, self.t_val.ptr, self.t_ind.ptr, t_pk.ptr, hmax)
                self.t_pk, self.real = t_pk, True
                self.t_val = self.t_ind = None                          # the complex copy of G'^H is not needed any more
                # samples sorted by the 8x8x8 grid tile they fall into, tiles grouped into 64^3 super-tiles: the
                # samples one CTA sweeps share operand lines in all three dimensions (L1) and the CTAs in
                # flight cover a compact block of the grid (L2)
                stile = (ctypes.c_int64 * 3)(*self.sample_tile)
                ssuper = (ctypes.c_int64 * 3)(*self.sample_super)
                lib.grid_tile_rank2(s, grid3, stile, ssuper, None, ctypes.byref(padded))
                nr8 = int(padded.value)
                rank8 = B.empty_array((self.on,), i32)
                lib.grid_tile_rank2(s, grid3, stile, ssuper, rank8.ptr, ctypes.byref(padded))
                self.g_ptr = B.empty_array((self.M + 1,), i32, name='G.sorted.rowPtrs')
                self.g_pk = B.zero_array((self.nnz + 2,), pk, name='G.sorted.packed')
                self.g_map = B.empty_array((max(self.M, 1),), i32, name='G.sorted.rowmap')
                lib.csr_permute_rows(s, self.M, self.nnz, self.G.rowPtrs.ptr, g_pk.ptr, rank8.ptr, nr8,
                                     self.g_ptr.ptr, self.g_pk.ptr, self.g_map.ptr)
                del rank8
                # separable Kaiser-Bessel records in the same tile-sorted order: the forward gather then
                # needs no stored entries at all (csrc/kbgrid.cu).  k-space between the two gridding steps is kept in this sorted order when both the separable
                # forward gather and the x-run adjoint gather serve it: samples that are neighbours on the grid
                # are then neighbours in memory (the original spoke order scatters them over 0.9 GB at cfg3)
                self.kb = None
                use_runs = self.allow_runs and C % 2 == 0 and self.tile[0] == 4 and kp % 4 == 0
                use_tiles = self._want_tiles() is not None
                self.ksp_sorted = bool(self.allow_separable and (use_runs or use_tiles) and self.allow_sorted_ksp)
                if self.allow_separable:
                    self.kb = kb_records_device(B, self.oN, coord, beta, weights, width, n, perm=self.g_map,
                                                out_sorted=self.ksp_sorted)
                if self.kb is None:
                    self.ksp_sorted = False
                if self.ksp_sorted:
                    self.pos = B.empty_array((max(self.M, 1),), i32, name='G.sorted.position')
                    lib.invert_perm(s, self.M, self.g_map.ptr, self.pos.ptr)
                if self.kb is not None:
                    self.g_pk = self.g_ptr = None
            del g_pk
        # rows of G'^H that are long enough to deserve a whole CTA (k-space centre of radial trajectories)
        cnt = ctypes.c_int()
        if not mf:
            lib.csr_long_rows(s, kp, self.t_ptr.ptr, self.long_thresh, None, 0, ctypes.byref(cnt))
        self.nlong, self.longrows = int(cnt.value), None
        if self.nlong:
            self.longrows = B.empty_array((self.nlong,), i32, name='G.H.longrows')
            lib.csr_long_rows(s, kp, self.t_ptr.ptr, self.long_thresh, self.longrows.ptr, self.nlong, ctypes.byref(cnt))
        # k-space support windows (csrc/kbgrid.cu, csrc/fft_pk.cuh): grid points no sample touches are neither
        # written by the last forward pass, nor zero-filled by the adjoint gather, nor read by the first
        # inverse pass.  Blocks of bx x 4 columns share one z interval; 16 interleaved lines (one FFT tile)
        # must not straddle two blocks.
        self.win, self.support_fraction = None, 1.0
        if self.allow_windows and self.nnz and (C % 16 == 0 or 16 % C == 0):
            bx = max(self.tile[0], 16 // C) if C < 16 else self.tile[0]
            if self.oN[0] % bx == 0 and bx % self.tile[0] == 0:
                win = B.empty_array((2 * self.oN[0] * self.oN[1],), i32, name='G.support')
                rowmap_w = B.empty_array((kp,), i32, name='G.H.rowmap.support')
                inside = ctypes.c_int64()
                blk = (ctypes.c_int64 * 3)(bx, self.tile[1], self.tile[2])
                if mf and self.kb is not None:
                    lib.kb_support_windows(s, self.M, self.kb.ptr, grid3, kp, self.rowmap.ptr, blk, win.ptr, rowmap_w.ptr,
                                           ctypes.byref(inside))
                elif not mf:
                    lib.grid_support_windows(s, grid3, kp, self.t_ptr.ptr, self.rowmap.ptr, blk, win.ptr, rowmap_w.ptr,
                                             ctypes.byref(inside))
                else:
                    inside.value = self.on
                frac = inside.value / float(self.on)
                if frac <= 1.0 - self.window_min_saving:
                    try:
                        lib.sense_plan_set_support(self._plan, win.ptr, bx)
                        self.win, self.rowmap, self.support_fraction = win, rowmap_w, frac
                    except RuntimeError:
                        pass                                            # geometry without persistent packed z passes
        # block entries built from the separable records: one entry and one gather per (sample, block of 4 x by x bz
        # grid points) pair -- whole tiles when the coils are few (the shard of a coil-sharded operator)
        self.tiles = None
        shape = self._want_tiles()
        if self.real and self.kb is not None and shape:
            from .sense import block_entries_device
            by, bz = shape
            t = block_entries_device(B, self.M, self.kb, self.oN, self.rowmap, kp, shape, self.tiles_seg_batches)
            cl = 1
            while cl < min(C, 16) // 2:
                cl *= 2
            t['scratch'] = B.empty_array((max(t['nslot'], 1) * 4 * by * bz * 2 * cl,), _C64, name='G.H.blocks.partial')
            self.tiles = t
        # x-run lists of the stored adjoint: one gather of a sample serves the four grid points of a tile row;
        # runs longer than run_long_thresh entries are cut into segments with their own lane groups
        self.runs = None
        if not mf and self.tiles is None and self.real and self.allow_runs and C % 2 == 0 and self.tile[0] == 4 and kp % 4 == 0:
            seg = max(4, int(self.run_long_thresh) // 4 * 4)
            run_ptr = B.empty_array((kp // 4 + 1,), i32, name='G.H.runs.ptr')
            nre, nsg, nsp = ctypes.c_int64(), ctypes.c_int(), ctypes.c_int()
            lib.csr_runs_count(s, kp, self.t_ptr.ptr, self.t_pk.ptr, seg, run_ptr.ptr,
                               ctypes.byref(nre), ctypes.byref(nsg), ctypes.byref(nsp))
            ne, nsg, nsp = max(int(nre.value), 4), int(nsg.value), int(nsp.value)
            ids = B.empty_array((ne,), i32, name='G.H.runs.ids')
            w4 = B.empty_array((4 * ne,), np.dtype('float32'), name='G.H.runs.w4')
            segd = B.empty_array((4 * max(nsg, 1),), i32, name='G.H.runs.segments')
            spld = B.empty_array((4 * max(nsp, 1),), i32, name='G.H.runs.split')
            lib.csr_runs_fill(s, kp, self.t_ptr.ptr, self.t_pk.ptr, seg, run_ptr.ptr, ids.ptr, w4.ptr, segd.ptr, spld.ptr,
                              self.pos.ptr if self.ksp_sorted else None)
            cl = 1
            while cl < C // 2:
                cl *= 2
            scratch = B.empty_array((max(nsg, 1) * 4 * 2 * cl,), _C64, name='G.H.runs.partial')
            self.runs = dict(ptr=run_ptr, ids=ids, w4=w4, seg=seg, segd=segd, nseg=nsg, spld=spld, nsplit=nsp,
                             scratch=scratch, entries=int(nre.value))
        # zero-initialised: with windows, parts of the grid are never written, and the separable gather
        # multiplies its zero-weight taps (6th tap of on-grid samples) with whatever is there
        if mf and (self.kb is None or self.tiles is None):
            # the records or the block entries could not be built (kernel wider than 6 taps): construct on stored matrices
            lib.sense_plan_destroy(self._plan)
            self._plan = None
            self.matrix_free_setup = False
            return self.__init__(B, N, coord, maps, oversamp, weights, width, n)
        if self.tiles is not None and self.kb is not None and not self.keep_stored:
            # both gridding steps are matrix-free now: the CSR matrix, its stored adjoint and the long-row list were
            # only the source of the support windows (17 GB at cfg3)
            self.G = self.t_pk = self.t_ptr = self.t_val = self.t_ind = self.longrows = None
            self.nlong = 0
        self.grid = B.zero_array((self.on * C,), _C64, name='grid[z][y][x][c]')
        self.ksp = B.empty_array((self.M * C,), _C64, name='ksp[m][c]')

    def _want_tiles(self):
        """Block shape (by, bz) of the matrix-free adjoint gather for this coil count, or None (x-runs / stored rows)."""
        if not (self.allow_tiles and self.allow_separable and self.C % 2 == 0 and tuple(self.tile) == (4, 4, 4)):
            return None
        if self.block_shape:
            return tuple(self.block_shape)
        if self.C <= self.tiles_max_coils:
            return (4, 4)
        if self.C <= self.blocks_max_coils:
            return (2, 2)
        return None

    def __del__(self):
        try:
            if getattr(self, '_plan', None):
                self.B._lib.sense_plan_destroy(self._plan)
        except Exception:
            pass

    # ---- the four fused steps ---------------------------------------------------------------
    # `probe`: optional callable label -> context manager (bench.py's KernelTimer).  When set, the two transforms
    # are issued pass by pass through ib200_sense_pass (the same kernels with the same arguments) so that every
    # kernel of the apply can be bracketed by CUDA events.
    probe = None

    def _step(self, label):
        import contextlib
        return self.probe(label) if self.probe is not None else contextlib.nullcontext()

    def expand_fft(self, x):
        lib, s = self.B._lib, self.B._stream
        if self.probe is None:
            lib.sense_expand_fft(self._plan, s, self.grid.ptr, x.ptr, self.pf.ptr)
            return
        for which, label in ((0, "sense_expand_pk[x]"), (1, "fft_pass[y fwd]"), (2, "fft_pass[z fwd]")):
            with self.probe(label):
                lib.sense_pass(self._plan, s, which, self.grid.ptr, x.ptr, None, self.pf.ptr, 1.0, 0.0, 0.0, 0.0)

    def grid_to_samples(self, alpha=1.0):
        with self._step("kb_gather"):
            self._grid_to_samples(alpha)

    def samples_to_grid(self):
        with self._step("kb_blocks" if self.tiles is not None else "csrmm_runs"):
            self._samples_to_grid()

    def _grid_to_samples(self, alpha=1.0):
        a = complex(alpha) * complex(self.gphase)
        G, lib, s = self.G, self.B._lib, self.B._stream
        if self.real and self.kb is not None:
            lib.kb_gather(s, self.M, self.C, a.real, a.imag, self.kb.ptr, self.grid.ptr, self.C,
                          (ctypes.c_int64 * 3)(*self.oN), self.ksp.ptr, self.C)
        elif self.real:
            lib.ccsrmm_ilr(s, self.M, self.on, self.C, self.nnz, a.real, a.imag, self.g_pk.ptr, self.g_ptr.ptr,
                           self.grid.ptr, self.C, self.ksp.ptr, self.C, self.g_map.ptr, self.staged_fwd, None, 0, 0)
        else:
            lib.ccsrmm_il(s, self.M, self.on, self.C, self.nnz, a.real, a.imag, G.values.ptr, G.colInds.ptr,
                          G.rowPtrs.ptr, self.grid.ptr, self.C, self.ksp.ptr, self.C, None, 0, None, 0, 0)

    def _samples_to_grid(self):
        lib, s = self.B._lib, self.B._stream
        lr = self.longrows.ptr if self.nlong else None
        u = complex(self.gphase).conjugate()
        ur, ui = float(u.real), float(u.imag)
        if self.real and self.tiles is not None:
            t = self.tiles
            lib.kb_blocks_apply(s, self.C, t['shape'][0], t['shape'][1], ur, ui, t['nwork'], t['work'].ptr, t['ent'].ptr,
                                self.ksp.ptr, self.C, self.grid.ptr, self.C, self.rowmap.ptr, t['nsplit'], t['split'].ptr,
                                t['scratch'].ptr, int(self.tiles_lanes))
        elif self.real and self.runs is not None:
            r = self.runs
            lib.ccsrmm_runs(s, self.kp, self.C, ur, ui, r['ptr'].ptr, r['ids'].ptr, r['w4'].ptr, self.ksp.ptr, self.C,
                            self.grid.ptr, self.C, self.rowmap.ptr, r['seg'], r['segd'].ptr, r['nseg'], r['spld'].ptr,
                            r['nsplit'], r['scratch'].ptr)
        elif self.real:
            lib.ccsrmm_ilr(s, self.kp, self.M, self.C, self.nnz, ur, ui, self.t_pk.ptr, self.t_ptr.ptr,
                           self.ksp.ptr, self.C, self.grid.ptr, self.C, self.rowmap.ptr, self.staged_adj, lr, self.nlong,
                           self.long_thresh)
        else:
            lib.ccsrmm_il(s, self.kp, self.M, self.C, self.nnz, ur, ui, self.t_val.ptr, self.t_ind.ptr,
                          self.t_ptr.ptr, self.ksp.ptr, self.C, self.grid.ptr, self.C, self.rowmap.ptr, 1,
                          lr, self.nlong, self.long_thresh)

    def ifft_combine(self, y, alpha=1.0, beta=0.0):
        a, b = complex(alpha), complex(beta)
        lib, s = self.B._lib, self.B._stream
        if self.probe is None:
            lib.sense_ifft_combine(self._plan, s, y.ptr, self.grid.ptr, self.pf.ptr, a.real, a.imag, b.real, b.imag)
            return
        for which, label in ((3, "fft_pass[z inv]"), (4, "fft_pass[y inv]"), (5, "sense_combine_pk[x]")):
            with self.probe(label):
                lib.sense_pass(self._plan, s, which, self.grid.ptr, None, y.ptr, self.pf.ptr, a.real, a.imag, b.real, b.imag)


def make_fused_classes(ops):
    """Fused node classes on top of the operator family `ops` (indigo_b200.linop or the
    reference's indigo.operators)."""

    class FusedSenseNUFFT(ops.Operator):
        """A = KronI(C, G' F) P : image (nvox) -> multi-coil k-space (M*C), and its adjoint."""

        def __init__(self, backend, dev, name='SENSE1.fused'):
            ops.Operator.__init__(self, backend, name=name)
            self._dev = dev

        shape = property(lambda self: (self._dev.M * self._dev.C, self._dev.nvox))
        dtype = property(lambda self: _C64)

        def _mem_usage(self, ncols=1):
            return 0

        def _eval(self, y, x, alpha=1, beta=0, forward=True, left=True):
            if not left:
                raise NotImplementedError("Right-multiplication not implemented for FusedSenseNUFFT.")
            assert x.shape[1] == 1, "fused SENSE operator takes one image / one multi-coil data set at a time"
            d, B = self._dev, self._backend
            lib, s = B._lib, B._stream
            b = complex(beta)
            if forward:
                d.expand_fft(x)
                d.grid_to_samples(alpha)
                if d.ksp_sorted:
                    lib.deinterleave_rows(s, d.M, d.C, d.ksp.ptr, d.C, b.real, b.imag, y.ptr, d.M, d.pos.ptr)
                else:
                    lib.deinterleave(s, d.M, d.C, d.ksp.ptr, d.C, b.real, b.imag, y.ptr, d.M)
            else:
                if d.ksp_sorted:
                    lib.interleave_rows(s, d.M, d.C, x.ptr, d.M, d.ksp.ptr, d.C, d.pos.ptr)
                else:
                    lib.interleave(s, d.M, d.C, x.ptr, d.M, d.ksp.ptr, d.C)
                d.samples_to_grid()
                d.ifft_combine(y, alpha, beta)

        @property
        def normal(self):
            return FusedSenseNormal(self._backend, self._dev)

    class FusedSenseNormal(ops.Operator):
        """A^H A : image -> image; k-space stays coil-interleaved between the two gathers."""

        def __init__(self, backend, dev, name='SENSE.fused'):
            ops.Operator.__init__(self, backend, name=name)
            self._dev = dev

        shape = property(lambda self: (self._dev.nvox, self._dev.nvox))
        dtype = property(lambda self: _C64)

        def _mem_usage(self, ncols=1):
            return 0

        def _eval(self, y, x, alpha=1, beta=0, forward=True, left=True):
            if not left:
                raise NotImplementedError("Right-multiplication not implemented for FusedSenseNormal.")
            assert x.shape[1] == 1
            d = self._dev
            d.expand_fft(x)
            d.grid_to_samples()
            d.samples_to_grid()
            d.ifft_combine(y, alpha, beta)

    class FusedSenseToeplitz(ops.Operator):
        """T ~ A^H A : image -> image as a zero-padded FFT convolution (toeplitz_normal); no gridding."""

        def __init__(self, backend, tdev, name='SENSE.toeplitz'):
            ops.Operator.__init__(self, backend, name=name)
            self._tdev = tdev

        shape = property(lambda self: (self._tdev.nvox, self._tdev.nvox))
        dtype = property(lambda self: _C64)

        def _mem_usage(self, ncols=1):
            return 0

        def _eval(self, y, x, alpha=1, beta=0, forward=True, left=True):
            if not left:
                raise NotImplementedError("Right-multiplication not implemented for FusedSenseToeplitz.")
            if x.shape[1] != 1:
                raise ValueError("FusedSenseToeplitz takes one image at a time (got %d columns)" % x.shape[1])
            self._tdev.apply(y, x, alpha, beta)

    return FusedSenseNUFFT, FusedSenseNormal, FusedSenseToeplitz


_cache = {}


def _classes(ops):
    if ops not in _cache:
        _cache[ops] = make_fused_classes(ops)
    return _cache[ops]


def sense_operator_fused(B, N, coord, maps, oversamp=2.0, weights=None, width=3, n=128):
    """The SENSE operator of examples/pics.py:92-95 as one fused node (same arguments as
    indigo_b200.sense.sense_operator).  Raises RuntimeError when the oversampled grid has no
    specialised FFT passes; callers then fall back to sense_operator_device / sense_operator."""
    from .sense import _ops_of
    Fwd = _classes(_ops_of(B))[0]
    dev = SenseDevice(B, N, coord, maps, oversamp, weights, width, n)
    return Fwd(B, dev)


# ---------------------------------------------------------------------------------------------------------
# Toeplitz embedding of the normal operator.  The normal operator of a non-uniform DFT is Toeplitz:
#     A^H A x = s^2 * sum_c conj(S_c) .* crop_N( IFFT_L( K .* FFT_L( pad_L(S_c .* x) ) ) ),
#     K = Re FFT_L(p_sym) / prod(L),   p(d) ~ sum_m w_m^2 exp(+2 pi i kappa_m . d),  d in (-L/2, L/2)^3,
# with L >= 2N - 1 per axis, so that every lag between two voxels of the image has its own grid point.  CG
# applies A^H A fifty times per solve; this form has no gridding, no per-sample work and no k-space buffer in
# the loop.  It is a different discretisation of the same model (DESIGN.md section 9): p comes from the gridded
# adjoint the fused operator already has, on an image of L points per axis, so it carries the same Kaiser-Bessel
# conventions, and s^2 is the least-squares fit of T to the gridded normal operator.
TOEPLITZ_LENGTHS = (32, 52, 64, 104, 128, 192, 208, 256, 320, 384, 416, 448, 512, 640, 768, 832, 1024)
TOEPLITZ_MAX = 512                  # longest axis of the convolution pass (ib200_sense_toeplitz_pass)
TOEPLITZ_AUX_MAX = 832              # longest oversampled axis of the PSF's auxiliary operator: the fused passes of
                                    # 1024-point axes do not fit shared memory (so 2-D 256^2 images are not served)
TOEPLITZ_PROBE_SEED = 20            # seed of the probe image of the scale fit


def toeplitz_grid(N, oversamp=2.0):
    """Padded grid L of the Toeplitz embedding: per axis the smallest length L_d >= 2 N_d - 1 such that L_d and
    the oversampled grid of an image of L_d points both have specialised passes that fit (1 for a one-point axis).
    Raises RuntimeError when no such length exists."""
    os3 = oversamp if isinstance(oversamp, tuple) else (oversamp,) * 3
    L = []
    for d, (nd, o) in enumerate(zip(N, os3)):
        nd = int(nd)
        if nd == 1:
            L.append(1)
            continue
        ok = [l for l in TOEPLITZ_LENGTHS if l >= 2 * nd - 1 and l <= TOEPLITZ_MAX and int(l * o) in TOEPLITZ_LENGTHS
              and int(l * o) <= TOEPLITZ_AUX_MAX]
        if not ok:
            raise RuntimeError("Toeplitz normal operator: no padded grid length with specialised passes for axis %d "
                               "of %d points (oversampling %g)" % (d, nd, o))
        L.append(ok[0])
    if int(N[2]) > 1 and L[2] == 1:
        raise RuntimeError("Toeplitz normal operator: bad image shape %s" % (tuple(N),))
    return tuple(L)


class ToeplitzDevice(object):
    """Device-resident pieces of one Toeplitz normal operator: plan on the padded grid, kernel K, scale s^2."""

    probe = None          # as SenseDevice.probe: label -> context manager around every pass of an apply

    def __init__(self, dev, team=None):
        from .sense import _ops_of
        B = self.B = dev.B
        lib, s = B._lib, B._stream
        self.N, self.C, self.nvox = dev.N, dev.C, dev.nvox
        self.L = L = toeplitz_grid(dev.N, dev.oversamp)
        self.nL = nL = int(np.prod(L))
        self.three = L[2] > 1
        self._plan = None
        # plan first: raises RuntimeError (unsupported) before anything large is built
        plan = ctypes.c_void_p()
        lib.sense_plan_create(ctypes.byref(plan), (ctypes.c_int64 * 3)(*self.N), (ctypes.c_int64 * 3)(*L), self.C)
        self._plan = plan
        # 1. PSF: adjoint of an auxiliary fused operator on an image of L points, applied to the k-space [w, 0]
        #    (maps (1, 0): two coils keep it on the matrix-free construction)
        aux_maps = np.zeros(L + (2,), dtype=_C64, order='F')
        aux_maps[..., 0] = 1
        aux = SenseDevice(B, L, dev.coord, aux_maps, dev.oversamp, dev.weights, dev.width, dev.n)
        del aux_maps
        ksp = np.zeros((aux.M * 2, 1), dtype=_C64, order='F')
        ksp[:aux.M, 0] = 1 if dev.weights is None else np.asarray(dev.weights, dtype=np.float32).reshape(-1, order='F')
        ksp_d = B.copy_array(ksp)
        del ksp
        img = B.empty_array((nL, 1), _C64, name='toeplitz.psf_image')
        _classes(_ops_of(B))[0](B, aux)._eval(img, ksp_d, forward=False)
        del ksp_d, aux
        # 2. symmetrise into circular order, 3. L-point FFT, 4. K = Re(.) / prod(L)
        psf = B.empty_array((nL, 1), _C64, name='toeplitz.psf')
        lib.toeplitz_psf(s, (ctypes.c_int64 * 3)(*L), img.ptr, psf.ptr)
        del img
        fplan = ctypes.c_void_p()
        lib.fft_plan_create(ctypes.byref(fplan), 3, (ctypes.c_int64 * 3)(*L), 1)
        try:
            lib.fft_exec(fplan, s, psf.ptr, psf.ptr, -1)
            self.kernel = B.empty_array((nL,), np.dtype('float32'), name='toeplitz.K')
            lib.toeplitz_kernel(s, nL, psf.ptr, 1.0 / nL, self.kernel.ptr)
            lib.stream_sync(s)
        finally:
            lib.fft_plan_destroy(fplan)
        del psf
        self.grid = B.empty_array((nL * self.C,), _C64, name='toeplitz.grid[z][y][x][c]')
        self.pf = B.copy_array(np.ascontiguousarray(dev.maps.reshape((self.nvox, self.C), order='F').astype(_C64)).reshape(-1))
        # 5. scale: s^2 = Re<T1 v, N v> / ||T1 v||^2 with T1 = T at s = 1 and N the gridded normal operator, both
        #    with the unit map on coil 0.  The fit depends on the trajectory only, not on the maps, so every coil
        #    shard of an operator finds the same s^2 and the shards' T add up to the whole operator's T; with a
        #    team the two sums are all-reduced as well, which makes s^2 bit-identical on every rank.
        self.s2 = 1.0
        rs = np.random.RandomState(TOEPLITZ_PROBE_SEED)
        v = B.copy_array((rs.rand(self.nvox, 1) + 1j * rs.rand(self.nvox, 1)).astype(_C64, order='F'))
        unit = np.zeros((self.nvox, self.C), dtype=_C64)
        unit[:, 0] = 1
        pf_t = B.copy_array(unit.reshape(-1))
        unit[:, 0] = dev.q
        pf_a = B.copy_array(unit.reshape(-1))
        del unit
        tv = B.empty_array((self.nvox, 1), _C64, name='toeplitz.probe.T')
        av = B.empty_array((self.nvox, 1), _C64, name='toeplitz.probe.AHA')
        self._passes(tv, v, pf_t, 1.0, 0.0)
        lib.sense_expand_fft(dev._plan, s, dev.grid.ptr, v.ptr, pf_a.ptr)
        dev.grid_to_samples()
        dev.samples_to_grid()
        lib.sense_ifft_combine(dev._plan, s, av.ptr, dev.grid.ptr, pf_a.ptr, 1.0, 0.0, 0.0, 0.0)
        num, den = B.dot(tv, av), B.norm2(tv)
        if team is not None:
            num, den = team.allreduce(num), team.allreduce(den)
        if not den > 0:
            raise RuntimeError("Toeplitz normal operator: the trajectory gives an empty point-spread function")
        self.s2 = float(num) / float(den)
        del v, pf_t, pf_a, tv, av

    def __del__(self):
        try:
            if getattr(self, '_plan', None):
                self.B._lib.sense_plan_destroy(self._plan)
        except Exception:
            pass

    def _step(self, label):
        import contextlib
        return self.probe(label) if self.probe is not None else contextlib.nullcontext()

    def _passes(self, y, x, pf, alpha, beta):
        lib, s, g = self.B._lib, self.B._stream, self.grid.ptr
        a, b = complex(alpha) * self.s2, complex(beta)
        with self._step("sense_expand_pk[x]"):
            lib.sense_pass(self._plan, s, 0, g, x.ptr, None, pf.ptr, 1.0, 0.0, 0.0, 0.0)
        if self.three:
            with self._step("fft_pass[y fwd]"):
                lib.sense_pass(self._plan, s, 1, g, None, None, None, 1.0, 0.0, 0.0, 0.0)
        with self._step("toeplitz_pass[%s]" % ("z" if self.three else "y")):
            lib.sense_toeplitz_pass(self._plan, s, g, self.kernel.ptr)
        if self.three:
            with self._step("fft_pass[y inv]"):
                lib.sense_pass(self._plan, s, 4, g, None, None, None, 1.0, 0.0, 0.0, 0.0)
        with self._step("sense_combine_pk[x]"):
            lib.sense_pass(self._plan, s, 5, g, None, y.ptr, pf.ptr, a.real, a.imag, b.real, b.imag)

    def apply(self, y, x, alpha=1.0, beta=0.0):
        """y = alpha * T x + beta * y (beta == 0 never reads y)."""
        self._passes(y, x, self.pf, alpha, beta)


def toeplitz_normal(A, team=None):
    """Toeplitz-embedded normal operator T ~ A^H A of a fused SENSE operator (from sense_operator_fused or
    fuse_transform): an operator of the same family, shape (nvox, nvox), applied as a zero-padded FFT convolution
    with a real kernel built once here.  It is not bit-parity with A^H A (DESIGN.md section 9): use it where the
    gridded normal operator would go, e.g. B.cg(toeplitz_normal(A), A.H * y, x, lamda=...).  With a coil-sharded
    operator pass the CoilTeam: every rank then uses the same scale.  Raises TypeError for any other operator and
    RuntimeError when the padded grid has no specialised passes."""
    dev = getattr(A, '_dev', None)
    if not isinstance(dev, SenseDevice):
        raise TypeError("toeplitz_normal takes a fused SENSE operator (sense_operator_fused / fuse_transform), got %s"
                        % type(A).__name__)
    from .sense import _ops_of
    Toep = _classes(_ops_of(A._backend))[2]
    return Toep(A._backend, ToeplitzDevice(dev, team), name=(getattr(A, '_name', '') or 'SENSE') + '.toeplitz')


# ---------------------------------------------------------------------------------------------------------
# The fusion as a Transform (SURVEY.md section 8f rank 1: "a new visitor in the style of pics.py:104-177 /
# transforms.py:202-249"): trees built by the unchanged recipe of examples/pics.py:92-95,
#     A = KronI(C, [Diag(dcf) *] B.NUFFT(M, N, coord)) * VStack_c Diag(maps_c),
# are recognised and replaced by the fused node; anything else is left as it is.  The interpolation matrix
# alone does not determine the trajectory, so B200Backend.NUFFT tags the product it returns with the
# arguments it was built from (`tag_nufft`); maps and row weights are read back from the diagonal matrices.
def tag_nufft(op, N, coord, width, n, oversamp):
    op._b200_nufft = dict(N=tuple(int(v) for v in N), coord=np.asarray(coord), width=width, n=n, oversamp=oversamp)
    return op


def _diagonal_of(node):
    """Diagonal of an SpMatrix node that holds a square diagonal matrix, else None."""
    if type(node).__name__ != 'SpMatrix':
        return None
    M = node._matrix
    if M.shape[0] != M.shape[1] or M.nnz > M.shape[0]:
        return None
    coo = M.tocoo()
    if not np.array_equal(coo.row, coo.col):
        return None
    return np.asarray(M.diagonal())


def match_sense_tree(node):
    """Arguments of the SENSE operator a Product node was built from (dict with N, coord, maps, weights, oversamp,
    width, n), or None when the node is not KronI(C, [Diag *] NUFFT) * VStack(Diag...)."""
    if type(node).__name__ != 'Product':
        return None
    kids = node.children
    if len(kids) != 2 or type(kids[0]).__name__ != 'Kron' or type(kids[1]).__name__ != 'VStack':
        return None
    eye, F1 = kids[0].children
    if type(eye).__name__ != 'Eye':
        return None
    C = int(eye.shape[0])
    weights, meta = None, getattr(F1, '_b200_nufft', None)
    if meta is None and type(F1).__name__ == 'Product' and len(F1.children) == 2:
        D, F2 = F1.children
        meta, weights = getattr(F2, '_b200_nufft', None), _diagonal_of(D)
        if meta is None or weights is None:
            return None
    if meta is None:
        return None
    N = meta['N']
    nvox = int(np.prod(N))
    coils = kids[1].children
    if len(coils) != C:
        return None
    cols = []
    for ch in coils:
        d = _diagonal_of(ch)
        if d is None or d.shape[0] != nvox:
            return None
        cols.append(d.astype(_C64))
    maps = np.stack(cols, axis=1).reshape(tuple(N) + (C,), order='F')
    if weights is not None:
        if np.abs(np.imag(weights)).max() > 0:
            return None                                    # complex row weights are not a density compensation
        weights = np.real(weights).astype(np.float32)
    return dict(N=N, coord=meta['coord'], maps=maps, weights=weights, oversamp=meta['oversamp'],
                width=meta['width'], n=meta['n'])


def fuse_transform(B):
    """Transform class of B's operator family whose visit() swaps recognised SENSE trees for the fused node:
        A = A.optimize([fuse_transform(B)])        # or: sense_operator(B, ..., recipe=[fuse_transform(B)])
    Grids without specialised passes (RuntimeError from the plan) keep their tree."""
    if getattr(B, 'ops', None) is not None:
        raise RuntimeError("fuse_transform rewrites trees of the reference's operator family; this backend was "
                           "built without the reference package (use sense_operator_fused directly)")
    from indigo.transforms import Transform

    class FuseSenseNUFFT(Transform):
        build = staticmethod(lambda backend, **kw: sense_operator_fused(backend, kw['N'], kw['coord'], kw['maps'], kw['oversamp'],
                                                                        kw['weights'], kw['width'], kw['n']))

        def visit_Product(self, node):
            hit = match_sense_tree(node)
            if hit is None:
                return self.generic_visit(node)
            try:
                fused = type(self).build(node._backend, **hit)
            except RuntimeError:
                return self.generic_visit(node)
            fused._name = (getattr(node, '_name', '') or 'SENSE1') + '.fused'
            return fused

    return FuseSenseNUFFT
