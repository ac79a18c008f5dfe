/*
 * indigo_b200.h -- C ABI of libindigo_b200.so, the B200 (sm_100a) execution
 * layer behind indigo's `Backend` interface.
 *
 * This header is the drop-in boundary.  Every entry point replaces one method
 * of the reference's abstract backend (indigo/backends/backend.py) exactly as
 * the reference's own GPU backend binds its libraries through ctypes
 * (indigo/backends/cuda.py:14-18,51-62): plain pointers and sizes, no C++ or
 * torch types, `int` status returns.  INTEGRATION.md shows the ctypes stub a
 * maintainer adds on the reference side.
 *
 * Conventions
 *   - status: 0 = OK; >0 = cudaError_t; <0 = IB200_E_* below.  Nothing throws.
 *     ib200_last_error() returns a thread-local message for the last failure.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *     Compute entry points enqueue work and DO NOT synchronise, except the few
 *     that return a host scalar (documented per function).
 *   - all matrices are complex64 (interleaved re,im floats), column-major,
 *     addressed as ptr[row + col*ld]; `ld` is in ELEMENTS and may be far larger
 *     than the row count (views into indigo's scratch arena, SURVEY.md
 *     landmine 4).  Pointers need only be 8-byte aligned.
 *   - beta == 0 means "overwrite": Y is never read (the arena is uninitialised,
 *     indigo/transforms.py:73-76).
 *   - sparse indices are 0-based int32 (indigo/backends/backend.py:539,549-550).
 */
#ifndef INDIGO_B200_H
#define INDIGO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IB200_E_INVALID   (-1)   /* bad argument                               */
#define IB200_E_UNSUPPORTED (-2) /* valid request this build cannot serve      */
#define IB200_E_NOMEM     (-3)   /* host allocation failed                     */

#define IB200_FFT_FORWARD (-1)   /* same sign convention as cuda.py:427-428    */
#define IB200_FFT_INVERSE (+1)

const char *ib200_last_error(void);
int ib200_version(void);
/* Fills sm_count, max opt-in shared memory per block, L2 bytes, total global
 * memory for device `dev`; any out pointer may be NULL. */
int ib200_device_info(int dev, int *sm_count, int64_t *smem_optin, int64_t *l2_bytes, int64_t *mem_bytes);
/* How many kernels this library has launched since load (bench.py's
 * `gpu_launches`); reset with ib200_launch_count_reset(). */
int64_t ib200_launch_count(void);
void ib200_launch_count_reset(void);

/* ------------------------------------------------------------------ arrays
 * Backend.dndarray._copy_from/_copy_to/_copy/_zero, backend.py:187-215;
 * pitched-copy model of cuda.py:127-181.  kind: 0 = D2D, 1 = H2D, 2 = D2H.
 * Asynchronous on `stream`; H2D/D2H from pageable memory behave like
 * cudaMemcpy2DAsync (staged).  ib200_stream_sync is Backend.barrier(),
 * backend.py:246 / cuda.py:120-121. */
int ib200_copy2d(void *stream, void *dst, int64_t dpitch_bytes, const void *src, int64_t spitch_bytes,
                 int64_t width_bytes, int64_t height, int kind);
int ib200_memset0(void *stream, void *dst, int64_t nbytes);
int ib200_stream_sync(void *stream);

/* ------------------------------------------------------------------ BLAS-1
 * Backend.axpby / scale / dot / norm2, backend.py:453-467 (oracle np.py:53-74).
 * n counts complex elements. */
int ib200_caxpby(void *stream, int64_t n, float beta_re, float beta_im, void *y,
                 float alpha_re, float alpha_im, const void *x);            /* y = beta*y + alpha*x */
int ib200_cscal(void *stream, int64_t n, float alpha_re, float alpha_im, void *x);
/* Device-resident results (no sync): out[0..1] = sum conj(x)*y as doubles. */
int ib200_cdotc_dev(void *stream, int64_t n, const void *x, const void *y, double *dev_out2);
/* out[0] = sum |x|^2 as a double. */
int ib200_scnrm2sq_dev(void *stream, int64_t n, const void *x, double *dev_out1);
/* Host-returning forms used by Backend.dot / Backend.norm2: run the reduction,
 * copy the scalar back and synchronise `stream`.  *host_re = Re(x^H y) (the
 * reference returns only the real part, np.py:64); *host_out = ||x||^2
 * (SQUARED, np.py:69). */
int ib200_cdotc(void *stream, int64_t n, const void *x, const void *y, double *host_re, double *host_im);
int ib200_scnrm2sq(void *stream, int64_t n, const void *x, double *host_out);

/* Fused CG vector updates for Backend.cg, backend.py:666-679.  All scalars
 * live in device memory (doubles) so one iteration needs no host round trip:
 *   ib200_cg_xr : alpha = rr/pAp;  x += alpha*p;  r -= alpha*Ap;  r2 = ||r||^2
 *   ib200_cg_p  : beta = r2/rr;    p = beta*p + r;                 rr = r2
 * `scal` points at 4 device doubles {rr, Re(p^H Ap), Im(p^H Ap), r2}; fill
 * scal[1..2] with ib200_cdotc_dev(stream, n, p, Ap, scal + 1). */
int ib200_cg_xr(void *stream, int64_t n, void *x, void *r, const void *p, const void *Ap, double *scal);
int ib200_cg_p(void *stream, int64_t n, void *p, const void *r, double *scal);

/* ------------------------------------------------------------------ sparse
 * Backend.ccsrmm, backend.py:514-519 (oracle np.py:120-127; native reference
 * _customcpu.c:14-114, _customgpu.cu:49-81, cuda.py:582-596):
 *   adjoint == 0 : Y(m x ncols) = alpha * A      * X(k x ncols) + beta * Y
 *   adjoint != 0 : Y(k x ncols) = alpha * A^H    * X(m x ncols) + beta * Y
 * A is m x k CSR (rowptr[m+1], colind[nnz], vals[nnz]; nnz is passed like
 * cusparseCcsrmm's, cuda.py:590, and only steers the thread-per-row split).
 * `exwrite` promises
 * that no two stored entries share a column (scatter without atomics). */
int ib200_ccsrmm(void *stream, int adjoint, int exwrite, int64_t m, int64_t k, int64_t ncols, int64_t nnz,
                 float alpha_re, float alpha_im, const void *vals, const int32_t *colind, const int32_t *rowptr,
                 const void *X, int64_t ldx, float beta_re, float beta_im, void *Y, int64_t ldy);
/* Coil-interleaved fast path of Backend.ccsrmm for 2..32 right-hand-side columns
 * (same reference interface: backend.py:514-519; the layout conversion replaces
 * the strided per-coil gathers the column-major interface would force).
 *   ib200_interleave   : Xil[r*pitch + c] = X[r + c*ldx]
 *   ib200_ccsrmm_il    : Yil[r*ypitch + c] = alpha * sum_p vals[p] * Xil[colind[p]*xpitch + c]
 *   ib200_deinterleave : Y[r + c*ldy] = Yil[r*pitch + c] + beta * Y[r + c*ldy]
 * The adjoint product uses the same entry on the stored conjugate transpose
 * (ib200_csr_transpose_conj), so neither direction needs atomics. */
int ib200_interleave(void *stream, int64_t rows, int64_t ncols, const void *X, int64_t ldx, void *Xil, int64_t pitch);
int ib200_deinterleave(void *stream, int64_t rows, int64_t ncols, const void *Yil, int64_t pitch,
                       float beta_re, float beta_im, void *Y, int64_t ldy);
/* Same with a row permutation on the interleaved side: row r of X goes to / comes from row perm[r] of the
 * interleaved array (fused SENSE recipe: k-space is kept in tile-sorted sample order internally).
 * ib200_invert_perm writes inv[perm[i]] = i. */
int ib200_interleave_rows(void *stream, int64_t rows, int64_t ncols, const void *X, int64_t ldx, void *Xil, int64_t pitch,
                          const int32_t *perm);
int ib200_deinterleave_rows(void *stream, int64_t rows, int64_t ncols, const void *Yil, int64_t pitch,
                            float beta_re, float beta_im, void *Y, int64_t ldy, const int32_t *perm);
int ib200_invert_perm(void *stream, int64_t n, const int32_t *perm, int32_t *inv);
int ib200_ccsrmm_il(void *stream, int64_t m, int64_t k, int64_t ncols, int64_t nnz, float alpha_re, float alpha_im,
                    const void *vals, const int32_t *colind, const int32_t *rowptr,
                    const void *Xil, int64_t xpitch, void *Yil, int64_t ypitch,
                    const int32_t *rowmap, int rows_per_group,
                    const int32_t *longrows, int nlong, int long_thresh);
/* Real-weight form of the same product for matrices whose values are real (gridding matrices on
 * grids whose extents are multiples of four: the centring phase is +-1).  ib200_csr_pack_real
 * writes packed[p] = {int32 colind[p], float Re vals[p]} (8 bytes per entry) and returns
 * host_max = {max |Re|, max |Im|} so that the caller can decide whether dropping the imaginary
 * parts is admissible (synchronises).  ib200_ccsrmm_ilr is ib200_ccsrmm_il on packed entries. */
int ib200_csr_pack_real(void *stream, int64_t nnz, const void *vals, const int32_t *colind, void *packed,
                        float host_max[2]);
int ib200_ccsrmm_ilr(void *stream, int64_t m, int64_t k, int64_t ncols, int64_t nnz, float alpha_re, float alpha_im,
                     const void *packed, const int32_t *rowptr, const void *Xil, int64_t xpitch,
                     void *Yil, int64_t ypitch, const int32_t *rowmap, int rows_per_group,
                     const int32_t *longrows, int nlong, int long_thresh);
/* rowmap (optional, m int32): row r of the matrix is written to output row rowmap[r]; negative
 * entries are padding rows and write nothing.  rows_per_group: consecutive-row blocking factor of
 * the kernel (0 = automatic).  Both exist for matrices whose rows were stored in tile-major
 * order of a 3-D grid so that the rows one CTA owns share their operands:
 * ib200_grid_tile_rank fills colrank[g] = padded tile-major rank of grid point g (x fastest)
 * and rowmap[rank] = g (or -1 for padding); *padded_rows = number of ranks.  Pass NULL for both
 * arrays to query the size only. */
/* Stable re-ordering of the ROWS of a packed CSR matrix by the key colrank[first column of the row]
 * (rows without entries go last): rowptr_out[m+1] / packed_out[nnz] hold the permuted matrix and
 * rowmap_out[i] the original index of permuted row i, to be passed as `rowmap` to the products
 * above.  With colrank from ib200_grid_tile_rank the samples of a trajectory end up grouped by
 * the grid tile they fall into, so consecutive rows share operand lines in all three dimensions,
 * not only along the readout.  nranks = number of distinct ranks (padded_rows).  Synchronises. */
int ib200_csr_permute_rows(void *stream, int64_t m, int64_t nnz, const int32_t *rowptr, const void *packed,
                           const int32_t *colrank, int64_t nranks, int32_t *rowptr_out, void *packed_out,
                           int32_t *rowmap_out);
/* Rows with more than long_thresh entries (the k-space centre of a radial trajectory puts ~80 000
 * entries into single rows of the stored adjoint) are listed once by ib200_csr_long_rows
 * (count returned through *host_count; call with capacity 0 to size the list; synchronises) and
 * passed to the two products above as longrows[nlong]: each such row is then served by a whole
 * CTA instead of one lane group.  nlong == 0 disables the split. */
int ib200_csr_long_rows(void *stream, int64_t m, const int32_t *rowptr, int thresh, int32_t *list, int capacity,
                        int *host_count);
/* Two-level form: tiles grouped into super-tiles of super[0] x super[1] x super[2] tiles (super-tile major,
 * then tile major, then point).  Only colrank is produced (NULL: size query); used as the sort key of the
 * samples for ib200_csr_permute_rows so that the samples in flight cover a compact, L2-sized block. */
int ib200_grid_tile_rank2(void *stream, const int64_t grid[3], const int64_t tile[3], const int64_t super[3],
                          int32_t *colrank, int64_t *nranks);
int ib200_grid_tile_rank(void *stream, const int64_t grid[3], const int64_t tile[3], int32_t *colrank, int32_t *rowmap,
                         int64_t *padded_rows);
/* Separable Kaiser-Bessel gridding (the product ccsrmm(G') of the -O3 SENSE tree, SURVEY.md 3.1,
 * without a stored matrix).  interp.py:19-60 emits every value of a row as li(x)*li(y)*li(z) and the
 * -O2 recipe multiplies in the centring phase and the grid scale (backend.py:349-364), all of which
 * factor over the axes.  ib200_kb_records writes one record of ib200_kb_record_bytes() (96) bytes per
 * sample: 3 x 6 float32 weights (f0/f1/f2 = per-axis real factors of mod*scale, indexed by grid
 * coordinate; rowweight = optional per-sample weight), the first tap of each axis wrapped into the grid,
 * the tap counts and the output row.  Record r describes sample perm[r] (perm NULL: identity), so the
 * records can be stored in the tile-sorted order ib200_csr_permute_rows produces while results land
 * in the original rows (out_is_record == 0) or in row r itself (out_is_record != 0: k-space kept in the
 * sorted order between the two gridding steps, so that neighbouring samples are neighbours in memory).  *host_flag != 0 on return means some sample needs more than 6 taps on an axis
 * (or the grid is smaller than the kernel): the caller must stay on the stored-matrix path.
 * Synchronises.  ib200_kb_gather computes Yil[out][c] = alpha * sum_taps w * Xil[tap][c] for ncols
 * interleaved columns (Xil = grid[z][y][x][c] with `xpitch` elements per grid point). */
int ib200_kb_record_bytes(void);
int ib200_kb_records(void *stream, int64_t m, const double *coord, const int64_t grid[3], double width,
                     const double *table, int ntable, const float *rowweight, const float *f0, const float *f1,
                     const float *f2, const int32_t *perm, int out_is_record, void *records, int *host_flag);
int ib200_kb_gather(void *stream, int64_t m, int64_t ncols, float alpha_re, float alpha_im, const void *records,
                    const void *grid_il, int64_t xpitch, const int64_t grid[3], void *Yil, int64_t ypitch);
/* Matrix-free construction of the fused SENSE operator (no CSR matrix, no stored adjoint):
 *   ib200_kb_sample_order: perm[r] = sample at position r when the samples are sorted (stably) by the two-level tile
 *     rank (ib200_grid_tile_rank2 with the same tile / super extents) of their first tap -- the order
 *     ib200_csr_permute_rows derives from the first column of every row of G'.
 *   ib200_kb_support_windows: the windows of ib200_grid_support_windows from the separable records (the hull along z of
 *     the taps of every record, zero-weight taps included, like the explicit zeros of the reference's matrix).
 * Both synchronise. */
int ib200_kb_sample_order(void *stream, int64_t m, const double *coord, const int64_t grid[3], double width,
                          const int64_t tile[3], const int64_t super[3], int32_t *perm);
int ib200_kb_support_windows(void *stream, int64_t m, const void *records, const int64_t grid[3], int64_t kp,
                             const int32_t *rowmap, const int64_t block[3], int32_t *win, int32_t *rowmap_out,
                             int64_t *host_inside);
/* x-run form of a stored adjoint in tile-major row order (fused SENSE recipe, csrc/csrmm_runs.cu): the four
 * consecutive rows that form one x-row of a 4x4x4 tile are merged into one list of (sample, 4 weights)
 * entries, padded to a multiple of four entries.  ib200_csr_runs_count fills run_ptr[kp/4 + 1] and returns
 * the number of run entries, and -- for runs longer than seg_len entries, which are cut into segments
 * of seg_len -- the number of segments and of such runs; ib200_csr_runs_fill writes ids[entries] (int32),
 * w4[entries] (4 floats each), seg_desc[4*segments] and split_desc[4*split runs] (int32 quadruples);
 * colmap (optional) renames the columns: ids hold colmap[col] (k-space kept in sorted sample order).
 * ib200_ccsrmm_runs computes Yil[rowmap[r]][c] = alpha * sum_p w(r,p) * Xil[col(r,p)][c] for all kp rows
 * (rowmap < 0: nothing stored) with an even number of interleaved columns; `scratch` holds the partial
 * sums of the segments: segments * 4 * 2*pow2ceil(ncols/2) complex words.  The first two synchronise. */
int ib200_csr_runs_count(void *stream, int64_t kp, const int32_t *rowptr, const void *packed, int seg_len,
                         int32_t *run_ptr, int64_t *host_entries, int *host_segments, int *host_split);
int ib200_csr_runs_fill(void *stream, int64_t kp, const int32_t *rowptr, const void *packed, int seg_len,
                        const int32_t *run_ptr, int32_t *ids, void *w4, int32_t *seg_desc, int32_t *split_desc,
                        const int32_t *colmap);
int ib200_ccsrmm_runs(void *stream, int64_t kp, int64_t ncols, float alpha_re, float alpha_im, const int32_t *run_ptr,
                      const int32_t *ids, const void *w4, const void *Xil, int64_t xpitch, void *Yil, int64_t ypitch,
                      const int32_t *rowmap, int seg_len, const int32_t *seg_desc, int nseg, const int32_t *split_desc,
                      int nsplit, void *scratch);
/* Block form of the adjoint gridding (csrc/kbblocks.cu; replaces ccsrmm(G', adjoint),
 * indigo/backends/backend.py:560-596, for the matrix that indigo/interp.py:19-80 emits).  Built from the
 * separable records of ib200_kb_records, no stored matrix: the grid is cut into blocks of 4 x by x bz points
 * ((by, bz) = (4,4), (2,2), (2,1) or (1,1), inside the 4x4x4 tiles of ib200_grid_tile_rank) and every (sample,
 * block) pair that meets is one entry (sample, wx[4], wy[by], wz[bz]); entries of a block are consecutive,
 * ordered by record, in batches of four (ib200_kb_blocks_batch_bytes(by, bz) bytes each, zero-weight padding).
 * rowmap[64*tile + (z*4 + y)*4 + x] is the output row of a point (< 0: nothing stored).  A block with more than
 * seg_batches batches is cut into several work items whose partial sums are added in a fixed order by a second
 * kernel.
 *   ib200_kb_blocks_count: fills bptr[blocks+1] (first batch of every block) and wptr[blocks+1] (first work item);
 *     host_totals[5] = {blocks, batches, work items, split blocks, work items of split blocks}.  Blocks without
 *     a row inside rowmap get nothing; blocks with rows but without samples get one empty work item (they are
 *     overwritten with zeros on every apply).
 *   ib200_kb_blocks_fill: writes entries[batches * batch_bytes], work[4 * work items], split[4 * split blocks].
 *   ib200_kb_blocks_apply: Yil[rowmap[point]][c] = alpha * sum_e wz_e wy_e wx_e * Xil[out(e)][c] for an even
 *     number of at most 64 interleaved columns (served in chunks of 16); scratch: (work items of split blocks) *
 *     4*by*bz * 2*pow2ceil(min(ncols,16)/2) complex words; lanes: 0 or the number of lanes (1, 2, 4, 8, 16) that
 *     share the rows of a block.
 * The first two synchronise. */
int ib200_kb_blocks_batch_bytes(int by, int bz);
int ib200_kb_blocks_count(void *stream, int64_t m, const void *records, const int64_t grid[3], int by, int bz,
                          const int32_t *rowmap, int seg_batches, int32_t *bptr, int32_t *wptr, int64_t *host_totals);
int ib200_kb_blocks_fill(void *stream, int64_t m, const void *records, const int64_t grid[3], int by, int bz, int seg_batches,
                         const int32_t *bptr, const int32_t *wptr, void *entries, int32_t *work, int32_t *split);
int ib200_kb_blocks_apply(void *stream, int64_t ncols, int by, int bz, float alpha_re, float alpha_im, int nwork,
                          const int32_t *work, const void *entries, const void *Xil, int64_t xpitch, void *Yil,
                          int64_t ypitch, const int32_t *rowmap, int nsplit, const int32_t *split, void *scratch, int lanes);
/* Pipe-Menon density compensation (csrc/dcf.cu; indigo_b200.sense.pipe_menon_dcf): w <- w / (I I^T w) with I the
 * Kaiser-Bessel interpolation matrix, on the structures of the block gather above with 4x4x4 blocks and of
 * ib200_kb_records (built without row weights, records in the sorted order with out = record position).
 *   ib200_kb_density_spread: grid[rowmap[point]] = sum_e wz_e wy_e wx_e * w[out(e)], a real grid of prod(oN)
 *     floats, for every point of a block that has a work item (points with rowmap < 0 are not written); scratch:
 *     (work items of split blocks) * 64 floats.  Deterministic (fixed summation order, no atomics).
 *   ib200_kb_density_update: per record q = inv_scale2 * sum_taps wz wy wx * grid[tap], then w[out] = w[out] / q, or
 *     0 when q <= 0 or is not finite.  inv_scale2 = 1 / scale^2 for the scale the records carry, so that q is
 *     (I I^T w) for the unscaled interpolation matrix.  residual (optional): 1 + ceil(m / 256) doubles of device
 *     memory; residual[0] receives sum_r (q_r - 1)^2 in a fixed summation order.
 * Neither synchronises. */
int ib200_kb_density_spread(void *stream, int nwork, const int32_t *work, const void *entries, const float *w, float *grid,
                            const int32_t *rowmap, int nsplit, const int32_t *split, float *scratch);
int ib200_kb_density_update(void *stream, int64_t m, const void *records, const float *grid, const int64_t dims[3],
                            float inv_scale2, float *w, double *residual);
/* k-space support windows of a trajectory (fused SENSE recipe only).  Given the stored adjoint of the
 * gridding matrix in tile-major row order (rowptr[kp+1], rowmap[kp] from ib200_grid_tile_rank) the
 * grid columns are grouped into blocks of block[0] x block[1] points; for each block the hull [lo, hi)
 * along z of the grid points that receive at least one sample is computed, rounded outwards to
 * multiples of block[2].  win[2*(y*n0+x)], win[2*(y*n0+x)+1] receive the interval of column (x, y)
 * ((0,0) when empty); rowmap_out is rowmap with every row outside its column's interval set to -1, so
 * that the adjoint gather stores nothing there.  *host_inside = grid points inside the windows.
 * Grid points outside are never read by the forward gridding and are exactly zero after the
 * adjoint gridding, so ib200_sense_plan_set_support lets the last forward FFT pass skip writing them
 * and the first inverse pass skip reading them (results are unchanged).  Synchronises. */
int ib200_grid_support_windows(void *stream, const int64_t grid[3], int64_t kp, const int32_t *rowptr,
                               const int32_t *rowmap, const int64_t block[3], int32_t *win, int32_t *rowmap_out,
                               int64_t *host_inside);
/* The inspector of _customcpu.c:179-215 on the device: out = {rows with >=1
 * entry, columns with >=1 entry, exwrite flag, max entries in one column}.
 * `work` is k int32 of device scratch.  Synchronises `stream`. */
int ib200_csr_inspect(void *stream, int64_t m, int64_t k, const int32_t *colind, const int32_t *rowptr,
                      int32_t *work, int64_t host_out[4]);
/* Device-side conjugate transpose of a CSR matrix (the "stored adjoint" used
 * for non-exclusive-write adjoints).  t_rowptr[k+1], t_colind[nnz], t_vals[nnz]
 * are caller-allocated device buffers; `work` is k+1 int32 of device scratch.
 * Output rows are sorted by column.  `colrank` (optional, k int32, a permutation
 * of 0..k-1) places the transposed row of column c at position colrank[c], so
 * that rows which are neighbours on a 3-D grid can be stored next to each other
 * (see ib200_grid_tile_rank); NULL keeps the natural order.  Synchronises `stream`. */
int ib200_csr_transpose_conj(void *stream, int64_t m, int64_t k, int64_t nnz,
                             const void *vals, const int32_t *colind, const int32_t *rowptr,
                             void *t_vals, int32_t *t_colind, int32_t *t_rowptr, int32_t *work,
                             const int32_t *colrank);
/* Backend.cdiamm, backend.py:521-526 (oracle np.py:129-136; _customgpu.cu:83-143).
 * A is m x k in DIA form; data is (data_cols x noffsets) column-major with column pitch
 * data_pitch, i.e. scipy's dia.data transposed (backend.py:610).  scipy does not promise
 * data_cols == k (todia() gives max column + 1, diags() can be wider): entry (d, j) is the value
 * in column j of diagonal d, columns >= data_cols hold nothing.
 *   adjoint == 0 : Y(m x n) = alpha*A*X(k x n) + beta*Y
 *   adjoint != 0 : Y(k x n) = alpha*A^H*X(m x n) + beta*Y */
int ib200_cdiamm(void *stream, int adjoint, int64_t m, int64_t k, int64_t ncols, int64_t noffsets,
                 const int32_t *offsets, const void *data, int64_t data_cols, int64_t data_pitch,
                 float alpha_re, float alpha_im,
                 const void *X, int64_t ldx, float beta_re, float beta_im, void *Y, int64_t ldy);
/* Backend.onemm, backend.py:528-533 (oracle np.py:95-97; _customgpu.cu:15-47):
 * Y(m x n) = beta*Y + alpha * ones(m,k) * X(k x n). */
int ib200_onemm(void *stream, int64_t m, int64_t ncols, int64_t k, float alpha_re, float alpha_im,
                const void *X, int64_t ldx, float beta_re, float beta_im, void *Y, int64_t ldy);
/* Backend.max, backend.py:734-736 (np.py:141-145; _customgpu.cu:7-13):
 * arr = max(arr, val) over nfloats floats (real and imaginary parts alike). */
int ib200_fmax(void *stream, int64_t nfloats, float val, void *arr);

/* ------------------------------------------------------------------ FFT
 * Backend.fftn / ifftn, backend.py:497-509 (oracle np.py:102-115; cuFFT
 * binding cuda.py:470-498): unscaled forward and UNSCALED inverse C2C over the
 * first `ndim` (1..3) axes of a column-major (d0[,d1[,d2]], batch) array with
 * contiguous batches.  Out of place or in place (y == x).  Any lengths: radices
 * 2,3,4,5,7,8,11,13,16 are specialised, other prime factors use a generic
 * butterfly.  No workspace (Backend._fft_workspace_size -> 0). */
typedef struct ib200_fft_plan_s *ib200_fft_plan;
int ib200_fft_plan_create(ib200_fft_plan *plan, int ndim, const int64_t *dims, int64_t batch);
int ib200_fft_plan_destroy(ib200_fft_plan plan);
/* Writes the radix sequence of axis `axis` into radices[0..max) and returns
 * the number of stages (host only, no device needed) or a negative error. */
int ib200_fft_plan_describe(ib200_fft_plan plan, int axis, int *radices, int max);
int ib200_fft_exec(ib200_fft_plan plan, void *stream, void *y, const void *x, int direction);
/* Fused variants (SURVEY.md section 8f rank 1, the north-star's "fused
 * elementwise"): d_in / d_out are optional length-prod(dims) complex64
 * diagonals applied on the first pass's load / the last pass's store,
 * broadcast over the batch; conj_* conjugates the diagonal. */
int ib200_fft_exec_diag(ib200_fft_plan plan, void *stream, void *y, const void *x, int direction,
                        const void *d_in, int conj_in, const void *d_out, int conj_out);

/* ------------------------------------------------------------------ fused SENSE transforms
 * Backend-specific fusion of the first two and last two calls of the -O3 SENSE apply
 * (SURVEY.md section 3.1):   ccsrmm(P^H, adjoint) -> fftn     and     ifftn -> ccsrmm(P^H),
 * P = kron(I_C, mod*zpad*apod) * vstack(maps) (examples/pics.py:111-126, indigo/backends/
 * backend.py:355-387).  The oversampled grid is kept coil-interleaved, grid[z][y][x][coil],
 * which is the layout ib200_ccsrmm_il gathers from; `pf` is the dense factor
 * pf[voxel*C + coil] = (mod*apod)[voxel] * maps[voxel, coil].  Zero-padding and cropping are
 * the input/output windows of the passes, so the zero rows of the padded volume are never
 * written, read or transformed before the pass that fills them.
 *   expand_fft   : grid = FFT3( zpad( pf .* img ) )                      (unscaled forward)
 *   ifft_combine : img  = alpha * sum_c conj(pf) .* crop( IFFT3(grid) ) + beta * img
 *                  (unscaled inverse; grid is overwritten; beta == 0 never reads img)
 * Grid extents must have a specialised FFT (32, 52, 64, 104, 128, 192, 208, 256, 320, 384, 416,
 * 448, 512, 640, 768, 832, 1024); otherwise plan creation returns IB200_E_UNSUPPORTED and the
 * caller stays on the six-call path. */
typedef struct ib200_sense_plan_s *ib200_sense_plan;
int ib200_sense_plan_create(ib200_sense_plan *plan, const int64_t N[3], const int64_t oN[3], int64_t ncoils);
int ib200_sense_plan_destroy(ib200_sense_plan plan);
/* win (device, 2 * oN[0]*oN[1] int32, see ib200_grid_support_windows; NULL disables) must stay valid
 * while the plan is used; block_x is the block extent along x the windows were built with (a tile of
 * 16 interleaved lines must not straddle two blocks: needs block_x*ncoils % 16 == 0 or ncoils % 16 == 0).
 * Returns IB200_E_UNSUPPORTED when the geometry does not allow per-tile windows. */
int ib200_sense_plan_set_support(ib200_sense_plan plan, const int32_t *win, int block_x);
int ib200_sense_expand_fft(ib200_sense_plan plan, void *stream, void *grid_il, const void *img, const void *pf);
int ib200_sense_ifft_combine(ib200_sense_plan plan, void *stream, void *img_out, void *grid_il, const void *pf,
                             float alpha_re, float alpha_im, float beta_re, float beta_im);
/* One pass of the two fused transforms on its own -- the same kernels with the same arguments as inside
 * ib200_sense_expand_fft / ib200_sense_ifft_combine -- so that a caller (bench.py) can bracket every
 * kernel of UnscaledFFT's replacement (operators.py:311-338) with CUDA events:
 *   which = 0 expand + x pass (img, pf -> grid), 1 forward y, 2 forward z,
 *           3 inverse z, 4 inverse y, 5 x pass + coil combine (grid, pf -> img_out, alpha/beta as above). */
int ib200_sense_pass(ib200_sense_plan plan, void *stream, int which, void *grid_il, const void *img,
                     void *img_out, const void *pf, float alpha_re, float alpha_im, float beta_re, float beta_im);

/* ------------------------------------------------------------------ Toeplitz normal operator
 * A^H A of a SENSE operator as a zero-padded convolution (indigo_b200.fused.toeplitz_normal):
 *   T x = s^2 * sum_c conj(S_c) .* crop( IFFT_L( K .* FFT_L( pad_L(S_c .* x) ) ) )
 * on a plan created with oN = L (the padded grid, ib200_sense_plan_create) and pf = maps (no apodisation,
 * no centring phase), without support windows.  One apply is five launches:
 *   ib200_sense_pass 0 -> [1] -> ib200_sense_toeplitz_pass -> [4] -> ib200_sense_pass 5 (alpha = s^2 * alpha)
 * (the bracketed y passes only when L[2] > 1).
 *   ib200_sense_toeplitz_pass: on the last transformed axis (z, or y when L[2] == 1) loads the image window of
 *     every line, transforms it forward, multiplies by kernel[pos * plane + point] (real float32, plane = L0*L1
 *     points, or L0 when L[2] == 1; kernel is laid out like one coil of the grid, z slowest), and runs the first
 *     inverse pass on it, storing the image window in the state ib200_sense_pass 3 leaves.  Lengths up to 512.
 *   ib200_toeplitz_psf: psf[j] = (p(d) + conj p(-d)) / 2 for the circular lag d = j (mod L) per axis, with
 *     p(d) = img[d + L/2] (column-major L0 x L1 x L2 complex64 images, x fastest; img != psf).
 *   ib200_toeplitz_kernel: kernel[i] = scale * Re spectrum[i] for n points (spectrum = ib200_fft_exec of psf,
 *     scale = 1 / prod(L)).
 * None synchronises. */
int ib200_sense_toeplitz_pass(ib200_sense_plan plan, void *stream, void *grid_il, const float *kernel);
int ib200_toeplitz_psf(void *stream, const int64_t L[3], const void *img, void *psf);
int ib200_toeplitz_kernel(void *stream, int64_t n, const void *spectrum, float scale, float *kernel);

/* ------------------------------------------------------------------ orthonormal wavelets, l1-wavelet FISTA
 * Separable periodized orthonormal wavelet transform W of a column-major dims[0] x dims[1] x dims[2] complex64
 * image (DESIGN.md section 11).  h (host, lf doubles, lf = 2 or 8) is the low-pass filter; the high-pass filter is
 * g[m] = (-1)^m h[lf-1-m].  Axes of one point are not transformed; every other axis must be divisible by
 * 2^levels and at most 512 points long (longer: IB200_E_UNSUPPORTED).  Level j transforms the sub-box of extent
 * dims[d] / 2^(j-1): an x pass, a y pass and a z pass, each in place on `work` (nvox complex64, device).
 *   ib200_wavelet: y = alpha * W x + beta * y (inverse == 0) or alpha * W^H x + beta * y (inverse != 0);
 *     beta == 0 never reads y.  work must not alias x or y.  A multi-level analysis ends with one elementwise
 *     pass from work to y (its last wavelet pass covers only the coarse sub-box); a multi-level synthesis starts
 *     with a device copy of x into work (its first pass covers only the coarse sub-box).
 *   ib200_wavelet_fista_step: one prox-and-update step of FISTA (indigo_b200.wavelet.l1wavelet_recon), given
 *     g = A^H A z:
 *         x_new = W^H soft_thresh(W (z - step (g - b)))   (the coarse band of the last level is not thresholded)
 *         z     = x_new + momentum[*counter] (x_new - x),   x = x_new,   *counter += 1
 *     with soft_thresh(c) = c max(0, 1 - thresh / |c|).  The first analysis pass reads z, g and b, the last pass
 *     of each analysis level thresholds on store and the last synthesis pass writes x and z.  stats (optional,
 *     IB200_WAVELET_STATS doubles of device memory) receives stats[0] = ||x_new - x||^2, stats[1] = ||x_new||^2,
 *     summed in a fixed order.  momentum and counter are device memory.
 * Both are deterministic (no atomics) and neither synchronises. */
#define IB200_WAVELET_STATS (2 + 2 * 4096)
int ib200_wavelet(void *stream, const int64_t dims[3], int lf, const double *h, int levels, int inverse,
                  float alpha_re, float alpha_im, float beta_re, float beta_im, const void *x, void *y, void *work);
int ib200_wavelet_fista_step(void *stream, const int64_t dims[3], int lf, const double *h, int levels, float step,
                             float thresh, const void *g, const void *b, void *z, void *x, void *work,
                             const double *momentum, int *counter, double *stats);

/* ------------------------------------------------------------------ ESPIRiT coil sensitivities (espirit.cu)
 * DESIGN.md section 12.  All three are deterministic (fixed summation order, no atomics) and none synchronises.
 * ib200_espirit_calib_gram: G = A^H A (n x n complex64, column-major, n = ncoils*k0*k1*k2) of the calibration
 *   matrix A of the (w0, w1, w2, ncoils) column-major calibration k-space: one row per kernel position s with the
 *   k0 x k1 x k2 patch inside the region, column (c, p) = p0 + k0 (p1 + k1 p2) + k0 k1 k2 c holding X_c(s + p).
 *   fp32 accumulation; the upper triangle is computed and mirrored, the diagonal is real.
 * ib200_espirit_lag_pass: out[o][x][i] = sum_{j < lags} in[o][j][i] * twiddle[x*lags + j], o < outer, x < n,
 *   i < inner (one axis of the separable evaluation of the lag form).
 * ib200_espirit_maps: per voxel (x, line), line = y + N1 z, M(x) = sum_j coef[line][j][c'][c] * twiddle0[x][j]
 *   (the C x C matrix, row c, column c', coef laid out [line][lags0][ncoils][ncoils], c fastest); max_iter power
 *   iterations from the all-ones vector, eig = the last norm, coil 0 rotated to real >= 0, zero where eig <= crop.
 *   maps is (N0 N1 N2, ncoils) column-major complex64, eig N0 N1 N2 floats.  1 <= ncoils <= 32; the lag matrices
 *   of one line must fit shared memory (lags0 * ncoils^2 * 8 bytes). */
int ib200_espirit_calib_gram(void *stream, const int64_t w[3], const int64_t k[3], int ncoils, const void *calib,
                             void *gram);
int ib200_espirit_lag_pass(void *stream, int64_t outer, int lags, int n, int64_t inner, const void *twiddle,
                           const void *in, void *out);
int ib200_espirit_maps(void *stream, const int64_t N[3], int lags0, int ncoils, int max_iter, float crop,
                       const void *twiddle0, const void *coef, void *maps, float *eig);

/* ------------------------------------------------------------------ operator construction on the device
 * Setup-time replacements for the host construction of the two sparse factors
 * of the -O3 SENSE tree (indigo/interp.py:19-80 + scipy COO->CSR + the -O2
 * products of indigo/transforms.py:86-96 / examples/pics.py:111-126).  All
 * buffers are device memory; results are ordinary CSR arrays for ib200_ccsrmm.
 *
 * Gridding matrix G' (m samples x prod(grid)):  count -> exclusive scan -> fill.
 *   coord     (3, m) doubles, coord[d + 3*i] in cycles/FOV
 *   table     Kaiser-Bessel half window (ntable doubles), backend.py:435-436
 *   rowweight optional m floats (sqrt density compensation) or NULL
 *   colscale  optional prod(grid) complex64 = diagonal of mod*scale, or NULL */
int ib200_kb_count(void *stream, int64_t m, const double *coord, const int64_t grid[3], double width,
                   int32_t *counts);
int ib200_exclusive_scan_i32(void *stream, int64_t n, const int32_t *in, int32_t *out /* n+1, synchronises */);
int ib200_kb_fill(void *stream, int64_t m, const double *coord, const int64_t grid[3], double width,
                  const double *table, int ntable, const float *rowweight, const void *colscale,
                  const int32_t *rowptr, int32_t *colind, void *vals);
/* Stored adjoint P^H (nvox x ncoils*ogrid) of P = kron(I, mod*zpad*apod) * vstack(maps):
 * row r holds conj(q[r]*maps[r,c]) at column c*ogrid + zp[r] for every coil c with a
 * non-zero product.  maps is (nvox, ncoils) column-major, q = mod[zp]*apod, zp the
 * zero-padded position of voxel r (backend.py:371-387). */
int ib200_sense_ph_count(void *stream, int64_t nvox, int ncoils, const void *maps, const void *q, int32_t *counts);
int ib200_sense_ph_fill(void *stream, int64_t nvox, int ncoils, int64_t ogrid, const void *maps, const void *q,
                        const int32_t *zp, const int32_t *rowptr, int32_t *colind, void *vals);

/* ------------------------------------------------------------------ dense
 * Backend.cgemm, backend.py:481-485 (oracle np.py:76-87; cuda.py:314-329):
 *   conjtrans == 0 : Y(m x n) = alpha * M(m x k)     * X(k x n) + beta*Y
 *   conjtrans != 0 : Y(m x n) = alpha * M(k x m)^H   * X(k x n) + beta*Y
 * Backend.csymm, backend.py:487-491 (np.py:89-90; cuda.py:355-366), M real
 * symmetric (stored full, complex64):
 *   left  != 0 : Y(m x n) = alpha * M(m x m) * X(m x n) + beta*Y
 *   left  == 0 : Y(m x n) = alpha * X(m x n) * M(n x n) + beta*Y */
int ib200_cgemm(void *stream, int conjtrans, int64_t m, int64_t n, int64_t k, float alpha_re, float alpha_im,
                const void *M, int64_t ldm, const void *X, int64_t ldx, float beta_re, float beta_im,
                void *Y, int64_t ldy);
int ib200_csymm(void *stream, int left, int64_t m, int64_t n, float alpha_re, float alpha_im,
                const void *M, int64_t ldm, const void *X, int64_t ldx, float beta_re, float beta_im,
                void *Y, int64_t ldy);
/* Products with at most 64 rows of op(M), an even k and 16-byte aligned X columns (coil compression:
 * M 12 x 48, millions of coil-fastest columns) run on the tensor cores as three TF32 MMAs per
 * product on (hi, lo) operand splits (mma.sync kernel); everything else on the SIMT fp32 kernel.
 * mode 1 forces the SIMT kernel, mode 3 selects the tcgen05/TMEM kernel where it applies (k % 4 == 0,
 * k <= 48, n >= 128, 16-byte aligned Y columns; tests compare all three), mode 0 restores the default. */
int ib200_cgemm_mode(int mode);

#ifdef __cplusplus
}
#endif
#endif /* INDIGO_B200_H */
