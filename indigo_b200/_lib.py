"""
ctypes binding of libindigo_b200.so (C ABI declared in include/indigo_b200.h).

This is the thin layer the north star asks for: every Backend method ends in
exactly one of these calls.  There is no fallback: if the shared library is
missing or a call fails, a RuntimeError is raised (same convention as the
reference's ctypes backends, indigo/backends/cuda.py:42-49).
"""
import ctypes
import os
from ctypes import c_int, c_int64, c_float, c_double, c_void_p, c_char_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IB200_LIB") or os.path.join(_HERE, "libindigo_b200.so")   # IB200_LIB: build variants (tools/)

_vp, _i, _i64, _f = c_void_p, c_int, c_int64, c_float

# name -> (restype, argtypes); mirrors include/indigo_b200.h one to one
SIGNATURES = {
    "ib200_last_error": (c_char_p, []),
    "ib200_version": (_i, []),
    "ib200_device_info": (_i, [_i, POINTER(_i), POINTER(_i64), POINTER(_i64), POINTER(_i64)]),
    "ib200_launch_count": (_i64, []),
    "ib200_launch_count_reset": (None, []),
    "ib200_copy2d": (_i, [_vp, _vp, _i64, _vp, _i64, _i64, _i64, _i]),
    "ib200_memset0": (_i, [_vp, _vp, _i64]),
    "ib200_stream_sync": (_i, [_vp]),
    "ib200_caxpby": (_i, [_vp, _i64, _f, _f, _vp, _f, _f, _vp]),
    "ib200_cscal": (_i, [_vp, _i64, _f, _f, _vp]),
    "ib200_cdotc_dev": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "ib200_scnrm2sq_dev": (_i, [_vp, _i64, _vp, _vp]),
    "ib200_cdotc": (_i, [_vp, _i64, _vp, _vp, POINTER(c_double), POINTER(c_double)]),
    "ib200_scnrm2sq": (_i, [_vp, _i64, _vp, POINTER(c_double)]),
    "ib200_cg_xr": (_i, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "ib200_cg_p": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "ib200_ccsrmm": (_i, [_vp, _i, _i, _i64, _i64, _i64, _i64, _f, _f, _vp, _vp, _vp, _vp, _i64, _f, _f, _vp, _i64]),
    "ib200_interleave": (_i, [_vp, _i64, _i64, _vp, _i64, _vp, _i64]),
    "ib200_deinterleave": (_i, [_vp, _i64, _i64, _vp, _i64, _f, _f, _vp, _i64]),
    "ib200_interleave_rows": (_i, [_vp, _i64, _i64, _vp, _i64, _vp, _i64, _vp]),
    "ib200_deinterleave_rows": (_i, [_vp, _i64, _i64, _vp, _i64, _f, _f, _vp, _i64, _vp]),
    "ib200_invert_perm": (_i, [_vp, _i64, _vp, _vp]),
    "ib200_ccsrmm_il": (_i, [_vp, _i64, _i64, _i64, _i64, _f, _f, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i,
                             _vp, _i, _i]),
    "ib200_csr_permute_rows": (_i, [_vp, _i64, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "ib200_csr_long_rows": (_i, [_vp, _i64, _vp, _i, _vp, _i, POINTER(_i)]),
    "ib200_csr_pack_real": (_i, [_vp, _i64, _vp, _vp, _vp, POINTER(c_float)]),
    "ib200_ccsrmm_ilr": (_i, [_vp, _i64, _i64, _i64, _i64, _f, _f, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i,
                              _vp, _i, _i]),
    "ib200_kb_record_bytes": (_i, []),
    "ib200_kb_records": (_i, [_vp, _i64, _vp, POINTER(_i64), c_double, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp,
                              POINTER(_i)]),
    "ib200_kb_gather": (_i, [_vp, _i64, _i64, _f, _f, _vp, _vp, _i64, POINTER(_i64), _vp, _i64]),
    "ib200_kb_sample_order": (_i, [_vp, _i64, _vp, POINTER(_i64), c_double, POINTER(_i64), POINTER(_i64), _vp]),
    "ib200_kb_support_windows": (_i, [_vp, _i64, _vp, POINTER(_i64), _i64, _vp, POINTER(_i64), _vp, _vp, POINTER(_i64)]),
    "ib200_grid_support_windows": (_i, [_vp, POINTER(_i64), _i64, _vp, _vp, POINTER(_i64), _vp, _vp, POINTER(_i64)]),
    "ib200_sense_plan_set_support": (_i, [_vp, _vp, _i]),
    "ib200_csr_runs_count": (_i, [_vp, _i64, _vp, _vp, _i, _vp, POINTER(_i64), POINTER(_i), POINTER(_i)]),
    "ib200_csr_runs_fill": (_i, [_vp, _i64, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ib200_ccsrmm_runs": (_i, [_vp, _i64, _i64, _f, _f, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i, _vp, _i, _vp, _i, _vp]),
    "ib200_kb_blocks_batch_bytes": (_i, [_i, _i]),
    "ib200_kb_blocks_count": (_i, [_vp, _i64, _vp, POINTER(_i64), _i, _i, _vp, _i, _vp, _vp, POINTER(_i64)]),
    "ib200_kb_blocks_fill": (_i, [_vp, _i64, _vp, POINTER(_i64), _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "ib200_kb_blocks_apply": (_i, [_vp, _i64, _i, _i, _f, _f, _i, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i, _vp, _vp, _i]),
    "ib200_grid_tile_rank2": (_i, [_vp, POINTER(_i64), POINTER(_i64), POINTER(_i64), _vp, POINTER(_i64)]),
    "ib200_grid_tile_rank": (_i, [_vp, POINTER(_i64), POINTER(_i64), _vp, _vp, POINTER(_i64)]),
    "ib200_csr_inspect": (_i, [_vp, _i64, _i64, _vp, _vp, _vp, POINTER(_i64)]),
    "ib200_csr_transpose_conj": (_i, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ib200_kb_count": (_i, [_vp, _i64, _vp, POINTER(_i64), c_double, _vp]),
    "ib200_exclusive_scan_i32": (_i, [_vp, _i64, _vp, _vp]),
    "ib200_kb_fill": (_i, [_vp, _i64, _vp, POINTER(_i64), c_double, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "ib200_sense_ph_count": (_i, [_vp, _i64, _i, _vp, _vp, _vp]),
    "ib200_sense_ph_fill": (_i, [_vp, _i64, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ib200_cdiamm": (_i, [_vp, _i, _i64, _i64, _i64, _i64, _vp, _vp, _i64, _i64, _f, _f, _vp, _i64, _f, _f, _vp, _i64]),
    "ib200_onemm": (_i, [_vp, _i64, _i64, _i64, _f, _f, _vp, _i64, _f, _f, _vp, _i64]),
    "ib200_fmax": (_i, [_vp, _i64, _f, _vp]),
    "ib200_fft_plan_create": (_i, [POINTER(_vp), _i, POINTER(_i64), _i64]),
    "ib200_fft_plan_destroy": (_i, [_vp]),
    "ib200_fft_plan_describe": (_i, [_vp, _i, POINTER(_i), _i]),
    "ib200_fft_exec": (_i, [_vp, _vp, _vp, _vp, _i]),
    "ib200_fft_exec_diag": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _i]),
    "ib200_sense_plan_create": (_i, [POINTER(_vp), POINTER(_i64), POINTER(_i64), _i64]),
    "ib200_sense_plan_destroy": (_i, [_vp]),
    "ib200_sense_expand_fft": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "ib200_sense_ifft_combine": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _f, _f, _f]),
    "ib200_sense_pass": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _f, _f, _f, _f]),
    "ib200_sense_toeplitz_pass": (_i, [_vp, _vp, _vp, _vp]),
    "ib200_toeplitz_psf": (_i, [_vp, POINTER(_i64), _vp, _vp]),
    "ib200_toeplitz_kernel": (_i, [_vp, _i64, _vp, _f, _vp]),
    "ib200_cgemm": (_i, [_vp, _i, _i64, _i64, _i64, _f, _f, _vp, _i64, _vp, _i64, _f, _f, _vp, _i64]),
    "ib200_csymm": (_i, [_vp, _i, _i64, _i64, _f, _f, _vp, _i64, _vp, _i64, _f, _f, _vp, _i64]),
    "ib200_cgemm_mode": (_i, [_i]),
}

# entry points that return something other than a status code
_NO_STATUS = {"ib200_last_error", "ib200_version", "ib200_launch_count", "ib200_launch_count_reset",
              "ib200_fft_plan_describe", "ib200_kb_record_bytes", "ib200_kb_blocks_batch_bytes"}


class Library(object):
    """Loaded libindigo_b200.so.  `lib.ccsrmm(...)` calls `ib200_ccsrmm` and
    raises RuntimeError on a non-zero status."""

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise RuntimeError(
                "libindigo_b200.so not found at %s: build it with `make -C indigo_b200/csrc` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback." % path)
        self.path = path
        self._dll = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(self._dll, name)          # AttributeError here = header/library mismatch
            fn.restype, fn.argtypes = res, args
            setattr(self, name[len("ib200_"):], self._wrap(name, fn))

    def _wrap(self, name, fn):
        if name in _NO_STATUS:
            return fn
        dll = self._dll

        def call(*args):
            rc = fn(*args)
            if rc != 0:
                msg = dll.ib200_last_error()
                raise RuntimeError("%s failed with status %d: %s" % (name, rc, msg.decode("ascii", "replace") if msg else ""))
        call.__name__ = name
        return call


_lib = None


def load():
    """Process-wide library handle (loaded on first use)."""
    global _lib
    if _lib is None:
        _lib = Library()
    return _lib
