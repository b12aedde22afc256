"""ctypes binding of libwisecondor_b200.so (the C ABI declared in include/wisecondor_b200.h).

There is no CPU fallback: if the library is missing it is built with nvcc; if that is impossible, or no B200 is
present when a compute entry point is called, the call raises.
"""
import ctypes
import os

from . import build as _build

_LIB = None
ABI_VERSION = 3      # include/wisecondor_b200.h: WC_ABI_VERSION

SYMBOLS = [
    "wc_create", "wc_destroy", "wc_last_error", "wc_version", "wc_abi_version", "wc_debug_filter_scores", "wc_debug_pivot_select", "wc_sm_count", "wc_last_phase_ms",
    "wc_last_counter", "wc_device_count", "wc_dev_alloc", "wc_dev_free", "wc_copy_h2d", "wc_copy_d2h", "wc_dev_sync", "wc_newref_topk", "wc_newref_topk_wide", "wc_newref_topk_host",
    "wc_newref_shard_dims", "wc_newref_shard_begin", "wc_newref_shard_sweep", "wc_newref_shard_finish", "wc_debug_sym_plan", "wc_debug_profile", "wc_set_option",
    "wc_newref_mask", "wc_newref_normalize", "wc_pca_gram", "wc_pca_apply",
    "wc_table_stride", "wc_test_table", "wc_test_prep", "wc_apply_pca", "wc_zscore_batch", "wc_segment_batch",
]


class WcCall(ctypes.Structure):
    _fields_ = [("sample", ctypes.c_int32), ("chrom", ctypes.c_int32), ("x", ctypes.c_int32),
                ("y", ctypes.c_int32), ("z", ctypes.c_double)]


class WisecondorError(RuntimeError):
    pass


def lib():
    """Load (building first if needed) the shared library and declare the prototypes."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB
    if not os.path.exists(path):
        path = _build.build_library()
    L = ctypes.CDLL(path)
    vp, ci, cd = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    # a stale binary under new prototypes would misalign arguments silently: refuse it
    have = L.wc_abi_version() if hasattr(L, "wc_abi_version") else 0
    if have != ABI_VERSION:
        raise WisecondorError("%s was built for C-ABI version %d, this binding needs %d: rebuild it "
                              "(python -m wisecondor_b200.build --force)" % (path, have, ABI_VERSION))
    L.wc_debug_filter_scores.restype = ci
    L.wc_debug_filter_scores.argtypes = [vp, vp, ci]
    L.wc_debug_pivot_select.restype = ci
    L.wc_debug_pivot_select.argtypes = [vp, vp, ci, ci, vp]
    L.wc_create.restype = vp
    L.wc_create.argtypes = [ci]
    L.wc_destroy.restype = None
    L.wc_destroy.argtypes = [vp]
    L.wc_last_error.restype = ctypes.c_char_p
    L.wc_version.restype = ctypes.c_char_p
    L.wc_sm_count.restype = ci
    L.wc_sm_count.argtypes = [vp]
    L.wc_last_phase_ms.restype = cd
    L.wc_last_phase_ms.argtypes = [vp, ci]
    L.wc_last_counter.restype = ctypes.c_longlong
    L.wc_last_counter.argtypes = [vp, ci]
    L.wc_device_count.restype = ci
    L.wc_device_count.argtypes = []
    L.wc_dev_alloc.restype = vp
    L.wc_dev_alloc.argtypes = [vp, ctypes.c_size_t]
    L.wc_dev_free.restype = ci
    L.wc_dev_free.argtypes = [vp, vp]
    L.wc_copy_h2d.restype = ci
    L.wc_copy_h2d.argtypes = [vp, vp, vp, ctypes.c_size_t]
    L.wc_copy_d2h.restype = ci
    L.wc_copy_d2h.argtypes = [vp, vp, vp, ctypes.c_size_t]
    L.wc_dev_sync.restype = ci
    L.wc_dev_sync.argtypes = [vp]
    L.wc_newref_topk.restype = ci
    L.wc_newref_topk.argtypes = [vp, vp, ci, ci, vp, ci, ci, ci, ci, vp, vp, vp]
    L.wc_newref_topk_wide.restype = ci
    L.wc_newref_topk_wide.argtypes = [vp, vp, ci, ci, vp, ci, ci, ci, ci, vp, vp, vp]
    L.wc_newref_topk_host.restype = ci
    L.wc_newref_topk_host.argtypes = [vp, vp, ci, ci, vp, ci, ci, ci, ci, vp, vp]
    L.wc_newref_shard_dims.restype = ci
    L.wc_newref_shard_dims.argtypes = [vp, ci, ci, ci, ci, vp]
    L.wc_newref_shard_begin.restype = ci
    L.wc_newref_shard_begin.argtypes = [vp, vp, ci, ci, vp, ci, ci, ci, ci, vp, vp]
    L.wc_newref_shard_sweep.restype = ci
    L.wc_newref_shard_sweep.argtypes = [vp, vp, vp, vp, vp, vp]
    L.wc_newref_shard_finish.restype = ci
    L.wc_newref_shard_finish.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.wc_debug_sym_plan.restype = ci
    L.wc_debug_sym_plan.argtypes = [ci, vp, ci, ci, ci, ci, ci, ci, ci, vp, ctypes.c_longlong, vp]
    L.wc_set_option.restype = ci
    L.wc_set_option.argtypes = [vp, ctypes.c_char_p, cd]
    L.wc_debug_profile.restype = ci
    L.wc_debug_profile.argtypes = [vp, ci, vp, ci]
    i32 = ci
    L.wc_newref_mask.restype = ci
    L.wc_newref_mask.argtypes = [vp, vp, i32, i32, vp, vp]
    L.wc_newref_normalize.restype = ci
    L.wc_newref_normalize.argtypes = [vp, vp, i32, i32, vp, i32, vp, vp]
    L.wc_pca_gram.restype = ci
    L.wc_pca_gram.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    L.wc_pca_apply.restype = ci
    L.wc_pca_apply.argtypes = [vp, vp, i32, i32, vp, vp, vp, i32, vp, vp, vp]
    L.wc_table_stride.restype = ci
    L.wc_table_stride.argtypes = [ci]
    L.wc_test_table.restype = ci
    L.wc_test_table.argtypes = [vp, vp, vp, i32, i32, vp, i32, cd, vp, vp, vp, vp, vp]
    L.wc_test_prep.restype = ci
    L.wc_test_prep.argtypes = [vp, vp, i32, i32, vp, i32, vp, vp, i32, vp, i32, vp]
    L.wc_apply_pca.restype = ci
    L.wc_apply_pca.argtypes = [vp, vp, i32, i32, vp, vp, i32, vp, i32, vp]
    L.wc_zscore_batch.restype = ci
    L.wc_zscore_batch.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, i32, cd, i32, vp, vp, vp, vp, vp]
    L.wc_segment_batch.restype = ci
    L.wc_segment_batch.argtypes = [vp, vp, vp, vp, i32, i32, vp, i32, vp, i32, i32, cd, cd, i32, vp, vp, vp, vp, i32, vp]
    _LIB = L
    return L


def check(rc):
    if rc != 0:
        raise WisecondorError("wisecondor_b200 error %d: %s" % (rc, lib().wc_last_error().decode()))


class Context(object):
    """One wc_ctx per CUDA device; owns the grow-only device workspaces."""

    def __init__(self, device=0):
        self._h = lib().wc_create(int(device))
        if not self._h:
            raise WisecondorError("wc_create(%d) failed: %s" % (device, lib().wc_last_error().decode()))
        self.device = int(device)
        for key in ("k5_group", "k5_stages", "k5_lag", "k5_sym", "k5_f16", "k5_pivots", "k6_split", "k6_select", "k6_parts", "k6_g4", "k6_chunk", "k6_warps", "k6_prod"):        # experiment knobs; results never depend on them
            val = os.environ.get("WC_" + key.upper())
            if val is not None:
                check(lib().wc_set_option(self._h, key.encode(), float(val)))

    @property
    def handle(self):
        return self._h

    def sm_count(self):
        return lib().wc_sm_count(self._h)

    def phase_ms(self, which):
        return lib().wc_last_phase_ms(self._h, which)

    def counter(self, which):
        return lib().wc_last_counter(self._h, which)

    def close(self):
        if self._h:
            lib().wc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_CONTEXTS = {}


def context(device=0):
    ctx = _CONTEXTS.get(device)
    if ctx is None:
        ctx = _CONTEXTS[device] = Context(device)
    return ctx
