"""ctypes binding of ``csrc/libfocusr_b200.so`` (declared in ``include/focusr_b200.h``).

There is no CPU fallback: if the library is missing, or no CUDA device is visible when a compute
entry point is first needed, the product raises.  PyTorch is used for device memory (its caching
allocator owns all HBM the library touches), streams and ``torch.distributed`` only.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# FOCUSR_B200_LIB: an alternative build of the same library (kernel A/B builds of tools/knn_ab.sh); never a fallback
LIB_PATH = os.environ.get("FOCUSR_B200_LIB") or os.path.join(_HERE, "csrc", "libfocusr_b200.so")

_vp = C.c_void_p
_i = C.c_int
_d = C.c_double
_sz = C.c_size_t

# name -> (restype, argtypes); mirrors include/focusr_b200.h one to one
SIGNATURES = {
    "focusr_last_error": (C.c_char_p, []),
    "focusr_version": (_i, []),
    "focusr_launch_count": (C.c_ulonglong, []),
    "focusr_laplacian_workspace_bytes": (_sz, [_i, _i]),
    "focusr_laplacian_build": (_i, [_vp, _i, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "focusr_laplacian_csr": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "focusr_mean_filter_workspace_bytes": (_sz, [_i, _i]),
    "focusr_mean_filter": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _i, _i, _vp, _sz, _vp]),
    "focusr_mean_filter_mapped_workspace_bytes": (_sz, [_i, _i, _i]),
    "focusr_mean_filter_mapped": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _i, _vp, _sz, _vp]),
    "focusr_gather_rows": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    "focusr_eigs_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "focusr_sell_entries_cap": (C.c_longlong, [_vp, _vp, _i]),
    "focusr_eigs_workspace_bytes_mixed": (_sz, [_i, C.c_longlong, _i, _i, _i]),
    "focusr_eigs_default_options": (None, [_vp]),
    "focusr_eigs_block_size": (_i, [_i, _i, _i, _i, _i]),
    "focusr_eigs_smallest": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _i, _i, _i, _d, _d, _i, _i, _d,
                                  _vp, _vp, _i, _vp, _vp, _vp, _sz, _vp, _vp]),
    "focusr_dist_unique_id": (_i, [_vp]),
    "focusr_dist_init": (_i, [_vp, _i, _i]),
    "focusr_dist_finalize": (_i, []),
    "focusr_eigs_dist_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i]),
    "focusr_dist_shared_bytes": (_sz, [_i, _i, _i]),
    "focusr_dist_shared_alloc": (_i, [_sz, _vp]),
    "focusr_dist_shared_open": (_i, [_vp, _i, _i]),
    "focusr_dist_shared_free": (_i, []),
    "focusr_eigs_smallest_dist": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, C.c_longlong, C.c_longlong, _vp, _i, _vp,
                                       _vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _d, _d, _i, _i, _d,
                                       _vp, _vp, _i, _vp, _vp, _vp, _sz, _vp, _vp]),
    "focusr_profile_reset": (None, []),
    "focusr_profile_get": (None, [_vp]),
    "focusr_profile_get_kind": (None, [_i, _vp]),
    "focusr_laplacian_apply": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _i, _vp]),
    "focusr_normalize_columns": (_i, [_vp, _i, _i, _vp, _i, _vp, _vp]),
    "focusr_flip_permute_columns": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "focusr_spectral_coords": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _i, _vp, _vp]),
    "focusr_eigsort_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "focusr_eigsort_costs": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp,
                                  _vp, _sz, _vp]),
    "focusr_eigsort_ragged_workspace_bytes": (_sz, [_vp, _vp, _i, _i]),
    "focusr_eigsort_costs_ragged": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp,
                                         _vp, _vp, _vp, _sz, _vp]),
    "focusr_eigsort_decide_workspace_bytes": (_sz, [_i, _i]),
    "focusr_eigsort_decide": (_i, [_vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp,
                                   _vp, _sz, _vp]),
    "focusr_knn_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "focusr_knn": (_i, [_vp, _i, _vp, _i, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "focusr_knn_mapped_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "focusr_knn_mapped": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _i, _vp, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _sz,
                               _vp]),
    "focusr_cdist": (_i, [_vp, _i, _vp, _i, _i, _vp, _vp]),
    "focusr_lsap_workspace_bytes": (_sz, [_i]),
    "focusr_lsap": (_i, [_vp, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "focusr_weighted_positions": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "focusr_curvature_workspace_bytes": (_sz, [_i, _i]),
    "focusr_curvatures": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "focusr_node_features_workspace_bytes": (_sz, [_i, _i, _i]),
    "focusr_node_features": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i, _d, _i, _vp, _vp, _vp, _sz, _vp]),
    "focusr_feature_coords": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _vp, _vp]),
    "focusr_icp_workspace_bytes": (_sz, [_i, _i]),
    "focusr_icp": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "focusr_icp_batch_workspace_bytes": (_sz, [_vp, _vp, _i, _vp, _vp, _i, _i]),
    "focusr_icp_batch": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp,
                              _sz, _vp]),
    "focusr_cpd_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "focusr_cpd_affine": (_i, [_vp, _i, _vp, _i, _i, _i, _d, _d, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "focusr_cpd_deformable": (_i, [_vp, _i, _vp, _i, _i, _i, _d, _d, _d, _d, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "focusr_cpd_kernel_matrix": (_i, [_vp, _i, _i, _d, _vp, _vp]),
    "focusr_cpd_affine_apply": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp]),
    "focusr_cpd_deformable_apply": (_i, [_vp, _i, _vp, _i, _i, _vp, _d, _vp, _vp]),
    "focusr_procrustes_fit": (_i, [_vp, _i, _i, _vp, _i, _vp, _vp, _vp]),
    "focusr_procrustes_mean_workspace_bytes": (_sz, [_i]),
    "focusr_procrustes_mean": (_i, [_vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "focusr_shape_gram_workspace_bytes": (_sz, [_i, _i]),
    "focusr_shape_gram": (_i, [_vp, _vp, _i, _i, _vp, _vp, _sz, _vp]),
    "focusr_shape_modes": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _vp]),
    "focusr_closest_points_workspace_bytes": (_sz, [_vp, _vp, _i, _vp, _i, _vp]),
    "focusr_closest_points": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "focusr_surface_distance_stats": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _vp]),
}

MESH_INFO_INTS = 8  # FOCUSR_MESH_INFO_INTS: {nnz, one-way entries, zero-degree rows, non-finite weights, longest row, ...}


class EigsOptions(C.Structure):
    """``focusr_eigs_options`` (include/focusr_b200.h): per-call options of the eigensolver; no process-wide state."""

    _fields_ = [("mixed_precision", _i), ("filter_policy", _i), ("filter_prefetch", _i), ("filter_min_blocks", _i),
                ("filter_pdl", _i), ("nonsym_device", _i), ("reserved", _i * 10)]

    def __init__(self, **kw):
        super().__init__()
        load().focusr_eigs_default_options(C.byref(self))
        for k, v in kw.items():
            if k not in dict(self._fields_):
                raise TypeError("unknown eigensolver option %r" % k)
            setattr(self, k, int(v))


_lib = None


class FocusrB200Error(RuntimeError):
    """Raised when a libfocusr_b200 entry point returns a non-zero status."""

    def __init__(self, fn, code, message):
        super().__init__("%s failed (status %d): %s" % (fn, code, message))
        self.fn = fn
        self.code = code
        self.message = message


def load():
    """Load the shared library (once).  Raises ImportError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libfocusr_b200.so is not built (%s). Run pyfocusr_b200/csrc/build.sh or "
            "`python -c 'import __graft_entry__ as g; g.build()'`; there is no CPU fallback." % LIB_PATH
        )
    import torch  # noqa: F401  (loads libcudart into the process before the library needs it)

    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def call(name, *args):
    """Call an int-returning entry point and raise on a non-zero status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise FocusrB200Error(name, rc, lib.focusr_last_error().decode("utf-8", "replace"))
    return rc


def launch_count():
    return int(load().focusr_launch_count())


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError(
            "pyfocusr_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback for the "
            "spectral-correspondence path."
        )
    return torch


def ptr(t):
    """Device (or host, for numpy arrays) address of a tensor/array, or NULL for None."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


def stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream
