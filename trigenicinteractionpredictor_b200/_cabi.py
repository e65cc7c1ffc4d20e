"""ctypes binding of libtip.so (include/tip.h).  No CPU fallback: if the library cannot be loaded
every call raises `TipLibraryError`."""
from __future__ import annotations

import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtip.so")
HEADER = os.path.join(os.path.dirname(HERE), "include", "tip.h")

c_void_p, c_int, c_int64, c_size_t, c_uint, c_double = (
    ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_uint, ctypes.c_double)
_pi64 = ctypes.POINTER(ctypes.c_int64)
_psz = ctypes.POINTER(ctypes.c_size_t)
_pdbl = ctypes.POINTER(ctypes.c_double)

TIP_EM_DEFAULT = 0
TIP_EM_FORCE_GENERIC = 1
TIP_EM_FP32_COMPUTE = 2
TIP_EM_WITH_LOGLIK = 4
TIP_EM_GENE_SEGMENTED = 8
TIP_ROWS_COMPACT8 = 16
TIP_EM_SLOT_SEGMENTED = 32
TIP_EM_GATHER_L1 = 64

# name -> (restype, argtypes); must list every function include/tip.h declares (tests check this)
SIGNATURES = {
    "tip_abi_version": (c_int, []),
    "tip_last_error": (ctypes.c_char_p, []),
    "tip_stats_len": (c_int64, [c_int, c_int]),
    "tip_rows_capacity": (c_int64, [c_int64]),
    "tip_pack_rows_workspace_bytes": (c_int, [c_int64, _psz]),
    "tip_pack_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_size_t,
                              c_void_p, _pi64, _pi64, c_void_p, c_void_p]),
    "tip_order_rows_workspace_bytes": (c_int, [c_int64, _psz]),
    "tip_order_rows_out_bytes": (c_int64, [c_int64]),
    "tip_order_rows_by_gene": (c_int, [c_void_p, c_int64, c_int64, c_int, c_void_p, c_size_t, c_void_p, c_void_p]),
    "tip_order_rows": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_size_t, c_void_p, c_void_p]),
    "tip_em_workspace_bytes": (c_int, [c_int, c_int, c_int64, c_uint, _psz]),
    "tip_em_step": (c_int, [c_int, c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                            c_uint, c_void_p]),
    "tip_em_step_host_rows": (c_int, [c_int, c_int, c_void_p, c_int64, c_int64, c_uint, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "tip_normalise": (c_int, [c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tip_loglik_workspace_bytes": (c_size_t, [c_int, c_int]),
    "tip_loglik": (c_int, [c_int, c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_uint,
                           c_void_p]),
    "tip_score": (c_int, [c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tip_metrics_workspace_bytes": (c_int, [c_int64, _psz]),
    "tip_metrics": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_size_t, c_void_p, c_void_p]),
    "tip_sort_scores_workspace_bytes": (c_int, [c_int64, _psz]),
    "tip_sort_scores": (c_int, [c_void_p, c_int64, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "tip_top_triplets_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int64, c_int64, _psz]),
    "tip_top_triplets": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int64, c_void_p,
                                 c_size_t, c_void_p, c_void_p, _pi64, c_void_p]),
    "tip_top_triplets_last_passes": (c_int, []),
    "tip_top_triplets_per_gene_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, c_int64, c_int64, _psz]),
    "tip_top_triplets_per_gene": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                          c_int64, c_int64, c_void_p, c_size_t, c_void_p, c_void_p, _pi64, c_void_p]),
    "tip_top_triplets_per_gene_last_passes": (c_int, []),
    "tip_top_triplets_per_pair_workspace_bytes": (c_int, [c_int, c_int64, c_int, c_int, c_int64, c_int64, _psz]),
    "tip_top_triplets_per_pair": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p,
                                          c_int64, c_int64, c_void_p, c_size_t, c_void_p, c_void_p, _pi64, c_void_p]),
    "tip_top_triplets_per_pair_last_passes": (c_int, []),
    "tip_score_histogram_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, c_int, _psz]),
    "tip_score_histogram": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                    ctypes.POINTER(c_int), c_void_p, c_void_p, c_size_t, c_void_p]),
    "tip_rank_per_pair_workspace_bytes": (c_int, [c_int, c_int64, c_int, c_int, c_int64, c_int64, _psz]),
    "tip_rank_per_pair": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p, c_int64,
                                  c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tip_rank_per_gene_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, c_int64, c_int64, _psz]),
    "tip_rank_per_gene": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int64,
                                  c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p,
                                  c_void_p]),
    "tip_score_pairs": (c_int, [c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "tip_top_pairs_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int64, _psz]),
    "tip_top_pairs": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int64, c_void_p,
                              c_size_t, c_void_p, c_void_p, _pi64, c_void_p]),
    "tip_top_pairs_last_chunks": (c_int, []),
    "tip_top_pairs_per_gene_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, c_int64, _psz]),
    "tip_top_pairs_per_gene": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                       c_int64, c_int64, c_void_p, c_size_t, c_void_p, c_void_p, _pi64, c_void_p]),
    "tip_top_pairs_per_gene_last_chunks": (c_int, []),
    "tip_reduce_samples":(c_int, [c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tip_em_iterations_host": (c_int, [c_int, c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int,
                                       c_uint]),
    "tip_rows_compact_host": (c_int, [c_void_p, c_int64, c_void_p]),
    "tip_rows_expand": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "tip_ipc_export": (c_int, [c_void_p, c_void_p, _pi64]),
    "tip_ipc_import": (c_int, [c_void_p, c_int64, ctypes.POINTER(c_void_p)]),
    "tip_peer_barrier": (c_int, [ctypes.POINTER(c_void_p), c_void_p, c_int, c_int, c_void_p]),
    "tip_normalise_peers": (c_int, [c_int, c_int, ctypes.POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tip_peer_mstep": (c_int, [c_int, c_int, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                               ctypes.POINTER(c_void_p), c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "tip_peer_push_mstep": (c_int, [c_int, c_int, c_void_p, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p), c_void_p, c_int,
                                    c_int, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tip_em_set_push_targets": (c_int, [ctypes.POINTER(c_void_p), c_int, c_int, c_int64]),
    "tip_pairs_step": (c_int, [c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tip_pairs_normalise": (c_int, [c_int, c_void_p, c_void_p, c_void_p]),
    "tip_pairs_loglik": (c_int, [c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tip_measure_fma_peak": (c_int, [c_int, _pdbl]),
    "tip_measure_red_f64": (c_int, [c_int64, c_int, _pdbl]),
    "tip_measure_l2_gather": (c_int, [c_int, c_int, _pdbl]),
    "tip_seg3_timing": (c_int, [c_int]),
    "tip_seg3_last_timing": (c_int, [ctypes.POINTER(ctypes.c_float)]),
}


class TipLibraryError(RuntimeError):
    pass


_lib = None


def header_functions() -> list[str]:
    """Names of all functions declared in include/tip.h."""
    text = open(HEADER, encoding="utf-8").read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(tip_[a-z0-9_]+)\s*\(", text)))


def load(build_if_missing: bool = True):
    """Load (building first if the .so is absent and nvcc exists).  Raises TipLibraryError otherwise."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) and build_if_missing:
        try:
            from . import build as _build
            _build.build()
        except Exception as exc:  # noqa: BLE001
            raise TipLibraryError(
                "libtip.so is missing and could not be built (%s); this package has no CPU path" % exc) from exc
    if not os.path.exists(LIB_PATH):
        raise TipLibraryError("libtip.so not found at %s; run `python -m trigenicinteractionpredictor_b200.build`"
                              % LIB_PATH)
    # a library older than the sources it sits next to must not run silently (ADVICE r1): the build writes the digest of
    # csrc/*.cu, *.cuh and include/tip.h beside the objects; on a mismatch rebuild (nvcc is in the image), else refuse
    try:
        from . import build as _build
        stamp = os.path.join(_build.OBJ_DIR, "stamp.sha256")
        if build_if_missing and os.path.exists(stamp) and open(stamp).read().strip() != _build._digest():
            try:
                _build.build()
            except Exception as exc:  # noqa: BLE001
                raise TipLibraryError("libtip.so is older than its sources and could not be rebuilt (%s)" % exc) from exc
    except ImportError:
        pass
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as exc:
        raise TipLibraryError("cannot load %s: %s" % (LIB_PATH, exc)) from exc
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise TipLibraryError("libtip.so does not export %s" % name) from exc
        fn.restype = res
        fn.argtypes = args
    if lib.tip_abi_version() != 1:
        raise TipLibraryError("libtip.so ABI version %d, expected 1" % lib.tip_abi_version())
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().tip_last_error()
        raise TipLibraryError("%s failed (%d): %s" % (what, rc, (msg or b"").decode("utf-8", "replace")))
