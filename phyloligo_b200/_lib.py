"""ctypes binding of libphyloligo_b200.so (the C ABI declared in include/phyloligo_b200.h).

There is no fallback: if the shared library cannot be loaded the import of any
compute entry point raises PhyloligoError, and on a machine without a CUDA
device the calls themselves fail with the library's own error message.
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "lib", "libphyloligo_b200.so")

PO_OK = 0
STRANDS = {"plus": 0, "minus": 1, "both": 2}
METRICS = {"Eucl": 0, "JSD": 1, "KT": 2, "BC": 3, "SC": 4,
           # Eucl in the Gram form on the tensor cores (what the reference's --large workers compute
           # through sklearn euclidean_distances, bin/phyloligo.py:200-202, 238-246)
           "EuclGram": 5}
PO_F32, PO_F64 = 0, 1
FLAG_SKIP_LOWER, FLAG_MIRROR, FLAG_MIRROR_ONLY = 1, 2, 4
TILE = 128  # largest kernel tile edge: row panels and rank boundaries are multiples of it

# every symbol include/phyloligo_b200.h declares (tests check the library exports them all)
EXPORTED = [
    "po_version", "po_last_error", "po_device_info", "po_pattern_info", "po_fasta_index_host",
    "po_profile_batch", "po_prepared_row_bytes", "po_prepared_bytes", "po_prepare_profiles", "po_rank_transform", "po_distance_block", "po_distance_block_ex",
    "po_ipc_export", "po_ipc_open", "po_ipc_close", "po_savetxt_host", "po_copy2d_async", "po_window_count_byte", "po_window_distances",
    "po_host_prefault", "po_host_premap", "po_host_register", "po_host_unregister", "po_host_copy2d", "po_host_pwrite2d",
    "po_host_pread", "po_host_transpose_f32",
    "po_host_mirror_open", "po_host_mirror_submit", "po_host_mirror_wait", "po_host_mirror_close",
    "po_matrix_rowsums", "po_matrix_argmin_rows", "po_cluster_argmin", "po_matrix_knn",
    "po_hdbscan_check", "po_matrix_kth", "po_hdbscan_mst_workspace", "po_hdbscan_mst_init", "po_hdbscan_mst_scan", "po_hdbscan_mst_merge", "po_hdbscan_tree",
    "po_tsne_check", "po_tsne_conditional", "po_tsne_sum", "po_tsne_workspace", "po_tsne_repulsion", "po_tsne_attraction_step",
    "po_linkage_workspace", "po_linkage_run", "po_linkage_tree",
    "po_nj_capacity", "po_nj_workspace", "po_nj_stage_bytes", "po_nj_run",
    "po_launch_count", "po_timing_enable", "po_timing_reset", "po_timing_read", "po_microbench",
]


class PhyloligoError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library once and set the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise PhyloligoError(
            "libphyloligo_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `python phyloligo_b200/build.py`; there is no CPU fallback." % LIB_PATH)
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as exc:  # pragma: no cover
        raise PhyloligoError("cannot load %s: %s" % (LIB_PATH, exc)) from exc
    vp, i64, i32, u32 = C.c_void_p, C.c_int64, C.c_int, C.c_uint
    lib.po_version.restype = C.c_char_p
    lib.po_last_error.restype = C.c_char_p
    lib.po_device_info.argtypes = [C.POINTER(i32)] * 3
    lib.po_device_info.restype = i32
    lib.po_pattern_info.argtypes = [C.c_char_p, C.POINTER(i32), C.POINTER(i32), C.POINTER(i64)]
    lib.po_pattern_info.restype = i32
    lib.po_fasta_index_host.argtypes = [vp, i64, vp, vp, i64, i32]
    lib.po_fasta_index_host.restype = i64
    lib.po_profile_batch.argtypes = [vp, vp, vp, i64, C.c_char_p, i32, vp, vp, vp, vp, vp]
    lib.po_profile_batch.restype = i32
    lib.po_prepared_row_bytes.argtypes = [i32, i64]
    lib.po_prepared_row_bytes.restype = i64
    lib.po_prepared_bytes.argtypes = [i32, i64, i64]
    lib.po_prepared_bytes.restype = i64
    lib.po_prepare_profiles.argtypes = [i32, vp, i32, i64, i64, i64, vp, vp, vp]
    lib.po_prepare_profiles.restype = i32
    lib.po_distance_block.argtypes = [i32, vp, vp, i64, i64, i64, i64, i64, i64, vp, i64, i64, i64, i32, u32, vp]
    lib.po_distance_block.restype = i32
    lib.po_distance_block_ex.argtypes = [i32, vp, vp, i64, i64, i64, i64, i64, i64, vp, i64, i64, i64,
                                         vp, i64, i64, i64, i32, u32, vp]
    lib.po_distance_block_ex.restype = i32
    lib.po_ipc_export.argtypes = [vp, vp, C.POINTER(i64)]
    lib.po_ipc_export.restype = i32
    lib.po_ipc_open.argtypes = [vp, C.POINTER(vp)]
    lib.po_ipc_open.restype = i32
    lib.po_ipc_close.argtypes = [vp]
    lib.po_ipc_close.restype = i32
    lib.po_window_count_byte.argtypes = [vp, vp, vp, i64, i32, vp, vp]
    lib.po_window_count_byte.restype = i32
    lib.po_window_distances.argtypes = [i32, vp, i64, i64, i64, vp, vp, vp]
    lib.po_window_distances.restype = i32
    lib.po_rank_transform.argtypes = [vp, i32, i64, i64, i64, vp, i64, vp]
    lib.po_rank_transform.restype = i32
    lib.po_copy2d_async.argtypes = [vp, i64, vp, i64, i64, i64, vp]
    lib.po_copy2d_async.restype = i32
    lib.po_savetxt_host.argtypes = [C.c_char_p, vp, i64, i64, i64, i32, i32]
    lib.po_savetxt_host.restype = i32
    lib.po_host_prefault.argtypes = [vp, i64, i32]
    lib.po_host_prefault.restype = i32
    lib.po_host_premap.argtypes = [i32, vp, i64, i32]
    lib.po_host_premap.restype = i32
    lib.po_host_register.argtypes = [vp, i64]
    lib.po_host_register.restype = i32
    lib.po_host_unregister.argtypes = [vp]
    lib.po_host_unregister.restype = i32
    lib.po_host_copy2d.argtypes = [vp, i64, vp, i64, i64, i64, i32]
    lib.po_host_copy2d.restype = i32
    lib.po_host_pwrite2d.argtypes = [i32, i64, i64, vp, i64, i64, i64, i32]
    lib.po_host_pwrite2d.restype = i32
    lib.po_host_pread.argtypes = [i32, i64, vp, i64, i32]
    lib.po_host_pread.restype = i32
    lib.po_host_transpose_f32.argtypes = [vp, i64, vp, i64, i64, i64, i32]
    lib.po_host_transpose_f32.restype = i32
    lib.po_host_mirror_open.argtypes = [i32]
    lib.po_host_mirror_open.restype = vp
    lib.po_host_mirror_submit.argtypes = [vp, vp, i32, vp, i64, vp, i64, i64, i64]
    lib.po_host_mirror_submit.restype = i32
    lib.po_host_mirror_wait.argtypes = [vp]
    lib.po_host_mirror_wait.restype = i32
    lib.po_host_mirror_close.argtypes = [vp]
    lib.po_host_mirror_close.restype = i32
    lib.po_matrix_rowsums.argtypes = [vp, i64, i32, vp, i64, i64, vp, vp, vp, vp]
    lib.po_matrix_rowsums.restype = i32
    lib.po_matrix_argmin_rows.argtypes = [vp, i64, i32, vp, i32, i64, vp, vp]
    lib.po_matrix_argmin_rows.restype = i32
    lib.po_cluster_argmin.argtypes = [vp, vp, i64, i32, vp, vp, vp, vp, vp]
    lib.po_cluster_argmin.restype = i32
    lib.po_matrix_knn.argtypes = [vp, i64, i32, i64, i64, i64, i32, vp, vp, vp]
    lib.po_matrix_knn.restype = i32
    lib.po_hdbscan_check.argtypes = [vp, i64, i32, i64, i64, i64, vp, i64, vp, vp]
    lib.po_hdbscan_check.restype = i32
    lib.po_matrix_kth.argtypes = [vp, i64, i32, i64, i64, i32, vp, vp]
    lib.po_matrix_kth.restype = i32
    lib.po_hdbscan_mst_workspace.argtypes = [i64]
    lib.po_hdbscan_mst_workspace.restype = i64
    lib.po_hdbscan_mst_init.argtypes = [i64, vp, vp]
    lib.po_hdbscan_mst_init.restype = i32
    lib.po_hdbscan_mst_scan.argtypes = [vp, i64, i32, i64, i64, i64, vp, vp, vp]
    lib.po_hdbscan_mst_scan.restype = i32
    lib.po_hdbscan_mst_merge.argtypes = [i64, i32, vp, vp, vp, vp, vp, C.POINTER(i64), vp]
    lib.po_hdbscan_mst_merge.restype = i32
    lib.po_hdbscan_tree.argtypes = [i64, i64] + [vp] * 14
    lib.po_hdbscan_tree.restype = i32
    lib.po_tsne_check.argtypes = [vp, i64, i32, i64, i64, i64, vp, vp]
    lib.po_tsne_check.restype = i32
    lib.po_tsne_conditional.argtypes = [vp, i64, i32, i64, vp, i32, C.c_double, vp, vp]
    lib.po_tsne_conditional.restype = i32
    lib.po_tsne_sum.argtypes = [vp, i64, vp, vp]
    lib.po_tsne_sum.restype = i32
    lib.po_tsne_workspace.argtypes = [i64]
    lib.po_tsne_workspace.restype = i64
    lib.po_tsne_repulsion.argtypes = [vp, i64, vp, vp]
    lib.po_tsne_repulsion.restype = i32
    lib.po_tsne_attraction_step.argtypes = [vp, vp, vp, i64, C.c_double, C.c_double, vp, vp, vp, vp, vp, vp, C.c_double,
                                            C.c_double, i32, C.POINTER(C.c_double), vp]
    lib.po_tsne_attraction_step.restype = i32
    lib.po_linkage_workspace.argtypes = [i64]
    lib.po_linkage_workspace.restype = i64
    lib.po_linkage_run.argtypes = [vp, i64, i32, i64, i32, vp, vp, vp, vp, vp, C.POINTER(i64), vp]
    lib.po_linkage_run.restype = i32
    lib.po_linkage_tree.argtypes = [i64, vp, vp, vp, vp]
    lib.po_linkage_tree.restype = i32
    for name in ("po_nj_capacity", "po_nj_workspace", "po_nj_stage_bytes"):
        getattr(lib, name).argtypes = [i64]
        getattr(lib, name).restype = i64
    lib.po_nj_run.argtypes = [vp, i64, i32, i64, i32, vp, vp, vp, vp, vp, C.POINTER(i64), vp]
    lib.po_nj_run.restype = i32
    lib.po_launch_count.restype = i64
    lib.po_timing_enable.argtypes = [i32]
    lib.po_timing_enable.restype = i32
    lib.po_timing_reset.restype = i32
    lib.po_timing_read.argtypes = [i32, C.POINTER(C.c_double), C.POINTER(i64)]
    lib.po_timing_read.restype = i32
    lib.po_microbench.argtypes = [i32, C.POINTER(C.c_double)]
    lib.po_microbench.restype = i32
    _lib = lib
    return lib


def check(rc, what="call"):
    if rc < 0:
        msg = load().po_last_error().decode("utf-8", "replace")
        raise PhyloligoError("%s failed (status %d): %s" % (what, rc, msg))
    return rc


def pattern_info(pattern: str):
    """(width, k, dim) of a spaced pattern string."""
    lib = load()
    w, k, d = C.c_int(), C.c_int(), C.c_int64()
    check(lib.po_pattern_info(str(pattern).encode(), C.byref(w), C.byref(k), C.byref(d)), "po_pattern_info")
    return w.value, k.value, d.value


def launch_count() -> int:
    return int(load().po_launch_count())


def timing_enable(on: bool):
    load().po_timing_enable(1 if on else 0)


def timing_reset():
    load().po_timing_reset()


def timing_read(family: int):
    ms, n = C.c_double(), C.c_int64()
    check(load().po_timing_read(family, C.byref(ms), C.byref(n)), "po_timing_read")
    return ms.value, n.value


def microbench(kind: int) -> float:
    """0: FP32 FFMA TFLOP/s, 1: MUFU.LG2 1e12 op/s, 2: POPC 1e12 op/s, 3: MUFU.RCP 1e12 op/s,
    4: microseconds per grid barrier of the linkage kernels' grid, 5..12: warp-instructions per SM per clock of
    the packed-f32x2 operand forms listed in csrc/po_microbench.cu."""
    out = C.c_double()
    check(load().po_microbench(kind, C.byref(out)), "po_microbench")
    return out.value
