"""ctypes binding of libsympa_b200.so (the C ABI of include/sympa_b200.h).  Fails loudly when the
library is missing - there is no fallback path."""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SYMPA_B200_LIB") or os.path.join(_PKG, "libsympa_b200.so")

KIND = {"upper": 0, "bounded": 1, "spd": 2}
METRIC = {"riem": 0, "fone": 1, "finf": 2, "fmin": 3, "wsum": 4}
MAX_N = 10
OPT_SPLIT_PATH = 1
OPT_SCATTER_PASS_MB = 2

STATUS_BITS = {
    1: "a point is outside the manifold (Cholesky pivot <= 0)",
    2: "a Takagi value exceeded 1.01 (reference assert siegel_manifold.py:66)",
    4: "Jacobi sweep cap reached",
    8: "non-finite distance",
    16: "table index out of range",
    32: "a sampling source reaches no other node",
}

EXPORTS = (
    "sympa_version",
    "sympa_error_string",
    "sympa_last_cuda_error",
    "sympa_workspace_bytes",
    "sympa_scratch_bytes",
    "sympa_rsgd_step",
    "sympa_rsgd_step_ex",
    "sympa_set_option",
    "sympa_probe_fp64",
    "sympa_dist_forward",
    "sympa_dist_backward",
    "sympa_distortion_step",
    "sympa_dist_matrix",
    "sympa_backward_workspace_bytes",
    "sympa_dist_backward_table",
    "sympa_table_grad_scatter",
    "sympa_table_grad_expand",
    "sympa_table_grad_scatter_rows",
    "sympa_table_grad_scatter_add",
    "sympa_distortion_loss_forward",
    "sympa_distortion_loss_backward",
    "sympa_bounded_rows_to_upper",
    "sympa_bounded_rows_backward",
    "sympa_check_points",
    "sympa_average_precision_workspace_bytes",
    "sympa_average_precision",
    "sympa_hop_distances_workspace_bytes",
    "sympa_hop_distances",
    "sympa_distortion_rows",
    "sympa_distortion_rows_full",
    "sympa_sample_pairs_workspace_bytes",
    "sympa_sample_pairs",
    "sympa_dist_rows",
    "sympa_row_topk_workspace_bytes",
    "sympa_row_topk",
    "sympa_target_ranks_workspace_bytes",
    "sympa_target_ranks",
)

_lib = None


class SympaLibraryError(RuntimeError):
    pass


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SympaLibraryError(
            f"{LIB_PATH} is missing: build it with `python -m sympa_b200.build` "
            "(or __graft_entry__.build()); sympa_b200 has no CPU / eager fallback")
    lib = ctypes.CDLL(LIB_PATH)
    P, I, L, D = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
    lib.sympa_version.restype = I
    lib.sympa_error_string.restype = ctypes.c_char_p
    lib.sympa_error_string.argtypes = [I]
    lib.sympa_last_cuda_error.restype = ctypes.c_char_p
    lib.sympa_workspace_bytes.restype = L
    lib.sympa_workspace_bytes.argtypes = [I, I, L]
    lib.sympa_rsgd_step.restype = I
    lib.sympa_rsgd_step.argtypes = [I, I, L, P, P, D, P, P, P]
    lib.sympa_rsgd_step_ex.restype = I
    lib.sympa_rsgd_step_ex.argtypes = [I, I, L, P, P, D, P, P, I, P]
    lib.sympa_probe_fp64.restype = L
    lib.sympa_probe_fp64.argtypes = [I, P, P]
    lib.sympa_set_option.restype = I
    lib.sympa_set_option.argtypes = [I, I]
    lib.sympa_scratch_bytes.restype = L
    lib.sympa_scratch_bytes.argtypes = [I, I, L]
    lib.sympa_dist_forward.restype = I
    lib.sympa_dist_forward.argtypes = [I, I, I, L, P, P, P, L, P, P, P, P, P, P, L, P, P]
    lib.sympa_dist_backward.restype = I
    lib.sympa_dist_backward.argtypes = [I, I, I, L, P, P, P, P, P, L, P, P, P, P, P]
    lib.sympa_distortion_step.restype = I
    lib.sympa_distortion_step.argtypes = [I, I, I, L, P, L, P, P, D, P, P, P, P, P, P, P, L, P, P]
    lib.sympa_dist_matrix.restype = I
    lib.sympa_dist_matrix.argtypes = [I, I, I, P, L, L, L, P, P, P, L, P, P]
    lib.sympa_backward_workspace_bytes.restype = L
    lib.sympa_backward_workspace_bytes.argtypes = [I, I, L]
    lib.sympa_dist_backward_table.restype = I
    lib.sympa_dist_backward_table.argtypes = [I, I, I, L, P, P, P, L, P, P, P, P, P, L, I, P]
    lib.sympa_table_grad_scatter.restype = I
    lib.sympa_table_grad_scatter.argtypes = [I, I, I, L, P, P, L, P, P, P, P, P, L, P]
    lib.sympa_table_grad_scatter_rows.restype = I
    lib.sympa_table_grad_scatter_rows.argtypes = [I, I, L, P, P, L, P, L, L, P, L, P]
    lib.sympa_table_grad_scatter_add.restype = I
    lib.sympa_table_grad_scatter_add.argtypes = [I, I, L, P, P, L, P, P, L, I, P, P]
    lib.sympa_table_grad_expand.restype = I
    lib.sympa_table_grad_expand.argtypes = [I, I, L, P, P, I, P]
    lib.sympa_distortion_loss_forward.restype = I
    lib.sympa_distortion_loss_forward.argtypes = [L, P, P, P, P]
    lib.sympa_distortion_loss_backward.restype = I
    lib.sympa_distortion_loss_backward.argtypes = [L, P, P, P, P, P]
    lib.sympa_check_points.restype = I
    lib.sympa_check_points.argtypes = [I, I, L, P, ctypes.c_double, ctypes.c_double, P, P]
    lib.sympa_bounded_rows_to_upper.restype = I
    lib.sympa_bounded_rows_to_upper.argtypes = [I, L, P, P, P, P]
    lib.sympa_bounded_rows_backward.restype = I
    lib.sympa_bounded_rows_backward.argtypes = [I, L, P, P, P, I, P]
    lib.sympa_average_precision_workspace_bytes.restype = L
    lib.sympa_average_precision_workspace_bytes.argtypes = [L, L]
    lib.sympa_average_precision.restype = I
    lib.sympa_average_precision.argtypes = [L, L, L, P, P, P, P, P, L, P, P]
    lib.sympa_hop_distances_workspace_bytes.restype = L
    lib.sympa_hop_distances_workspace_bytes.argtypes = [L]
    lib.sympa_hop_distances.restype = I
    lib.sympa_hop_distances.argtypes = [L, L, L, P, P, P, P, L, P, P]
    lib.sympa_distortion_rows.restype = I
    lib.sympa_distortion_rows.argtypes = [L, L, L, P, P, D, P, P, P, P, P, P]
    lib.sympa_distortion_rows_full.restype = I
    lib.sympa_distortion_rows_full.argtypes = [L, L, L, P, P, D, P, P, P, P, P, P]
    lib.sympa_sample_pairs_workspace_bytes.restype = L
    lib.sympa_sample_pairs_workspace_bytes.argtypes = [L]
    lib.sympa_sample_pairs.restype = I
    lib.sympa_sample_pairs.argtypes = [L, P, P, L, P, L, ctypes.c_uint64, ctypes.c_uint64, P, P, P, L, P, P]
    lib.sympa_dist_rows.restype = I
    lib.sympa_dist_rows.argtypes = [I, I, I, P, L, P, L, P, P, P, L, P, P]
    lib.sympa_row_topk_workspace_bytes.restype = L
    lib.sympa_row_topk_workspace_bytes.argtypes = [L, L, L]
    lib.sympa_row_topk.restype = I
    lib.sympa_row_topk.argtypes = [L, L, P, P, L, P, P, P, L, P, P]
    lib.sympa_target_ranks_workspace_bytes.restype = L
    lib.sympa_target_ranks_workspace_bytes.argtypes = [L, L]
    lib.sympa_target_ranks.restype = I
    lib.sympa_target_ranks.argtypes = [L, L, P, P, P, P, P, P, P, P, P, L, P, P]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        lib = load()
        msg = lib.sympa_error_string(rc).decode()
        if rc == 3:
            msg += ": " + lib.sympa_last_cuda_error().decode()
        raise RuntimeError(f"sympa_b200: {msg} (code {rc})")
