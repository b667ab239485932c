"""ctypes binding of librnvp_b200.so (C ABI declared in include/rnvp.h).

The library is built in-tree by ``__graft_entry__.build()`` /
``make -C probaforms_b200/csrc``.  Loading fails loudly if it is missing: the
product has no other execution path.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "librnvp_b200.so")

_lib = None

c_desc_p = C.c_void_p
c_f32_p = C.c_void_p      # raw device pointers (tensor.data_ptr())
c_i64_p = C.c_void_p
c_stream = C.c_void_p

# name -> (restype, argtypes); every symbol include/rnvp.h declares
SIGNATURES = {
    "rnvp_desc_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int,
                                   C.POINTER(c_desc_p)]),
    "rnvp_desc_destroy": (None, [c_desc_p]),
    "rnvp_param_count": (C.c_int64, [c_desc_p]),
    "rnvp_packed_count": (C.c_int64, [c_desc_p]),
    "rnvp_grad_count": (C.c_int64, [c_desc_p]),
    "rnvp_workspace_bytes": (C.c_int64, [c_desc_p, C.c_int64]),
    "rnvp_param_tensors": (C.c_int, [c_desc_p, C.POINTER(C.c_int64), C.c_int]),
    "rnvp_plan_info": (C.c_int, [c_desc_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                 C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "rnvp_pack_params": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_stream]),
    "rnvp_unpack_grads": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_stream]),
    "rnvp_forward": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, C.c_int64, C.c_int, C.c_int,
                               c_f32_p, c_f32_p, c_f32_p, c_stream]),
    "rnvp_inverse": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, C.c_int64, C.c_int, C.c_int,
                               c_f32_p, c_stream]),
    "rnvp_sample": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, C.c_int64, C.c_uint64, C.c_int64, c_f32_p, c_stream]),
    "rnvp_backward": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, C.c_int64, C.c_float,
                                c_f32_p, c_f32_p, c_f32_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_adam_step": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p,
                                 C.c_float, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                 C.c_int64, C.c_int, c_f32_p, c_f32_p, C.c_float, c_stream]),
    "rnvp_fit_epoch": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, C.c_int64,
                                 C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int64, c_f32_p,
                                 c_f32_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_wgrad_record_floats": (C.c_int, [c_desc_p]),
    "rnvp_wgrad_sweep": (C.c_int, [c_desc_p, c_f32_p, C.c_int64, c_f32_p, c_f32_p, c_stream]),
    "rnvp_set_path": (C.c_int, [c_desc_p, C.c_int]),
    "rnvp_debug_set_trace": (C.c_int, [C.c_void_p]),
    "rnvp_perm_create": (C.c_int, [C.c_uint64, C.c_int64, C.c_void_p, C.POINTER(C.c_void_p)]),
    "rnvp_perm_advance": (C.c_int64, [C.c_void_p, C.c_int64]),
    "rnvp_perm_destroy": (None, [C.c_void_p]),
    "rnvp_host_gather_xc": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_int64, C.c_void_p,
                                         C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int]),
    "rnvp_host_copy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "rnvp_mma_selftest": (C.c_int, [c_f32_p, c_f32_p, c_f32_p, C.c_int, C.c_int, C.c_int, c_stream]),
    "rnvp_mmd_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int64, C.c_int, C.c_int]),
    "rnvp_mmd_draws": (C.c_int, [c_f32_p, C.c_int64, c_f32_p, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_mmd_layout": (C.c_int, [C.c_int64, C.c_int64, C.c_int, C.POINTER(C.c_int64)]),
    "rnvp_mmd_begin": (C.c_int, [c_f32_p, C.c_int64, c_f32_p, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                 C.c_void_p, C.c_int64, c_stream]),
    "rnvp_mmd_hist_pass": (C.c_int, [c_f32_p, C.c_int64, c_f32_p, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                     C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, c_stream]),
    "rnvp_mmd_select": (C.c_int, [c_f32_p, C.c_int64, c_f32_p, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                  C.c_void_p, C.c_int64, C.c_int, C.c_void_p, c_stream]),
    "rnvp_mmd_sum_pass": (C.c_int, [c_f32_p, C.c_int64, c_f32_p, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                    C.c_void_p, C.c_int64, C.c_int, C.c_int, c_stream]),
    "rnvp_mmd_finish": (C.c_int, [c_f32_p, C.c_int64, c_f32_p, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                  C.c_void_p, C.c_int64, C.c_void_p, c_stream]),
    "rnvp_boot_moments": (C.c_int, [c_f32_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                    c_stream]),
    "rnvp_rank_workspace_bytes": (C.c_int64, [C.c_int, C.c_int, C.c_int]),
    "rnvp_rank_draws": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                  C.c_double, C.c_void_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_kde_draws": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                 C.c_double, C.c_double, C.c_void_p, c_stream]),
    "rnvp_cn_desc_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int,
                                      C.POINTER(c_desc_p)]),
    "rnvp_cn_desc_destroy": (None, [c_desc_p]),
    "rnvp_cn_param_count": (C.c_int64, [c_desc_p]),
    "rnvp_cn_workspace_bytes": (C.c_int64, [c_desc_p, C.c_int64]),
    "rnvp_cn_inverse": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, C.c_void_p, c_stream]),
    "rnvp_cn_forward": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, C.c_int64, C.c_uint64, C.c_int64,
                                  c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_stream]),
    "rnvp_cn_log_prob": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, C.c_int64, C.c_void_p, C.c_void_p,
                                   C.c_void_p, c_stream]),
    "rnvp_cn_grad": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, C.c_int64, c_f32_p, c_f32_p,
                               C.c_void_p, C.c_int64, c_stream]),
    "rnvp_cn_fit_epoch": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, C.c_int64,
                                    C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int64,
                                    c_f32_p, C.c_void_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_cn_rng_advance": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64]),
    "rnvp_cv_desc_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int,
                                      C.POINTER(c_desc_p)]),
    "rnvp_cv_desc_destroy": (None, [c_desc_p]),
    "rnvp_cv_param_count": (C.c_int64, [c_desc_p]),
    "rnvp_cv_workspace_bytes": (C.c_int64, [c_desc_p, C.c_int64, C.c_int64]),
    "rnvp_cv_encode": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, C.c_int64, c_f32_p, c_f32_p, c_stream]),
    "rnvp_cv_decode": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, C.c_int64, C.c_uint64, C.c_int64, c_f32_p,
                                 c_stream]),
    "rnvp_cv_grad": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, c_f32_p, C.c_int64, C.c_double, c_f32_p,
                               c_f32_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_cv_loss": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, c_f32_p, C.c_int64, C.c_double, c_f32_p,
                               C.c_void_p, C.c_int64, c_stream]),
    "rnvp_cv_fit_epoch": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, C.c_int64,
                                    C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                    C.c_int64, c_f32_p, C.c_uint64, c_f32_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_wg_desc_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int,
                                      C.POINTER(C.c_int), C.c_int, C.POINTER(c_desc_p)]),
    "rnvp_wg_desc_destroy": (None, [c_desc_p]),
    "rnvp_wg_param_count": (C.c_int64, [c_desc_p, C.c_int]),
    "rnvp_wg_workspace_bytes": (C.c_int64, [c_desc_p, C.c_int64, C.c_int64]),
    "rnvp_wg_generate": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, C.c_int64, C.c_uint64, C.c_int64, c_f32_p,
                                   c_stream]),
    "rnvp_wg_critic": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, C.c_int64, c_f32_p, c_stream]),
    "rnvp_wg_grad": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, c_f32_p, C.c_int64, C.c_int, c_f32_p,
                               c_f32_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_wg_loss": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, c_f32_p, C.c_int64, c_f32_p, c_f32_p,
                               C.c_void_p, C.c_int64, c_stream]),
    "rnvp_wg_fit_epoch": (C.c_int, [c_desc_p, c_f32_p, c_f32_p, c_f32_p, c_f32_p, c_i64_p, C.c_int64, C.c_int64,
                                    C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                    c_f32_p, C.c_uint64, c_f32_p, c_f32_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_draw_summary": (C.c_int, [c_f32_p, C.c_int64, C.c_int64, C.POINTER(C.c_double), C.c_int, c_f32_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, c_stream]),
    "rnvp_draw_joint_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int64, C.c_int]),
    "rnvp_draw_joint": (C.c_int, [c_f32_p, C.c_int64, C.c_int64, C.c_int, c_f32_p, C.c_double, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_draw_density": (C.c_int, [c_f32_p, C.c_int64, C.c_int64, C.c_int, c_f32_p, C.c_double, C.c_double,
                                    C.c_void_p, C.c_void_p, C.c_void_p, c_stream]),
    "rnvp_knn_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int64, C.c_int, C.c_int]),
    "rnvp_knn_radii": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_knn_cross": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, c_stream]),
    "rnvp_knn_prdc": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, c_stream]),
    "rnvp_last_error": (C.c_char_p, []),
    "rnvp_version": (C.c_int, []),
}


def build(verbose=False):
    """Compile librnvp_b200.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", f"-j{min(os.cpu_count() or 1, 8)}", "-C", CSRC], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("building librnvp_b200.so failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout)
    return LIB_PATH


def load():
    """dlopen the library and attach the prototypes.  No GPU is needed for this."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C probaforms_b200/csrc` (probaforms_b200 has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class RnvpError(RuntimeError):
    pass


def check(rc, what):
    if rc != 0:
        msg = load().rnvp_last_error()
        raise RnvpError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
