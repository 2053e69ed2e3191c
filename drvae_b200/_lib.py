"""ctypes binding of the C ABI declared in include/drvae_b200.h.

There is no CPU fallback: if the shared library has not been built (python -m drvae_b200.build)
or a call fails, a RuntimeError is raised with the library's own message.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libdrvae_b200.so")
if os.environ.get("DRVAE_B200_LIB"):  # measurement knob: an instrumented build (tools/wait_profile.py)
    LIB_PATH = os.environ["DRVAE_B200_LIB"]
_lib = None

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_ll = ctypes.c_longlong
c_float = ctypes.c_float
MAX_HIDDEN = 4

KIND = {"drvae": 0, "pvae": 1, "vfae": 2}


class Arch(ctypes.Structure):
    _fields_ = [("kind", c_int), ("dim_x", c_int), ("dim_y", c_int), ("dim_z1", c_int), ("dim_z3", c_int),
                ("n_enc_z1", c_int), ("enc_z1", c_int * MAX_HIDDEN),
                ("n_dec_x", c_int), ("dec_x", c_int * MAX_HIDDEN),
                ("n_enc_z3", c_int), ("enc_z3", c_int * MAX_HIDDEN),
                ("n_dec_z1", c_int), ("dec_z1", c_int * MAX_HIDDEN),
                ("weight_norm", c_int), ("L", c_int), ("max_batch", c_int)]


class Batch(ctypes.Structure):
    _fields_ = [("x1", c_void_p), ("x2", c_void_p), ("y", c_void_p), ("has_x2", c_void_p), ("has_y", c_void_p),
                ("N", c_int), ("row_index", c_void_p), ("dataset_rows", c_int)]


class Noise(ctypes.Structure):
    _fields_ = [("eps", c_void_p), ("seed", ctypes.c_ulonglong), ("row_offset", c_ll)]


class HParams(ctypes.Structure):
    _fields_ = [("step", c_int), ("training", c_int), ("add_noise", c_int), ("noise_std", c_float),
                ("beta_pert", c_float), ("pertloss_rate", c_float), ("kl_qz2pz2_rate", c_float),
                ("yloss_rate", c_float), ("kl_min", c_float), ("lr", c_float), ("beta1", c_float),
                ("beta2", c_float), ("adam_eps", c_float), ("weight_decay", c_float),
                ("global_N", c_int), ("global_Np", c_int), ("global_Nlab", c_int),
                ("log_prior_y", c_float * 8), ("global_counts_dev", c_void_p)]


class MemberHParams(ctypes.Structure):
    _fields_ = [("yloss_rate", c_float), ("pertloss_rate", c_float), ("kl_qz2pz2_rate", c_float), ("noise_std", c_float),
                ("lr", c_float), ("weight_decay", c_float), ("log_prior_y", c_float * 8)]


class EpsLayout(ctypes.Structure):
    _fields_ = [("off_x1", c_ll), ("off_x2", c_ll), ("off_z1", c_ll), ("off_z2", c_ll), ("off_z2f", c_ll),
                ("off_z3", c_ll), ("total", c_ll)]


class DpPeers(ctypes.Structure):
    _fields_ = [("rank", c_int), ("world", c_int), ("grad_ptrs", ctypes.POINTER(c_void_p)), ("ctl_ptrs", ctypes.POINTER(c_void_p)),
                ("grads_multicast", c_void_p)]


class InferOut(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ("z1_mu", "z1_lv", "z2_mu", "z2_lv", "proba", "pred", "px1_mu", "px1_sg",
                                        "px2_mu", "px2_sg")]


# every symbol include/drvae_b200.h declares (tests check the library exports all of them)
EXPORTS = ["drvae_last_error", "drvae_plan_create", "drvae_plan_destroy", "drvae_plan_param_count",
           "drvae_plan_num_tensors", "drvae_plan_tensor_info", "drvae_plan_eps_layout",
           "drvae_plan_workspace_bytes", "drvae_plan_bind", "drvae_sync_shadows", "drvae_train_step",
           "drvae_loss_forward", "drvae_grad_step", "drvae_adam_step", "drvae_infer", "drvae_set_gemm_impl",
           "drvae_plan_launch_count", "drvae_debug_buffer", "drvae_debug_gemm", "drvae_profile_begin",
           "drvae_profile_end", "drvae_plan_num_buckets", "drvae_plan_bucket_info", "drvae_stream_wait_bucket", "drvae_set_graph", "drvae_plan_graph_replays", "drvae_debug_wait_stats",
           "drvae_debug_side_delay", "drvae_plan_tensor_ld", "drvae_trace_begin", "drvae_trace_end", "drvae_debug_dwa_stats", "drvae_set_infer_precision", "drvae_dp_attach", "drvae_dp_grad_floats",
           "drvae_dp_counts_ptr", "drvae_dp_exchange_counts", "drvae_dp_train_step", "drvae_plan_graph_failures", "drvae_set_step_kernel", "drvae_plan_step_kernel_launches",
           "drvae_eval_workspace_bytes", "drvae_eval_x_reconstruction", "drvae_set_member_hparams", "drvae_plan_create_clf"]


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "drvae_b200: %s is missing. Build it with `python -m drvae_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    P = ctypes.POINTER
    lib.drvae_last_error.restype = ctypes.c_char_p
    lib.drvae_plan_create.restype = c_int
    lib.drvae_plan_create.argtypes = [P(Arch), c_int, P(c_void_p)]
    lib.drvae_plan_create_clf.restype = c_int
    lib.drvae_plan_create_clf.argtypes = [P(Arch), c_int, P(c_int), c_int, P(c_void_p)]
    lib.drvae_plan_destroy.restype = c_int
    lib.drvae_plan_destroy.argtypes = [c_void_p]
    lib.drvae_plan_param_count.restype = c_ll
    lib.drvae_plan_param_count.argtypes = [c_void_p]
    lib.drvae_plan_num_tensors.restype = c_int
    lib.drvae_plan_num_tensors.argtypes = [c_void_p]
    lib.drvae_plan_tensor_info.restype = c_int
    lib.drvae_plan_tensor_info.argtypes = [c_void_p, c_int, ctypes.c_char_p, c_int, P(c_int), P(c_int), P(c_ll)]
    lib.drvae_plan_tensor_ld.restype = c_int
    lib.drvae_plan_tensor_ld.argtypes = [c_void_p, c_int]
    lib.drvae_plan_eps_layout.restype = c_int
    lib.drvae_plan_eps_layout.argtypes = [c_void_p, P(EpsLayout)]
    lib.drvae_plan_workspace_bytes.restype = c_ll
    lib.drvae_plan_workspace_bytes.argtypes = [c_void_p]
    lib.drvae_plan_launch_count.restype = c_ll
    lib.drvae_plan_launch_count.argtypes = [c_void_p]
    lib.drvae_plan_bind.restype = c_int
    lib.drvae_plan_bind.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.drvae_sync_shadows.restype = c_int
    lib.drvae_sync_shadows.argtypes = [c_void_p, c_void_p]
    for name in ("drvae_train_step", "drvae_loss_forward", "drvae_grad_step", "drvae_dp_train_step"):
        fn = getattr(lib, name)
        fn.restype = c_int
        fn.argtypes = [c_void_p, P(Batch), P(Noise), P(HParams), c_void_p, c_void_p]
    lib.drvae_adam_step.restype = c_int
    lib.drvae_adam_step.argtypes = [c_void_p, P(HParams), c_void_p]
    lib.drvae_plan_num_buckets.restype = c_int
    lib.drvae_plan_num_buckets.argtypes = [c_void_p]
    lib.drvae_plan_bucket_info.restype = c_int
    lib.drvae_plan_bucket_info.argtypes = [c_void_p, c_int, P(c_ll), P(c_ll)]
    lib.drvae_stream_wait_bucket.restype = c_int
    lib.drvae_stream_wait_bucket.argtypes = [c_void_p, c_int, c_void_p]
    lib.drvae_set_graph.restype = c_int
    lib.drvae_set_graph.argtypes = [c_void_p, c_int]
    lib.drvae_plan_graph_failures.restype = c_ll
    lib.drvae_plan_graph_failures.argtypes = [c_void_p]
    lib.drvae_eval_workspace_bytes.restype = c_ll
    lib.drvae_eval_workspace_bytes.argtypes = [c_int, c_int]
    lib.drvae_eval_x_reconstruction.restype = c_int
    lib.drvae_eval_x_reconstruction.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]
    lib.drvae_set_step_kernel.restype = c_int
    lib.drvae_set_step_kernel.argtypes = [c_void_p, c_int]
    lib.drvae_plan_step_kernel_launches.restype = c_ll
    lib.drvae_plan_step_kernel_launches.argtypes = [c_void_p]
    lib.drvae_plan_graph_replays.restype = c_ll
    lib.drvae_plan_graph_replays.argtypes = [c_void_p]
    lib.drvae_infer.restype = c_int
    lib.drvae_infer.argtypes = [c_void_p, c_void_p, c_int, P(InferOut), c_void_p]
    lib.drvae_set_member_hparams.restype = c_int
    lib.drvae_set_member_hparams.argtypes = [c_void_p, P(MemberHParams), c_int, c_void_p]
    lib.drvae_debug_wait_stats.restype = c_int
    lib.drvae_debug_wait_stats.argtypes = [c_void_p, c_int]
    lib.drvae_debug_dwa_stats.restype = c_int
    lib.drvae_debug_dwa_stats.argtypes = [c_void_p, c_int, c_void_p]
    lib.drvae_dp_attach.restype = c_int
    lib.drvae_dp_attach.argtypes = [c_void_p, P(DpPeers)]
    lib.drvae_dp_grad_floats.restype = c_ll
    lib.drvae_dp_grad_floats.argtypes = [c_void_p]
    lib.drvae_dp_counts_ptr.restype = c_void_p
    lib.drvae_dp_counts_ptr.argtypes = [c_void_p]
    lib.drvae_dp_exchange_counts.restype = c_int
    lib.drvae_dp_exchange_counts.argtypes = [c_void_p, c_ll, c_ll, c_ll, c_ll, c_void_p]
    lib.drvae_set_infer_precision.restype = c_int
    lib.drvae_set_infer_precision.argtypes = [c_void_p, c_int]
    lib.drvae_trace_begin.restype = c_int
    lib.drvae_trace_begin.argtypes = [c_void_p, c_int]
    lib.drvae_trace_end.restype = c_int
    lib.drvae_trace_end.argtypes = [c_void_p, ctypes.c_char_p, c_int]
    lib.drvae_debug_side_delay.restype = c_int
    lib.drvae_debug_side_delay.argtypes = [c_void_p, c_ll]
    lib.drvae_set_gemm_impl.restype = c_int
    lib.drvae_set_gemm_impl.argtypes = [c_void_p, c_int]
    lib.drvae_profile_begin.restype = c_int
    lib.drvae_profile_begin.argtypes = [c_void_p]
    lib.drvae_profile_end.restype = c_int
    lib.drvae_profile_end.argtypes = [c_void_p, ctypes.c_char_p, c_int]
    lib.drvae_debug_buffer.restype = c_int
    lib.drvae_debug_buffer.argtypes = [c_void_p, ctypes.c_char_p, P(c_void_p), P(c_ll), P(c_ll), P(c_int), P(c_int)]
    lib.drvae_debug_gemm.restype = c_int
    lib.drvae_debug_gemm.argtypes = [
        c_int, c_int, c_void_p, c_int, c_int, c_ll, c_void_p, c_int, c_int, c_ll, c_void_p, c_int, c_ll,
        c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p]
    _lib = lib
    return lib


def check(status, what=""):
    if status != 0:
        msg = load().drvae_last_error()
        raise RuntimeError("drvae_b200 %s failed (status %d): %s" % (what, status, msg.decode() if msg else "?"))
