"""ctypes binding of librcmarl.so (C ABI declared in include/rcmarl.h).

There is deliberately NO fallback: if the shared library is missing or a call
fails, an exception is raised.  The library is built in-tree by
``__graft_entry__.build()`` / ``make -C resilient-consensus-based-marl_b200/csrc``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RCMARL_LIB", os.path.join(_HERE, "librcmarl.so"))   # override: kernel experiments only

MAX_JOBS = 32
MAX_TERMS = 3
MAX_NEIGHBOURS = 16
MAX_H = 7
MAX_GRID = 32
HIDDEN = 20
N_ACTIONS = 5

IN_S, IN_SA, IN_NS = 0, 1, 2
LOSS_MSE, LOSS_CE = 0, 1

c_fp = C.c_void_p  # device pointers travel as integers


class Rows(C.Structure):
    _fields_ = [("sa", c_fp), ("ns", c_fp), ("r", c_fp), ("row_begin", C.c_int64), ("n_rows", C.c_int64),
                ("time_idx", c_fp), ("n_envs", C.c_int32), ("n_agents", C.c_int32)]


class ConsensusJob(C.Structure):
    _fields_ = [("dst", c_fp), ("msgs", c_fp), ("msg_stride", C.c_int64), ("n_hidden", C.c_int32),
                ("n_in", C.c_int32), ("H", C.c_int32), ("in_nodes", C.c_int32 * MAX_NEIGHBOURS)]


class ValueJob(C.Structure):
    _fields_ = [("w", c_fp * MAX_TERMS), ("kind", C.c_int32 * MAX_TERMS), ("scale", C.c_float * MAX_TERMS),
                ("n_terms", C.c_int32), ("n_out", C.c_int32), ("softmax", C.c_int32), ("add_off", C.c_int32),
                ("add", c_fp), ("add_stride", C.c_int64), ("add_scale", C.c_float), ("out", c_fp)]


class GradJob(C.Structure):
    _fields_ = [("w", c_fp), ("target", c_fp), ("sums", c_fp), ("time_idx", c_fp), ("target_stride", C.c_int64),
                ("kind", C.c_int32), ("action_agent", C.c_int32)]


class SgdJob(C.Structure):
    _fields_ = [("dst", c_fp), ("src", c_fp), ("sums", c_fp), ("loss_out", c_fp), ("n", C.c_int32),
                ("first", C.c_int32), ("coef", C.c_float), ("loss_coef", C.c_float), ("loss_accumulate", C.c_int32),
                ("reserved", C.c_int32)]


class AdamJob(C.Structure):
    _fields_ = [("theta", c_fp), ("m", c_fp), ("v", c_fp), ("sums", c_fp), ("loss_out", c_fp), ("n", C.c_int32),
                ("grad_scale", C.c_float), ("lr_t", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float),
                ("eps", C.c_float), ("loss_coef", C.c_float), ("loss_accumulate", C.c_int32), ("reserved", C.c_int32)]


class TeamJob(C.Structure):
    _fields_ = [("w", c_fp), ("msgs", c_fp), ("msg_stride", C.c_int64), ("sums", c_fp), ("agg_out", c_fp),
                ("agg_in", c_fp), ("kind", C.c_int32), ("n_in", C.c_int32), ("H", C.c_int32),
                ("in_nodes", C.c_int32 * MAX_NEIGHBOURS)]


class RolloutArgs(C.Structure):
    _fields_ = [("actor_w", c_fp), ("critic_w", c_fp), ("desired", c_fp), ("sa", c_fp), ("ns", c_fp), ("r", c_fp),
                ("time_begin", C.c_int64), ("est", c_fp), ("ret", c_fp), ("uniforms", c_fp), ("init_state", c_fp),
                ("seed", C.c_uint64), ("env_offset", C.c_int64), ("episode_offset", C.c_int64),
                ("n_envs", C.c_int32), ("n_agents", C.c_int32), ("n_episodes", C.c_int32), ("max_ep_len", C.c_int32),
                ("nrow", C.c_int32), ("ncol", C.c_int32), ("gamma", C.c_float), ("mu", C.c_float),
                ("n_active", C.c_int32), ("reserved", C.c_int32),
                ("state_tab_x", C.c_float * MAX_GRID), ("state_tab_y", C.c_float * MAX_GRID)]


# every symbol include/rcmarl.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("rcmarl_version", C.c_char_p, []),
    ("rcmarl_status_string", C.c_char_p, [C.c_int]),
    ("rcmarl_last_cuda_error", C.c_int, []),
    ("rcmarl_device_info", C.c_int, [C.POINTER(C.c_int)] * 3),
    ("rcmarl_param_count", C.c_int64, [C.c_int, C.c_int]),
    ("rcmarl_workspace_bytes", C.c_int64, [C.c_int, C.c_int]),
    ("rcmarl_grad_grid_plan", C.c_int, [C.c_int, C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int,
                                        C.POINTER(C.c_int32)]),
    ("rcmarl_clip_mean", C.c_int, [c_fp, C.c_int, C.c_int64, C.c_int64, C.c_int, c_fp, c_fp]),
    ("rcmarl_consensus_hidden", C.c_int, [C.POINTER(ConsensusJob), C.c_int, c_fp]),
    ("rcmarl_values", C.c_int, [C.POINTER(Rows), C.POINTER(ValueJob), C.c_int, c_fp]),
    ("rcmarl_grad", C.c_int, [C.POINTER(Rows), C.POINTER(GradJob), C.c_int, C.c_int, c_fp, C.c_int64, C.c_int, c_fp]),
    ("rcmarl_sgd_apply", C.c_int, [C.POINTER(SgdJob), C.c_int, c_fp]),
    ("rcmarl_adam_apply", C.c_int, [C.POINTER(AdamJob), C.c_int, c_fp]),
    ("rcmarl_minibatch_sgd", C.c_int, [C.POINTER(Rows), C.POINTER(GradJob), C.POINTER(SgdJob), C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_float, c_fp, C.c_int64, c_fp]),
    ("rcmarl_minibatch_cells_bytes", C.c_int64, [C.c_int, C.c_int]),
    ("rcmarl_minibatch_steps", C.c_int64, [C.c_int, C.c_int, C.c_int]),
    ("rcmarl_minibatch_fit", C.c_int, [C.POINTER(Rows), C.POINTER(GradJob), C.POINTER(SgdJob), C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_float, c_fp, C.c_int64, C.c_uint32, C.c_int, c_fp]),
    ("rcmarl_overlap_split", C.c_int, [C.c_int, C.POINTER(C.c_int32), C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_int32),
                                       C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int32)]),
    ("rcmarl_team", C.c_int, [C.POINTER(Rows), C.POINTER(TeamJob), C.c_int, c_fp, C.c_int64, c_fp]),
    ("rcmarl_reward_mix", C.c_int, [c_fp, C.c_int64, C.c_int, C.POINTER(C.c_int32), C.c_int, C.c_float, c_fp, c_fp]),
    ("rcmarl_comm_create", C.c_int, [C.c_int, C.c_int, C.c_int64, C.POINTER(C.c_void_p)]),
    ("rcmarl_comm_handle_bytes", C.c_int, []),
    ("rcmarl_comm_export", C.c_int, [C.c_void_p, C.c_char_p]),
    ("rcmarl_comm_connect", C.c_int, [C.c_void_p, C.c_char_p]),
    ("rcmarl_comm_bind", C.c_int, [C.c_void_p]),
    ("rcmarl_comm_error", C.c_int, [C.c_void_p]),
    ("rcmarl_comm_destroy", C.c_int, [C.c_void_p]),
    ("rcmarl_rollout", C.c_int, [C.POINTER(RolloutArgs), c_fp]),
    ("rcmarl_episode_means", C.c_int, [c_fp, C.c_int, C.c_int, C.c_int, c_fp, c_fp]),
    ("rcmarl_env_step", C.c_int, [c_fp, c_fp, c_fp, C.c_int, C.c_int, C.c_int, c_fp, c_fp]),
]

_lib = None


class RcmarlError(RuntimeError):
    pass


def lib():
    """Load librcmarl.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RcmarlError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / PyTorch fallback for the RPBCAC kernels)")
        l = C.CDLL(LIB_PATH)
        lax = os.environ.get("RCMARL_LIB_LAX") == "1"      # kernel A/B runs against older builds only (tools/ab_grad.py)
        for name, res, args in SYMBOLS:
            if lax and not hasattr(l, name):
                continue
            f = getattr(l, name)          # AttributeError if the ABI and the header diverge
            f.restype = res
            f.argtypes = args
        _lib = l
    return _lib


def check(status, what):
    if status != 0:
        l = lib()
        msg = l.rcmarl_status_string(status).decode()
        raise RcmarlError(f"{what}: {msg} (status {status}, cudaError {l.rcmarl_last_cuda_error()})")


def param_count(d_in, n_out):
    return d_in * HIDDEN + HIDDEN + HIDDEN * HIDDEN + HIDDEN + HIDDEN * n_out + n_out
