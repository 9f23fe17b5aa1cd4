"""ctypes binding of libswimmer_ars.so (C ABI declared in include/swimmer_ars.h).

PyTorch is used only as plumbing: device memory (tensor.data_ptr()), streams
(torch.cuda.current_stream()) and torch.distributed.  All arithmetic happens in the CUDA
library; there is no CPU fallback -- if the library or a GPU is missing, calls raise.
"""
import ctypes
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SWM_LIB_PATH", os.path.join(_HERE, "libswimmer_ars.so"))

GYM, RLGLUE = 0, 1
POLICY_FIXED_ACTION, POLICY_EXPLICIT, POLICY_PHILOX, POLICY_DELTAS = 0, 1, 2, 3
DELTA_PM1, DELTA_01 = 0, 1
ARS_AGENT, ARS_TOPB, ARS_RLGLUE = 0, 1, 2
KERNEL_AUTO, KERNEL_THREAD, KERNEL_LANES, KERNEL_LANES2, KERNEL_LANES3 = 0, 1, 2, 3, 4  # swm_rollout_kernel
MIN_SEGMENTS, MAX_SEGMENTS = 2, 10
ABI_VERSION = 3  # include/swimmer_ars.h SWM_ABI_VERSION
MAX_MODELS_PER_STEP = 24  # SWM_MAX_MODELS_PER_STEP
MAX_COST_FORMS = 32  # SWM_MAX_COST_FORMS
MAX_SIM_MODELS = 16  # SWM_MAX_SIM_MODELS
MAX_LOOKAHEAD = 1024  # SWM_MAX_LOOKAHEAD
MAX_CANDIDATES = 1024  # SWM_MAX_CANDIDATES
CMAES_MIN_POPSIZE = 2  # SWM_CMAES_MIN_POPSIZE
FIELDS = {"m_i": 0, "l_i": 1, "k": 2}  # swm_field
CMAES_STOP = {0: "running", 1: "maxiter", 2: "tolfun", 3: "tolx", 4: "conditioncov"}  # swm_cmaes_status

_dp = ctypes.c_void_p


class SwmParams(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int32), ("_pad", ctypes.c_int32), ("l_i", ctypes.c_double),
                ("m_i", ctypes.c_double), ("k", ctypes.c_double), ("h", ctypes.c_double),
                ("max_u", ctypes.c_double), ("direction", ctypes.c_double * 2)]


class SwmPhilox(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64), ("iteration", ctypes.c_uint32), ("dir0", ctypes.c_uint32),
                ("dist", ctypes.c_int32), ("_pad", ctypes.c_int32), ("iteration_dev", _dp)]


class SwmScreen(ctypes.Structure):
    _fields_ = [("enabled", ctypes.c_int32), ("_pad", ctypes.c_int32), ("sim", SwmParams),
                ("sim_thresh", ctypes.c_double), ("real_thresh", ctypes.c_double),
                ("violations", _dp), ("frozen_at", _dp)]


class SwmRollout(ctypes.Structure):
    _fields_ = [("variant", ctypes.c_int32), ("policy_mode", ctypes.c_int32),
                ("normalize", ctypes.c_int32), ("clip_actions", ctypes.c_int32),
                ("H", ctypes.c_int32), ("rollouts_per_policy", ctypes.c_int32),
                ("B", ctypes.c_int64), ("actions", _dp), ("policies", _dp), ("deltas", _dp),
                ("nu", ctypes.c_double), ("philox", SwmPhilox), ("dir_mask", _dp), ("mean", _dp),
                ("inv_sigma", _dp), ("init_state", _dp), ("init_state_count", ctypes.c_int64),
                ("init_perturb", ctypes.c_double), ("returns", _dp), ("final_state", _dp),
                ("trajectory", _dp), ("stats_partial", _dp), ("stats_pivot", _dp),
                ("screen", SwmScreen), ("accumulate_returns", ctypes.c_int32), ("kernel", ctypes.c_int32),
                ("schedule_sub", ctypes.c_int32), ("schedule_chunk", ctypes.c_int32)]


class SwmPack(ctypes.Structure):
    """swm_pack_t (include/swimmer_ars.h): arguments of the fused pack + exchange + unpack launch."""
    _fields_ = [("returns_local", _dp), ("n_local", ctypes.c_int32), ("rollouts_per_policy", ctypes.c_int32),
                ("mask_local", _dp), ("stats_partial", _dp), ("n_blocks", ctypes.c_int64),
                ("n_features", ctypes.c_int32), ("gathered_world", ctypes.c_int32), ("samples", ctypes.c_double),
                ("units", _dp), ("pivot", _dp), ("returns_all", _dp), ("mask_all", _dp), ("records", _dp),
                ("record_out", _dp), ("gathered_in", _dp)]


class SwmRlglueProtocol(ctypes.Structure):
    """swm_rlglue_protocol_t (include/swimmer_ars.h)."""
    _fields_ = [("N", ctypes.c_int32), ("b", ctypes.c_int32), ("H", ctypes.c_int32), ("n_it", ctypes.c_int32),
                ("alpha", ctypes.c_double), ("nu", ctypes.c_double), ("deltas", _dp), ("seed", ctypes.c_uint64),
                ("iteration0", ctypes.c_uint32), ("_pad", ctypes.c_int32), ("state", _dp), ("results", _dp),
                ("table", _dp), ("replicas", ctypes.c_int64)]


class SwmEstimateData(ctypes.Structure):
    """swm_estimate_data_t (include/swimmer_ars.h): recorded data and field map of the estimation objective."""
    _fields_ = [("trajectories", _dp), ("policies", _dp), ("K", ctypes.c_int32), ("H", ctypes.c_int32),
                ("d", ctypes.c_int32), ("fields", ctypes.c_int32 * 3), ("workspace", _dp)]


IPC_HANDLE_BYTES = 64  # SWM_IPC_HANDLE_BYTES


class SwimmerLibError(RuntimeError):
    pass


_lib = None


def build_library(verbose=False):
    """Compiles libswimmer_ars.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j", str(os.cpu_count() or 4)]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout)
    if out.returncode != 0:
        raise SwimmerLibError("building libswimmer_ars.so failed")
    return LIB_PATH


def lib():
    """Loads the CUDA library; raises loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SwimmerLibError(
            "%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C <package>/csrc`). There is no CPU fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    pp = ctypes.POINTER(SwmParams)
    i64, c_int, dbl = ctypes.c_int64, ctypes.c_int, ctypes.c_double
    L.swm_abi_version.restype = c_int
    L.swm_strerror.restype = ctypes.c_char_p
    L.swm_strerror.argtypes = [c_int]
    L.swm_last_cuda_error.restype = ctypes.c_char_p
    L.swm_device_info.argtypes = [ctypes.POINTER(c_int)] * 3
    L.swm_step_batched.argtypes = [pp, c_int, _dp, _dp, _dp, _dp, i64, _dp]
    L.swm_accelerations_batched.argtypes = [pp, c_int, _dp, _dp, _dp, i64, _dp]
    L.swm_step_batched_models.argtypes = [pp, c_int, i64, _dp, _dp, _dp, _dp, _dp]
    L.swm_rollout.argtypes = [pp, ctypes.POINTER(SwmRollout), _dp]
    L.swm_rollout_costed.argtypes = [pp, ctypes.POINTER(SwmRollout), _dp, c_int, _dp]
    L.swm_rollout_ensemble.argtypes = [pp, ctypes.POINTER(SwmRollout), pp, c_int, _dp, c_int, _dp]
    L.swm_rollout_shielded.argtypes = [pp, ctypes.POINTER(SwmRollout), pp, c_int, _dp, c_int, _dp, _dp, _dp]
    L.swm_rollout_lookahead.argtypes = [pp, ctypes.POINTER(SwmRollout), pp, c_int, _dp, c_int, _dp, c_int, _dp, _dp]
    L.swm_rollout_models.argtypes = [pp, c_int, ctypes.POINTER(SwmRollout), _dp]
    L.swm_rollout_stats_blocks.argtypes = [pp, ctypes.POINTER(SwmRollout), _dp]
    L.swm_rollout_stats_blocks.restype = i64
    L.swm_rollout_kernel_choice.argtypes = [pp, ctypes.POINTER(SwmRollout)]
    L.swm_rollout_schedule.argtypes = [pp, ctypes.POINTER(SwmRollout), _dp, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]
    L.swm_stats_finalize.argtypes = [_dp, i64, c_int, dbl, _dp, _dp, _dp, _dp]
    L.swm_stats_merge.argtypes = [_dp, _dp, c_int, c_int, _dp, _dp, _dp]
    L.swm_reduce_returns.argtypes = [_dp, i64, c_int, _dp, _dp]
    L.swm_ars_topb.argtypes = [_dp, _dp, c_int, _dp, _dp]
    L.swm_ars_update.argtypes = [_dp, c_int, _dp, c_int, _dp, c_int, _dp, dbl, c_int, dbl,
                                 ctypes.POINTER(SwmPhilox), _dp, _dp, _dp]
    L.swm_screen_mask.argtypes = [_dp, c_int, dbl, _dp, _dp, _dp, _dp]
    L.swm_screen_mask_models.argtypes = [_dp, c_int, c_int, dbl, _dp, _dp, _dp, _dp]
    L.swm_policy_actions.argtypes = [pp, _dp, _dp, c_int, _dp, _dp, c_int, _dp, i64, _dp]
    L.swm_philox_deltas.argtypes = [ctypes.POINTER(SwmPhilox), c_int, c_int, _dp, _dp]
    L.swm_fp64_probe.argtypes = [c_int, c_int, c_int, _dp, ctypes.POINTER(dbl), _dp]
    L.swm_counter_add.argtypes = [_dp, ctypes.c_uint32, _dp]
    L.swm_record_nanmean.argtypes = [_dp, c_int, _dp, _dp, ctypes.c_uint32, _dp]
    L.swm_rlglue_set_params.argtypes = [pp]
    L.swm_rlglue_protocol_state_doubles.argtypes = [c_int]
    L.swm_rlglue_protocol_state_doubles.restype = i64
    L.swm_rlglue_protocol.argtypes = [pp, ctypes.POINTER(SwmRlglueProtocol), _dp]
    L.swm_pack_record_doubles.argtypes = [c_int, c_int, c_int]
    L.swm_pack_record_doubles.restype = i64
    L.swm_exchange_create.argtypes = [c_int, c_int, i64, ctypes.POINTER(_dp)]
    L.swm_exchange_ipc_handle.argtypes = [_dp, _dp]
    L.swm_exchange_open_peers.argtypes = [_dp, _dp]
    L.swm_exchange_status.argtypes = [_dp, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
    L.swm_exchange_destroy.argtypes = [_dp]
    L.swm_ars_pack_exchange.argtypes = [_dp, ctypes.POINTER(SwmPack), _dp]
    ed, u64 = ctypes.POINTER(SwmEstimateData), ctypes.c_uint64
    L.swm_prediction_error_workspace_doubles.argtypes = [c_int, c_int, c_int]
    L.swm_prediction_error_workspace_doubles.restype = i64
    L.swm_prediction_error.argtypes = [pp, ed, _dp, c_int, _dp, _dp]
    L.swm_cmaes_state_doubles.argtypes = [c_int, c_int]
    L.swm_cmaes_state_doubles.restype = i64
    L.swm_cmaes_init.argtypes = [_dp, c_int, c_int, ctypes.POINTER(dbl), dbl, dbl, dbl, i64, _dp]
    L.swm_cmaes_sample.argtypes = [_dp, c_int, c_int, u64, _dp, _dp]
    L.swm_cmaes_update.argtypes = [_dp, c_int, c_int, _dp, _dp, _dp]
    L.swm_cmaes_generation.argtypes = [_dp, c_int, c_int, u64, pp, ed, _dp, _dp, _dp]
    if L.swm_abi_version() != ABI_VERSION:
        raise SwimmerLibError("ABI version mismatch")
    _lib = L
    return L


def check(rc):
    if rc != 0:
        L = lib()
        msg = L.swm_strerror(rc).decode()
        if rc == -3:
            msg += ": " + L.swm_last_cuda_error().decode()
        raise SwimmerLibError("libswimmer_ars: %s (status %d)" % (msg, rc))


def require_cuda():
    if not torch.cuda.is_available():
        raise SwimmerLibError("a CUDA device is required: this package has no CPU fallback")


def make_params(n=3, l_i=1.0, m_i=1.0, k=10.0, h=0.001, max_u=5.0, direction=(1.0, 0.0)):
    n = int(n)
    if not (MIN_SEGMENTS <= n <= MAX_SEGMENTS):
        raise ValueError("n must be in [%d, %d], got %d" % (MIN_SEGMENTS, MAX_SEGMENTS, n))
    p = SwmParams()
    p.n = n
    p.l_i, p.m_i, p.k, p.h, p.max_u = float(l_i), float(m_i), float(k), float(h), float(max_u)
    p.direction[0], p.direction[1] = float(direction[0]), float(direction[1])
    return p


def ptr(t):
    """Device pointer of a contiguous float64/int32 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda or not t.is_contiguous():
        raise ValueError("expected a contiguous CUDA tensor")
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def f64(t, shape=None):
    if t.dtype != torch.float64:
        raise ValueError("expected float64, got %s" % t.dtype)
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (tuple(shape), tuple(t.shape)))
    return t
