"""ctypes binding of libssd_b200.so (the C ABI declared in include/ssd_b200.h).

There is NO CPU fallback: if the CUDA library is missing or no GPU is present every entry
point raises.  The library is built in-tree by `contracts_b200.build.build()` /
`__graft_entry__.build()`.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# SSD_LIB_PATH: development only (A/B runs of differently built libraries); the shipped library is the in-tree one
LIB_PATH = os.environ.get("SSD_LIB_PATH") or os.path.join(_HERE, "libssd_b200.so")

SSD_ABI_VERSION = 3
ENV_KIND = {"cleanup_new": 0, "harvest_new": 1, "cleanup": 2, "harvest": 3, "selfdrive": 4}
CONTRACT_KIND = {None: 0, "CleanupContract": 1, "HarvestFeaturemodLocalContract": 2,
                 "SelfdriveContractDistprop": 3}
FLAG_COLLECTIVE_REWARD, FLAG_INEQUITY_AVERSE = 1, 2     # SSD_FLAG_* (ssd_config.flags)
SOLVER_RULE = {"max": 0, "majority": 1}                 # SSD_SOLVER_RULE_* (two_stage_train.py:751,758)
OBS_BYTES_PER_AGENT = 675
METRIC_STRIDE = 56


class SsdError(RuntimeError):
    pass


class ssd_config(ctypes.Structure):
    _fields_ = [
        ("abi_version", ctypes.c_int32), ("struct_size", ctypes.c_int32), ("env_kind", ctypes.c_int32), ("num_envs", ctypes.c_int32),
        ("num_agents", ctypes.c_int32), ("map_h", ctypes.c_int32), ("map_w", ctypes.c_int32),
        ("ascii_map", ctypes.c_char_p), ("horizon", ctypes.c_int32), ("contract_kind", ctypes.c_int32),
        ("theta_low", ctypes.c_double), ("theta_high", ctypes.c_double), ("null_prob", ctypes.c_double),
        ("seed", ctypes.c_uint32), ("first_env_id", ctypes.c_uint32), ("device", ctypes.c_int32),
        ("flags", ctypes.c_int32), ("env_params", ctypes.c_double * 8),
    ]


class ssd_step_io(ctypes.Structure):
    _fields_ = [
        ("actions_dev", ctypes.c_void_p), ("obs_dev", ctypes.c_void_p), ("obs_env_stride", ctypes.c_int64),
        ("rew_dev", ctypes.c_void_p), ("base_rew_dev", ctypes.c_void_p), ("transfers_dev", ctypes.c_void_p),
        ("info_dev", ctypes.c_void_p), ("feature_obs_dev", ctypes.c_void_p), ("done_dev", ctypes.c_void_p),
        ("auto_reset", ctypes.c_int32), ("neg_proposals_dev", ctypes.c_void_p), ("neg_accept_dev", ctypes.c_void_p),
        ("neg_decision_dev", ctypes.c_void_p),
    ]


class ssd_host_layout(ctypes.Structure):
    _fields_ = [
        ("total_bytes", ctypes.c_int64), ("count_offset", ctypes.c_int64), ("done_offset", ctypes.c_int64),
        ("rew_i8_offset", ctypes.c_int64), ("records_offset", ctypes.c_int64), ("record_bytes", ctypes.c_int32),
        ("record_capacity", ctypes.c_int32),
    ]


class ssd_checkpoint_layout(ctypes.Structure):
    _fields_ = [("row_bytes", ctypes.c_int64), ("config_tag", ctypes.c_uint64)]


class ssd_policy_out(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_int32), ("dtype", ctypes.c_int32), ("image_dev", ctypes.c_void_p),
                ("contract_dev", ctypes.c_void_p)]


class ssd_flat_policy_out(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_int32), ("dtype", ctypes.c_int32), ("obs_dev", ctypes.c_void_p)]


class ssd_feature_out(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_int32), ("dtype", ctypes.c_int32), ("obs_dev", ctypes.c_void_p)]


class ssd_global_out(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_int32), ("dtype", ctypes.c_int32), ("obs_dev", ctypes.c_void_p)]


POLICY_DTYPE = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}     # SSD_POLICY_F32 / _F16 / _BF16
FEATURE_F64 = 3                                                           # SSD_FEATURE_F64 (ssd_set_feature_output)
GLOBAL_U8 = 4                                                             # SSD_GLOBAL_U8 (ssd_set_global_output)


def policy_dtype_code(dtype):
    """the SSD_POLICY_* code of a policy tensor's torch dtype"""
    if dtype not in POLICY_DTYPE:
        raise ValueError("policy_dtype must be None, torch.float32, torch.float16 or torch.bfloat16, got %r" % (dtype,))
    return POLICY_DTYPE[dtype]



STATS_LEN = 8


class ssd_episode_record(ctypes.Structure):
    _fields_ = [("env_id", ctypes.c_uint32), ("episode", ctypes.c_uint32), ("t", ctypes.c_int32), ("ended", ctypes.c_uint32),
                ("theta", ctypes.c_double), ("pad", ctypes.c_double), ("metrics", ctypes.c_double * METRIC_STRIDE)]


class ssd_episode_log(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_int32), ("capacity", ctypes.c_int32), ("records_dev", ctypes.c_void_p),
                ("count_dev", ctypes.c_void_p)]


def resolve_device(device):
    """torch.device with an explicit index ('cuda' / None mean torch's CURRENT device, not GPU 0).  The C entry points
    switch to the handle's device themselves (and restore the caller's), so a handle on cuda:1 works whatever the
    current device is; streams are always taken from that device."""
    import torch
    if device is None:
        return torch.device("cuda", torch.cuda.current_device())
    device = torch.device(device)
    if device.type != "cuda":
        raise SsdError("contracts_b200 needs a CUDA device, got %r (there is no CPU fallback)" % (device,))
    return device if device.index is not None else torch.device("cuda", torch.cuda.current_device())


def make_config(**kw):
    """ssd_config with abi_version / struct_size filled in."""
    return ssd_config(abi_version=SSD_ABI_VERSION, struct_size=ctypes.sizeof(ssd_config), **kw)


class ssd_solver_window(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_int32), ("num_samples", ctypes.c_int32), ("capacity", ctypes.c_int32),
                ("env_dev", ctypes.c_void_p), ("episode_dev", ctypes.c_void_p), ("count_dev", ctypes.c_void_p),
                ("params_dev", ctypes.c_void_p), ("rows_dev", ctypes.c_void_p)]


class ssd_selfdrive_io(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in ("actions_dev", "obs_dev", "rew_dev", "base_rew_dev", "transfers_dev",
                                               "info_dev", "done_dev")] + [("auto_reset", ctypes.c_int32)]


class ssd_feat_io(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in ("actions_dev", "obs_dev", "rew_dev", "base_rew_dev", "transfers_dev",
                                               "info_dev", "done_dev")] + [("auto_reset", ctypes.c_int32)]


EXPORTS = [
    "ssd_abi_version", "ssd_create", "ssd_destroy", "ssd_last_error", "ssd_reset", "ssd_step",
    "ssd_set_contract_params", "ssd_negotiate", "ssd_get_state", "ssd_set_state", "ssd_get_metrics",
    "ssd_random_actions", "ssd_philox4x32_10", "ssd_feature_dim", "ssd_state_bytes_per_env",
    "ssd_kernel_launches", "ssd_enable_timing", "ssd_get_step_times", "ssd_selfdrive_reset", "ssd_selfdrive_step", "ssd_selfdrive_get_state",
    "ssd_selfdrive_random_actions", "ssd_feat_reset", "ssd_feat_step", "ssd_feat_get_state", "ssd_feat_get_metrics",
    "ssd_global_view", "ssd_concat_obs", "ssd_solver_sample", "ssd_solver_choose", "ssd_policy_inputs", "ssd_record_beams", "ssd_render", "ssd_step_host",
    "ssd_step_host_async", "ssd_step_host_wait", "ssd_host_result_layout", "ssd_host_result_expand", "ssd_set_episode_stats",
    "ssd_feat_step_host_async", "ssd_selfdrive_step_host_async",
    "ssd_checkpoint_get_layout", "ssd_checkpoint_save", "ssd_checkpoint_load", "ssd_set_policy_output",
    "ssd_set_episode_log", "ssd_set_flat_policy_output", "ssd_set_feature_output", "ssd_set_global_output",
    "ssd_solver_enable", "ssd_solver_rows", "ssd_solver_resolve",
]

_LIB = None


def load():
    """Load the shared library (raises SsdError with build instructions if it is missing)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise SsdError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, u32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32
    L.ssd_abi_version.restype = i32
    L.ssd_create.argtypes = [ctypes.POINTER(ssd_config), ctypes.POINTER(vp)]
    L.ssd_destroy.argtypes = [vp]
    L.ssd_destroy.restype = None
    L.ssd_last_error.argtypes = [vp]
    L.ssd_last_error.restype = ctypes.c_char_p
    L.ssd_reset.argtypes = [vp, vp, vp, i64, vp]
    L.ssd_step.argtypes = [vp, ctypes.POINTER(ssd_step_io), vp]
    L.ssd_set_contract_params.argtypes = [vp, vp, vp]
    L.ssd_negotiate.argtypes = [vp, vp, vp, vp, vp, vp]
    L.ssd_step_host_async.argtypes = [vp, ctypes.POINTER(ssd_step_io), vp, vp, ctypes.POINTER(i64), vp]
    L.ssd_step_host_wait.argtypes = [vp, i64]
    L.ssd_feat_step_host_async.argtypes = [vp, ctypes.POINTER(ssd_feat_io), vp, vp, ctypes.POINTER(i64), vp]
    L.ssd_selfdrive_step_host_async.argtypes = [vp, ctypes.POINTER(ssd_selfdrive_io), vp, vp, ctypes.POINTER(i64), vp]
    L.ssd_host_result_layout.argtypes = [vp, ctypes.POINTER(ssd_host_layout)]
    L.ssd_host_result_expand.argtypes = [vp, vp, vp]
    L.ssd_set_episode_stats.argtypes = [vp, vp]
    L.ssd_set_episode_log.argtypes = [vp, ctypes.POINTER(ssd_episode_log)]
    L.ssd_get_state.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.ssd_set_state.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.ssd_get_metrics.argtypes = [vp, vp, vp]
    L.ssd_random_actions.argtypes = [vp, u32, i32, vp, vp]
    L.ssd_philox4x32_10.argtypes = [vp, vp, vp]
    L.ssd_philox4x32_10.restype = None
    L.ssd_selfdrive_reset.argtypes = [vp, vp, vp, vp]
    L.ssd_selfdrive_step.argtypes = [vp, ctypes.POINTER(ssd_selfdrive_io), vp]
    L.ssd_selfdrive_get_state.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.ssd_selfdrive_random_actions.argtypes = [vp, u32, ctypes.c_float, ctypes.c_float, vp, vp]
    L.ssd_feat_reset.argtypes = [vp, vp, vp, vp]
    L.ssd_feat_step.argtypes = [vp, ctypes.POINTER(ssd_feat_io), vp]
    L.ssd_feat_get_state.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.ssd_feat_get_metrics.argtypes = [vp, vp, vp]
    L.ssd_global_view.argtypes = [vp, vp, vp]
    L.ssd_concat_obs.argtypes = [vp, vp, i64, vp, vp]
    L.ssd_solver_sample.argtypes = [vp, i32, vp, vp]
    L.ssd_step_host.argtypes = [vp, ctypes.POINTER(ssd_step_io), vp, vp, vp, vp]
    L.ssd_record_beams.argtypes = [vp, i32]
    L.ssd_render.argtypes = [vp, vp, vp]
    L.ssd_policy_inputs.argtypes = [vp, vp, i64, i32, vp, vp, vp]
    L.ssd_set_policy_output.argtypes = [vp, ctypes.POINTER(ssd_policy_out)]
    L.ssd_set_flat_policy_output.argtypes = [vp, ctypes.POINTER(ssd_flat_policy_out)]
    L.ssd_set_feature_output.argtypes = [vp, ctypes.POINTER(ssd_feature_out)]
    L.ssd_set_global_output.argtypes = [vp, ctypes.POINTER(ssd_global_out)]
    L.ssd_solver_choose.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp]
    L.ssd_solver_enable.argtypes = [vp, i32]
    L.ssd_solver_rows.argtypes = [vp, ctypes.POINTER(ssd_solver_window), vp, vp]
    L.ssd_solver_resolve.argtypes = [vp, ctypes.POINTER(ssd_solver_window), i32, vp, vp, vp, vp, vp]
    L.ssd_feature_dim.argtypes = [vp]
    L.ssd_state_bytes_per_env.argtypes = [vp]
    L.ssd_state_bytes_per_env.restype = i64
    L.ssd_kernel_launches.argtypes = [vp]
    L.ssd_kernel_launches.restype = i64
    L.ssd_enable_timing.argtypes = [vp, ctypes.c_int32]
    L.ssd_get_step_times.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
    L.ssd_checkpoint_get_layout.argtypes = [vp, ctypes.POINTER(ssd_checkpoint_layout)]
    L.ssd_checkpoint_save.argtypes = [vp, vp, i32, vp, vp]
    L.ssd_checkpoint_load.argtypes = [vp, ctypes.c_uint64, vp, i32, vp, vp, vp]
    if L.ssd_abi_version() != SSD_ABI_VERSION:
        raise SsdError("libssd_b200.so ABI %d != binding ABI %d" % (L.ssd_abi_version(), SSD_ABI_VERSION))
    _LIB = L
    return L


def check(handle, rc):
    if rc != 0:
        msg = load().ssd_last_error(handle)
        raise SsdError("libssd_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))
