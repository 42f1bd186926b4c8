"""ctypes binding of the C ABI in include/pve_mcc.h (libpve_mcc.so, built in-tree by build.py).

There is no CPU fallback: if the CUDA library is missing or cannot be loaded this module raises.
"""
import ctypes as C
import os

import numpy as np

from .config import NLANE, OBS_W, PveConfig

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(CSRC_DIR, "libpve_mcc.so")
CUDA_BACKEND = "cuda-sm_100a"

HDR_DTYPE = np.dtype([
    ("tick", "<i4"), ("id_seq", "<i4"), ("passed_veh", "<i4"), ("overflow", "<i4"),
    ("passed_step_total", "<i8"), ("n_veh", "<i4"), ("n_ctrl", "<i4"),
    ("next_spawn", "<i4", (NLANE,)), ("veh_rec", "<u2", (NLANE,)), ("lane_n", "u1", (NLANE,)),
    ("head_lane", "i1", (NLANE,)), ("head_j", "u1", (NLANE,)), ("pad_", "u1", (4,))])
META_DTYPE = np.dtype([("uid", "<i4"), ("packed", "<u4")])
#: pve_agent_record: the per-agent scalars of one output row in 16 bytes
RECORD_DTYPE = np.dtype([("reward", "<f4"), ("uid", "<i4"), ("lane", "u1"), ("j", "u1"), ("status", "u1"), ("cpv", "u1"),
                         ("jerk_sum", "<f4")])
assert HDR_DTYPE.itemsize == 144 and META_DTYPE.itemsize == 8 and RECORD_DTYPE.itemsize == 16

F_CONTROL, F_FINISH, F_LOCK = 1, 2, 4
ST_DONE, ST_REMOVED, ST_FINISHED = 1, 2, 4
COUNTER_NAMES = ["agent_steps", "vehicle_steps", "env_steps", "spawned", "passed", "passed_step_total",
                 "passed_jerk_sum", "collided_agent_steps", "lock_events", "reward_sum", "reward_sq_sum",
                 "removed", "overflow", "q5_undefined", "reserved0", "reserved1"]


class PveStateView(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("hdr", "p", "v", "a", "jerk_sum", "meta", "row0")]


class PveOutputs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("agent_offset", "obs", "reward", "ids", "cpv", "status", "jerk_sum",
                 "env_collisions", "env_lock", "env_removed", "nbr_src", "packed", "row0_out", "prev_row0", "obs_src")]


class PvePoisson(C.Structure):
    """pve_poisson: the arrival stream of pve_reset_poisson"""
    _fields_ = [("seed", C.c_uint64), ("rate_veh_per_hour", C.c_double), ("min_headway", C.c_double), ("first_env", C.c_int64)]


class PveReplayView(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("state", "action", "reward", "next_state", "done")] + [("capacity", C.c_int64)]


class NativeError(RuntimeError):
    pass


def load_library(path=None):
    """Load libpve_mcc.so and declare the prototypes of every symbol in include/pve_mcc.h."""
    path = path or os.environ.get("PVE_MCC_LIBRARY") or LIB_PATH      # the env override is for A/B measurements of builds
    if not os.path.exists(path):
        raise NativeError(
            "CUDA extension %s is missing; build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback." % path)
    lib = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.pve_backend.restype = C.c_char_p
    lib.pve_config_bytes.restype = i32
    lib.pve_default_config.argtypes = [C.POINTER(PveConfig), i32, C.c_double]
    lib.pve_create.argtypes = [C.POINTER(PveConfig), i32, C.POINTER(vp)]
    lib.pve_destroy.argtypes = [vp]
    lib.pve_destroy.restype = None
    lib.pve_last_error.argtypes = [vp]
    lib.pve_last_error.restype = C.c_char_p
    lib.pve_reset.argtypes = [vp, vp, i32, i32, vp]
    lib.pve_reset_poisson.argtypes = [vp, C.POINTER(PvePoisson), i32, vp]
    lib.pve_reset_poisson_rates.argtypes = [vp, C.POINTER(PvePoisson), vp, i32, vp]
    lib.pve_set_intention_draws.argtypes = [vp, vp]
    lib.pve_step.argtypes = [vp, vp, C.POINTER(PveOutputs), vp]
    lib.pve_step_host.argtypes = [vp, vp, C.POINTER(PveOutputs), C.POINTER(PveOutputs), i32, vp]
    lib.pve_step_host_async.argtypes = [vp, vp, C.POINTER(PveOutputs), C.POINTER(PveOutputs), i32, vp]
    lib.pve_expand_obs_host.argtypes = [vp, i32, i32, i64, vp, vp, vp, vp]
    lib.pve_expand_obs_host.restype = i64
    lib.pve_expand_obs.argtypes = [vp, i32, i64, vp, vp, vp, vp, vp]
    lib.pve_host_wait.argtypes = [vp]
    lib.pve_host_wait.restype = i64
    lib.pve_next_agent_total.argtypes = [vp, vp]
    lib.pve_next_agent_total.restype = i64
    lib.pve_set_state.argtypes = [vp, C.POINTER(PveStateView), vp]
    lib.pve_get_state.argtypes = [vp, C.POINTER(PveStateView), vp]
    for name in ("pve_row0_dev", "pve_row0_prev_dev", "pve_meta_dev", "pve_hdr_dev", "pve_env_stats_dev"):
        getattr(lib, name).argtypes = [vp]
        getattr(lib, name).restype = vp
    lib.pve_smem_bytes.argtypes = [vp]
    lib.pve_smem_bytes.restype = i64
    lib.pve_threads.argtypes = [vp]
    lib.pve_launch_info.argtypes = [vp, C.POINTER(C.c_int32 * 8)]
    lib.pve_veh_cap.argtypes = [vp]
    lib.pve_agent_cap.argtypes = [vp]
    lib.pve_stats.argtypes = [vp, vp, vp]
    lib.pve_set_profiling.argtypes = [vp, i32]
    lib.pve_kernel_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.pve_actor_create.argtypes = [vp, i32, i32, C.POINTER(vp)]
    lib.pve_actor_destroy.argtypes = [vp]
    lib.pve_actor_destroy.restype = None
    lib.pve_actor_forward.argtypes = [vp, vp, i64, vp, vp]
    lib.pve_act.argtypes = [vp, vp, vp, C.c_float, vp, vp]
    lib.pve_rollout.argtypes = [vp, vp, i32, vp, C.c_float, vp, C.POINTER(PveOutputs), vp]
    lib.pve_actor_forward_n.argtypes = [vp, vp, i64, vp, i32, vp, vp]
    lib.pve_critic_create.argtypes = [vp, i32, i32, C.POINTER(vp)]
    lib.pve_critic_destroy.argtypes = [vp]
    lib.pve_critic_destroy.restype = None
    lib.pve_critic_forward.argtypes = [vp, vp, vp, i64, vp, vp, vp]
    lib.pve_nstep_create.argtypes = [i32, i32, i32, i64, i64, i32, C.POINTER(vp)]
    lib.pve_nstep_destroy.argtypes = [vp]
    lib.pve_nstep_destroy.restype = None
    lib.pve_nstep_push.argtypes = [vp, C.POINTER(PveOutputs), C.c_double, vp, vp, vp]
    lib.pve_nstep_push_scene.argtypes = [vp, vp, C.POINTER(PveOutputs), C.c_double, vp, vp, vp]
    lib.pve_nstep_create_factored.argtypes = [i32, i32, i32, i64, i64, i32, C.POINTER(vp)]
    lib.pve_nstep_push_factored.argtypes = [vp, C.POINTER(PveOutputs), C.c_double, vp, vp, vp]
    lib.pve_nstep_factored_slot.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    lib.pve_nstep_log_bytes.argtypes = [vp]
    lib.pve_nstep_log_bytes.restype = i64
    lib.pve_nstep_last_error.argtypes = [vp]
    lib.pve_nstep_last_error.restype = C.c_char_p
    lib.pve_nstep_set_profiling.argtypes = [vp, i32]
    lib.pve_nstep_fold_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.pve_nstep_reset.argtypes = [vp, vp]
    lib.pve_nstep_obs_slot.argtypes = [vp, C.POINTER(vp)]
    lib.pve_nstep_replay.argtypes = [vp, C.POINTER(PveReplayView)]
    lib.pve_nstep_counters.argtypes = [vp, C.POINTER(i64), vp]
    lib.pve_nstep_q_dev.argtypes = [vp]
    lib.pve_nstep_q_dev.restype = vp
    if lib.pve_config_bytes() != C.sizeof(PveConfig):
        raise NativeError("pve_config layout mismatch: library %d bytes, binding %d bytes"
                          % (lib.pve_config_bytes(), C.sizeof(PveConfig)))
    return lib


# -------------------------------------------------------------------------------------------
# friendly <-> packed state
# -------------------------------------------------------------------------------------------
def pack_state(st, B, cap):
    """Friendly flat state (dict of arrays, see ``empty_state``) -> device layout arrays."""
    hdr = np.zeros(B, HDR_DTYPE)
    hdr["tick"] = st["tick"]
    hdr["id_seq"] = st["id_seq"]
    hdr["passed_veh"] = st["passed_veh"]
    hdr["passed_step_total"] = st["passed_step_total"]
    hdr["veh_rec"] = st["veh_rec"]
    hdr["lane_n"] = st["lane_n"]
    hdr["head_lane"] = np.where(st["head_lane"] >= 0, st["head_lane"], -1)
    hdr["head_j"] = np.where(st["head_lane"] >= 0, st["head_j"], 0)
    hdr["next_spawn"] = 2**31 - 1          # recomputed on the device from veh_rec
    meta = np.zeros((B, cap), META_DTYPE)
    meta["uid"] = st["uid"]
    flags = st["flags"].astype(np.uint32) & 7
    lock_a = (st["lock_a"].astype(np.int32) + 1).astype(np.uint32) & 3
    intention = (st["intention"].astype(np.uint32) & 3) if "intention" in st else np.uint32(0)      # lane_num = 4 only
    meta["packed"] = (np.minimum(st["step"], 0xFFFF).astype(np.uint32)
                      | (np.minimum(st["collision"], 255).astype(np.uint32) << 16)
                      | ((flags | (lock_a << 3) | (intention << 5)) << 24))
    if "intention_re" in st:
        hdr["pad_"][:, 0] = np.asarray(st["intention_re"]) % 3
    out = {"hdr": hdr, "meta": meta,
           "row0": np.ascontiguousarray(st["row0"], dtype=np.float32)}
    for k in ("p", "v", "a", "jerk_sum"):
        out[k] = np.ascontiguousarray(st[k], dtype=np.float64)
    return out


def unpack_state(dev, B, cap):
    hdr, meta = dev["hdr"], dev["meta"]
    packed = meta["packed"]
    fl = packed >> 24
    st = {
        "tick": hdr["tick"].astype(np.int32), "lane_n": hdr["lane_n"].astype(np.int32),
        "veh_rec": hdr["veh_rec"].astype(np.int32),
        "head_lane": hdr["head_lane"].astype(np.int32),
        "head_j": np.where(hdr["head_lane"] >= 0, hdr["head_j"].astype(np.int32), -1),
        "id_seq": hdr["id_seq"].astype(np.int32), "passed_veh": hdr["passed_veh"].astype(np.int32),
        "passed_step_total": hdr["passed_step_total"].astype(np.int64),
        "overflow": hdr["overflow"].astype(np.int32), "n_veh": hdr["n_veh"].astype(np.int32),
        "n_ctrl": hdr["n_ctrl"].astype(np.int32), "next_spawn": hdr["next_spawn"].astype(np.int32),
        "p": dev["p"], "v": dev["v"], "a": dev["a"], "jerk_sum": dev["jerk_sum"],
        "collision": ((packed >> 16) & 0xFF).astype(np.int32), "step": (packed & 0xFFFF).astype(np.int32),
        "uid": meta["uid"].astype(np.int32),
        "seq_in_lane": np.full((B, cap), -1, np.int32),      # logging-only field, not kept on device
        "flags": (fl & 7).astype(np.uint8), "lock_a": (((fl >> 3) & 3).astype(np.int32) - 1).astype(np.int8),
        "intention": ((fl >> 5) & 3).astype(np.uint8),            # lane_num = 4: TIS:387; 0 on the 12-lane path
        "intention_re": hdr["pad_"][:, 0].astype(np.int32),       # lane_num = 4: intention_re % 3
        "row0": dev["row0"],
    }
    # zero the dead slots so that states compare equal
    live = np.arange(cap)[None, :] < st["n_veh"][:, None]
    for k in ("p", "v", "a", "jerk_sum", "collision", "step", "uid", "flags", "lock_a", "intention"):
        st[k] = np.where(live, st[k], 0).astype(st[k].dtype)
    st["row0"] = np.where(live[:, :, None], st["row0"], 0).astype(np.float32)
    return st


def empty_state(B, cap):
    z = lambda *s, dt=np.int32: np.zeros(s, dt)
    st = {"tick": z(B), "lane_n": z(B, NLANE), "veh_rec": z(B, NLANE), "head_lane": z(B, NLANE) - 1,
          "head_j": z(B, NLANE) - 1, "id_seq": z(B), "passed_veh": z(B), "passed_step_total": z(B, dt=np.int64),
          "p": z(B, cap, dt=np.float64), "v": z(B, cap, dt=np.float64), "a": z(B, cap, dt=np.float64),
          "jerk_sum": z(B, cap, dt=np.float64), "collision": z(B, cap), "step": z(B, cap),
          "seq_in_lane": z(B, cap), "uid": z(B, cap), "flags": z(B, cap, dt=np.uint8),
          "lock_a": z(B, cap, dt=np.int8), "row0": z(B, cap, OBS_W, dt=np.float32)}
    return st
