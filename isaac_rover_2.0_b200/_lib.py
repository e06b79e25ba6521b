"""ctypes binding of librover_b200.so (the C ABI declared in include/rover_b200.h).

There is no fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

import torch

from . import _build

_lib = None

SEM_TORCH_CUDA = 0
SEM_TORCH_CPU = 1
LAYER_INDEX_ONLY = 1          # RVB_LAYER_INDEX_ONLY, a `flags` bit of rvb_terrain_create
N_STATS = 16

p = C.c_void_p
i64 = C.c_int64
i32 = C.c_int32
f32 = C.c_float


class RewardParams(C.Structure):
    _fields_ = [("pos_reward", f32), ("heading_contraint_reward", f32), ("motion_contraint_reward", f32),
                ("goal_angle_reward", f32), ("boogie_contraint_reward", f32),
                ("max_episode_length", i32), ("curriculum_level", i32), ("num_envs_total", i64),
                ("sem", i32), ("reserved", i32)]


class Linear(C.Structure):
    """rvb_linear (include/rover_b200.h): one torch nn.Linear, borrowed device pointers."""
    _fields_ = [("weight", p), ("bias", p), ("in_features", i32), ("out_features", i32)]


ACTIVATIONS = {"leakyrelu": 0, "relu": 1, "elu": 2, "tanh": 3, "sigmoid": 4, "relu6": 5}   # rvb_activation


class StepIO(C.Structure):
    """rvb_step_io (include/rover_b200.h)."""
    _fields_ = [(n, p) for n in ("pos", "quat", "joints", "target", "lin_hist", "ang_hist", "progress", "euler", "heading",
                                 "obs")] + [("obs_ld", i64)] + \
               [(n, p) for n in ("dist", "wheel_dist", "body_dist", "rock_collision", "rew", "reset", "ex_pos_reward", "ex_collision",
                                 "ex_uprightness", "ex_heading", "ex_motion", "ex_goal_angle", "stats", "stats_scratch", "obs_h16")] + \
               [("obs_h16_ld", i64)]


_SIGNATURES = {
    "rvb_abi_version": (C.c_int, []),
    "rvb_last_error": (C.c_char_p, []),
    "rvb_terrain_create": (C.c_int, [C.POINTER(p), p, i64, i64, i64, i64, i64, i64, p, i64, p, i64, f32, f32, f32, C.c_int, C.c_int, p]),
    "rvb_terrain_destroy": (C.c_int, [p]),
    "rvb_terrain_bytes": (i64, [p]),
    "rvb_terrain_release_index": (C.c_int, [p]),
    "rvb_terrain_has_index": (C.c_int, [p]),
    "rvb_terrain_unbounded_triangles": (i64, [p]),
    "rvb_heightmap_raycast": (C.c_int, [p, p, p, p, p, i64, i64, p, p, p, p, p, p, i64, p, i64, C.c_int, p, p, C.c_int, p]),
    "rvb_cast_rays": (C.c_int, [p, p, p, i64, p, p, p, p, p]),
    "rvb_ray_distance": (C.c_int, [p, p, p, i64, p, p, p]),
    "rvb_rock_collision": (C.c_int, [p, p, p, p, p, p, i64, p, p, p, p, p, p]),
    "rvb_check_collision": (C.c_int, [p, p, i64, p, p]),
    "rvb_quat_to_euler": (C.c_int, [p, i64, p, p]),
    "rvb_ackermann": (C.c_int, [p, i64, p, i64, i64, p, p, p, p, C.c_int, p]),
    "rvb_history_push": (C.c_int, [p, i64, i64, p, i64, p]),
    "rvb_obs_proprio": (C.c_int, [p, p, p, p, p, i64, p, i64, p, C.c_int, p]),
    "rvb_obs_gather": (C.c_int, [p, i64, i64, p, i64, p, i64, i64, p]),
    "rvb_stats_scratch_len": (i64, [i64]),
    "rvb_reward_reset": (C.c_int, [C.POINTER(RewardParams)] + [p] * 11 + [i64] + [p] * 10 + [p]),
    "rvb_env_pre": (C.c_int, [p, p, i64, i64, p, p, p, p, p, C.c_int, p]),
    "rvb_env_post": (C.c_int, [p, p, C.POINTER(RewardParams), C.POINTER(StepIO), p, p, i64, p, p, i64, i64, p]),
    "rvb_timing_enable": (C.c_int, [C.c_int]),
    "rvb_timing_read": (C.c_int, [C.POINTER(f32), C.c_int]),
    "rvb_stone_validate": (C.c_int, [p, i64, i64, p, i64, f32, C.c_int, p, p, p, p]),
    "rvb_spawn_validate": (C.c_int, [p, i64, p, i64, i32, p, p]),
    "rvb_height_lookup": (C.c_int, [p, i64, i64, p, i64, i64, f32, f32, f32, f32, p, C.c_int, p]),
    "rvb_build_knn_index": (C.c_int, [p, i64, p, i64, p, p, i64, i64, i64, p, p]),
    "rvb_reset_targets": (C.c_int, [p, i64, i64, C.c_uint64, C.c_uint64, p, f32, p, i64, f32, i32, p, i64, i64, f32, f32, f32, f32,
                                    p, p, p, p, C.c_int, p]),
    "rvb_policy_create": (C.c_int, [C.POINTER(p), i32, i32, i32, C.POINTER(Linear), C.POINTER(Linear), C.POINTER(Linear),
                                    C.POINTER(Linear), i32, i32, C.c_int, p]),
    "rvb_policy_destroy": (C.c_int, [p]),
    "rvb_policy_bytes": (i64, [p]),
    "rvb_policy_forward": (C.c_int, [p, p, i64, i64, p, i64, p]),
    "rvb_policy_forward_pair": (C.c_int, [p, p, p, i64, i64, p, i64, p, i64, p]),
    "rvb_policy_forward_packed": (C.c_int, [p, p, p, i64, p, i64, i64, p, i64, p, i64, p]),
    "rvb_policy_variant": (C.c_int, [C.c_int]),
    "rvb_obs_hooks": (C.c_int, [p, i64, i64, i64, i64, f32, f32, f32, p, C.c_uint64, C.c_uint64, i64, p]),
    "rvb_teacher_record": (C.c_int, [p, p, i64, p, i64, i64, i64, p, i64, p]),
    "rvb_teacher_record_packed": (C.c_int, [p, p, i64, p, i64, i64, p, i64, i64, i64, p, i64, p, i64, p]),
}

EXPORTS = tuple(_SIGNATURES)


def lib_path():
    return _build.LIB


# kernels launched per entry point (for bench.py's `gpu_launches` claim)
KERNELS_PER_CALL = {"rvb_terrain_create": 2, "rvb_heightmap_raycast": 4, "rvb_cast_rays": 2, "rvb_ray_distance": 1,
                    "rvb_rock_collision": 1, "rvb_check_collision": 1, "rvb_quat_to_euler": 1, "rvb_ackermann": 1,
                    "rvb_history_push": 1, "rvb_obs_proprio": 1, "rvb_obs_gather": 1, "rvb_reward_reset": 2, "rvb_env_pre": 1,
                    "rvb_env_post": 8,
    "rvb_stone_validate": 1, "rvb_spawn_validate": 1, "rvb_height_lookup": 1, "rvb_build_knn_index": 6, "rvb_reset_targets": 1,
                    "rvb_policy_create": 7, "rvb_policy_forward": 1, "rvb_policy_forward_pair": 1,
                    "rvb_policy_forward_packed": 2,
                    "rvb_obs_hooks": 1, "rvb_teacher_record": 1, "rvb_teacher_record_packed": 1}
launch_count = 0


class _Counted:
    """Thin callable around a ctypes function that counts the kernels it launches."""
    __slots__ = ("fn", "n")

    def __init__(self, fn, n):
        self.fn, self.n = fn, n

    def __call__(self, *args):
        global launch_count
        launch_count += self.n
        return self.fn(*args)


class _Lib:
    pass


def load():
    """Load (building first if the sources are newer and nvcc is present).  Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_build.LIB) or (_build.needs_build() and os.environ.get("ROVER_B200_NO_REBUILD") != "1"):
        try:
            _build.build()
        except Exception as e:
            if not os.path.exists(_build.LIB):
                raise RuntimeError("librover_b200.so is missing and could not be built: %s" % e)
            if "nvcc failed" in str(e):             # the sources do not compile: never run yesterday's kernels in their place
                raise RuntimeError("librover_b200.so is stale and its sources do not compile: %s" % e)
            import warnings                         # no compiler on this box: a present library is still usable, but say so
            warnings.warn("librover_b200.so is older than its sources and could not be rebuilt (%s); using it as is" % e)
    # ROVER_B200_LIB: another build of the same ABI (same-box A/B of two builds; tools/shadow_quick.py)
    raw = C.CDLL(os.environ.get("ROVER_B200_LIB") or _build.LIB)
    lib = _Lib()
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(raw, name)                     # AttributeError here = ABI mismatch, fail loudly
        fn.restype = res
        fn.argtypes = args
        setattr(lib, name, _Counted(fn, KERNELS_PER_CALL[name]) if name in KERNELS_PER_CALL else fn)
    if lib.rvb_abi_version() != 5:
        raise RuntimeError("librover_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError("%s [status %d]" % (load().rvb_last_error().decode(), rc))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream_of(t):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("rover_b200: expected a CUDA tensor (there is no CPU path)")
