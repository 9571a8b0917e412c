"""ctypes binding of libmerlin_b200.so (the C ABI in include/merlin_b200.h).

The library is the product: there is no Python or CPU fallback.  If it has not been built, loading fails
with an explicit message; if no CUDA device is present, every entry point returns MERLIN_ECUDA and the
host layer raises RuntimeError.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("MERLIN_B200_LIB") or os.path.join(_PKG_ROOT, "lib", "libmerlin_b200.so")

OK, EINVAL, ECUDA, ESTATE, ENOMEM = 0, -1, -2, -3, -4
F_AUTO_RESET, F_RESET_SAME, F_SEVEN_ACTIONS, F_STUCK_PENALTY, F_EXPLORE_BONUS = 0x1, 0x2, 0x4, 0x8, 0x10

EXPORTS = (
    "merlin_env_default_config", "merlin_env_create", "merlin_env_destroy", "merlin_env_upload_layouts",
    "merlin_env_generate_layouts", "merlin_env_generate_seeded_layouts", "merlin_env_read_layouts",
    "merlin_env_layout_count", "merlin_env_set_tile_atlas", "merlin_env_set_cursors", "merlin_env_reset", "merlin_env_step",
    "merlin_env_state_ptrs", "merlin_env_read_state", "merlin_env_bad_actions", "merlin_env_launch_count",
    "merlin_set_kernel_choice", "merlin_set_observation_path", "merlin_env_step_kernel", "merlin_env_render", "merlin_env_render_f32", "merlin_env_full_obs", "merlin_gae",
    "merlin_pack_cell", "merlin_last_error", "merlin_version",
    "merlin_env_policy_step", "merlin_env_seed_sampler", "merlin_env_rearm", "merlin_env_set_kernel_choice",
    "merlin_env_set_observation_path", "merlin_env_write_state", "merlin_env_step_final",
    "merlin_env_policy_step_final", "merlin_env_final_step_kernel",
)


class EnvConfig(C.Structure):
    _fields_ = [
        ("device", C.c_int32), ("n_envs", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
        ("max_steps", C.c_int32), ("view", C.c_int32), ("tile", C.c_int32), ("flags", C.c_uint32),
        ("stuck_max_stay", C.c_int32), ("stuck_penalty", C.c_double), ("explore_bonus", C.c_double),
    ]


class StepExtras(C.Structure):
    _fields_ = [("episode_return", C.c_void_p), ("episode_length", C.c_void_p), ("stuck", C.c_void_p),
                ("done", C.c_void_p)]


class PolicyIO(C.Structure):
    """merlin_policy_io_t: device pointers of one fused act -> sample -> step -> store transition."""
    _fields_ = [("logits", C.c_void_p), ("value", C.c_void_p), ("action", C.c_void_p), ("logprob", C.c_void_p),
                ("value_out", C.c_void_p), ("greedy", C.c_int32), ("logits_stride", C.c_int32),
                ("value_stride", C.c_int32), ("finished", C.c_void_p),
                ("first_return", C.c_void_p), ("first_length", C.c_void_p), ("first_goal", C.c_void_p)]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build the CUDA library first (python -c 'import __graft_entry__ as g; g.build()' "
            "or make -C ppo-2dgrid_b200/csrc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.merlin_env_default_config.argtypes = [C.POINTER(EnvConfig)]
    lib.merlin_env_default_config.restype = None
    lib.merlin_env_create.argtypes = [C.POINTER(EnvConfig), C.POINTER(vp)]
    lib.merlin_env_destroy.argtypes = [vp]
    lib.merlin_env_upload_layouts.argtypes = [vp, vp, vp, i32]
    lib.merlin_env_generate_layouts.argtypes = [vp, i32, C.c_uint64, i64, i32, vp]
    lib.merlin_env_generate_seeded_layouts.argtypes = [vp, i32, vp, i32, vp]
    lib.merlin_env_read_layouts.argtypes = [vp, vp, vp]
    lib.merlin_env_layout_count.argtypes = [vp]
    lib.merlin_env_set_tile_atlas.argtypes = [vp, vp, i32]
    lib.merlin_env_set_cursors.argtypes = [vp, vp]
    lib.merlin_env_reset.argtypes = [vp, vp, vp, vp, vp]
    lib.merlin_env_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.POINTER(StepExtras), vp]
    lib.merlin_env_policy_step.argtypes = [vp, C.POINTER(PolicyIO), vp, vp, vp, vp, vp, C.POINTER(StepExtras), vp]
    lib.merlin_env_step_final.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.POINTER(StepExtras), vp, vp]
    lib.merlin_env_policy_step_final.argtypes = [vp, C.POINTER(PolicyIO), vp, vp, vp, vp, vp, C.POINTER(StepExtras),
                                                 vp, vp]
    lib.merlin_env_seed_sampler.argtypes = [vp, C.c_uint64]
    lib.merlin_env_rearm.argtypes = [vp, vp]
    lib.merlin_env_set_kernel_choice.argtypes = [vp, C.c_int]
    lib.merlin_env_set_observation_path.argtypes = [vp, C.c_int]
    lib.merlin_env_state_ptrs.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(i32), C.POINTER(vp)]
    lib.merlin_env_read_state.argtypes = [vp, vp, vp, vp]
    lib.merlin_env_write_state.argtypes = [vp, vp, vp, vp]
    lib.merlin_env_write_state.restype = C.c_int
    lib.merlin_env_bad_actions.argtypes = [vp, C.POINTER(C.c_uint64)]
    lib.merlin_env_launch_count.argtypes = [vp]
    lib.merlin_env_launch_count.restype = i64
    lib.merlin_set_kernel_choice.argtypes = [C.c_int]
    lib.merlin_set_kernel_choice.restype = C.c_int
    lib.merlin_set_observation_path.argtypes = [C.c_int]
    lib.merlin_set_observation_path.restype = C.c_int
    lib.merlin_env_full_obs.argtypes = [vp, vp, vp]
    lib.merlin_env_full_obs.restype = C.c_int
    lib.merlin_env_render.argtypes = [vp, vp, i64, vp, i32, vp, i32, vp]
    lib.merlin_env_render.restype = C.c_int
    lib.merlin_env_render_f32.argtypes = [vp, vp, i64, vp, i32, vp, i32, vp]
    lib.merlin_env_render_f32.restype = C.c_int
    lib.merlin_env_step_kernel.argtypes = [vp, C.c_int]
    lib.merlin_env_step_kernel.restype = C.c_char_p
    lib.merlin_env_final_step_kernel.argtypes = [vp, C.c_int]
    lib.merlin_env_final_step_kernel.restype = C.c_char_p
    lib.merlin_gae.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, C.c_double, C.c_double, vp]
    lib.merlin_pack_cell.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.merlin_pack_cell.restype = C.c_uint8
    lib.merlin_last_error.restype = C.c_char_p
    lib.merlin_version.restype = C.c_char_p
    for name in ("merlin_env_create", "merlin_env_destroy", "merlin_env_upload_layouts", "merlin_env_set_tile_atlas",
                 "merlin_env_generate_layouts", "merlin_env_generate_seeded_layouts", "merlin_env_read_layouts", "merlin_env_layout_count",
                 "merlin_env_set_cursors", "merlin_env_reset", "merlin_env_step", "merlin_env_state_ptrs",
                 "merlin_env_read_state", "merlin_env_bad_actions", "merlin_gae", "merlin_env_policy_step",
                 "merlin_env_seed_sampler", "merlin_env_rearm", "merlin_env_set_kernel_choice",
                 "merlin_env_set_observation_path", "merlin_env_step_final", "merlin_env_policy_step_final"):
        getattr(lib, name).restype = C.c_int
    _lib = lib
    if os.environ.get("MERLIN_OBSERVATION_PATH"):
        check(lib.merlin_set_observation_path(int(os.environ["MERLIN_OBSERVATION_PATH"])))
    if os.environ.get("MERLIN_KERNEL_CHOICE"):
        check(lib.merlin_set_kernel_choice(int(os.environ["MERLIN_KERNEL_CHOICE"])))
    return lib


def set_kernel_choice(choice):
    """0 = automatic, 1 = group kernel, 2 = warp-per-env kernel, 3 = CTA-tile kernel, 4 = CTA-tile kernel with TMA frame
    stores, 5 = symbolic-only kernel, 6 = group kernel with in-order hand-out.  Process-wide DEFAULT for envs without a
    setting of their own (`BatchedMerlinEnv.set_kernel_choice`); identical results."""
    check(load().merlin_set_kernel_choice(int(choice)))


def set_observation_path(path):
    """0 = automatic (row-parallel gen_obs in the symbolic-only kernel), 1 = per-cell everywhere, 2 = row-parallel in
    every kernel that has it (symbolic-only, tile, ordered).  Process-wide; identical results."""
    check(load().merlin_set_observation_path(int(path)))


def check(rc):
    if rc == OK:
        return
    msg = load().merlin_last_error().decode("utf-8", "replace")
    if rc == EINVAL:
        raise ValueError(msg)
    if rc == ENOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)
