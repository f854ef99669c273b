"""ctypes binding of libsoccer2d.so - the C ABI declared in include/soccer2d.h.

This is the only place the Python host touches native code.  There is NO CPU fallback: if the shared
library is missing, or no CUDA device is usable, the caller gets an exception, never a silent slow path.
"""
from __future__ import annotations

import ctypes as C
import os

ABI_VERSION = 13
MAX_PIPELINE_SLOTS = 4

# ---- constants (mirror include/soccer2d.h) ----------------------------------------------------------
S2D_OK, S2D_ERR_INVALID, S2D_ERR_UNBOUND, S2D_ERR_CUDA, S2D_ERR_NO_DEVICE = 0, -1, -2, -3, -4
SCENARIO_REACHBALL, SCENARIO_SHOOT, SCENARIO_FULLGAME = 0, 1, 2
ACT_DISCRETE, ACT_CONTINUOUS, ACT_TURNING, ACT_COMMAND = 0, 1, 2, 3
CMD_NONE, CMD_DASH, CMD_TURN, CMD_KICK, CMD_GOTO = 0, 1, 2, 3, 4
CMD_TURN_TO_POINT, CMD_TURN_TO_BALL, CMD_TURN_TO_ANGLE, CMD_KICK_ONE_STEP, CMD_STOP_BALL, CMD_INTERCEPT = 5, 6, 7, 8, 9, 10
CMD_TACKLE, CMD_CATCH, CMD_SMART_KICK = 11, 12, 13
RESULT_NONE, RESULT_GOAL, RESULT_OUT, RESULT_TIMEOUT = 0, 1, 2, 3
RESULT_NAMES = (None, "Goal", "Out", "Timeout")  # info['result'], reach_ball_env.py:126,140,145,150
FLAG_BALL_COLLIDED, FLAG_PLAYER_COLLIDED, FLAG_KICKED, FLAG_DONE = 1, 2, 4, 8
COLLISION_MIDPOINT, COLLISION_BACKTRACE = 0, 1
COLLISION_MODELS = {"midpoint": COLLISION_MIDPOINT, "backtrace": COLLISION_BACKTRACE}

_SP_FIELDS = (
    "pitch_half_length pitch_half_width goal_width goal_post_radius "
    "ball_size ball_decay ball_rand ball_speed_max ball_accel_max "
    "player_size player_decay player_rand player_speed_max player_accel_max "
    "dash_power_rate inertia_moment "
    "min_dash_power max_dash_power min_dash_angle max_dash_angle dash_angle_step "
    "side_dash_rate back_dash_rate "
    "min_power max_power min_moment max_moment "
    "kick_power_rate kickable_margin kick_rand "
    "stamina_max stamina_inc_max extra_stamina stamina_capacity "
    "recover_init recover_min recover_dec recover_dec_thr "
    "effort_init effort_max effort_min effort_dec effort_dec_thr effort_inc effort_inc_thr "
    "slowness_on_top_for_left_team slowness_on_top_for_right_team"
).split()


class ServerParam(C.Structure):
    _fields_ = [(n, C.c_float) for n in _SP_FIELDS] + [("reserved", C.c_float * 5)]


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("scenario", C.c_int32),
        ("num_envs", C.c_int64), ("env_id_offset", C.c_int64), ("seed", C.c_uint64),
        ("device", C.c_int32), ("action_mode", C.c_int32), ("action_space_size", C.c_int32),
        ("max_steps", C.c_int32), ("auto_reset", C.c_int32),
        ("change_ball_position", C.c_int32), ("change_ball_velocity", C.c_int32), ("noise", C.c_int32),
        ("players_per_side", C.c_int32), ("half_time_cycles", C.c_int32),
        ("kick_actions", C.c_int32), ("collision_model", C.c_int32), ("reserved_i", C.c_int32 * 2),
        ("min_distance_to_ball", C.c_float),
        ("ball_position_x", C.c_float), ("ball_position_y", C.c_float),
        ("ball_speed", C.c_float), ("ball_direction", C.c_float),
        ("goto_dist_thr", C.c_float), ("reserved_f", C.c_float * 3),
        ("sp", ServerParam),
    ]


class Buffers(C.Structure):
    _fields_ = [
        ("state", C.c_void_p), ("actions", C.c_void_p), ("obs", C.c_void_p), ("reward", C.c_void_p),
        ("done", C.c_void_p), ("result", C.c_void_p), ("terminal_obs", C.c_void_p), ("stats", C.c_void_p),
    ]


class OutputLayout(C.Structure):
    """S2DOutputLayout: byte offsets of obs | reward | done | result (| terminal_obs) inside one output block"""
    _fields_ = [(n, C.c_size_t) for n in
                "obs reward done result step_bytes terminal_obs bytes bytes_with_terminal_obs".split()]


class Stats(C.Structure):
    _fields_ = [
        ("episodes", C.c_uint64), ("goals", C.c_uint64), ("outs", C.c_uint64), ("timeouts", C.c_uint64),
        ("episode_steps", C.c_uint64), ("env_steps", C.c_uint64), ("return_sum", C.c_double), ("reserved", C.c_double),
    ]


class PlayerSnapshot(C.Structure):
    _fields_ = [(n, C.c_float) for n in
                "x y vx vy body_direction stamina effort recovery stamina_capacity".split()] + \
               [(n, C.c_int32) for n in "side uniform_number collided kicked".split()]


class EnvSnapshot(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                "cycle stoped_cycle game_mode_type game_mode_side step_number episode left_score right_score".split()] + \
               [(n, C.c_float) for n in
                "ball_x ball_y ball_vx ball_vy mem_distance_to_ball mem_body_ball_angle_diff episode_return".split()] + \
               [(n, C.c_int32) for n in "ball_collided num_players flags".split()] + \
               [("players", PlayerSnapshot * 22)]


MAX_PLAYER_TYPES = 18
_PT_FIELDS = ("player_decay inertia_moment dash_power_rate stamina_inc_max kickable_margin kick_rand extra_stamina "
              "effort_max effort_min kick_power_rate").split()


class PlayerType(C.Structure):
    """proto PlayerType (idl/service.proto:1697-1732): the fields the cycle reads"""
    _fields_ = [(n, C.c_float) for n in _PT_FIELDS] + [("reserved", C.c_float * 6)]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n in _PT_FIELDS}


class MlpPolicy(C.Structure):
    """S2DMlpPolicy: device pointers to a 64-64 Q-network in torch nn.Linear layout"""
    _fields_ = [("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p), ("w3", C.c_void_p),
                ("b3", C.c_void_p), ("hidden", C.c_int32), ("precision", C.c_int32)]


class Trajectory(C.Structure):
    """S2DTrajectory: optional time-major device buffers for the transitions of a fused rollout"""
    _fields_ = [("obs", C.c_void_p), ("actions", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
                ("actions_f", C.c_void_p)]


# every symbol include/soccer2d.h declares: (restype, argtypes)
_H = C.c_void_p
SIGNATURES = {
    "s2d_abi_version": (C.c_int, []),
    "s2d_error_string": (C.c_char_p, [C.c_int]),
    "s2d_last_error": (C.c_char_p, [_H]),
    "s2d_default_server_param": (C.c_int, [C.POINTER(ServerParam)]),
    "s2d_default_config": (C.c_int, [C.POINTER(Config), C.c_int]),
    "s2d_state_bytes": (C.c_size_t, [C.POINTER(Config)]),
    "s2d_action_bytes": (C.c_size_t, [C.POINTER(Config)]),
    "s2d_stats_bytes": (C.c_size_t, [C.POINTER(Config)]),
    "s2d_obs_dim": (C.c_int, [C.POINTER(Config)]),
    "s2d_num_players": (C.c_int, [C.POINTER(Config)]),
    "s2d_create": (C.c_int, [C.POINTER(Config), C.POINTER(_H)]),
    "s2d_destroy": (C.c_int, [_H]),
    "s2d_bind": (C.c_int, [_H, C.POINTER(Buffers)]),
    "s2d_reset": (C.c_int, [_H, C.c_void_p, C.c_void_p]),
    "s2d_step": (C.c_int, [_H, C.c_int, C.c_void_p]),
    "s2d_step_host": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "s2d_bind_pipeline": (C.c_int, [_H, C.POINTER(Buffers)]),
    "s2d_bind_pipeline_slot": (C.c_int, [_H, C.c_int, C.POINTER(Buffers)]),
    "s2d_output_layout": (C.c_int, [C.POINTER(Config), C.POINTER(OutputLayout)]),
    "s2d_fence": (C.c_int, [_H, C.c_void_p]),
    "s2d_clear": (C.c_int, [_H, C.c_void_p]),
    "s2d_submit_host": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "s2d_wait_host": (C.c_int, [_H, C.c_int]),
    "s2d_stats": (C.c_int, [_H, C.POINTER(Stats), C.c_void_p]),
    "s2d_stats_reset": (C.c_int, [_H, C.c_void_p]),
    "s2d_env_steps": (C.c_int, [_H, C.POINTER(C.c_uint64)]),
    "s2d_export_env": (C.c_int, [_H, C.c_int64, C.POINTER(EnvSnapshot), C.c_void_p]),
    "s2d_pipeline_info": (C.c_int, [_H, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "s2d_launch_info": (C.c_int, [_H, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "s2d_generate_player_types": (C.c_int, [C.c_uint64, C.POINTER(ServerParam), C.POINTER(PlayerType), C.c_int]),
    "s2d_set_player_types": (C.c_int, [_H, C.POINTER(PlayerType), C.c_int, C.POINTER(C.c_uint8)]),
    "s2d_set_player_types_per_match": (C.c_int, [_H, C.POINTER(PlayerType), C.c_int, C.POINTER(C.c_uint8)]),
    "s2d_set_scripted_players": (C.c_int, [_H, C.c_uint32]),
    "s2d_rollout_mlp": (C.c_int, [_H, C.POINTER(MlpPolicy), C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "s2d_rollout_mlp_collect": (C.c_int, [_H, C.POINTER(MlpPolicy), C.c_int, C.c_float, C.POINTER(Trajectory), C.c_void_p]),
    "s2d_rollout_actor_collect": (C.c_int, [_H, C.POINTER(MlpPolicy), C.c_int, C.c_float, C.POINTER(Trajectory), C.c_void_p]),
}

# S2D_LIB: alternative build of the same library (kernel tuning experiments); default = the in-tree build
LIB_PATH = os.environ.get("S2D_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libsoccer2d.so")


class Soccer2DError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libsoccer2d error {code}: {message}")
        self.code = code


_lib = None


def load():
    """dlopen libsoccer2d.so (built by `__graft_entry__.build()` / csrc/Makefile) and type its entry points."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  soccer2d_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = the library does not export what the header declares
        fn.restype, fn.argtypes = res, args
    got = lib.s2d_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"libsoccer2d ABI version {got}, python host expects {ABI_VERSION}: rebuild the library")
    _lib = lib
    return lib


def check(rc: int, handle=None):
    if rc == S2D_OK:
        return
    lib = load()
    msg = lib.s2d_last_error(handle) or b""
    text = msg.decode("utf-8", "replace") or lib.s2d_error_string(rc).decode()
    raise Soccer2DError(rc, text)
