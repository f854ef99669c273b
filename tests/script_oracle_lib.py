"""ctypes access to the CPU oracle with FULLGAME's scripted players (tests/script_oracle: oracle/s2d_oracle.c plus the
script's rules -> tests/script_oracle/_build/libscript_oracle_{f64,f32}.so).  Test-side only."""
import ctypes as C
import glob
import os
import subprocess

import numpy as np

import oracle_lib as OL

HERE = os.path.dirname(os.path.abspath(__file__))
SCRIPT_DIR = os.path.join(HERE, "script_oracle")

_libs = {}
_V, _I64, _D = C.c_void_p, C.c_int64, C.c_double
# what this library exports and OracleSim calls (oracle/s2d_oracle.c's s2do_* entry points, plus the script's own)
_SIGNATURES = {
    "s2do_is_f32": (C.c_int, []),
    "s2do_create": (C.c_int, [_V, C.POINTER(_V)]),
    "s2do_destroy": (None, [_V]),
    "s2do_obs_dim": (C.c_int, [_V]),
    "s2do_reset": (None, [_V, _V]),
    "s2do_reset_masked": (None, [_V, _V, _V]),
    "s2do_step": (None, [_V, _V, C.c_int] + [_V] * 5),
    "s2do_stats": (None, [_V, _V]),
    "s2do_get_state_fg": (C.c_int, [_V, _I64, _V]),
    "s2do_set_state_fg": (None, [_V, _I64, _V]),
    "s2do_get_extra_fg": (C.c_int, [_V, _I64, _V]),
    "s2do_set_extra_fg": (None, [_V, _I64, _V]),
    "s2do_set_player_types": (C.c_int, [_V, _V, C.c_int, _V]),
    "s2do_set_player_types_per_match": (C.c_int, [_V, _V, C.c_int, _V]),
    "s2dos_step": (None, [_V, C.c_uint32, _V, C.c_int] + [_V] * 5),
    "s2dos_script_commands": (None, [_V, C.c_uint32, _V]),
}


def lib(kind: str):
    """the script oracle of one build (it carries the oracle's s2do_* entry points as well)"""
    if kind not in _libs:
        path = os.path.join(SCRIPT_DIR, "_build", f"libscript_oracle_{kind}.so")
        srcs = glob.glob(os.path.join(SCRIPT_DIR, "*.c")) + [os.path.join(OL.ORACLE_DIR, "s2d_oracle.c"),
                                                             os.path.join(OL.ROOT, "include", "soccer2d.h")]
        if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(s) for s in srcs):
            subprocess.run(["make", "-s", "-C", SCRIPT_DIR], check=True, capture_output=True)
        L = C.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _libs[kind] = L
    return _libs[kind]


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def team_mask(np_players, who):
    """"left" / "right" / "all" / an iterable of player indices -> the bit mask"""
    pps = np_players // 2
    if who == "left":
        return (1 << pps) - 1
    if who == "right":
        return ((1 << np_players) - 1) & ~((1 << pps) - 1)
    if who == "all":
        return (1 << np_players) - 1
    m = 0
    for j in who:
        m |= 1 << int(j)
    return m


class ScriptedOracleSim(OL.OracleSim):
    """OracleSim whose step plays the players of `mask` by the built-in script (mask 0: exactly OracleSim.step).  The
    state accessors, statistics and player types are OracleSim's, called on this library."""

    def __init__(self, cfg, kind="f64", mask=0):
        self.L = lib(kind)
        self.kind = kind
        self.real = np.float64 if kind == "f64" else np.float32
        assert self.L.s2do_is_f32() == (kind == "f32")
        self.cfg = cfg
        self.n = int(cfg.num_envs)
        self.h = C.c_void_p()
        if self.L.s2do_create(C.byref(cfg), C.byref(self.h)) != 0:
            raise ValueError("oracle rejected the config")
        self.obs_dim = int(self.L.s2do_obs_dim(self.h))
        self.obs = np.zeros((self.n, self.obs_dim), self.real)
        self.term_obs = np.zeros((self.n, self.obs_dim), self.real)
        self.reward = np.zeros(self.n, self.real)
        self.done = np.zeros(self.n, np.uint8)
        self.result = np.zeros(self.n, np.uint8)
        self.mask = int(mask)

    def set_scripted(self, mask):
        self.mask = int(mask)

    def step(self, actions, k=1):
        a = np.ascontiguousarray(actions, dtype=np.float32)
        self.L.s2dos_step(self.h, self.mask, _ptr(a), int(k), _ptr(self.obs), _ptr(self.reward), _ptr(self.done),
                          _ptr(self.result), _ptr(self.term_obs))
        return self.obs, self.reward, self.done, self.result

    def script_commands(self, mask=None):
        """[N, np, 4] float32: what the script would command the players of `mask` (default: the sim's) this cycle (others 0)"""
        np_ = 2 * int(self.cfg.players_per_side)
        rows = np.zeros((self.n, np_, 4), np.float32)
        self.L.s2dos_script_commands(self.h, self.mask if mask is None else int(mask), _ptr(rows))
        return rows
