"""Test-side tools for SHOOT's parameterized actions (S2D_ACT_PARAMETERIZED, include/soccer2d.h): the C oracle
(tests/param_oracle: oracle/s2d_oracle.c plus the translation of the rows), the kernel source on the host (tests/param_emu:
tests/emu plus step_kernel's translation), a Python restatement of the translation for the Python oracle, and row
generators.  Test-side only."""
import ctypes as C
import glob
import math
import os
import subprocess

import numpy as np

import emu_lib as EL
import helpers as H
import oracle_lib as OL
from oracle import soccer2d_oracle as O
from soccer2d_b200 import _abi

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(HERE, "param_oracle")
EMU_DIR = os.path.join(HERE, "param_emu")
_V = C.c_void_p


def _build(directory, path, srcs):
    if not os.path.exists(path) or os.path.getmtime(path) < max(os.path.getmtime(s) for s in srcs):
        subprocess.run(["make", "-s", "-C", directory], check=True, capture_output=True)


# ---- rows -------------------------------------------------------------------------------------------------------------

def config(num_envs, **kw):
    """S2DConfig of SHOOT with parameterized actions (helpers.make_config's overrides)"""
    return H.make_config(num_envs, _abi.ACT_PARAMETERIZED, scenario=_abi.SCENARIO_SHOOT, **kw)


def command_config(num_envs, **kw):
    return H.make_config(num_envs, "command", scenario=_abi.SCENARIO_SHOOT, **kw)


def random_rows(rng, n, k=1):
    """[n, k, 8] float32 parameterized rows: values beyond [-1, 1], exact ties between the weights, the bounds -1 / +1
    and NaN now and then (the clamps and the tie rule are part of the contract)"""
    a = rng.uniform(-1.3, 1.3, size=(n, k, 8)).astype(np.float32)
    pick = rng.uniform(size=(n, k, 8))
    a = np.where(pick < 0.05, np.float32(1.0), a)
    a = np.where((pick >= 0.05) & (pick < 0.1), np.float32(-1.0), a)
    a = np.where((pick >= 0.1) & (pick < 0.12), np.float32(np.nan), a)
    tie = rng.uniform(size=(n, k)) < 0.1  # two or three equal weights
    a[..., 1] = np.where(tie, a[..., 0], a[..., 1])
    a[..., 2] = np.where(tie & (rng.uniform(size=(n, k)) < 0.5), a[..., 0], a[..., 2])
    return a


def to_command(a):
    """the S2D_ACT_COMMAND rows [.., 4] float32 that parameterized rows [.., 8] stand for, in float32 numpy (one rounding
    per operation, as the header specifies)"""
    a = np.asarray(a, np.float32)
    c = np.fmax(np.float32(-1), np.fmin(a, np.float32(1)))  # fmin / fmax: a NaN becomes +1
    dash = (c[..., 0] >= c[..., 1]) & (c[..., 0] >= c[..., 2])
    turn = ~dash & (c[..., 1] >= c[..., 2])
    one, fifty, deg = np.float32(1), np.float32(50), np.float32(180)
    out = np.zeros(a.shape[:-1] + (4,), np.float32)
    out[..., 0] = np.where(dash, 1, np.where(turn, 2, 3))
    out[..., 1] = np.where(dash, (c[..., 3] + one) * fifty, np.where(turn, c[..., 5] * deg, (c[..., 6] + one) * fifty))
    out[..., 2] = np.where(dash, c[..., 4] * deg, np.where(turn, np.float32(0), c[..., 7] * deg))
    return out


def to_command_f64(row):
    """one row -> (cmd, a, b, c): the translation in double, each argument rounded to float where it enters the command
    row (what the f64 oracle does); the Python oracle's restatement"""
    c = [1.0 if math.isnan(float(v)) else O.clamp(-1.0, float(v), 1.0) for v in row]
    if c[0] >= c[1] and c[0] >= c[2]:
        return O.CMD_DASH, O.f32((c[3] + 1.0) * 50.0), O.f32(c[4] * 180.0), 0.0
    if c[1] >= c[2]:
        return O.CMD_TURN, O.f32(c[5] * 180.0), 0.0, 0.0
    return O.CMD_KICK, O.f32((c[6] + 1.0) * 50.0), O.f32(c[7] * 180.0), 0.0


def chase_and_shoot(obs, rng, k=1, random_share=0.2):
    """helpers.chase_and_shoot in the parameterized space: Dash(100, towards the ball) while far, Kick(100, towards the
    goal centre) within 1 m; every row is replaced by a random_rows one with probability random_share.  [n, k, 8] float32
    (the same row for all k cycles)."""
    c = H.chase_and_shoot(obs)[:, 0]  # {3, 100, goal direction, 0} near the ball, else {4, bx, by, 100}
    obs = np.asarray(obs, np.float64)
    n = obs.shape[0]
    a = np.full((n, 8), -1.0, np.float32)
    near = c[:, 0] == 3
    a[:, 0] = np.where(near, -1.0, 1.0)
    a[:, 2] = np.where(near, 1.0, -1.0)
    a[:, 3] = 1.0
    a[:, 4] = np.clip(obs[:, 0], -1, 1)  # body-to-ball angle / 180
    a[:, 6] = 1.0
    a[:, 7] = np.where(near, c[:, 2] / 180.0, 0.0)
    a = np.repeat(a[:, None, :], k, axis=1)
    return np.where(rng.uniform(size=(n, k, 1)) < random_share, random_rows(rng, n, k), a).astype(np.float32)


# ---- the C oracle ------------------------------------------------------------------------------------------------------

_oracles = {}


def oracle_lib(kind: str):
    if kind not in _oracles:
        path = os.path.join(ORACLE_DIR, "build", f"libparam_oracle_{kind}.so")
        _build(ORACLE_DIR, path, glob.glob(os.path.join(ORACLE_DIR, "*.c")) +
               [os.path.join(OL.ORACLE_DIR, "s2d_oracle.c"), os.path.join(OL.ROOT, "include", "soccer2d.h")])
        L = C.CDLL(path)
        for name, (res, args) in {
                "s2do_is_f32": (C.c_int, []), "s2dop_create": (C.c_int, [_V, C.POINTER(_V)]),
                "s2do_destroy": (None, [_V]), "s2do_obs_dim": (C.c_int, [_V]), "s2do_reset": (None, [_V, _V]),
                "s2do_reset_masked": (None, [_V, _V, _V]), "s2dop_step": (None, [_V, _V, C.c_int] + [_V] * 5),
                "s2dop_translate": (None, [_V, C.c_int64, _V]), "s2do_stats": (None, [_V, _V]),
                "s2do_get_state": (None, [_V, C.c_int64, _V]), "s2do_set_state": (None, [_V, C.c_int64, _V])}.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _oracles[kind] = L
    return _oracles[kind]


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class ParamOracleSim(OL.OracleSim):
    """OracleSim for SHOOT + S2D_ACT_PARAMETERIZED: `step` takes [N, K, 8] rows.  Reset, state and statistics are
    OracleSim's, called on this library."""

    def __init__(self, cfg, kind="f64"):
        self.L = oracle_lib(kind)
        self.kind = kind
        self.real = np.float64 if kind == "f64" else np.float32
        assert self.L.s2do_is_f32() == (kind == "f32")
        self.cfg = cfg
        self.n = int(cfg.num_envs)
        self.h = C.c_void_p()
        if self.L.s2dop_create(C.byref(cfg), C.byref(self.h)) != 0:
            raise ValueError("oracle rejected the config")
        self.obs_dim = int(self.L.s2do_obs_dim(self.h))
        self.obs = np.zeros((self.n, self.obs_dim), self.real)
        self.term_obs = np.zeros((self.n, self.obs_dim), self.real)
        self.reward = np.zeros(self.n, self.real)
        self.done = np.zeros(self.n, np.uint8)
        self.result = np.zeros(self.n, np.uint8)

    def step(self, actions, k=1):
        a = np.ascontiguousarray(actions, dtype=np.float32)
        self.L.s2dop_step(self.h, _ptr(a), int(k), _ptr(self.obs), _ptr(self.reward), _ptr(self.done),
                          _ptr(self.result), _ptr(self.term_obs))
        return self.obs, self.reward, self.done, self.result

    def translate(self, actions):
        """the command rows this build's translation makes of `actions` [.., 8]"""
        a = np.ascontiguousarray(actions, dtype=np.float32)
        out = np.zeros(a.shape[:-1] + (4,), np.float32)
        self.L.s2dop_translate(_ptr(a), a.size // 8, _ptr(out))
        return out


class ParamShootOracle(O.ShootOracle):
    """the Python oracle's Shoot episode stream, fed parameterized rows through to_command_f64"""

    def step(self, action):
        return super().step(to_command_f64(action))


# ---- the kernel source on the host -------------------------------------------------------------------------------------

_emu = None


def emu_lib():
    global _emu
    if _emu is None:
        path = os.path.join(EMU_DIR, "build", "libemu_shoot_param.so")
        _build(EMU_DIR, path, glob.glob(os.path.join(HERE, "..", "gym-soccer-2d-env_b200", "csrc", "*.cuh")) +
               glob.glob(os.path.join(EMU_DIR, "*.cpp")) + glob.glob(os.path.join(EL.EMU_DIR, "*.cpp")) +
               glob.glob(os.path.join(EL.EMU_DIR, "*.h")))
        L = C.CDLL(path)
        L.emu_create.restype = C.c_void_p
        L.emu_create.argtypes = [C.c_void_p]
        L.emu_destroy.argtypes = [C.c_void_p]
        L.emu_state.restype = C.c_void_p
        L.emu_state.argtypes = [C.c_void_p]
        L.emu_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.emu_step_param.argtypes = [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 6
        L.emu_uses_default_sp.argtypes = [C.c_void_p]
        _emu = L
    return _emu


class ParamEmuSim(EL.EmuSim):
    """EmuSim whose step takes [N, K, 8] parameterized rows through the kernels' translation"""

    def __init__(self, cfg):
        self.L = emu_lib()
        self.n = int(cfg.num_envs)
        self.h = self.L.emu_create(C.byref(cfg))
        self.obs = np.zeros((self.n, 10), np.float32)
        self.term_obs = np.zeros((self.n, 10), np.float32)
        self.reward = np.zeros(self.n, np.float32)
        self.done = np.zeros(self.n, np.uint8)
        self.result = np.zeros(self.n, np.uint8)
        self.stats6 = np.zeros(6, np.float64)

    def step(self, actions, k=1):
        a = np.ascontiguousarray(actions, dtype=np.float32)
        self.L.emu_step_param(self.h, _ptr(a), int(k), _ptr(self.obs), _ptr(self.reward), _ptr(self.done),
                              _ptr(self.result), _ptr(self.term_obs), _ptr(self.stats6))
        return self.obs, self.reward, self.done, self.result
