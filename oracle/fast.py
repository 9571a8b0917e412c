"""ORACLE (test infrastructure, NOT product code) -- ctypes binding of oracle/fast_oracle.c plus a
numpy vector-env (`OracleVecEnv`) that states, on the CPU, the batched semantics the CUDA library
implements: layout pool + per-env cursor, optional auto-reset, StuckPenalty counters
(src/wrappers/stuck_penalty_wrapper.py:19-58), the builder-specified first-visit ExplorationBonus
(absent from the reference, SURVEY F5) and per-episode return/length bookkeeping (src/ppo.py:88-98).

Tiles come from the literal per-pixel renderer in oracle/minigrid_restated.py (Grid.render_tile).
Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this module.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

from . import minigrid_restated as mg

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libfast_oracle.so")
_lib = None


def build(force=False):
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(
            os.path.join(_HERE, "fast_oracle.c")):
        subprocess.check_call(["make", "-C", _HERE, "-B" if force else "-s"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.fo_step.restype = ctypes.c_int
        _lib.fo_obs.restype = ctypes.c_int
        _lib.fo_set_threads.restype = ctypes.c_int
        _lib.fo_gae.restype = None
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def set_threads(n):
    return lib().fo_set_threads(ctypes.c_int(int(n)))


# ---- tile atlas from the literal renderer ----------------------------------------------------
N_TILE_SLOTS = 11 * 6 * 3 * 2 * 2


def tile_slot(type_, color, state, agent, hl):
    return (((type_ * 6 + color) * 3 + state) * 2 + agent) * 2 + hl


class TileAtlas:
    """Dense atlas filled lazily by Grid.render_tile for the (type,color,state) triples asked for."""

    def __init__(self, tile=8):
        self.tile = tile
        self.tiles = np.zeros((N_TILE_SLOTS, tile, tile, 3), dtype=np.uint8)
        self.present = np.zeros(N_TILE_SLOTS, dtype=np.uint8)
        self.ensure([(1, 0, 0)])  # empty / None

    def ensure(self, triples):
        for (t, c, s) in triples:
            t, c, s = int(t), int(c), int(s)
            obj = mg.WorldObj.decode(t, c, s) if t != 1 else None
            for agent in (0, 1):
                for hl in (0, 1):
                    k = tile_slot(t, c, s, agent, hl)
                    if self.present[k]:
                        continue
                    img = mg.Grid.render_tile(obj, agent_dir=3 if agent else None, highlight=bool(hl),
                                              tile_size=self.tile)
                    buf = np.zeros((self.tile, self.tile, 3), dtype=np.uint8)
                    buf[:, :, :] = img  # the same float64 -> uint8 assignment Grid.render performs
                    self.tiles[k] = buf
                    self.present[k] = 1


def split_enc(enc):
    """Grid.encode() layout enc[L,W,H,3] (index [i=x][j=y]) -> row-major type/color/state [L,H*W]."""
    enc = np.asarray(enc, dtype=np.uint8)
    L, W, H, _ = enc.shape
    rm = np.ascontiguousarray(enc.transpose(0, 2, 1, 3)).reshape(L, H * W, 3)
    return (np.ascontiguousarray(rm[:, :, 0]), np.ascontiguousarray(rm[:, :, 1]),
            np.ascontiguousarray(rm[:, :, 2]))


class OracleVecEnv:
    def __init__(self, num_envs, enc, agent, max_steps=None, view=7, tile=8, n_actions=3, auto_reset=True,
                 reset_mode="next", stuck_penalty=False, stuck_max_stay=3, stuck_penalty_value=-0.1,
                 exploration_bonus=0.0, want_rgb=True, atlas=None):
        enc = np.asarray(enc, dtype=np.uint8)
        self.N = int(num_envs)
        self.L, self.W, self.H = enc.shape[0], enc.shape[1], enc.shape[2]
        self.max_steps = int(max_steps) if max_steps is not None else 4 * self.W * self.H
        self.V, self.T = view, tile
        self.n_actions = n_actions
        self.auto_reset = auto_reset
        assert reset_mode in ("next", "same")
        self.reset_mode = reset_mode
        self.stuck_on, self.max_stay, self.penalty = stuck_penalty, stuck_max_stay, float(stuck_penalty_value)
        self.bonus = float(exploration_bonus)
        self.want_rgb = want_rgb
        self.pool_t, self.pool_c, self.pool_s = split_enc(enc)
        self.pool_agent = np.asarray(agent, dtype=np.int32).reshape(self.L, 3)
        self.atlas = atlas or TileAtlas(tile)
        if want_rgb:
            trip = np.unique(enc.reshape(-1, 3), axis=0)
            need = {tuple(int(v) for v in x) for x in trip}
            need |= {(4, c, st) for (t, c, _s) in list(need) if t == 4 for st in (0, 1, 2)}  # toggling changes door state
            self.atlas.ensure(sorted(need))
        N, HW = self.N, self.W * self.H
        self.gt = np.ones((N, HW), np.uint8)
        self.gc = np.zeros((N, HW), np.uint8)
        self.gs = np.zeros((N, HW), np.uint8)
        self.ax = np.zeros(N, np.int32)
        self.ay = np.zeros(N, np.int32)
        self.adir = np.zeros(N, np.int32)
        self.stepc = np.zeros(N, np.int32)
        self.carry_t = np.zeros(N, np.uint8)
        self.carry_c = np.zeros(N, np.uint8)
        self.cursor = (np.arange(N, dtype=np.int64) % self.L).astype(np.int32)
        self.stay = np.zeros(N, np.int32)
        self.last_x = np.zeros(N, np.int32)
        self.last_y = np.zeros(N, np.int32)
        self.visited = np.zeros((N, HW), bool)
        self.ep_return = np.zeros(N, np.float32)

    # ------------------------------------------------------------------------------------------
    def _load(self, idx):
        """(Re)start the envs in `idx` from pool[cursor]; advance the cursor in 'next' mode."""
        if len(idx) == 0:
            return
        cur = self.cursor[idx]
        self.gt[idx] = self.pool_t[cur]
        self.gc[idx] = self.pool_c[cur]
        self.gs[idx] = self.pool_s[cur]
        self.ax[idx] = self.pool_agent[cur, 0]
        self.ay[idx] = self.pool_agent[cur, 1]
        self.adir[idx] = self.pool_agent[cur, 2]
        self.stepc[idx] = 0
        self.carry_t[idx] = 0
        self.carry_c[idx] = 0
        self.stay[idx] = 0
        self.last_x[idx] = self.ax[idx]
        self.last_y[idx] = self.ay[idx]
        self.visited[idx] = False
        self.visited[idx, self.ay[idx] * self.W + self.ax[idx]] = True
        self.ep_return[idx] = 0
        if self.reset_mode == "next":
            # a restart moves on by N pool slots (mod L), or by one slot when L divides N: always a different layout
            stride = self.N % self.L or (1 if self.L > 1 else 0)
            self.cursor[idx] = ((cur.astype(np.int64) + stride) % self.L).astype(np.int32)

    def observe(self, want_sym=True, want_rgb=None):
        want_rgb = self.want_rgb if want_rgb is None else want_rgb
        N, V, T = self.N, self.V, self.T
        sym = np.zeros((N, V, V, 3), np.uint8) if want_sym else None
        rgb = np.zeros((N, V * T, V * T, 3), np.uint8) if want_rgb else None
        r = lib().fo_obs(N, self.W, self.H, V, T, _p(self.gt), _p(self.gc), _p(self.gs), _p(self.ax), _p(self.ay),
                         _p(self.adir), _p(self.carry_t), _p(self.carry_c), _p(self.atlas.tiles),
                         _p(self.atlas.present), _p(sym), _p(rgb))
        if r != 0:
            raise RuntimeError(f"fo_obs failed: {r} (tile missing from atlas?)")
        return rgb, sym

    def reset(self, mask=None):
        idx = np.arange(self.N) if mask is None else np.nonzero(np.asarray(mask))[0]
        self._load(idx)
        return self.observe()

    def step(self, actions):
        actions = np.ascontiguousarray(actions, dtype=np.int64)
        if np.any((actions < 0) | (actions >= self.n_actions)):
            raise ValueError("Unknown action")
        N = self.N
        reward = np.zeros(N, np.float64)
        term = np.zeros(N, np.uint8)
        trunc = np.zeros(N, np.uint8)
        r = lib().fo_step(N, self.W, self.H, self.max_steps, self.V, self.T, _p(self.gt), _p(self.gc), _p(self.gs),
                          _p(self.ax), _p(self.ay), _p(self.adir), _p(self.stepc), _p(self.carry_t),
                          _p(self.carry_c), _p(actions), _p(reward), _p(term), _p(trunc))
        if r != 0:
            raise RuntimeError(f"fo_step failed: {r}")
        reward_env = reward  # MiniGridEnv's own reward, before the shaping wrappers
        stuck = np.zeros(N, bool)
        if self.stuck_on:
            same = (self.ax == self.last_x) & (self.ay == self.last_y)
            self.stay = np.where(same, self.stay + 1, 0).astype(np.int32)
            stuck = self.stay >= self.max_stay
            reward = np.where(stuck, reward + self.penalty, reward)
            self.last_x[:] = self.ax
            self.last_y[:] = self.ay
        if self.bonus != 0.0:
            cell = self.ay * self.W + self.ax
            fresh = ~self.visited[np.arange(N), cell]
            self.visited[np.arange(N), cell] = True
            reward = np.where(fresh, reward + self.bonus, reward)
        reward32 = reward.astype(np.float32)
        self.ep_return = (self.ep_return + reward32).astype(np.float32)
        done = (term | trunc).astype(bool)
        ep_ret = np.where(done, self.ep_return, np.float32(0)).astype(np.float32)
        ep_len = np.where(done, self.stepc, 0).astype(np.int32)
        if self.auto_reset:
            self._load(np.nonzero(done)[0])
        rgb, sym = self.observe()
        info = {"episode_return": ep_ret, "episode_length": ep_len, "stuck": stuck, "obs_symbolic": sym,
                "reward_f64": reward, "reward_env": reward_env}
        return rgb, reward32, term.astype(bool), trunc.astype(bool), info


def gae(rew, val, done, last_val, gamma, lam):
    """[T,N] fp32 GAE + returns through fo_gae."""
    rew = np.ascontiguousarray(rew, np.float32)
    val = np.ascontiguousarray(val, np.float32)
    done = np.ascontiguousarray(done, np.float32)
    T, N = rew.shape
    last_val = np.ascontiguousarray(np.broadcast_to(np.asarray(last_val, np.float32), (N,)))
    adv = np.empty_like(rew)
    ret = np.empty_like(rew)
    lib().fo_gae(T, N, _p(rew), _p(val), _p(done), _p(last_val), ctypes.c_double(gamma), ctypes.c_double(lam),
                 _p(adv), _p(ret))
    return adv, ret
