"""Final observations on top of the oracle (test infrastructure): `FinalObsOracle.step` is `OracleVecEnv.step` plus
info["final_obs_symbolic"] / info["final_obs"] -- for every env whose episode ends in the step, the observation of its
terminal state (what the reference's `env.step(a)` returns before its caller runs `env.reset()`), computed by
`observe()` before the auto-reset reloads the env; zero rows for the others.  Without auto-reset it is the step's own
observation."""
from __future__ import annotations

import numpy as np

from oracle import fast


class FinalObsOracle(fast.OracleVecEnv):
    _capturing = False
    _terminal = None

    def _load(self, idx):
        if self._capturing and len(idx):
            self._terminal = self.observe()   # the state after the action, before the restart
        super()._load(idx)

    def step(self, actions):
        self._capturing, self._terminal = True, None
        try:
            rgb, reward, term, trunc, info = super().step(actions)
        finally:
            self._capturing = False
        frgb, fsym = self._terminal if self._terminal is not None else (rgb, info["obs_symbolic"])
        done = term | trunc
        final_sym = np.zeros_like(info["obs_symbolic"])
        final_sym[done] = fsym[done]
        final_rgb = None
        if frgb is not None:
            final_rgb = np.zeros_like(frgb)
            final_rgb[done] = frgb[done]
        info["final_obs_symbolic"], info["final_obs"] = final_sym, final_rgb
        return rgb, reward, term, trunc, info
