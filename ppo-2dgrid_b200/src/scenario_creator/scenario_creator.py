"""ScenarioCreator -- YAML scenario table -> environments (reference
src/scenario_creator/scenario_creator.py:10-73, same constructor, methods, attributes and errors).

`create_env` builds the reference's single-env wrapper stack (RGB partial obs -> image only -> optional
flatten -> three actions) over a CUDA-backed env; `create_batched_env` is the additive batched surface: N envs
of one difficulty stepped by one kernel launch, observations / rewards / flags as device tensors.
"""
from __future__ import annotations

import os

import numpy as np
import yaml

import src.custom_envs.register as _register  # noqa: F401  (registration side effect, as in the reference)
from src.wrappers.obs_wrappers import FlattenObservation, FullyObsWrapper, ImgObsWrapper, RGBImgPartialObsWrapper
from src.wrappers.three_action_wrapper import ThreeActionWrapper

DEFAULT_CONFIG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "config", "scenario.yaml")


_PACKAGED_DEFAULT = "src/config/scenario.yaml"
# attribute <- (top-level YAML key, value when the key is absent); the reference reads the same five sections
_SECTIONS = (("seed", "seed", 42), ("global_cfg", "global", None), ("obs_cfg", "observation", None),
             ("rewards_cfg", "rewards", None), ("logging_cfg", "logging", None))


class ScenarioCreator:
    def __init__(self, config_path: str = _PACKAGED_DEFAULT):
        path = config_path
        if not os.path.exists(path) and path == _PACKAGED_DEFAULT and os.path.exists(DEFAULT_CONFIG):
            path = DEFAULT_CONFIG  # the packaged table, when not run from the repo root
        if not os.path.exists(path):
            raise FileNotFoundError(f"Config not found: {config_path}")
        with open(path) as fh:
            table = yaml.safe_load(fh)
        self.config = table
        for attr, key, missing in _SECTIONS:
            setattr(self, attr, table.get(key, {} if missing is None else missing))
        self._validate_grid_sizes()

    def _validate_grid_sizes(self):
        """One table, one grid size: ids shaped like `...-16x16-v0` must agree on the `16x16` part."""
        seen = []
        for entry in self.config["difficulties"].values():
            parts = entry["env_id"].split("-")
            if len(parts) > 1 and "x" in entry["env_id"] and parts[-2] not in seen:
                seen.append(parts[-2])
        if len(seen) > 1:
            raise ValueError(f"Multiple grid sizes detected: {set(seen)}")

    def _difficulty_cfg(self, difficulty):
        entry = self.config["difficulties"].get(difficulty)
        if entry:
            return entry
        raise ValueError(f"Unknown difficulty: {difficulty}")

    def _env_params(self, entry):
        merged = dict(self.global_cfg)
        merged.update(entry.get("params", {}))
        return merged

    # ---- the reference's single-env path ----------------------------------------------------------------
    def create_env(self, difficulty: str = "easy", seed=None):
        """`seed` is accepted and ignored, as in the reference (the env is seeded by `reset(seed=...)`)."""
        entry = self._difficulty_cfg(difficulty)
        full = bool(self.obs_cfg.get("fully_observable", False))
        stack = [FullyObsWrapper if full else RGBImgPartialObsWrapper, ImgObsWrapper]
        if self.obs_cfg.get("flatten", False):
            stack.append(FlattenObservation)
        stack.append(ThreeActionWrapper)
        env = _register.make(entry["env_id"], **self._env_params(entry))
        for wrap in stack:
            env = wrap(env)
        return env

    def sample_scenarios(self, n: int = 5, difficulty: str = "easy"):
        return [self.create_env(difficulty) for _ in range(n)]

    # ---- batched surface (additive) ---------------------------------------------------------------------
    def create_batched_env(self, difficulty="easy", num_envs=1, device="cuda", layouts=None, seeds=None,
                           stuck_penalty=False, exploration_bonus=0.0, fomaml_mode=False, size=None,
                           want_symbolic=False, n_layouts=None, **env_kwargs):
        """N envs of `difficulty` on `device`.  Layout pool: `layouts=(cells u8[L, H*W], agent i32[L, 3])`, or
        generated on the host from `seeds` (one `reset(seed=s)` layout per seed; default: seeds 0..max(N, 1024)-1).
        `layouts="device"` generates the pool on the GPU instead:
          - `seeds` a sequence of ints: one `reset(seed=s)` layout per seed, the same pool `layouts=None` builds on the
            host (`n_layouts` is ignored, as there);
          - `seeds` an int or None: `n_layouts` entries (default max(N, 1024)) from a counter-based stream keyed by the
            int -- fresh layouts of the right distribution, not the reference's per-seed layouts.
        `fomaml_mode`: finished envs restart on their own layout (src/fomaml.py:92) instead of the next one."""
        from merlin_b200 import BatchedMerlinEnv
        from merlin_b200 import layouts as _layouts

        cfg = self._difficulty_cfg(difficulty)
        params = self._env_params(cfg)
        size = int(size if size is not None else params.get("size", 16))
        diff = _register.DIFFICULTY_OF[cfg["env_id"]]
        common = dict(width=size, height=size)
        if isinstance(layouts, str):
            if layouts != "device":
                raise ValueError("layouts must be (cells, agent), None (host-generated from seeds) or 'device'")
            if seeds is None or np.ndim(seeds) == 0:
                pool = dict(generate=(diff, int(seeds or 0), int(n_layouts or max(int(num_envs), 1024))))
            else:
                pool = dict(generate_seeded=(diff, seeds))
            cells = agent = None
        else:
            if layouts is None:
                if seeds is None:
                    seeds = range(int(n_layouts or max(int(num_envs), 1024)))
                layouts = _layouts.generate(diff, size, seeds)
            cells, agent = (np.asarray(a) for a in layouts)
            pool = {}
        env = BatchedMerlinEnv(int(num_envs), cells, agent, **common, **pool,
                               max_steps=env_kwargs.pop("max_steps", params.get("max_steps")), device=device,
                               reset_mode="same" if fomaml_mode else "next", stuck_penalty=stuck_penalty,
                               exploration_bonus=exploration_bonus, want_symbolic=want_symbolic, **env_kwargs)
        env.difficulty = diff
        return env

    # ---- accessors --------------------------------------------------------------------------------------
    def get_env_id(self, difficulty: str) -> str:
        return self.config["difficulties"][difficulty]["env_id"]

    def get_observation_params(self) -> dict:
        return self.obs_cfg

    def get_logging_params(self) -> dict:
        return self.logging_cfg

    def get_env_size_str(self, difficulty: str) -> str:
        side = self.config["difficulties"][difficulty].get("params", {}).get("size", 16)
        return "x".join((str(side),) * 2)
