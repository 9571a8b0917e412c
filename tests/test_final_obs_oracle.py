"""CPU tests: the oracle's final observations (`info["final_obs_symbolic"]` / `info["final_obs"]` of
`FinalObsOracle.step`, tests/final_obs_oracle.py) are the observation the literal restatement
(oracle/minigrid_restated.py) returns for the step that ends an episode, before anything resets it -- the image the GPU
tests hold the step kernels' `final_sym` to."""
from __future__ import annotations

import numpy as np
import pytest

from final_obs_oracle import FinalObsOracle
from oracle import minigrid_restated as mg

LEFT, RIGHT, FORWARD, PICKUP, DROP, TOGGLE = 0, 1, 2, 3, 4, 5

# (objects by (x, y), agent (x, y, dir), max_steps, actions, how the episode ends)
SCENARIOS = {
    "goal": ({(3, 1): mg.Goal(), (1, 3): mg.Lava()}, (1, 1, 0), 60, [FORWARD, FORWARD], "terminated"),
    "lava": ({(1, 2): mg.Lava(), (4, 4): mg.Goal()}, (1, 1, 0), 60, [LEFT, RIGHT, RIGHT, FORWARD], "terminated"),
    "truncation": ({(5, 5): mg.Goal(), (3, 2): mg.Wall()}, (2, 2, 0), 5, [LEFT, FORWARD, RIGHT, FORWARD, LEFT],
                   "truncated"),
    # seven actions: pick the key up, drop it, pick it up again, open the locked door with it, turn to the box and
    # empty it, drop the key where the box stood, pick it up once more and step there -- cut by the step limit
    "pickup_drop_toggle": ({(2, 1): mg.Key("yellow"), (3, 1): mg.Door("yellow", is_locked=True), (3, 2): mg.Wall(),
                            (3, 3): mg.Wall(), (2, 2): mg.Box("purple"), (5, 2): mg.Ball("red"), (6, 6): mg.Goal()},
                           (1, 1, 0), 12,
                           [PICKUP, DROP, PICKUP, FORWARD, TOGGLE, LEFT, LEFT, LEFT, TOGGLE, DROP, PICKUP, FORWARD],
                           "truncated"),
}


class _Scratch(mg.MiniGridEnv):
    def __init__(self, objects, agent, max_steps):
        self._objects, self._agent = objects, agent
        super().__init__(mission_space=mg.MissionSpace(lambda: "x"), grid_size=9, max_steps=max_steps)

    def _gen_grid(self, w, h):
        self.grid = mg.Grid(w, h)
        self.grid.wall_rect(0, 0, w, h)
        for (x, y), obj in self._objects.items():
            self.grid.set(x, y, obj)
        self.agent_pos, self.agent_dir = self._agent[:2], self._agent[2]


@pytest.mark.parametrize("name", list(SCENARIOS))
def test_oracle_final_obs_is_the_restated_terminal_observation(name):
    objects, agent, max_steps, actions, ending = SCENARIOS[name]
    penv = _Scratch(objects, agent, max_steps)
    pobs, _ = penv.reset(seed=0)
    enc = penv.grid.encode()[None]
    n_actions = 7 if name == "pickup_drop_toggle" else 3
    kw = dict(max_steps=max_steps, n_actions=n_actions)
    auto = FinalObsOracle(1, enc, np.array([agent], np.int32), **kw)
    manual = FinalObsOracle(1, enc, np.array([agent], np.int32), auto_reset=False, **kw)
    _, sym0 = auto.reset()
    manual.reset()
    assert np.array_equal(sym0[0], pobs["image"])
    for t, a in enumerate(actions):
        pobs, _, pte, ptr, _ = penv.step(a)
        rgb, _, te, tr, info = auto.step(np.array([a]))
        mrgb, _, _, _, minfo = manual.step(np.array([a]))
        assert (bool(te[0]), bool(tr[0])) == (pte, ptr), t
        # without auto-reset the final row is the step's own observation
        want = minfo["obs_symbolic"][0] if (pte or ptr) else np.zeros_like(minfo["obs_symbolic"][0])
        assert np.array_equal(minfo["final_obs_symbolic"][0], want), t
        if not (pte or ptr):
            assert not info["final_obs_symbolic"].any() and not info["final_obs"].any(), t
            assert np.array_equal(info["obs_symbolic"][0], pobs["image"]), t
            continue
        assert t == len(actions) - 1
        assert (ending == "terminated") == pte and (ending == "truncated") == ptr
        frame = penv.get_frame(tile_size=8, agent_pov=True)
        assert np.array_equal(info["final_obs_symbolic"][0], pobs["image"])
        assert np.array_equal(info["final_obs"][0], frame)
        assert np.array_equal(mrgb[0], frame)
        # the step's own observation is already the next episode's
        assert not np.array_equal(info["obs_symbolic"][0], pobs["image"])
    if name == "pickup_drop_toggle":
        img = pobs["image"]
        assert tuple(img[3, 6]) == (5, 4, 0)        # the carried yellow key, shown in the agent's cell
        assert penv.carrying is not None and penv.grid.get(3, 1).is_open
        assert penv.grid.get(2, 2) is None and tuple(penv.agent_pos) == (2, 2)   # the box was emptied


def test_ppo_bootstrap_truncated_needs_a_batched_env():
    from src.ppo import PPO
    from src.scenario_creator.scenario_creator import ScenarioCreator
    env = ScenarioCreator().create_env("medium")
    with pytest.raises(ValueError, match="BatchedMerlinEnv"):
        PPO(env, batch_size=16, minibatch_size=8, bootstrap_truncated=True)
