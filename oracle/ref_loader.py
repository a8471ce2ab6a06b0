"""Import the UNMODIFIED Python reference (TEST INFRASTRUCTURE ONLY).

Only the fixture generators (oracle/gen_golden.py) use this module; the tests read what they recorded under
tests/golden/ and never need the reference. gymnasium and pygame may be missing: oracle/ref_shim supplies import
stand-ins (our own code); a real gymnasium, if installed, takes precedence.
"""
from __future__ import annotations

import importlib.util
import os
import sys

REFERENCE_ROOT = os.environ.get("MINIGRID_REFERENCE_ROOT", "/root/reference")
_SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_shim")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "minigrid"))


def load():
    """Returns (gymnasium_module, minigrid_module) with the reference's envs registered."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    if importlib.util.find_spec("gymnasium") is None or importlib.util.find_spec("pygame") is None:
        if _SHIM not in sys.path:
            sys.path.append(_SHIM)  # appended: real packages win
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import gymnasium  # noqa: E402
    import minigrid  # noqa: E402

    return gymnasium, minigrid


class ReferenceVecEnv:
    """N reference MiniGridEnv objects stepped in lockstep with SyncVectorEnv autoreset rules
    (gymnasium >= 1.0: NEXT_STEP default; SAME_STEP optional). Implemented here so the result does
    not depend on which gymnasium (if any) is installed (SURVEY.md Appendix A)."""

    def __init__(self, env_id, num_envs, autoreset="next_step", wrap=None, **kwargs):
        """wrap: optional callable env -> wrapped env (the reference's NoDeath / ActionBonus / PositionBonus, as a
        SyncVectorEnv of wrapped envs would hold them): step() and reset() then go through the wrapper."""
        import numpy as np

        gym, _ = load()
        self.np = np
        self.envs = [gym.make(env_id, **kwargs).unwrapped for _ in range(num_envs)]
        self.wrapped = [wrap(e) for e in self.envs] if wrap is not None else self.envs
        self.num_envs = num_envs
        e0 = self.envs[0]
        self.width, self.height, self.max_steps, self.see_through = e0.width, e0.height, e0.max_steps, e0.see_through_walls
        self.autoreset = autoreset
        self.pending = [False] * num_envs

    def reset(self, seed=None):
        np = self.np
        obs, dirs = [], []
        for i, e in enumerate(self.wrapped):
            s = None if seed is None else (int(seed) + i if np.isscalar(seed) else int(seed[i]))
            o, _ = e.reset(seed=s)
            obs.append(o["image"]); dirs.append(o["direction"])
        self.pending = [False] * self.num_envs
        return np.stack(obs), np.asarray(dirs, np.int32)

    def step(self, actions):
        np = self.np
        obs, dirs, rew, term, trunc = [], [], [], [], []
        for i, e in enumerate(self.wrapped):
            if self.autoreset == "next_step" and self.pending[i]:
                o, _ = e.reset()
                r, te, tr = 0.0, False, False
                self.pending[i] = False
            else:
                o, r, te, tr, _ = e.step(int(actions[i]))
                done = te or tr
                if self.autoreset == "next_step":
                    self.pending[i] = done
                elif self.autoreset == "same_step" and done:
                    o, _ = e.reset()
            obs.append(o["image"]); dirs.append(o["direction"]); rew.append(float(r)); term.append(te); trunc.append(tr)
        return (np.stack(obs), np.asarray(dirs, np.int32), np.asarray(rew, np.float64),
                np.asarray(term, bool), np.asarray(trunc, bool))

    def get_state(self):
        np = self.np
        n = self.num_envs
        e0 = self.envs[0]
        grid = np.zeros((n, e0.width, e0.height, 3), np.uint8)
        agent = np.zeros((n, 6), np.int32)
        rng = np.zeros((n, 6), np.uint64)
        for i, e in enumerate(self.envs):
            grid[i] = e.grid.encode()
            c = e.carrying
            enc = c.encode() if c is not None else (-1, 0, 0)
            agent[i] = [e.agent_pos[0], e.agent_pos[1], e.agent_dir, enc[0], enc[1], e.step_count]
            st = e.np_random.bit_generator.state
            s, inc = st["state"]["state"], st["state"]["inc"]
            m = (1 << 64) - 1
            rng[i] = [s >> 64, s & m, inc >> 64, inc & m, st["has_uint32"], st["uinteger"]]
        return {"grid": grid, "agent": agent, "rng": rng, "pending": np.asarray(self.pending, np.uint8)}

    def set_state(self, agent):
        """Agent records as OracleVecEnv.set_state takes them: x, y, dir, carried object type / colour (-1: none),
        step_count."""
        from minigrid.core.world_object import WorldObj

        for e, (x, y, d, ctype, ccolor, steps) in zip(self.envs, self.np.asarray(agent).tolist()):
            e.agent_pos, e.agent_dir, e.step_count = (x, y), d, steps
            e.carrying = None if ctype < 0 else WorldObj.decode(ctype, ccolor, 0)

    def full_obs(self):
        from minigrid.wrappers import FullyObsWrapper

        np = self.np
        return np.stack([FullyObsWrapper(e).observation({})["image"] for e in self.envs])

    # ---- observation wrappers of the reference, applied to the current state of every env (wrappers.py) ----
    def _last_obs(self, e):
        return e.gen_obs()

    def view_obs(self, view_size):
        """ViewSizeWrapper.observation (wrappers.py:663-673)."""
        from minigrid.wrappers import ViewSizeWrapper

        np = self.np
        return np.stack([ViewSizeWrapper(e, agent_view_size=view_size).observation(self._last_obs(e))["image"] for e in self.envs])

    def symbolic_obs(self):
        """SymbolicObsWrapper.observation (wrappers.py:762-782)."""
        from minigrid.wrappers import SymbolicObsWrapper

        np = self.np
        return np.stack([np.asarray(SymbolicObsWrapper(e).observation(self._last_obs(e))["image"]) for e in self.envs])

    def one_hot_obs(self):
        """OneHotPartialObsWrapper.observation (wrappers.py:268-284)."""
        from minigrid.wrappers import OneHotPartialObsWrapper

        np = self.np
        return np.stack([OneHotPartialObsWrapper(e).observation(self._last_obs(e))["image"] for e in self.envs])

    def flat_obs(self):
        """FlatObsWrapper.observation (wrappers.py:589-626)."""
        from minigrid.wrappers import FlatObsWrapper

        np = self.np
        return np.stack([FlatObsWrapper(e).observation(self._last_obs(e)) for e in self.envs])

    def rgb_partial_obs(self, tile_size=8):
        """RGBImgPartialObsWrapper.observation (wrappers.py:371-380): get_frame(tile_size, agent_pov=True)."""
        np = self.np
        return np.stack([e.get_frame(tile_size=tile_size, agent_pov=True) for e in self.envs])

    def rgb_full_obs(self, tile_size=8):
        """RGBImgObsWrapper.observation (wrappers.py:325-331): get_frame(highlight=True, tile_size)."""
        np = self.np
        return np.stack([e.get_frame(highlight=True, tile_size=tile_size) for e in self.envs])
