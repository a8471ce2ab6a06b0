"""A small, fixed workload for compute-sanitizer (memcheck / racecheck / synccheck): both K1 layouts (tiled, window),
both autoreset modes with episodes forced to end (sparse and whole-tile waves), ragged last tile,
the reset / state / full-obs kernels and the observation-only pass. Compared with the oracle so that a sanitizer run is
also a parity run. Usage: compute-sanitizer --tool racecheck --kernel-regex kns=2mg python scripts/sanitize_smoke.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from minigrid_b200 import MinigridVecEnv
from oracle.oracle import OracleVecEnv

cases = [("MiniGrid-DoorKey-8x8-v0", None, None), ("MiniGrid-DoorKey-8x8-v0", "1", None),
         ("MiniGrid-FourRooms-v0", None, None), ("MiniGrid-LavaCrossingS9N1-v0", None, None), ("MiniGrid-Empty-8x8-v0", None, None),
         ("MiniGrid-Fetch-8x8-N3-v0", None, None), ("MiniGrid-MemoryS13Random-v0", None, None),
         # two CTAs of three warps: every warp goes through several tiles (mbarrier phase, prefetch, order list)
         ("MiniGrid-DoorKey-8x8-v0", None, "3", "2"), ("MiniGrid-FourRooms-v0", None, "3", "2"), ("MiniGrid-LavaCrossingS9N1-v0", None, "3", "2")]
if len(sys.argv) > 1:
    cases = cases[: int(sys.argv[1])]
n, steps = 1024 + 5, 14
for case in cases:
    env_id, layout, cfg = case[:3]
    grid_cap = case[3] if len(case) > 3 else None
    for mode in ("next_step", "same_step"):
        os.environ.pop("MINIGRID_B200_LAYOUT", None)
        os.environ.pop("MINIGRID_B200_CFG", None)
        os.environ.pop("MINIGRID_B200_GRID", None)
        if grid_cap is not None:
            os.environ["MINIGRID_B200_GRID"] = grid_cap
        if layout is not None:
            os.environ["MINIGRID_B200_LAYOUT"] = layout
        if cfg is not None:
            os.environ["MINIGRID_B200_CFG"] = cfg
        e = MinigridVecEnv(env_id, n, autoreset_mode=mode)
        o = OracleVecEnv(env_id, n, autoreset=mode, n_threads=0)
        obs, _ = e.reset(seed=3)
        oo, _ = o.reset(seed=3)
        assert np.array_equal(obs["image"].cpu().numpy(), oo)
        rng = np.random.default_rng(1)
        agent = o.get_state()["agent"].copy()
        agent[:, 5] = o.max_steps - rng.integers(1, 9, n)   # every env truncates within 8 steps: sparse ends
        agent[: n // 2, 5] = o.max_steps - 3                # and a dense wave in the first half of the tiles
        e.set_state(agent=agent)
        o.set_state(agent=agent)
        for t in range(steps):
            a = rng.integers(0, 7, n).astype(np.int32)
            r = e.step(torch.as_tensor(a, device="cuda"))
            q = o.step(a)
            assert np.array_equal(r[0]["image"].cpu().numpy(), q[0]), (env_id, layout, cfg, mode, t)
            assert r[1].cpu().numpy().tobytes() == q[2].tobytes()
        assert np.array_equal(e.full_obs().cpu().numpy(), o.full_obs())
        assert np.array_equal(e.gen_obs()["image"].cpu().numpy(), o.gen_obs()[0])
        st = e.get_state()
        assert np.array_equal(st["grid"].cpu().numpy(), o.get_state()["grid"])
        if env_id == "MiniGrid-LavaCrossingS9N1-v0" and grid_cap is None:  # the reward wrappers' branch of K1 (wrap_step)
            e.set_no_death(("lava",), -1.0); o.set_no_death(("lava",), -1.0)
            e.set_bonus("action"); o.set_bonus("action")
            for t in range(6):
                a = np.where(rng.random(n) < 0.5, 2, rng.integers(0, 7, n)).astype(np.int32)
                r = e.step(torch.as_tensor(a, device="cuda")); q = o.step(a)
                assert r[1].cpu().numpy().tobytes() == q[2].tobytes() and np.array_equal(r[2].cpu().numpy(), q[3])
        e.close()
        print("ok", env_id, "layout", layout, "cfg", cfg, "grid cap", grid_cap, mode, flush=True)
print("sanitize_smoke: all cases bit-exact")
