"""Generate tests/golden/*.npz from the UNMODIFIED Python reference (build container only).

Run:  python -m oracle.gen_golden          (needs /root/reference; see oracle/ref_loader.py)

Run:  python -m oracle.gen_golden next     (only the next_rollout_* fixtures of generators that have no device kernel yet)

Run:  python -m oracle.gen_golden traces   (only traces_reference.npz: the reference's side of the scenarios of
                                           tests/test_oracle_vs_reference.py and tests/test_oracle_next.py)

Two families of fixtures, both produced by the reference's own MiniGridEnv objects:
  rollout_<id>.npz   seeded reset + T lockstep steps of N envs with SyncVectorEnv NEXT_STEP
                     autoreset, uniform-random actions (np.random.default_rng(1234)); records every
                     obs/direction/reward/terminated/truncated, final state and FullyObs.
  inject_<id>.npz    random object soups (every type/colour/door state, random carrying) written
                     into a reference env through Grid.decode, then T steps without reset: pins the
                     transition + gen_obs for objects the four generators never create.
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.ref_loader import ReferenceVecEnv, load  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

ROLLOUTS = {  # id -> (N, T, seed)
    "MiniGrid-Empty-5x5-v0": (8, 260, 0),
    "MiniGrid-Empty-8x8-v0": (8, 600, 100),
    "MiniGrid-DoorKey-8x8-v0": (8, 1400, 7),
    "MiniGrid-LavaCrossingS9N1-v0": (8, 420, 2),
    "MiniGrid-FourRooms-v0": (8, 260, 31),
    "MiniGrid-Empty-Random-6x6-v0": (4, 200, 5),
    "MiniGrid-DoorKey-5x5-v0": (4, 300, 11),
    "MiniGrid-DoorKey-16x16-v0": (4, 200, 3),
    "MiniGrid-LavaCrossingS11N5-v0": (4, 200, 9),
    "MiniGrid-SimpleCrossingS9N2-v0": (4, 350, 21),
    "MiniGrid-LavaGapS5-v0": (4, 200, 13),
    "MiniGrid-LavaGapS7-v0": (4, 300, 17),
    "MiniGrid-DistShift1-v0": (4, 300, 19),
    "MiniGrid-DistShift2-v0": (4, 300, 23),
    "MiniGrid-MultiRoom-N2-S4-v0": (6, 130, 29),
    "MiniGrid-MultiRoom-N6-v0": (4, 260, 37),
    "MiniGrid-LockedRoom-v0": (4, 420, 41),
    "MiniGrid-Playground-v0": (4, 330, 43),
    "MiniGrid-GoToDoor-5x5-v0": (6, 260, 47),
    "MiniGrid-GoToDoor-8x8-v0": (6, 400, 53),
    "MiniGrid-Fetch-5x5-N2-v0": (6, 260, 59),
    "MiniGrid-Fetch-8x8-N3-v0": (6, 500, 61),
    "MiniGrid-RedBlueDoors-6x6-v0": (8, 900, 67),
    "MiniGrid-GoToObject-8x8-N2-v0": (6, 400, 71),
    "MiniGrid-PutNear-8x8-N3-v0": (8, 300, 73),
    "MiniGrid-MemoryS13Random-v0": (6, 600, 79),
    "MiniGrid-MemoryS7-v0": (6, 400, 83),
    "MiniGrid-Dynamic-Obstacles-Random-6x6-v0": (8, 400, 89),
    "MiniGrid-Dynamic-Obstacles-8x8-v0": (8, 500, 97),
    "MiniGrid-Unlock-v0": (6, 600, 101),
    "MiniGrid-UnlockPickup-v0": (6, 600, 103),
    "MiniGrid-BlockedUnlockPickup-v0": (6, 700, 107),
    "MiniGrid-KeyCorridorS3R2-v0": (6, 560, 109),
    "MiniGrid-KeyCorridorS4R3-v0": (4, 500, 113),
    "MiniGrid-KeyCorridorS6R3-v0": (4, 300, 127),
    "MiniGrid-ObstructedMaze-1Dlhb-v0": (6, 600, 131),
    "MiniGrid-ObstructedMaze-2Dlh-v0": (4, 600, 137),
    "MiniGrid-ObstructedMaze-2Q-v0": (4, 400, 139),
    "MiniGrid-ObstructedMaze-Full-v0": (4, 300, 149),
    "MiniGrid-ObstructedMaze-Full-v1": (4, 300, 151),
}
NEXT_ROLLOUTS = {  # SURVEY 8(f-1) generators whose device kernels do not exist yet: next_rollout_<id>.npz (oracle only)
}
INJECTS = {  # id (host env whose size/see_through/max_steps are used) -> (N, T)
    "MiniGrid-DoorKey-8x8-v0": (16, 120),
    "MiniGrid-Empty-8x8-v0": (8, 80),
    "MiniGrid-LavaCrossingS9N1-v0": (8, 80),
    "MiniGrid-FourRooms-v0": (8, 80),
    "MiniGrid-Empty-5x5-v0": (8, 60),
    "MiniGrid-DistShift1-v0": (8, 80),  # 9 x 7: width != height
}


# SURVEY 8(f-4): the reference's reward wrappers around every env (wrappers.py:68-184, 809-882), bonus outermost:
# rewardwrap_<name>.npz = a rollout fixture + the wrapper configuration. name -> (id, N, T, seed, no_death_types, death_cost, bonus, mode)
REWARD_WRAPS = {
    "nodeath_lava": ("MiniGrid-LavaCrossingS9N1-v0", 8, 500, 2, ("lava",), -1.0, None, "next_step"),
    "nodeath_lava_action": ("MiniGrid-DistShift1-v0", 8, 400, 3, ("lava",), -0.75, "action", "next_step"),
    "nodeath_ball": ("MiniGrid-Dynamic-Obstacles-6x6-v0", 8, 400, 2, ("ball",), -1.0, None, "next_step"),
    "nodeath_ball_position_samestep": ("MiniGrid-Dynamic-Obstacles-8x8-v0", 8, 400, 5, ("ball",), -2.5, "position", "same_step"),
    "action_doorkey": ("MiniGrid-DoorKey-8x8-v0", 8, 800, 7, (), 0.0, "action", "next_step"),
    "position_fourrooms": ("MiniGrid-FourRooms-v0", 8, 330, 31, (), 0.0, "position", "next_step"),
    "action_fourrooms_samestep": ("MiniGrid-FourRooms-v0", 8, 330, 33, (), 0.0, "action", "same_step"),
}


def reward_wrap(no_death, death_cost, bonus):
    load()
    from minigrid.wrappers import ActionBonus, NoDeath, PositionBonus

    def w(e):
        if no_death:
            e = NoDeath(e, no_death_types=tuple(no_death), death_cost=death_cost)
        if bonus == "action":
            e = ActionBonus(e)
        elif bonus == "position":
            e = PositionBonus(e)
        return e
    return w


def gen_rollout(env_id, n, t_steps, seed, mode="next_step", wrap=None, forward_share=0.0):
    ref = ReferenceVecEnv(env_id, n, autoreset=mode, wrap=wrap)
    obs0, dir0 = ref.reset(seed=seed)
    state0 = ref.get_state()
    full0 = ref.full_obs()
    rng = np.random.default_rng(1234)
    actions = rng.integers(0, 7, (t_steps, n)).astype(np.int32)
    if forward_share > 0:  # walk into things more often than uniform actions do
        actions = np.where(rng.random((t_steps, n)) < forward_share, 2, actions).astype(np.int32)
    obs = np.zeros((t_steps, n, 7, 7, 3), np.uint8)
    dirs = np.zeros((t_steps, n), np.int32)
    rew = np.zeros((t_steps, n), np.float64)
    term = np.zeros((t_steps, n), bool)
    trunc = np.zeros((t_steps, n), bool)
    for t in range(t_steps):
        obs[t], dirs[t], rew[t], term[t], trunc[t] = ref.step(actions[t])
    st = ref.get_state()
    e0 = ref.envs[0]
    return dict(env_id=env_id, mode=mode, seed=seed, actions=actions, obs0=obs0, dir0=dir0, obs=obs, dir=dirs,
                reward=rew, terminated=term, truncated=trunc, full_obs0=full0, full_obs=ref.full_obs(),
                grid0=state0["grid"], agent0=state0["agent"], rng0=state0["rng"],
                grid=st["grid"], agent=st["agent"], rng=st["rng"], pending=st["pending"],
                width=e0.width, height=e0.height, max_steps=e0.max_steps, see_through=e0.see_through_walls)


def random_soup(rng, W, H):
    """A random encoded grid [W][H][3]: grey border walls, interior of every object kind."""
    g = np.zeros((W, H, 3), np.uint8)
    g[:, :, 0] = 1
    for x in range(W):
        for y in range(H):
            if x in (0, W - 1) or y in (0, H - 1):
                g[x, y] = (2, 5, 0)
                continue
            r = rng.random()
            if r < 0.50:
                continue
            t = int(rng.choice([2, 3, 4, 4, 4, 5, 6, 7, 8, 9]))
            col = int(rng.integers(0, 6))
            state = int(rng.integers(0, 3)) if t == 4 else 0
            if t == 8:
                col = 1  # Goal() is always green after decode
            if t == 9:
                col = 0  # Lava() is always red
            g[x, y] = (t, col, state)
    return g


def gen_inject(env_id, n, t_steps, seed=99):
    gym, _ = load()
    from minigrid.core.grid import Grid
    from minigrid.core.world_object import Ball, Box, Key

    rng = np.random.default_rng(seed)
    envs = [gym.make(env_id).unwrapped for _ in range(n)]
    W, H = envs[0].width, envs[0].height
    grid0 = np.zeros((n, W, H, 3), np.uint8)
    agent0 = np.zeros((n, 6), np.int32)
    for i, e in enumerate(envs):
        e.reset(seed=i)
        g = random_soup(rng, W, H)
        # agent on a cell it could legally stand on: empty, floor, goal, lava, open door
        while True:
            ax, ay = int(rng.integers(1, W - 1)), int(rng.integers(1, H - 1))
            t, _, s = g[ax, ay]
            if t in (1, 3, 8, 9) or (t == 4 and s == 0):
                break
        grid, _ = Grid.decode(g)
        e.grid = grid
        e.agent_pos = (ax, ay)
        e.agent_dir = int(rng.integers(0, 4))
        c = int(rng.integers(0, 4))
        colors = ["red", "green", "blue", "purple", "yellow", "grey"]
        col = colors[int(rng.integers(0, 6))]
        e.carrying = [None, Key(col), Ball(col), Box(col)][c]
        e.step_count = int(rng.integers(0, 20))
        grid0[i] = e.grid.encode()
        enc = e.carrying.encode() if e.carrying is not None else (-1, 0, 0)
        agent0[i] = [ax, ay, e.agent_dir, enc[0], enc[1], e.step_count]
    obs0 = np.stack([e.gen_obs()["image"] for e in envs])
    actions = rng.integers(0, 7, (t_steps, n)).astype(np.int32)
    obs = np.zeros((t_steps, n, 7, 7, 3), np.uint8)
    dirs = np.zeros((t_steps, n), np.int32)
    rew = np.zeros((t_steps, n), np.float64)
    term = np.zeros((t_steps, n), bool)
    trunc = np.zeros((t_steps, n), bool)
    for t in range(t_steps):
        for i, e in enumerate(envs):
            o, r, te, tr, _ = e.step(int(actions[t, i]))
            obs[t, i], dirs[t, i], rew[t, i], term[t, i], trunc[t, i] = o["image"], o["direction"], r, te, tr
    grid = np.stack([e.grid.encode() for e in envs])
    agent = np.zeros((n, 6), np.int32)
    for i, e in enumerate(envs):
        enc = e.carrying.encode() if e.carrying is not None else (-1, 0, 0)
        agent[i] = [e.agent_pos[0], e.agent_pos[1], e.agent_dir, enc[0], enc[1], e.step_count]
    e0 = envs[0]
    return dict(env_id=env_id, actions=actions, obs0=obs0, obs=obs, dir=dirs, reward=rew, terminated=term,
                truncated=trunc, grid0=grid0, agent0=agent0, grid=grid, agent=agent,
                width=W, height=H, max_steps=e0.max_steps, see_through=e0.see_through_walls)


WRAPPER_FIXTURES = {  # id -> (N, steps before the snapshot): the reference's observation wrappers on the same states
    "MiniGrid-DoorKey-8x8-v0": (6, 90),
    "MiniGrid-FourRooms-v0": (5, 40),
    "MiniGrid-Playground-v0": (5, 60),
    "MiniGrid-Empty-5x5-v0": (4, 7),
    "MiniGrid-LavaCrossingS9N1-v0": (4, 12),
}


def gen_wrappers(env_id, n, t_steps, seed=77):
    """State after t_steps random steps + what the reference's wrapper classes (minigrid/wrappers.py) return on it."""
    ref = ReferenceVecEnv(env_id, n, autoreset="next_step")
    ref.reset(seed=seed)
    rng = np.random.default_rng(4)
    obs = None
    for t in range(t_steps):
        obs = ref.step(rng.integers(0, 6, n))  # no `done`: keeps the post-filter envs of other fixtures out of this one
    st = ref.get_state()
    out = dict(env_id=env_id, seed=seed, grid=st["grid"], agent=st["agent"], obs=obs[0], one_hot=ref.one_hot_obs(),
               symbolic=ref.symbolic_obs(), rgb_partial=ref.rgb_partial_obs(), rgb_full=ref.rgb_full_obs(), full_obs=ref.full_obs())
    for V in (3, 5, 9, 11):
        out[f"view{V}"] = ref.view_obs(V)
    try:
        out["flat"] = ref.flat_obs()
    except Exception:  # noqa: BLE001  (missions with characters FlatObsWrapper rejects)
        pass
    return out


def main_wrappers():
    os.makedirs(OUT, exist_ok=True)
    for env_id, (n, t) in WRAPPER_FIXTURES.items():
        d = gen_wrappers(env_id, n, t)
        np.savez_compressed(os.path.join(OUT, f"wrappers_{env_id}.npz"), **d)
        print("wrappers", env_id, {k: v.shape for k, v in d.items() if hasattr(v, "shape") and k.startswith(("rgb", "flat", "view9"))})


def main_reward_wrappers():
    os.makedirs(OUT, exist_ok=True)
    for name, (env_id, n, t, seed, no_death, cost, bonus, mode) in REWARD_WRAPS.items():
        d = gen_rollout(env_id, n, t, seed, mode=mode, wrap=reward_wrap(no_death, cost, bonus), forward_share=0.4)
        d.update(no_death=np.array(list(no_death), dtype="U8"), death_cost=cost, bonus=bonus or "")
        np.savez_compressed(os.path.join(OUT, f"rewardwrap_{name}.npz"), **d)
        print("rewardwrap", name, "episodes ended:", int((d["terminated"] | d["truncated"]).sum()),
              "negative rewards on live envs:", int(((d["reward"] < 0) & ~d["terminated"]).sum()))


def main_next():
    os.makedirs(OUT, exist_ok=True)
    for env_id, (n, t, seed) in NEXT_ROLLOUTS.items():
        d = gen_rollout(env_id, n, t, seed)
        np.savez_compressed(os.path.join(OUT, f"next_rollout_{env_id}.npz"), **d)
        print("next_rollout", env_id, "episodes ended:", int((d["terminated"] | d["truncated"]).sum()))


def main_traces():
    """Every scenario of tests/test_oracle_vs_reference.py and tests/test_oracle_next.py run on the reference's env
    objects with a recording trace (oracle/trace.py), under the names the tests replay."""
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
    import test_oracle_next as tn
    import test_oracle_vs_reference as tv

    from oracle import trace
    from oracle.oracle import ENV_SPECS, NEXT_SPECS

    gym, _ = load()
    from minigrid.wrappers import DictObservationSpaceWrapper

    def make(env_id, n, autoreset="next_step", spec=None, gym_kwargs=None, no_death=(), death_cost=-1.0, bonus=None):
        wrap = reward_wrap(no_death, death_cost, bonus) if (no_death or bonus) else None
        return ReferenceVecEnv(env_id, n, autoreset=autoreset, wrap=wrap, **(gym_kwargs or {}))

    out = {}

    def record(name, scenario, *args):
        t = trace.Trace(name)
        scenario(make, t, *args)
        out[name] = t.close()

    def registry(make, t):
        for env_id in ENV_SPECS:
            e = gym.make(env_id).unwrapped
            t.exact(env_id, [e.width, e.height, e.max_steps, e.see_through_walls])

    def dict_observation(make, t):
        words = DictObservationSpaceWrapper.get_minigrid_words()
        assert sorted(words.values()) == list(range(len(words)))
        t.exact("words", sorted(words, key=words.get))
        for env_id in tv.constant_mission_ids():
            obs, _ = DictObservationSpaceWrapper(gym.make(env_id)).reset(seed=0)
            t.exact(f"mission {env_id}", obs["mission"])

    for mode in ("next_step", "same_step"):
        for env_id in ENV_SPECS:
            record(f"lockstep {env_id} {mode}", tv.lockstep, env_id, mode)
        for env_id in NEXT_SPECS:
            record(f"next lockstep {env_id} {mode}", tv.lockstep, env_id, mode, 5, 420, 2024, 78)
        for env_id, no_death, bonus in tv.REWARD_WRAPPER_CASES:
            record(f"reward wrappers {env_id} {mode}", tv.reward_wrappers, env_id, no_death, bonus, mode)
    record("registry", registry)
    record("dict observation", dict_observation)
    for case in tv.UNREGISTERED_SIZES:
        record(f"unregistered {case[0]} {case[2]}", tv.unregistered_size, *case)
    for env_id in tv.WRAPPER_IDS:
        record(f"observation wrappers {env_id}", tv.observation_wrappers, env_id)
    for env_id in tn.MEMORY_IDS:
        record(f"memory cells {env_id}", tn.memory_cells, env_id)
    for env_id in tn.ROOMGRID_IDS:
        record(f"roomgrid post-filters {env_id}", tn.roomgrid_post_filters, env_id)
    for env_id in tn.BOX_IDS:
        record(f"boxes {env_id}", tn.boxes_hide_keys, env_id)
    os.makedirs(OUT, exist_ok=True)
    trace.save(os.path.join(OUT, "traces_reference.npz"), out)
    print("traces", len(out), "scenarios")


def main():
    os.makedirs(OUT, exist_ok=True)
    for env_id, (n, t, seed) in ROLLOUTS.items():
        d = gen_rollout(env_id, n, t, seed)
        np.savez_compressed(os.path.join(OUT, f"rollout_{env_id}.npz"), **d)
        print("rollout", env_id, "episodes ended:", int((d["terminated"] | d["truncated"]).sum()))
    d = gen_rollout("MiniGrid-FourRooms-v0", 8, 260, 31, mode="same_step")
    np.savez_compressed(os.path.join(OUT, "rollout_samestep_MiniGrid-FourRooms-v0.npz"), **d)
    for env_id, (n, t) in INJECTS.items():
        d = gen_inject(env_id, n, t)
        np.savez_compressed(os.path.join(OUT, f"inject_{env_id}.npz"), **d)
        print("inject", env_id, "terminated:", int(d["terminated"].sum()))
    # known-answer vectors of the reference's own tests/doctests, re-derived from the reference here
    gym, _ = load()
    kat = {}
    for s in (0, 1, 123):
        e = gym.make("MiniGrid-Empty-5x5-v0").unwrapped
        e.reset(seed=s)
        kat[f"empty5_seed{s}_integers10"] = np.array([int(e.np_random.integers(10)) for _ in range(10)])
    np.savez_compressed(os.path.join(OUT, "kat.npz"), **kat)


if __name__ == "__main__":
    if sys.argv[1:] == ["next"]:   # python -m oracle.gen_golden next: only the next_rollout_* fixtures
        main_next()
    elif sys.argv[1:] == ["wrappers"]:
        main_wrappers()
    elif sys.argv[1:] == ["reward_wrappers"]:
        main_reward_wrappers()
    elif sys.argv[1:] == ["traces"]:
        main_traces()
    else:
        main()
        main_next()
        main_wrappers()
        main_reward_wrappers()
        main_traces()
