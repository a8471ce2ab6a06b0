"""The C oracle against the unmodified Python reference. Every scenario below runs on either side: on the reference's
own env objects it was recorded once into tests/golden/traces_reference.npz (python -m oracle.gen_golden traces), and
the tests replay it on the oracle against that recording (oracle/trace.py)."""
import os

import numpy as np
import pytest

from oracle import trace as tr
from oracle.oracle import ENV_SPECS, OracleVecEnv

TRACES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "traces_reference.npz")
_recorded = None


class OracleEnv(OracleVecEnv):
    """The oracle under the method names oracle.ref_loader.ReferenceVecEnv gives the reference's wrappers."""

    def view_obs(self, view_size):
        return self.gen_obs_view(view_size)

    def one_hot_obs(self):
        return self.one_hot(self.obs)


def make_oracle(env_id, n, autoreset="next_step", spec=None, gym_kwargs=None, no_death=(), death_cost=-1.0, bonus=None):
    """The oracle side of a scenario's env maker (gym_kwargs is what the reference's constructor takes instead of spec)."""
    e = OracleEnv(env_id, n, spec=spec, autoreset=autoreset)
    if no_death or bonus:
        e.set_no_death(no_death, death_cost)
        e.set_bonus(bonus)
    return e


def replay(name, scenario, *args):
    """Runs scenario(make_oracle, trace, *args) against the recording stored under `name`."""
    global _recorded
    if _recorded is None:
        _recorded = tr.load(TRACES)
    if name not in _recorded:
        raise AssertionError(f"no recording of {name}: regenerate the traces (python -m oracle.gen_golden traces)")
    t = tr.Trace(name, _recorded[name])
    scenario(make_oracle, t, *args)
    t.close()


# ---- scenarios: make(env_id, n, ...) builds the reference's or the oracle's vector env, trace records or checks ----
def lockstep(make, trace, env_id, mode, n=6, t_steps=250, seed=1000, action_seed=77, **make_kw):
    env = make(env_id, n, autoreset=mode, **make_kw)
    trace.exact("dims", [env.width, env.height, env.max_steps, env.see_through])
    trace.reset(env.reset(seed=seed))
    rng = np.random.default_rng(action_seed)
    for t in range(t_steps):
        a = rng.integers(0, 7, n)
        trace.step(env.step(a), a)
    trace.state(env)


UNREGISTERED_SIZES = [
    ("MiniGrid-Empty-5x5-v0", "empty", 26, 4 * 26 * 26, True, [1, 0, 0, 0]),  # agent_start_pos=None: random start
    ("MiniGrid-DoorKey-5x5-v0", "doorkey", 26, 10 * 26 * 26, False, []),
    ("MiniGrid-DoorKey-5x5-v0", "doorkey", 6, 10 * 6 * 6, False, []),
]


def unregistered_size(make, trace, base_id, kind, size, max_steps, see_through, params):
    gym_kwargs = {"size": size}
    if kind == "empty":
        gym_kwargs["agent_start_pos"] = None
    lockstep(make, trace, base_id, "next_step", n=4, t_steps=200, seed=5, action_seed=6,
             spec=(kind, size, size, max_steps, see_through, params), gym_kwargs=gym_kwargs)


WRAPPER_IDS = ["MiniGrid-DoorKey-8x8-v0", "MiniGrid-FourRooms-v0", "MiniGrid-Empty-5x5-v0", "MiniGrid-MultiRoom-N6-v0",
               "MiniGrid-Playground-v0", "MiniGrid-Dynamic-Obstacles-6x6-v0"]


def observation_wrappers(make, trace, env_id):
    n = 6
    env = make(env_id, n)
    env.reset(seed=31)
    rng = np.random.default_rng(5)
    for t in range(120):
        a = rng.integers(0, 7, n)
        trace.step(env.step(a), a)
        if t % 6 == 0:
            for V in (3, 5, 7, 9, 11):
                trace.digest(f"view {V} t={t}", env.view_obs(V))
            sym = env.symbolic_obs()
            assert sym.dtype == np.int64
            trace.digest(f"symbolic t={t}", sym)
            trace.digest(f"one-hot t={t}", env.one_hot_obs())


REWARD_WRAPPER_CASES = [
    ("MiniGrid-LavaCrossingS9N1-v0", ("lava",), None),
    ("MiniGrid-LavaCrossingS9N3-v0", ("lava",), "action"),
    ("MiniGrid-DistShift1-v0", ("lava",), "position"),
    ("MiniGrid-LavaGapS5-v0", ("lava", "wall"), None),
    ("MiniGrid-Dynamic-Obstacles-5x5-v0", ("ball",), None),
    ("MiniGrid-Dynamic-Obstacles-6x6-v0", ("ball",), "action"),
    ("MiniGrid-Empty-5x5-v0", (), "action"),
    ("MiniGrid-DoorKey-5x5-v0", (), "position"),
    ("MiniGrid-FourRooms-v0", (), "action"),
    ("MiniGrid-GoToDoor-5x5-v0", ("door",), "position"),
]


def reward_wrappers(make, trace, env_id, no_death, bonus, mode):
    n, t_steps = 6, 400
    env = make(env_id, n, autoreset=mode, no_death=no_death, death_cost=-1.5, bonus=bonus)
    env.reset(seed=2)
    rng = np.random.default_rng(11)
    saved = 0
    for t in range(t_steps):
        # forward-heavy actions: walk into lava / obstacles often
        a = np.where(rng.random(n) < 0.5, 2, rng.integers(0, 7, n))
        r = trace.step(env.step(a), a)
        saved += int(((r[2] < -0.4) & ~r[3]).sum())  # a negative reward on a live env: the death cost
    if no_death and "Empty" not in env_id and "GoToDoor" not in env_id:
        assert saved > 0, "NoDeath never triggered: the test does not cover it"


# ---- tests ----
@pytest.mark.parametrize("env_id", list(ENV_SPECS))
@pytest.mark.parametrize("mode", ["next_step", "same_step"])
def test_lockstep_rollout(env_id, mode):
    replay(f"lockstep {env_id} {mode}", lockstep, env_id, mode)


def test_spec_table_matches_registry():
    """(width, height, max_steps, see_through_walls) of gym.make(id).unwrapped, recorded for every id of ENV_SPECS."""
    def check(make, trace):
        for env_id, spec in ENV_SPECS.items():
            trace.exact(env_id, list(spec[1:5]))

    replay("registry", check)


@pytest.mark.parametrize("base_id,kind,size,max_steps,see_through,params", UNREGISTERED_SIZES)
def test_lockstep_rollout_at_unregistered_sizes(base_id, kind, size, max_steps, see_through, params):
    """The engine's size limit (26) and a small DoorKey that no id registers: the reference classes take `size`."""
    replay(f"unregistered {base_id} {size}", unregistered_size, base_id, kind, size, max_steps, see_through, params)


@pytest.mark.parametrize("env_id", WRAPPER_IDS)
def test_observation_wrappers_against_live_reference(env_id):
    """SURVEY 8(f-3): ViewSizeWrapper (V = 3, 5, 9, 11), SymbolicObsWrapper and OneHotPartialObsWrapper restated in the
    oracle (gen_obs_view, symbolic_obs, one_hot) against the reference's own wrapper classes on the same states."""
    replay(f"observation wrappers {env_id}", observation_wrappers, env_id)


# ---- SURVEY 8(f-4), second half: the reward wrappers (wrappers.py:68-184, 809-882) ----
@pytest.mark.parametrize("env_id,no_death,bonus", REWARD_WRAPPER_CASES)
@pytest.mark.parametrize("mode", ["next_step", "same_step"])
def test_reward_wrappers_against_live_reference(env_id, no_death, bonus, mode):
    """NoDeath, ActionBonus and PositionBonus as a SyncVectorEnv of wrapped envs applies them (bonus outermost), restated
    in the oracle (wrapped_step): rewards bit for bit, and the episodes NoDeath keeps alive stay alive."""
    replay(f"reward wrappers {env_id} {mode}", reward_wrappers, env_id, no_death, bonus, mode)


def test_reward_wrapper_known_answers():
    """The reference's own doctests: wrappers.py:81-93 (ActionBonus 1.0, 1.0), :137-145 (PositionBonus 1.0, 0.7071067811865475),
    :818-834 (NoDeath: LavaCrossingS9N1 seed 2 -> (-1.0, False); Dynamic-Obstacles-5x5 seed 2 -> (-2.0, False))."""
    o = OracleVecEnv("MiniGrid-Empty-5x5-v0", 1); o.set_bonus("action"); o.reset(seed=0)
    assert [float(o.step([1])[2][0]) for _ in range(2)] == [1.0, 1.0]
    o = OracleVecEnv("MiniGrid-Empty-5x5-v0", 1); o.set_bonus("position"); o.reset(seed=0)
    assert [float(o.step([1])[2][0]) for _ in range(2)] == [1.0, 0.7071067811865475]
    o = OracleVecEnv("MiniGrid-LavaCrossingS9N1-v0", 1); o.reset(seed=2); o.step([1])
    r = o.step([2]); assert (float(r[2][0]), bool(r[3][0])) == (0.0, True)
    o = OracleVecEnv("MiniGrid-LavaCrossingS9N1-v0", 1); o.set_no_death(("lava",), -1.0); o.reset(seed=2); o.step([1])
    r = o.step([2]); assert (float(r[2][0]), bool(r[3][0])) == (-1.0, False)
    o = OracleVecEnv("MiniGrid-Dynamic-Obstacles-5x5-v0", 1); o.reset(seed=2)
    r = o.step([2]); assert (float(r[2][0]), bool(r[3][0])) == (-1.0, True)
    o = OracleVecEnv("MiniGrid-Dynamic-Obstacles-5x5-v0", 1); o.set_no_death(("ball",), -1.0); o.reset(seed=2)
    r = o.step([2]); assert (float(r[2][0]), bool(r[3][0])) == (-2.0, False)


def constant_mission_ids():
    from minigrid_b200 import specs

    return [env_id for env_id in (specs.all_ids() if hasattr(specs, "all_ids") else list(ENV_SPECS))
            if "{" not in specs.get(env_id).mission]


def test_dict_observation_space_wrapper_mission_indices():
    """minigrid_b200.wrappers.mission_to_indices against the reference's DictObservationSpaceWrapper (wrappers.py:428-554) on the
    constant mission strings of the registered ids (its doctest value included: LavaCrossingS11N5 -> [19, 31, 17, 36, 20, 38, ...]).
    The recording holds the wrapper's word list (get_minigrid_words, in index order) and obs["mission"] after reset(seed=0)."""
    from minigrid_b200 import specs
    from minigrid_b200.wrappers import MINIGRID_WORDS, mission_to_indices

    def check(make, trace):
        trace.exact("words", list(MINIGRID_WORDS))
        for env_id in constant_mission_ids():
            trace.exact(f"mission {env_id}", mission_to_indices(specs.get(env_id).mission))

    replay("dict observation", check)
    assert len(constant_mission_ids()) >= 20
    assert mission_to_indices("avoid the lava and get to the green goal square")[:10] == [19, 31, 17, 36, 20, 38, 31, 2, 15, 35]
