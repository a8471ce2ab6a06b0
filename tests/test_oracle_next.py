"""SURVEY 8(f) rows restated in the oracle ahead of their device kernels (f-1: LockedRoom, Playground; f-2, the first
step post-filter: GoToDoor): the oracle
against fixtures produced by the Python reference and against recordings of the reference's side of the scenarios
below (tests/golden/traces_reference.npz). The product does not register these ids yet, so there is no GPU counterpart
of this file."""
import os

import numpy as np
import pytest
from conftest import golden_files
from test_oracle_golden import test_rollout_matches_reference_fixture as check_rollout_fixture
from test_oracle_vs_reference import lockstep, replay

from oracle.oracle import ENV_SPECS, NEXT_SPECS, OracleVecEnv


@pytest.mark.parametrize("path", golden_files("next_rollout"), ids=os.path.basename)
def test_next_rollout_matches_reference_fixture(path):
    check_rollout_fixture(path)


def test_next_ids_are_not_product_ids_yet():
    from minigrid_b200 import specs

    assert not (set(NEXT_SPECS) & set(ENV_SPECS))
    for env_id in NEXT_SPECS:
        with pytest.raises(Exception):
            specs.get(env_id)


@pytest.mark.parametrize("env_id", list(NEXT_SPECS))
@pytest.mark.parametrize("mode", ["next_step", "same_step"])
def test_next_lockstep_rollout_against_live_reference(env_id, mode):
    replay(f"next lockstep {env_id} {mode}", lockstep, env_id, mode, 5, 420, 2024, 78)


# ---- the device generators of these kinds (mg_levels.cuh), compiled for the CPU by tests/host_emu ----
import sys  # noqa: E402

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emu"))
import parity  # noqa: E402
from conftest import load_golden  # noqa: E402
from emu import EmuVecEnv  # noqa: E402


# ids whose device generators exist in mg_levels.cuh (the step post-filter kinds are oracle-only so far)
DEVICE_NEXT = []
# ... and, for the step post-filter kinds, also mg_postfilter.cuh (Dynamic-Obstacles is oracle-only: RNG inside step)
DEVICE_NEXT += []


def make_next_emu(env_id, n, mode, layout=-1):
    return EmuVecEnv(NEXT_SPECS[env_id], n, autoreset=mode, layout=layout)


@pytest.mark.parametrize("layout", [0, 1], ids=["tiled", "window"])
@pytest.mark.parametrize("path", [p for p in golden_files("next_rollout") if any(i in p for i in DEVICE_NEXT)], ids=os.path.basename)
def test_next_device_generators_replay_reference_fixture(path, layout):
    """draw_level / cell_of / level_word / patch_level of the next kinds, through K2's fill and K1's template + patch
    autoreset as replayed by the host emulation, against what the Python reference produced."""
    parity.check_rollout_fixture(lambda env_id, n, mode: make_next_emu(env_id, n, mode, layout), load_golden(path))


@pytest.mark.parametrize("env_id", DEVICE_NEXT)
@pytest.mark.parametrize("mode,n", [("next_step", 70), ("same_step", 45)])
def test_next_device_generators_lockstep_vs_oracle(env_id, mode, n):
    emu = make_next_emu(env_id, n, mode)
    orc = OracleVecEnv(env_id, n, autoreset=mode)
    parity.check_lockstep_vs_oracle(emu, orc, 450, seed=99, check_state_every=150)


# ---- the post-filter branches random actions never reach, driven on purpose (scenarios as in test_oracle_vs_reference) ----
def memory_cells(make, trace, env_id):
    """Random actions almost never walk the hallway: drive every env to its end, half of them up and half down, so that
    both post-filter branches (memory.py:156-164) fire."""
    n = 24
    env = make(env_id, n)
    trace.reset(env.reset(seed=300))
    size = env.width
    turn = np.where(np.arange(n) % 2 == 0, 0, 1)  # left = up, right = down
    script = [np.full(n, 2)] * size + [turn] + [np.full(n, 2)] * 2 + [np.full(n, 3)] * 2
    rewards, ended = [], 0
    for a in script * 2:  # the second pass runs on the autoreset episodes
        r = trace.step(env.step(a), a)
        rewards.append(np.array(r[2]))  # a copy: the oracle reuses its output buffers
        ended += int(np.asarray(r[3]).sum())
    rewards = np.concatenate(rewards)
    assert ended >= n and (rewards > 0).any() and ended > int((rewards > 0).sum())  # successes and failures both seen


def _roomgrid_targets(ref, unlock):
    """From the reference's env objects: every agent next to its target (Unlock: in front of the locked door, with its
    key; the pickup variants: facing the object). Returns the agent records and how many envs were moved."""
    from minigrid.core.constants import COLOR_TO_IDX

    agent = ref.get_state()["agent"].copy()
    moved = 0
    for i, e in enumerate(ref.envs):
        tx, ty = (e.door.cur_pos if unlock else e.obj.cur_pos)
        for d, (dx, dy) in enumerate([(1, 0), (0, 1), (-1, 0), (0, -1)]):  # stand at target - d, face d
            ax, ay = tx - dx, ty - dy
            here = e.grid.get(ax, ay) if 0 < ax < e.width - 1 and 0 < ay < e.height - 1 else False
            if here is None or (here and here.type == "door" and not unlock):  # (S3 rooms: the only free neighbour is the doorway)
                agent[i, :3] = (ax, ay, d)
                agent[i, 3:5] = (5, COLOR_TO_IDX[e.door.color]) if unlock else (-1, 0)
                moved += 1
                break
    return agent, moved


def roomgrid_post_filters(make, trace, env_id):
    """Random actions practically never unlock a door or reach the object behind it: put every agent next to its target
    (the same injection on both sides) so that the success branches of unlock.py:88-96 and of the `carrying == self.obj`
    filters run."""
    n = 16
    env = make(env_id, n)
    trace.reset(env.reset(seed=700))
    unlock = env_id == "MiniGrid-Unlock-v0"
    targets = _roomgrid_targets(env, unlock) if trace.recording else None
    agent = trace.input("injected agent", lambda: targets[0])
    moved = int(trace.input("moved", lambda: targets[1]))
    assert moved >= n // 2
    env.set_state(agent=agent)
    act = np.full(n, 5 if unlock else 3)
    ended = 0
    for a in (act, act, np.full(n, 2)):
        r = trace.step(env.step(a), a)
        ended += int((np.asarray(r[3]) & (np.asarray(r[2]) > 0)).sum())
    assert ended >= moved  # every injected env succeeded once
    trace.state(env, full_obs=False)


def boxes_hide_keys(make, trace, env_id):
    """Box.contains / Box.toggle (world_object.py:273-293): agents put in front of a box, then toggle / pick up / drop
    scripts."""
    n = 24
    env = make(env_id, n)
    trace.reset(env.reset(seed=11))
    agent, moved = parity.face_first_cell_of_type(env, 7)
    assert moved.sum() >= n // 2
    env.set_state(agent=trace.exact("injected agent", agent))
    half = np.arange(n) % 2 == 0
    script = [np.where(half, 5, 3), np.where(half, 3, 0), np.where(half, 6, 4), np.where(half, 6, 5), np.where(half, 4, 3), np.full(n, 2)]
    for a in script:
        trace.step(env.step(a), a)
    st = trace.state(env, full_obs=False)
    assert (st["agent"][moved, 3] == 5).sum() >= moved.sum() // 4


MEMORY_IDS = ["MiniGrid-MemoryS7-v0", "MiniGrid-MemoryS13Random-v0"]
ROOMGRID_IDS = ["MiniGrid-Unlock-v0", "MiniGrid-UnlockPickup-v0", "MiniGrid-BlockedUnlockPickup-v0", "MiniGrid-KeyCorridorS3R3-v0",
                "MiniGrid-KeyCorridorS6R3-v0"]
BOX_IDS = ["MiniGrid-ObstructedMaze-1Dlh-v0", "MiniGrid-ObstructedMaze-Full-v1"]


@pytest.mark.parametrize("env_id", MEMORY_IDS)
def test_memory_success_and_failure_cells_against_live_reference(env_id):
    replay(f"memory cells {env_id}", memory_cells, env_id)


@pytest.mark.parametrize("env_id", ROOMGRID_IDS)
def test_roomgrid_post_filters_fire_against_live_reference(env_id):
    replay(f"roomgrid post-filters {env_id}", roomgrid_post_filters, env_id)


@pytest.mark.parametrize("env_id", BOX_IDS)
def test_boxes_hide_keys_against_live_reference(env_id):
    replay(f"boxes {env_id}", boxes_hide_keys, env_id)
