"""What a scenario produced, kept compactly so that the oracle can be compared with the Python reference where the
reference is not installed. TEST INFRASTRUCTURE ONLY.

A scenario is a function of an environment maker and a `Trace`. `python -m oracle.gen_golden traces` runs it once on
the reference's own env objects with a recording trace and stores the result under tests/golden/; the tests run the
same function on the oracle with a checking trace, which fails at the first value that differs from the recording.

What is kept: small arrays as they are (rewards, flags, dimensions, injected inputs); large ones as 64-bit digests of
their values; the actions, observations and directions of a rollout as running digests taken every CHECKPOINT steps.
"""
from __future__ import annotations

import hashlib
import json

import numpy as np

CHECKPOINT = 50


def _value_bytes(a) -> bytes:
    """The values of `a` whatever its dtype (as np.testing.assert_array_equal compares them), with its shape."""
    a = np.asarray(a)
    canon = a.astype("<f8") if a.dtype.kind == "f" else a.astype("<i8")
    return repr(a.shape).encode() + np.ascontiguousarray(canon).tobytes()


def digest(a) -> np.uint64:
    return np.uint64(int.from_bytes(hashlib.blake2b(_value_bytes(a), digest_size=8).digest(), "little"))


class Trace:
    """recorded: None to record (then `data` holds what to store), or the stored arrays of this scenario to check."""

    def __init__(self, name: str, recorded: dict | None = None):
        self.name = name
        self.recording = recorded is None
        self.data = {} if recorded is None else recorded
        self._used = set()
        self._t = 0
        self._rows = {"reward": [], "terminated": [], "truncated": []}
        self._actions = hashlib.blake2b(digest_size=8)
        self._obs = hashlib.blake2b(digest_size=8)
        self._marks = []

    def _get(self, key):
        if key not in self.data:
            raise AssertionError(f"{self.name}: nothing recorded under {key!r}; regenerate the traces (python -m oracle.gen_golden traces)")
        self._used.add(key)
        return self.data[key]

    def exact(self, key, a):
        """A small array, compared value for value."""
        if self.recording:
            self.data[key] = np.asarray(a)
        else:
            np.testing.assert_array_equal(np.asarray(a), self._get(key), err_msg=f"{self.name}: {key}")
        return a

    def digest(self, key, a):
        """A large array, compared through the digest of its values."""
        if self.recording:
            self.data[key] = digest(a)
        else:
            assert digest(a) == self._get(key), f"{self.name}: {key} differs from the reference"
        return a

    def input(self, key, make):
        """A value the scenario derives from the reference's env objects (an injected state, say): computed by
        `make()` while recording, read back from the recording otherwise."""
        if self.recording:
            self.data[key] = np.asarray(make())
            return self.data[key]
        return self._get(key)

    def reset(self, out):
        obs, d = out[0], out[1]
        self.digest(f"reset obs {self._t}", obs)
        self.exact(f"reset dir {self._t}", d)
        return out

    def step(self, out, actions):
        """One vector step: actions in, (obs, dir, reward, terminated, truncated) out. Rewards are compared as IEEE bit
        patterns and the flags exactly at every step; actions, observations and directions every CHECKPOINT steps."""
        obs, d, r, te, tr = out[:5]
        t = self._t
        self._actions.update(_value_bytes(actions))
        self._obs.update(_value_bytes(obs))
        self._obs.update(_value_bytes(d))
        rows = {"reward": np.asarray(r, np.float64), "terminated": np.asarray(te, bool), "truncated": np.asarray(tr, bool)}
        for k, v in rows.items():
            if self.recording:
                self._rows[k].append(v)
            else:
                want = self._get(k)
                assert t < len(want), f"{self.name}: more steps than the recording's {len(want)}"
                if k == "reward":
                    assert v.tobytes() == want[t].tobytes(), f"{self.name}: reward bits t={t}: {v} != {want[t]}"
                else:
                    np.testing.assert_array_equal(v, want[t], err_msg=f"{self.name}: {k} t={t}")
        self._t += 1
        if self._t % CHECKPOINT == 0:
            self._checkpoint()
        return out

    def _checkpoint(self):
        first = self._marks[-1] if self._marks else 0
        k = len(self._marks)
        self._marks.append(self._t)
        a, o = (np.frombuffer(h.digest(), "<u8")[0] for h in (self._actions, self._obs))
        if self.recording:
            self._rows.setdefault("actions_digest", []).append(a)
            self._rows.setdefault("obs_digest", []).append(o)
        else:
            steps = f"steps {first}..{self._t - 1}"
            assert a == self._get("actions_digest")[k], f"{self.name}: the actions of {steps} are not the recorded ones"
            assert o == self._get("obs_digest")[k], f"{self.name}: obs / direction of {steps} differ from the reference"

    def state(self, env, full_obs=True):
        """get_state() (grid, agent, rng, pending) and, optionally, FullyObsWrapper's image."""
        st = env.get_state()
        self.digest("grid", st["grid"])
        self.exact("agent", st["agent"])
        self.digest("rng", st["rng"])
        self.exact("pending", st["pending"])
        if full_obs:
            self.digest("full_obs", env.full_obs())
        return st

    def close(self):
        if self._t % CHECKPOINT:
            self._checkpoint()
        if self.recording:
            for k, v in self._rows.items():
                if v:
                    self.data[k] = np.stack(v)
            return self.data
        if self._t:
            assert self._t == len(self._get("reward")), f"{self.name}: {self._t} steps, the recording has {len(self._get('reward'))}"
        missed = set(self.data) - self._used
        assert not missed, f"{self.name}: recorded but never compared: {sorted(missed)}"
        return None


def save(path, traces: dict):
    """traces: scenario name -> Trace.data. Stored as one byte buffer and an index (one npz member per array would
    cost more in zip headers than the arrays themselves)."""
    entries = sorted(((k, name, np.array(v, order="C")) for name, data in traces.items() for k, v in data.items()),
                     key=lambda e: (e[0].split(" ")[0], e[1], e[0]))  # like with like: better compression
    np.savez_compressed(path, name=np.array([f"{name}::{k}" for k, name, _ in entries]),
                        dtype=np.array([v.dtype.str for _, _, v in entries]),
                        shape=np.array([json.dumps(v.shape) for _, _, v in entries]),
                        size=np.array([v.nbytes for _, _, v in entries], np.int64),
                        data=np.frombuffer(b"".join(v.tobytes() for _, _, v in entries), np.uint8))


def load(path) -> dict:
    out = {}
    with np.load(path, allow_pickle=False) as f:
        data, ends = f["data"], np.cumsum(f["size"])
        for full, dt, shape, end, size in zip(f["name"], f["dtype"], f["shape"], ends, f["size"]):
            name, k = str(full).split("::", 1)
            a = np.frombuffer(data[end - size:end].tobytes(), np.dtype(str(dt))).reshape(json.loads(str(shape)))
            out.setdefault(name, {})[k] = a
    return out
