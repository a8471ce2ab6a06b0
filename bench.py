#!/usr/bin/env python
"""bench.py — env-steps/s of the batched Minigrid hot path (BASELINE.json's metric).

    python bench.py --gpus 1 --steps K --warmup W            # this engine, 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   # N GPUs, weak scaling
    python bench.py --impl reference ...                      # the reference algorithm on the host CPUs
    python bench.py ... --dump-outputs DIR                    # + the last timed step's arrays as DIR/*.npy (A/B of builds)

One "step" = one lockstep vector step (action -> state', obs, reward, terminated, truncated, autoreset) of the
whole batch. Headline workload (config.workload): BASELINE.json configs[2], MiniGrid-DoorKey-8x8-v0 with 262144
environments per GPU (the configuration the >=1e8 steps/s target is quoted on), uniform random actions generated
on the device before timing, NEXT_STEP autoreset with DESYNCHRONISED episodes: before timing every env's step_count
is drawn from U[0, max_steps) (mg_set_state), so each timed step regenerates ~n / max_steps environments — the steady
state of a long run — instead of none (a batch that was just reset) or all of them (the synchronised truncation
wave, reported separately as `sync_wave`). The other BASELINE configs are timed the same way and reported under
`configs`. Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALGO_BYTES_PER_STEP = 348  # SURVEY.md 8(d): action 4 + patch 147 + obs 147 + reward 8 + flags 2 + agent 20 r + 20 w
L2_BYTES = 126e6
HEADLINE_ENV = "MiniGrid-DoorKey-8x8-v0"
# BASELINE.json configs[1], [3], [4] (per-GPU share); configs[0] (Empty-5x5, 1 env, CPU) is the `config1` key
DUMP_ENVS = 65536  # --dump-outputs: at most this many environments of the last step
OTHER_CONFIGS = [("MiniGrid-Empty-8x8-v0", 65536), ("MiniGrid-LavaCrossingS9N1-v0", 262144), ("MiniGrid-FourRooms-v0", 262144)]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--env", default=HEADLINE_ENV)
    ap.add_argument("--envs-per-gpu", type=int, default=262144)
    ap.add_argument("--rotate", type=int, default=0, help="independent env batches cycled through so the working set exceeds L2 (0 = auto)")
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configs and the long single-batch runs")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--graph", type=int, default=1, help="replay the step loop as CUDA graphs (0 = eager launches)")
    ap.add_argument("--sync-episodes", action="store_true", help="do NOT desynchronise the episodes (round-1 behaviour: no autoreset in the timed region)")
    ap.add_argument("--host-format", default="packed", choices=["packed", "full"], help="D2H format of the e2e leg (packed: 52 B/env expanded on the host)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned as DIR/<name>.npy "
                    "(float32, reward float64; a fixed sample of DUMP_ENVS environments of larger batches) to compare two builds")
    return ap.parse_args()


def dump_outputs(out_dir, env, seed=0):
    """Writes the arrays env.step() returned last: step() hands back the same tensors on every call (the copy=False
    convention), so after the timed loop they hold its last step. Batches above DUMP_ENVS envs are sampled, the same
    sorted subset of env indices on every run (65536 envs: 39 MB of float32 images)."""
    import torch

    n = env.num_envs
    idx = np.arange(n) if n <= DUMP_ENVS else np.sort(np.random.default_rng(seed).choice(n, DUMP_ENVS, replace=False))
    sel = torch.as_tensor(idx, device=env.device)
    outputs = {"image": (env._obs_dict["image"], torch.float32), "direction": (env._obs_dict["direction"], torch.float32),
               "reward": (env._reward, torch.float64), "terminated": (env._terminated, torch.float32),
               "truncated": (env._truncated, torch.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, (t, dtype) in outputs.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.index_select(0, sel).to(dtype).cpu().numpy())


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(env_id, n):
    """dram__bytes_read.sum + dram__bytes_write.sum per k_step launch, from the committed ncu capture of this workload
    (profiles/traffic.json, written by scripts/ncu_traffic.py from >= 16 consecutive launches, caches not flushed
    between them: steady-state write-back included)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f).get(f"{env_id}|{n}")
        return (float(t["bytes_per_launch"]), t["source"]) if t else (None, None)
    except Exception:
        return None, None


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML from a background thread DURING the timed region."""

    def __init__(self, gpu_index, period_s=0.02):
        self.gpu, self.period = gpu_index, period_s
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = None
        self._thread = None

    def start(self):
        import threading

        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except (ValueError, IndexError):
                    idx = self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            return
        names = {
            pynvml.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            pynvml.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            pynvml.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            pynvml.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        self._stop = threading.Event()

        def loop():
            while not self._stop.is_set():
                try:
                    self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
                self._stop.wait(self.period)

        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if self.samples:
            out["sm_mhz"] = float(np.median(self.samples))
        return out


def usable_cores():
    """Host threads this process can actually run at once: min(online CPUs, cgroup CPU quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(np.ceil(int(quota) / int(period)))))
    except Exception:
        pass
    return n


def make_config(env_id, n, world, sync_episodes=False):
    """The workload description: identical for the engine arm and the reference arm."""
    total = n * world
    episodes = ("synchronised (all envs reset together before timing)" if sync_episodes else
                "desynchronised: step_count ~ U[0, max_steps) per env before timing, so every timed step autoresets ~n/max_steps envs")
    return {"workload": f"{env_id}, {n} envs per GPU ({total} total), uniform random actions, NEXT_STEP autoreset, episodes {episodes.split(':')[0]}",
            "env": env_id, "envs_per_gpu": n, "total_envs": total, "autoreset": "next_step", "episodes": episodes}


def desync_oracle(env, seed=4321):
    """step_count ~ U[0, max_steps) per env (the engine arm does the same through mg_set_state)."""
    st = env.get_state()
    agent = st["agent"].copy()
    agent[:, 5] = np.random.default_rng(seed).integers(0, env.max_steps, env.num_envs)
    env.set_state(agent=agent)


def run_reference(args, rank, world):
    """The reference algorithm on the host CPUs: the oracle port (C restatement of MiniGridEnv.step/gen_obs,
    validated against the Python reference), one env slice per host thread. The Python reference itself cannot
    travel to the GPU box (no gymnasium in the image)."""
    if rank != 0:
        return
    from oracle.oracle import OracleVecEnv, max_threads

    n = args.envs_per_gpu
    cores = min(max_threads(), usable_cores())
    env = OracleVecEnv(args.env, n, autoreset="next_step", n_threads=cores)
    env.reset(seed=0)
    if not args.sync_episodes:
        desync_oracle(env)
    rng = np.random.default_rng(1234)
    # bounded sample: keep the whole run to a few minutes whatever the core count
    probe_steps = 2
    secs, _ = env.rollout(rng.integers(0, 7, (probe_steps, n)).astype(np.int32), n_threads=cores)
    per_step = max(secs / probe_steps, 1e-6)
    budget = 120.0
    steps = int(max(3, min(args.steps, budget / per_step)))
    warm = int(max(1, min(args.warmup, 10.0 / per_step)))
    env.rollout(rng.integers(0, 7, (warm, n)).astype(np.int32), n_threads=cores)
    secs, _ = env.rollout(rng.integers(0, 7, (steps, n)).astype(np.int32), n_threads=cores)
    value = n * steps / secs
    line = {
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * secs / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": make_config(args.env, n, world, args.sync_episodes),
        "run": {"host_threads": cores, "sample_envs": n},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "per_core": value / cores, "kind": "port",
                         "sample": f"{n} envs x {steps} lockstep steps (one GPU's share of the workload), C port of the reference algorithm "
                                   f"(oracle/mg_oracle.c), {cores} threads"},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def cpu_baseline(args):
    from oracle.oracle import OracleVecEnv, max_threads

    cores = min(max_threads(), usable_cores())
    n = 65536
    env = OracleVecEnv(args.env, n, autoreset="next_step", n_threads=cores)
    env.reset(seed=0)
    if not args.sync_episodes:
        desync_oracle(env)
    rng = np.random.default_rng(1234)
    secs, _ = env.rollout(rng.integers(0, 7, (2, n)).astype(np.int32), n_threads=cores)
    steps = int(max(4, min(2000, args.cpu_seconds / max(secs / 2, 1e-6))))
    secs, _ = env.rollout(rng.integers(0, 7, (steps, n)).astype(np.int32), n_threads=cores)
    return {"value": n * steps / secs, "unit": "env-steps/s", "cores": cores, "per_core": n * steps / secs / cores, "kind": "port",
            "sample": f"{n} envs x {steps} lockstep steps of {args.env} ({secs:.1f} s), oracle C port on {cores} host threads "
                      f"(os.cpu_count()={os.cpu_count()}, cgroup CPU quota respected)"}


def config1_cpu():
    """BASELINE.json configs[0]: MiniGrid-Empty-5x5-v0, ONE env, random actions on the CPU (minigrid/benchmark.py's loop):
    the oracle port, single thread."""
    from oracle.oracle import OracleVecEnv

    env = OracleVecEnv("MiniGrid-Empty-5x5-v0", 1, autoreset="next_step", n_threads=1)
    env.reset(seed=0)
    a = np.random.default_rng(1234).integers(0, 7, (200000, 1)).astype(np.int32)
    env.rollout(a[:20000], n_threads=1)
    secs, _ = env.rollout(a, n_threads=1)
    return a.shape[0] / secs


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from minigrid_b200 import MinigridVecEnv, bind_to_gpu_numa_node, make_sharded

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # torch's CPU thread pool is not used by anything measured here, but its workers keep spinning for a while after any
    # parallel CPU op (OpenMP block time) — next to the host threads that expand packed step records in the e2e leg
    torch.set_num_threads(1)
    # pinned host buffers (the e2e leg) should live on the GPU's own NUMA node: with 8 ranks copying at once, remote
    # pinned memory costs a quarter of the D2H bandwidth (round 1: 37 instead of 50 GB/s per GPU at N = 8)
    cores_total = usable_cores()  # before the NUMA binding narrows this process's affinity mask to one node's CPUs
    numa = bind_to_gpu_numa_node(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    K, W = args.steps, max(3, args.warmup)  # never fewer than 3 untimed steps before a timed region
    peak, peak_src = load_peaks()

    def desync(env, seed):
        st = env.get_state()
        g = torch.Generator(device=dev).manual_seed(seed)
        st["agent"][:, 5] = torch.randint(0, env.max_steps, (env.num_envs,), generator=g, device=dev, dtype=torch.int32)
        env.set_state(agent=st["agent"])

    def time_workload(env_id, n, K, W, *, rotate=0, sync_episodes=False, autoreset="next_step", want_graph=True):
        """W untimed + K timed vector steps of R rotating batches of n envs; returns the measurement and the batches."""
        total = n * world
        probe = make_sharded(env_id, total, rank, world, device=dev, autoreset_mode=autoreset)
        wpe_bytes = ((probe.height + 2) * ((probe.width + 3) // 4) + (probe.width + 2) * ((probe.height + 3) // 4)) * 4
        ws = n * (min(wpe_bytes, 224 + 32) + 147 + 16 + 16 + 4 + 4 + 8 + 2)  # bytes a step touches per env (window layout: 7 lines)
        R = rotate if rotate > 0 else max(1, int(np.ceil(2.2 * L2_BYTES / ws)))
        batches = [probe] + [make_sharded(env_id, total, rank, world, device=dev, autoreset_mode=autoreset) for _ in range(R - 1)]
        for b, e in enumerate(batches):
            e.reset(seed=1_000_003 * b)  # env i of batch b: seed 1000003*b + global index
            if not sync_episodes:
                desync(e, 77 + 1000 * b + rank)
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        T = int(min(max(K + W, 64), 512))  # action table rows, cycled
        actions = torch.randint(0, 7, (T, n), generator=gen, device=dev, dtype=torch.int32)
        torch.cuda.synchronize()
        act_rows = [actions[i] for i in range(T)]  # views made once: the timed loop is launches only
        step_fns = [b.step for b in batches]

        def eager_run(steps, first=0):
            for t in range(first, first + steps):
                step_fns[t % R](act_rows[t % T])

        eager_run(W)
        barrier()
        # The step loop is launch-bound for small batches (one ~20 us kernel per step vs ~8 us of Python + driver per
        # launch), so it is captured once as a CUDA graph through the same public step() calls and replayed. K steps
        # are still exactly K kernel launches on the device. G = steps per graph: a multiple of R (every batch), at
        # most 128 and at most K, so that a short --steps run replays graphs too.
        # K <= 128: ONE graph of exactly K steps (a short --steps run, the driver's 20, is then a single graph launch and not
        # a graph plus a few eager launches with their host gaps); beyond that, graphs of G steps and one graph for the rest.
        graph, graph_rem, G, graph_error = None, None, 0, None
        if want_graph and K >= 1:
            G = K if K <= 128 else R * max(1, 128 // R if R <= 128 else 1)
            rem = K % G
            try:
                cap_stream = torch.cuda.Stream(device=dev)
                cap_stream.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(cap_stream):
                    eager_run(G)  # warm the capture stream
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph, stream=cap_stream):
                        eager_run(G)
                    if rem:
                        graph_rem = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(graph_rem, stream=cap_stream):
                            eager_run(rem, G * (K // G))
                torch.cuda.current_stream(dev).wait_stream(cap_stream)
                torch.cuda.synchronize()
            except Exception as exc:  # noqa: BLE001  (fall back to eager launches, and say so)
                graph, graph_rem, G, graph_error = None, None, 0, repr(exc)
                torch.cuda.synchronize()

        def run(steps, first=0):
            if graph is None:
                return eager_run(steps, first)
            for _ in range(steps // G):
                graph.replay()
            if steps % G:
                if graph_rem is not None and steps % G == K % G:
                    graph_rem.replay()
                else:
                    eager_run(steps % G, first)

        if graph is not None:
            run(G)
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        l0 = sum(b.launch_count for b in batches)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        h0 = time.perf_counter()
        run(K, W)
        host_enqueue_s = time.perf_counter() - h0
        ev1.record()
        barrier()
        clocks = sampler.stop()
        ms = max_over_ranks(ev0.elapsed_time(ev1))
        launches = sum(b.launch_count for b in batches) - l0
        if graph is not None:
            launches += (K // G) * G  # launches replayed by the graphs (each captured step() is one kernel node)
            if graph_rem is not None:
                launches += K % G
        # the batch that took the last timed step: graphs replay the steps t = 0 .. K-1 they were captured with (the
        # remainder graph its tail), eager launches continue from t = W
        last_batch = ((K if graph is not None else W + K) - 1) % R
        for b in batches:
            b.check_actions()
        # share of envs that were regenerated per timed step (pending flags after the run, averaged over the batches)
        pend = float(np.mean([float(b.get_state()["pending"].float().mean().item()) for b in batches]))
        res = {"env": env_id, "envs_per_gpu": n, "total_envs": total, "steps": K, "ms": ms, "ms_per_step": ms / K,
               "value": total * K / (ms * 1e-3), "launches": int(launches), "R": R, "ws": ws, "G": G, "graph": graph is not None,
               "graph_error": graph_error, "clocks": clocks, "host_enqueue_us_per_step": 1e6 * host_enqueue_s / K,
               "autoreset_fraction_per_step": pend, "last_batch": last_batch}
        achieved = ALGO_BYTES_PER_STEP * n / (ms / K * 1e-3) / 1e9
        res["achieved_gbs"], res["frac"] = achieved, achieved / peak
        return res, batches, (eager_run, act_rows, step_fns, T, R)

    # ---- headline ----
    n = args.envs_per_gpu
    total = n * world
    head, batches, (eager_run, act_rows, step_fns, T, R) = time_workload(args.env, n, K, W, rotate=args.rotate,
                                                                         sync_episodes=args.sync_episodes, want_graph=bool(args.graph))
    ms, launches = head["ms"], head["launches"]
    value = head["value"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, batches[head["last_batch"]])

    # per-launch events (perturbs the stream; reported, not used for the headline)
    kstep_ms = ms / K if launches == K else None
    kstep_ms_events = None
    try:
        for b in batches:
            b.profile_kernels(True)
        eager_run(min(K, 200), W)  # graph replays bypass the C-ABI call that records the events
        torch.cuda.synchronize()
        tot, cnt = 0.0, 0
        for b in batches:
            t_ms, c = b.kernel_time_ms()
            tot += t_ms; cnt += c
            b.profile_kernels(False)
        kstep_ms_events = tot / max(cnt, 1)
    except AttributeError:
        pass

    # ---- end to end through the host-buffer API: pinned host actions in, pinned host obs/reward/flags out ----
    Ke = max(1, args.e2e_steps)  # its own count: a short --steps run (the driver's 20) must not shorten this leg
    host_actions = torch.from_numpy(np.random.default_rng(4321 + rank).integers(0, 7, (min(Ke, 64), n)).astype(np.int32)).pin_memory()
    act_views = [host_actions[i] for i in range(host_actions.shape[0])]

    def e2e_run(fmt):
        """Ke synchronous step_host calls (pinned host actions in, host arrays out), three times; the median repetition."""
        # expander threads per rank: this rank's share of the host's cores; with several ranks on one host the calling
        # thread of every rank (it polls the copy events) needs a core of its own as well
        threads = max(1, min(cores_total // max(1, world), usable_cores()) - (1 if world > 1 else 0))
        for b in batches:
            b.set_host_format(fmt, threads)
        # every batch allocates its pinned staging on first use, and a handle's first 20 packed steps calibrate the
        # expander's store form (mg_abi.cu): keep both out of the timing
        for t in range(max(3, 22 * R)):
            batches[t % R].step_host(act_views[t % len(act_views)])
        reps = []
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            for t in range(Ke):
                batches[t % R].step_host(act_views[t % len(act_views)])
            torch.cuda.synchronize()
            reps.append(total * Ke / max_over_ranks(time.perf_counter() - t0))
        return float(np.median(reps)), reps

    e2e_value, e2e_reps = e2e_run(args.host_format)
    h2d = n * 4
    d2h = batches[0].host_d2h_bytes_per_step
    e2e_threads = batches[0].host_threads
    e2e_full = None
    if args.host_format != "full":  # the same loop with the arrays crossing PCIe as they are, for comparison
        v_full, reps_full = e2e_run("full")
        e2e_full = {"value": v_full, "repetitions": reps_full, "d2h_bytes_per_step": batches[0].host_d2h_bytes_per_step}

    # ---- the other BASELINE configs, the synchronised long run and the autoreset cost (one batch, L2-resident) ----
    configs, sync_wave, autoreset_cost, full_obs = [], None, None, None
    del batches, step_fns, eager_run
    torch.cuda.empty_cache()
    if not args.no_configs:
        for env_id, n_c in OTHER_CONFIGS:
            if env_id == args.env and n_c == n:
                continue
            r, bs, _ = time_workload(env_id, n_c, K, W, want_graph=bool(args.graph))
            tr, tr_src = load_traffic(env_id, n_c)
            configs.append({"env": env_id, "envs_per_gpu": n_c, "total_envs": r["total_envs"], "value": r["value"],
                            "ms_per_step": r["ms_per_step"], "frac": r["frac"], "achieved_gbs": r["achieved_gbs"], "steps": K,
                            "batches_cycled": r["R"], "launch": "graph" if r["graph"] else "eager",
                            "autoreset_fraction_per_step": r["autoreset_fraction_per_step"], "traffic": tr})
            if env_id == "MiniGrid-FourRooms-v0":  # K3 (FullyObsWrapper.observation) on the largest grid
                e = bs[0]
                out = torch.empty((n_c, e.width, e.height, 3), dtype=torch.uint8, device=dev)
                for _ in range(3):
                    e.full_obs(out)
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                for _ in range(20):
                    e.full_obs(out)
                a1.record()
                torch.cuda.synchronize()
                fo_ms = max_over_ranks(a0.elapsed_time(a1)) / 20
                fo_bytes = n_c * (e.width * e.height * 4 + 16)  # read W*H one-byte cell codes + the agent record, write 3*W*H
                full_obs = {"kernel": "k_full_obs (K3, FullyObsWrapper.observation)", "env": env_id, "envs_per_gpu": n_c,
                            "ms": fo_ms, "algorithmic_bytes_per_launch": fo_bytes, "achieved_gbs": fo_bytes / (fo_ms * 1e-3) / 1e9,
                            "frac": fo_bytes / (fo_ms * 1e-3) / 1e9 / peak}
            del bs
            torch.cuda.empty_cache()
        # one synchronised batch over >= 2 episodes: contains the truncation waves (every env truncates in the same step)
        spec_steps = MinigridVecEnv(args.env, 32, device=dev).max_steps
        Kl = int(min(max(2 * spec_steps + 64, 1024), 6000))
        rs, bs, _ = time_workload(args.env, n, Kl, W, rotate=1, sync_episodes=True, want_graph=bool(args.graph))
        del bs
        ro, bs, _ = time_workload(args.env, n, Kl, W, rotate=1, sync_episodes=True, autoreset="disabled", want_graph=bool(args.graph))
        del bs
        rd, bs, _ = time_workload(args.env, n, Kl, W, rotate=1, sync_episodes=False, want_graph=bool(args.graph))
        del bs
        torch.cuda.empty_cache()
        sync_wave = {"value": rs["value"], "ms_per_step": rs["ms_per_step"], "steps": Kl,
                     "note": "ONE batch reset together, never desynchronised: every env truncates in the same step every max_steps steps"}
        autoreset_cost = {"steps": Kl, "one_batch_l2_resident": True, "us_per_step_autoreset_disabled": 1e3 * ro["ms_per_step"],
                          "us_per_step_desynchronised": 1e3 * rd["ms_per_step"], "us_per_step_synchronised_waves": 1e3 * rs["ms_per_step"],
                          "desynchronised_over_disabled": rd["ms_per_step"] / ro["ms_per_step"],
                          "synchronised_over_disabled": rs["ms_per_step"] / ro["ms_per_step"]}

    tr, tr_src = load_traffic(args.env, n)
    roof = None
    if kstep_ms:
        roof = {"bound": "hbm", "kernel": "k_step (K1: transition + autoreset + gen_obs)", "achieved": head["achieved_gbs"], "peak": peak,
                "unit": "GB/s", "frac": head["frac"], "traffic": tr, "traffic_source": tr_src,
                "peak_source": peak_src, "kernel_ms": kstep_ms, "kernel_ms_per_launch_events": kstep_ms_events,
                "algorithmic_bytes_per_launch": ALGO_BYTES_PER_STEP * n}

    if rank == 0:
        line = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": make_config(args.env, n, world, args.sync_episodes),
            "run": {"l2": f"{head['R']} independent env batches cycled, working set {head['R'] * head['ws'] / 1e6:.0f} MB per GPU > 126 MB L2 (inputs larger than L2)",
                    "parallelism": f"env-sharded x{world}, no collective on the step path",
                    "launch": (f"CUDA graph replay, {head['G']} steps per graph" if head["graph"] else "eager launches"),
                    "graph_error": head["graph_error"], "numa": numa,
                    "autoreset_fraction_per_step": head["autoreset_fraction_per_step"]},
            "clocks": {k: head["clocks"][k] for k in ("sm_mhz", "sm_max_mhz", "reasons")},
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": Ke,
                    "format": args.host_format, "host_threads": e2e_threads, "repetitions": e2e_reps,
                    "protocol": "3 repetitions of `steps` synchronous step_host calls, the median", "full_format": e2e_full},
            "gpu_launches": int(launches),
            "host_enqueue_us_per_step": head["host_enqueue_us_per_step"],
        }
        if roof:
            line["roofline"] = roof
        if configs:
            line["configs"] = configs
        if full_obs:
            line["full_obs"] = full_obs
        if sync_wave:
            line["sync_wave"] = sync_wave
            line["autoreset_cost"] = autoreset_cost
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args)
            # BASELINE.json configs[0]: Empty-5x5, ONE env — CPU port beside the engine at n = 1 (launch-latency bound)
            e1 = MinigridVecEnv("MiniGrid-Empty-5x5-v0", 1, device=dev)
            e1.reset(seed=0)
            a1 = torch.randint(0, 7, (256, 1), device=dev, dtype=torch.int32)
            rows = [a1[i] for i in range(256)]
            for t in range(64):
                e1.step(rows[t])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for t in range(2000):
                e1.step(rows[t & 255])
            torch.cuda.synchronize()
            line["config1"] = {"env": "MiniGrid-Empty-5x5-v0", "envs": 1, "cpu_port_steps_per_s": config1_cpu(),
                               "engine_steps_per_s": 2000 / (time.perf_counter() - t0),
                               "note": "BASELINE.json configs[0]; one env is a launch-latency measurement on a GPU"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
