#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched gym-cellular step on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg4|cfg2|cfg3|cfg5] [--impl reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path (env.step for every env of the batch) over one batch of
synthetic random actions.  Rank 0 prints ONE JSON line (contract in the task statement):
  value      whole-job env-steps/s with actions already resident in HBM (device path, one kernel
             launch per step per GPU), timed with CUDA events, max over ranks
  e2e        the same metric through the host-facing call (numpy in, numpy out, H2D + kernel + D2H every
             step).  Cellular workloads use the packed wire format (gc_step_host_packed: one action word in,
             state word + reward + flag byte out per env); grid world the int8 one (gc_step_host)
  packed     device path of the packed layout (25 B per env-step instead of 3C + 20), with its own roofline
  roofline   algorithmic HBM bytes per launch / measured launch time, against MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle port (oracle/gc_oracle.c) on all host cores, bounded sample

Workloads (BASELINE.json configs; per-GPU batch fixed => weak scaling):
  cfg4 (default)  polarisation scaled to 16 cells x 4 levels, 2^24 envs per GPU (68 B/env-step,
                  1.14 GB per step: larger than the 126 MB L2, genuinely HBM-bound)
  cfg2            default polarisation env (3 cells x 3 levels), 65,536 envs (1.9 MB: L2-resident)
  cfg3            grid world, 2^20 envs, stochastic dispersal + fused auto-reset (27 MB: L2-resident)
  cfg5            mixed: per GPU 4M stochastic polarisation + 4M grid world envs (64M at 8 GPUs)
The default line also carries cfg2/cfg3/cfg5 results under "workloads" on 1 GPU, and cfg5 (the multi-GPU
config of BASELINE.json) at every N > 1, where the line also holds a shard check run on the hardware.

--dump-outputs DIR writes what the timed device path computed in its last step (see dump_outputs); the inputs
are seeded, so two builds run with the same arguments can be compared output for output.  The script writes
nothing into the tree it runs from.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

WORKLOADS = {
    # name: description, list of sub-batches (kind, fraction, kwargs), bytes per env-step
    "cfg4": dict(desc="polarisation 16 cells x 4 levels, 2^24 envs per GPU, deterministic (BASELINE config 4)",
                 n_envs=1 << 24, parts=[("cellular", 1.0, dict(n_cells=16, n_states=4))], l2_resident=False),
    "cfg2": dict(desc="polarisation 3 cells x 3 levels, 65,536 envs (BASELINE config 2)",
                 n_envs=1 << 16, parts=[("cellular", 1.0, dict(n_cells=3, n_states=3))], l2_resident=True),
    "cfg3": dict(desc="grid world, 2^20 envs, stochastic dispersal, auto-reset every 128 steps (BASELINE config 3)",
                 n_envs=1 << 20, parts=[("gridworld", 1.0, dict(max_episode_steps=128))], l2_resident=True),
    "cfg5": dict(desc="mixed sweep: half stochastic polarisation (Cells3ResetVDeadlock), half grid world, "
                      "2^23 envs per GPU, auto-reset every 128 steps (BASELINE config 5 = 2^26 envs on 8 GPUs)",
                 n_envs=1 << 23,
                 parts=[("cellular", 0.5, dict(n_cells=3, n_states=3, stochastic=True, max_episode_steps=128)),
                        ("gridworld", 0.5, dict(max_episode_steps=128))], l2_resident=False),
}
RING = 8            # pre-generated action buffers per sub-batch
DUMP_ENVS = 1 << 16  # --dump-outputs: envs per sub-batch in the written sample (every env of a smaller one)


def bytes_per_env_step(kind, n_cells):
    """Algorithmic HBM bytes of one env-step (SURVEY.md 8d): state r/w + action r (3C), t r/w (8),
    reward (4), index (4), terminated/truncated/unsafe/count (4)."""
    return 3 * n_cells + 20


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons while the timed region runs (NVML, else nvidia-smi)."""

    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4, "hw_power_brake": 0x80}
    # NVML queries go through the driver and slow concurrent kernel launches down: polled every 5 ms they
    # doubled the per-step time of the launch-bound workloads (15 us against 6-7 us per step)
    PERIOD_S = 0.05

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _poll_once(self):
        if self.nv is not None:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            try:
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                mask = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for name, bit in {**self.BAD, **self.NOTE}.items():
                if mask & bit:
                    self.reasons.add(name)
        else:
            out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm,"
                                  "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                                  "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True).stdout.strip()
            f = [x.strip() for x in out.split(",")]
            if len(f) >= 6:
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)

    def _run(self):
        # first sample 1 ms into the region: by then the launches of a short region are queued (an NVML query
        # takes a driver lock that concurrent kernel launches also need), and the kernels are running
        self._stop.wait(0.001)
        while not self._stop.is_set():
            try:
                self._poll_once()
            except Exception:
                pass
            self._stop.wait(self.PERIOD_S)

    def __enter__(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc):
        try:
            self._poll_once()           # at least one sample while the last kernels are in flight
        except Exception:
            pass
        self._stop.set()
        self._thread.join()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------
HOST_CHUNK_ENVS = 1 << 20


STATS_EVERY = 64     # steps per "iteration": the episode statistics are all-reduced once per iteration


def build_batches(workload, device, rank, n_override=None, packed=False):
    """Creates the vector envs of one rank and their pre-generated device action rings.  `packed`: the
    cellular sub-batches use the packed-word layout (PackedCellularVectorEnv)."""
    import torch
    from gym_cellular_b200 import CellularVectorEnv, PackedCellularVectorEnv
    w = WORKLOADS[workload]
    n_total = int(n_override or w["n_envs"])
    batches, offset = [], rank * n_total
    gen = torch.Generator(device=device).manual_seed(1234 + rank)
    for kind, frac, kw in w["parts"]:
        n = int(n_total * frac) // 16 * 16
        use_packed = packed and kind == "cellular"
        cls = PackedCellularVectorEnv if use_packed else CellularVectorEnv
        env = cls(kind=kind, num_envs=n, device=device, env_seed=0, env_id_offset=offset,
                  emit_side_effects=False, collect_stats=True,
                  # host-path chunk: 1 M envs on the int8 wire, 2 M on the packed wire (sweeps in profiles/r0*_tuning_log.md)
                  host_chunk_envs=HOST_CHUNK_ENVS * (2 if use_packed else 1), **kw)
        offset += n
        ring = []
        for _ in range(RING):
            if kind == "gridworld":
                # the reference sampler's distribution: exactly one jurisdiction names a position (grid_world.py:191-195)
                a = torch.full((2, env.ld), 4, dtype=torch.int8, device=device)
                jur = torch.randint(0, 2, (env.ld,), device=device, generator=gen)
                pos = torch.randint(0, 4, (env.ld,), device=device, generator=gen).to(torch.int8)
                a[0] = torch.where(jur == 0, pos, a[0])
                a[1] = torch.where(jur == 1, pos, a[1])
            else:
                a = torch.randint(0, env.n_actions, (env.n_cells, env.ld), dtype=torch.int8, device=device, generator=gen)
            if use_packed:                  # the same actions as packed words (2 bits per cell)
                w32 = torch.zeros(env.ld, dtype=torch.int32, device=device)
                w32[:n] = env.pack(a[:, :n])
                a = w32
            ring.append(a)
        batches.append(dict(env=env, ring=ring, kind=kind, n=n, packed=use_packed,
                            bytes=env.hbm_bytes_per_env_step if use_packed else bytes_per_env_step(kind, env.n_cells)))
    return batches



def time_device_path(batches, steps, warmup, dist, device, sampler_index, reducer=None):
    """Device path.  Every step of a sub-batch is one kernel launch on the sub-batch's own stream
    (independent sub-batches -- the mixed config 5 -- overlap tail and head); the launches are issued by
    gc_step_many, STATS_EVERY steps per foreign call, chained by programmatic dependent launch.  After
    every STATS_EVERY steps (one "iteration") the episode statistics are all-reduced over the ranks (NCCL,
    ordered in the stepping stream: see StatsReducer) -- INSIDE the timed region."""
    import torch
    main = torch.cuda.current_stream(device)
    streams = [main] if len(batches) == 1 else [torch.cuda.Stream(device=device) for _ in batches]
    slots = [[b["env"]._bind(a) for a in b["ring"]] for b in batches]
    for b, sl in zip(batches, slots):
        b["env"].prepare_step_many(sl)          # small shards: the graph gc_step_many replays, built before any timing

    def run(lo, hi):
        for s in streams:
            if s is not main:
                s.wait_stream(main)
        pending = None
        for c0 in range(lo, hi, STATS_EVERY):
            c1 = min(hi, c0 + STATS_EVERY)
            for b, sl, s in zip(batches, slots, streams):
                order = [sl[i % RING] for i in range(c0, min(c1, c0 + RING))]
                b["env"].step_many(order, c1 - c0, stream=s)
            if reducer is not None:
                for s in streams:
                    if s is not main:
                        main.wait_stream(s)
                if pending is not None:
                    pending.wait()
                pending = reducer.start(sum_stats(batches))
                for s in streams:
                    if s is not main:
                        s.wait_stream(main)
        for s in streams:
            if s is not main:
                main.wait_stream(s)
        if pending is not None:
            pending.wait()

    run(0, warmup)
    if reducer is not None:                 # (untimed) let NCCL finish whatever it sets up lazily for this collective
        for _ in range(3):
            reducer.start(sum_stats(batches)).wait()
    torch.cuda.synchronize(device)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(device)
    launches0 = sum(b["env"].launch_count for b in batches)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host = 0.0
    with ClockSampler(sampler_index) as clk:
        if dist is not None:
            # align the ranks ON THE DEVICE: the start event of every rank follows one NCCL all-reduce in the
            # stepping stream, which completes everywhere within microseconds -- a host-side barrier leaves the ranks
            # up to milliseconds apart, and with a collective inside the region every rank would pay for that skew
            # at the first reduction (8 GPUs, 200 steps: 218.8 instead of 195 us per step)
            dist.all_reduce(torch.zeros(1, device=device))
        else:
            # one rank: a ~100 us spin kernel plays the same role -- the start event and the first step launches are
            # queued behind it, so the region starts with the first step kernel already in the queue instead of with
            # the host latency of issuing it (20-50 us of Python: 1-2 % of a 20-step region)
            torch.cuda._sleep(200_000)
        start.record(main)
        t0 = time.perf_counter()
        run(warmup, warmup + steps)
        t_host = time.perf_counter() - t0
        stop.record(main)
        stop.synchronize()
    ms = start.elapsed_time(stop)
    launches = sum(b["env"].launch_count for b in batches) - launches0
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    torch.cuda.synchronize(device)
    return ms, launches, clk.summary(), 1e6 * t_host / max(launches, 1)


def dump_outputs(batches, out_dir):
    """What the last step handed its caller -- observation, reward, terminated, truncated and the infos unsafe,
    count, time_step and tabular_state -- for a fixed, seeded sample of each sub-batch's envs, as float64 arrays
    out_dir/<kind>_<name>.npy (at most 13 MB per sub-batch); <kind>_env_ids.npy holds the sampled env indices."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for b in batches:
        env, n = b["env"], b["n"]
        ids = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ENVS), replace=False))
        sel = torch.from_numpy(ids).to(env.device)
        infos = env._v_infos
        out = {"env_ids": ids, "state": env.state[:, sel], "reward": env._v_reward[sel], "terminated": env._v_term[sel],
               "truncated": env._v_trunc[sel], "unsafe": infos["unsafe"][sel], "count": infos["count"][sel],
               "time_step": infos["time_step"][sel], "tabular_state": env.tabular_state()[sel]}
        for name, a in out.items():
            a = a.cpu().numpy() if torch.is_tensor(a) else a
            np.save(os.path.join(out_dir, f"{b['kind']}_{name}.npy"), a.astype(np.float64))


def sum_stats(batches):
    import torch
    return torch.stack([b["env"]._stats for b in batches]).sum(0)


def time_graph_path(batches, steps, device):
    """Launch-bound batch sizes: RING captured steps per CUDA graph, replayed steps/RING times."""
    import torch
    graphs = [b["env"].capture_steps(b["ring"]) for b in batches]
    reps = max(1, steps // RING)
    for g in graphs:
        g.replay()
    torch.cuda.synchronize(device)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        for g in graphs:
            g.replay()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop), reps * RING


def measure_pcie(device, dist=None, nbytes=1 << 27):
    """Pinned-memory copy bandwidth of this box (GB/s per GPU): each direction alone and both at once --
    the ceiling of the e2e figure, which moves h2d + d2h bytes per step.  With several ranks all of them
    measure at the same time (barrier first), so the figure is the per-GPU share of the host's aggregate."""
    import torch
    h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_in = torch.empty(nbytes, dtype=torch.uint8, device=device)
    d_out = torch.empty(nbytes, dtype=torch.uint8, device=device)
    s1, s2 = torch.cuda.Stream(device=device), torch.cuda.Stream(device=device)

    def run(h2d, d2h, reps=4):
        torch.cuda.synchronize(device)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for _ in range(reps):
            if h2d:
                with torch.cuda.stream(s1):
                    d_in.copy_(h_in, non_blocking=True)
            if d2h:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_out, non_blocking=True)
        torch.cuda.synchronize(device)
        return reps * nbytes / (time.perf_counter() - t0) / 1e9
    run(True, True, 1)
    out = {"h2d_gbs": round(run(True, False), 1), "d2h_gbs": round(run(False, True), 1)}
    out["duplex_gbs_each"] = round(run(True, True), 1)
    if dist is not None:
        t = torch.tensor([out["h2d_gbs"], out["d2h_gbs"], out["duplex_gbs_each"]], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        out["all_ranks_concurrent_sum"] = {"h2d_gbs": round(float(t[0]), 1), "d2h_gbs": round(float(t[1]), 1),
                                           "duplex_gbs_each": round(float(t[2]), 1)}
    return out


def time_host_path(batches, steps, warmup, dist, device):
    """End to end through the host-facing call: pinned numpy actions in, numpy results out."""
    import torch
    host_rings = []
    for b in batches:
        ring = [b["ring"][i].cpu().pin_memory() for i in range(2)]
        host_rings.append([(t, t.numpy()[:b["n"]] if b["packed"] else t.numpy()[:, :b["n"]]) for t in ring])
    h2d = sum(b["env"].host_bytes_per_env_step[0] * b["n"] for b in batches)
    d2h = sum(b["env"].host_bytes_per_env_step[1] * b["n"] for b in batches)

    def one(i):
        sink = 0.0
        for b, hr in zip(batches, host_rings):
            obs, rew, term, trunc, info = b["env"].step(hr[i % 2][1])
            sink += float(rew[0])
        return sink
    for i in range(warmup):
        one(i)
    torch.cuda.synchronize(device)
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        one(i)
    torch.cuda.synchronize(device)
    el = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([el], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        el = float(t.item())
    return el, h2d, d2h


# ------------------------------------------------------------------------------------------------
def oracle_envs(workload, n_sample):
    """The CPU oracle configured like `workload` (bench cpu_baseline / --impl reference legs only)."""
    import numpy as np
    from oracle import oracle as O
    out = []
    rng = np.random.default_rng(1234)
    for kind, frac, kw in WORKLOADS[workload]["parts"]:
        n = max(16, int(n_sample * frac))
        if kind == "gridworld":
            env = O.OracleEnv(kind="gridworld", n_envs=n, seed=0, max_episode_steps=kw.get("max_episode_steps", 0))
            a = np.full((2, n), 4, np.int8)
            a[rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
        else:
            st = kw.get("stochastic", False)
            env = O.OracleEnv(n_envs=n, n_cells=kw["n_cells"], n_states=kw["n_states"], noise=st, rng_episodic=True,
                              reward="nonlinear_rp" if st else "right_polarizing", seed=0,
                              max_episode_steps=kw.get("max_episode_steps", 0))
            a = rng.integers(0, kw["n_states"], size=(kw["n_cells"], n)).astype(np.int8)
        out.append((env, a, n))
    return out


def time_oracle(envs, steps, warmup, threads):
    for _ in range(warmup):
        for env, a, n in envs:
            env.step_parallel(a, threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        for env, a, n in envs:
            env.step_parallel(a, threads)
    el = time.perf_counter() - t0
    return sum(n for _, _, n in envs) * steps / el, el


ORACLE_REPS = 3


def oracle_rate(workload, steps, warmup, budget_s):
    """The C oracle port on all host cores, the same sampling for the cpu_baseline leg and the reference
    arm: a calibration pass sizes the sample so that one repetition of (warmup + steps) steps takes about
    budget_s / ORACLE_REPS seconds; ORACLE_REPS repetitions, the MEDIAN rate is reported (the spread between
    repetitions on one box was 40 % in round 1: thread placement / first touch)."""
    threads = os.cpu_count() or 1
    rate, _ = time_oracle(oracle_envs(workload, 1 << 16), 2, 1, threads)          # calibration
    per_rep = budget_s / ORACLE_REPS
    n_sample = int(min(1 << 22, max(1 << 12, rate * per_rep / max(steps + warmup, 1))))
    envs = oracle_envs(workload, n_sample)
    reps = sorted(time_oracle(envs, steps, warmup if i == 0 else 0, threads) for i in range(ORACLE_REPS))
    rate, el = reps[len(reps) // 2]
    n = sum(n for _, _, n in envs)
    return {"rate": rate, "seconds": el, "envs": n, "threads": threads, "steps": steps,
            "reps": [round(r) for r, _ in reps]}


def python_port_rate(workload):
    """What the reference's own execution model (one Python object per env) costs on this box: the
    pure-Python port oracle/pyport.py in a fresh process (fork pool over all cores).  Context only."""
    part = next((kw for kind, _, kw in WORKLOADS[workload]["parts"] if kind == "cellular"), None)
    if part is None:
        return None
    try:
        out = subprocess.run([sys.executable, "-B", "-m", "oracle.pyport", "--envs", "64", "--steps", "150", "--cells",
                              str(part["n_cells"]), "--levels", str(part["n_states"])], cwd=REPO, capture_output=True,
                             text=True, timeout=120).stdout.strip().splitlines()[-1]
        return json.loads(out)
    except Exception as exc:
        return {"error": type(exc).__name__}


def _pyport_env_fn(n_cells, n_levels):
    """env_fn for the AsyncVectorEnv baseline: the pure-Python port of the reference step with the reference's
    spaces attached (cells3states3actions3.py:65-89)."""
    def make():
        from gym_cellular_b200._gym import gym
        from oracle.pyport import PolarisationEnv
        env = PolarisationEnv(n_cells, n_levels)
        sp = gym.spaces
        env.observation_space = sp.Tuple([sp.Discrete(n_levels) for _ in range(n_cells)])
        env.action_space = sp.Tuple([sp.Discrete(n_levels) for _ in range(n_cells)])
        return env
    return make


def async_vector_env_rate(n_cells, n_levels, envs_per_worker, steps):
    """The CPU baseline BASELINE.json names: the reference's step loop (its pure-Python port -- the reference
    itself cannot travel to the GPU box) under gymnasium.vector.AsyncVectorEnv (the multiprocessing
    stand-in of gym_cellular_b200/compat when gymnasium is absent): one worker per core, one pipe round trip
    per step, num_envs = workers x envs_per_worker."""
    import numpy as np
    from gym_cellular_b200._gym import gym
    workers = os.cpu_count() or 1
    n = workers * envs_per_worker
    fns = [_pyport_env_fn(n_cells, n_levels) for _ in range(n)]
    try:
        env = gym.vector.AsyncVectorEnv(fns, shared_memory=False, envs_per_worker=envs_per_worker)
        layout = f"{workers} workers x {envs_per_worker} envs"
    except TypeError:                      # real gymnasium: one process per env
        n = workers
        env = gym.vector.AsyncVectorEnv(fns[:n], shared_memory=False)
        layout = f"{workers} workers x 1 env"
    try:
        env.reset()
        rng = np.random.default_rng(0)
        acts = [tuple(rng.integers(0, n_levels, n) for _ in range(n_cells)) for _ in range(8)]
        for i in range(3):
            env.step(acts[i % 8])
        t0 = time.perf_counter()
        for i in range(steps):
            env.step(acts[i % 8])
        el = time.perf_counter() - t0
    finally:
        env.close()
    return {"value": n * steps / el, "unit": "env-steps/s", "layout": layout, "steps": steps,
            "shape": f"{n_cells} cells x {n_levels} levels", "harness": gym.vector.AsyncVectorEnv.__module__}


def config1_rates():
    """BASELINE config 1: Cells3States3Actions3-v0, ONE env, 10 000 random-action steps.  The reference's
    Python cannot travel to the GPU box; its pure-Python port is timed in-process (the reference itself:
    2.4e5 steps/s on one core, BASELINE.md).  Also the drop-in single-env class of this package through
    gymnasium.make, whose step() is one N = 1 kernel launch plus a device-to-host read."""
    import numpy as np
    from oracle.pyport import PolarisationEnv
    out = {}
    rng = np.random.default_rng(0)
    acts = [tuple(int(x) for x in rng.integers(0, 3, 3)) for _ in range(10000)]
    env = PolarisationEnv(3, 3)
    env.reset()
    t0 = time.perf_counter()
    for a in acts:
        env.step(a)
    out["python_port_one_env"] = {"value": len(acts) / (time.perf_counter() - t0), "unit": "env-steps/s", "steps": len(acts)}
    try:
        import gym_cellular_b200  # noqa: F401
        from gym_cellular_b200._gym import gym
        env = gym.make("gym_cellular/Cells3States3Actions3-v0")
        env.reset()
        for a in acts[:50]:
            env.step(a)
        t0 = time.perf_counter()
        for a in acts[:2000]:
            env.step(a)
        out["native_single_env_drop_in"] = {"value": 2000 / (time.perf_counter() - t0), "unit": "env-steps/s", "steps": 2000,
                                            "note": "gymnasium.make id, one N=1 kernel launch + D2H per step"}
        env.close()
    except Exception as exc:            # pragma: no cover
        out["native_single_env_drop_in"] = {"error": f"{type(exc).__name__}: {exc}"}
    return out


def cpu_baseline(workload, budget_s=18.0):
    r = oracle_rate(workload, 8, 1, budget_s)
    out = {"value": r["rate"], "unit": "env-steps/s", "cores": r["threads"], "kind": "port",
           "sample": f"C oracle (oracle/gc_oracle.c), {r['envs']} envs x {r['steps']} steps of {workload}, {r['threads']} threads, "
                     f"median of {ORACLE_REPS} repetitions {r['reps']} ({r['seconds']:.1f} s each)",
           "python_port": python_port_rate(workload)}
    part = next((kw for kind, _, kw in WORKLOADS[workload]["parts"] if kind == "cellular"), None)
    try:
        out["async_vector_env"] = {"config1_shape": async_vector_env_rate(3, 3, 64, 60)}
        if part is not None and (part["n_cells"], part["n_states"]) != (3, 3):
            out["async_vector_env"]["bench_shape"] = async_vector_env_rate(part["n_cells"], part["n_states"], 16, 30)
    except Exception as exc:            # pragma: no cover - depends on the box
        out["async_vector_env"] = {"error": f"{type(exc).__name__}: {exc}"}
    out["config1"] = config1_rates()
    return out


def workload_config(workload, world):
    """The `config` object of the JSON line: a function of the workload and the world size only, so that
    the native and the reference arm print the same one."""
    w = WORKLOADS[workload]
    return {"workload": workload, "description": w["desc"], "envs_per_gpu": w["n_envs"] // 16 * 16,
            "global_envs": w["n_envs"] // 16 * 16 * world,
            "parallelism": f"env-sharded x{world}, NCCL all-reduce of episode statistics once per iteration "
                           f"({STATS_EVERY} steps), in the stepping stream, inside the timed region",
            "l2": "per-step working set larger than L2" if not w["l2_resident"]
                  else "working set is L2-resident (launch-bound, not an HBM measurement)",
            "actions": f"ring of {RING} pre-generated buffers, uniform random"}


def run_reference_arm(args, workload):
    """--impl reference: the CPU implementation on the host cores (the reference is pure Python and
    cannot travel to the GPU box; the oracle port stands in, see DESIGN.md).  Each step is a bounded sample
    of the workload (cpu_baseline.sample says how many envs); same sampling as the native arm's
    cpu_baseline leg."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = oracle_rate(workload, args.steps, args.warmup, 60.0)
    sample = (f"C oracle (oracle/gc_oracle.c), {r['envs']} envs per step of {workload}, {r['threads']} threads, "
              f"median of {ORACLE_REPS} repetitions {r['reps']}")
    line = {"impl": "reference", "metric": "env-steps/sec", "value": r["rate"], "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8/int32 state, f32 reward",
            "data": "synthetic", "config": workload_config(workload, args.gpus),
            "cpu_baseline": {"value": r["rate"], "unit": "env-steps/s", "cores": r["threads"], "kind": "port", "sample": sample},
            "e2e": {"value": r["rate"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def bind_near_gpu(device):
    """Pin this rank's host threads (and hence its pinned staging buffers, by first touch) to the CPUs
    of the GPU's NUMA node; matters for the host path when 8 ranks share the host.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bdf = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(device.index)).busId
        bdf = bdf.decode() if isinstance(bdf, bytes) else bdf
        bdf = bdf.lower()
        if len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]
        path = f"/sys/bus/pci/devices/{bdf}/local_cpulist"
        cpus = set()
        for part in open(path).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"{len(allowed)} cpus of the GPU's NUMA node"
        return "no local cpu allowed"
    except Exception as exc:           # pragma: no cover - depends on the box
        return f"unbound ({type(exc).__name__})"


def measured_peak():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload):
    """dram read+write bytes per step from the committed ncu capture, if any (profiles/traffic.json)."""
    path = os.path.join(REPO, "profiles", "traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path)).get(workload)
        except Exception:
            return None
    return None


def roofline_of(workload, batches, step_s, tag=None, resident_state=False):
    # resident_state: the many-step kernel keeps state and episode step in registers between two steps, so a step
    # moves C + 4 bytes per env less than SURVEY 8d's figure (it still writes both at every step)
    def not_reread(b):                       # state + t: one packed word + 4, or C bytes + 4
        return 8 if (b["packed"] and b["kind"] == "cellular") else b["env"].n_cells + 4
    alg_bytes = sum((b["bytes"] - (not_reread(b) if resident_state else 0)) * b["n"] for b in batches)   # per step, per rank
    n_rank = sum(b["n"] for b in batches)
    peak, peak_src = measured_peak()
    traffic = ncu_traffic(tag or workload)
    static = WORKLOADS[workload]["l2_resident"]
    # A working set below the 126 MB L2 stays there from step to step (ncu's DRAM bytes for such a launch are the
    # cold-cache reads of its replay mode, not steady-state traffic); above it, the measured traffic says how much
    # of the algorithmic bytes actually reaches DRAM
    dram_share = None if not isinstance(traffic, (int, float)) else traffic / alg_bytes
    if alg_bytes < 100e6:
        resident = True
    elif dram_share is None:
        resident = static
    else:
        resident = "partly" if dram_share < 0.75 else False
    return {"bound": "hbm", "achieved": alg_bytes / step_s / 1e9, "peak": peak, "unit": "GB/s",
            "frac": alg_bytes / step_s / 1e9 / peak, "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg_bytes // len(batches), "bytes_per_env_step": alg_bytes / n_rank,
            "kernels_per_step": len(batches),
            "dram_bytes_over_algorithmic": None if dram_share is None else round(dram_share, 3),
            "l2_resident": resident}


def bench_workload(workload, steps, warmup, dist, device, world, rank, e2e_steps, side=True, dump_dir=None):
    """`side` = also time the CUDA-graph and fused-rollout variants (single process only).  `dump_dir`: where rank 0
    writes the outputs of the timed path's last step (dump_outputs)."""
    import torch
    from gym_cellular_b200.distributed import StatsReducer
    batches = build_batches(workload, device, rank)
    n_rank = sum(b["n"] for b in batches)
    reducer = StatsReducer()
    # the per-iteration all-reduce of the statistics belongs to the multi-GPU path; one rank has nothing to reduce
    in_loop = reducer if dist is not None else None
    ms, launches, clocks, host_us = time_device_path(batches, steps, warmup, dist, device, device.index, in_loop)
    if dump_dir is not None and rank == 0:          # before anything below steps these envs again
        dump_outputs(batches, dump_dir)
    # Small shards: gc_step_many runs the bound steps of a call inside ONE kernel (state in registers between the steps,
    # every per-step output written at every step; include/gym_cellular_b200.h).  The same loop is then timed with one
    # launch per step as well (GC_B200_STEP_MANY_FUSED=0, read by the library at every call) and reported beside it.
    sep_res, sep_steps = None, 0
    if launches < steps * len(batches):
        os.environ["GC_B200_STEP_MANY_FUSED"] = "0"
        try:
            s_ms, s_launches, _, s_host_us = time_device_path(batches, steps, warmup, dist, device, device.index, in_loop)
        finally:
            os.environ.pop("GC_B200_STEP_MANY_FUSED", None)
        sep_steps = steps + warmup
        sep_res = {"value": world * n_rank * steps / (s_ms * 1e-3), "ms_per_step": s_ms / steps, "gpu_launches": s_launches * world,
                   "host_us_per_launch": round(s_host_us, 2),
                   "roofline_frac": roofline_of(workload, batches, s_ms * 1e-3 / steps)["frac"],
                   "note": "one kernel launch per step (programmatic dependent launch, cached graph replay)"}
    single = dist is None and side
    graph_res = None
    if WORKLOADS[workload]["l2_resident"] and single:
        g_ms, g_steps = time_graph_path(batches, steps, device)
        graph_res = {"value": n_rank * g_steps / (g_ms * 1e-3), "ms_per_step": g_ms / g_steps,
                     "steps_per_graph": RING}
    ro_res = None
    if single:              # K-step fused rollout (random actions generated in the kernel)
        K = 64
        main = torch.cuda.current_stream(device)
        ro_streams = [main] if len(batches) == 1 else [torch.cuda.Stream(device=device) for _ in batches]

        def rollouts(reps):                # independent sub-batches on one stream each, as in the step path
            for s in ro_streams:
                if s is not main:
                    s.wait_stream(main)
            for _ in range(reps):
                for b, s in zip(batches, ro_streams):
                    with torch.cuda.stream(s):
                        b["env"].rollout(K)
            for s in ro_streams:
                if s is not main:
                    main.wait_stream(s)
        rollouts(1)
        torch.cuda.synchronize(device)
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 4
        r0.record(main)
        rollouts(reps)
        r1.record(main)
        r1.synchronize()
        ro_res = {"value": n_rank * K * reps / (r0.elapsed_time(r1) * 1e-3), "steps_per_launch": K,
                  "note": "fused rollout: state in registers, actions generated in-kernel (not per-step step())"}
    # episode statistics over all ranks: the path's only collective; totals must add up exactly
    totals = reducer.start(sum_stats(batches)).result()
    expect = world * n_rank * (steps + warmup + sep_steps + (g_steps + RING if graph_res else 0) + (K * (reps + 1) if ro_res else 0))
    stats_ok = totals["env_steps"] == expect
    step_s = ms * 1e-3 / steps
    res = {
        "value": world * n_rank * steps / (ms * 1e-3),
        "ms_per_step": ms / steps,
        "envs_per_gpu": n_rank,
        "gpu_launches": launches * world,
        "host_us_per_launch": round(host_us, 2),
        "clocks": clocks,
        "roofline": roofline_of(workload, batches, step_s, resident_state=sep_res is not None),
        "episode_stats": dict(totals, env_steps_expected=expect, consistent=stats_ok),
        "cuda_graph": graph_res,
        "fused_rollout": ro_res,
        "steps_per_launch": round(steps * len(batches) / max(launches, 1), 1),
        "separate_launches": sep_res,
    }
    if sep_res is not None:
        # the dominant kernel is the many-step kernel: its launch moves the algorithmic bytes of all its steps
        spl = steps * len(batches) / max(launches, 1)
        res["roofline"]["algorithmic_bytes_per_step"] = res["roofline"]["algorithmic_bytes_per_launch"]
        res["roofline"]["algorithmic_bytes_per_launch"] = int(res["roofline"]["algorithmic_bytes_per_launch"] * spl)
        res["roofline"]["kernels_per_step"] = round(len(batches) / spl, 4)
        # DRAM bytes of one launch of the many-step kernel (ncu capture of a 64-step launch, profiles/r02_kernel_*_many.md)
        many_traffic = ncu_traffic(workload + "_many")
        res["roofline"]["traffic"] = many_traffic
        res["roofline"]["dram_bytes_over_algorithmic"] = (
            None if not isinstance(many_traffic, (int, float)) else
            round(many_traffic / (res["roofline"]["algorithmic_bytes_per_step"] * STATS_EVERY), 3))
        res["roofline"]["bytes_note"] = ("state and t are read once per launch, not once per step: the step's algorithmic bytes are "
                                         "SURVEY 8d's 3C + 20 minus C + 4")
        res["step_many"] = ("bound steps of one gc_step_many call run inside ONE kernel (shards <= 2^21 envs): state and episode "
                            "step in registers between the steps, actions read and every per-step output written at every step; "
                            "bit-identical to separate launches (tests/test_gpu_many.py); `separate_launches` = the same loop with "
                            "one launch per step")
    for b in batches:
        b["env"].close()
    del batches
    torch.cuda.empty_cache()

    # ---- packed layout: device path (cellular sub-batches as packed words) and the e2e host path ---------
    has_cell = any(kind == "cellular" for kind, _, _ in WORKLOADS[workload]["parts"])
    pbatches = build_batches(workload, device, rank, packed=True)
    if has_cell:
        p_ms, p_launches, _, p_host_us = time_device_path(pbatches, steps, warmup, dist, device, device.index, in_loop)
        res["packed"] = {"value": world * n_rank * steps / (p_ms * 1e-3), "ms_per_step": p_ms / steps,
                         "gpu_launches": p_launches * world, "host_us_per_launch": round(p_host_us, 2),
                         "layout": "cellular sub-batches: one 32-bit word per env for the state, one for the action "
                                   "(2 bits per cell), reward + one flag byte out",
                         "steps_per_launch": round(steps * len(pbatches) / max(p_launches, 1), 1),
                         "roofline": roofline_of(workload, pbatches, p_ms * 1e-3 / steps, tag=workload + "_packed",
                                                 resident_state=p_launches < steps * len(pbatches))}
    el_host, h2d, d2h = time_host_path(pbatches, e2e_steps, 2, dist, device)
    res["e2e"] = {"value": world * n_rank * e2e_steps / el_host, "unit": "env-steps/s",
                  "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world, "steps": e2e_steps,
                  "ms_per_step": 1e3 * el_host / e2e_steps,
                  "wire": "packed words for the cellular sub-batches (4 B in, 9 B out per env-step; state word = "
                          "tabular index at 4 levels), int8 layout for grid world (2 B in, 13 B out); the constant "
                          "`terminated` flag is not copied",
                  "link_gbs_per_gpu": {"h2d": h2d / el_host * e2e_steps / 1e9, "d2h": d2h / el_host * e2e_steps / 1e9}}
    for b in pbatches:
        b["env"].close()
    del pbatches
    torch.cuda.empty_cache()
    return res


def shard_check(dist, device, rank, world):
    """On the hardware, over NCCL: rank r re-steps the first 65,536 envs of rank (r+1) % N's shard of the
    mixed config (stochastic polarisation + grid world, Philox keyed by GLOBAL env id) on its own GPU and
    the CRCs are compared with the owner's -- results must not depend on which GPU owns an env."""
    import zlib
    import torch
    from gym_cellular_b200 import CellularVectorEnv
    n, T = 1 << 16, 6
    n_total = WORKLOADS["cfg5"]["n_envs"]

    def crc_of(owner):
        gen = torch.Generator(device=device).manual_seed(777 + owner)
        offset, h = owner * n_total, 0
        for kind, frac, kw in WORKLOADS["cfg5"]["parts"]:
            env = CellularVectorEnv(kind=kind, num_envs=n, device=device, env_seed=0, env_id_offset=offset,
                                    emit_side_effects=False, **kw)
            offset += int(n_total * frac) // 16 * 16
            for _ in range(T):
                if kind == "gridworld":
                    a = torch.full((2, n), 4, dtype=torch.int8, device=device)
                    jur = torch.randint(0, 2, (n,), device=device, generator=gen)
                    pos = torch.randint(0, 4, (n,), device=device, generator=gen).to(torch.int8)
                    a[0] = torch.where(jur == 0, pos, a[0])
                    a[1] = torch.where(jur == 1, pos, a[1])
                else:
                    a = torch.randint(0, env.n_actions, (env.n_cells, n), dtype=torch.int8, device=device, generator=gen)
                env.step_device(a)
                for t in (env.state, env._index[:n], env._reward[:n], env._unsafe[:n], env._count[:n]):
                    h = zlib.crc32(t.cpu().numpy().tobytes(), h)
            env.close()
        return h
    mine, neighbour = crc_of(rank), crc_of((rank + 1) % world)
    t = torch.tensor([mine, neighbour], dtype=torch.int64, device=device)
    allv = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(allv, t)
    ok = all(int(allv[r][1]) == int(allv[(r + 1) % world][0]) for r in range(world))
    distinct = len({int(v[0]) for v in allv}) == world            # different shards really differ
    return {"result": "ok" if (ok and distinct) else "MISMATCH", "envs_per_rank_checked": 2 * n, "steps": T,
            "what": "rank r re-steps the head of rank (r+1)%N's shard (env_id_offset); CRC32 of state/index/reward/flags all-gathered"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the cfg2/cfg3/cfg5 side measurements")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side", action="store_true",
                    help="skip the CUDA-graph and fused-rollout side measurements (profiling runs: launch lists)")
    ap.add_argument("--host-chunk", type=int, default=None, help="envs per chunk of the host (e2e) path")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the timed path's last step as DIR/<name>.npy (rank 0; a fixed sample "
                         f"of {DUMP_ENVS} envs per sub-batch)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.host_chunk:
        global HOST_CHUNK_ENVS
        HOST_CHUNK_ENVS = args.host_chunk
    # nothing is written into the tree, which may be read-only: no bytecode caches, and a CPU oracle that is
    # missing or older than its source is compiled into a temporary directory
    sys.dont_write_bytecode = True
    from oracle import oracle as O
    oracle_dir = tempfile.TemporaryDirectory(prefix="gc_bench_oracle_")
    O.build_dir = oracle_dir.name

    if args.impl == "reference":
        run_reference_arm(args, args.workload)
        return

    # stdout carries the one JSON line and nothing else: libraries that write to file descriptor 1 behind
    # Python's back (NCCL prints its version banner there, and its log at NCCL_DEBUG=INFO) are sent to
    # stderr by pointing descriptor 1 at it; Python's own sys.stdout keeps the original descriptor
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    affinity = bind_near_gpu(device) if world > 1 else "single rank: unbound"
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    e2e_steps = max(3, min(args.steps, 10))
    main_res = bench_workload(args.workload, args.steps, args.warmup, dist, device, world, rank, e2e_steps,
                              side=not args.no_side, dump_dir=args.dump_outputs)
    # side workloads, over the same --steps: the launch-bound configs 2 and 3 on one GPU, the mixed multi-GPU
    # config 5 at every N (a run of a few steps times the launch-bound ones mostly filling the pipeline)
    extra = {}
    if not args.no_extra:
        for w in (("cfg2", "cfg3", "cfg5") if world == 1 else ("cfg5",)):
            if w != args.workload:
                r = bench_workload(w, args.steps, args.warmup, dist, device, world, rank, e2e_steps, side=not args.no_side)
                extra[w] = {"description": WORKLOADS[w]["desc"], "value": r["value"], "ms_per_step": r["ms_per_step"],
                            "steps": args.steps, "host_us_per_launch": r["host_us_per_launch"],
                            "roofline_frac": r["roofline"]["frac"], "achieved_gbs": r["roofline"]["achieved"],
                            "traffic": r["roofline"]["traffic"],
                            "dram_bytes_over_algorithmic": r["roofline"]["dram_bytes_over_algorithmic"],
                            "l2_resident": r["roofline"]["l2_resident"], "e2e": r["e2e"]["value"],
                            "e2e_bytes_per_step": [r["e2e"]["h2d_bytes_per_step"], r["e2e"]["d2h_bytes_per_step"]],
                            "kernels_per_step": r["roofline"]["kernels_per_step"], "cuda_graph": r["cuda_graph"],
                            "steps_per_launch": r["steps_per_launch"], "separate_launches": r["separate_launches"],
                            "step_many": r.get("step_many"),
                            "fused_rollout": r["fused_rollout"], "episode_stats_consistent": r["episode_stats"]["consistent"],
                            "packed": None if "packed" not in r else
                            {k: r["packed"][k] for k in ("value", "ms_per_step", "steps_per_launch")} | {"roofline_frac": r["packed"]["roofline"]["frac"],
                                                                                    "bytes_per_env_step": r["packed"]["roofline"]["bytes_per_env_step"]}}
    pcie = measure_pcie(device, dist)
    check = shard_check(dist, device, rank, world) if dist is not None else None
    if rank == 0:
        e2e = dict(main_res["e2e"], pcie_measured=pcie)
        dup, d2h_bw = pcie.get("duplex_gbs_each"), pcie.get("d2h_gbs")
        if dup and d2h_bw:
            # ideal overlapped schedule on this box's link (per GPU, all ranks busy): both directions at the duplex
            # rate until the actions are in, the rest of the results at the device-to-host rate alone
            h2d_b, d2h_b = e2e["h2d_bytes_per_step"] / world, e2e["d2h_bytes_per_step"] / world
            t1 = h2d_b / (dup * 1e9)
            ideal = t1 + max(0.0, d2h_b - dup * 1e9 * t1) / (d2h_bw * 1e9)
            e2e["link_ideal_ms_per_step"] = 1e3 * ideal
            e2e["link_ceiling_env_steps_per_s"] = world * main_res["envs_per_gpu"] / ideal
            e2e["frac_of_link_ceiling"] = e2e["value"] / e2e["link_ceiling_env_steps_per_s"]
        line = {
            "metric": "env-steps/sec", "value": main_res["value"], "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8/int32 state, f32 reward",
            "data": "synthetic",
            "config": workload_config(args.workload, world),
            "host_affinity": affinity,
            "e2e": e2e,
            "gpu_launches": main_res["gpu_launches"], "host_us_per_launch": main_res["host_us_per_launch"],
            "clocks": main_res["clocks"],
            "roofline": main_res["roofline"], "packed": main_res.get("packed"),
            "episode_stats": main_res["episode_stats"],
            "fused_rollout": main_res["fused_rollout"], "cuda_graph": main_res["cuda_graph"],
            "steps_per_launch": main_res["steps_per_launch"],
        }
        if main_res["separate_launches"] is not None:
            line["separate_launches"], line["step_many"] = main_res["separate_launches"], main_res["step_many"]
        if check is not None:
            line["shard_check"] = check["result"]
            line["shard_check_detail"] = check
        if extra:
            line["workloads"] = extra
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.workload)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
