"""Experience counts on one GPU: `collect_counts` against the rollout floor and against `collect` followed by the torch
aggregation a model-based tabular agent runs on its record, K = 64 steps per call, on the README's three collect
workloads.  Arms are timed in alternating rounds; each arm reports the median time per call over the rounds and the
spread (min, max).  Writes one JSON file (the card's name and power limit are read in the same run).

    python scripts/count_bench.py [--out profiles/r04_count_bench.json] [--k 64] [--rounds 5] [--reps 5]

Tables: the joint visits / next / reward_q24 / unsafe tables where they exist (config 2: 27 x 27 states and actions,
grid world: 400 x 25), only the per-cell N_c(s_c, a_c, s'_c) for 16 x 4 (4^16 states have no joint table).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import torch                                                          # noqa: E402

import gym_cellular_b200 as B                                         # noqa: E402

WORKLOADS = {
    "cfg2": ("polarisation 3 cells x 3 levels, stochastic, 65,536 envs",
             dict(kind="cellular", num_envs=1 << 16, n_cells=3, n_states=3, stochastic=True), True),
    "cfg3": ("grid world, 2^20 envs, auto-reset every 128 steps",
             dict(kind="gridworld", num_envs=1 << 20, max_episode_steps=128), True),
    "16x4": ("polarisation 16 cells x 4 levels with noise (r03's 16x4 collect workload is deterministic), 2^22 envs, "
             "per-cell counts only",
             dict(kind="cellular", num_envs=1 << 22, n_cells=16, n_states=4, stochastic=True), False),
}
GRID_RANDOM = [4, 9, 14, 19, 20, 21, 22, 23]         # a_0 + 5 a_1 of the reference sampler's actions


def policy_table(env):
    n_s = 400 if env.kind == "gridworld" else env.n_states ** env.n_cells
    if env.kind == "gridworld":
        return torch.tensor(GRID_RANDOM, device=env.device)[torch.randint(0, 8, (n_s,), device=env.device)].to(torch.int32)
    return torch.randint(0, env.n_actions ** env.n_cells, (n_s,), device=env.device, dtype=torch.int32)


def aggregate(env, tr, counts):
    """The torch aggregation of a `collect` record into the tables `collect_counts` fills."""
    u32 = lambda t: t.long() & 0xFFFFFFFF                              # noqa: E731  (uint32 payload of int32 views)
    s, a, nx = u32(tr.obs).view(-1), u32(tr.action).view(-1), u32(tr.next_obs).view(-1)
    if counts.visits is not None:
        nS, nA = env._joint_sizes()
        sa = s * nA + a
        counts.visits.view(-1).add_(torch.bincount(sa, minlength=nS * nA))
        counts.next.view(-1).add_(torch.bincount(sa * nS + nx, minlength=nS * nA * nS))
        q = torch.round(tr.reward.view(-1).double() * 2.0 ** 24).long()
        counts.reward_q24.view(-1).index_add_(0, sa, q)
        counts.unsafe.view(-1).index_add_(0, sa, (tr.flags.view(-1) & 1).long())
    if counts.cell_next is not None:
        S, A = env.n_states, env.n_actions
        for c in range(env.n_cells):
            d = lambda x, R: (x // R ** c) % R                          # noqa: E731
            counts.cell_next[c].view(-1).add_(torch.bincount((d(s, S) * A + d(a, A)) * S + d(nx, S), minlength=S * A * S))


def time_calls(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps * 1e-3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r04_count_bench.json"))
    ap.add_argument("--k", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("count_bench needs a CUDA device")
    K = a.k
    out = {"card": card(), "k": K, "rounds": a.rounds, "reps_per_round": a.reps, "workloads": {}}
    for name in a.workloads.split(","):
        desc, kw, joint = WORKLOADS[name]
        env = B.CellularVectorEnv(env_seed=1, emit_side_effects=False, **kw)
        n = env.num_envs
        pols = [("random", None, 0.0)] + ([("table_eps0.1", policy_table(env), 0.1)] if joint else [])
        res = {"desc": desc, "envs": n, "joint_tables": joint}
        for pname, pol, eps in pols:
            counts, agg = env.zero_counts(joint=joint), env.zero_counts(joint=joint)

            def collect_agg():
                aggregate(env, env.collect(K, pol, eps, next_obs=True), agg)
            arms = {"collect_counts": lambda: env.collect_counts(K, pol, eps, counts),
                    "rollout_floor": lambda: env.rollout(K, pol),
                    "collect_plus_torch": collect_agg}
            if joint:
                # attribution: the same call counting one group of tables at a time (the others None), into tables of
                # its own so that the check below still compares like with like
                keep = {"counts_joint_only": ("visits", "next", "reward_q24", "unsafe"), "counts_visits_only": ("visits",),
                        "counts_next_only": ("next",), "counts_reward_unsafe_only": ("reward_q24", "unsafe")}
                if counts.cell_next is not None:
                    keep["counts_cell_next_only"] = ("cell_next",)
                for arm, fields in keep.items():
                    part = env.zero_counts()._replace(**{f: None for f in counts._fields if f not in fields})
                    arms[arm] = (lambda part: lambda: env.collect_counts(K, pol, eps, part))(part)
            for fn in arms.values():                                # warm-up: modules, allocator, record buffers
                fn()
            times = {k: [] for k in arms}
            for _ in range(a.rounds):
                for k, fn in arms.items():
                    times[k].append(time_calls(fn, a.reps))
            r = {}
            floor = statistics.median(times["rollout_floor"])
            for k, ts in times.items():
                med = statistics.median(ts)
                r[k] = {"s_per_call_median": med, "s_per_call_min": min(ts), "s_per_call_max": max(ts),
                        "env_steps_per_s": n * K / med, "over_rollout_floor": med / floor}
            r["collect_plus_torch_over_counts"] = r["collect_plus_torch"]["s_per_call_median"] / r["collect_counts"]["s_per_call_median"]
            r["counts_over_rollout"] = r["collect_counts"]["s_per_call_median"] / r["rollout_floor"]["s_per_call_median"]
            # both paths saw the same kind of trajectories; the tables are sanity-checked for their sums
            r["check_visits_sum_equal"] = (bool(counts.visits.sum() == agg.visits.sum()) if joint
                                           else bool((counts.cell_next.sum((1, 2, 3)) == agg.cell_next.sum((1, 2, 3))).all()))
            res[pname] = r
            print(name, pname, json.dumps(r), flush=True)
            del counts, agg, arms
        out["workloads"][name] = res
        env.close()
        del env
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
