"""Policy stacks on one GPU: what GC_POLICY_TABLE_STACK costs, and whether the existing policy kinds kept their speed.

    python scripts/policy_stack_bench.py [--parent-tree DIR [--parent-lib-dir DIR]] [--out FILE] [--k 64]

Workloads: BASELINE config 2 (3 cells x 3 levels with noise, 65,536 envs), config 3 (grid world, 2^20 envs) and 2^22 envs
of 8 cells x 4 levels with noise (per-cell counts only: 4^8 x 4^8 joint bins exceed 2^31).  K = 64 steps per call.

1. existing kinds, before and after: rollout (random and table policy), collect and collect_counts (table policy, epsilon
   0.1), each in a fresh process per side and round, the sides alternating.  --parent-tree is a checkout of the commit
   before the stack; its library is built into a temporary directory through GC_B200_LIB_DIR unless --parent-lib-dir
   names one already built from it.  Each side also hashes the outputs of one seeded call sequence; the hashes must agree.
2. the stack: rollout and collect_counts of P = 1, 8 and 64 tables over the batch (env e acts by table e % P) in one
   launch, against the same P tables run as P envs of num_envs / P envs each (one launch per table and round, what a
   caller without stacks runs), and against GC_POLICY_TABLE on the whole batch.

Every arm reports the median time per call (or per round of P calls) over the rounds and its spread (min, max).  Writes
one JSON file; the card's name and power limit are read in the same run.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKLOADS = {
    "cfg2": ("polarisation 3 cells x 3 levels, stochastic, 65,536 envs",
             dict(kind="cellular", num_envs=1 << 16, n_cells=3, n_states=3, stochastic=True), True),
    "cfg3": ("grid world, 2^20 envs, auto-reset every 128 steps",
             dict(kind="gridworld", num_envs=1 << 20, max_episode_steps=128), True),
    "8x4": ("polarisation 8 cells x 4 levels, stochastic, 2^22 envs, per-cell counts only",
            dict(kind="cellular", num_envs=1 << 22, n_cells=8, n_states=4, stochastic=True), False),
}
GRID_RANDOM = [4, 9, 14, 19, 20, 21, 22, 23]         # a_0 + 5 a_1 of the reference sampler's actions
EPS = 0.1


def _torch():
    import torch
    return torch


def policy_tables(env, n_tables, seed):
    """[n_tables, nS] int32 device tables, the same on every run (drawn on the host)."""
    torch = _torch()
    g = torch.Generator().manual_seed(seed)
    nS, nA = env._joint_sizes()
    if env.kind == "gridworld":
        pick = torch.randint(0, 8, (n_tables, nS), generator=g)
        return torch.tensor(GRID_RANDOM, dtype=torch.int32)[pick].to(env.device)
    return torch.randint(0, nA, (n_tables, nS), generator=g, dtype=torch.int32).to(env.device)


def time_calls(fn, reps):
    torch = _torch()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps * 1e-3


def summary(ts, work):
    med = statistics.median(ts)
    return {"s_median": med, "s_min": min(ts), "s_max": max(ts), "env_steps_per_s": work / med}


def card():
    torch = _torch()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


# ---------------------------------------------------------------------------------------------
# 1. the existing kinds (runs in a worker process, against whichever library GC_B200_LIB_DIR selects)

def existing_arms(B, env, K, joint):
    pol = policy_tables(env, 1, 1)[0]
    counts = env.zero_counts(joint=joint)
    return {"rollout_random": lambda: env.rollout(K),
            "rollout_table": lambda: env.rollout(K, pol),
            "collect_table_eps": lambda: env.collect(K, pol, EPS, next_obs=True),
            "counts_table_eps": lambda: env.collect_counts(K, pol, EPS, counts)}


def output_hash(B, kw, K, joint):
    """sha256 of every output of one seeded sequence of the four calls on a fresh env."""
    torch = _torch()
    env = B.CellularVectorEnv(env_seed=3, emit_side_effects=False, **kw)
    pol = policy_tables(env, 1, 2)[0]
    h = hashlib.sha256()
    add = lambda t: h.update(t.contiguous().view(torch.uint8).cpu().numpy().tobytes())      # noqa: E731
    for x in env.rollout(K):
        add(x)
    for x in env.rollout(K, pol):
        add(x)
    tr = env.collect(K, pol, EPS, next_obs=True)
    for x in tr:
        add(x)
    counts = env.collect_counts(K, pol, EPS, env.zero_counts(joint=joint))
    for x in counts:
        if x is not None:
            add(x)
    for x in (env.state, env.time_step, env.tabular_state(torch.int32), env._stats):
        add(x)
    add(torch.tensor([env.sync_step_counter(), env.launch_count]))
    env.close()
    return h.hexdigest()


def worker(a):
    torch = _torch()
    import gym_cellular_b200 as B
    out = {"lib": B._lib.LIB_PATH, "workloads": {}}
    for name in a.workloads.split(","):
        _, kw, joint = WORKLOADS[name]
        env = B.CellularVectorEnv(env_seed=1, emit_side_effects=False, **kw)
        arms = existing_arms(B, env, a.k, joint)
        for fn in arms.values():
            fn()
        out["workloads"][name] = {"times": {k: time_calls(fn, a.reps) for k, fn in arms.items()},
                                  "output_sha256": output_hash(B, kw, a.k, joint)}
        env.close()
        del env, arms
        torch.cuda.empty_cache()
    print("WORKER " + json.dumps(out), flush=True)


def run_worker(a, pkg_root, lib_dir):
    env = dict(os.environ)
    if lib_dir:
        env["GC_B200_LIB_DIR"] = lib_dir
    else:
        env.pop("GC_B200_LIB_DIR", None)
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--pkg-root", pkg_root, "--k", str(a.k),
           "--reps", str(a.reps), "--workloads", a.workloads]
    p = subprocess.run(cmd, env=env, capture_output=True, text=True)
    line = [x for x in p.stdout.splitlines() if x.startswith("WORKER ")]
    if p.returncode or not line:
        raise RuntimeError(f"worker failed ({pkg_root}):\n{p.stdout}\n{p.stderr}")
    return json.loads(line[-1][len("WORKER "):])


def before_after(a):
    lib_dir, tmp = a.parent_lib_dir, None
    if lib_dir is None:
        tmp = tempfile.TemporaryDirectory()
        lib_dir = tmp.name
        subprocess.check_call([sys.executable, "-m", "gym_cellular_b200.build"], cwd=a.parent_tree,
                              env=dict(os.environ, GC_B200_LIB_DIR=lib_dir))
    sides = {"parent": (os.path.abspath(a.parent_tree), os.path.abspath(lib_dir)), "this": (REPO, None)}
    runs = {s: [] for s in sides}
    for rnd in range(a.ab_rounds):
        for s in (("parent", "this") if rnd % 2 == 0 else ("this", "parent")):     # alternating which side goes first
            runs[s].append(run_worker(a, *sides[s]))
    res = {}
    for name in a.workloads.split(","):
        K, n = a.k, WORKLOADS[name][1]["num_envs"]
        r = {}
        for s in sides:
            r[s] = {arm: summary([run["workloads"][name]["times"][arm] for run in runs[s]], K * n)
                    for arm in runs[s][0]["workloads"][name]["times"]}
        r["this_over_parent"] = {arm: r["this"][arm]["s_median"] / r["parent"][arm]["s_median"] for arm in r["this"]}
        hashes = {s: {run["workloads"][name]["output_sha256"] for run in runs[s]} for s in sides}
        r["outputs_identical"] = len(hashes["parent"] | hashes["this"]) == 1
        res[name] = r
        print(name, json.dumps(r), flush=True)
    if tmp is not None:
        tmp.cleanup()
    return {"rounds": a.ab_rounds, "reps_per_round": a.reps, "parent_lib": lib_dir, "workloads": res}


# ---------------------------------------------------------------------------------------------
# 2. the stack against separate launches

def stack_cost(a):
    torch = _torch()
    import gym_cellular_b200 as B
    K, res = a.k, {}
    for name in a.workloads.split(","):
        desc, kw, joint = WORKLOADS[name]
        n = kw["num_envs"]
        r = {"desc": desc, "envs": n}
        for P in (int(x) for x in a.tables.split(",")):
            whole = B.CellularVectorEnv(env_seed=1, emit_side_effects=False, **kw)
            tables = policy_tables(whole, P, 7)
            table_of_env = (torch.arange(n, device=whole.device) % P).to(torch.int32)
            part = dict(kw, num_envs=n // P)
            parts = [B.CellularVectorEnv(env_seed=1, emit_side_effects=False, env_id_offset=j * (n // P), **part)
                     for j in range(P)]
            c_whole, c_one = whole.zero_counts(joint=joint), whole.zero_counts(joint=joint)
            c_parts = parts[0].zero_counts(joint=joint)

            def separate(call):
                def go():
                    for j, e in enumerate(parts):
                        call(e, tables[j])
                return go
            arms = {"rollout_stack": lambda: whole.rollout(K, tables, policy_of_env=table_of_env),
                    "rollout_separate": separate(lambda e, t: e.rollout(K, t)),
                    "rollout_one_table": lambda: whole.rollout(K, tables[0]),
                    "counts_stack": lambda: whole.collect_counts(K, tables, EPS, c_whole, policy_of_env=table_of_env),
                    "counts_separate": separate(lambda e, t: e.collect_counts(K, t, EPS, c_parts)),
                    "counts_one_table": lambda: whole.collect_counts(K, tables[0], EPS, c_one)}
            for fn in arms.values():
                fn()
            times = {k: [] for k in arms}
            keys = list(arms)
            for rnd in range(a.rounds):
                for k in keys[rnd % len(keys):] + keys[:rnd % len(keys)]:     # rotated, so no arm always runs first
                    times[k].append(time_calls(arms[k], a.reps))
            rr = {k: summary(ts, K * n) for k, ts in times.items()}
            for kind in ("rollout", "counts"):
                st = rr[f"{kind}_stack"]["s_median"]
                rr[f"{kind}_separate_over_stack"] = rr[f"{kind}_separate"]["s_median"] / st
                rr[f"{kind}_stack_over_one_table"] = st / rr[f"{kind}_one_table"]["s_median"]
            rr["launches_per_round"] = {"stack": 1, "separate": P}
            r[f"P{P}"] = rr
            print(name, P, json.dumps(rr), flush=True)
            for e in [whole] + parts:
                e.close()
            del whole, parts, arms, c_whole, c_one, c_parts, tables
            torch.cuda.empty_cache()
        res[name] = r
    return {"rounds": a.rounds, "reps_per_round": a.reps, "workloads": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r06_policy_stack_bench.json"))
    ap.add_argument("--k", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--ab-rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--tables", default="1,8,64")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--parent-lib-dir", default=None)
    ap.add_argument("--part", choices=("both", "ab", "stack"), default="both",
                    help="ab: only the existing kinds before / after; stack: only the stack against separate launches")
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--pkg-root", default=REPO)
    a = ap.parse_args()
    sys.path.insert(0, a.pkg_root)
    torch = _torch()
    if not torch.cuda.is_available():
        raise SystemExit("policy_stack_bench needs a CUDA device")
    if a.worker:
        return worker(a)
    out = {"card": card(), "k": a.k, "epsilon": EPS}
    if a.parent_tree and a.part != "stack":
        out["existing_kinds_before_after"] = before_after(a)
    if a.part != "ab":
        out["stack"] = stack_cost(a)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
