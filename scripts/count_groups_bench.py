"""Grouped counts on one GPU: P independent count sets over one batch in one launch, against what a caller runs without
them, and whether the existing count kinds kept their speed.

    python scripts/count_groups_bench.py [--parent-tree DIR [--parent-lib-dir DIR]] [--out FILE] [--k 64]

Workloads: those of scripts/policy_stack_bench.py -- BASELINE config 2 (3 cells x 3 levels with noise, 65,536 envs),
config 3 (grid world, 2^20 envs) and 2^22 envs of 8 cells x 4 levels with noise (per-cell counts only).  K = 64 steps per
call, epsilon 0.1, env e in group e % P, P = 8 and 64.  Arms, each the median time per round and its spread:
1. grouped: one `collect_counts` with counts of P groups (gc_collect_counts_grouped), one launch;
2. separate: P envs of num_envs / P envs, each with its own counts, P launches;
3. collect + bincount: one stacked `collect` and a per-group histogram of its record in torch;
4. ungrouped: the stacked `collect_counts` into one count set, what grouping costs;
5. existing kinds before and after (--parent-tree, a checkout of the commit before grouped counts): `collect_counts`
   with a table policy and with a stack of 8 tables, each side in fresh processes, the sides alternating, each side
   hashing the outputs of one seeded call sequence (the hashes must agree).
Writes one JSON file; the card's name and power limit are read in the same run.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "scripts"))
from policy_stack_bench import EPS, WORKLOADS, card, policy_tables, summary, time_calls     # noqa: E402

STACK_P = 8                 # the stack of arm 5


def _torch():
    import torch
    return torch


# ---------------------------------------------------------------------------------------------
# 5. the existing count kinds (a worker process, against whichever library GC_B200_LIB_DIR selects)

def existing_arms(env, K, joint):
    torch = _torch()
    tables = policy_tables(env, STACK_P, 1)
    m = (torch.arange(env.num_envs, device=env.device) % STACK_P).to(torch.int32)
    c_table, c_stack = env.zero_counts(joint=joint), env.zero_counts(joint=joint)
    return {"counts_table_eps": lambda: env.collect_counts(K, tables[0], EPS, c_table),
            "counts_stack_eps": lambda: env.collect_counts(K, tables, EPS, c_stack, policy_of_env=m)}


def output_hash(B, kw, K, joint):
    """sha256 of every output of one seeded sequence of table and stack `collect_counts` calls on a fresh env."""
    torch = _torch()
    env = B.CellularVectorEnv(env_seed=3, emit_side_effects=False, **kw)
    tables = policy_tables(env, STACK_P, 2)
    m = (torch.arange(env.num_envs, device=env.device) % STACK_P).to(torch.int32)
    h = hashlib.sha256()
    add = lambda t: h.update(t.contiguous().view(torch.uint8).cpu().numpy().tobytes())      # noqa: E731
    for counts in (env.collect_counts(K, tables[0], EPS, env.zero_counts(joint=joint)),
                   env.collect_counts(K, tables, EPS, env.zero_counts(joint=joint), policy_of_env=m)):
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
        arms = existing_arms(env, a.k, joint)
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
    return {"rounds": a.ab_rounds, "reps_per_round": a.reps, "workloads": res}


# ---------------------------------------------------------------------------------------------
# 1-4. grouped counts against the alternatives

def bincount_groups(rec, group, P, nS, nA, S, A, Cn, joint, cellular):
    """Per-group histograms of a stacked record in torch: what a caller without grouped counts computes."""
    torch = _torch()
    g = group.long()[None, :].expand_as(rec.obs).reshape(-1)
    s, a_, nx = (x.long().reshape(-1) & 0xFFFFFFFF for x in (rec.obs, rec.action, rec.next_obs))
    out = []
    if joint:
        sa = g * (nS * nA) + s * nA + a_
        out.append(torch.bincount(sa, minlength=P * nS * nA))
        out.append(torch.bincount(sa * nS + nx, minlength=P * nS * nA * nS) if nS * nA * nS * P <= 2 ** 31 else None)
        q = torch.round(rec.reward.double().reshape(-1) * 2.0 ** 24)
        out.append(torch.bincount(sa, weights=q, minlength=P * nS * nA))
        out.append(torch.bincount(sa, weights=rec.unsafe.reshape(-1).double(), minlength=P * nS * nA))
    if cellular:
        for c in range(Cn):
            sc, ac, nc = (s // S ** c) % S, (a_ // A ** c) % A, (nx // S ** c) % S
            out.append(torch.bincount(((g * Cn + c) * S + sc) * A * S + ac * S + nc, minlength=P * Cn * S * A * S))
    return out


def groups_cost(a):
    torch = _torch()
    import gym_cellular_b200 as B
    K, res = a.k, {}
    for name in a.workloads.split(","):
        desc, kw, joint = WORKLOADS[name]
        n = kw["num_envs"]
        cellular = kw["kind"] == "cellular"
        r = {"desc": desc, "envs": n}
        for P in (int(x) for x in a.groups.split(",")):
            whole = B.CellularVectorEnv(env_seed=1, emit_side_effects=False, **kw)
            nS, nA = whole._joint_sizes()
            # 'next' is counted where P of it fit 2^31 entries (config 2 and 3 at P = 8 and 64)
            trans = joint and P * nS * nA * nS <= 2 ** 31
            tables = policy_tables(whole, P, 7)
            group = (torch.arange(n, device=whole.device) % P).to(torch.int32)
            part = dict(kw, num_envs=n // P)
            parts = [B.CellularVectorEnv(env_seed=1, emit_side_effects=False, env_id_offset=j * (n // P), **part)
                     for j in range(P)]
            c_grouped = whole.zero_counts(joint=joint, transitions=trans, groups=P)
            c_plain = whole.zero_counts(joint=joint, transitions=trans)
            c_parts = [e.zero_counts(joint=joint, transitions=trans) for e in parts]

            def separate():
                for j, e in enumerate(parts):
                    e.collect_counts(K, tables[j], EPS, c_parts[j])

            def collect_bincount():
                rec = whole.collect(K, tables, EPS, next_obs=True, policy_of_env=group)
                return bincount_groups(rec, group, P, nS, nA, whole.n_states, whole.n_actions, whole.n_cells, joint,
                                       cellular)

            arms = {"grouped": lambda: whole.collect_counts(K, tables, EPS, c_grouped, policy_of_env=group),
                    "separate": separate,
                    "collect_bincount": collect_bincount,
                    "ungrouped": lambda: whole.collect_counts(K, tables, EPS, c_plain, policy_of_env=group)}
            for fn in arms.values():
                fn()
            times = {k: [] for k in arms}
            keys = list(arms)
            for rnd in range(a.rounds):
                for k in keys[rnd % len(keys):] + keys[:rnd % len(keys)]:     # rotated, so no arm always runs first
                    times[k].append(time_calls(arms[k], a.reps))
            rr = {k: summary(ts, K * n) for k, ts in times.items()}
            g = rr["grouped"]["s_median"]
            rr["separate_over_grouped"] = rr["separate"]["s_median"] / g
            rr["collect_bincount_over_grouped"] = rr["collect_bincount"]["s_median"] / g
            rr["grouped_over_ungrouped"] = g / rr["ungrouped"]["s_median"]
            rr["launches_per_round"] = {"grouped": 1, "separate": P, "ungrouped": 1}
            rr["tables"] = {"joint": joint, "next": trans, "cell_next": cellular}
            r[f"P{P}"] = rr
            print(name, P, json.dumps(rr), flush=True)
            for e in [whole] + parts:
                e.close()
            del whole, parts, arms, c_grouped, c_plain, c_parts, tables
            torch.cuda.empty_cache()
        res[name] = r
    return {"rounds": a.rounds, "reps_per_round": a.reps, "workloads": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r07_count_groups_bench.json"))
    ap.add_argument("--k", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--ab-rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--groups", default="8,64")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--parent-lib-dir", default=None)
    ap.add_argument("--part", choices=("both", "ab", "groups"), default="both",
                    help="ab: only the existing kinds before / after; groups: only arms 1-4")
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--pkg-root", default=REPO)
    a = ap.parse_args()
    sys.path.insert(0, a.pkg_root)
    torch = _torch()
    if not torch.cuda.is_available():
        raise SystemExit("count_groups_bench needs a CUDA device")
    if a.worker:
        return worker(a)
    out = {"card": card(), "k": a.k, "epsilon": EPS}
    if a.part != "ab":
        out["groups"] = groups_cost(a)
    if a.parent_tree and a.part != "groups":
        out["existing_kinds_before_after"] = before_after(a)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
