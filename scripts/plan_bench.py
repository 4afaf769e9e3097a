"""Device value iteration (`gcb.value_iteration`, one launch) against the examples' torch planners, on one GPU.

    python scripts/plan_bench.py [--out profiles/r08_plan_bench.json] [--repeats 5]

Every case plans 300 iterations at gamma 0.95, both arms in this process on the same inputs:
  counts    config 2 (3 cells x 3 levels with noise, 65,536 envs) grouped counts at P = 1, 8, 64 and config 3 (grid
            world, 2^20 envs) at P = 1, 8, collected by one grouped `collect_counts` of K = 64 steps, epsilon 0.1;
            torch arm: independent_agents.value_iteration over `counts.group(j)` for every j;
  dirichlet config-2 models sampled as in posterior_sampling.py, M = 8 and 64; torch arm: posterior_sampling.plan;
  exact     grid world `exact_model`; torch arm: count_and_plan.value_iteration;
  round     one round of examples/device_planning.py (grouped collect + one device plan) against one round of
            examples/independent_agents.py (the same collect + P torch plans), P = 8, config 2.
Each arm is warmed up, then timed with CUDA events over `reps` calls, `repeats` times; the medians are reported with
their spread.  `input_bytes` is what a call reads from global memory at least once; `l2_resident` says whether it fits
the 126 MB L2 (the torch arms read their dense float64 P in every iteration).  The card's name and power limit are read
in the same run.
"""
import argparse
import json
import os
import statistics
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "examples"))
sys.path.insert(0, os.path.join(REPO, "scripts"))
from policy_stack_bench import card, time_calls     # noqa: E402

GAMMA, ITERS, K, EPS = 0.95, 300, 64, 0.1
L2_BYTES = 126 * 2 ** 20


def timed(fn, reps, repeats):
    fn()
    ts = [time_calls(fn, reps) for _ in range(repeats)]
    return {"s_median": statistics.median(ts), "s_min": min(ts), "s_max": max(ts), "reps": reps, "repeats": repeats}


def grouped_counts(gcb, torch, kw, P):
    env = gcb.CellularVectorEnv(env_seed=1, emit_side_effects=False, **kw)
    nS, nA = env._joint_sizes()
    g = torch.Generator().manual_seed(0)
    if env.kind == "gridworld":
        grid = torch.tensor([4, 9, 14, 19, 20, 21, 22, 23], dtype=torch.int32)
        pol = grid[torch.randint(0, 8, (P, nS), generator=g)].cuda()
    else:
        pol = torch.randint(0, nA, (P, nS), generator=g, dtype=torch.int32).cuda()
    m = (torch.arange(env.num_envs, device="cuda") % P).to(torch.int32)
    counts = env.collect_counts(K, pol, EPS, env.zero_counts(groups=P), policy_of_env=m)
    env.close()
    return counts


def agree(a, b):
    return float((a == b).double().mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r08_plan_bench.json"))
    ap.add_argument("--repeats", type=int, default=5)
    a = ap.parse_args()
    import torch
    import gym_cellular_b200 as gcb
    from gym_cellular_b200.model import exact_model
    import count_and_plan
    import device_planning      # noqa: F401  (the example the round arm runs)
    import independent_agents as ia
    import posterior_sampling as ps
    assert torch.cuda.is_available(), "plan_bench needs a GPU"
    out = {"card": card(), "iters": ITERS, "gamma": GAMMA, "cases": []}
    cfg2 = dict(kind="cellular", num_envs=1 << 16, n_cells=3, n_states=3, stochastic=True)
    cfg3 = dict(kind="gridworld", num_envs=1 << 20, max_episode_steps=128)

    def case(name, dev_fn, torch_fn, input_bytes, reps_dev, reps_torch, **extra):
        dev, ref = dev_fn(), torch_fn()
        row = {"case": name, "device": timed(dev_fn, reps_dev, a.repeats), "torch": timed(torch_fn, reps_torch, a.repeats),
               "input_bytes": input_bytes, "l2_resident": input_bytes <= L2_BYTES,
               "policy_agreement": agree(dev.cpu(), ref.cpu()), **extra}
        row["speedup"] = row["torch"]["s_median"] / row["device"]["s_median"]
        out["cases"].append(row)
        print(json.dumps({k: row[k] for k in ("case", "speedup", "policy_agreement")}), flush=True)

    for cname, kw, Ps in (("cfg2", cfg2, (1, 8, 64)), ("cfg3", cfg3, (1, 8))):
        for P in Ps:
            counts = grouped_counts(gcb, torch, kw, P)
            nbytes = sum(t.numel() * 8 for t in (counts.visits, counts.next, counts.reward_q24))
            case(f"{cname}_counts_P{P}", lambda: gcb.value_iteration(counts, GAMMA, ITERS).policy,
                 lambda: torch.stack([ia.value_iteration(*ia.estimate(counts.group(j)), GAMMA, ITERS) for j in range(P)]),
                 nbytes, 20, 1, models=P, shape=list(counts.next.shape[-3:]),
                 unvisited_share=float((counts.visits == 0).double().mean()))
    for M in (8, 64):
        torch.manual_seed(M)
        c1 = grouped_counts(gcb, torch, cfg2, 1).group(0)
        P, R = ps.sample_models(c1, M).contiguous(), ps.sample_rewards(c1, M).contiguous()
        case(f"cfg2_dirichlet_M{M}", lambda: gcb.value_iteration((P, R), GAMMA, ITERS).policy,
             lambda: ps.plan(P, R, GAMMA, ITERS), P.numel() * 8 + R.numel() * 8, 20, 2, models=M, shape=[27, 27, 27])
    Pn, Rn, _ = exact_model(kind="gridworld")
    Pg, Rg = torch.from_numpy(Pn).cuda(), torch.from_numpy(Rn).cuda()
    case("gridworld_exact_model", lambda: gcb.value_iteration((Pg, Rg), GAMMA, ITERS).policy,
         lambda: count_and_plan.value_iteration(Pg, Rg, GAMMA, ITERS), Pg.numel() * 8 + Rg.numel() * 8, 5, 2, models=1,
         shape=[400, 25, 400])

    # one learning round of the two examples: the same collect, then the device plan or the P torch plans
    agents = 8
    env = gcb.CellularVectorEnv(num_envs=1 << 16, env_seed=1, max_episode_steps=50, emit_side_effects=False, **ia.ENV)
    agent = (torch.arange(env.num_envs, device="cuda") % agents).to(torch.int32)
    counts = env.zero_counts(groups=agents)
    nS, nA = counts.visits.shape[1:]
    state = {"pol": ia.initial_policies(agents, nS, nA, env.device)}
    ev = lambda: torch.cuda.Event(enable_timing=True)      # noqa: E731

    def round_ms(planner):
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        env.collect_counts(K, state["pol"], 0.2, counts, policy_of_env=agent)
        e1.record()
        state["pol"] = planner()
        e2.record()
        e2.synchronize()
        return e0.elapsed_time(e1) * 1e-3, e1.elapsed_time(e2) * 1e-3

    arms = {"device_planning": lambda: gcb.value_iteration(counts, GAMMA, ITERS).policy,
            "independent_agents": lambda: torch.stack([ia.value_iteration(*ia.estimate(counts.group(j)), GAMMA, ITERS)
                                                       for j in range(agents)])}
    rounds = {k: [] for k in arms}
    for k, fn in arms.items():
        round_ms(fn)                                        # warm-up
    for _ in range(a.repeats):
        for k, fn in arms.items():                          # alternating arms
            rounds[k].append(round_ms(fn))
    env.close()
    out["round"] = {k: {"collect_s_median": statistics.median(c for c, _ in v),
                        "plan_s_median": statistics.median(p for _, p in v),
                        "round_s_median": statistics.median(c + p for c, p in v),
                        "rounds": [list(x) for x in v]} for k, v in rounds.items()}
    out["round"]["agents"] = agents
    out["round"]["speedup"] = out["round"]["independent_agents"]["round_s_median"] / out["round"]["device_planning"]["round_s_median"]
    print(json.dumps({"round_speedup": out["round"]["speedup"]}), flush=True)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(a.out)


if __name__ == "__main__":
    main()
