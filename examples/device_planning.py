#!/usr/bin/env python
"""P independent count-and-plan agents, collecting AND planning on the device: two launches per round.

    python examples/device_planning.py [--agents 8] [--envs 65536] [--rounds 8] [--steps 64] [--epsilon 0.2]

The loop of independent_agents.py (same envs, agents, initial policies, grouped `collect_counts` and evaluation),
with the per-agent torch value iteration replaced by ONE `gcb.value_iteration` on the grouped counts: the kernel
forms each agent's estimate P_hat / R_hat from its own counts and plans all P of them in one launch, returning the
[P, nS] policy stack the next round's collect acts by.  Prints each round's time, split into collect and plan, from
CUDA events.
"""
import argparse
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import gym_cellular_b200 as gcb                                                          # noqa: E402
from gym_cellular_b200.model import exact_model                                         # noqa: E402
from independent_agents import ENV, evaluate, initial_policies                          # noqa: E402


def learn(agents=8, envs=1 << 16, rounds=8, steps=64, epsilon=0.2, eval_steps=128, gamma=0.95, iters=300):
    env = gcb.CellularVectorEnv(num_envs=envs, env_seed=1, max_episode_steps=50, emit_side_effects=False, **ENV)
    agent = (torch.arange(envs, device=env.device) % agents).to(torch.int32)
    counts = env.zero_counts(groups=agents)
    nS, nA = counts.visits.shape[1:]
    policies = initial_policies(agents, nS, nA, env.device)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(rounds)]
    for r in range(rounds):
        ev[r][0].record()
        env.collect_counts(steps, policies, epsilon, counts, policy_of_env=agent)
        ev[r][1].record()
        policies = gcb.value_iteration(counts, gamma, iters).policy
        ev[r][2].record()
    torch.cuda.synchronize()
    collect_ms = [e[0].elapsed_time(e[1]) for e in ev]
    plan_ms = [e[1].elapsed_time(e[2]) for e in ev]
    learned = evaluate(policies, envs, eval_steps)
    P, R, _ = exact_model(**ENV)
    planned = gcb.value_iteration((torch.from_numpy(P).cuda(), torch.from_numpy(R).cuda()), gamma, iters).policy
    out = {"agents": agents, "collect_ms": collect_ms, "plan_ms": plan_ms,
           "counted_transitions": [int(v) for v in counts.visits.sum((1, 2)).cpu()],
           "learned_return": [float(x) for x in learned],
           "exact_model_return": float(evaluate(planned[None], envs, eval_steps)[0]),
           "random_return": float(evaluate(initial_policies(1, nS, nA, env.device), envs, eval_steps)[0])}
    env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--agents", type=int, default=8)
    ap.add_argument("--envs", type=int, default=1 << 16)
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--epsilon", type=float, default=0.2)
    a = ap.parse_args()
    out = learn(a.agents, a.envs, a.rounds, a.steps, a.epsilon)
    for r, (c, p) in enumerate(zip(out["collect_ms"], out["plan_ms"])):
        print(f"round {r}: collect {c:7.3f} ms  plan {p:7.3f} ms")
    r = torch.tensor(out["learned_return"])
    print(f"{out['agents']} agents, {sum(out['counted_transitions'])} transitions counted")
    print(f"learned return over 128 steps  mean {float(r.mean()):8.3f}  min {float(r.min()):8.3f}  max {float(r.max()):8.3f}")
    print(f"exact_model policy             {out['exact_model_return']:8.3f}")
    print(f"a random table policy          {out['random_return']:8.3f}")
    return out


if __name__ == "__main__":
    main()
