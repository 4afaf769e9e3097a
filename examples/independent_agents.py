#!/usr/bin/env python
"""P independent count-and-plan agents over one batch, one launch per round -- everything on one B200.

    python examples/independent_agents.py [--agents 8] [--envs 65536] [--rounds 8] [--steps 64] [--epsilon 0.2]

Agent j owns the envs e with e % P == j and starts from its own random greedy policy (seed j).  Each round runs ONE
grouped `collect_counts` (a policy stack of the P greedy policies, counts with a leading [P] group dimension): every env
acts by its agent's table and adds its transitions to its agent's counts only.  Each agent then plans on its own
counts alone with the value iteration of count_and_plan.py, so the P learners share the launch but no experience
(seeds of one agent for error bars, or a sweep over epsilon or priors).  At the end one stacked `rollout` evaluates all
P learned policies, next to the policy planned on `exact_model`.
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gym_cellular_b200 as gcb                                      # noqa: E402
from gym_cellular_b200.model import exact_model                     # noqa: E402

ENV = dict(stochastic=True)


def value_iteration(P, R, gamma=0.95, iters=300):
    V = torch.zeros(P.shape[0], dtype=torch.float64, device=P.device)
    for _ in range(iters):
        Q = R + gamma * (P @ V)
        V = Q.max(dim=1).values
    return Q.argmax(dim=1).to(torch.int32)


def estimate(counts):
    """P_hat[s, a, s'] and R_hat[s, a] of one agent's counts (unvisited pairs: no successor, reward 0)."""
    n = counts.visits.to(torch.float64)
    seen = n.clamp(min=1.0)
    return counts.next.to(torch.float64) / seen[..., None], counts.reward_q24.to(torch.float64) * 2.0 ** -24 / seen


def initial_policies(agents, nS, nA, device):
    """One random greedy table per agent, drawn from generator seed j."""
    return torch.stack([torch.randint(0, nA, (nS,), generator=torch.Generator().manual_seed(j), dtype=torch.int32)
                        for j in range(agents)]).to(device)


def evaluate(policies, envs, steps):
    """Mean return of each table of `policies` [P, nS] over its envs (e % P), all P evaluated by one stacked rollout."""
    P = policies.shape[0]
    env = gcb.CellularVectorEnv(num_envs=envs, env_seed=2, emit_side_effects=False, **ENV)
    agent = (torch.arange(envs, device=env.device) % P).to(torch.int32)
    ret, _ = env.rollout(steps, policies, policy_of_env=agent)
    out = torch.zeros(P, dtype=torch.float64, device=env.device).index_add_(0, agent.long(), ret.double())
    out /= torch.bincount(agent.long(), minlength=P).double()
    env.close()
    return out.cpu()


def learn(agents=8, envs=1 << 16, rounds=8, steps=64, epsilon=0.2, eval_steps=128):
    env = gcb.CellularVectorEnv(num_envs=envs, env_seed=1, max_episode_steps=50, emit_side_effects=False, **ENV)
    agent = (torch.arange(envs, device=env.device) % agents).to(torch.int32)
    counts = env.zero_counts(groups=agents)
    nS, nA = counts.visits.shape[1:]
    policies = initial_policies(agents, nS, nA, env.device)
    launches = env.launch_count
    for _ in range(rounds):
        env.collect_counts(steps, policies, epsilon, counts, policy_of_env=agent)
        policies = torch.stack([value_iteration(*estimate(counts.group(j))) for j in range(agents)])
    learned = evaluate(policies, envs, eval_steps)
    P, R, _ = exact_model(**ENV)
    planned = value_iteration(torch.from_numpy(P).cuda(), torch.from_numpy(R).cuda())
    out = {"agents": agents, "count_launches": env.launch_count - launches,
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
    r = torch.tensor(out["learned_return"])
    print(f"{out['agents']} agents, {sum(out['counted_transitions'])} transitions counted in {out['count_launches']} "
          f"launches (each agent {min(out['counted_transitions'])}..{max(out['counted_transitions'])})")
    print(f"learned return over 128 steps  mean {float(r.mean()):8.3f}  min {float(r.min()):8.3f}  max {float(r.max()):8.3f}")
    print(f"exact_model policy             {out['exact_model_return']:8.3f}")
    print(f"a random table policy          {out['random_return']:8.3f}")
    return out


if __name__ == "__main__":
    main()
