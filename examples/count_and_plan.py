#!/usr/bin/env python
"""Model-based tabular learning from experience counts -- everything on one B200.

    python examples/count_and_plan.py [--envs 65536] [--rounds 8] [--steps 64] [--epsilon 0.2]

Each round runs one `collect_counts` launch (every env, K steps, epsilon-greedy on the current greedy policy), which
adds the visit, transition and reward counts of all K x num_envs transitions into the same tables.  The model is then
P_hat = next / visits and R_hat = reward_q24 * 2^-24 / visits, and value iteration (torch, as in
plan_and_rollout.py) on it gives the next greedy policy.  At the end the learned policy and the policy planned on
`exact_model` are evaluated with `rollout`.
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
    """P_hat[s, a, s'] and R_hat[s, a] from the counts (unvisited pairs: no successor, reward 0)."""
    n = counts.visits.to(torch.float64)
    seen = n.clamp(min=1.0)
    return counts.next.to(torch.float64) / seen[..., None], counts.reward_q24.to(torch.float64) * 2.0 ** -24 / seen


def evaluate(policy, envs, steps):
    env = gcb.CellularVectorEnv(num_envs=envs, env_seed=2, emit_side_effects=False, **ENV)
    ret, _ = env.rollout(steps, policy)
    out = float(ret.mean())
    env.close()
    return out


def learn(envs=1 << 16, rounds=8, steps=64, epsilon=0.2, eval_steps=128):
    env = gcb.CellularVectorEnv(num_envs=envs, env_seed=1, max_episode_steps=50, emit_side_effects=False, **ENV)
    counts = env.zero_counts()
    policy = torch.zeros(27, dtype=torch.int32, device="cuda")
    for _ in range(rounds):
        env.collect_counts(steps, policy, epsilon, counts)
        policy = value_iteration(*estimate(counts))
    P, R, _ = exact_model(**ENV)
    planned = value_iteration(torch.from_numpy(P).cuda(), torch.from_numpy(R).cuda())
    out = {"counted_transitions": int(counts.visits.sum()), "count_launches": env.launch_count,
           "learned_return": evaluate(policy, envs, eval_steps), "exact_model_return": evaluate(planned, envs, eval_steps),
           "random_return": evaluate(None, envs, eval_steps)}
    env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 16)
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--epsilon", type=float, default=0.2)
    a = ap.parse_args()
    out = learn(a.envs, a.rounds, a.steps, a.epsilon)
    print(f"{out['counted_transitions']} transitions counted in {out['count_launches']} launches")
    for k in ("learned_return", "exact_model_return", "random_return"):
        print(f"{k:20s} mean return over 128 steps = {out[k]:8.3f}")
    return out


if __name__ == "__main__":
    main()
