#!/usr/bin/env python
"""Posterior sampling (PSRL) on experience counts -- P sampled models acted on in ONE launch per round.

    python examples/posterior_sampling.py [--envs 65536] [--models 8] [--rounds 8] [--steps 64]

Each round draws P models from the posterior of the counts on the device -- transitions from a Dirichlet per (s, a)
with parameters counts.next + prior, mean rewards from a normal around the counted mean with standard deviation
reward_scale / sqrt(visits + 1) -- plans each of them with batched value iteration in torch, and runs one
`collect_counts` over the whole batch with the P greedy policies as a stack: env e acts by model e % P.  Every
transition of every model lands in the one set of counts the next round samples from.  The spread of the sampled
models is all the exploration there is (epsilon 0).
At the end the policy planned on the posterior mean, the policy planned on `exact_model` and the random policy are
evaluated with `rollout`, as in count_and_plan.py.
"""
import argparse
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import gym_cellular_b200 as gcb                                      # noqa: E402
from count_and_plan import ENV, estimate, evaluate, value_iteration  # noqa: E402
from gym_cellular_b200.model import exact_model                     # noqa: E402


def sample_models(counts, n_models, prior=1.0):
    """n_models draws of P(s' | s, a) ~ Dirichlet(next[s, a] + prior): float64 [n_models, nS, nA, nS]."""
    alpha = counts.next.to(torch.float64) + prior
    return torch.distributions.Dirichlet(alpha).sample((n_models,))


def sample_rewards(counts, n_models, reward_scale=1.0):
    """n_models draws of the mean reward R(s, a) ~ N(counted mean, reward_scale^2 / (visits + 1)): [n_models, nS, nA]."""
    n = counts.visits.to(torch.float64)
    mean = counts.reward_q24.to(torch.float64) * 2.0 ** -24 / n.clamp(min=1.0)
    noise = torch.randn(n_models, *n.shape, dtype=torch.float64, device=n.device)
    return mean + reward_scale * noise / (n + 1.0).sqrt()


def plan(P, R, gamma=0.95, iters=300):
    """Value iteration on a batch of models P [M, nS, nA, nS] with rewards R [M, nS, nA] (or [nS, nA] shared by all):
    greedy policies int32 [M, nS]."""
    V = torch.zeros(P.shape[0], P.shape[1], dtype=torch.float64, device=P.device)
    for _ in range(iters):
        Q = R + gamma * torch.einsum("msat,mt->msa", P, V)
        V = Q.max(dim=2).values
    return Q.argmax(dim=2).to(torch.int32)


def learn(envs=1 << 16, models=8, rounds=8, steps=64, prior=1.0, reward_scale=1.0, eval_steps=128, seed=0):
    torch.manual_seed(seed)
    env = gcb.CellularVectorEnv(num_envs=envs, env_seed=1, max_episode_steps=50, emit_side_effects=False, **ENV)
    counts = env.zero_counts()
    table_of_env = (torch.arange(envs, device=env.device) % models).to(torch.int32)
    launches = env.launch_count
    for _ in range(rounds):
        policies = plan(sample_models(counts, models, prior), sample_rewards(counts, models, reward_scale))
        env.collect_counts(steps, policies, 0.0, counts, policy_of_env=table_of_env)
    count_launches = env.launch_count - launches
    policy = value_iteration(*estimate(counts))
    P, R, _ = exact_model(**ENV)
    planned = value_iteration(torch.from_numpy(P).cuda(), torch.from_numpy(R).cuda())
    out = {"counted_transitions": int(counts.visits.sum()), "count_launches": count_launches,
           "learned_return": evaluate(policy, envs, eval_steps), "exact_model_return": evaluate(planned, envs, eval_steps),
           "random_return": evaluate(None, envs, eval_steps)}
    env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 16)
    ap.add_argument("--models", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--prior", type=float, default=1.0)
    ap.add_argument("--reward-scale", type=float, default=1.0)
    a = ap.parse_args()
    out = learn(a.envs, a.models, a.rounds, a.steps, a.prior, a.reward_scale)
    print(f"{out['counted_transitions']} transitions of {a.models} sampled models counted in {out['count_launches']} launches")
    for k in ("learned_return", "exact_model_return", "random_return"):
        print(f"{k:20s} mean return over 128 steps = {out[k]:8.3f}")
    return out


if __name__ == "__main__":
    main()
