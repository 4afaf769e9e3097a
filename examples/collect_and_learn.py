#!/usr/bin/env python
"""Batched Q-learning on experience collected K steps at a time: one kernel launch per K env-steps.

    python examples/collect_and_learn.py [--envs 16384] [--rounds 40] [--k 32]

The agent of examples/packed_tabular_agent.py, rebuilt on `collect`: instead of one step launch plus a dozen small
torch launches per step, each round asks the env for K steps of every env under the epsilon-greedy policy of the
current greedy table, recorded as [K, num_envs] tensors of (obs, action, reward, flags, next_obs), and makes one
batched update over the K x num_envs transitions.  The update bootstraps from `next_obs`, the successor before the
time-limit auto-reset: at a truncated step the episode was cut, not ended, so its value still counts.
"""
import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gym_cellular_b200 as gcb                                      # noqa: E402


def evaluate(policy, n, k, seed):
    """Mean per-env return and unsafe-step rate of `k` steps of `policy` (None = random play) from the reset state."""
    env = gcb.CellularVectorEnv(num_envs=n, n_cells=3, n_states=3, stochastic=True, env_seed=seed, max_episode_steps=50)
    ret, uns = env.rollout(k, policy)
    return float(ret.mean()), float(uns.sum()) / (n * k)


def learn(envs=16384, rounds=40, k=32, gamma=0.9, unsafe_penalty=0.0, eval_steps=64, seed=1):
    n, C, S, A = envs, 3, 3, 3
    env = gcb.CellularVectorEnv(num_envs=n, n_cells=C, n_states=S, stochastic=True, env_seed=seed, max_episode_steps=50)
    n_s, n_a = S ** C, A ** C
    Q = torch.zeros(n_s, n_a, device=env.device)
    visits = torch.zeros(n_s * n_a, device=env.device)
    torch.cuda.synchronize()
    t0, launches0 = time.perf_counter(), env.launch_count
    for r in range(rounds):
        eps = max(0.05, 1.0 - r / (0.6 * rounds))
        tr = env.collect(k, Q.argmax(1), eps, next_obs=True)           # one kernel launch: k steps of every env
        obs, act, nxt = (x.reshape(-1).to(torch.int64) for x in (tr.obs, tr.action, tr.next_obs))
        target = tr.reward.reshape(-1) - unsafe_penalty * tr.unsafe.reshape(-1) + gamma * Q[nxt].max(1).values
        flat = obs * n_a + act
        visits.index_add_(0, flat, torch.ones_like(target))
        Q.view(-1).index_add_(0, flat, (target - Q.view(-1)[flat]) / visits[flat].clamp(min=1.0))
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    greedy = Q.argmax(1)
    g_ret, g_uns = evaluate(greedy, n, eval_steps, seed + 100)
    r_ret, r_uns = evaluate(None, n, eval_steps, seed + 100)
    return {"env_steps": rounds * k * n, "collect_launches": env.launch_count - launches0, "wall_s": wall,
            "env_steps_per_s": rounds * k * n / wall, "greedy_return": g_ret, "random_return": r_ret,
            "greedy_unsafe_rate": g_uns, "random_unsafe_rate": r_uns}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--rounds", type=int, default=40)
    ap.add_argument("--k", type=int, default=32)
    ap.add_argument("--unsafe-penalty", type=float, default=0.0)
    args = ap.parse_args()
    out = learn(args.envs, args.rounds, args.k, unsafe_penalty=args.unsafe_penalty)
    print(out)
    return out


if __name__ == "__main__":
    main()
