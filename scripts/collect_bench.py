"""Experience collection on one GPU: the fused rollout, `collect` with the full record (ε = 0 and ε = 0.1), and
the per-step loop an agent writes without it (`step_device` plus torch policy lookup, ε draw and record copies),
K = 64 steps per call, at the sizes where launches or HBM bound the step.  Writes one JSON file to --out.

    python scripts/collect_bench.py --out DIR [--k 64] [--reps 20] [--warmup 3]

Record bytes per env-step: obs, action, reward and next_obs 4 B each, flags 1 B (17 B); the rate of those writes is
reported against the project's measured HBM bandwidth (6554.2 GB/s on the B200, profiles/README.md).
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                                          # noqa: E402

import gym_cellular_b200 as B                                         # noqa: E402

HBM_GBS = 6554.2
RECORD_BYTES = 17
SIZES = {
    "cfg2": ("polarisation 3 cells x 3 levels, stochastic, 65,536 envs",
             dict(kind="cellular", num_envs=1 << 16, n_cells=3, n_states=3, stochastic=True)),
    "cfg3": ("grid world, 2^20 envs, auto-reset every 128 steps",
             dict(kind="gridworld", num_envs=1 << 20, max_episode_steps=128)),
    "16x4": ("polarisation 16 cells x 4 levels, 2^22 envs",
             dict(kind="cellular", num_envs=1 << 22, n_cells=16, n_states=4)),
}
GRID_RANDOM = [4, 9, 14, 19, 20, 21, 22, 23]         # a_0 + 5 a_1 of the reference sampler's actions


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps * 1e-3


def policy_table(env):
    """A fixed random table policy, or None where no table fits (4^16 states)."""
    n_s = env.n_states ** env.n_cells
    if n_s > 1 << 20:
        return None
    if env.kind == "gridworld":
        return torch.tensor(GRID_RANDOM, device=env.device)[torch.randint(0, 8, (n_s,), device=env.device)].to(torch.int32)
    return torch.randint(0, env.n_actions ** env.n_cells, (n_s,), device=env.device, dtype=torch.int32)


def step_loop(env, K, policy, eps):
    """K steps of the per-step loop recording what `collect` records (obs, action, reward, flags)."""
    n, dev = env.num_envs, env.device
    rec = {"obs": torch.empty(K, n, dtype=torch.int32, device=dev), "action": torch.empty(K, n, dtype=torch.int64, device=dev),
           "reward": torch.empty(K, n, device=dev), "flags": torch.empty(K, n, dtype=torch.uint8, device=dev)}
    grid = env.kind == "gridworld"
    n_joint = 25 if grid else env.n_actions ** env.n_cells
    codes = torch.tensor(GRID_RANDOM, device=dev)
    info = env._v_infos

    def run():
        for k in range(K):
            idx = env.tabular_state(torch.int32)
            rec["obs"][k].copy_(idx)
            rnd = codes[torch.randint(0, 8, (n,), device=dev)] if grid else torch.randint(0, n_joint, (n,), device=dev)
            if policy is not None:
                rnd = torch.where(torch.rand(n, device=dev) < eps, rnd, policy[idx.long()].long())
            rec["action"][k].copy_(rnd)
            env.step_device(env.detabularize(rnd, "action"))
            rec["reward"][k].copy_(env._v_reward)
            rec["flags"][k].copy_(info["unsafe"].to(torch.uint8) | (env._v_trunc.to(torch.uint8) << 1) | (info["count"] << 2))
    return run


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--k", type=int, default=64)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sizes", default=",".join(SIZES))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("collect_bench needs a CUDA device")
    K = a.k
    out = {"card": card(), "k": K, "reps": a.reps, "warmup": a.warmup, "record_bytes_per_env_step": RECORD_BYTES,
           "hbm_gbs_measured": HBM_GBS, "sizes": {}}
    for name in a.sizes.split(","):
        desc, kw = SIZES[name]
        env = B.CellularVectorEnv(env_seed=1, emit_side_effects=False, **kw)
        n, pol = env.num_envs, policy_table(env)
        res = {"desc": desc, "envs": n}
        arms = {"a_rollout": lambda: env.rollout(K),
                "b_collect": lambda: env.collect(K, pol, 0.0, next_obs=True)}
        if pol is not None:
            arms["c_collect_eps0.1"] = lambda: env.collect(K, pol, 0.1, next_obs=True)
        for arm, fn in arms.items():
            s = timed(fn, a.reps, a.warmup)
            r = {"s_per_call": s, "env_steps_per_s": n * K / s}
            if arm != "a_rollout":
                r["record_gbs"] = RECORD_BYTES * n * K / s / 1e9
                r["record_frac_of_hbm"] = r["record_gbs"] / HBM_GBS
            res[arm] = r
        loop = step_loop(env, K, pol, 0.1)
        s = timed(loop, max(1, a.reps // 10), 1)
        res["d_step_loop"] = {"s_per_call": s, "env_steps_per_s": n * K / s, "policy": "table, eps 0.1" if pol is not None else "random"}
        res["b_over_a"] = res["a_rollout"]["s_per_call"] / res["b_collect"]["s_per_call"]
        res["b_over_d"] = res["d_step_loop"]["s_per_call"] / res["b_collect"]["s_per_call"]
        out["sizes"][name] = res
        print(name, json.dumps(res), flush=True)
        env.close()
        del env, arms, loop
        torch.cuda.empty_cache()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "collect_bench.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
