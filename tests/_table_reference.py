"""The table contract of `gc_set_tables` (include/gym_cellular_b200.h, gc_cell_tables) restated in numpy, float64.

The kernels never see rules: they see the tables lowered into bit-packed LUTs (gc_tables.cu).  The C oracle hard-codes
the reference's rules, so it can only check tables of the reference's structure.  This module steps ANY table set the
header admits, one cell at a time and vectorised over envs, without a LUT or a bit trick:

  draw     cell c of env g fires iff draws[s][a], noise is on and v < ceil(p * 2^32), v the 32-bit draw of DESIGN §4
           (`_noise_draws.cell_draws`) at counter T = t[e] (rng_episodic) or the global step; replay: u < p in float64
  next     noisy[s][a] if fired, else move[s][a]
  reward   sum over cells of (reward_noisy if fired, else reward)[s][a], in float64, then log2(1 + .) if asked for
  se_row   se_row[j] = side_effects[j][s'_0][s'_p] of the next state s' before the time-limit reset, p = 1 for j = 0
           (p = 0 when C = 1), p = j otherwise; unsafe = any code 2; count = sum of counted[s'_c]
  limit    tn = t + 1; limit > 0 and tn >= limit: truncated, the state becomes initial_state, t = 0
  index    sum_c s_c * place_c mod 2^32 of the returned state, place values from radix (default: n_states)
  stats    steps, unsafe, count, truncated exact; reward = sum of rint(float64(float32 reward) * 2^24)

The reward table is used as given: pass the float32-rounded values the device receives when comparing with a GPU, the
float64 tables of the rules when comparing with the oracle.  Policies of rollout / collect are restated as well
(DESIGN §4): random actions from stream 0x40000000 + c, table actions from the digits of policy[index], and the
epsilon-greedy rule of `_collect_oracle.explore_actions`.
"""
from types import SimpleNamespace

import numpy as np

import _noise_draws as ND
from _collect_oracle import _words, philox

ROLLOUT_STREAM = 0x40000000
EXPLORE_STREAM, EXPLORE_ACTION_STREAM = 0x50000000, 0x50000001
UNSAFE = 2


def threshold(p):
    """ceil(p * 2^32), clamped as gc_api.cu's threshold_of."""
    if not p > 0.0:
        return 0
    return 1 << 32 if p >= 1.0 else int(np.ceil(p * 2.0 ** 32))


def q24(reward):
    """The reward statistic of one step: sum of rint(float64(reward) * 2^24), in int64 (reward: float32 values)."""
    return int(np.rint(np.asarray(reward, np.float64) * 2.0 ** 24).astype(np.int64).sum())


class TableEnv:
    """A batch of n envs stepped by the table contract.  `tabs` is the dict `CellularVectorEnv(cell_tables=...)` takes;
    arrays are cell-major [C][n] as in the oracle."""

    def __init__(self, tabs, n, *, noise_prob=0.1, seed=0, env_id_offset=0, rng_episodic=False, max_episode_steps=0,
                 reward_log2=False, replay=False, radix=None):
        self.C, self.S, self.A = (int(tabs[k]) for k in ("n_cells", "n_states", "n_actions"))
        C, S, A = self.C, self.S, self.A
        self.move = np.asarray(tabs["move"], np.int64).reshape(S, A)
        self.noise = tabs.get("draws") is not None
        self.noisy = np.asarray(tabs["noisy"] if self.noise else self.move, np.int64).reshape(S, A)
        self.draws = (np.asarray(tabs["draws"]).reshape(S, A) != 0) if self.noise else np.zeros((S, A), bool)
        self.reward = np.asarray(tabs["reward"], np.float64).reshape(S, A)
        rn = tabs.get("reward_noisy")
        self.reward_noisy = self.reward if rn is None else np.asarray(rn, np.float64).reshape(S, A)
        self.se = np.asarray(tabs["side_effects"], np.int64).reshape(C, S, S)
        self.counted = (np.asarray(tabs["counted"]).reshape(S) != 0).astype(np.int64)
        init = tabs.get("initial_state")
        self.init = np.zeros(C, np.int64) if init is None else np.asarray(init, np.int64).reshape(C)
        self.noise_prob = float(tabs.get("noise_prob", noise_prob))
        self.thr = threshold(self.noise_prob)
        self.n, self.seed, self.env_id_offset = int(n), int(seed), int(env_id_offset)
        self.rng_episodic, self.limit = bool(rng_episodic), int(max_episode_steps)
        self.reward_log2, self.replay = bool(reward_log2), bool(replay)
        radix = [S] * C if radix is None else [int(r) for r in radix]
        self.place = np.cumprod([1] + radix[:-1]).astype(np.uint64)
        self.se_partner = [(1 if C > 1 else 0) if j == 0 else j for j in range(C)]
        self.global_step = 0
        self.stats = np.zeros(8, np.int64)
        self.reset()

    # ---- state ---------------------------------------------------------------------------------
    def encode(self, cells):
        return ((np.asarray(cells).astype(np.uint64) * self.place[:, None]).sum(0) & np.uint64(0xFFFFFFFF)).astype(np.uint32)

    def reset(self):
        self.state = np.repeat(self.init[:, None], self.n, 1).astype(np.int8)
        self.t = np.zeros(self.n, np.int32)
        self.index = self.encode(self.state)

    def set_state(self, cells, t=None):
        self.state = np.asarray(cells, np.int8).reshape(self.C, self.n).copy()
        if t is not None:
            self.t = np.broadcast_to(np.asarray(t, np.int32), (self.n,)).copy()
        self.index = self.encode(self.state)

    def counter(self):
        """Per-env RNG counter T: the episode step under rng_episodic, else the global step (low 32 bits)."""
        if self.rng_episodic:
            return self.t.astype(np.uint64)
        return np.full(self.n, self.global_step & 0xFFFFFFFF, np.uint64)

    # ---- one step ------------------------------------------------------------------------------
    def fired(self, s, a, replay_u=None):
        """bool [C, n]: which cells' draws fire at this step."""
        want = self.draws[s, a]
        if not self.noise:
            return want
        if self.replay:
            return want & (np.asarray(replay_u, np.float64).T < self.noise_prob)
        v = ND.cell_draws(self.seed, self.C, self.env_id_offset, self.n, self.counter())
        return want & (v.astype(np.uint64) < np.uint64(self.thr))

    def step(self, actions, replay_u=None):
        s = self.state.astype(np.int64)
        a = np.asarray(actions, np.int64).reshape(self.C, self.n)
        fire = self.fired(s, a, replay_u)
        ns = np.where(fire, self.noisy[s, a], self.move[s, a])
        cell_r = np.where(fire, self.reward_noisy[s, a], self.reward[s, a])
        r = self.reward_pre_log = cell_r.sum(0)
        self.reward_abs = np.abs(cell_r).sum(0)
        if self.reward_log2:
            r = np.log2(1.0 + r)
        se_row = np.stack([self.se[j, ns[0], ns[p]] for j, p in enumerate(self.se_partner)])
        unsafe = (se_row == UNSAFE).any(0)
        count = self.counted[ns].sum(0)
        tn = self.t.astype(np.int64) + 1
        trunc = (tn >= self.limit) if self.limit > 0 else np.zeros(self.n, bool)
        self.final_state = ns.astype(np.int8)
        ns = np.where(trunc[None, :], self.init[:, None], ns)
        tn[trunc] = 0
        self.last_s, self.last_a = s, a
        self.last_fire, self.last_draws = fire, self.draws[s, a] & self.noise
        self.state, self.t, self.index = ns.astype(np.int8), tn.astype(np.int32), self.encode(ns)
        self.reward_out, self.se_row = r, se_row.astype(np.int8)
        self.unsafe, self.count, self.truncated = unsafe.astype(np.uint8), count.astype(np.uint8), trunc.astype(np.uint8)
        self.stats[:4] += (self.n, unsafe.sum(), count.sum(), trunc.sum())
        self.stats[4] += q24(r.astype(np.float32))
        self.global_step += 1
        return self

    # ---- policies of rollout / collect ---------------------------------------------------------
    def _ids(self):
        return np.arange(self.n, dtype=np.uint64) + np.uint64(self.env_id_offset)

    def random_actions(self):
        """Cell c of env g: floor(word * A / 2^32), word = word g % 4 of philox(g / 4, T, 0x40000000 + c)."""
        g, T = self._ids(), self.counter()
        out = np.zeros((self.C, self.n), np.int8)
        for c in range(self.C):
            w = np.stack(philox(g >> np.uint64(2), g >> np.uint64(34), T, ROLLOUT_STREAM + c, self.seed))
            word = w[(g & np.uint64(3)).astype(np.int64), np.arange(self.n)].astype(np.uint64)
            out[c] = ((word * np.uint64(self.A)) >> np.uint64(32)).astype(np.int8)
        return out

    def table_actions(self, policy):
        p = np.asarray(policy, np.int64)[self.index.astype(np.int64)]
        return np.stack([(p // self.A ** c) % self.A for c in range(self.C)]).astype(np.int8)

    def policy_actions(self, policy=None, epsilon=0.0):
        """Actions the fused kernels generate for the current step; exploration keyed by the global step."""
        if policy is None:
            return self.random_actions()
        a = self.table_actions(policy)
        if not epsilon > 0.0:
            return a
        batch = SimpleNamespace(n=self.n, cfg=SimpleNamespace(seed=self.seed, env_id_offset=self.env_id_offset))
        G = np.uint64(self.global_step & 0xFFFFFFFF)
        explore = _words(batch, G, EXPLORE_STREAM).astype(np.float64) * 2.0 ** -32 < epsilon
        joint = (_words(batch, G, EXPLORE_ACTION_STREAM).astype(np.uint64) * np.uint64(self.A ** self.C)) >> np.uint64(32)
        rnd = np.stack([(joint // np.uint64(self.A ** c)) % np.uint64(self.A) for c in range(self.C)]).astype(np.int8)
        return np.where(explore[None, :], rnd, a)

    def collect(self, n_steps, policy=None, epsilon=0.0):
        """n_steps x (policy actions -> step), recording obs, action, reward, flags and next_obs per step."""
        K, n = int(n_steps), self.n
        rec = dict(obs=np.zeros((K, n), np.uint32), action=np.zeros((K, n), np.uint32), reward=np.zeros((K, n)),
                   flags=np.zeros((K, n), np.uint8), next_obs=np.zeros((K, n), np.uint32))
        aplace = np.array([self.A ** c for c in range(self.C)], np.uint64)
        for k in range(K):
            a = self.policy_actions(policy, epsilon)
            rec["obs"][k] = self.index
            rec["action"][k] = (a.astype(np.uint64) * aplace[:, None]).sum(0).astype(np.uint32)
            self.step(a)
            rec["reward"][k] = self.reward_out
            rec["flags"][k] = self.unsafe | (self.truncated << 1) | (self.count << 2)
            rec["next_obs"][k] = self.encode(self.final_state)
        return rec
