"""Reference for experience collection (gc_collect), built on the oracle's existing step and policy actions.

The epsilon-greedy draws are restated here in numpy (DESIGN.md §4, RNG table) rather than taken from the kernels:
env g at global step G explores when u * 2^-32 < epsilon for u = word (g % 4) of
philox(key, ((g/4)_lo, (g/4)_hi, G, 0x50000000)); an exploring env takes, with v = word (g % 4) of
philox(key, ((g/4)_lo, (g/4)_hi, G, 0x50000001)), the joint action floor(v * A^C / 2^32) (cellular, digits cell 0
first) or the rollout's random grid-world action (jurisdiction = bit 31, position = bits 29-30); any other env the
table action.  G is the global step also for episodic envs.
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)


def philox(c0, c1, c2, c3, seed):
    """Philox4x32-10 over arrays of counters; returns the four output words as uint32 arrays."""
    c = [np.asarray(x, np.uint64) & _LO for x in (c0, c1, c2, c3)]
    c = np.broadcast_arrays(*c)
    c0, c1, c2, c3 = (x.copy() for x in c)
    k0, k1 = int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & _LO, (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & _LO
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return tuple(x.astype(np.uint32) for x in (c0, c1, c2, c3))


def _words(ora, G, stream):
    g = np.arange(ora.n, dtype=np.uint64) + np.uint64(ora.cfg.env_id_offset)
    w = np.stack(philox(g >> np.uint64(2), g >> np.uint64(34), G, stream, ora.cfg.seed))
    return w[(g & np.uint64(3)).astype(np.int64), np.arange(ora.n)]


def explore_actions(ora, policy, epsilon):
    """int8 [C, n] actions of the epsilon-greedy table policy for the oracle's current step."""
    a = ora.policy_actions(policy)
    if not epsilon > 0.0:
        return a
    G = np.uint64(ora.global_step & 0xFFFFFFFF)
    explore = _words(ora, G, 0x50000000).astype(np.float64) * 2.0 ** -32 < epsilon
    v = _words(ora, G, 0x50000001).astype(np.uint64)
    if ora.cfg.kind == 1:                                      # grid world
        jur, pos = (v >> np.uint64(31)).astype(np.int64), ((v >> np.uint64(29)) & np.uint64(3)).astype(np.int8)
        rnd = np.stack([np.where(jur == 0, pos, 4), np.where(jur == 1, pos, 4)]).astype(np.int8)
    else:
        A = ora.cfg.n_actions
        joint = (v * np.uint64(A ** ora.C)) >> np.uint64(32)             # A^C <= 2^32: the product fits 64 bits
        rnd = np.stack([(joint // np.uint64(A ** c)) % np.uint64(A) for c in range(ora.C)]).astype(np.int8)
    return np.where(explore[None, :], rnd, a)


def collect(ora, n_steps, policy=None, epsilon=0.0):
    """n_steps x (actions -> oracle step), recording every step: (obs, action, reward, flags), each [n_steps, n].
    obs = tabular index the step starts from, action = tabular index of the executed action (radix n_actions;
    grid world a_0 + 5 a_1), flags = unsafe | truncated << 1 | count << 2."""
    K, n = int(n_steps), ora.n
    obs = np.zeros((K, n), np.uint32)
    act = np.zeros((K, n), np.uint32)
    rew = np.zeros((K, n), np.float64)
    flags = np.zeros((K, n), np.uint8)
    radix = 5 if ora.cfg.kind == 1 else ora.cfg.n_actions
    place = np.array([radix ** c for c in range(ora.C)], np.uint64)
    for k in range(K):
        a = ora.policy_actions(None) if policy is None else explore_actions(ora, policy, epsilon)
        obs[k] = ora.index
        act[k] = (a.astype(np.uint64) * place[:, None]).sum(0).astype(np.uint32)
        ora.step(a)
        rew[k] = ora.reward
        flags[k] = ora.unsafe | (ora.truncated << 1) | (ora.count << 2)
    return obs, act, rew, flags
