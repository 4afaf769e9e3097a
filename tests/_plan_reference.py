"""numpy restatement of the planner's arithmetic (include/gym_cellular_b200_plan.h), bit for bit.

Per model: V_0 = +0.0; for k = 1..iters, sum = +0.0 plus p * V_{k-1}(s') over s' ascending, skipping p = 0, each
product and sum rounded on its own; Q_k = r + gamma * sum; pi_k = the first maximising action; V_k = Q_k(s, pi_k).
Vectorised over the (model, s, a) rows, one s' column at a time: numpy's float64 `*` and `+` are elementwise IEEE
operations without contraction, and a row receives at most one term per column, in ascending s'."""
import numpy as np


def estimate(visits, next_, reward_q24):
    """The counts' estimate, as count_and_plan.estimate: n = max(visits, 1) as a double, p = next / n,
    r = (reward_q24 * 2^-24) / n (unvisited pairs: no successor, reward 0)."""
    n = np.maximum(np.asarray(visits).astype(np.float64), 1.0)
    return np.asarray(next_).astype(np.float64) / n[..., None], np.asarray(reward_q24).astype(np.float64) * 2.0 ** -24 / n


def value_iteration(P, R, gamma, iters):
    """P float64 [..., nS, nA, nS], R [..., nS, nA] -> (policy int32 [..., nS], value float64 [..., nS],
    Q_iters float64 [..., nS, nA])."""
    P = np.asarray(P, dtype=np.float64)
    R = np.asarray(R, dtype=np.float64)
    lead, (nS, nA) = P.shape[:-3], P.shape[-3:-1]
    M = int(np.prod(lead, dtype=np.int64))
    flat = P.reshape(M * nS * nA, nS)
    model_of_row = np.arange(M * nS * nA) // (nS * nA)
    cols = []
    for t in range(nS):                       # the nonzeros of column s' = t: rows and p
        rows = np.flatnonzero(flat[:, t] != 0.0)
        cols.append((rows, flat[rows, t], model_of_row[rows] * nS + t))
    r = R.reshape(M * nS * nA)
    V = np.zeros(M * nS)
    for _ in range(iters):
        acc = np.zeros(M * nS * nA)
        for rows, p, vi in cols:
            acc[rows] = acc[rows] + p * V[vi]
        Q = (r + gamma * acc).reshape(M * nS, nA)
        pi = Q.argmax(axis=1)                 # the first maximum
        V = Q[np.arange(M * nS), pi]
    return (pi.astype(np.int32).reshape(*lead, nS), V.reshape(*lead, nS), Q.reshape(*lead, nS, nA))


def greedy_gap(Q):
    """Best minus second-best Q of every state (inf with one action)."""
    if Q.shape[-1] < 2:
        return np.full(Q.shape[:-1], np.inf)
    top = np.sort(Q, axis=-1)
    return top[..., -1] - top[..., -2]
