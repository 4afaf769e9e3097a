"""Value iteration on the device: every model of a batch planned in one kernel launch (libgymcellular_b200_plan.so).

    plan = value_iteration(counts, gamma=0.95, iters=300)   # Counts of zero_counts() or zero_counts(groups=P)
    plan.policy                                             # int32 [nS] or [P, nS]: rollout(policy) / policy_of_env=
    plan.value                                              # float64, the same leading shape
    plan = value_iteration((P, R), gamma, iters)            # float64 P [nS, nA, nS] / [M, nS, nA, nS], R [.., nS, nA]

The arithmetic is that of the examples' torch planners, stated exactly in include/gym_cellular_b200_plan.h: the counts
give P_hat = next / max(visits, 1) and R_hat = reward_q24 * 2^-24 / max(visits, 1) (count_and_plan.estimate), V_0 = 0,
Q_k = R + gamma * (P @ V_{k-1}) with every product and sum rounded on its own, ascending s', V_k = max_a Q_k, and the
policy is the first maximising action of Q_iters (torch.argmax's rule).
"""
import ctypes as C
import math
from collections import namedtuple

import torch

from . import _plan_lib


class Plan(namedtuple("Plan", "policy value")):
    """Result of `value_iteration`: the greedy policy int32 and its value V_iters float64, [nS] or [M, nS]."""
    __slots__ = ()


def _tables(model):
    """-> (kind, tables, leading shape, (M, nS, nA)) of Counts or a (P, R) pair, after every check."""
    from .vector_env import Counts
    if isinstance(model, Counts):
        vis, nxt, rq = model.visits, model.next, model.reward_q24
        if vis is None or nxt is None or rq is None:
            raise ValueError("value_iteration needs counts with visits, next and reward_q24 (zero_counts() with "
                             "joint=True and transitions=True)")
        tabs, dtype, names, trans = (vis, nxt, rq), torch.int64, ("visits", "next", "reward_q24"), nxt
    elif isinstance(model, (tuple, list)) and len(model) == 2:
        tabs, dtype, names = tuple(model), torch.float64, ("P", "R")
        trans = tabs[0]
    else:
        raise ValueError("value_iteration takes a Counts or a (P, R) pair of float64 tensors")
    for name, t in zip(names, tabs):
        if not isinstance(t, torch.Tensor):
            raise ValueError(f"{name} must be a torch tensor")
        if t.dtype != dtype:
            raise ValueError(f"{name} must be {dtype}, not {t.dtype}")
    if trans.dim() not in (3, 4) or trans.shape[-1] != trans.shape[-3]:
        raise ValueError(f"{'P' if dtype == torch.float64 else 'next'} must have shape [nS, nA, nS] or "
                         f"[M, nS, nA, nS]; got {tuple(trans.shape)}")
    lead = tuple(trans.shape[:-3])
    nS, nA = trans.shape[-3], trans.shape[-2]
    for name, t in zip(names, tabs):
        want = lead + ((nS, nA, nS) if t is trans else (nS, nA))
        if tuple(t.shape) != want:
            raise ValueError(f"{name} has shape {tuple(t.shape)}; expected {want}")
        if not t.is_contiguous():
            raise ValueError(f"{name} must be contiguous")
        if t.device != trans.device:
            raise ValueError(f"{name} lives on {t.device}, the transitions on {trans.device}")
    M = lead[0] if lead else 1
    if M < 1 or nS < 1 or nA < 1:
        raise ValueError(f"empty models: {M} x {nS} states x {nA} actions")
    if nS > _plan_lib.MAX_STATES:
        raise ValueError(f"{nS} states exceed the planner's limit of {_plan_lib.MAX_STATES}")
    if nS * nA > _plan_lib.MAX_STATE_ACTIONS:
        raise ValueError(f"{nS} x {nA} state-action pairs exceed the planner's limit of {_plan_lib.MAX_STATE_ACTIONS}")
    if M * nS * nA * nS > 2 ** 31:
        raise ValueError(f"{M} models of {nS} x {nA} x {nS} exceed 2**31 entries in all")
    if trans.device.type != "cuda":
        raise ValueError(f"value_iteration runs on a CUDA device; the tables live on {trans.device}")
    return ("counts" if dtype == torch.int64 else "model"), tabs, lead, (M, nS, nA)


def value_iteration(model, gamma=0.95, iters=300):
    """Value iteration of every model in one kernel launch on the current stream of the tables' device.

    model: `Counts` (from `zero_counts()` or `zero_counts(groups=P)`, visits / next / reward_q24 required), planned on
    the estimate P_hat / R_hat formed inside the kernel; or a pair (P, R) of float64 tensors, P [nS, nA, nS] or
    [M, nS, nA, nS] and R [nS, nA] or [M, nS, nA], assumed finite (e.g. `exact_model`, or sampled models).  Every table
    contiguous on one CUDA device; nS <= 4096, nS * nA <= 2**17, M * nS * nA * nS <= 2**31; gamma finite in [0, 1];
    iters >= 1.  A failed check raises ValueError before any launch.

    Returns Plan(policy int32, value float64), [nS] or [M, nS] (M = the groups of grouped counts): the policy feeds
    `rollout(policy)` or, as a stack, `policy_of_env=`.  Nothing here reads the data on the host, so a call adds no
    synchronisation and can be captured into a CUDA graph; non-finite entries give non-finite values, never an access
    outside the tables."""
    if isinstance(gamma, bool) or not isinstance(gamma, (int, float)) or not math.isfinite(gamma) or not 0 <= gamma <= 1:
        raise ValueError(f"gamma must be a finite number in [0, 1] (got {gamma!r})")
    if isinstance(iters, bool) or not isinstance(iters, int) or not 1 <= iters < 2 ** 31:
        raise ValueError(f"iters must be an int >= 1 (got {iters!r})")
    kind, tabs, lead, (M, nS, nA) = _tables(model)
    L = _plan_lib.load()
    device = tabs[0].device
    policy = torch.empty(*lead, nS, dtype=torch.int32, device=device)
    value = torch.empty(*lead, nS, dtype=torch.float64, device=device)
    ptrs = [t.data_ptr() for t in tabs]
    m = _plan_lib.GcpModel(C.sizeof(_plan_lib.GcpModel), M, nS, nA,
                           *(ptrs + [None, None] if kind == "counts" else [None, None, None] + ptrs))
    stream = torch.cuda.current_stream(device).cuda_stream
    _plan_lib.check(L.gcp_value_iteration(device.index, C.byref(m), float(gamma), int(iters), policy.data_ptr(),
                                          value.data_ptr(), stream))
    return Plan(policy, value)
