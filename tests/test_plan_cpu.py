"""The planner (libgymcellular_b200_plan.so, `value_iteration`) without a device: its exports, ABI version and ctypes
prototype against its header, every refusal of the C entry point, the ValueError cases of the Python surface, and the
numpy restatement of the arithmetic (tests/_plan_reference.py) against the examples' torch planners on CPU tensors."""
import ctypes as C
import importlib.util
import os
import re

import numpy as np
import pytest

import _plan_reference as PR
from conftest import REPO

torch = pytest.importorskip("torch")

HEADER = os.path.join(REPO, "include", "gym_cellular_b200_plan.h")


def _load():
    import __graft_entry__
    __graft_entry__.build()
    from gym_cellular_b200 import _plan_lib
    return _plan_lib, _plan_lib.load()


def test_planner_exports_and_abi_version():
    P, L = _load()
    header = open(HEADER).read()
    declared = sorted(set(re.findall(r"\b(gcp_[a-z_]+)\s*\(", header)))
    assert declared == sorted(P.EXPORTS)
    for name in declared:
        assert hasattr(L, name), name
    assert L.gcp_abi_version() == P.ABI_VERSION == int(re.search(r"GCP_ABI_VERSION (\d+)", header).group(1))
    assert P.MAX_STATES == int(re.search(r"GCP_MAX_STATES (\d+)", header).group(1))
    assert P.MAX_STATE_ACTIONS == int(re.search(r"GCP_MAX_STATE_ACTIONS (\d+)", header).group(1))
    # the env library is untouched: none of its exports is the planner's, and the planner's are not in it
    from gym_cellular_b200 import _lib
    assert not any(n.startswith("gcp_") for n in _lib.EXPORTS)
    assert not hasattr(C.CDLL(_lib.LIB_PATH), "gcp_value_iteration")


def test_prototype_and_struct_match_the_header():
    P, L = _load()
    header = open(HEADER).read()
    m = re.search(r"\bint\s+gcp_value_iteration\s*\(([^)]*)\)\s*;", header)
    params = [" ".join(p.split()) for p in m.group(1).split(",")]
    want = {"int": C.c_int, "double": C.c_double, "int32_t": C.c_int32}
    fn = L.gcp_value_iteration
    assert len(fn.argtypes) == len(params) == 7
    for p, t in zip(params, fn.argtypes):
        if p.startswith("const gcp_model"):
            assert t is C.POINTER(P.GcpModel), p
        elif "*" in p:
            assert t is C.c_void_p, p
        else:
            assert t is want[p.split()[0]], p
    body = re.search(r"typedef struct \{(.*?)\} gcp_model;", header, re.S).group(1)
    fields = re.findall(r"\b(\w+);", body)
    assert fields == [f for f, _ in P.GcpModel._fields_]
    assert C.sizeof(P.GcpModel) == 4 * 4 + 5 * 8


def _model(lib, **kw):
    base = dict(n_models=2, n_states=27, n_actions=27, visits=0x1000, next=0x2000, reward_q24=0x3000)
    base.update(kw)
    return lib.GcpModel(C.sizeof(lib.GcpModel), *(base.get(f) for f, _ in lib.GcpModel._fields_[1:]))


REFUSALS = [
    (dict(), dict(model=None), "model is NULL"),
    (dict(), dict(struct_size=8), "struct_size"),
    (dict(), dict(device=-1), "device"),
    (dict(n_models=0), dict(), ">= 1"),
    (dict(n_states=0), dict(), ">= 1"),
    (dict(n_actions=-3), dict(), ">= 1"),
    (dict(n_states=4097, n_actions=1), dict(), "limit of 4096"),
    (dict(n_states=4096, n_actions=33), dict(), "limit of 131072"),
    (dict(n_models=2 ** 16, n_states=64, n_actions=16), dict(), "2\\^31"),       # 2^32 entries
    (dict(P=0x4000, R=0x5000), dict(), "both"),
    (dict(visits=None, next=None, reward_q24=None), dict(), "neither"),
    (dict(next=None), dict(), "one is NULL"),
    (dict(visits=None, next=None, reward_q24=None, P=0x4000), dict(), "one is NULL"),
    (dict(reward_q24=0x3004), dict(), "8-byte aligned"),
    (dict(visits=None, next=None, reward_q24=None, P=0x4000, R=0x5002), dict(), "8-byte aligned"),
    (dict(), dict(policy=None), "must not be NULL"),
    (dict(), dict(value=None), "must not be NULL"),
    (dict(), dict(policy=0x6002), "aligned"),
    (dict(), dict(value=0x7004), "aligned"),
    (dict(), dict(gamma=-0.1), "gamma"),
    (dict(), dict(gamma=1.0000001), "gamma"),
    (dict(), dict(gamma=float("nan")), "gamma"),
    (dict(), dict(gamma=float("inf")), "gamma"),
    (dict(), dict(iters=0), "iters"),
]


@pytest.mark.parametrize("fields,call,msg", REFUSALS)
def test_every_refusal_needs_no_device(fields, call, msg):
    """Validated before any CUDA call: the fake addresses are never touched."""
    P, L = _load()
    m = _model(P, **fields)
    if "struct_size" in call:
        m.struct_size = call["struct_size"]
    args = dict(device=0, model=C.byref(m), gamma=0.95, iters=300, policy=0x6000, value=0x7000)
    args.update({k: v for k, v in call.items() if k != "struct_size"})
    rc = L.gcp_value_iteration(args["device"], args["model"], args["gamma"], args["iters"], args["policy"],
                               args["value"], None)
    assert rc == P.ERR_INVALID
    assert re.search(msg, L.gcp_last_error().decode()), L.gcp_last_error()


# ---------------------------------------------------------------------------------------------
# value_iteration: the checks of the Python surface (CPU and meta tensors: every one raises before the library is used)

def _counts(lead=(), nS=27, nA=27, device="cpu"):
    from gym_cellular_b200 import Counts
    z = lambda *s: torch.zeros(*lead, *s, dtype=torch.int64, device=device)      # noqa: E731
    return Counts(z(nS, nA), z(nS, nA, nS), z(nS, nA), z(nS, nA), None)


def test_value_iteration_value_errors():
    from gym_cellular_b200 import value_iteration
    c = _counts()
    for gamma in (-0.5, 1.5, float("nan"), float("inf"), True, "0.9", None):
        with pytest.raises(ValueError, match="gamma"):
            value_iteration(c, gamma=gamma)
    for iters in (0, -1, 2.0, True, 2 ** 31):
        with pytest.raises(ValueError, match="iters"):
            value_iteration(c, iters=iters)
    with pytest.raises(ValueError, match="transitions=True"):
        value_iteration(c._replace(next=None))
    with pytest.raises(ValueError, match="transitions=True"):
        value_iteration(c._replace(visits=None, next=None, reward_q24=None))
    with pytest.raises(ValueError, match="takes a Counts"):
        value_iteration(c.next)
    with pytest.raises(ValueError, match="takes a Counts"):
        value_iteration((c.next,))
    with pytest.raises(ValueError, match="int64"):
        value_iteration(c._replace(visits=c.visits.int()))
    with pytest.raises(ValueError, match="float64"):
        value_iteration((c.next.double(), c.visits))
    with pytest.raises(ValueError, match="float64"):
        value_iteration((c.next.float(), c.visits.double()))
    with pytest.raises(ValueError, match="torch tensor"):
        value_iteration((c.next.double().numpy(), c.visits.double()))
    with pytest.raises(ValueError, match="shape"):
        value_iteration(c._replace(next=torch.zeros(27, 27, 26, dtype=torch.int64)))
    with pytest.raises(ValueError, match="shape"):
        value_iteration(c._replace(next=torch.zeros(2, 2, 27, 27, 27, dtype=torch.int64)))
    with pytest.raises(ValueError, match="visits has shape"):
        value_iteration(c._replace(visits=torch.zeros(27, 26, dtype=torch.int64)))
    with pytest.raises(ValueError, match="R has shape"):                       # one R for many models: not taken
        value_iteration((torch.zeros(3, 27, 27, 27, dtype=torch.float64), torch.zeros(27, 27, dtype=torch.float64)))
    g = _counts((4,))
    with pytest.raises(ValueError, match="reward_q24 has shape"):              # groups must agree
        value_iteration(g._replace(reward_q24=g.reward_q24[:3]))
    with pytest.raises(ValueError, match="contiguous"):
        value_iteration(c._replace(visits=torch.zeros(27, 27, dtype=torch.int64).t()))
    with pytest.raises(ValueError, match="CUDA device"):
        value_iteration(c)
    with pytest.raises(ValueError, match="CUDA device"):
        value_iteration(g)
    with pytest.raises(ValueError, match="lives on"):
        value_iteration(c._replace(visits=c.visits.to("meta")))
    # limits, on meta tensors (shapes without memory)
    with pytest.raises(ValueError, match="limit of 4096"):
        value_iteration(_counts((), 4097, 1, "meta"))
    with pytest.raises(ValueError, match="limit of 131072"):
        value_iteration(_counts((), 4096, 33, "meta"))
    with pytest.raises(ValueError, match="2\\*\\*31"):
        value_iteration(_counts((65,), 1024, 32, "meta"))                      # 64 groups would be 2^31 exactly
    with pytest.raises(ValueError, match="CUDA device"):
        value_iteration(_counts((64,), 1024, 32, "meta"))
    with pytest.raises(ValueError, match="empty"):
        value_iteration(_counts((0,), 27, 27, "meta"))


# ---------------------------------------------------------------------------------------------
# the restatement against the examples' torch planners

def _example(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REPO, "examples", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def random_counts(rng, M, nS, nA, succ, unvisited=0.2):
    """Counts-like int64 tables: up to `succ` successors per (s, a), a share of unvisited pairs."""
    nxt = np.zeros((M, nS, nA, nS), np.int64)
    for idx in np.ndindex(M, nS, nA):
        if rng.random() < unvisited:
            continue
        to = rng.choice(nS, size=rng.integers(1, succ + 1), replace=False)
        nxt[idx + (to,)] = rng.integers(1, 50, size=to.size)
    visits = nxt.sum(-1)
    reward_q24 = (rng.normal(size=visits.shape) * visits * 2.0 ** 24).astype(np.int64)
    return visits, nxt, reward_q24


def _assert_close_to_torch(P, R, pol_t, V_t=None, gamma=0.95, iters=300):
    pi, V, Q = PR.value_iteration(P, R, gamma, iters)
    gap = PR.greedy_gap(Q)
    clear = gap > 1e-9
    assert clear.mean() > 0.5
    assert (pi[clear] == pol_t[clear]).all()
    if V_t is not None:
        np.testing.assert_allclose(V, V_t, rtol=1e-12, atol=0)
    return pi, V


def test_reference_matches_count_and_plan_on_counts():
    cp = _example("count_and_plan")
    rng = np.random.default_rng(0)
    for nS, nA, succ in ((27, 27, 8), (400, 25, 9)):
        visits, nxt, rq = random_counts(rng, 1, nS, nA, succ)
        from gym_cellular_b200 import Counts
        c = Counts(*(torch.from_numpy(x[0]) for x in (visits, nxt, rq)), None, None)
        Pt, Rt = cp.estimate(c)
        Pn, Rn = PR.estimate(visits[0], nxt[0], rq[0])
        assert np.array_equal(Pt.numpy(), Pn) and np.array_equal(Rt.numpy(), Rn)        # the estimate: bit for bit
        # torch's value of the same iteration, for the 1e-12 comparison
        V = torch.zeros(nS, dtype=torch.float64)
        for _ in range(300):
            V = (Rt + 0.95 * (Pt @ V)).max(dim=1).values
        _assert_close_to_torch(Pn, Rn, cp.value_iteration(Pt, Rt).numpy(), V.numpy())


def test_reference_matches_batched_posterior_plan():
    ps = _example("posterior_sampling")
    g = torch.Generator().manual_seed(1)
    M, nS, nA = 8, 27, 27
    alpha = torch.rand(nS, nA, nS, generator=g, dtype=torch.float64) + 0.1
    P = torch.distributions.Dirichlet(alpha).sample((M,))
    R = torch.randn(M, nS, nA, generator=g, dtype=torch.float64)
    V = torch.zeros(M, nS, dtype=torch.float64)
    for _ in range(300):
        V = (R + 0.95 * torch.einsum("msat,mt->msa", P, V)).max(dim=2).values
    pi, _ = _assert_close_to_torch(P.numpy(), R.numpy(), ps.plan(P, R).numpy(), V.numpy())
    assert pi.shape == (M, nS) and pi.dtype == np.int32


def test_reference_rules():
    """gamma = 0 is the argmax of R; exact ties go to the smallest action; iters = 1; skipped zeros change no bit."""
    rng = np.random.default_rng(2)
    R = rng.integers(0, 3, size=(5, 4)).astype(np.float64)
    P = rng.dirichlet(np.ones(5), size=(5, 4))
    pi, V, _ = PR.value_iteration(P, R, 0.0, 7)
    assert (pi == R.argmax(1)).all() and (V == R.max(1)).all()
    pi1, V1, Q1 = PR.value_iteration(P, R, 0.9, 1)
    assert (Q1 == R).all() and (pi1 == R.argmax(1)).all()
    # a deterministic chain 0 -> 1 -> ... -> 4 -> 4, reward 1 a step, gamma 1: V_k(s) = k
    chain = np.zeros((5, 2, 5))
    for s in range(5):
        chain[s, :, min(s + 1, 4)] = 1.0
    pi, V, _ = PR.value_iteration(chain, np.ones((5, 2)), 1.0, 6)
    assert (V == 6.0).all() and (pi == 0).all()
