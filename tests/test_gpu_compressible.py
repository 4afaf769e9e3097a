"""Env-owned step buffers in generic compressible memory give bit-identical results to ordinary memory: config 4 at
2^24 envs on both layouts, config 5's cellular part with a time limit, the host path, and a sequence with
load_state_dict and a table swap.  With compression forced off the allocator falls back to ordinary memory."""
import ctypes as C
import gc

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from test_gpu_tables import make_tables      # noqa: E402


@pytest.fixture(scope="module")
def B():
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


def outputs(env):
    torch.cuda.synchronize()
    return {name: t.clone() for name, t in zip(("state", "t", "reward", "index", "f4", "f5", "f6", "f7"),
                                                env._step_buffers())} | {"stats": env._stats.clone()}


def assert_same(a, b):
    for k in a:
        assert torch.equal(a[k], b[k]), k


def pair(cls, **kw):
    comp = cls(compressible_buffers=True, **kw)
    plain = cls(compressible_buffers=False, **kw)
    assert not plain.compressible
    return comp, plain


def supported(B):
    return bool(B._lib.load().gc_compressible_supported(torch.cuda.current_device()))


@pytest.mark.parametrize("packed", [False, True])
def test_config4_bit_identical(B, packed):
    cls = B.PackedCellularVectorEnv if packed else B.CellularVectorEnv
    comp, plain = pair(cls, num_envs=1 << 24, n_cells=16, n_states=4, emit_side_effects=False)
    assert comp.compressible == supported(B)
    gen = torch.Generator(device="cuda").manual_seed(5)
    ring = []
    for _ in range(3):
        a = torch.randint(0, 4, (16, comp.ld), dtype=torch.int8, device="cuda", generator=gen)
        if packed:
            w = torch.zeros(comp.ld, dtype=torch.int32, device="cuda")
            w[:comp.num_envs] = comp.pack(a[:, :comp.num_envs])
            a = w
        ring.append(a)
    for env in (comp, plain):
        env.step_many([env._bind(a) for a in ring], 10)
    assert_same(outputs(comp), outputs(plain))


def test_config5_cellular_time_limit(B):
    kw = dict(num_envs=(1 << 22) + 48, n_cells=3, n_states=3, stochastic=True, max_episode_steps=4, env_seed=3,
              emit_final_obs=True)
    comp, plain = pair(B.CellularVectorEnv, **kw)
    gen = torch.Generator(device="cuda").manual_seed(7)
    for _ in range(9):
        a = torch.randint(0, 3, (3, comp.ld), dtype=torch.int8, device="cuda", generator=gen)
        comp.step_device(a)
        plain.step_device(a)
    assert_same(outputs(comp), outputs(plain))
    assert torch.equal(comp._final, plain._final)


@pytest.mark.parametrize("packed", [False, True])
def test_host_path(B, packed):
    cls = B.PackedCellularVectorEnv if packed else B.CellularVectorEnv
    comp, plain = pair(cls, num_envs=(1 << 21) + 16, n_cells=16, n_states=4, stochastic=True, max_episode_steps=3,
                       host_chunk_envs=1 << 19)
    rng = np.random.default_rng(1)
    for _ in range(4):
        a = rng.integers(0, 4, size=(16, comp.num_envs)).astype(np.int8)
        if packed:
            from gym_cellular_b200.packed_env import pack_host
            a = pack_host(a)
        ra, rb = comp.step(a), plain.step(a)
        for x, y in zip(ra[:4], rb[:4]):
            for u, v in zip(x if isinstance(x, tuple) else (x,), y if isinstance(y, tuple) else (y,)):
                assert np.array_equal(np.asarray(u), np.asarray(v))
    assert_same(outputs(comp), outputs(plain))


def test_state_dict_and_table_swap(B):
    from gym_cellular_b200 import _lib
    tabs, alt = (make_tables(s, 5, 4, 3, noise=True, se_mode="pair") for s in (11, 12))
    for t in (tabs, alt):
        t["noise_prob"] = 0.3
    comp, plain = pair(B.CellularVectorEnv, num_envs=4099, cell_tables=tabs, env_seed=2, max_episode_steps=6)
    rng = np.random.default_rng(2)
    acts = [torch.from_numpy(rng.integers(0, 3, size=(5, 4099)).astype(np.int8)).cuda() for _ in range(12)]
    for a in acts[:4]:
        comp.step_device(a)
        plain.step_device(a)
    sd = plain.state_dict()
    for a in acts[4:7]:
        comp.step_device(a)
    comp.load_state_dict(sd)
    arr = {k: None if alt.get(k) is None else np.ascontiguousarray(alt[k], dt) for k, dt in (
        ("move", np.int8), ("noisy", np.int8), ("draws", np.uint8), ("reward", np.float32), ("side_effects", np.int8),
        ("counted", np.uint8), ("initial_state", np.int8), ("reward_noisy", np.float32))}
    t = _lib.GcCellTables(*[None if arr[k] is None else arr[k].ctypes.data for k in (
        "move", "noisy", "draws", "reward", "side_effects", "counted", "initial_state", "reward_noisy")], None)
    torch.cuda.synchronize()
    for env in (comp, plain):
        _lib.check(env._lib.gc_set_tables(env._h, C.byref(t)))
    for a in acts[7:]:
        comp.step_device(a)
        plain.step_device(a)
    assert_same(outputs(comp), outputs(plain))
    assert comp.sync_step_counter() == plain.sync_step_counter()


def test_forced_off_falls_back(B, monkeypatch):
    monkeypatch.setenv("GC_B200_COMPRESSIBLE", "0")
    assert B._lib.load().gc_compressible_supported(torch.cuda.current_device()) == 0
    comp, plain = pair(B.CellularVectorEnv, num_envs=1 << 16, n_cells=16, n_states=4)
    assert not comp.compressible
    a = torch.randint(0, 4, (16, comp.ld), dtype=torch.int8, device="cuda")
    for env in (comp, plain):
        env.step_device(a)
    assert_same(outputs(comp), outputs(plain))
    auto = B.CellularVectorEnv(num_envs=1 << 10)
    assert not auto._compressible_buffers


@pytest.mark.parametrize("packed", [False, True])
def test_auto_only_for_large_shards(B, packed):
    cls = B.PackedCellularVectorEnv if packed else B.CellularVectorEnv
    assert not cls(num_envs=1 << 16, n_cells=3, n_states=3)._compressible_buffers     # config 2: latency-bound
    assert cls(num_envs=1 << 24, n_cells=16, n_states=4).compressible == supported(B)


def test_views_keep_the_memory(B):
    L = B._lib.load()
    if not supported(B):
        pytest.skip("the device grants no compressible memory")
    env = B.CellularVectorEnv(num_envs=1 << 16, n_cells=16, n_states=4, compressible_buffers=True)
    env.step_device(torch.ones(16, env.ld, dtype=torch.int8, device="cuda"))
    view, ptr = env._v_reward, env._reward.data_ptr()
    expect = view.clone()
    env.close()
    del env
    gc.collect()
    assert L.gc_is_compressible(C.c_void_p(ptr)) == 1       # the view returned by step() still holds its allocation
    assert torch.equal(view, expect)
    del view
    gc.collect()
    assert L.gc_is_compressible(C.c_void_p(ptr)) == 0       # the last view gone, the mapping is released
