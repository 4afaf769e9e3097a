"""Compressible step buffers without a GPU: the allocator's symbols resolve through ctypes and report no device, and
compressible_buffers=False keeps the env's step buffers on torch's own allocator."""
import ctypes as C
from types import SimpleNamespace

import pytest

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def L():
    from gym_cellular_b200 import _lib
    return _lib.load()


def test_symbols_resolve(L):
    for name in ("gc_compressible_supported", "gc_alloc_compressible", "gc_free_compressible", "gc_is_compressible"):
        assert C.cast(getattr(L, name), C.c_void_p).value


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the answers on a machine without a device")
def test_no_device_no_memory(L):
    assert L.gc_compressible_supported(0) == 0
    assert not L.gc_alloc_compressible(1 << 20, 0, None)
    assert L.gc_is_compressible(None) == 0
    L.gc_free_compressible(None, 0, 0, None)          # freeing NULL is a no-op, as for cudaFree


def test_disabled_uses_torch_zeros():
    from gym_cellular_b200 import CellularVectorEnv
    stub = SimpleNamespace(device=torch.device("cpu"), _compressible_buffers=False)
    zeros = CellularVectorEnv._step_buffer_zeros(stub)
    t = zeros(3, 32, dtype=torch.int8)
    assert t.shape == (3, 32) and t.dtype == torch.int8 and t.device.type == "cpu" and not t.any()
