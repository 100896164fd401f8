"""GPU tests (-m gpu): the record array in compressible device memory (pom_batch_records_compressed).  Every other GPU
test runs on such records too; these check what the allocation itself decides: that a device with generic compression
gets it, that sizes which do not fill the allocation granularity step right, and that destroy gives everything back."""
import ctypes as C
import os

import pytest

from test_gpu_parity import _run_vs_oracle

pytestmark = pytest.mark.gpu


class _AllocProp(C.Structure):
    """CUmemAllocationProp (cuda.h)"""
    _fields_ = [("type", C.c_int), ("requestedHandleTypes", C.c_int), ("loc_type", C.c_int), ("loc_id", C.c_int),
                ("win32HandleMetaData", C.c_void_p), ("compressionType", C.c_ubyte), ("gpuDirectRDMACapable", C.c_ubyte),
                ("usage", C.c_ushort), ("reserved", C.c_ubyte * 4)]


@pytest.fixture(scope="module")
def pb():
    import pomcpp_b200 as pb
    assert os.path.exists(pb.LIB_PATH), "libpom_b200.so missing on the GPU box"
    assert pb.device_count() > 0, "no CUDA device"
    return pb


@pytest.fixture(scope="module")
def cu():
    cu = C.CDLL("libcuda.so.1")
    assert cu.cuInit(0) == 0
    return cu


def _compression(cu, device=0):
    """(CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, minimum granularity of a compressible allocation or None)"""
    dev, v, g = C.c_int(), C.c_int(), C.c_size_t()
    assert cu.cuDeviceGet(C.byref(dev), device) == 0
    assert cu.cuDeviceGetAttribute(C.byref(v), 107, dev) == 0
    p = _AllocProp(type=1, loc_type=1, loc_id=dev.value, compressionType=1)
    gran = g.value if v.value and cu.cuMemGetAllocationGranularity(C.byref(g), C.byref(p), 0) == 0 else None
    return v.value, gran


def _free_bytes(cu):
    free, total = C.c_size_t(), C.c_size_t()
    assert cu.cuMemGetInfo_v2(C.byref(free), C.byref(total)) == 0
    return free.value


def test_one_mi_env_records_are_compressed_where_the_device_supports_it(pb, cu):
    supported, _ = _compression(cu)
    b = pb.Batch(1 << 20, n_templates=16)
    assert b.records_compressed() == bool(supported)
    b.close()


def test_ragged_sizes_step_like_the_oracle(pb, orc, cu):
    _, gran = _compression(cu)
    past_one_granule = (gran or 2 << 20) // pb.REC_BYTES + 1      # the records need a second granule
    for n in (1, 31, 33, 4099, past_one_granule):
        _run_vs_oracle(pb, orc, n, 40, 6, 1, 47 + n, n_templates=7)


def test_create_and_destroy_give_the_memory_back(pb, cu):
    _, gran = _compression(cu)

    def one():
        b = pb.Batch(4099, n_templates=7)
        mv = b.alloc(4 * 4099)
        b.generate_moves(mv, 5, 0, 6)
        b.step(mv, pb.STEP_AUTORESET)
        b.sync()
        b.free(mv)
        b.close()
    one()                                   # module loads, the context's own allocations
    before = _free_bytes(cu)
    for _ in range(50):
        one()
    after = _free_bytes(cu)
    # a handle's records alone are one granule (2 MiB) or more: 50 leaked handles would be far outside this margin
    assert abs(before - after) <= 2 * (gran or 2 << 20), (before, after)
