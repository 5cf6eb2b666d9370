"""CPU: the KV cache set entry points without a device, the argument checks of speckv_ext_cache_set_create, and the
host-side parts of KVCacheSet and CxlSpeckvKVAllocator.register_kv_caches (geometry checks, the cache-major groups
and the default block ids of offload_request) on CPU tensors."""
import ctypes as C

import numpy as np
import pytest
import torch

import cxl_speckv_b200 as pkg
from cxl_speckv_b200 import build as pkg_build
from cxl_speckv_b200.codec import KVCacheSet
from cxl_speckv_b200.vllm_speckv_backend import CxlSpeckvKVAllocator


@pytest.fixture(scope="module")
def L():
    pkg_build.build()
    return pkg.lib()


def _bases(*addrs):
    return (C.c_void_p * len(addrs))(*addrs)


def test_set_entry_points_fail_loudly_without_gpu(L):
    if L.speckv_ext_device_count() > 0:
        pytest.skip("a GPU is present")
    out = C.c_void_p()
    fake = C.c_void_p(0x1000)
    assert L.speckv_ext_cache_set_create(_bases(0x1000, 0x2000), 2, 2048, 2048, 0, C.byref(out)) == pkg.SPECKV_ERR_DRIVER
    assert not out
    assert L.speckv_ext_compress_gather_set(fake, fake, fake, None, 1, fake, 4096, fake, fake, 2, None) == \
        pkg.SPECKV_ERR_DRIVER
    assert L.speckv_ext_decompress_scatter_set(fake, 4096, fake, fake, None, fake, fake, fake, 1, None, 2, None) == \
        pkg.SPECKV_ERR_DRIVER
    ids = np.zeros(1, dtype=np.uint64)
    assert L.speckv_ext_tier_offload_set(fake, fake, fake, fake, None, 1, ids.ctypes.data, None) == pkg.SPECKV_ERR_DRIVER
    assert L.speckv_ext_tier_restore_set(fake, ids.ctypes.data, 1, fake, fake, fake, None) == pkg.SPECKV_ERR_DRIVER
    assert L.speckv_ext_tier_fetch_set(fake, fake, None, 1, fake, fake, fake, 2, None, None, fake, 1 << 20, None) == \
        pkg.SPECKV_ERR_DRIVER
    L.speckv_ext_cache_set_destroy(None)   # a no-op


def test_set_create_rejects_bad_arguments(L):
    out = C.c_void_p()
    ok = _bases(0x1000, 0x2000)
    assert L.speckv_ext_cache_set_create(None, 2, 2048, 2048, 0, C.byref(out)) == pkg.SPECKV_ERR_INVAL
    assert L.speckv_ext_cache_set_create(ok, 0, 2048, 2048, 0, C.byref(out)) == pkg.SPECKV_ERR_INVAL        # no cache
    assert L.speckv_ext_cache_set_create(ok, 2, 0, 2048, 0, C.byref(out)) == pkg.SPECKV_ERR_INVAL           # empty block
    assert L.speckv_ext_cache_set_create(ok, 2, 2048, 2047, 0, C.byref(out)) == pkg.SPECKV_ERR_INVAL        # stride < block
    assert L.speckv_ext_cache_set_create(ok, 2, 2048, 4096, 3, C.byref(out)) == pkg.SPECKV_ERR_INVAL        # dtype
    assert L.speckv_ext_cache_set_create(_bases(0x1000, 0), 2, 2048, 2048, 0, C.byref(out)) == pkg.SPECKV_ERR_INVAL
    assert L.speckv_ext_cache_set_create(ok, 2, 2048, 2048, 0, None) == pkg.SPECKV_ERR_INVAL
    assert not out


def test_kv_cache_set_checks_and_groups():
    caches = [torch.zeros(6, 4, 2, 8, dtype=torch.float16) for _ in range(3)]
    s = KVCacheSet(caches)
    assert (len(s), s.num_blocks, s.block_elems, s.block_stride, s.dtype) == (3, 6, 64, 64, torch.float16)
    ci, b = s.groups(torch.tensor([5, 0, 3], dtype=torch.int32))
    assert ci.dtype == torch.int32 and b.dtype == torch.int32
    assert ci.tolist() == [0, 0, 0, 1, 1, 1, 2, 2, 2]
    assert b.tolist() == [5, 0, 3] * 3
    with pytest.raises(ValueError):
        s.handle()                                               # no native set on CPU tensors
    # [num_blocks, 2, ...] views: blocks twice as far apart
    kv = torch.zeros(6, 2, 4, 2, 8, dtype=torch.bfloat16)
    s2 = KVCacheSet([kv[:, 0], kv[:, 1]])
    assert (s2.block_elems, s2.block_stride) == (64, 128)
    with pytest.raises(ValueError):
        KVCacheSet([])
    with pytest.raises(ValueError):
        KVCacheSet([caches[0], torch.zeros(5, 4, 2, 8, dtype=torch.float16)])            # shape
    with pytest.raises(ValueError):
        KVCacheSet([caches[0], torch.zeros(6, 4, 2, 8, dtype=torch.bfloat16)])           # dtype
    with pytest.raises(ValueError):
        KVCacheSet([kv[:, 0], caches[0].bfloat16()])                                     # strides
    with pytest.raises(ValueError):
        KVCacheSet([torch.zeros(6, 4, 2, 8).transpose(1, 2)])                           # a block not contiguous
    with pytest.raises(TypeError):
        KVCacheSet([torch.zeros(6, 4, dtype=torch.int32)])


@pytest.mark.parametrize("layout", ["2nb", "nb2"])
def test_register_kv_caches_and_default_ids(layout):
    shape = (2, 10, 16, 2, 8) if layout == "2nb" else (10, 2, 16, 2, 8)
    kv = {f"layer{i}": torch.zeros(shape, dtype=torch.float16) for i in range(3)}
    alloc = CxlSpeckvKVAllocator(pkg.lib_path(), "/dev/null")
    try:
        _check_register(alloc, kv, layout)
    finally:
        alloc._speckv.finalize()


def _check_register(alloc, kv, layout):
    with pytest.raises(RuntimeError):
        alloc.request_block_ids([1, 2])                                                  # nothing registered yet
    s = alloc.register_kv_caches(kv)
    assert len(s) == 6 and s.block_elems == 256 and s.block_stride == (256 if layout == "2nb" else 512)
    first = kv["layer1"][1] if layout == "2nb" else kv["layer1"][:, 1]
    assert s.caches[3].data_ptr() == first.data_ptr()                                   # cache 2 * layer + 1: V
    ids = alloc.request_block_ids(torch.tensor([9, 0, 4], dtype=torch.int32))
    assert ids.dtype == np.uint64 and ids.shape == (6, 3)
    for c in range(6):
        for j, b in enumerate([9, 0, 4]):
            assert int(ids[c, j]) == (c << 40) | b
    assert alloc._request_ids(s, torch.tensor([9, 0, 4]), None).tolist() == ids.reshape(-1).tolist()
    with pytest.raises(ValueError):
        alloc._request_ids(s, torch.tensor([9, 0, 4]), np.zeros((6, 2), dtype=np.uint64))
    with pytest.raises(ValueError):
        alloc.register_kv_caches([torch.zeros(3, 3, 16, 2, 8)])
