"""CPU checks of the ragged-group entry points: without a CUDA device they fail loudly, like every codec call."""
import ctypes as C

import numpy as np
import pytest
import torch

import cxl_speckv_b200 as pkg
from cxl_speckv_b200 import codec


@pytest.fixture(scope="module")
def L():
    try:
        return pkg.lib()
    except ImportError as e:  # pragma: no cover
        pytest.skip(str(e))


def test_ragged_entry_points_fail_loudly_without_gpu(L):
    if L.speckv_ext_device_count() > 0:
        pytest.skip("a GPU is present")
    assert L.speckv_ext_compress_ragged(None, None, None, 0, 2048, 1, None, 4096, None, None, 2, None) == pkg.SPECKV_ERR_DRIVER
    assert L.speckv_ext_compress_ragged(None, None, None, 0, 2048, 1, None, 4096, None, None, 0, None) == pkg.SPECKV_ERR_DRIVER
    ids = np.zeros(1, dtype=np.uint64)
    assert L.speckv_ext_tier_offload_ragged(None, None, None, None, 0, 2048, 1, ids.ctypes.data, None) == pkg.SPECKV_ERR_DRIVER
    tier = C.c_void_p()
    assert L.speckv_ext_tier_create(1 << 20, C.byref(tier)) == pkg.SPECKV_ERR_DRIVER


def test_compress_ragged_rejects_host_tensors():
    with pytest.raises(ValueError):
        codec.compress_ragged(torch.zeros(2048, dtype=torch.float16), 2048, torch.zeros(1, dtype=torch.int32))
