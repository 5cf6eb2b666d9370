"""CPU checks of the device-side tier fetch: without a CUDA device the calls fail loudly, and the workspace size is
plain arithmetic over the slot sizes."""
import numpy as np
import pytest

import cxl_speckv_b200 as pkg


@pytest.fixture(scope="module")
def L():
    try:
        return pkg.lib()
    except ImportError as e:  # pragma: no cover
        pytest.skip(str(e))


def test_fetch_entry_points_fail_loudly_without_gpu(L):
    if L.speckv_ext_device_count() > 0:
        pytest.skip("a GPU is present")
    assert L.speckv_ext_tier_enable_fetch(None, None) == pkg.SPECKV_ERR_DRIVER
    ids = np.zeros(4, dtype=np.uint64)
    ws = np.zeros(64, dtype=np.uint8)
    assert L.speckv_ext_tier_fetch(None, ids.ctypes.data, None, 4, 2048, 0, 2, ws.ctypes.data, None, None, None,
                                   ws.ctypes.data, ws.size, None) == pkg.SPECKV_ERR_DRIVER
    assert L.speckv_ext_tier_fetch(None, None, None, 0, 2048, 0, 2, None, None, None, None, None, 0,
                                   None) == pkg.SPECKV_ERR_DRIVER


@pytest.mark.parametrize("G", [1, 1000, 2048, 4096, 131072])
@pytest.mark.parametrize("n", [0, 1, 7, 1024])
def test_workspace_bytes_covers_every_slot(L, G, n):
    ws = L.speckv_ext_tier_fetch_workspace_bytes(n, G)
    slots = [L.speckv_ext_slot_bytes(G, s) for s in range(5)]
    assert ws == n * (L.speckv_ext_slot_bytes(G, pkg.COMP_INT8_DELTA_RLE) + 24) + 8
    assert ws >= n * max(slots) + 24 * n + 8     # staging at the largest slot + offsets, pool offsets, sizes, scales, total
    assert max(slots) % 16 == 0                  # the metadata behind the staging stays 8-byte aligned
