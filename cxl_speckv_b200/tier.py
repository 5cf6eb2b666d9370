"""Host tier: a pinned-DRAM pool standing in for the CXL memory pool (speckv_ext_tier_*).
Offload = compress on the GPU and move the payload to host memory; restore = the inverse."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import COMP_INT8_DELTA_RLE, check, lib
from .codec import _DTYPES, _stream


class HostTier:
    def __init__(self, pool_bytes: int):
        self._h = C.c_void_p()
        self._fetch_ws = {}   # fetch() workspaces by (requests, group_elems, device)
        check(lib().speckv_ext_tier_create(pool_bytes, C.byref(self._h)), "speckv_ext_tier_create")

    def close(self):
        if self._h:
            lib().speckv_ext_tier_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def set_scheme(self, scheme: int) -> None:
        """Scheme new offloads are stored under (0 .. 4); stored blocks keep theirs."""
        check(lib().speckv_ext_tier_set_scheme(self._h, int(scheme)), "speckv_ext_tier_set_scheme")

    def offload(self, x: torch.Tensor, group_elems: int, block_ids: np.ndarray) -> None:
        x = x.contiguous()
        ids = np.ascontiguousarray(block_ids, dtype=np.uint64)
        n = x.numel() // group_elems
        assert ids.size == n and x.numel() % group_elems == 0
        with torch.cuda.device(x.device):
            check(lib().speckv_ext_tier_offload(self._h, x.data_ptr(), _DTYPES[x.dtype], group_elems, n, ids.ctypes.data,
                                                _stream()), "speckv_ext_tier_offload")

    def restore(self, block_ids: np.ndarray, group_elems: int, dtype: torch.dtype, device="cuda:0",
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
        ids = np.ascontiguousarray(block_ids, dtype=np.uint64)
        if out is None:
            out = torch.empty((ids.size, group_elems), dtype=dtype, device=device)
        with torch.cuda.device(out.device):
            check(lib().speckv_ext_tier_restore(self._h, ids.ctypes.data, ids.size, group_elems, _DTYPES[dtype],
                                                out.data_ptr(), _stream()), "speckv_ext_tier_restore")
        return out

    def offload_blocks(self, cache: torch.Tensor, block_table: torch.Tensor, block_ids: np.ndarray) -> None:
        """Paged form: compress the blocks of a paged KV cache ([num_blocks, ...], one block = one codec
        group) named by `block_table` (CUDA int32) into the pool under `block_ids`, reading them in place."""
        assert cache.is_cuda and cache.is_contiguous()
        ids = np.ascontiguousarray(block_ids, dtype=np.uint64)
        table = block_table.to(device=cache.device, dtype=torch.int32).contiguous()
        assert ids.size == table.numel()
        with torch.cuda.device(cache.device):
            check(lib().speckv_ext_tier_offload_paged(self._h, cache.data_ptr(), table.data_ptr(), _DTYPES[cache.dtype],
                                                      cache[0].numel(), ids.size, ids.ctypes.data, _stream()),
                  "speckv_ext_tier_offload_paged")

    def offload_ragged(self, x: torch.Tensor, group_elems: int, lengths: torch.Tensor, block_ids: np.ndarray,
                       block_table: Optional[torch.Tensor] = None) -> None:
        """Store the filled prefix of blocks: block i (block block_table[i] of x, or block i of x without a table) is
        stored from its first min(lengths[i], group_elems) elements.  lengths: CUDA int32 element counts.  Restores
        write those elements back and leave the rest of each destination block untouched."""
        assert x.is_cuda and x.is_contiguous() and x.numel() % group_elems == 0
        ids = np.ascontiguousarray(block_ids, dtype=np.uint64)
        lengths = lengths.to(device=x.device, dtype=torch.int32).contiguous()
        assert ids.size == lengths.numel()
        if bool((lengths < 0).any()):   # the offload synchronises anyway; a negative length would store the whole block
            raise ValueError("offload_ragged: negative length")
        table = None
        if block_table is not None:
            table = block_table.to(device=x.device, dtype=torch.int32).contiguous()
            assert ids.size == table.numel()
        else:
            assert ids.size == x.numel() // group_elems
        with torch.cuda.device(x.device):
            check(lib().speckv_ext_tier_offload_ragged(self._h, x.data_ptr(), table.data_ptr() if table is not None else None,
                                                       lengths.data_ptr(), _DTYPES[x.dtype], group_elems, ids.size,
                                                       ids.ctypes.data, _stream()), "speckv_ext_tier_offload_ragged")

    def restore_blocks(self, block_ids: np.ndarray, cache: torch.Tensor, block_table: torch.Tensor) -> torch.Tensor:
        """Paged form: decompress the stored blocks `block_ids` straight into cache blocks `block_table`."""
        assert cache.is_cuda and cache.is_contiguous()
        ids = np.ascontiguousarray(block_ids, dtype=np.uint64)
        table = block_table.to(device=cache.device, dtype=torch.int32).contiguous()
        assert ids.size == table.numel()
        with torch.cuda.device(cache.device):
            check(lib().speckv_ext_tier_restore_paged(self._h, ids.ctypes.data, ids.size, cache[0].numel(),
                                                      _DTYPES[cache.dtype], cache.data_ptr(), table.data_ptr(), _stream()),
                  "speckv_ext_tier_restore_paged")
        return cache

    def drop(self, block_ids: np.ndarray) -> None:
        ids = np.ascontiguousarray(block_ids, dtype=np.uint64)
        check(lib().speckv_ext_tier_drop(self._h, ids.ctypes.data, ids.size), "speckv_ext_tier_drop")

    def enable_fetch(self) -> None:
        """Keep a device copy of the block directory from now on, so that fetch() finds blocks without the host.
        Call it on the tier's device (the current one when the tier was created)."""
        check(lib().speckv_ext_tier_enable_fetch(self._h, _stream()), "speckv_ext_tier_enable_fetch")

    def fetch(self, block_ids: torch.Tensor, group_elems: int, dtype: torch.dtype, scheme: int = COMP_INT8_DELTA_RLE,
              out: Optional[torch.Tensor] = None, block_table: Optional[torch.Tensor] = None,
              count: Optional[torch.Tensor] = None, out_elems: Optional[torch.Tensor] = None,
              status: Optional[torch.Tensor] = None):
        """Restore blocks named on the device (speckv_ext_tier_fetch): request i < count[0] (all of block_ids without
        a count) decodes stored block block_ids[i] into out[i], or into cache block block_table[i] of `out` (a paged
        cache of blocks of group_elems elements).  No host synchronisation, so a warm call can be captured into a CUDA
        graph.  block_ids: CUDA int64 ids; count: CUDA int32 [1] (e.g. from prefetch.route); block_table: CUDA int32.
        scheme names the decoder: 1 and 4 decode alike, so do 2 and 3; blocks stored under the other pair are not
        served.  -> (out, out_elems int32 [n], status uint8 [n]): status 1 = served; an unserved request (unknown id,
        other geometry, dtype or decoder, raw block) leaves its destination as it is and gets out_elems 0.  Entries
        at and behind the count are not written.  The workspace is cached per (len(block_ids), group_elems) and
        allocated on the first eager call of that shape: run one before capturing."""
        if not block_ids.is_cuda or block_ids.dtype not in (torch.int64, torch.uint64) or not block_ids.is_contiguous():
            raise TypeError("block_ids must be a contiguous CUDA int64 tensor")
        if dtype not in _DTYPES:
            raise TypeError(f"unsupported dtype {dtype}")
        dev = block_ids.device
        n = block_ids.numel()
        if count is not None and (not count.is_cuda or count.dtype != torch.int32 or count.device != dev):
            raise TypeError("count must be a CUDA int32 tensor on the device of block_ids")
        if block_table is not None:
            if out is None:
                raise ValueError("a block table needs the cache to write into (out)")
            if not block_table.is_cuda or block_table.dtype != torch.int32 or block_table.numel() < n or \
                    not block_table.is_contiguous():
                raise TypeError("block_table must be a contiguous CUDA int32 tensor with one entry per request")
        if out is None:
            out = torch.empty((n, group_elems), dtype=dtype, device=dev)
        if out.dtype != dtype or out.device != dev or not out.is_contiguous() or out.numel() % group_elems or \
                (block_table is None and out.numel() < n * group_elems):
            raise ValueError("out must be a contiguous tensor of whole blocks of `dtype` on the device of block_ids")
        if out_elems is None:
            out_elems = torch.zeros(n, dtype=torch.int32, device=dev)
        if status is None:
            status = torch.zeros(n, dtype=torch.uint8, device=dev)
        assert out_elems.numel() >= n and status.numel() >= n and out_elems.is_cuda and status.is_cuda
        ws = self._workspace(n, group_elems, dev)
        with torch.cuda.device(dev):
            check(lib().speckv_ext_tier_fetch(self._h, block_ids.data_ptr(), count.data_ptr() if count is not None else None,
                                              n, group_elems, _DTYPES[dtype], int(scheme), out.data_ptr(),
                                              block_table.data_ptr() if block_table is not None else None,
                                              out_elems.data_ptr(), status.data_ptr(), ws.data_ptr(), ws.numel(),
                                              _stream()), "speckv_ext_tier_fetch")
        return out, out_elems, status

    def _workspace(self, n: int, group_elems: int, dev: torch.device) -> torch.Tensor:
        key = (n, group_elems, dev)
        ws = self._fetch_ws.get(key)
        if ws is None:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("HostTier.fetch: no workspace for this shape yet; run one eager call before capturing")
            ws = torch.empty(max(lib().speckv_ext_tier_fetch_workspace_bytes(n, group_elems), 1), dtype=torch.uint8,
                             device=dev)
            self._fetch_ws[key] = ws
        return ws

    def stats(self) -> dict:
        s = _lib.TierStats()
        lib().speckv_ext_tier_get_stats(self._h, C.byref(s))
        return {k: getattr(s, k) for k, _ in s._fields_}


L1, L2, L3, UNALLOCATED = 0, 1, 2, 255


class TierPolicy:
    """Residency bookkeeping of the KV pages (speckv_ext_policy_*): the reference's
    CXLMemoryManager policy (src/cxl_memory/cxl_memory_manager.cpp:28-324) with the per-page state
    in device memory.  Page ids are dense indices; capacities count pages."""

    def __init__(self, n_pages: int, l1_pages: int, l2_pages: int = 1 << 62, l3_pages: int = 1 << 62):
        self._h = C.c_void_p()
        self.n_pages = n_pages
        check(lib().speckv_ext_policy_create(n_pages, l1_pages, l2_pages, l3_pages, C.byref(self._h)),
              "speckv_ext_policy_create")

    def close(self):
        if self._h:
            lib().speckv_ext_policy_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _ids(ids) -> np.ndarray:
        return np.ascontiguousarray(ids, dtype=np.uint64).ravel()

    def place(self, ids, tier: int) -> np.ndarray:
        ids = self._ids(ids)
        out = np.zeros(ids.size, dtype=np.uint8)
        check(lib().speckv_ext_policy_place(self._h, ids.ctypes.data, ids.size, tier, out.ctypes.data),
              "speckv_ext_policy_place")
        return out

    def release(self, ids) -> None:
        ids = self._ids(ids)
        check(lib().speckv_ext_policy_release(self._h, ids.ctypes.data, ids.size), "speckv_ext_policy_release")

    def touch(self, ids) -> None:
        """ids: a CUDA int64 tensor (stream-ordered, no synchronisation) or anything array-like on the host."""
        if isinstance(ids, torch.Tensor) and ids.is_cuda:
            ids = ids.contiguous()
            assert ids.dtype in (torch.int64, torch.uint64)
            with torch.cuda.device(ids.device):
                check(lib().speckv_ext_policy_touch(self._h, ids.data_ptr(), ids.numel(), 1, _stream()),
                      "speckv_ext_policy_touch")
            return
        ids = self._ids(ids)
        check(lib().speckv_ext_policy_touch(self._h, ids.ctypes.data, ids.size, 0, None), "speckv_ext_policy_touch")

    def is_hot(self, ids: torch.Tensor) -> torch.Tensor:
        ids = ids.contiguous()
        out = torch.empty(ids.numel(), dtype=torch.uint8, device=ids.device)
        with torch.cuda.device(ids.device):
            check(lib().speckv_ext_policy_is_hot(self._h, ids.data_ptr(), ids.numel(), out.data_ptr(), _stream()),
                  "speckv_ext_policy_is_hot")
        return out

    def promote(self, ids):
        """-> (ok[n] uint8, evicted page ids in order)"""
        ids = self._ids(ids)
        ok = np.zeros(ids.size, dtype=np.uint8)
        ev = np.zeros(max(ids.size, 1), dtype=np.uint64)
        n_ev = C.c_size_t()
        check(lib().speckv_ext_policy_promote(self._h, ids.ctypes.data, ids.size, ok.ctypes.data, ev.ctypes.data,
                                              C.byref(n_ev)), "speckv_ext_policy_promote")
        return ok, ev[:n_ev.value].copy()

    def demote(self, ids) -> np.ndarray:
        ids = self._ids(ids)
        ok = np.zeros(ids.size, dtype=np.uint8)
        check(lib().speckv_ext_policy_demote(self._h, ids.ctypes.data, ids.size, ok.ctypes.data),
              "speckv_ext_policy_demote")
        return ok

    def tiers(self, ids=None) -> np.ndarray:
        ids = self._ids(np.arange(self.n_pages) if ids is None else ids)
        out = np.zeros(ids.size, dtype=np.uint8)
        check(lib().speckv_ext_policy_get_tiers(self._h, ids.ctypes.data, ids.size, out.ctypes.data),
              "speckv_ext_policy_get_tiers")
        return out

    def lru_order(self) -> np.ndarray:
        out = np.zeros(self.n_pages, dtype=np.uint64)
        n = C.c_size_t()
        check(lib().speckv_ext_policy_lru_order(self._h, out.ctypes.data, out.size, C.byref(n)),
              "speckv_ext_policy_lru_order")
        return out[:n.value].copy()

    def stats(self) -> dict:
        s = _lib.PolicyStats()
        check(lib().speckv_ext_policy_get_stats(self._h, C.byref(s)), "speckv_ext_policy_get_stats")
        return {k: getattr(s, k) for k, _ in s._fields_}


class CxlAddressMap:
    """The address map of the reference's CXLMemoryManager (allocate / deallocate /
    translate_virtual_to_physical / is_in_cache, src/cxl_memory/cxl_memory_manager.cpp:28-128):
    host bookkeeping in libcxlspeckv.so, batched translation on the device through the page-lookup kernel."""
    VA_BASE = 0x100000000

    def __init__(self, l1_bytes: int = 12 << 30, l2_bytes: int = 3 << 30, l3_bytes: int = 128 << 30):
        self._h = C.c_void_p()
        check(lib().speckv_ext_memmgr_create(l1_bytes, l2_bytes, l3_bytes, C.byref(self._h)), "speckv_ext_memmgr_create")

    def close(self):
        if self._h:
            lib().speckv_ext_memmgr_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def allocate(self, size_bytes: int, layer_id: int = 0, tier: int = L3):
        va, used = C.c_uint64(), C.c_int()
        check(lib().speckv_ext_memmgr_allocate(self._h, size_bytes, layer_id, tier, C.byref(va), C.byref(used)),
              "speckv_ext_memmgr_allocate")
        return va.value, used.value

    def deallocate(self, va: int) -> None:
        check(lib().speckv_ext_memmgr_deallocate(self._h, va), "speckv_ext_memmgr_deallocate")

    def set_tier(self, va: int, n_pages: int, tier: int) -> None:
        check(lib().speckv_ext_memmgr_set_tier(self._h, va, n_pages, tier), "speckv_ext_memmgr_set_tier")

    def translate_host(self, va: int):
        pa, tier = C.c_uint64(), C.c_int()
        check(lib().speckv_ext_memmgr_translate_host(self._h, va, C.byref(pa), C.byref(tier)), "speckv_ext_memmgr_translate_host")
        return pa.value, tier.value

    def export(self, device="cuda:0") -> torch.Tensor:
        """The page table as a CUDA uint8 [n_pages, 24] tensor of speckv_page_t records."""
        n = C.c_size_t()
        check(lib().speckv_ext_memmgr_export(self._h, None, 0, C.byref(n), None, None), "speckv_ext_memmgr_export")
        table = torch.zeros((max(n.value, 1), 24), dtype=torch.uint8, device=device)
        with torch.cuda.device(table.device):
            check(lib().speckv_ext_memmgr_export(self._h, table.data_ptr(), n.value, C.byref(n), None, _stream()),
                  "speckv_ext_memmgr_export")
        return table[: n.value]

    def translate(self, table: torch.Tensor, va: torch.Tensor):
        """Batched translate_virtual_to_physical + tier flags (bit0 L1, bit1 L2) on the device:
        (pa int64, flags int32); unknown addresses give 0 / 0."""
        va = va.contiguous()
        pa = torch.empty_like(va)
        flags = torch.empty(va.numel(), dtype=torch.int32, device=va.device)
        with torch.cuda.device(va.device):
            check(lib().speckv_ext_page_lookup(table.data_ptr(), table.shape[0], self.VA_BASE, va.data_ptr(), pa.data_ptr(),
                                               flags.data_ptr(), va.numel(), _stream()), "speckv_ext_page_lookup")
        return pa, flags
