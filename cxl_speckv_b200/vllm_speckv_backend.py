"""CxlSpeckvKVAllocator -- the vLLM-facing allocator of the reference
(host/python/vllm_speckv_backend.py:9-100), same constructor and method
signatures, over the B200 libcxlspeckv.so.

The KV region of one handle is laid out [req][layer][kind (K=0,V=1)][pos][head] x
entry_bytes (`_calc_offset`, reference :87-100); `get_kv_ptr` turns that offset
into an address through speckv_access and `prefetch_step` forwards the recent
token history to speckv_prefetch.
"""
import ctypes
from typing import Any, Dict, List, Optional

import numpy as np

try:  # the reference imports it relatively (:5); its tests import it top-level
    from .speckv_ctypes import SpeckvLib
except ImportError:  # pragma: no cover
    from speckv_ctypes import SpeckvLib


class CxlSpeckvKVAllocator:
    def __init__(self, lib_path: str, dev_path: str = "/dev/speckv0", page_size: int = 4096):
        self._speckv = SpeckvLib(lib_path, dev_path)
        self._page_size = page_size
        self._handle: Optional[int] = None
        self._req_id_counter = 1
        self._req_state: Dict[int, Dict[str, Any]] = {}
        self._num_layers = 0
        self._num_heads = 0
        self._num_tokens = 0
        self._head_dim = 0
        self._bytes_per_element = 0
        self._pool = None      # CUDA tensor backing the region (bind_pool)
        self._tier = None      # keeps the HostTier alive as long as the binding refers to it
        self._policy = None    # TierPolicy (attach_policy)
        self._kv_set = None    # KVCacheSet of the registered per-layer caches (register_kv_caches)
        lib = self._speckv.lib
        if hasattr(lib, "speckv_ext_bind_pool"):   # additive entry points of the B200 library, declared once
            lib.speckv_ext_bind_pool.argtypes = [ctypes.c_uint64, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
            lib.speckv_ext_set_kv_layout.argtypes = [ctypes.c_uint64] + [ctypes.c_uint32] * 4
            lib.speckv_ext_set_pool_dtype.argtypes = [ctypes.c_uint64, ctypes.c_int]
            lib.speckv_ext_offload_pages.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p]
            lib.speckv_ext_fetch_pages.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p]
            for f in ("speckv_ext_bind_pool", "speckv_ext_set_kv_layout", "speckv_ext_set_pool_dtype",
                      "speckv_ext_offload_pages", "speckv_ext_fetch_pages"):
                getattr(lib, f).restype = ctypes.c_int

    def allocate(self, num_tokens: int, num_layers: int, num_heads: int, head_dim: int, bytes_per_element: int):
        """Allocate the KV region of one request: tokens x layers x heads x head_dim x bytes x 2 (K+V)."""
        self._num_tokens = num_tokens
        self._num_layers = num_layers
        self._num_heads = num_heads
        self._head_dim = head_dim
        self._bytes_per_element = bytes_per_element
        total_bytes = num_tokens * num_layers * num_heads * head_dim * bytes_per_element * 2
        self._handle = self._speckv.alloc(total_bytes, preferred_node=0)
        return self._handle

    def get_kv_ptr(self, req_id: int, layer: int, head: int, pos: int, kind: int, entry_bytes: int) -> int:
        """Address of one KV entry (ensures its page is resident, fetching it if needed)."""
        offset = self._calc_offset(req_id, layer, head, pos, kind, entry_bytes)
        gpu_ptr = ctypes.c_void_p()
        ret = self._speckv.lib.speckv_access(self._handle, offset, entry_bytes, ctypes.byref(gpu_ptr))
        if ret != 0:
            raise RuntimeError(f"speckv_access failed: {ret}")
        return gpu_ptr.value

    def prefetch_step(self, req_id: int, layer: int, cur_pos: int, recent_tokens: List[int], depth_k: int = 4):
        """Issue the speculative prefetch for the next tokens of (req_id, layer)."""
        hist_len = len(recent_tokens)
        arr = (ctypes.c_int32 * hist_len)(*recent_tokens)
        ret = self._speckv.lib.speckv_prefetch(req_id, layer, cur_pos, depth_k, arr, hist_len)
        if ret != 0:
            raise RuntimeError(f"speckv_prefetch failed: {ret}")

    # ---- additive: serve real device pointers (not in the reference, SURVEY.md section 8f row 1) ----
    def bind_pool(self, pool, tier=None):
        """Back the allocated region with a CUDA tensor (`pool`, >= the region's bytes).  After this
        get_kv_ptr() returns addresses inside `pool`; with a HostTier, pages can be demoted with
        offload_pages() and come back on access / prefetch_step()."""
        lib = self._speckv.lib
        if self._handle is None:
            raise RuntimeError("bind_pool: call allocate() first")
        ret = lib.speckv_ext_bind_pool(self._handle, pool.data_ptr(), pool.numel() * pool.element_size(),
                                       tier._h if tier is not None else None)
        if ret != 0:
            raise RuntimeError(f"speckv_ext_bind_pool failed: {ret}")
        ret = lib.speckv_ext_set_kv_layout(self._handle, self._num_layers, self._num_tokens, self._num_heads,
                                           self._head_dim * self._bytes_per_element)
        if ret != 0:
            raise RuntimeError(f"speckv_ext_set_kv_layout failed: {ret}")
        # the codec quantises the pool's own element type (fp16 / bf16 / fp32 pages)
        import torch
        code = {torch.float16: 0, torch.bfloat16: 1, torch.float32: 2}.get(pool.dtype)
        if code is None:
            raise TypeError(f"bind_pool: unsupported pool dtype {pool.dtype}")
        ret = lib.speckv_ext_set_pool_dtype(self._handle, code)
        if ret != 0:
            raise RuntimeError(f"speckv_ext_set_pool_dtype failed: {ret}")
        self._pool = pool
        self._tier = tier

    def offload_pages(self, first_page: int, n_pages: int):
        lib = self._speckv.lib
        if self._pool is None:
            raise RuntimeError("offload_pages: no pool bound (bind_pool)")
        ret = lib.speckv_ext_offload_pages(self._handle, first_page, n_pages, None)
        if ret != 0:
            raise RuntimeError(f"speckv_ext_offload_pages failed: {ret}")

    def fetch_pages(self, first_page: int, n_pages: int):
        lib = self._speckv.lib
        if self._pool is None:
            raise RuntimeError("fetch_pages: no pool bound (bind_pool)")
        ret = lib.speckv_ext_fetch_pages(self._handle, first_page, n_pages, None)
        if ret != 0:
            raise RuntimeError(f"speckv_ext_fetch_pages failed: {ret}")

    # ---- additive: vLLM block tables (SURVEY.md section 8f row 1) ----
    @staticmethod
    def offload_kv_blocks(kv_cache, block_table, tier, block_ids=None, num_tokens=None):
        """Compress the cache blocks `block_table` (CUDA int32 tensor of block numbers) of a paged KV cache
        tensor ([num_blocks, block_size, kv_heads, head_dim], contiguous) out to the host tier, reading them
        in place.  They are stored under `block_ids` (default: the block numbers themselves).

        `num_tokens` (optional, one entry per block of `block_table`, tensor or sequence): the filled tokens of each
        block.  Only they are stored -- the stale K/V a reused block holds behind them takes no part -- and a restore
        writes them back and leaves the rest of the block as it is.  None stores whole blocks."""
        ids = block_table.cpu().numpy().astype("uint64") if block_ids is None else block_ids
        if num_tokens is None:
            tier.offload_blocks(kv_cache, block_table, ids)
            return
        tier.offload_ragged(kv_cache, kv_cache[0].numel(), _token_lengths(num_tokens, kv_cache), ids,
                            block_table=block_table)

    @staticmethod
    def restore_kv_blocks(kv_cache, block_table, tier, block_ids=None):
        """Bring stored blocks back into the cache blocks `block_table` (decompressed in place)."""
        ids = block_table.cpu().numpy().astype("uint64") if block_ids is None else block_ids
        tier.restore_blocks(ids, kv_cache, block_table)

    # ---- additive: whole requests across all layers (one KV cache set) ----
    def register_kv_caches(self, kv_caches):
        """Register the model's per-layer KV caches once (a list, or vLLM's layer name -> tensor dict, in layer
        order).  Each tensor is [2, num_blocks, ...] (FlashAttention backend: K = kv[0], V = kv[1]) or
        [num_blocks, 2, ...] (FlashInfer backend: K = kv[:, 0], V = kv[:, 1]); a tensor whose first two dimensions are
        both 2 is taken as the first.  Cache 2 * layer is the layer's K, cache 2 * layer + 1 its V.  Returns the
        KVCacheSet that offload_request / restore_request move blocks through."""
        from .codec import KVCacheSet
        tensors = list(kv_caches.values()) if isinstance(kv_caches, dict) else list(kv_caches)
        views = []
        for kv in tensors:
            if kv.dim() >= 3 and kv.shape[0] == 2:
                views += [kv[0], kv[1]]
            elif kv.dim() >= 3 and kv.shape[1] == 2:
                views += [kv[:, 0], kv[:, 1]]
            else:
                raise ValueError(f"register_kv_caches: {tuple(kv.shape)} is neither [2, num_blocks, ...] nor "
                                 "[num_blocks, 2, ...]")
        if self._kv_set is not None:
            self._kv_set.close()
        self._kv_set = KVCacheSet(views)
        return self._kv_set

    def request_block_ids(self, block_table):
        """The default ids of a request's blocks: (cache c, block b) -> (c << 40) | b, a uint64 [n_caches, n_blocks]
        array.  Block numbers are below 2^32 (the tables are int32), so the cache index in bits 40 and up never meets
        them; cache 0's ids are the block numbers themselves, the ids offload_kv_blocks gives by default."""
        b = np.asarray(block_table.cpu() if hasattr(block_table, "cpu") else block_table).reshape(-1).astype(np.uint64)
        c = np.arange(len(self._registered()), dtype=np.uint64)
        return (c[:, None] << np.uint64(40)) | b[None, :]

    def offload_request(self, block_table, tier, block_ids=None, num_tokens=None):
        """Compress one request's blocks `block_table` (CUDA int32, the request's block numbers) of every registered
        cache out to the host tier in one call, cache-major.  block_ids: uint64 [n_caches, n_blocks] (default
        request_block_ids).  num_tokens (optional, one entry per block): the filled tokens of each block, as in
        offload_kv_blocks, applied to every cache."""
        cset, table, ids = self._request(block_table, block_ids)
        lengths = None
        if num_tokens is not None:
            lengths = _token_lengths(num_tokens, cset.caches[0])
            if lengths.numel() != table.numel():
                raise ValueError("num_tokens must hold one entry per block")
            lengths = lengths.repeat(len(cset))
        tier.offload_set(cset, *cset.groups(table), ids, lengths=lengths)

    def restore_request(self, block_table, tier, block_ids=None):
        """Bring one request's blocks of every registered cache back from the host tier in one call."""
        cset, table, ids = self._request(block_table, block_ids)
        tier.restore_set(ids, cset, *cset.groups(table))

    def _request(self, block_table, block_ids):
        """-> (the registered set, the request's block numbers as int32 on its device, their ids cache-major)"""
        import torch
        cset = self._registered()
        table = torch.as_tensor(block_table).to(device=cset.device, dtype=torch.int32).reshape(-1)
        return cset, table, self._request_ids(cset, table, block_ids)

    def _registered(self):
        if self._kv_set is None:
            raise RuntimeError("no KV caches registered (register_kv_caches)")
        return self._kv_set

    def _request_ids(self, cset, table, block_ids):
        if block_ids is None:
            return self.request_block_ids(table).reshape(-1)
        ids = np.ascontiguousarray(block_ids, dtype=np.uint64)
        if ids.shape != (len(cset), table.numel()):
            raise ValueError(f"block_ids must be [{len(cset)}, {table.numel()}] (caches x blocks)")
        return ids.reshape(-1)

    # ---- additive: residency policy driving the data path (SURVEY.md section 8f row 2) ----
    def attach_policy(self, policy):
        """`policy`: a cxl_speckv_b200.tier.TierPolicy over this region's pages (page i of the policy =
        page i of the region).  residency_step() then keeps the pool in line with its decisions."""
        self._policy = policy

    def residency_step(self, touched=None, promote=None):
        """One policy round: record the pages the step read (`touched`: CUDA tensor or array of page
        indices), promote the pages in `promote` (e.g. the prefetcher's predictions) to L1, and move
        data accordingly -- promoted pages are restored into the pool, the pages the policy evicted
        to make room are compressed out to the host tier.  Returns (ok, evicted)."""
        pol = self._policy
        if pol is None:
            raise RuntimeError("residency_step: no policy attached (attach_policy)")
        if touched is not None:
            pol.touch(touched)
        if promote is None or len(promote) == 0:
            return [], []
        ok, evicted = pol.promote(promote)
        for a, b in _runs(sorted(int(p) for p in evicted)):
            self.offload_pages(a, b - a)
        for a, b in _runs(sorted({int(p) for p, o in zip(promote, ok) if o})):
            self.fetch_pages(a, b - a)
        return ok, evicted

    def _calc_offset(self, req_id: int, layer: int, head: int, pos: int, kind: int, entry_bytes: int) -> int:
        # [req][layer][kind][pos][head] * entry_bytes  (reference :95-100)
        return ((((req_id * self._num_layers + layer) * 2 + kind) * self._num_tokens + pos)
                * self._num_heads + head) * entry_bytes


def _token_lengths(num_tokens, cache):
    """Filled tokens per block of a paged KV cache [num_blocks, block_size, ...] -> int32 element lengths on its device"""
    import torch
    lengths = torch.as_tensor(num_tokens, device=cache.device).to(torch.int64).reshape(-1) * cache[0, 0].numel()
    return lengths.clamp_(0, cache[0].numel()).to(torch.int32)


def _runs(pages):
    """[3, 4, 5, 9] -> [(3, 6), (9, 10)]: contiguous page ranges for the range-based offload / fetch calls."""
    out = []
    for p in pages:
        if out and out[-1][1] == p:
            out[-1][1] = p + 1
        else:
            out.append([p, p + 1])
    return [(a, b) for a, b in out]


def decode_step_example(model, kv_allocator: CxlSpeckvKVAllocator, state, depth_k: int = 4):
    """The decode-loop sketch of the reference (:104-129), made importable: one forward
    step, then a prefetch per layer on the last 16 tokens."""
    logits = model(state)
    new_token = int(logits.argmax(-1))
    state.tokens.append(new_token)
    last_tokens = state.tokens[-16:]
    for layer in range(model.num_layers):
        kv_allocator.prefetch_step(req_id=state.req_id, layer=layer, cur_pos=state.cur_pos,
                                   recent_tokens=last_tokens, depth_k=depth_k)
    state.cur_pos += 1
    return logits, new_token
