"""Torch-tensor front end of the batch codec entry points (speckv_ext_compress /
speckv_ext_decompress / speckv_ext_translate).  PyTorch is used for device memory
and streams only; all arithmetic happens in libcxlspeckv.so's CUDA kernels."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import COMP_INT8_DELTA_RLE, DTYPE_BF16, DTYPE_F16, DTYPE_F32, check, lib

_DTYPES = {torch.float16: DTYPE_F16, torch.bfloat16: DTYPE_BF16, torch.float32: DTYPE_F32}


def slot_bytes(group_elems: int, scheme: int = COMP_INT8_DELTA_RLE) -> int:
    return lib().speckv_ext_slot_bytes(group_elems, scheme)


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@dataclass
class CompressedKV:
    """Device-resident container: group g owns payload[g, :comp_bytes[g]], scales[g]."""
    payload: torch.Tensor      # uint8 [n_groups, slot_bytes]
    scales: torch.Tensor       # float32 [n_groups]
    comp_bytes: torch.Tensor   # int32 [n_groups] (bit pattern of uint32)
    group_elems: int
    dtype: torch.dtype
    scheme: int

    @property
    def n_groups(self) -> int:
        return self.scales.numel()


def _compressed(n_groups: int, group_elems: int, dtype: torch.dtype, scheme: int, device) -> CompressedKV:
    """An empty container for n_groups groups (one slot of the scheme's worst case each)."""
    return CompressedKV(torch.empty((n_groups, slot_bytes(group_elems, scheme)), dtype=torch.uint8, device=device),
                        torch.empty(n_groups, dtype=torch.float32, device=device),
                        torch.empty(n_groups, dtype=torch.int32, device=device), group_elems, dtype, scheme)


def _i32(t: torch.Tensor, device) -> torch.Tensor:
    """An index tensor as the C entry points take it: contiguous int32 on `device`."""
    return t.to(device=device, dtype=torch.int32).contiguous()


def _lengths(lengths: torch.Tensor, device, n=None, convert=False, check_negative=False) -> torch.Tensor:
    """The lengths of a ragged call as contiguous int32 on `device`, n of them when n is given (ValueError otherwise).
    `convert` converts any integer tensor; without it they must be an int32 tensor on `device` already (TypeError).
    `check_negative` reads them on the host and refuses a negative one: as unsigned, it would store the whole block."""
    if convert:
        lengths = lengths.to(device=device, dtype=torch.int32)
    elif not lengths.is_cuda or lengths.dtype != torch.int32 or lengths.device != device:
        raise TypeError(f"lengths must be an int32 tensor on {device}")
    lengths = lengths.contiguous()
    if n is not None and lengths.numel() != n:
        raise ValueError(f"lengths must hold one entry per group ({n})")
    if check_negative and bool((lengths < 0).any()):
        raise ValueError("negative length")
    return lengths


def compress(x: torch.Tensor, group_elems: int, scheme: int = COMP_INT8_DELTA_RLE,
             out: Optional[CompressedKV] = None) -> CompressedKV:
    """Compress x (flat view, contiguous) as consecutive groups of group_elems elements."""
    if not x.is_cuda:
        raise ValueError("compress() takes a CUDA tensor (use compress_host for host buffers)")
    if x.dtype not in _DTYPES:
        raise TypeError(f"unsupported dtype {x.dtype}")
    x = x.contiguous()
    n = x.numel()
    if group_elems <= 0 or n % group_elems:
        raise ValueError("numel must be a multiple of group_elems")
    n_groups = n // group_elems
    if out is None:
        out = _compressed(n_groups, group_elems, x.dtype, scheme, x.device)
    with torch.cuda.device(x.device):
        st = lib().speckv_ext_compress(x.data_ptr(), _DTYPES[x.dtype], group_elems, n_groups,
                                       out.payload.data_ptr(), out.payload.shape[1], out.scales.data_ptr(),
                                       out.comp_bytes.data_ptr(), scheme, _stream())
    check(st, "speckv_ext_compress")
    return out


def decompress(c: CompressedKV, out: Optional[torch.Tensor] = None, out_elems: Optional[torch.Tensor] = None,
               dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    dtype = dtype or c.dtype
    if out is None:
        out = torch.empty((c.n_groups, c.group_elems), dtype=dtype, device=c.payload.device)
    with torch.cuda.device(c.payload.device):
        st = lib().speckv_ext_decompress(c.payload.data_ptr(), c.payload.shape[1], c.scales.data_ptr(),
                                         c.comp_bytes.data_ptr(), c.group_elems, c.n_groups, _DTYPES[dtype],
                                         out.data_ptr(), out_elems.data_ptr() if out_elems is not None else None,
                                         c.scheme, _stream())
    check(st, "speckv_ext_decompress")
    return out


def decompress_indexed(c: CompressedKV, block_index: torch.Tensor, out: Optional[torch.Tensor] = None,
                       dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """Decompress only the stored blocks listed in block_index (int32 CUDA tensor)."""
    dtype = dtype or c.dtype
    block_index = block_index.to(torch.int32).contiguous()
    n = block_index.numel()
    if out is None:
        out = torch.empty((n, c.group_elems), dtype=dtype, device=c.payload.device)
    with torch.cuda.device(c.payload.device):
        st = lib().speckv_ext_decompress_indexed(c.payload.data_ptr(), c.payload.shape[1], c.scales.data_ptr(),
                                                 c.comp_bytes.data_ptr(), block_index.data_ptr(), n, c.group_elems,
                                                 _DTYPES[dtype], out.data_ptr(), None, c.scheme, _stream())
    check(st, "speckv_ext_decompress_indexed")
    return out


def decompress_routed(c: CompressedKV, block_index: torch.Tensor, count: torch.Tensor, out: torch.Tensor,
                      dtype: Optional[torch.dtype] = None) -> torch.Tensor:
    """decompress_indexed with the request count on the device (count: int32 [1], from prefetch.route): out has
    room for block_index.numel() blocks, the first count[0] of them are written.  No host synchronisation."""
    dtype = dtype or c.dtype
    cap = min(block_index.numel(), out.shape[0])
    with torch.cuda.device(c.payload.device):
        st = lib().speckv_ext_decompress_routed(c.payload.data_ptr(), c.payload.shape[1], c.scales.data_ptr(),
                                                c.comp_bytes.data_ptr(), block_index.data_ptr(), count.data_ptr(), cap,
                                                c.group_elems, _DTYPES[dtype], out.data_ptr(), None, c.scheme, _stream())
    check(st, "speckv_ext_decompress_routed")
    return out


def engine_stats(wait: bool = True) -> dict:
    """FPGACacheEngine::get_statistics (EngineStatistics, cache_engine.h:65-72)."""
    s = _lib.EngineStats()
    lib().speckv_ext_engine_stats(C.byref(s), int(wait))
    return {k: getattr(s, k) for k, _ in s._fields_}


def compress_gather(cache: torch.Tensor, block_table: torch.Tensor, scheme: int = COMP_INT8_DELTA_RLE,
                    out: Optional[CompressedKV] = None) -> CompressedKV:
    """Compress the blocks of a paged KV cache named by block_table, reading them where they lie.

    cache: [num_blocks, ...] contiguous CUDA tensor (one block = one codec group, e.g. vLLM's
    [num_blocks, block_size, kv_heads, head_dim]); block_table: int32 CUDA tensor of block ids.
    Stored group i encodes cache block block_table[i]."""
    if not cache.is_cuda or cache.dtype not in _DTYPES or not cache.is_contiguous():
        raise ValueError("compress_gather() takes a contiguous CUDA fp16/bf16/fp32 cache tensor")
    group_elems = cache[0].numel()
    block_table = _i32(block_table, cache.device)
    n_groups = block_table.numel()
    if out is None:
        out = _compressed(n_groups, group_elems, cache.dtype, scheme, cache.device)
    with torch.cuda.device(cache.device):
        st = lib().speckv_ext_compress_gather(cache.data_ptr(), block_table.data_ptr(), _DTYPES[cache.dtype],
                                              group_elems, n_groups, out.payload.data_ptr(), out.payload.shape[1],
                                              out.scales.data_ptr(), out.comp_bytes.data_ptr(), scheme, _stream())
    check(st, "speckv_ext_compress_gather")
    return out


def compress_ragged(x: torch.Tensor, group_elems: int, lengths: torch.Tensor,
                    block_table: Optional[torch.Tensor] = None, scheme: int = COMP_INT8_DELTA_RLE,
                    out: Optional[CompressedKV] = None) -> CompressedKV:
    """Compress the filled prefix of each block: group i is the first min(lengths[i], group_elems) elements of block
    block_table[i] of x (block i when block_table is None), where x is a contiguous CUDA tensor of whole blocks of
    group_elems elements.  lengths: CUDA int32 tensor of element counts, one per group; it stays on the device (no
    synchronisation, graph-capturable).  Elements behind a group's length take no part in its scale or payload.
    Schemes 1-4.  The decoders give lengths[i] elements per group and leave the rest of the destination as it is.
    The lengths are not read on the host: the kernels take them as unsigned and clamp them to group_elems, so a
    negative entry stores the whole block.  Callers that cannot rule that out check (lengths >= 0) themselves."""
    if not x.is_cuda or x.dtype not in _DTYPES or not x.is_contiguous():
        raise ValueError("compress_ragged() takes a contiguous CUDA fp16/bf16/fp32 tensor")
    if group_elems <= 0 or x.numel() % group_elems:
        raise ValueError("numel must be a multiple of group_elems")
    n_groups = block_table.numel() if block_table is not None else x.numel() // group_elems
    lengths = _lengths(lengths, x.device, n_groups)
    if block_table is not None:
        block_table = _i32(block_table, x.device)
    if out is None:
        out = _compressed(n_groups, group_elems, x.dtype, scheme, x.device)
    with torch.cuda.device(x.device):
        st = lib().speckv_ext_compress_ragged(x.data_ptr(), block_table.data_ptr() if block_table is not None else None,
                                              lengths.data_ptr(), _DTYPES[x.dtype], group_elems, n_groups,
                                              out.payload.data_ptr(), out.payload.shape[1], out.scales.data_ptr(),
                                              out.comp_bytes.data_ptr(), scheme, _stream())
    check(st, "speckv_ext_compress_ragged")
    return out


def decompress_scatter(c: CompressedKV, cache: torch.Tensor, block_table: torch.Tensor,
                       src_index: Optional[torch.Tensor] = None,
                       out_elems: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Decode stored blocks straight into the paged KV cache: request i decodes stored block
    src_index[i] (block i when src_index is None) into cache block block_table[i]."""
    if not cache.is_cuda or cache.dtype not in _DTYPES or not cache.is_contiguous():
        raise ValueError("decompress_scatter() takes a contiguous CUDA fp16/bf16/fp32 cache tensor")
    if cache[0].numel() != c.group_elems:
        raise ValueError("cache block size differs from the stored group size")
    block_table = _i32(block_table, cache.device)
    n = block_table.numel()
    if src_index is not None:
        src_index = _i32(src_index, cache.device)
        if src_index.numel() != n:
            raise ValueError("src_index and block_table differ in length")
    elif n != c.n_groups:
        raise ValueError("block_table must name one cache block per stored block")
    with torch.cuda.device(cache.device):
        st = lib().speckv_ext_decompress_scatter(c.payload.data_ptr(), c.payload.shape[1], c.scales.data_ptr(),
                                                 c.comp_bytes.data_ptr(),
                                                 src_index.data_ptr() if src_index is not None else None,
                                                 block_table.data_ptr(), n, c.group_elems, _DTYPES[cache.dtype],
                                                 cache.data_ptr(),
                                                 out_elems.data_ptr() if out_elems is not None else None,
                                                 c.scheme, _stream())
    check(st, "speckv_ext_decompress_scatter")
    return cache


class KVCacheSet:
    """A model's paged KV caches registered as one set (speckv_ext_cache_set_create): one tensor per layer and K|V,
    all of the same shape, dtype, strides and device, each [num_blocks, ...] with block b at index b.  A block must be
    contiguous; consecutive blocks may lie further apart (a K or V view of vLLM's [num_blocks, 2, ...] layout).

    Calls through the set name each group by (cache index, block number): see groups().  The set keeps the tensors
    alive; close() (or garbage collection) releases the native set, which must not happen while calls that use it
    are in flight or captured in a graph that is still replayed.  On CPU tensors only the geometry and groups() are
    available (no native set is created)."""

    def __init__(self, caches):
        caches = list(caches)
        if not caches:
            raise ValueError("KVCacheSet needs at least one cache")
        c0 = caches[0]
        for c in caches:
            if not isinstance(c, torch.Tensor):
                raise TypeError("KVCacheSet takes tensors")
            if c.dtype not in _DTYPES:
                raise TypeError(f"unsupported dtype {c.dtype}")
            if c.dim() < 2 or c.shape[0] == 0 or c[0].numel() == 0:
                raise ValueError("each cache must be [num_blocks, ...] with non-empty blocks")
            if c.shape != c0.shape or c.dtype != c0.dtype or c.stride() != c0.stride() or c.device != c0.device:
                raise ValueError("the caches of a set must agree in shape, dtype, strides and device")
        if not c0[0].is_contiguous():
            raise ValueError("a cache block must be contiguous")
        self.caches = caches
        self.num_blocks = c0.shape[0]
        self.block_elems = c0[0].numel()
        self.block_stride = c0.stride(0)
        if self.block_stride < self.block_elems:
            raise ValueError("the blocks of a cache overlap (stride(0) < block size)")
        self.dtype = c0.dtype
        self.device = c0.device
        self._h = C.c_void_p()
        if c0.is_cuda:
            bases = (C.c_void_p * len(caches))(*[c.data_ptr() for c in caches])
            with torch.cuda.device(self.device):
                check(lib().speckv_ext_cache_set_create(bases, len(caches), self.block_elems, self.block_stride,
                                                        _DTYPES[self.dtype], C.byref(self._h)),
                      "speckv_ext_cache_set_create")

    def __len__(self) -> int:
        return len(self.caches)

    def handle(self) -> C.c_void_p:
        if not self._h:
            raise ValueError("this KVCacheSet has no native set (CPU tensors, or closed)")
        return self._h

    def groups(self, block_table: torch.Tensor):
        """The cache-major cross product of all caches with block_table: (cache_index, block_index), int32 tensors of
        len(self) * block_table.numel() entries on block_table's device, all blocks of cache 0 first.  Torch ops only
        (capturable)."""
        b = block_table.reshape(-1).to(torch.int32)
        n, nc = b.numel(), len(self.caches)
        cache_index = torch.arange(nc, dtype=torch.int32, device=b.device).view(nc, 1).expand(nc, n).reshape(-1)
        return cache_index, b.view(1, n).expand(nc, n).reshape(-1)

    def close(self):
        if self._h:
            lib().speckv_ext_cache_set_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


def _set_groups(cset: KVCacheSet, cache_index: torch.Tensor, block_table: torch.Tensor):
    """Checked (cache_index, block_table) of a set call: contiguous int32 on the set's device, equal lengths."""
    if not isinstance(cset, KVCacheSet):
        raise TypeError("expected a KVCacheSet")
    cache_index, block_table = _i32(cache_index, cset.device), _i32(block_table, cset.device)
    if cache_index.numel() != block_table.numel():
        raise ValueError("cache_index and block_table differ in length")
    return cache_index, block_table


def compress_gather_set(cset: KVCacheSet, cache_index: torch.Tensor, block_table: torch.Tensor,
                        lengths: Optional[torch.Tensor] = None, scheme: int = COMP_INT8_DELTA_RLE,
                        out: Optional[CompressedKV] = None) -> CompressedKV:
    """compress_gather across a cache set: stored group i encodes block block_table[i] of cache cache_index[i]
    (e.g. from cset.groups(table)).  lengths (optional, CUDA int32, one per group) stores only the first lengths[i]
    elements of each block, as compress_ragged does.  Schemes 1-4."""
    cache_index, block_table = _set_groups(cset, cache_index, block_table)
    n_groups = block_table.numel()
    if lengths is not None:
        lengths = _lengths(lengths, cset.device, n_groups)
    if out is None:
        out = _compressed(n_groups, cset.block_elems, cset.dtype, scheme, cset.device)
    with torch.cuda.device(cset.device):
        st = lib().speckv_ext_compress_gather_set(cset.handle(), cache_index.data_ptr(), block_table.data_ptr(),
                                                  lengths.data_ptr() if lengths is not None else None, n_groups,
                                                  out.payload.data_ptr(), out.payload.shape[1], out.scales.data_ptr(),
                                                  out.comp_bytes.data_ptr(), scheme, _stream())
    check(st, "speckv_ext_compress_gather_set")
    return out


def decompress_scatter_set(c: CompressedKV, cset: KVCacheSet, cache_index: torch.Tensor, block_table: torch.Tensor,
                           src_index: Optional[torch.Tensor] = None,
                           out_elems: Optional[torch.Tensor] = None) -> KVCacheSet:
    """decompress_scatter across a cache set: request i decodes stored block src_index[i] (block i when src_index is
    None) into block block_table[i] of cache cache_index[i].  (cache, block) pairs must be distinct."""
    if cset.block_elems != c.group_elems:
        raise ValueError("cache block size differs from the stored group size")
    cache_index, block_table = _set_groups(cset, cache_index, block_table)
    n = block_table.numel()
    if src_index is not None:
        src_index = _i32(src_index, cset.device)
        if src_index.numel() != n:
            raise ValueError("src_index and block_table differ in length")
    elif n != c.n_groups:
        raise ValueError("block_table must name one cache block per stored block")
    with torch.cuda.device(cset.device):
        st = lib().speckv_ext_decompress_scatter_set(c.payload.data_ptr(), c.payload.shape[1], c.scales.data_ptr(),
                                                     c.comp_bytes.data_ptr(),
                                                     src_index.data_ptr() if src_index is not None else None,
                                                     cset.handle(), cache_index.data_ptr(), block_table.data_ptr(), n,
                                                     out_elems.data_ptr() if out_elems is not None else None,
                                                     c.scheme, _stream())
    check(st, "speckv_ext_decompress_scatter_set")
    return cset


def translate(va: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Batched FPGACacheEngine::translate_address over an int64 tensor of (uint64) addresses."""
    if va.dtype != torch.int64 or not va.is_cuda:
        raise TypeError("translate() takes a CUDA int64 tensor holding uint64 bit patterns")
    va = va.contiguous()
    if out is None:
        out = torch.empty_like(va)
    with torch.cuda.device(va.device):
        st = lib().speckv_ext_translate(va.data_ptr(), out.data_ptr(), va.numel(), _stream())
    check(st, "speckv_ext_translate")
    return out


def stats() -> dict:
    s = _lib.Stats()
    lib().speckv_ext_get_stats(C.byref(s))
    return {k: getattr(s, k) for k, _ in s._fields_}
