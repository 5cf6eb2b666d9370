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
    sb = slot_bytes(group_elems, scheme)
    if out is None:
        out = CompressedKV(torch.empty((n_groups, sb), dtype=torch.uint8, device=x.device),
                           torch.empty(n_groups, dtype=torch.float32, device=x.device),
                           torch.empty(n_groups, dtype=torch.int32, device=x.device),
                           group_elems, x.dtype, scheme)
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
    block_table = block_table.to(device=cache.device, dtype=torch.int32).contiguous()
    n_groups = block_table.numel()
    sb = slot_bytes(group_elems, scheme)
    if out is None:
        out = CompressedKV(torch.empty((n_groups, sb), dtype=torch.uint8, device=cache.device),
                           torch.empty(n_groups, dtype=torch.float32, device=cache.device),
                           torch.empty(n_groups, dtype=torch.int32, device=cache.device),
                           group_elems, cache.dtype, scheme)
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
    if not lengths.is_cuda or lengths.dtype != torch.int32 or lengths.device != x.device:
        raise TypeError("lengths must be an int32 tensor on the device of x")
    lengths = lengths.contiguous()
    if block_table is not None:
        block_table = block_table.to(device=x.device, dtype=torch.int32).contiguous()
        if block_table.numel() != lengths.numel():
            raise ValueError("block_table and lengths differ in length")
    elif lengths.numel() != x.numel() // group_elems:
        raise ValueError("lengths must hold one entry per block of x")
    n_groups = lengths.numel()
    sb = slot_bytes(group_elems, scheme)
    if out is None:
        out = CompressedKV(torch.empty((n_groups, sb), dtype=torch.uint8, device=x.device),
                           torch.empty(n_groups, dtype=torch.float32, device=x.device),
                           torch.empty(n_groups, dtype=torch.int32, device=x.device),
                           group_elems, x.dtype, scheme)
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
    block_table = block_table.to(device=cache.device, dtype=torch.int32).contiguous()
    n = block_table.numel()
    if src_index is not None:
        src_index = src_index.to(device=cache.device, dtype=torch.int32).contiguous()
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
