"""ctypes loaders for the CPU oracle.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module, and only as the checker or the timed CPU baseline.
The product package (cxl_speckv_b200) never imports it.

Two libraries:
  * Port  -- oracle/libspeckv_oracle.so: our C restatement (speckv_oracle.c).
  * Ref   -- oracle/_ref/libspeckv_ref.so: the reference's unmodified C++ sources
             behind our extern "C" shim (ref_shim.cpp).  Built in the authoring
             container where /root/reference exists; the prebuilt .so travels to
             the GPU box.  `Ref.available()` says whether it is there.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional, Tuple

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "libspeckv_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libspeckv_ref.so")
REF_CAPI_SO = os.path.join(HERE, "_ref", "libspeckv_ref_capi.so")

F16, BF16, F32 = 0, 1, 2

_u8p = C.POINTER(C.c_uint8)
_i8p = C.POINTER(C.c_int8)
_f32p = C.POINTER(C.c_float)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)
_f64p = C.POINTER(C.c_double)


def build(ref: bool = True) -> None:
    """Compile the restatement and, when the reference tree is present, oracle/_ref."""
    subprocess.check_call(["make", "-s", "-C", HERE, "port"])
    if ref and os.path.isdir(os.environ.get("REF", "/root/reference")):
        subprocess.check_call(["make", "-s", "-C", HERE, "ref"])


def _ptr(a: np.ndarray, t):
    return a.ctypes.data_as(t)


def np_dtype_code(a: np.ndarray, dtype: Optional[int]) -> int:
    if dtype is not None:
        return dtype
    if a.dtype == np.float16:
        return F16
    if a.dtype == np.float32:
        return F32
    raise ValueError("pass dtype=BF16 explicitly for bf16 bit patterns (uint16)")


class Port:
    """The C restatement (oracle/speckv_oracle.c)."""

    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            srcs = [os.path.join(HERE, f) for f in ("speckv_oracle.c", "speckv_oracle.h")]
            # a library older than its sources lacks what was added since: rebuild it
            if not os.path.exists(PORT_SO) or os.path.getmtime(PORT_SO) < max(map(os.path.getmtime, srcs)):
                build(ref=False)
            L = C.CDLL(PORT_SO)
            L.oracle_scale.restype = C.c_float
            L.oracle_scale.argtypes = [_f32p, C.c_size_t]
            L.oracle_quantize.argtypes = [_f32p, C.c_size_t, C.c_float, _i8p]
            L.oracle_delta_encode.argtypes = [_i8p, C.c_size_t, _i8p]
            L.oracle_compress.restype = C.c_size_t
            L.oracle_compress.argtypes = [_f32p, C.c_size_t, _f32p, _u8p]
            L.oracle_decompress.restype = C.c_size_t
            L.oracle_decompress.argtypes = [_u8p, C.c_size_t, C.c_float, _f32p, C.c_size_t]
            L.oracle_compress_batch.restype = C.c_int
            L.oracle_compress_batch.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, _u8p,
                                                C.c_size_t, _f32p, _u32p, C.c_int]
            L.oracle_decompress_batch.restype = C.c_int
            L.oracle_decompress_batch.argtypes = [_u8p, C.c_size_t, _f32p, _u32p, C.c_size_t,
                                                  C.c_size_t, C.c_int, C.c_void_p, _u32p, C.c_int]
            L.oracle_compress_batch_scheme.restype = C.c_int
            L.oracle_compress_batch_scheme.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, _u8p, C.c_size_t,
                                                       _f32p, _u32p, C.c_int, C.c_int]
            L.oracle_decompress_batch_scheme.restype = C.c_int
            L.oracle_decompress_batch_scheme.argtypes = [_u8p, C.c_size_t, _f32p, _u32p, C.c_size_t, C.c_size_t, C.c_int,
                                                         C.c_void_p, _u32p, C.c_int, C.c_int]
            L.oracle_translate.restype = C.c_uint64
            L.oracle_translate.argtypes = [C.c_uint64]
            L.oracle_atu_new.restype = C.c_void_p
            L.oracle_atu_new.argtypes = [C.c_size_t]
            L.oracle_atu_free.argtypes = [C.c_void_p]
            L.oracle_atu_translate.restype = C.c_uint64
            L.oracle_atu_translate.argtypes = [C.c_void_p, C.c_uint64]
            L.oracle_atu_invalidate.argtypes = [C.c_void_p, C.c_uint64]
            L.oracle_atu_invalidate_all.argtypes = [C.c_void_p]
            L.oracle_atu_stats.argtypes = [C.c_void_p, _u64p, _u64p]
            for f in ("oracle_virt_page_id", "oracle_phys_page_id"):
                getattr(L, f).restype = C.c_uint64
                getattr(L, f).argtypes = [C.c_uint64, C.c_uint64]
            L.oracle_access_addr.restype = C.c_uint64
            L.oracle_access_addr.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64]
            L.oracle_fetch_gpu_addr.restype = C.c_uint64
            L.oracle_fetch_gpu_addr.argtypes = [C.c_uint64]
            L.oracle_lstm_predict_topk.argtypes = [_f32p, _f32p, C.c_size_t, C.c_size_t, C.c_size_t,
                                                   C.c_size_t, C.c_size_t, _u32p, C.c_size_t,
                                                   C.c_size_t, _u32p, _f32p, _f32p]
            L.oracle_kv_address.restype = C.c_uint64
            L.oracle_kv_address.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32]
            L.oracle_lstm_init_weights.argtypes = [C.c_uint, _f32p, C.c_size_t, _f32p, C.c_size_t,
                                                   _f32p, C.c_size_t]
            L.oracle_fnv1a64.restype = C.c_uint64
            L.oracle_fnv1a64.argtypes = [C.c_void_p, C.c_size_t]
            L.oracle_policy_new.restype = C.c_void_p
            L.oracle_policy_new.argtypes = [C.c_uint64] * 4
            L.oracle_policy_free.argtypes = [C.c_void_p]
            for f in ("oracle_policy_touch", "oracle_policy_release"):
                getattr(L, f).restype = None
                getattr(L, f).argtypes = [C.c_void_p, C.c_uint64]
            for f in ("oracle_policy_is_hot", "oracle_policy_demote", "oracle_policy_tier"):
                getattr(L, f).restype = C.c_int
                getattr(L, f).argtypes = [C.c_void_p, C.c_uint64]
            L.oracle_policy_place.restype = C.c_int
            L.oracle_policy_place.argtypes = [C.c_void_p, C.c_uint64, C.c_int]
            L.oracle_policy_promote.restype = C.c_int
            L.oracle_policy_promote.argtypes = [C.c_void_p, C.c_uint64, _u64p]
            L.oracle_policy_lru.restype = C.c_size_t
            L.oracle_policy_lru.argtypes = [C.c_void_p, _u64p, C.c_size_t]
            L.oracle_policy_stats.argtypes = [C.c_void_p, C.c_void_p]
            for f in ("oracle_policy_touch_n", "oracle_policy_release_n"):
                getattr(L, f).restype = None
                getattr(L, f).argtypes = [C.c_void_p, _u64p, C.c_size_t]
            L.oracle_policy_place_n.restype = None
            L.oracle_policy_place_n.argtypes = [C.c_void_p, _u64p, C.c_size_t, C.c_int, C.POINTER(C.c_int32)]
            for f in ("oracle_policy_demote_n", "oracle_policy_is_hot_n"):
                getattr(L, f).restype = None
                getattr(L, f).argtypes = [C.c_void_p, _u64p, C.c_size_t, _u8p]
            L.oracle_policy_promote_n.restype = C.c_size_t
            L.oracle_policy_promote_n.argtypes = [C.c_void_p, _u64p, C.c_size_t, _u8p, _u64p]
            L.oracle_policy_tiers.restype = None
            L.oracle_policy_tiers.argtypes = [C.c_void_p, _u8p]
            cls._lib = L
        return cls._lib

    # -- single group, fp32 in (what the reference engine consumes) --------------------
    @classmethod
    def compress(cls, x: np.ndarray) -> Tuple[np.float32, np.ndarray]:
        x = np.ascontiguousarray(x, dtype=np.float32).ravel()
        out = np.zeros(max(2 * x.size, 2), dtype=np.uint8)
        s = C.c_float()
        n = cls.lib().oracle_compress(_ptr(x, _f32p), x.size, C.byref(s), _ptr(out, _u8p))
        return np.float32(s.value), out[:n].copy()

    @classmethod
    def decompress(cls, scale, payload: np.ndarray, cap: int) -> np.ndarray:
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        out = np.zeros(max(cap, 1), dtype=np.float32)
        n = cls.lib().oracle_decompress(_ptr(payload, _u8p), payload.size, C.c_float(float(scale)),
                                        _ptr(out, _f32p), cap)
        return out[:n].copy()

    @classmethod
    def quantize(cls, x: np.ndarray, scale) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32).ravel()
        q = np.zeros(x.size, dtype=np.int8)
        cls.lib().oracle_quantize(_ptr(x, _f32p), x.size, C.c_float(float(scale)), _ptr(q, _i8p))
        return q

    @classmethod
    def scale(cls, x: np.ndarray) -> np.float32:
        x = np.ascontiguousarray(x, dtype=np.float32).ravel()
        return np.float32(cls.lib().oracle_scale(_ptr(x, _f32p), x.size))

    # -- batched, fp16/bf16/fp32 boundary ------------------------------------------------
    @classmethod
    def compress_batch(cls, x: np.ndarray, group_elems: int, dtype: Optional[int] = None,
                       slot_bytes: Optional[int] = None, threads: int = 1, scheme: int = 2):
        """scheme: 1 INT8 codes, 2 the reference pipeline, 3 / 4 the clamped (non-reference) schemes"""
        code = np_dtype_code(x, dtype)
        x = np.ascontiguousarray(x).ravel()
        n_groups = x.size // group_elems if group_elems else 0
        if slot_bytes is None:
            slot_bytes = (2 * group_elems + 15) // 16 * 16
        payload = np.zeros(max(n_groups * slot_bytes, 1), dtype=np.uint8)
        scales = np.zeros(max(n_groups, 1), dtype=np.float32)
        comp = np.zeros(max(n_groups, 1), dtype=np.uint32)
        cls.lib().oracle_compress_batch_scheme(x.ctypes.data, code, group_elems, n_groups, _ptr(payload, _u8p),
                                               slot_bytes, _ptr(scales, _f32p), _ptr(comp, _u32p), scheme, threads)
        return payload[: n_groups * slot_bytes].reshape(n_groups, slot_bytes), scales[:n_groups], comp[:n_groups]

    @classmethod
    def decompress_batch(cls, payload: np.ndarray, scales: np.ndarray, comp: np.ndarray,
                         group_elems: int, dtype: int, threads: int = 1, scheme: int = 2):
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        n_groups = scales.size
        slot_bytes = payload.size // n_groups if n_groups else 0
        npdt = np.float32 if dtype == F32 else (np.float16 if dtype == F16 else np.uint16)
        out = np.zeros(max(n_groups * group_elems, 1), dtype=npdt)
        out_elems = np.zeros(max(n_groups, 1), dtype=np.uint32)
        scales = np.ascontiguousarray(scales, dtype=np.float32)
        comp = np.ascontiguousarray(comp, dtype=np.uint32)
        cls.lib().oracle_decompress_batch_scheme(_ptr(payload, _u8p), slot_bytes, _ptr(scales, _f32p),
                                                 _ptr(comp, _u32p), group_elems, n_groups, dtype,
                                                 out.ctypes.data, _ptr(out_elems, _u32p), scheme, threads)
        return out[: n_groups * group_elems].reshape(n_groups, group_elems), out_elems[:n_groups]

    # -- addresses ---------------------------------------------------------------------
    @classmethod
    def translate(cls, va: np.ndarray) -> np.ndarray:
        va = np.asarray(va, dtype=np.uint64)
        return np.uint64(0x4000000000) + (va & np.uint64(0xFFFFFFFFFFFF))

    @classmethod
    def atu_sequence(cls, vas, tlb_size: int = 1024):
        L = cls.lib()
        a = L.oracle_atu_new(tlb_size)
        a = C.c_void_p(a)
        out = [L.oracle_atu_translate(a, int(v)) for v in vas]
        h, m = C.c_uint64(), C.c_uint64()
        L.oracle_atu_stats(a, C.byref(h), C.byref(m))
        L.oracle_atu_free(a)
        return np.array(out, dtype=np.uint64), h.value, m.value

    @classmethod
    def access_addr(cls, handle: int, alloc_bytes: int, offset: int) -> int:
        return cls.lib().oracle_access_addr(handle, alloc_bytes, offset)

    # -- LSTM --------------------------------------------------------------------------
    @classmethod
    def lstm_weights(cls, seed: int = 1, vocab=32000, emb_dim=64, hidden=128, layers=2):
        emb = np.zeros(vocab * emb_dim, dtype=np.float32)
        wout = np.zeros(hidden * vocab, dtype=np.float32)
        cls.lib().oracle_lstm_init_weights(seed, _ptr(emb, _f32p), emb.size, None,
                                           layers * hidden * hidden * 4, _ptr(wout, _f32p), wout.size)
        return emb.reshape(vocab, emb_dim), wout.reshape(vocab, hidden)

    @classmethod
    def lstm_predict(cls, emb, wout, hist, k=4, layers=2, hist_len=16):
        emb = np.ascontiguousarray(emb, dtype=np.float32)
        wout = np.ascontiguousarray(wout, dtype=np.float32)
        vocab, emb_dim = emb.shape
        hidden = wout.shape[1]
        hist = np.ascontiguousarray(hist, dtype=np.uint32)
        ids = np.zeros(k, dtype=np.uint32)
        conf = np.zeros(k, dtype=np.float32)
        hid = np.zeros(hidden, dtype=np.float32)
        cls.lib().oracle_lstm_predict_topk(_ptr(emb, _f32p), _ptr(wout, _f32p), vocab, emb_dim, hidden,
                                           layers, hist_len, _ptr(hist, _u32p), hist.size, k,
                                           _ptr(ids, _u32p), _ptr(conf, _f32p), _ptr(hid, _f32p))
        return ids, conf, hid

    @classmethod
    def fnv1a64(cls, a: np.ndarray) -> int:
        a = np.ascontiguousarray(a)
        return cls.lib().oracle_fnv1a64(a.ctypes.data, a.nbytes)


class Ref:
    """The reference's own C++ model (oracle/_ref/libspeckv_ref.so)."""

    _lib = None

    @staticmethod
    def available() -> bool:
        return os.path.exists(REF_SO)

    @classmethod
    def lib(cls):
        if cls._lib is None:
            L = C.CDLL(REF_SO)
            L.ref_engine_new.restype = C.c_void_p
            L.ref_engine_free.argtypes = [C.c_void_p]
            L.ref_compress.restype = C.c_size_t
            L.ref_compress.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f32p, _u8p, C.c_size_t,
                                       C.POINTER(C.c_size_t)]
            L.ref_decompress.restype = C.c_size_t
            L.ref_decompress.argtypes = [C.c_void_p, C.c_float, _u8p, C.c_size_t, _f32p, C.c_size_t]
            L.ref_scale.restype = C.c_float
            L.ref_scale.argtypes = [C.c_void_p, _f32p, C.c_size_t]
            L.ref_quantize.argtypes = [C.c_void_p, _f32p, C.c_size_t, C.c_float, _i8p]
            L.ref_delta_encode.argtypes = [C.c_void_p, _i8p, C.c_size_t, _i8p]
            L.ref_engine_translate.restype = C.c_uint64
            L.ref_engine_translate.argtypes = [C.c_void_p, C.c_uint64]
            L.ref_engine_stats.argtypes = [C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t),
                                           C.POINTER(C.c_double), C.POINTER(C.c_double)]
            L.ref_engine_layer_ratio.restype = C.c_double
            L.ref_engine_layer_ratio.argtypes = [C.c_void_p, C.c_uint32]
            L.ref_roundtrip_batch.restype = C.c_int
            L.ref_roundtrip_batch.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_size_t, _u8p,
                                              C.c_size_t, _f32p, _u32p, C.c_void_p, C.c_int,
                                              C.c_int, C.c_int]
            L.ref_atu_new.restype = C.c_void_p
            L.ref_atu_new.argtypes = [C.c_size_t]
            L.ref_atu_free.argtypes = [C.c_void_p]
            L.ref_atu_translate.restype = C.c_uint64
            L.ref_atu_translate.argtypes = [C.c_void_p, C.c_uint64]
            L.ref_atu_invalidate.argtypes = [C.c_void_p, C.c_uint64]
            L.ref_atu_invalidate_all.argtypes = [C.c_void_p]
            L.ref_atu_stats.argtypes = [C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
            L.ref_lstm_new.restype = C.c_void_p
            L.ref_lstm_new.argtypes = [C.c_uint, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t, C.c_size_t]
            L.ref_lstm_free.argtypes = [C.c_void_p]
            L.ref_lstm_weights.argtypes = [C.c_void_p, _f32p, _f32p]
            L.ref_lstm_model_size.restype = C.c_size_t
            L.ref_lstm_model_size.argtypes = [C.c_void_p]
            L.ref_lstm_predict.restype = C.c_size_t
            L.ref_lstm_predict.argtypes = [C.c_void_p, _u32p, C.c_size_t, C.c_size_t, _u32p, _f32p]
            L.ref_prefetcher_new.restype = C.c_void_p
            L.ref_prefetcher_new.argtypes = [C.c_uint, C.c_size_t, C.c_size_t]
            L.ref_prefetcher_free.argtypes = [C.c_void_p]
            L.ref_prefetcher_weights.argtypes = [C.c_void_p, _f32p, _f32p]
            L.ref_prefetcher_prefetch.restype = C.c_size_t
            L.ref_prefetcher_prefetch.argtypes = [C.c_void_p, _u32p, C.c_size_t, C.c_uint32, C.c_size_t,
                                                  _u64p, _u32p, _u32p, _f32p]
            L.ref_prefetcher_mm_allocate.restype = C.c_uint64
            L.ref_prefetcher_mm_allocate.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_int]
            L.ref_prefetcher_mispredict.argtypes = [C.c_void_p, C.c_uint32, _u32p, C.c_size_t]
            L.ref_prefetcher_stats.argtypes = [C.c_void_p, _u64p, _f64p, C.c_int]
            L.ref_prefetcher_is_outstanding.restype = C.c_int
            L.ref_prefetcher_is_outstanding.argtypes = [C.c_void_p, C.c_uint64]
            L.ref_prefetcher_queue.restype = C.c_size_t
            L.ref_prefetcher_queue.argtypes = [C.c_void_p, _u64p, _u32p, C.c_size_t]
            L.ref_kv_address.restype = C.c_uint64
            L.ref_kv_address.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
            L.ref_mm_new.restype = C.c_void_p
            L.ref_mm_free.argtypes = [C.c_void_p]
            L.ref_mm_allocate.restype = C.c_uint64
            L.ref_mm_allocate.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_int]
            L.ref_mm_translate.restype = C.c_uint64
            L.ref_mm_translate.argtypes = [C.c_void_p, C.c_uint64]
            L.ref_mm_is_in_cache.restype = C.c_int
            L.ref_mm_is_in_cache.argtypes = [C.c_void_p, C.c_uint64, C.c_int]
            for f in ("ref_mm_touch", "ref_mm_release"):
                getattr(L, f).restype = None
                getattr(L, f).argtypes = [C.c_void_p, C.c_uint64]
            for f in ("ref_mm_is_hot", "ref_mm_promote", "ref_mm_demote", "ref_mm_tier"):
                getattr(L, f).restype = C.c_int
                getattr(L, f).argtypes = [C.c_void_p, C.c_uint64]
            L.ref_mm_lru.restype = C.c_size_t
            L.ref_mm_lru.argtypes = [C.c_void_p, _u64p, C.c_size_t]
            L.ref_mm_stats.argtypes = [C.c_void_p, _u64p, _f64p]
            cls._lib = L
            cls._engine = C.c_void_p(L.ref_engine_new())
        return cls._lib

    @classmethod
    def compress(cls, x: np.ndarray):
        L = cls.lib()
        x = np.ascontiguousarray(x, dtype=np.float32).ravel()
        out = np.zeros(max(2 * x.size, 2), dtype=np.uint8)
        s = C.c_float()
        orig = C.c_size_t()
        n = L.ref_compress(cls._engine, _ptr(x, _f32p), x.size, C.byref(s), _ptr(out, _u8p), out.size,
                           C.byref(orig))
        return np.float32(s.value), out[:n].copy()

    @classmethod
    def decompress(cls, scale, payload: np.ndarray, cap: int) -> np.ndarray:
        L = cls.lib()
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        out = np.zeros(max(cap, 1), dtype=np.float32)
        n = L.ref_decompress(cls._engine, C.c_float(float(scale)), _ptr(payload, _u8p), payload.size,
                             _ptr(out, _f32p), cap)
        return out[: min(n, cap)].copy()

    @classmethod
    def quantize(cls, x: np.ndarray, scale) -> np.ndarray:
        L = cls.lib()
        x = np.ascontiguousarray(x, dtype=np.float32).ravel()
        q = np.zeros(x.size, dtype=np.int8)
        L.ref_quantize(cls._engine, _ptr(x, _f32p), x.size, C.c_float(float(scale)), _ptr(q, _i8p))
        return q

    @classmethod
    def scale(cls, x: np.ndarray) -> np.float32:
        L = cls.lib()
        x = np.ascontiguousarray(x, dtype=np.float32).ravel()
        return np.float32(L.ref_scale(cls._engine, _ptr(x, _f32p), x.size))

    @classmethod
    def engine_translate(cls, vas) -> np.ndarray:
        L = cls.lib()
        return np.array([L.ref_engine_translate(cls._engine, int(v)) for v in vas], dtype=np.uint64)

    @classmethod
    def atu_sequence(cls, vas, tlb_size: int = 1024):
        L = cls.lib()
        a = C.c_void_p(L.ref_atu_new(tlb_size))
        out = np.array([L.ref_atu_translate(a, int(v)) for v in vas], dtype=np.uint64)
        h, m = C.c_size_t(), C.c_size_t()
        L.ref_atu_stats(a, C.byref(h), C.byref(m))
        L.ref_atu_free(a)
        return out, h.value, m.value

    @classmethod
    def roundtrip_batch(cls, x_u16: np.ndarray, dtype: int, group_elems: int, threads: int,
                        do_compress=True, do_decompress=True, state=None):
        """Reference engine round trip over fp16/bf16 bit patterns (timed CPU baseline)."""
        L = cls.lib()
        x_u16 = np.ascontiguousarray(x_u16).view(np.uint16).ravel()
        n_groups = x_u16.size // group_elems
        slot = (2 * group_elems + 15) // 16 * 16
        if state is None:
            payload = np.zeros(n_groups * slot, dtype=np.uint8)
            scales = np.zeros(n_groups, dtype=np.float32)
            comp = np.zeros(n_groups, dtype=np.uint32)
        else:
            payload, scales, comp = state
        out = np.zeros(n_groups * group_elems, dtype=np.uint16)
        L.ref_roundtrip_batch(x_u16.ctypes.data, dtype, group_elems, n_groups, _ptr(payload, _u8p), slot,
                              _ptr(scales, _f32p), _ptr(comp, _u32p), out.ctypes.data, threads,
                              int(do_compress), int(do_decompress))
        return payload.reshape(n_groups, slot), scales, comp, out.reshape(n_groups, group_elems)


class PolicyStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("l1_hits", "l1_misses", "l2_hits", "l2_misses", "l3_accesses",
                                          "migrations_l1_to_l3", "migrations_l3_to_l1")] + \
               [("l1_hit_rate", C.c_double), ("l2_hit_rate", C.c_double)] + \
               [(n, C.c_uint64) for n in ("l1_pages", "l2_pages", "l3_pages")]


class PolicyOracle:
    """oracle_policy_* of the C restatement driven a batch at a time (its *_n forms: the single-page calls in
    order), for traces too long for one ctypes call per page.  Ids are taken as uint64, so a negative id is a
    page past the end."""

    def __init__(self, n_pages: int, caps=(1 << 40, 1 << 40, 1 << 40)):
        self.L = Port.lib()
        self.n_pages = n_pages
        self.h = C.c_void_p(self.L.oracle_policy_new(n_pages, *caps))

    def close(self):
        if self.h:
            self.L.oracle_policy_free(self.h)
            self.h = C.c_void_p()

    @staticmethod
    def _ids(ids) -> np.ndarray:
        return np.ascontiguousarray(np.asarray(ids).astype(np.uint64, copy=False).ravel())

    def place(self, ids, tier: int) -> np.ndarray:
        """-> the tier each page went to, -1 where it was rejected"""
        ids = self._ids(ids)
        out = np.zeros(ids.size, dtype=np.int32)
        self.L.oracle_policy_place_n(self.h, _ptr(ids, _u64p), ids.size, tier, _ptr(out, C.POINTER(C.c_int32)))
        return out

    def touch(self, ids) -> None:
        ids = self._ids(ids)
        self.L.oracle_policy_touch_n(self.h, _ptr(ids, _u64p), ids.size)

    def release(self, ids) -> None:
        ids = self._ids(ids)
        self.L.oracle_policy_release_n(self.h, _ptr(ids, _u64p), ids.size)

    def demote(self, ids) -> np.ndarray:
        ids = self._ids(ids)
        ok = np.zeros(ids.size, dtype=np.uint8)
        self.L.oracle_policy_demote_n(self.h, _ptr(ids, _u64p), ids.size, _ptr(ok, _u8p))
        return ok

    def is_hot(self, ids) -> np.ndarray:
        ids = self._ids(ids)
        hot = np.zeros(ids.size, dtype=np.uint8)
        self.L.oracle_policy_is_hot_n(self.h, _ptr(ids, _u64p), ids.size, _ptr(hot, _u8p))
        return hot

    def promote(self, ids):
        """-> (ok[n] uint8, evicted page ids in order)"""
        ids = self._ids(ids)
        ok = np.zeros(ids.size, dtype=np.uint8)
        ev = np.zeros(max(ids.size, 1), dtype=np.uint64)
        k = self.L.oracle_policy_promote_n(self.h, _ptr(ids, _u64p), ids.size, _ptr(ok, _u8p), _ptr(ev, _u64p))
        return ok, ev[:k].copy()

    def tiers(self) -> np.ndarray:
        out = np.zeros(max(self.n_pages, 1), dtype=np.uint8)
        self.L.oracle_policy_tiers(self.h, _ptr(out, _u8p))
        return out[: self.n_pages]

    def lru_order(self) -> np.ndarray:
        out = np.zeros(max(self.n_pages, 1), dtype=np.uint64)
        k = self.L.oracle_policy_lru(self.h, _ptr(out, _u64p), self.n_pages)
        return out[:k].copy()

    def stats(self) -> dict:
        st = PolicyStats()
        self.L.oracle_policy_stats(self.h, C.byref(st))
        return {n: getattr(st, n) for n, _ in PolicyStats._fields_}


def run_policy_trace(ops, n_pages: int, caps=(1 << 40, 1 << 40, 1 << 40), impl: str = "port"):
    """Runs a residency-policy trace and returns what an observer can see.

    ops: list of (op, page[, tier]) with op in place / touch / hot / promote / demote / release.
    impl "port" = oracle/speckv_oracle.c; impl "ref" = the reference's CXLMemoryManager through
    oracle/_ref (one page per allocation; its capacities are whole GiB, so `caps` is ignored and a
    trace for it must never fill L1 -- the reference's eviction path deadlocks).
    Returns {"results": [...], "tiers": [...], "lru": [...], "stats": {...}}."""
    results = []
    if impl == "port":
        L = Port.lib()
        h = C.c_void_p(L.oracle_policy_new(n_pages, *caps))
        for op in ops:
            name, page = op[0], op[1]
            if name == "place":
                results.append(L.oracle_policy_place(h, page, op[2]))
            elif name == "touch":
                L.oracle_policy_touch(h, page); results.append(0)
            elif name == "hot":
                results.append(L.oracle_policy_is_hot(h, page))
            elif name == "promote":
                ev = C.c_uint64()
                ok = L.oracle_policy_promote(h, page, C.byref(ev))
                results.append((ok, None if ev.value == 0xFFFFFFFFFFFFFFFF else ev.value))
            elif name == "demote":
                results.append(L.oracle_policy_demote(h, page))
            elif name == "release":
                L.oracle_policy_release(h, page); results.append(0)
            else:
                raise ValueError(name)
        tiers = [L.oracle_policy_tier(h, g) for g in range(n_pages)]
        buf = (C.c_uint64 * max(n_pages, 1))()
        k = L.oracle_policy_lru(h, buf, n_pages)
        lru = [int(buf[i]) for i in range(k)]
        st = PolicyStats()
        L.oracle_policy_stats(h, C.byref(st))
        stats = {n: getattr(st, n) for n, _ in PolicyStats._fields_}
        L.oracle_policy_free(h)
    else:
        L = Ref.lib()
        m = C.c_void_p(L.ref_mm_new())
        va_of, page_of = {}, {}
        for op in ops:
            name, page = op[0], op[1]
            if name == "place":
                if page in va_of:
                    results.append(-1)
                    continue
                va = L.ref_mm_allocate(m, 4096, 0, op[2])
                va_of[page] = va; page_of[va] = page
                results.append(L.ref_mm_tier(m, va))
                continue
            va = va_of.get(page, 0x10)           # an address the manager has never seen
            if name == "touch":
                L.ref_mm_touch(m, va); results.append(0)
            elif name == "hot":
                results.append(L.ref_mm_is_hot(m, va))
            elif name == "promote":
                results.append((L.ref_mm_promote(m, va), None))
            elif name == "demote":
                results.append(L.ref_mm_demote(m, va))
            elif name == "release":
                L.ref_mm_release(m, va); va_of.pop(page, None); results.append(0)
            else:
                raise ValueError(name)
        tiers = [L.ref_mm_tier(m, va_of[g]) if g in va_of else 255 for g in range(n_pages)]
        k = L.ref_mm_lru(m, None, 0)
        buf = (C.c_uint64 * max(k, 1))()
        k = L.ref_mm_lru(m, buf, k)
        # entries of released L2/L3 pages dangle in the reference's list (:89-100); their addresses are
        # never handed out again, so only the entries of live pages are observable
        lru = [page_of[int(buf[i])] for i in range(k) if va_of.get(page_of.get(int(buf[i]))) == int(buf[i])]
        c7 = (C.c_uint64 * 7)(); r2 = (C.c_double * 2)()
        L.ref_mm_stats(m, c7, r2)
        names = ["l1_hits", "l1_misses", "l2_hits", "l2_misses", "l3_accesses", "migrations_l1_to_l3", "migrations_l3_to_l1"]
        stats = {n: int(c7[i]) for i, n in enumerate(names)}
        stats["l1_hit_rate"], stats["l2_hit_rate"] = r2[0], r2[1]
        for t, n in enumerate(("l1_pages", "l2_pages", "l3_pages")):
            stats[n] = sum(1 for x in tiers if x == t)
        L.ref_mm_free(m)
    return {"results": results, "tiers": tiers, "lru": lru, "stats": stats}


def random_policy_trace(seed: int):
    """-> (ops, n_pages): a random residency-policy trace for run_policy_trace that never fills L1 (the reference's
    eviction path deadlocks).  The traces of tests/golden/reference_traces.json."""
    import random
    rng = random.Random(seed)
    n = rng.choice([8, 64, 300])
    ops = [("place", g, rng.choice([0, 1, 2, 2])) for g in range(n) if rng.random() < 0.9]
    for _ in range(3000):
        r, g = rng.random(), rng.randrange(n)
        if r < 0.6:
            ops.append(("touch", g))
        elif r < 0.7:
            ops.append(("hot", g))
        elif r < 0.8:
            ops.append(("promote", g))
        elif r < 0.9:
            ops.append(("demote", g))
        elif r < 0.93:
            ops.append(("release", g))
        else:
            ops.append(("place", g, rng.choice([0, 1, 2])))
    return ops, n


def random_codec_cases(seed: int = 11):
    """-> (inputs, payloads): fp32 groups of mixed magnitude for compress, and arbitrary (not produced by compress)
    (scale, payload) pairs for decompress.  The codec cases of tests/golden/reference_traces.json."""
    rng = np.random.default_rng(seed)
    inputs = []
    for trial in range(60):
        n = int(rng.integers(1, 5000))
        kind = trial % 4
        if kind == 0:
            x = rng.standard_normal(n).astype(np.float16).astype(np.float32)
        elif kind == 1:
            x = np.repeat(rng.standard_normal(n // 97 + 1), 97)[:n].astype(np.float16).astype(np.float32)
        elif kind == 2:
            b = np.ascontiguousarray(rng.standard_normal(n) * np.exp(rng.uniform(-90, 80)), dtype=np.float32)
            u = b.view(np.uint32).astype(np.uint64)                          # to bf16, RN-even, and back
            x = (((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint32) << 16).view(np.float32)
        else:
            x = (rng.standard_normal(n) * np.exp(rng.uniform(-30, 30, n))).astype(np.float32)
        inputs.append(x)
    payloads = []
    for trial in range(20):
        p = rng.integers(0, 256, int(rng.integers(0, 400)), dtype=np.uint8)
        if trial % 2:
            p[1::2] = rng.integers(0, 4, p[1::2].size)
        payloads.append((np.float32(rng.uniform(0.001, 3)), p))
    return inputs, payloads


def splitmix64_block(seed: int, n: int) -> np.ndarray:
    """The cross-language integer generator of SURVEY.md section 8c: splitmix64(seed) ->
    k = sum of four 11-bit fields - 4094, x = k / 1024 (exactly representable in fp16)."""
    mask = (1 << 64) - 1
    out = np.empty(n, dtype=np.float32)
    s = seed & mask
    for i in range(n):
        s = (s + 0x9E3779B97F4A7C15) & mask
        z = s
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & mask
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & mask
        z = z ^ (z >> 31)
        k = (z & 0x7FF) + ((z >> 11) & 0x7FF) + ((z >> 22) & 0x7FF) + ((z >> 33) & 0x7FF) - 4094
        out[i] = k / 1024.0
    return out
