#!/usr/bin/env python
"""Generate tests/golden/ from the REFERENCE's own C++ model (oracle/_ref).

TEST INFRASTRUCTURE ONLY.  Run in the authoring container, where /root/reference
exists and `make -C oracle ref` has produced oracle/_ref/libspeckv_ref.so:

    python oracle/make_golden.py
    python oracle/make_golden.py traces [ref|port]   # only tests/golden/reference_traces.json

Every fixture in golden.json, codec_cases.npz and translate_cases.npz is the output of
the reference's unmodified sources (FPGACacheEngine::compress/decompress,
translate_address, AddressTranslationUnit, LSTMPredictor::predict_top_k,
SpeculativePrefetcher::prefetch, the host C API with /dev/null as the device).
tests/test_oracle_golden.py pins the C restatement to them on CPU;
tests/test_codec_gpu.py pins the CUDA path to them on a B200.

reference_traces.json is the exception that names its source in its "source" field.
`traces ref` records it from the reference.  `traces port` records it from the C
restatement, for a checkout without the reference's sources: the tests then pin the
restatement to its own recorded answers, and compare it with the reference itself
wherever oracle/_ref is built.  A `traces port` run refuses to replace a recording
made from the reference.
"""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[0] = ROOT  # replace the script dir (it would shadow the package with oracle.py)
from oracle.oracle import Port, Ref, REF_CAPI_SO, splitmix64_block, F16, BF16, F32  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def f32_bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def bf16_from_f32(a):
    """fp32 -> bf16 bit patterns, RN-even (numpy has no bf16)."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = u + 0x7FFF + ((u >> 16) & 1)
    return (u >> 16).astype(np.uint16)


def bf16_to_f32(b):
    return (b.astype(np.uint32) << 16).view(np.float32)


def codec_cases():
    rng = np.random.default_rng(20251017)
    cases = {}

    def add(name, x, dtype):
        cases[name] = (np.ascontiguousarray(x), dtype)

    # known-answer vectors of SURVEY.md section 8c (fp32 at the engine boundary)
    add("kat1_mixed", np.array([0, 1, -1, 0.5, 0.25, 0.25, 0.25, 2, -2, 1e-3], np.float32), F32)
    add("kat2_zeros1000", np.zeros(1000, np.float32), F32)
    add("kat3_const600", np.full(600, 3.0, np.float32), F32)
    add("kat4_nan", np.array([1, np.nan, -3], np.float32), F32)
    add("kat5_nan_inf", np.array([1, np.nan, -3, np.inf], np.float32), F32)
    add("single", np.array([-0.75], np.float32), F32)
    add("f32_randn_1000", rng.standard_normal(1000).astype(np.float32), F32)
    add("f32_tiny_denormal", (rng.standard_normal(300) * 1e-41).astype(np.float32), F32)
    add("f32_huge", (rng.standard_normal(300) * 1e37).astype(np.float32), F32)
    # fp16 groups, N(0,1): the headline distribution (nearly every code wraps)
    for n in (1, 2, 7, 8, 9, 255, 256, 257, 2048, 4099):
        add(f"f16_randn_{n}", rng.standard_normal(n).astype(np.float16), F16)
    add("f16_randn_scaled_small", (rng.standard_normal(2048) * 1e-3).astype(np.float16), F16)
    add("f16_denormals", (rng.standard_normal(512) * 3e-6).astype(np.float16), F16)
    # runs and the 255 cap
    for n in (254, 255, 256, 509, 510, 511, 512, 765, 766, 1021):
        add(f"f16_const_{n}", np.full(n, 0.5, np.float16), F16)
    runs = np.repeat(rng.standard_normal(14).astype(np.float16), 300)[:4096]
    add("f16_runs300", runs, F16)
    ramp = (np.arange(3000) % 97).astype(np.float16) / np.float16(8)
    add("f16_ramp", ramp, F16)                      # constant deltas -> long delta runs
    lin = (np.arange(2048, dtype=np.float32) * (1.0 / 2048)).astype(np.float16)
    add("f16_linear", lin, F16)
    mix = rng.standard_normal(4096).astype(np.float16)
    mix[700:1500] = 0
    mix[2000:2600] = mix[1999]
    add("f16_mixed_runs", mix, F16)
    # special values in fp16
    sp = rng.standard_normal(2048).astype(np.float16)
    sp[5] = np.nan
    sp[77] = np.nan
    add("f16_nan", sp, F16)
    sp2 = sp.copy()
    sp2[100] = np.inf
    add("f16_nan_inf", sp2, F16)
    sp3 = rng.standard_normal(300).astype(np.float16)
    sp3[17] = -np.inf
    add("f16_neg_inf", sp3, F16)
    add("f16_all_nan", np.full(64, np.nan, np.float16), F16)
    add("f16_maxval", np.array([65504, -65504, 1, 0.5, 6e-8, -6e-8] * 20, np.float16), F16)
    # tie-heavy: values k/ (2*127*127) * max make (x/s)*127 land on .5 often
    k = rng.integers(-16129, 16129, 4096)
    tie = ((2 * k + 1) / 2.0 / 16129.0 * 4.0).astype(np.float16)
    tie[0] = 4.0
    add("f16_ties", tie, F16)
    # bf16 bit patterns (uint16)
    add("bf16_randn_2048", bf16_from_f32(rng.standard_normal(2048)), BF16)
    add("bf16_randn_257", bf16_from_f32(rng.standard_normal(257) * 37.0), BF16)
    add("bf16_tiny", bf16_from_f32(rng.standard_normal(512) * 1e-30), BF16)     # max < 2^-60 path
    add("bf16_subnormal", bf16_from_f32(rng.standard_normal(512) * 1e-39), BF16)
    add("bf16_mixed_mag", bf16_from_f32(rng.standard_normal(1024) * np.exp(rng.uniform(-80, 20, 1024))), BF16)
    add("bf16_huge", bf16_from_f32(rng.standard_normal(512) * 1e38), BF16)
    return cases


def widen(x, dtype):
    if dtype == BF16:
        return bf16_to_f32(x)
    return x.astype(np.float32)


def main():
    assert Ref.available(), "build oracle/_ref first: make -C oracle ref"
    os.makedirs(OUT, exist_ok=True)
    meta = {"generator": "oracle/make_golden.py", "source": "oracle/_ref (reference C++ model, unmodified)",
            "codec": {}, "bulk": {}, "translate": {}, "capi": {}, "lstm": {}, "adaptive_depth": {}}

    # ---- codec fixtures ------------------------------------------------------------
    arrays = {}
    for name, (x, dtype) in codec_cases().items():
        xf = widen(x, dtype)
        s, p = Ref.compress(xf)
        y = Ref.decompress(s, p, xf.size + 8)
        q = Ref.quantize(xf, s)
        arrays[name + ".in"] = x if dtype != F16 else x.view(np.uint16)
        arrays[name + ".payload"] = p
        arrays[name + ".out_f32_bits"] = f32_bits(y)
        arrays[name + ".codes"] = q
        meta["codec"][name] = {"dtype": int(dtype), "n": int(x.size), "scale_bits": int(f32_bits([s])[0]),
                               "comp_bytes": int(p.size), "out_elems": int(y.size)}
        # the restatement must agree before anything is written
        s2, p2 = Port.compress(xf)
        assert f32_bits([s2])[0] == f32_bits([s])[0] and np.array_equal(p, p2), name
        assert np.array_equal(f32_bits(Port.decompress(s, p, xf.size + 8)), f32_bits(y)), name
    np.savez_compressed(os.path.join(OUT, "codec_cases.npz"), **arrays)

    # ---- bulk digests (one full 1024x128 group; inputs regenerated by the tests) -----
    x = splitmix64_block(42, 131072)
    s, p = Ref.compress(x)
    y = Ref.decompress(s, p, x.size)
    meta["bulk"]["splitmix42_131072"] = {
        "scale_bits": int(f32_bits([s])[0]), "comp_bytes": int(p.size),
        "payload_fnv1a64": "%016x" % Port.fnv1a64(p), "out_f32_fnv1a64": "%016x" % Port.fnv1a64(y),
        "out_f16_fnv1a64": "%016x" % Port.fnv1a64(y.astype(np.float16)),
        "in_f16_fnv1a64": "%016x" % Port.fnv1a64(x.astype(np.float16))}

    # ---- address translation -------------------------------------------------------
    rng = np.random.default_rng(7)
    vas = np.concatenate([
        np.array([0x100000123, 0x100000FFF, 0xFFFF000000000ABC, 0, 0xFFF, 0x1000, 2**48 - 1, 2**48, 2**64 - 1],
                 dtype=np.uint64),
        rng.integers(0, 2**63, 64, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, 64, dtype=np.uint64),
        (np.uint64(0x100000000) + rng.integers(0, 64, 128, dtype=np.uint64) * np.uint64(4096)
         + rng.integers(0, 4096, 128, dtype=np.uint64)),
    ])
    eng = Ref.engine_translate(vas)
    atu, hits, misses = Ref.atu_sequence(vas)
    meta["translate"] = {"n": int(vas.size), "atu_hits": int(hits), "atu_misses": int(misses)}
    np.savez_compressed(os.path.join(OUT, "translate_cases.npz"), va=vas, engine_pa=eng, atu_pa=atu)

    # ---- host C API with /dev/null as the device (SURVEY.md section 4) ------------------
    L = C.CDLL(REF_CAPI_SO)
    L.speckv_init.argtypes = [C.c_char_p]
    L.speckv_alloc.argtypes = [C.c_size_t, C.c_void_p, C.POINTER(C.c_uint64)]
    L.speckv_free.argtypes = [C.c_uint64]
    L.speckv_access.argtypes = [C.c_uint64, C.c_uint64, C.c_size_t, C.POINTER(C.c_void_p)]
    L.speckv_prefetch.argtypes = [C.c_uint32, C.c_uint16, C.c_uint32, C.c_uint32, C.POINTER(C.c_int32), C.c_uint32]
    log = []
    h = C.c_uint64()
    ptr = C.c_void_p()
    toks = (C.c_int32 * 4)(1, 2, 3, 4)
    log.append(["alloc_before_init", L.speckv_alloc(4096, None, C.byref(h))])
    log.append(["access_before_init", L.speckv_access(1, 0, 1, C.byref(ptr))])
    log.append(["free_before_init", L.speckv_free(1)])
    log.append(["prefetch_before_init", L.speckv_prefetch(0, 0, 0, 4, toks, 4)])
    log.append(["set_depth_before_init", L.speckv_set_prefetch_depth(4)])
    log.append(["set_scheme_before_init", L.speckv_set_compression_scheme(2)])
    log.append(["init_bad_path", L.speckv_init(b"/nonexistent/speckv0")])
    log.append(["init", L.speckv_init(b"/dev/null")])
    log.append(["init_twice", L.speckv_init(b"/dev/null")])
    log.append(["alloc_null_out", L.speckv_alloc(4096, None, None)])
    accesses = []
    for size in (1 << 20, 1 << 20, 5000, 3 << 20, 1):
        rc = L.speckv_alloc(size, None, C.byref(h))
        log.append([f"alloc_{size}", rc, int(h.value)])
        for off in (0, 100, 4095, 4096, 8191, 8192, size - 1, size, ((size + 4095) // 4096) * 4096 - 1,
                    ((size + 4095) // 4096) * 4096):
            ptr.value = 0xDEAD
            rc = L.speckv_access(h.value, off, 64, C.byref(ptr))
            accesses.append([int(h.value), int(size), int(off), rc, int(ptr.value or 0)])
    log.append(["access_unknown_handle", L.speckv_access(99, 0, 1, C.byref(ptr))])
    log.append(["access_null_out", L.speckv_access(1, 0, 1, None)])
    log.append(["free_unknown", L.speckv_free(12345)])
    log.append(["free_2", L.speckv_free(2)])
    log.append(["access_freed", L.speckv_access(2, 0, 1, C.byref(ptr))])
    log.append(["prefetch", L.speckv_prefetch(1, 3, 17, 4, toks, 4)])
    log.append(["prefetch_null_tokens", L.speckv_prefetch(1, 3, 17, 4, None, 4)])
    log.append(["prefetch_zero_len", L.speckv_prefetch(1, 3, 17, 4, toks, 0)])
    log.append(["set_depth_devnull", L.speckv_set_prefetch_depth(4)])
    log.append(["set_scheme_devnull", L.speckv_set_compression_scheme(2)])
    L.speckv_finalize()
    log.append(["alloc_after_finalize", L.speckv_alloc(4096, None, C.byref(h))])
    log.append(["reinit", L.speckv_init(b"/dev/null")])
    rc = L.speckv_alloc(4096, None, C.byref(h))
    log.append(["alloc_after_reinit", rc, int(h.value)])
    L.speckv_finalize()
    meta["capi"] = {"log": log, "accesses": accesses}

    # ---- LSTM predictor / prefetcher (weights = glibc rand() after srand(1)) ---------
    lib = Ref.lib()
    pred = C.c_void_p(lib.ref_lstm_new(1, 32000, 64, 128, 2, 16))
    emb = np.zeros(32000 * 64, np.float32)
    wout = np.zeros(32000 * 128, np.float32)
    lib.ref_lstm_weights(pred, emb.ctypes.data_as(C.POINTER(C.c_float)), wout.ctypes.data_as(C.POINTER(C.c_float)))
    pe, pw = Port.lstm_weights(1)
    assert np.array_equal(pe.ravel(), emb) and np.array_equal(pw.ravel(), wout), "rand() weight replay differs"
    rng = np.random.default_rng(7)
    hists = [rng.integers(0, 32000, 16).tolist() for _ in range(12)]
    hists += [[5, 6, 7], list(range(40)), [31999] * 16, [0] * 16, [40000, 3, 9, 100000, 12]]
    preds = []
    for hst in hists:
        a = np.array(hst, np.uint32)
        ids = np.zeros(8, np.uint32)
        conf = np.zeros(8, np.float32)
        n = lib.ref_lstm_predict(pred, a.ctypes.data_as(C.POINTER(C.c_uint32)), a.size, 8,
                                 ids.ctypes.data_as(C.POINTER(C.c_uint32)), conf.ctypes.data_as(C.POINTER(C.c_float)))
        preds.append({"hist": hst, "ids": ids[:n].tolist(), "conf_bits": f32_bits(conf[:n]).tolist()})
    meta["lstm"] = {"seed": 1, "emb_fnv1a64": "%016x" % Port.fnv1a64(emb), "wout_fnv1a64": "%016x" % Port.fnv1a64(wout),
                    "model_size": int(lib.ref_lstm_model_size(pred)), "predictions": preds}
    lib.ref_lstm_free(pred)
    # prefetcher: request emission (addresses, order) for depth 4
    pf = C.c_void_p(lib.ref_prefetcher_new(1, 4, 16))
    a = np.array(hists[0], np.uint32)
    va = np.zeros(8, np.uint64); lay = np.zeros(8, np.uint32); tok = np.zeros(8, np.uint32); cf = np.zeros(8, np.float32)
    n = lib.ref_prefetcher_prefetch(pf, a.ctypes.data_as(C.POINTER(C.c_uint32)), a.size, 5, 4,
                                    va.ctypes.data_as(C.POINTER(C.c_uint64)), lay.ctypes.data_as(C.POINTER(C.c_uint32)),
                                    tok.ctypes.data_as(C.POINTER(C.c_uint32)), cf.ctypes.data_as(C.POINTER(C.c_float)))
    meta["lstm"]["prefetch"] = {"hist": hists[0], "layer": 5, "depth": 4, "va": va[:n].tolist(),
                                "layer_out": lay[:n].tolist(), "tok": tok[:n].tolist(),
                                "conf_bits": f32_bits(cf[:n]).tolist()}
    # adaptive depth trace (update_prediction_accuracy / get_adaptive_depth)
    lib.ref_prefetcher_feedback.argtypes = [C.c_void_p, C.c_int]
    lib.ref_prefetcher_adaptive_depth.restype = C.c_size_t
    lib.ref_prefetcher_adaptive_depth.argtypes = [C.c_void_p]
    rng = np.random.default_rng(5)
    outcomes = np.concatenate([rng.random(150) < 0.99, rng.random(150) < 0.5, rng.random(200) < 0.9,
                               np.ones(60, bool)]).astype(int).tolist()
    trace = []
    for o in outcomes:
        lib.ref_prefetcher_feedback(pf, int(o))
        trace.append(int(lib.ref_prefetcher_adaptive_depth(pf)))
    meta["adaptive_depth"] = {"initial": 4, "outcomes": outcomes, "depth_trace": trace}
    lib.ref_prefetcher_free(pf)

    with open(os.path.join(OUT, "golden.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    print("wrote", OUT, {k: len(v) if hasattr(v, "__len__") else v for k, v in meta.items() if k != "generator"})
    record_traces("ref")


TRACE_SOURCES = {
    "ref": "oracle/_ref (reference C++ model, unmodified): FPGACacheEngine::compress/decompress, CXLMemoryManager",
    "port": "oracle/speckv_oracle.c (the C restatement), recorded where the reference was not built; the restatement "
            "matched the reference on these same cases while oracle/_ref was built alongside it",
}


def record_traces(impl: str):
    """tests/golden/reference_traces.json: what the reference answers on the random codec cases and residency-policy
    traces of oracle.random_codec_cases / random_policy_trace (digests for the codec, full traces for the policy)."""
    from oracle.oracle import random_codec_cases, random_policy_trace, run_policy_trace
    E = {"ref": Ref, "port": Port}[impl]
    path = os.path.join(OUT, "reference_traces.json")
    if impl == "port" and os.path.exists(path):
        with open(path) as f:
            if json.load(f).get("source") == TRACE_SOURCES["ref"]:
                raise SystemExit(f"{path} holds the reference's own answers; the restatement does not replace them")
    inputs, payloads = random_codec_cases()
    comp, dec = [], []
    for x in inputs:
        s, p = E.compress(x)
        y = E.decompress(s, p, x.size)
        comp.append([int(f32_bits([s])[0]), int(p.size), "%016x" % Port.fnv1a64(p), "%016x" % Port.fnv1a64(f32_bits(y))])
    for s, p in payloads:
        y = E.decompress(s, p, 200000)
        dec.append([int(y.size), "%016x" % Port.fnv1a64(f32_bits(y))])
    policy = []
    for seed in range(4):
        ops, n = random_policy_trace(seed)
        r = run_policy_trace(ops, n, impl=impl)
        policy.append(dict(r, seed=seed, n_pages=n, n_ops=len(ops)))
    out = {"generator": "oracle/make_golden.py", "source": TRACE_SOURCES[impl],
           "codec_random": {"compress": comp, "decompress": dec}, "policy": policy}
    # one line per top-level entry: the traces are data, not meant to be read line by line
    with open(path, "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(out[k], sort_keys=True, separators=(',', ':'))}"
                                  for k in sorted(out)) + "\n}\n")
    print("wrote", path, "from", impl)


if __name__ == "__main__":
    if sys.argv[1:2] == ["traces"]:
        record_traces(sys.argv[2] if len(sys.argv) > 2 else "ref")
    else:
        main()
