"""CPU: the C restatement (oracle/speckv_oracle.c) against the fixtures produced by the
reference's own C++ model (tests/golden, see oracle/make_golden.py) and, when
oracle/_ref is present, against the reference itself on the same random inputs."""
import numpy as np
import pytest

from oracle.oracle import Port, Ref, splitmix64_block
from tests.helpers import F16, BF16, F32, bf16_from_f32, bf16_to_f32, case_input, f32_bits


@pytest.fixture(scope="module")
def reference_traces():
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_traces.json")) as f:
        return json.load(f)


def test_codec_fixtures(golden):
    meta, codec = golden["meta"], golden["codec"]
    assert len(meta["codec"]) >= 40
    for name, m in meta["codec"].items():
        _, xf, _ = case_input(codec, meta, name)
        s, p = Port.compress(xf)
        assert int(f32_bits([s])[0]) == m["scale_bits"], name
        assert p.size == m["comp_bytes"], name
        assert np.array_equal(p, codec[name + ".payload"]), name
        assert np.array_equal(Port.quantize(xf, s), codec[name + ".codes"]), name
        y = Port.decompress(s, p, xf.size + 8)
        assert y.size == m["out_elems"] == xf.size, name
        assert np.array_equal(f32_bits(y), codec[name + ".out_f32_bits"]), name


def test_survey_known_answers():
    # SURVEY.md section 8c KAT-1..5 (measured on the reference)
    s, p = Port.compress(np.array([0, 1, -1, 0.5, 0.25, 0.25, 0.25, 2, -2, 1e-3], np.float32))
    assert float(s).hex() == "0x1.0204080000000p-6"
    assert p.view(np.int8).tolist() == [0, 1, -127, 1, -2, 1, 65, 1, 32, 1, 0, 2, 33, 1, -2, 1, 9, 1]
    s, p = Port.compress(np.zeros(1000, np.float32))
    assert s == 1.0 and p.tolist() == [0, 255, 0, 255, 0, 255, 0, 235]
    s, p = Port.compress(np.full(600, 3.0, np.float32))
    assert float(s).hex() == "0x1.83060c0000000p-6" and p.tolist() == [1, 1, 0, 255, 0, 255, 0, 89]
    s, p = Port.compress(np.array([1, np.nan, -3], np.float32))
    assert p.tolist() == [0, 2, 255, 1]
    s, p = Port.compress(np.array([1, np.nan, -3, np.inf], np.float32))
    assert np.isinf(s) and p.tolist() == [0, 4]


def test_bulk_digest(golden):
    m = golden["meta"]["bulk"]["splitmix42_131072"]
    x = splitmix64_block(42, 131072)
    assert "%016x" % Port.fnv1a64(x.astype(np.float16)) == m["in_f16_fnv1a64"]
    s, p = Port.compress(x)
    assert int(f32_bits([s])[0]) == m["scale_bits"] and p.size == m["comp_bytes"]
    assert "%016x" % Port.fnv1a64(p) == m["payload_fnv1a64"]
    y = Port.decompress(s, p, x.size)
    assert "%016x" % Port.fnv1a64(y) == m["out_f32_fnv1a64"]
    assert "%016x" % Port.fnv1a64(y.astype(np.float16)) == m["out_f16_fnv1a64"]


def test_decode_edge_cases():
    # trailing odd byte ignored, zero-count pair emits nothing (cache_engine.cpp:241-258)
    y = Port.decompress(1.0, np.array([5, 2, 7, 0, 1, 3, 9], np.uint8), 64)
    q = np.round(y * 127).astype(np.int64)
    assert q.tolist() == [5, 10, 11, 12, 13]
    assert Port.decompress(1.0, np.array([], np.uint8), 8).size == 0
    assert Port.decompress(1.0, np.array([3], np.uint8), 8).size == 0
    # empty input compresses to nothing with scale 1
    s, p = Port.compress(np.zeros(0, np.float32))
    assert s == 1.0 and p.size == 0


def test_batch_forms_match_single():
    rng = np.random.default_rng(3)
    x = rng.standard_normal(8 * 512).astype(np.float16)
    x[512:1024] = 0.25
    payload, scales, comp = Port.compress_batch(x, 512, threads=3)
    for g in range(8):
        s, p = Port.compress(x[g * 512:(g + 1) * 512].astype(np.float32))
        assert f32_bits([s])[0] == f32_bits([scales[g]])[0]
        assert comp[g] == p.size and np.array_equal(payload[g, :p.size], p)
    out, n = Port.decompress_batch(payload, scales, comp, 512, F16, threads=2)
    assert (n == 512).all()
    for g in range(8):
        y = Port.decompress(scales[g], payload[g, :comp[g]], 512)
        with np.errstate(over="ignore"):
            assert np.array_equal(out[g].view(np.uint16), y.astype(np.float16).view(np.uint16))
    # bf16 boundary
    xb = bf16_from_f32(rng.standard_normal(4 * 256))
    payload, scales, comp = Port.compress_batch(xb, 256, dtype=BF16)
    s, p = Port.compress(bf16_to_f32(xb[:256]))
    assert comp[0] == p.size and np.array_equal(payload[0, :p.size], p)


def test_translate_fixtures(golden):
    tr, meta = golden["translate"], golden["meta"]["translate"]
    va = tr["va"]
    assert np.array_equal(Port.translate(va), tr["engine_pa"])
    L = Port.lib()
    assert all(L.oracle_translate(int(v)) == int(p) for v, p in zip(va, tr["engine_pa"]))
    pa, hits, misses = Port.atu_sequence(va)
    assert np.array_equal(pa, tr["atu_pa"])
    assert (hits, misses) == (meta["atu_hits"], meta["atu_misses"])
    # SURVEY.md section 8a A10 measured values (engine model)
    assert L.oracle_translate(0x100000123) == 0x4100000123
    assert L.oracle_translate(0xFFFF000000000ABC) == 0x4000000ABC


def test_capi_address_fixtures(golden):
    for handle, size, off, rc, ptr in golden["meta"]["capi"]["accesses"]:
        a = Port.access_addr(handle, size, off)
        if rc == 0:
            assert a == ptr, (handle, size, off)
        else:
            assert a == 0
    # SURVEY.md section 8b measured: h=1,off=100 -> 0x4000100064; h=2,off=8191 -> 0x4000201fff
    assert Port.access_addr(1, 1 << 20, 100) == 0x4000100064
    assert Port.access_addr(2, 1 << 20, 8191) == 0x4000201FFF
    assert Port.access_addr(3, 5000, 4096) == 0x4000301000 and Port.access_addr(3, 5000, 8192) == 0


def same_topk(ids_a, ids_b, conf_bits):
    """std::sort (lstm_predictor.cpp:83-84) is unstable: ids may permute inside a tie."""
    groups_a, groups_b = {}, {}
    for i, c in enumerate(conf_bits):
        groups_a.setdefault(c, set()).add(ids_a[i])
        groups_b.setdefault(c, set()).add(ids_b[i])
    last = conf_bits[-1]  # a tie straddling the k-th place may pick different members
    return all(groups_a[c] == groups_b[c] for c in groups_a if c != last) and \
        len(groups_a[last]) == len(groups_b[last])


def test_lstm_fixtures(golden):
    m = golden["meta"]["lstm"]
    emb, wout = Port.lstm_weights(m["seed"])
    assert "%016x" % Port.fnv1a64(emb) == m["emb_fnv1a64"]
    assert "%016x" % Port.fnv1a64(wout) == m["wout_fnv1a64"]
    for pr in m["predictions"]:
        ids, conf, _ = Port.lstm_predict(emb, wout, np.array(pr["hist"], np.uint32), k=len(pr["ids"]))
        assert f32_bits(conf).tolist() == pr["conf_bits"]
        assert same_topk(ids.tolist(), pr["ids"], pr["conf_bits"]), pr["hist"]
    pf = m["prefetch"]
    L = Port.lib()
    assert [L.oracle_kv_address(0, pf["layer"], i + 1) for i in range(pf["depth"])] == pf["va"]


def test_port_vs_reference_random(reference_traces):
    """The restatement on random inputs against the answers recorded in tests/golden/reference_traces.json (its
    "source" names the reference or the restatement) and, where oracle/_ref is built, against the reference itself."""
    from oracle.oracle import random_codec_cases
    want = reference_traces["codec_random"]
    inputs, payloads = random_codec_cases()
    assert len(inputs) == len(want["compress"]) and len(payloads) == len(want["decompress"])
    for x, w in zip(inputs, want["compress"]):
        s1, p1 = Port.compress(x)
        y1 = Port.decompress(s1, p1, x.size)
        assert [int(f32_bits([s1])[0]), int(p1.size), "%016x" % Port.fnv1a64(p1),
                "%016x" % Port.fnv1a64(f32_bits(y1))] == w, x.size
        if Ref.available():
            s2, p2 = Ref.compress(x)
            assert f32_bits([s1])[0] == f32_bits([s2])[0] and np.array_equal(p1, p2)
            assert np.array_equal(f32_bits(y1), f32_bits(Ref.decompress(s2, p2, x.size)))
    # arbitrary (not produced by compress) payloads through the decoder
    for (s, p), w in zip(payloads, want["decompress"]):
        a = Port.decompress(s, p, 200000)
        assert [int(a.size), "%016x" % Port.fnv1a64(f32_bits(a))] == w, p.size
        if Ref.available():
            assert np.array_equal(f32_bits(a), f32_bits(Ref.decompress(s, p, 200000)))


def test_division_identities_quick():
    """oracle/verify_fastdiv: the FMA-residual quantiser, the q/127 identities and the rounding
    trick used by the CUDA kernels equal the reference arithmetic (every 16th fp16/bf16 max value
    here; the full exhaustive run is `./oracle/verify_fastdiv`, ~15 s on 8 cores)."""
    import os
    import subprocess

    here = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle")
    subprocess.check_call(["make", "-s", "-C", here, "verify"])
    out = subprocess.run([os.path.join(here, "verify_fastdiv"), "quick"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip().endswith("OK"), out.stdout


def test_policy_port_matches_reference_manager(reference_traces):
    """oracle_policy_* against the reference's CXLMemoryManager on random traces that never fill L1 (its eviction
    path deadlocks): per-call results, final tiers, LRU order, stats -- against the answers recorded in
    tests/golden/reference_traces.json (its "source" names the reference or the restatement) and, where oracle/_ref
    is built, against the reference itself."""
    import json
    from oracle.oracle import random_policy_trace, run_policy_trace
    assert len(reference_traces["policy"]) == 4
    for want in reference_traces["policy"]:
        ops, n = random_policy_trace(want["seed"])
        assert (n, len(ops)) == (want["n_pages"], want["n_ops"])
        a = json.loads(json.dumps(run_policy_trace(ops, n, impl="port")))     # tuples -> lists, as stored
        refs = [want] + ([json.loads(json.dumps(run_policy_trace(ops, n, impl="ref")))] if Ref.available() else [])
        for b in refs:
            assert a["results"] == b["results"]
            assert a["tiers"] == b["tiers"]
            assert a["lru"] == b["lru"]
            assert a["stats"] == b["stats"]


def test_policy_port_eviction_semantics():
    """The defined eviction (the reference's evict_l1_lru step repeated until it frees a page)."""
    from oracle.oracle import run_policy_trace
    ops = [("place", g, 2) for g in range(6)] + [("place", 6, 1)]
    ops += [("touch", 5), ("touch", 6)]                    # non-L1 entries at the front of the LRU list
    ops += [("promote", 0), ("promote", 1)]                # L1 (capacity 2) now holds 0, 1; LRU: 5 6 0 1
    ops += [("promote", 2)]                                # full: pops 5, 6 (dropped), then evicts 0
    ops += [("touch", 1), ("promote", 3)]                  # LRU: 2 1 -> evicts 2
    r = run_policy_trace(ops, 7, caps=(2, 1 << 40, 1 << 40), impl="port")
    assert r["results"][-3:] == [(1, 0), 0, (1, 2)]
    assert r["tiers"] == [2, 0, 2, 0, 2, 2, 1]
    assert r["lru"] == [1, 3]
    assert r["stats"]["migrations_l1_to_l3"] == 2 and r["stats"]["migrations_l3_to_l1"] == 4


# ---- the extension schemes (NOT reference behaviour; see oracle/speckv_oracle.c) ------------------------------
def test_clamped_scheme_restatement_known_answers():
    """Schemes 3 / 4: s = max|x|, q = clamp(round_half_away((x / s) * 127)), y = (q / 127) * s -- pinned against a
    hand-computed vector and an independent numpy formulation; scheme 1 = the reference's codes alone."""
    from oracle.oracle import Port
    x = np.array([0, 1, -1, 0.5, 0.25, 0.25, 0.25, 2, -2, 1e-3], dtype=np.float32)
    p, s, c = Port.compress_batch(x, x.size, threads=1, scheme=4)
    assert s[0] == np.float32(2.0) and c[0] == x.size
    assert p[0, :x.size].view(np.int8).tolist() == [0, 64, -64, 32, 16, 16, 16, 127, -127, 0]
    p3, s3, c3 = Port.compress_batch(x, x.size, threads=1, scheme=3)
    # deltas 0 64 -128 96 -16 0 0 111 2 127 -> pairs (value, count)
    want = [(0, 1), (64, 1), (-128, 1), (96, 1), (-16, 1), (0, 2), (111, 1), (2, 1), (127, 1)]
    assert c3[0] == 2 * len(want)
    got = p3[0, :c3[0]].reshape(-1, 2)
    assert [(int(np.int8(v)), int(n)) for v, n in got] == want
    y, n = Port.decompress_batch(p3, s3, c3, x.size, 2, threads=1, scheme=3)
    assert n[0] == x.size
    q = np.array([0, 64, -64, 32, 16, 16, 16, 127, -127, 0], dtype=np.float32)
    assert np.array_equal(y[0], (q / np.float32(127.0)) * np.float32(2.0))
    # independent numpy formulation on random fp16 groups (incl. zero group and NaN)
    rng = np.random.default_rng(12)
    G = 4096
    xs = rng.standard_normal(6 * G).astype(np.float16).reshape(6, G)
    xs[1] = 0
    xs[2, 9] = np.nan
    pc, sc, cc = Port.compress_batch(xs.reshape(-1), G, threads=2, scheme=4)
    for g in range(6):
        xf = xs[g].astype(np.float32)
        m = np.nanmax(np.abs(xf)) if np.isfinite(np.nanmax(np.abs(xf))) else np.inf
        sg = np.float32(m) if m > 0 else np.float32(1.0)
        t = (xf / sg) * np.float32(127.0)
        r = np.sign(t) * np.floor(np.abs(t) + np.float32(0.5))
        r = np.where(np.isnan(r), 0, np.clip(r, -128, 127)).astype(np.int8)
        assert sc[g] == sg and np.array_equal(pc[g, :G].view(np.int8), r), g
    # scheme 1 == the reference's quantiser alone: the codes whose deltas scheme 2 encodes
    p1, s1, c1 = Port.compress_batch(xs.reshape(-1), G, threads=2, scheme=1)
    p2, s2, c2 = Port.compress_batch(xs.reshape(-1), G, threads=2, scheme=2)
    y1, _ = Port.decompress_batch(p1, s1, c1, G, 0, threads=2, scheme=1)
    y2, _ = Port.decompress_batch(p2, s2, c2, G, 0, threads=2, scheme=2)
    assert np.array_equal(s1.view(np.uint32), s2.view(np.uint32)) and np.array_equal(y1.view(np.uint16), y2.view(np.uint16))
