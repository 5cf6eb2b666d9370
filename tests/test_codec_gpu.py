"""GPU parity tests: the CUDA codec (through the C ABI of libcxlspeckv.so) against
the fixtures recorded from the reference's C++ model and against the CPU oracle on
the same seeded inputs.  Bar: compressed bytes, scales, int8 codes, byte counts and
translated addresses bit-exact; decompressed fp32 bit-exact; fp16/bf16 outputs
within 1 ulp of the oracle's fp32 value rounded to the type (in practice equal)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.oracle import Port, splitmix64_block
from tests.helpers import F16, BF16, F32, bf16_from_f32, bf16_to_f32, case_input, f32_bits, narrow

pytestmark = pytest.mark.gpu

from cxl_speckv_b200 import codec  # noqa: E402
from cxl_speckv_b200 import COMP_FP16, COMP_INT8, COMP_INT8_DELTA_RLE  # noqa: E402

DEV = "cuda:0"
TORCH_DT = {F16: torch.float16, BF16: torch.bfloat16, F32: torch.float32}


def to_dev(raw, dtype):
    if dtype == BF16:
        return torch.from_numpy(raw.astype(np.int16)).to(DEV).view(torch.bfloat16)
    return torch.from_numpy(np.ascontiguousarray(raw)).to(DEV)


def out_bits(t):
    if t.dtype == torch.float32:
        return t.cpu().numpy().view(np.uint32)
    return t.view(torch.int16).cpu().numpy().view(np.uint16)


def ulp_diff16(a_bits, b_bits):
    """distance in representable values between two fp16/bf16 bit patterns (sign-magnitude order)"""
    def key(u):
        u = u.astype(np.int32)
        return np.where(u & 0x8000, -(u & 0x7FFF), u & 0x7FFF)
    return np.abs(key(a_bits) - key(b_bits))


def check_group_against_oracle(c, g, xf):
    s, p = Port.compress(xf)
    assert f32_bits(c.scales[g:g + 1].cpu().numpy())[0] == f32_bits([s])[0]
    nb = int(c.comp_bytes[g].item()) & 0xFFFFFFFF
    assert nb == p.size
    assert np.array_equal(c.payload[g, :nb].cpu().numpy(), p)
    return s, p


def test_golden_fixtures_rle(golden):
    meta, cz = golden["meta"], golden["codec"]
    for name, m in meta["codec"].items():
        raw, xf, dtype = case_input(cz, meta, name)
        x = to_dev(raw, dtype)
        c = codec.compress(x, m["n"])
        torch.cuda.synchronize()
        assert f32_bits(c.scales.cpu().numpy())[0] == m["scale_bits"], name
        nb = int(c.comp_bytes[0].item())
        assert nb == m["comp_bytes"], name
        assert np.array_equal(c.payload[0, :nb].cpu().numpy(), cz[name + ".payload"]), name
        # fp32 output: bit-exact against the reference's decompress()
        oel = torch.zeros(1, dtype=torch.int32, device=DEV)
        y32 = codec.decompress(c, dtype=torch.float32, out_elems=oel)
        assert int(oel.item()) == m["out_elems"], name
        assert np.array_equal(out_bits(y32)[0, :m["out_elems"]], cz[name + ".out_f32_bits"]), name
        # native dtype: reference fp32 rounded to the type, tolerance 1 ulp (north_star)
        if dtype != F32:
            y = codec.decompress(c)
            want = narrow(cz[name + ".out_f32_bits"].view(np.float32), dtype)
            got = out_bits(y)[0]
            finite = ~np.isnan(cz[name + ".out_f32_bits"].view(np.float32))
            assert (ulp_diff16(got[finite], want[finite]) <= 1).all(), name
            assert np.array_equal(got[finite], want[finite]), name   # in practice exact


def test_golden_fixtures_int8_codes(golden):
    meta, cz = golden["meta"], golden["codec"]
    for name, m in meta["codec"].items():
        raw, xf, dtype = case_input(cz, meta, name)
        c = codec.compress(to_dev(raw, dtype), m["n"], scheme=COMP_INT8)
        assert f32_bits(c.scales.cpu().numpy())[0] == m["scale_bits"], name
        assert int(c.comp_bytes[0].item()) == m["n"]
        assert np.array_equal(c.payload[0, :m["n"]].cpu().numpy().view(np.int8), cz[name + ".codes"]), name
        y = codec.decompress(c, dtype=torch.float32)
        want = (cz[name + ".codes"].astype(np.float32) / np.float32(127.0)) * np.uint32(m["scale_bits"]).view(np.float32)
        assert np.array_equal(out_bits(y)[0], f32_bits(want)), name


def test_bulk_group_digest(golden):
    m = golden["meta"]["bulk"]["splitmix42_131072"]
    x = splitmix64_block(42, 131072)          # fp32: values in [2,4) are not all fp16-representable
    c = codec.compress(torch.from_numpy(x).to(DEV), 131072)
    assert f32_bits(c.scales.cpu().numpy())[0] == m["scale_bits"]
    nb = int(c.comp_bytes[0].item())
    assert nb == m["comp_bytes"]
    assert "%016x" % Port.fnv1a64(c.payload[0, :nb].cpu().numpy()) == m["payload_fnv1a64"]
    y32 = codec.decompress(c, dtype=torch.float32)
    assert "%016x" % Port.fnv1a64(y32.cpu().numpy()) == m["out_f32_fnv1a64"]
    y16 = codec.decompress(c, dtype=torch.float16)
    assert "%016x" % Port.fnv1a64(y16.cpu().numpy()) == m["out_f16_fnv1a64"]


def make_inputs(rng, n_groups, G, kind):
    n = n_groups * G
    if kind == "randn":
        x = rng.standard_normal(n).astype(np.float16)
    elif kind == "runs":
        x = np.repeat(rng.standard_normal(n // 300 + 1), 300)[:n].astype(np.float16)
    elif kind == "zeros":
        x = np.zeros(n, np.float16)
    elif kind == "mixed":
        x = rng.standard_normal(n).astype(np.float16)
        for _ in range(max(1, n // 5000)):
            a = int(rng.integers(0, n))
            b = min(n, a + int(rng.integers(1, 1500)))
            x[a:b] = x[a]
        x[rng.integers(0, n, max(1, n // 4000))] = np.nan
    elif kind == "ramp":
        x = ((np.arange(n) % 251) / 16.0).astype(np.float16)
    else:
        raise ValueError(kind)
    return x


@pytest.mark.parametrize("G,n_groups", [(2048, 96), (131072, 5), (1000, 37), (4099, 11), (8, 300), (1, 17),
                                        (65536, 3), (16384, 9), (32768, 4), (262144, 2), (131080, 2)])
@pytest.mark.parametrize("kind", ["randn", "mixed", "runs", "zeros", "ramp"])
def test_batches_vs_oracle_f16(G, n_groups, kind):
    rng = np.random.default_rng(hash((G, n_groups, kind)) % (2**32))
    x = make_inputs(rng, n_groups, G, kind)
    xd = torch.from_numpy(x).to(DEV)
    c = codec.compress(xd, G)
    payload, scales, comp = Port.compress_batch(x, G, threads=8)
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(scales))
    got_comp = c.comp_bytes.cpu().numpy().view(np.uint32)
    assert np.array_equal(got_comp, comp)
    gp = c.payload.cpu().numpy()
    for g in range(n_groups):
        assert np.array_equal(gp[g, :comp[g]], payload[g, :comp[g]]), (g, comp[g])
    oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
    y = codec.decompress(c, out_elems=oel)
    want, want_n = Port.decompress_batch(payload, scales, comp, G, F16, threads=8)
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n) and (want_n == G).all()
    assert np.array_equal(out_bits(y), want.view(np.uint16))
    # INT8 scheme on the same data
    c8 = codec.compress(xd, G, scheme=COMP_INT8)
    g0 = int(rng.integers(0, n_groups))
    q = Port.quantize(x[g0 * G:(g0 + 1) * G].astype(np.float32), scales[g0])
    assert np.array_equal(c8.payload[g0, :G].cpu().numpy().view(np.int8), q)


@pytest.mark.parametrize("G,n_groups", [(2048, 40), (131072, 3), (777, 9)])
def test_batches_vs_oracle_bf16_f32(G, n_groups):
    rng = np.random.default_rng(G)
    # bf16, including groups whose max is below 2^-60 (exact-division path) and huge values
    mags = np.exp(rng.uniform(-75, 60, n_groups)).repeat(G)
    xb = bf16_from_f32(rng.standard_normal(n_groups * G) * mags)
    xd = torch.from_numpy(xb.astype(np.int16)).to(DEV).view(torch.bfloat16)
    c = codec.compress(xd, G)
    payload, scales, comp = Port.compress_batch(xb, G, dtype=BF16, threads=8)
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(scales))
    assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp)
    gp = c.payload.cpu().numpy()
    for g in range(n_groups):
        assert np.array_equal(gp[g, :comp[g]], payload[g, :comp[g]]), g
    y = codec.decompress(c)
    want, _ = Port.decompress_batch(payload, scales, comp, G, BF16, threads=8)
    assert np.array_equal(out_bits(y), want)
    # fp32 in / fp32 out: what the reference engine itself consumes and produces
    xf = (rng.standard_normal(n_groups * G) * np.exp(rng.uniform(-20, 20, n_groups * G))).astype(np.float32)
    c = codec.compress(torch.from_numpy(xf).to(DEV), G)
    payload, scales, comp = Port.compress_batch(xf, G, threads=8)
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(scales))
    assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp)
    gp = c.payload.cpu().numpy()
    for g in range(n_groups):
        assert np.array_equal(gp[g, :comp[g]], payload[g, :comp[g]]), g
    y = codec.decompress(c)
    want, _ = Port.decompress_batch(payload, scales, comp, G, F32, threads=8)
    assert np.array_equal(out_bits(y), f32_bits(want))


def test_unaligned_input_pointer():
    rng = np.random.default_rng(5)
    G, n_groups = 2048, 6
    x = rng.standard_normal(n_groups * G + 3).astype(np.float16)
    xd = torch.from_numpy(x).to(DEV)[3:]          # 6-byte offset: no 128-bit loads possible
    c = codec.compress(xd, G)
    payload, scales, comp = Port.compress_batch(x[3:], G)
    assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp)
    for g in range(n_groups):
        assert np.array_equal(c.payload[g, :comp[g]].cpu().numpy(), payload[g, :comp[g]])
    buf = torch.zeros(n_groups * G + 1, dtype=torch.float16, device=DEV)
    y = codec.decompress(c, out=buf[1:].view(n_groups, G))
    want, _ = Port.decompress_batch(payload, scales, comp, G, F16)
    assert np.array_equal(out_bits(y), want.view(np.uint16))


def test_decode_arbitrary_payloads():
    """payloads the encoder never produces: zero counts, odd trailing byte, overlong output."""
    rng = np.random.default_rng(9)
    G, n_groups = 3000, 24
    sb = codec.slot_bytes(G)
    payload = np.zeros((n_groups, sb), np.uint8)
    comp = np.zeros(n_groups, np.uint32)
    scales = rng.uniform(0.01, 2.0, n_groups).astype(np.float32)
    for g in range(n_groups):
        nbytes = int(rng.integers(0, 700))
        p = rng.integers(0, 256, nbytes, dtype=np.uint8)
        if g % 3 == 0:
            p[1::2] = rng.integers(0, 3, p[1::2].size)       # many zero counts, short output
        if g % 3 == 1:
            p[1::2] = 255                                    # overlong: clipped at G
        payload[g, :nbytes] = p
        comp[g] = nbytes
    c = codec.CompressedKV(torch.from_numpy(payload).to(DEV), torch.from_numpy(scales).to(DEV),
                           torch.from_numpy(comp.view(np.int32)).to(DEV), G, torch.float32, COMP_INT8_DELTA_RLE)
    out = torch.full((n_groups, G), -7.0, dtype=torch.float32, device=DEV)
    oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
    codec.decompress(c, out=out, out_elems=oel)
    got, got_n = out.cpu().numpy(), oel.cpu().numpy()
    for g in range(n_groups):
        want = Port.decompress(scales[g], payload[g, :comp[g]], G)
        assert got_n[g] == want.size, g
        assert np.array_equal(f32_bits(got[g, :want.size]), f32_bits(want)), g
        assert (got[g, want.size:] == -7.0).all()            # nothing written past the decoded length


def test_fp16_passthrough_scheme():
    x = torch.randn(8 * 2048, device=DEV).half()
    c = codec.compress(x, 2048, scheme=COMP_FP16)
    assert (c.comp_bytes == 4096).all() and (c.scales == 1).all()
    y = codec.decompress(c)
    assert torch.equal(y.view(-1), x)


def test_translate(golden):
    tr = golden["translate"]
    va = torch.from_numpy(tr["va"].view(np.int64)).to(DEV)
    pa = codec.translate(va)
    assert np.array_equal(pa.cpu().numpy().view(np.uint64), tr["engine_pa"])
    rng = np.random.default_rng(1)
    big = rng.integers(0, 2**63, 1_000_003, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    pa = codec.translate(torch.from_numpy(big.view(np.int64)).to(DEV))
    assert np.array_equal(pa.cpu().numpy().view(np.uint64), Port.translate(big))
    pa = codec.translate(torch.from_numpy(big.view(np.int64)).to(DEV)[1:])      # 8-byte aligned only
    assert np.array_equal(pa.cpu().numpy().view(np.uint64), Port.translate(big[1:]))


def test_host_buffer_api_matches_device_api():
    from cxl_speckv_b200 import lib
    L = lib()
    rng = np.random.default_rng(2)
    G, n_groups = 131072, 300                 # 75 MiB: several pipeline chunks
    x = rng.standard_normal(n_groups * G).astype(np.float16)
    x[5 * G:6 * G] = 0
    sb = codec.slot_bytes(G)
    payload = np.zeros((n_groups, sb), np.uint8)
    scales = np.zeros(n_groups, np.float32)
    comp = np.zeros(n_groups, np.uint32)
    st = L.speckv_ext_compress_host(x.ctypes.data, 0, G, n_groups, payload.ctypes.data, sb, scales.ctypes.data,
                                    comp.ctypes.data, 2)
    assert st == 0
    c = codec.compress(torch.from_numpy(x).to(DEV), G)
    assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp)
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(scales))
    gp = c.payload.cpu().numpy()
    for g in range(0, n_groups, 17):
        assert np.array_equal(gp[g, :comp[g]], payload[g, :comp[g]])
    out = np.zeros((n_groups, G), np.float16)
    oel = np.zeros(n_groups, np.uint32)
    st = L.speckv_ext_decompress_host(payload.ctypes.data, sb, scales.ctypes.data, comp.ctypes.data, G, n_groups, 0,
                                      out.ctypes.data, oel.ctypes.data, 2)
    assert st == 0 and (oel == G).all()
    y = codec.decompress(c)
    assert np.array_equal(out.view(np.uint16), out_bits(y))
    for g in (0, 5, 299):
        want = Port.decompress(scales[g], payload[g, :comp[g]], G)
        assert np.array_equal(out[g].view(np.uint16), want.astype(np.float16).view(np.uint16))


def test_bad_arguments_are_rejected():
    from cxl_speckv_b200 import SpeckvError
    x = torch.randn(4096, device=DEV).half()
    with pytest.raises(ValueError):
        codec.compress(x, 1000)
    c = codec.compress(x, 2048)
    bad = codec.CompressedKV(c.payload[:, :4080].contiguous(), c.scales, c.comp_bytes, 2048, c.dtype, c.scheme)
    with pytest.raises(SpeckvError):
        codec.decompress(bad)                  # slot smaller than the worst case
    # the C entry points: each rejected argument on its own, and an empty call, which checks no buffer
    import cxl_speckv_b200 as pkg
    L = pkg.lib()
    sb, o = c.payload.shape[1], torch.empty_like(x)
    idx = torch.zeros(2, dtype=torch.int32, device=DEV)
    cnt = torch.full((1,), 2, dtype=torch.int32, device=DEV)
    buf = dict(p=c.payload.data_ptr(), sb=sb, s=c.scales.data_ptr(), cb=c.comp_bytes.data_ptr(), dt=0, G=2048, n=2,
               scheme=2, x=x.data_ptr(), o=o.data_ptr(), idx=idx.data_ptr(), cnt=cnt.data_ptr())
    calls = {
        "compress": lambda a: L.speckv_ext_compress(a["x"], a["dt"], a["G"], a["n"], a["p"], a["sb"], a["s"], a["cb"],
                                                    a["scheme"], None),
        "decompress": lambda a: L.speckv_ext_decompress(a["p"], a["sb"], a["s"], a["cb"], a["G"], a["n"], a["dt"], a["o"],
                                                        None, a["scheme"], None),
        "indexed": lambda a: L.speckv_ext_decompress_indexed(a["p"], a["sb"], a["s"], a["cb"], a["idx"], a["n"], a["G"],
                                                             a["dt"], a["o"], None, a["scheme"], None),
        "routed": lambda a: L.speckv_ext_decompress_routed(a["p"], a["sb"], a["s"], a["cb"], a["idx"], a["cnt"], a["n"],
                                                           a["G"], a["dt"], a["o"], None, a["scheme"], None),
    }
    common = [dict(dt=3), dict(dt=-1), dict(scheme=5), dict(scheme=-1), dict(dt=2, scheme=0), dict(sb=sb - 8),
              dict(sb=sb - 16), dict(sb=1 << 32), dict(G=1 << 31), dict(n=1 << 32), dict(p=None), dict(s=None),
              dict(cb=None), dict(p=c.payload.data_ptr() + 8)]
    own = {"compress": [dict(x=None)], "decompress": [dict(o=None)], "indexed": [dict(o=None), dict(idx=None)],
           "routed": [dict(o=None), dict(idx=None), dict(cnt=None)]}
    for name, call in calls.items():
        for bad_arg in common + own[name]:
            assert call({**buf, **bad_arg}) == pkg.SPECKV_ERR_INVAL, (name, bad_arg)
        assert call({**buf, "n": 0, "p": None, "s": None, "cb": None, "x": None, "o": None, "idx": None,
                     "cnt": None}) == pkg.SPECKV_OK, name
        assert call({**buf, "n": 0, "dt": 3}) == pkg.SPECKV_ERR_INVAL, name


def test_full_size_properties_llama70b_layer():
    """BASELINE config 3 geometry at full per-layer size (8 KV heads x 8192 tokens x 128,
    K and V: 128 groups of 1024x128), several layers at once: size-independent properties +
    oracle spot checks."""
    torch.manual_seed(1234)
    G, layers = 131072, 8
    n_groups = layers * 2 * 8 * 8
    x = torch.randn(n_groups * G, device=DEV, dtype=torch.float32).half()
    c = codec.compress(x, G)
    comp = c.comp_bytes.cpu().numpy().view(np.uint32)
    assert (comp % 2 == 0).all() and (comp <= 2 * G).all() and (comp > 1.9 * G).all()
    # scale == max|x| / 127 in IEEE fp32 for every group
    amax = x.view(n_groups, G).float().abs().amax(dim=1).cpu().numpy()
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(amax / np.float32(127.0)))  # IEEE divide on the host
    # every pair count >= 1 and counts sum to G (decoder length) for every group
    oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
    y = codec.decompress(c, out_elems=oel)
    assert (oel == G).all()
    # decode is the inverse of delta+RLE: re-encoding the INT8 codes path agrees with it
    c8 = codec.compress(x, G, scheme=COMP_INT8)
    y8 = codec.decompress(c8)
    assert torch.equal(y8.view(torch.int16), y.view(torch.int16))
    # reconstruction error equals the reference's (SURVEY.md fact 1: ~0.996 MSE for N(0,1))
    mse = ((y.float() - x.view(n_groups, G).float()) ** 2).mean().item()
    assert 0.9 < mse < 1.1
    xs = x.view(n_groups, G)
    for g in (0, 1, n_groups // 2, n_groups - 1):
        s, p = check_group_against_oracle(c, g, xs[g].cpu().numpy().astype(np.float32))
        want = Port.decompress(s, p, G).astype(np.float16)
        assert np.array_equal(out_bits(y[g]), want.view(np.uint16))


def test_page_table_lookup_on_device(golden):
    """speckv_ext_page_table_export + speckv_ext_page_lookup against the reference's recorded
    speckv_access results (tests/golden, host C API with /dev/null) and the oracle formulas."""
    import cxl_speckv_b200 as pkg
    L = pkg.lib()
    assert L.speckv_init(b"cuda:0") == 0
    try:
        sizes = (1 << 20, 1 << 20, 5000, 3 << 20, 1)
        handles = []
        for sz in sizes:
            h = C.c_uint64()
            assert L.speckv_alloc(sz, None, C.byref(h)) == 0
            handles.append(h.value)
        assert handles == [1, 2, 3, 4, 5]
        ptr = C.c_void_p()
        assert L.speckv_access(4, 8192 + 5, 4, C.byref(ptr)) == 0           # marks page 2 of handle 4 as L2
        for h, sz in zip(handles, sizes):
            npages = (sz + 4095) // 4096
            pages = torch.zeros(npages * 3, dtype=torch.int64, device=DEV)   # 24-byte records
            cnt = C.c_size_t()
            assert L.speckv_ext_page_table_export(h, pages.data_ptr(), npages, C.byref(cnt), None) == 0
            assert cnt.value == npages
            rec = pages.cpu().numpy().view(np.uint64).reshape(npages, 3)
            assert all(int(rec[i, 0]) == Port.lib().oracle_virt_page_id(h, i) for i in range(npages))
            assert all(int(rec[i, 1]) == Port.lib().oracle_phys_page_id(h, i) for i in range(npages))
            offs = np.array([a[2] for a in golden["meta"]["capi"]["accesses"] if a[0] == h], dtype=np.uint64)
            rng = np.random.default_rng(h)
            offs = np.concatenate([offs, rng.integers(0, npages * 4096 + 9000, 5000, dtype=np.uint64)])
            va = torch.from_numpy(((np.uint64(h) << np.uint64(32)) + offs).view(np.int64)).to(DEV)
            pa = torch.empty_like(va)
            fl = torch.empty(va.numel(), dtype=torch.int32, device=DEV)
            st = L.speckv_ext_page_lookup(pages.data_ptr(), npages, h << 32, va.data_ptr(), pa.data_ptr(), fl.data_ptr(),
                                          va.numel(), None)
            assert st == 0
            want = np.array([Port.access_addr(h, sz, int(o)) for o in offs], dtype=np.uint64)
            assert np.array_equal(pa.cpu().numpy().view(np.uint64), want)
            flags = fl.cpu().numpy()
            if h == 4:
                assert (flags[(offs >= 8192) & (offs < 12288)] == 2).all() and (flags[offs < 8192] == 0).all()
            else:
                assert (flags == 0).all()
        # golden: every recorded (handle, offset) -> address / failure
        for h, sz, off, rc, addr in golden["meta"]["capi"]["accesses"]:
            assert Port.access_addr(h, sz, off) == (addr if rc == 0 else 0)
    finally:
        L.speckv_finalize()


def test_stateful_atu_matches_reference_sequence(golden):
    """AddressTranslationUnit with its TLB state: per-address results (offset counted twice on a
    miss), hit/miss counters and invalidation, against the reference's recorded sequence and the
    oracle's model on a longer random sequence."""
    import cxl_speckv_b200 as pkg
    L = pkg.lib()
    tr, meta = golden["translate"], golden["meta"]["translate"]
    atu = C.c_void_p()
    assert L.speckv_ext_atu_create(1024, C.byref(atu)) == 0
    try:
        va = torch.from_numpy(tr["va"].view(np.int64)).to(DEV)
        pa = torch.empty_like(va)
        assert L.speckv_ext_atu_translate(atu, va.data_ptr(), pa.data_ptr(), va.numel(), None) == 0
        assert np.array_equal(pa.cpu().numpy().view(np.uint64), tr["atu_pa"])
        h, m = C.c_uint64(), C.c_uint64()
        assert L.speckv_ext_atu_get_stats(atu, C.byref(h), C.byref(m), 1) == 0
        assert (h.value, m.value) == (meta["atu_hits"], meta["atu_misses"])
        # longer sequence with reuse, continuing from the TLB state left by the first batch
        rng = np.random.default_rng(3)
        seq = (np.uint64(0x100000000) + rng.integers(0, 3000, 20000, dtype=np.uint64) * np.uint64(4096)
               + rng.integers(0, 4096, 20000, dtype=np.uint64))
        Lp = Port.lib()
        ref = Lp.oracle_atu_new(1024)
        ref = C.c_void_p(ref)
        for v in tr["va"]:
            Lp.oracle_atu_translate(ref, int(v))
        want = np.array([Lp.oracle_atu_translate(ref, int(v)) for v in seq], dtype=np.uint64)
        va2 = torch.from_numpy(seq.view(np.int64)).to(DEV)
        pa2 = torch.empty_like(va2)
        assert L.speckv_ext_atu_translate(atu, va2.data_ptr(), pa2.data_ptr(), va2.numel(), None) == 0
        assert np.array_equal(pa2.cpu().numpy().view(np.uint64), want)
        # invalidate one page, then everything
        Lp.oracle_atu_invalidate(ref, int(seq[-1]))
        assert L.speckv_ext_atu_invalidate(atu, int(seq[-1]), 0, None) == 0
        probe = np.array([seq[-1], seq[-2], seq[-1]], dtype=np.uint64)
        want = np.array([Lp.oracle_atu_translate(ref, int(v)) for v in probe], dtype=np.uint64)
        vp_ = torch.from_numpy(probe.view(np.int64)).to(DEV); pp_ = torch.empty_like(vp_)
        assert L.speckv_ext_atu_translate(atu, vp_.data_ptr(), pp_.data_ptr(), 3, None) == 0
        assert np.array_equal(pp_.cpu().numpy().view(np.uint64), want)
        Lp.oracle_atu_invalidate_all(ref)
        assert L.speckv_ext_atu_invalidate(atu, 0, 1, None) == 0
        want = np.array([Lp.oracle_atu_translate(ref, int(v)) for v in probe], dtype=np.uint64)
        assert L.speckv_ext_atu_translate(atu, vp_.data_ptr(), pp_.data_ptr(), 3, None) == 0
        assert np.array_equal(pp_.cpu().numpy().view(np.uint64), want)
        hh, mm = C.c_uint64(), C.c_uint64()
        Lp.oracle_atu_stats(ref, C.byref(hh), C.byref(mm))
        assert L.speckv_ext_atu_get_stats(atu, C.byref(h), C.byref(m), 0) == 0
        assert h.value + meta["atu_hits"] == hh.value and m.value + meta["atu_misses"] == mm.value
        Lp.oracle_atu_free(ref)
    finally:
        L.speckv_ext_atu_destroy(atu)


def test_ratio_stats_match_reference_accounting():
    """avg_compression_ratio the way the reference accounts it (fp32 original size, mean of ratios)."""
    import cxl_speckv_b200 as pkg
    L = pkg.lib()
    G, n = 2048, 500
    x = torch.randn(n * G, device=DEV).half()
    x[: 100 * G] = 0
    c = codec.compress(x, G)
    tot, mean = C.c_double(), C.c_double()
    assert L.speckv_ext_ratio_stats(c.comp_bytes.data_ptr(), n, G, C.byref(tot), C.byref(mean), None) == 0
    comp = c.comp_bytes.cpu().numpy().view(np.uint32).astype(np.float64)
    assert tot.value == comp.sum()
    assert abs(mean.value - (G * 4.0 / comp).mean()) < 1e-9 * mean.value
    # zeros: 2048 elements -> 9 pairs (255 cap) -> ratio 8192 / 18; N(0,1): ~2.0 (SURVEY.md section 6)
    assert comp[0] == 18 and 1.99 < (G * 4.0 / comp[200:]).mean() < 2.03


@pytest.mark.parametrize("G,num_blocks,n_sel", [(2048, 600, 257), (131072, 9, 5), (16384, 40, 40), (1000, 50, 21)])
@pytest.mark.parametrize("tdt", [F16, BF16])
def test_paged_gather_scatter_matches_staged_path(G, num_blocks, n_sel, tdt):
    """speckv_ext_compress_gather / _decompress_scatter (paged KV cache + block table) give
    the oracle's bytes for the listed blocks, and scatter writes only the blocks named."""
    rng = np.random.default_rng(G + num_blocks)
    x = make_inputs(rng, num_blocks, G, "mixed")
    if tdt == BF16:
        raw = bf16_from_f32(x.astype(np.float32))
        xf = bf16_to_f32(raw)
    else:
        raw, xf = x, x.astype(np.float32)
    cache = to_dev(raw, tdt).view(num_blocks, G)
    table = rng.permutation(num_blocks)[:n_sel].astype(np.int32)
    td = torch.from_numpy(table).to(DEV)
    c = codec.compress_gather(cache, td)
    torch.cuda.synchronize()
    sel = np.ascontiguousarray(xf.reshape(num_blocks, G)[table]).reshape(-1)
    payload, scales, comp = Port.compress_batch(sel, G, threads=8)
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(scales))
    assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp)
    gp = c.payload.cpu().numpy()
    for g in range(n_sel):
        assert np.array_equal(gp[g, :comp[g]], payload[g, :comp[g]]), g
    # scatter into a fresh cache through a different table, picking stored blocks in reverse
    sentinel = 0x1234
    dst = torch.full((num_blocks, G), sentinel, dtype=torch.int16, device=DEV).view(TORCH_DT[tdt])
    dst_table = rng.permutation(num_blocks)[:n_sel].astype(np.int32)
    src_index = np.arange(n_sel - 1, -1, -1).astype(np.int32)
    oel = torch.zeros(n_sel, dtype=torch.int32, device=DEV)
    codec.decompress_scatter(c, dst, torch.from_numpy(dst_table).to(DEV), torch.from_numpy(src_index).to(DEV), oel)
    torch.cuda.synchronize()
    want, want_n = Port.decompress_batch(payload, scales, comp, G, tdt, threads=8)
    got = out_bits(dst)
    want = want.view(np.uint16).reshape(n_sel, G)
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n[src_index])
    for i in range(n_sel):
        assert np.array_equal(got[dst_table[i]], want[src_index[i]]), i
    untouched = np.setdiff1d(np.arange(num_blocks), dst_table)
    assert (got[untouched] == sentinel).all()
    # INT8 scheme through the same tables
    c8 = codec.compress_gather(cache, td, scheme=COMP_INT8)
    q = Port.quantize(sel[:G], scales[0])
    assert np.array_equal(c8.payload[0, :G].cpu().numpy().view(np.int8), q)


def test_paged_gather_scatter_rejects_bad_arguments():
    cache = torch.zeros((4, 2048), dtype=torch.float16, device=DEV)
    table = torch.arange(4, dtype=torch.int32, device=DEV)
    with pytest.raises(Exception):
        codec.compress_gather(cache, table, scheme=COMP_FP16)      # raw passthrough has no gather form
    c = codec.compress_gather(cache, table)
    with pytest.raises(ValueError):
        codec.decompress_scatter(c, torch.zeros((4, 4096), dtype=torch.float16, device=DEV), table)
    with pytest.raises(ValueError):
        codec.decompress_scatter(c, cache, table[:2])
    lens = torch.full((4,), 100, dtype=torch.int32, device=DEV)
    with pytest.raises(TypeError):
        codec.compress_ragged(cache, 2048, lens.long())
    with pytest.raises(TypeError):
        codec.compress_ragged(cache, 2048, lens.cpu())
    with pytest.raises(ValueError):
        codec.compress_ragged(cache, 2048, lens[:3])                     # one length per block of x
    with pytest.raises(ValueError):
        codec.compress_ragged(cache, 2048, lens, block_table=table[:3])  # one length per table entry
    with pytest.raises(ValueError):
        codec.compress_ragged(cache, 1000, lens)
    with pytest.raises(ValueError):
        codec.compress_gather(cache.t(), table)
    # the C entry points: each rejected argument on its own; the raw scheme is refused even for an empty call
    import cxl_speckv_b200 as pkg
    L = pkg.lib()
    buf = dict(p=c.payload.data_ptr(), sb=c.payload.shape[1], s=c.scales.data_ptr(), cb=c.comp_bytes.data_ptr(), dt=0,
               G=2048, n=4, scheme=2, x=cache.data_ptr(), t=table.data_ptr(), len=lens.data_ptr())
    calls = {
        "gather": lambda a: L.speckv_ext_compress_gather(a["x"], a["t"], a["dt"], a["G"], a["n"], a["p"], a["sb"], a["s"],
                                                         a["cb"], a["scheme"], None),
        "ragged": lambda a: L.speckv_ext_compress_ragged(a["x"], a["t"], a["len"], a["dt"], a["G"], a["n"], a["p"],
                                                         a["sb"], a["s"], a["cb"], a["scheme"], None),
        "scatter": lambda a: L.speckv_ext_decompress_scatter(a["p"], a["sb"], a["s"], a["cb"], None, a["t"], a["n"],
                                                             a["G"], a["dt"], a["x"], None, a["scheme"], None),
    }
    own = {"gather": [dict(t=None)], "ragged": [dict(len=None)], "scatter": [dict(t=None)]}
    for name, call in calls.items():
        for bad_arg in [dict(scheme=0), dict(scheme=5), dict(dt=3), dict(x=None), dict(p=None), dict(s=None),
                        dict(cb=None), dict(sb=16), dict(p=c.payload.data_ptr() + 8)] + own[name]:
            assert call({**buf, **bad_arg}) == pkg.SPECKV_ERR_INVAL, (name, bad_arg)
        assert call({**buf, "n": 0, "scheme": 0}) == pkg.SPECKV_ERR_INVAL, name
        assert call({**buf, "n": 0, "p": None, "s": None, "cb": None, "x": None, "t": None,
                     "len": None}) == pkg.SPECKV_OK, name


@pytest.mark.parametrize("G", [2048, 8192, 32768, 131072])
def test_zero_groups_closed_form(G):
    """max-abs 0 (zeros, -0.0, NaNs: the reference's max skips NaN and the cast sends it to code 0) is
    emitted by the tuned kernel itself; its decode fills without staging.  Mixed with ordinary groups."""
    rng = np.random.default_rng(G)
    n_groups = 12
    x = rng.standard_normal(n_groups * G).astype(np.float16).reshape(n_groups, G)
    x[1] = 0.0
    x[4] = -0.0
    x[7] = 0.0
    x[7, rng.integers(0, G, 9)] = np.nan
    x[10] = 0.0
    x = x.reshape(-1)
    xd = torch.from_numpy(x).to(DEV)
    c = codec.compress(xd, G)
    payload, scales, comp = Port.compress_batch(x, G, threads=8)
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(scales))
    assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp)
    gp = c.payload.cpu().numpy()
    for g in range(n_groups):
        assert np.array_equal(gp[g, :comp[g]], payload[g, :comp[g]]), g
    oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
    y = torch.full((n_groups, G), 3.0, dtype=torch.float16, device=DEV)
    codec.decompress(c, out=y, out_elems=oel)
    want, want_n = Port.decompress_batch(payload, scales, comp, G, F16, threads=8)
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n)
    assert np.array_equal(out_bits(y), want.view(np.uint16))


@pytest.mark.parametrize("tdt", [F16, BF16])
def test_decode_zero_valued_regions(tdt):
    """Hand-built payloads whose 2048-pair regions hold only zero values (long constant stretches starting
    from a non-zero code, ragged element offsets, negative scales) between ordinary regions."""
    rng = np.random.default_rng(5 + tdt)
    G, n_groups = 131072, 6
    sb = codec.slot_bytes(G)
    payload = np.zeros((n_groups, sb), np.uint8)
    comp = np.zeros(n_groups, np.uint32)
    scales = rng.uniform(0.01, 2.0, n_groups).astype(np.float32)
    scales[3] = -0.75
    for g in range(n_groups):
        parts = []
        total = 0
        for r in range(20):
            if r % 3 == g % 3:        # a zero-valued region: counts 1..33 (region total 2048..~35000 elements)
                cnt = rng.integers(1, 34 if g % 2 else 3, 2048).astype(np.uint8)
                val = np.zeros(2048, np.uint8)
            else:                     # an ordinary region: counts of 1, one count of 2 here and there
                cnt = np.ones(2048, np.uint8)
                cnt[rng.integers(0, 2048, 5)] = 2
                val = rng.integers(0, 256, 2048, dtype=np.uint8)
            if total + int(cnt.sum()) > G:
                break
            total += int(cnt.sum())
            parts.append(np.stack([val, cnt], axis=1).reshape(-1))
        p = np.concatenate(parts)
        payload[g, :p.size] = p
        comp[g] = p.size
    c = codec.CompressedKV(torch.from_numpy(payload).to(DEV), torch.from_numpy(scales).to(DEV),
                           torch.from_numpy(comp.view(np.int32)).to(DEV), G, TORCH_DT[tdt], COMP_INT8_DELTA_RLE)
    out = torch.full((n_groups, G), 0x1234, dtype=torch.int16, device=DEV).view(TORCH_DT[tdt])
    oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
    codec.decompress(c, out=out, out_elems=oel)
    want, want_n = Port.decompress_batch(payload, scales, comp, G, tdt, threads=8)
    got = out_bits(out)
    want = want.view(np.uint16).reshape(n_groups, G)
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n)
    for g in range(n_groups):
        n = int(want_n[g])
        assert np.array_equal(got[g, :n], want[g, :n]), g
        assert (got[g, n:] == 0x1234).all(), g


def test_plain_c_host_program_on_the_gpu(tmp_path):
    """tests/c/frozen_abi.c with a CUDA device: C host code -> C ABI -> kernels, no Python in the data path.
    Checks the reference's KAT-1 bytes / scale / decompressed values and the three translate_address
    results recorded from the reference."""
    import subprocess
    from tests.test_abi_cpu import _build_c_program
    exe = _build_c_program(tmp_path, with_cuda=True)
    r = subprocess.run([exe, "cuda:0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.parametrize("G,n_groups,dtype", [(131072, 2048, "f16"), (2048, 131072, "bf16"), (16384, 8192, "f16")])
def test_tuned_and_generic_kernels_agree_at_scale(G, n_groups, dtype):
    """512 MiB of KV per case (BASELINE config 1 size), structured and unstructured groups mixed: the tuned
    TMA / cluster kernels and the generic kernels (SPECKV_FORCE_GENERIC=1, a separate implementation that the
    oracle tests pin on small sizes) give the same sizes, scales, payload bytes and decoded values."""
    import json
    import os
    import subprocess
    import sys
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_digest_worker.py")
    res = {}
    for force in ("0", "1"):
        env = dict(os.environ, SPECKV_FORCE_GENERIC=force)
        r = subprocess.run([sys.executable, worker, str(G), str(n_groups), dtype], capture_output=True, text=True,
                           env=env, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        res[force] = json.loads(r.stdout.strip().splitlines()[-1])
    a, b = res["0"], res["1"]
    for k in ("comp_sum", "comp_xor", "scale_bits_sum", "payload_weighted_sum", "output_weighted_sum"):
        assert a[k] == b[k], (k, a[k], b[k])
    assert a["launches"] > b["launches"]      # the tuned path really ran (fast kernel + flagged second pass)


@pytest.mark.parametrize("tdt", [F16, BF16])
def test_infinite_group_decodes_to_the_oracles_nan_bits(tdt):
    """A group that contains +-inf has an infinite scale; the reference then decodes 0 * inf = NaN (x86's real
    indefinite 0xFFC00000) and +-inf.  At the fp16 / bf16 boundary the NaN keeps its sign and payload bits
    (0xFE00 / 0xFFC0, what x86 F16C and the oracle give), not the GPU's canonical 0x7FFF."""
    rng = np.random.default_rng(77)
    G, n_groups = 2048, 6
    x = rng.standard_normal(n_groups * G).astype(np.float32).reshape(n_groups, G)
    x[1, 5] = np.inf
    x[3, 100] = -np.inf
    x[4, 7] = np.inf
    x[4, 9] = np.nan
    if tdt == F16:
        raw = x.astype(np.float16).reshape(-1)
    else:
        raw = bf16_from_f32(x.reshape(-1))
    c = codec.compress(to_dev(raw, tdt), G)
    y = codec.decompress(c)
    payload, scales, comp = Port.compress_batch(raw, G, dtype=tdt, threads=4)
    want, _ = Port.decompress_batch(payload, scales, comp, G, tdt, threads=4)
    got = out_bits(y)
    assert np.array_equal(got, want.view(np.uint16).reshape(n_groups, G))
    assert (got[1] == (0xFE00 if tdt == F16 else 0xFFC0)).any()


@pytest.mark.parametrize("G", [2048, 16384, 32768, 131072])
@pytest.mark.parametrize("tdt", [F16, BF16])
def test_long_runs_then_dense_heads(G, tdt):
    """Regions that start inside a long constant stretch (only forced heads: the 255 cap of cache_engine.cpp:223) and
    turn into noise at an arbitrary position -- every lane chunk then holds a different number of run boundaries.
    The first head-stationary emission of the long-run path lost all pairs after such a turn (fuzz seed 13, case 840:
    the lanes without a boundary ran on without the others behind a lane-divergent store ladder); sizes, scales and
    every payload byte against the oracle."""
    rng = np.random.default_rng(840 + G)
    n_groups = max(4, min(64, (2 << 20) // G))
    x = rng.standard_normal(n_groups * G).astype(np.float32)
    for g in range(n_groups):
        pos = g * G + int(rng.integers(0, 8))
        end = (g + 1) * G
        while pos < end:
            run = int(rng.choice([300, 700, 2048 + 3, 4904, 1016, 255, 256, 8 * int(rng.integers(1, 600)) + int(rng.integers(0, 8))]))
            x[pos:min(end, pos + run)] = x[pos] if rng.random() < 0.5 else 0.0
            pos += run
            dense = int(rng.choice([1, 7, 9, 130, 1144, 2500])) + int(rng.integers(0, 16))
            if rng.random() < 0.5:      # sparse boundaries: short runs of 1 .. 12
                q = pos
                while q < min(end, pos + dense):
                    r = int(rng.integers(1, 13))
                    x[q:min(end, q + r)] = x[q]
                    q += r
            pos += dense
    raw = x.astype(np.float16) if tdt == F16 else bf16_from_f32(x)
    xd = torch.from_numpy(raw).to(DEV) if tdt == F16 else torch.from_numpy(raw.astype(np.int16)).to(DEV).view(torch.bfloat16)
    c = codec.compress(xd, G)
    payload, scales, comp = Port.compress_batch(raw, G, dtype=tdt, threads=8)
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(scales))
    assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp)
    gp = c.payload.cpu().numpy()
    for g in range(n_groups):
        assert np.array_equal(gp[g, :comp[g]], payload[g, :comp[g]]), (g, comp[g])
    y = codec.decompress(c)
    want, _ = Port.decompress_batch(payload, scales, comp, G, tdt, threads=8)
    assert np.array_equal(out_bits(y).reshape(-1), want.view(np.uint16).reshape(-1))


@pytest.mark.parametrize("G", [8192, 32768, 131072])
@pytest.mark.parametrize("tdt", [F16, BF16])
@pytest.mark.parametrize("scheme", [2, 3])
def test_partially_filled_blocks(G, tdt, scheme):
    """KV blocks filled up to an arbitrary token and zero (or constant, or NaN-sprinkled zero) behind it: compress skips
    the quantiser for all-zero regions of a non-zero group, decompress expands the dense front of the boundary region in
    place and writes the tail as a fill (the group stays off the run-expansion path).  Sizes, scales, payload bytes and
    decoded bits against the oracle; fill levels around region and iteration edges; the reference's scheme and the
    clamped extension (NaN codes as 0 in both)."""
    rng = np.random.default_rng(7 * G + (1 if tdt == BF16 else 0))
    levels = [1, 9, 255, 256, 2047, 2048, 2049, 2048 + 1016, 5000, G // 2 - 1, G // 2, G - 2048 - 3, G - 300, G - 9, G - 1]
    n_groups = len(levels) * 3
    x = rng.standard_normal(n_groups * G).astype(np.float32)
    for i in range(n_groups):
        lvl = levels[i % len(levels)]
        tail = x[i * G + lvl:(i + 1) * G]
        kind = i // len(levels)
        tail[:] = 0.0 if kind != 1 else 0.625
        if kind == 2 and tail.size > 40:
            tail[rng.integers(0, tail.size, 3)] = np.nan          # NaN quantises to code 0 like the zeros around it
    raw = x.astype(np.float16) if tdt == F16 else bf16_from_f32(x)
    xd = torch.from_numpy(raw).to(DEV) if tdt == F16 else torch.from_numpy(raw.astype(np.int16)).to(DEV).view(torch.bfloat16)
    c = codec.compress(xd, G, scheme=scheme)
    payload, scales, comp = Port.compress_batch(raw, G, dtype=tdt, threads=8, scheme=scheme)
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(scales))
    assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp)
    gp = c.payload.cpu().numpy()
    for g in range(n_groups):
        assert np.array_equal(gp[g, :comp[g]], payload[g, :comp[g]]), (g, levels[g % len(levels)], comp[g])
    oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
    y = codec.decompress(c, out_elems=oel)
    want, want_n = Port.decompress_batch(payload, scales, comp, G, tdt, threads=8, scheme=scheme)
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n)
    got = out_bits(y).reshape(n_groups, G)
    wantb = want.view(np.uint16).reshape(n_groups, G)
    bad = np.argwhere(got != wantb)
    assert bad.size == 0, (bad[:3], levels[int(bad[0][0]) % len(levels)])


def test_randomised_differential_run():
    """tests/fuzz_codec.py for a few seconds: random geometries, dtypes and value structures against the oracle."""
    from tests import fuzz_codec
    fuzz_codec.main(seconds=8.0, seed=11)
    fuzz_codec.main_decode(seconds=6.0, seed=12)


def test_memory_manager_address_map_on_device():
    """The reference's CXLMemoryManager address map (allocate / deallocate / set_tier), exported to the device:
    one page-lookup launch answers translate_virtual_to_physical and is_in_cache for a batch of addresses,
    identical to the oracle restatement (which tests/test_abi_cpu.py pins to the reference's own class)."""
    import ctypes as C
    from cxl_speckv_b200.tier import CxlAddressMap
    from tests.test_abi_cpu import _mm_port, mm_random_ops
    P = _mm_port()
    rng = np.random.default_rng(8)
    m = C.c_void_p(P.oracle_mm_new(12 << 30, 3 << 30, 128 << 30, 4096))
    prod = CxlAddressMap()
    allocs = []
    for op, a, b in mm_random_ops(rng, 4000):
        if op == "alloc":
            va = P.oracle_mm_allocate(m, a, 0, b)
            assert prod.allocate(a, 0, b)[0] == va
            allocs.append((va, a))
        elif op == "free":
            va = allocs[a][0] + min(b, (allocs[a][1] + 4095) // 4096 - 1) * 4096
            P.oracle_mm_deallocate(m, va)
            prod.deallocate(va)
    table = prod.export(DEV)
    q = np.concatenate([np.array([va + int(rng.integers(0, size + 9000)) for va, size in allocs for _ in range(4)], dtype=np.uint64),
                        np.array([0, 0xFFFFFFFF, 0x100000000 - 1, 1 << 60, 0x100000000 + (1 << 40)], dtype=np.uint64)])
    pa, flags = prod.translate(table, torch.from_numpy(q.view(np.int64)).to(DEV))
    pa, flags = pa.cpu().numpy().view(np.uint64), flags.cpu().numpy()
    want = np.array([P.oracle_mm_translate(m, int(v)) for v in q], dtype=np.uint64)
    assert np.array_equal(pa, want)
    for i in rng.integers(0, q.size, 2000):
        for t, bit in ((0, 1), (1, 2)):
            assert bool(flags[i] & bit) == bool(P.oracle_mm_is_in_cache(m, int(q[i]), t))
    # a promotion decided by the residency policy shows up after set_tier + export
    va0, size0 = allocs[0]
    if prod.translate_host(va0)[0]:
        prod.set_tier(va0, 1, 0)
        t2 = prod.export(DEV)
        _, f2 = prod.translate(t2, torch.tensor([va0], dtype=torch.int64, device=DEV))
        assert int(f2[0]) & 1
    prod.close()
    P.oracle_mm_free(m)


@pytest.mark.parametrize("G,n_groups,tdt", [(131072, 128, torch.float16), (131072, 128, torch.bfloat16),
                                            (2048, 16384, torch.float16), (2048, 8192, torch.bfloat16)])
def test_full_layer_bit_exact_against_reference_engine(G, n_groups, tdt):
    """One whole Llama-2-70B layer (config 3: 2 x 8 KV heads x 8 blocks = 128 groups of 1024 x 128) and a config-4
    layer slice (4 KiB page groups), EVERY group compared with the reference's own FPGACacheEngine (oracle/_ref,
    else the C restatement): compressed bytes, sizes, scale bits and decoded bits.  A tenth of the groups carry
    constant stretches (runs past the 255 cap) and zero tails, the rest is N(0,1)."""
    from oracle.oracle import Ref
    dcode = F16 if tdt == torch.float16 else BF16
    gen = torch.Generator(device=DEV)
    gen.manual_seed(99 + G)
    x = torch.empty(n_groups * G, dtype=torch.float32, device=DEV).normal_(generator=gen).to(tdt).view(n_groups, G)
    for g in range(0, n_groups, 10):
        x[g, G // 3: G // 3 + 777] = 0.125
        x[g, G - min(G // 4, 600):] = 0
    x = x.reshape(-1).contiguous()
    c = codec.compress(x, G)
    y = codec.decompress(c)
    torch.cuda.synchronize()
    xh = x.view(torch.int16).cpu().numpy().view(np.uint16)
    if Ref.available():
        rp, rs, rc, ro = Ref.roundtrip_batch(xh, dcode, G, threads=8)
    else:
        xf = xh.view(np.float16) if dcode == F16 else xh
        rp, rs, rc = Port.compress_batch(xf, G, dtype=dcode, threads=8)
        ro, _ = Port.decompress_batch(rp, rs, rc, G, dcode, threads=8)
        ro = ro.view(np.uint16).reshape(n_groups, G)
    comp = c.comp_bytes.cpu().numpy().view(np.uint32)
    assert np.array_equal(comp, rc)
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(rs))
    gp = c.payload.cpu().numpy()
    mask = np.arange(gp.shape[1])[None, :] < comp[:, None]
    assert np.array_equal(np.where(mask, gp, 0), np.where(mask, rp[:, :gp.shape[1]], 0))
    assert np.array_equal(y.view(torch.int16).cpu().numpy().view(np.uint16), ro.view(np.uint16).reshape(n_groups, G))
