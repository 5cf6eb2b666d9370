"""GPU parity tests of ragged groups: the filled prefix of each KV block (speckv_ext_compress_ragged,
speckv_ext_tier_offload_ragged, CxlSpeckvKVAllocator.offload_kv_blocks(num_tokens=...)).

A ragged group of length n is the reference engine's compress on the vector x[g, :n] (cache_engine.cpp:40-82 takes
a vector of any length), so the bar is the oracle on that prefix: scale bits, comp_bytes and payload[:comp_bytes]
equal Port's, whatever the block holds behind n (+-inf, NaN, 65504, random garbage: the stale K/V of an earlier
request).  Decodes give n elements and leave the destination behind them untouched (sentinel-filled buffers)."""
import numpy as np
import pytest
import torch

from oracle.oracle import Port
from tests.helpers import BF16, F16, F32, bf16_from_f32, f32_bits

pytestmark = pytest.mark.gpu

from cxl_speckv_b200 import SpeckvError, codec  # noqa: E402
from cxl_speckv_b200.tier import HostTier  # noqa: E402
from cxl_speckv_b200.vllm_speckv_backend import CxlSpeckvKVAllocator  # noqa: E402
from tests.test_codec_paths_gpu import CLASSES, class_group  # noqa: E402

DEV = "cuda:0"
TORCH_DT = {F16: torch.float16, BF16: torch.bfloat16, F32: torch.float32}
SENT16 = 0x1234
SENT32 = 0x3F9E0419   # an fp32 pattern no decode of these inputs produces by chance


def narrow(x, tdt):
    if tdt == F16:
        with np.errstate(over="ignore", invalid="ignore"):
            return x.astype(np.float16)
    if tdt == BF16:
        return bf16_from_f32(x.reshape(-1)).reshape(x.shape)
    return x.astype(np.float32)


def to_dev(raw, tdt):
    if tdt == BF16:
        return torch.from_numpy(np.ascontiguousarray(raw).view(np.int16)).to(DEV).view(torch.bfloat16)
    return torch.from_numpy(np.ascontiguousarray(raw)).to(DEV)


def bits(t):
    if t.dtype == torch.float32:
        return t.view(torch.int32).cpu().numpy().view(np.uint32)
    return t.view(torch.int16).cpu().numpy().view(np.uint16)


def sentinel(shape, tdt):
    if tdt == F32:
        return torch.full(shape, SENT32, dtype=torch.int32, device=DEV).view(torch.float32)
    return torch.full(shape, SENT16, dtype=torch.int16, device=DEV).view(TORCH_DT[tdt])


def sent_value(tdt):
    return np.uint32(SENT32) if tdt == F32 else np.uint16(SENT16)


def lengths_for(G, rng, n_random=6):
    """Every boundary the kernels treat specially, plus random ones (whole 64-element tokens and arbitrary)."""
    base = [0, 1, 7, 8, 63, 64, 128, 255, 256, 2047, 2048, 2049, G - 128, G - 1, G, G + 5, 3 * G]
    k = max(1, G // 2048 - 1)
    base.append(2048 * k + 5)   # inside the halo of region k
    out = [n for n in base if n >= 0 and (n <= G or n in (G + 5, 3 * G))]
    out += [int(rng.integers(1, G // 64 + 1)) * 64 for _ in range(n_random // 2)]
    out += [int(rng.integers(1, G + 1)) for _ in range(n_random - n_random // 2)]
    return out


def garbage_tail(rng, x, lengths, G, tdt, variant):
    """Fill every block behind its length with stale-looking data: +-inf, NaN, 65504 or random large values."""
    x = x.copy()
    for g, n in enumerate(lengths):
        n = min(n, G)
        m = G - n
        if m == 0:
            continue
        kind = (g + variant) % 4
        if kind == 0:
            t = np.where(rng.random(m) < 0.5, np.inf, -np.inf)
        elif kind == 1:
            t = np.full(m, np.nan)
        elif kind == 2:
            t = np.full(m, 65504.0)
        else:
            t = rng.standard_normal(m) * 1e4
        x[g, n:] = t.astype(np.float32)
    return x


def special_prefix(rng, x, lengths, G):
    """Content around the end: a run that straddles n, a run of exactly 255 ending at n, inf / tiny in the prefix."""
    x = x.copy()
    for g, n in enumerate(lengths):
        n = min(n, G)
        kind = g % 5
        if kind == 0 and n >= 300:
            x[g, n - 150: min(G, n + 150)] = 0.25                  # straddles n
        elif kind == 1 and n >= 256:
            x[g, n - 255: n] = -0.5                                # exactly 255 ending at n
        elif kind == 2 and n >= 1:
            x[g, int(rng.integers(0, n))] = np.inf                 # inside the prefix
        elif kind == 3 and n >= 1:
            x[g, :n] *= np.float32(1e-39)                          # tiny (bf16 generic range; fp16 zeros)
    return x


def oracle_prefix(raw, lengths, G, tdt, scheme):
    """Port on x[g, :n] for every group: (scale bits, comp_bytes, payload bytes per group)."""
    sc, cb, pl = [], [], []
    for g, n in enumerate(lengths):
        n = min(n, G)
        if n == 0:
            sc.append(np.float32(1.0))
            cb.append(0)
            pl.append(np.zeros(0, np.uint8))
            continue
        p, s, c = Port.compress_batch(np.ascontiguousarray(raw[g, :n]), n, dtype=tdt, scheme=scheme)
        sc.append(s[0])
        cb.append(int(c[0]))
        pl.append(p[0, :c[0]].copy())
    return f32_bits(np.array(sc, np.float32)), np.array(cb, np.uint32), pl


def assert_container(c, want, tag):
    sbits, comp, pl = want
    got_s = f32_bits(c.scales.cpu().numpy())
    got_c = c.comp_bytes.cpu().numpy().view(np.uint32)
    bad = np.flatnonzero(got_s != sbits)
    assert bad.size == 0, (tag, "scale", bad[:5])
    bad = np.flatnonzero(got_c != comp)
    assert bad.size == 0, (tag, "comp_bytes", bad[:5], got_c[bad[:5]], comp[bad[:5]])
    gp = c.payload.cpu().numpy()
    for g, p in enumerate(pl):
        assert np.array_equal(gp[g, :p.size], p), (tag, "payload of group", g)


def make_batch(rng, G, tdt, lengths):
    cls = [CLASSES[i % len(CLASSES)] for i in range(len(lengths))]
    x = np.stack([class_group(rng, c, G, tdt if tdt != F32 else F16) for c in cls])
    return special_prefix(rng, x, lengths, G)


def lens_dev(lengths):
    return torch.tensor(lengths, dtype=torch.int64).clamp(max=2**31 - 1).to(torch.int32).to(DEV)


# ---- 1. parity sweep ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scheme", [1, 2, 3, 4])
@pytest.mark.parametrize("tdt", [F16, BF16, F32])
@pytest.mark.parametrize("G", [2048, 16384, 131072, 6144])
def test_ragged_parity_sweep(G, tdt, scheme):
    rng = np.random.default_rng(G * 31 + tdt * 7 + scheme)
    lengths = lengths_for(G, rng)
    x = make_batch(rng, G, tdt, lengths)
    want = None
    results = []
    for variant in range(2):   # two different garbage tails: the outputs must not move
        raw = narrow(garbage_tail(rng, x, lengths, G, tdt, variant), tdt)
        if want is None:
            want = oracle_prefix(raw, lengths, G, tdt, scheme)
        c = codec.compress_ragged(to_dev(raw, tdt), G, lens_dev(lengths), scheme=scheme)
        torch.cuda.synchronize()
        assert_container(c, want, (G, tdt, scheme, variant))
        results.append(c)
    # the payload bytes themselves, not only the prefix the oracle fixes, are the same under both tails
    for g, p in enumerate(want[2]):
        a = results[0].payload[g, :p.size].cpu().numpy()
        b = results[1].payload[g, :p.size].cpu().numpy()
        assert np.array_equal(a, b)


# ---- 2. decode --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scheme", [1, 2, 3, 4])
@pytest.mark.parametrize("tdt", [F16, BF16])
@pytest.mark.parametrize("G", [2048, 131072])
def test_ragged_decode(G, tdt, scheme):
    rng = np.random.default_rng(G + 13 * scheme + tdt)
    lengths = lengths_for(G, rng)
    raw = narrow(garbage_tail(rng, make_batch(rng, G, tdt, lengths), lengths, G, tdt, 0), tdt)
    ng = len(lengths)
    c = codec.compress_ragged(to_dev(raw, tdt), G, lens_dev(lengths), scheme=scheme)
    torch.cuda.synchronize()
    n = np.minimum(np.array(lengths), G)
    want_y, want_n = Port.decompress_batch(c.payload.cpu().numpy(), c.scales.cpu().numpy(),
                                           c.comp_bytes.cpu().numpy().view(np.uint32), G, tdt, scheme=scheme)
    assert np.array_equal(want_n, n)
    want = np.where(np.arange(G)[None, :] < n[:, None], want_y.view(np.uint16).reshape(ng, G), np.uint16(SENT16))

    out = sentinel((ng, G), tdt)
    oe = torch.full((ng,), -1, dtype=torch.int32, device=DEV)
    codec.decompress(c, out=out, out_elems=oe)
    torch.cuda.synchronize()
    assert np.array_equal(oe.cpu().numpy(), n)
    assert np.array_equal(bits(out), want), "decompress"

    idx = torch.tensor(list(range(ng))[::-1], dtype=torch.int32, device=DEV)
    out = sentinel((ng, G), tdt)
    codec.decompress_indexed(c, idx, out=out)
    torch.cuda.synchronize()
    assert np.array_equal(bits(out), want[::-1]), "decompress_indexed"

    cache = sentinel((ng + 3, G), tdt)
    table = torch.from_numpy(rng.permutation(ng + 3)[:ng].astype(np.int32)).to(DEV)
    oe = torch.full((ng,), -1, dtype=torch.int32, device=DEV)
    codec.decompress_scatter(c, cache, table, out_elems=oe)
    torch.cuda.synchronize()
    assert np.array_equal(oe.cpu().numpy(), n)
    got = bits(cache)
    assert np.array_equal(got[table.cpu().numpy()], want), "decompress_scatter"
    untouched = np.setdiff1d(np.arange(ng + 3), table.cpu().numpy())
    assert (got[untouched] == SENT16).all()


# ---- 1b. ends at a 256-element boundary inside a region, with long runs before it ------------------------------
@pytest.mark.parametrize("scheme", [2, 3])
@pytest.mark.parametrize("tdt", [F16, BF16])
@pytest.mark.parametrize("G", [2048, 16384, 131072])
def test_ragged_long_run_region_ending_on_256(G, tdt, scheme):
    """n a multiple of 256 but not of 2048 (every odd token count of 1024-element tokens), with a stretch of 40 equal
    values inside the boundary region (or across its start) so that it takes the long-run emission, and noise up to
    n: the reference's last pair closes at n with delta[n - 1]."""
    rng = np.random.default_rng(G + 101 * scheme + tdt)
    R = G // 2048
    lengths = [256, 1024, 1280, 1792]
    for r in sorted(set([1, R // 2, R - 1])):
        if 1 <= r < R:
            lengths += [2048 * r + 256, 2048 * r + 1024, 2048 * r + 1792]
    x = rng.standard_normal((len(lengths), G)).astype(np.float32)
    for g, n in enumerate(lengths):
        rs = (n - 1) // 2048 * 2048
        kind = g % 3
        if kind == 2 and rs >= 2048:
            x[g, rs - 8: rs + 24] = 0.0           # across the region start: the halo sees the run
        else:
            x[g, rs + 8: rs + 48] = 0.0 if kind == 0 else 0.5
    x = garbage_tail(rng, x, lengths, G, tdt, 0)
    raw = narrow(x, tdt)
    want = oracle_prefix(raw, lengths, G, tdt, scheme)
    assert sum(int(p[-2]) != 0 for p in want[2]) >= len(lengths) // 2   # last pairs with a non-zero delta
    c = codec.compress_ragged(to_dev(raw, tdt), G, lens_dev(lengths), scheme=scheme)
    torch.cuda.synchronize()
    assert_container(c, want, ("256-boundary", G, tdt, scheme))
    n = np.array(lengths)
    y = sentinel((len(lengths), G), tdt)
    codec.decompress(c, out=y)
    torch.cuda.synchronize()
    want_y, want_n = Port.decompress_batch(c.payload.cpu().numpy(), c.scales.cpu().numpy(),
                                           c.comp_bytes.cpu().numpy().view(np.uint32), G, tdt, scheme=scheme)
    assert np.array_equal(want_n, n)
    assert np.array_equal(bits(y), np.where(np.arange(G)[None, :] < n[:, None],
                                            want_y.view(np.uint16).reshape(len(lengths), G), np.uint16(SENT16)))


# ---- 3. block table, graphs, streams -------------------------------------------------------------------------------
@pytest.mark.parametrize("scheme", [2, 4])
@pytest.mark.parametrize("G", [2048, 16384, 131072])
def test_ragged_gather_with_block_table(G, scheme):
    rng = np.random.default_rng(G + scheme)
    nb = 12
    blocks = narrow(rng.standard_normal((nb, G)).astype(np.float32) * 1e3, F16)   # garbage everywhere
    sel = [7, 2, 9, 0, 11, 5]
    lengths = [G // 2 + 64, 64, G, 0, 2048 + 128, G - 64]
    vals = make_batch(rng, G, F16, lengths)
    for i, b in enumerate(sel):
        blocks[b, :lengths[i]] = narrow(vals[i, :lengths[i]], F16)
    table = torch.tensor(sel, dtype=torch.int32, device=DEV)
    c = codec.compress_ragged(to_dev(blocks, F16), G, lens_dev(lengths), block_table=table, scheme=scheme)
    torch.cuda.synchronize()
    assert_container(c, oracle_prefix(blocks[sel], lengths, G, F16, scheme), ("gather", G, scheme))


@pytest.mark.parametrize("scheme", [2, 3, 1])
@pytest.mark.parametrize("G", [2048, 131072])
def test_ragged_graph_replay_new_lengths_and_inputs(G, scheme):
    rng = np.random.default_rng(5 + G + scheme)
    ng = 8
    x = torch.empty((ng, G), dtype=torch.float16, device=DEV)
    lens = torch.zeros(ng, dtype=torch.int32, device=DEV)
    out = codec.CompressedKV(torch.empty((ng, codec.slot_bytes(G, scheme)), dtype=torch.uint8, device=DEV),
                             torch.empty(ng, dtype=torch.float32, device=DEV),
                             torch.empty(ng, dtype=torch.int32, device=DEV), G, torch.float16, scheme)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        codec.compress_ragged(x, G, lens, scheme=scheme, out=out)   # grows the per-stream scratch before capture
        s.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            codec.compress_ragged(x, G, lens, scheme=scheme, out=out)
    for rep in range(3):
        lengths = [int(rng.integers(0, G + 1)) for _ in range(ng)]
        lengths[rep] = G
        raw = narrow(garbage_tail(rng, make_batch(rng, G, F16, lengths), lengths, G, F16, rep), F16)
        x.copy_(to_dev(raw, F16))
        lens.copy_(lens_dev(lengths))
        graph.replay()
        torch.cuda.synchronize()
        assert_container(out, oracle_prefix(raw, lengths, G, F16, scheme), ("graph", G, scheme, rep))


def test_ragged_two_streams_concurrently():
    rng = np.random.default_rng(77)
    G, ng = 16384, 24
    jobs = []
    for k in range(2):
        lengths = [int(rng.integers(0, G // 64 + 1)) * 64 for _ in range(ng)]
        raw = narrow(garbage_tail(rng, make_batch(rng, G, F16, lengths), lengths, G, F16, k), F16)
        jobs.append((raw, lengths, to_dev(raw, F16), lens_dev(lengths), torch.cuda.Stream()))
    torch.cuda.synchronize()
    outs = []
    for raw, lengths, xd, ld, st in jobs:
        with torch.cuda.stream(st):
            outs.append(codec.compress_ragged(xd, G, ld, scheme=2))
    torch.cuda.synchronize()
    for (raw, lengths, _, _, _), c in zip(jobs, outs):
        assert_container(c, oracle_prefix(raw, lengths, G, F16, 2), "two streams")


# ---- 4. tier ----------------------------------------------------------------------------------------------------
def _roundtrip_want(raw, lengths, G, tdt, scheme):
    """Oracle round trip of each prefix as 16-bit patterns, SENT16 behind it."""
    want = np.full((len(lengths), G), SENT16, np.uint16)
    for g, n in enumerate(lengths):
        n = min(n, G)
        if n == 0:
            continue
        p, s, c = Port.compress_batch(np.ascontiguousarray(raw[g, :n]), n, dtype=tdt, scheme=scheme)
        y, m = Port.decompress_batch(p, s, c, n, tdt, scheme=scheme)
        assert m[0] == n
        want[g, :n] = y.view(np.uint16).reshape(-1)[:n]
    return want


@pytest.mark.parametrize("scheme", [2, 4])
@pytest.mark.parametrize("tdt", [F16, BF16])
@pytest.mark.parametrize("G", [2048, 131072])
def test_tier_offload_ragged_flat_and_paged(G, tdt, scheme):
    rng = np.random.default_rng(G + tdt + scheme)
    lengths = lengths_for(G, rng, n_random=4)[:12]
    ng = len(lengths)
    raw = narrow(garbage_tail(rng, make_batch(rng, G, tdt, lengths), lengths, G, tdt, 1), tdt)
    esz = 2
    valid = sum(min(n, G) for n in lengths) * esz
    want = _roundtrip_want(raw, lengths, G, tdt, scheme)
    tier = HostTier(256 << 20)
    try:
        tier.set_scheme(scheme)
        ids = np.arange(ng, dtype=np.uint64) + 1000
        s0 = tier.stats()
        tier.offload_ragged(to_dev(raw, tdt), G, lens_dev(lengths), ids)
        s1 = tier.stats()
        assert s1["bytes_offloaded_raw"] - s0["bytes_offloaded_raw"] == valid
        out = sentinel((ng, G), tdt)
        tier.restore(ids, G, TORCH_DT[tdt], out=out)
        s2 = tier.stats()
        assert s2["bytes_restored_raw"] - s1["bytes_restored_raw"] == valid
        assert np.array_equal(bits(out), want), "flat restore"

        # paged: the blocks sit in a larger cache at the positions the table names; restore into other blocks
        cache = np.asarray(narrow(rng.standard_normal((ng + 5, G)).astype(np.float32) * 100, tdt))
        put = rng.permutation(ng + 5)[:ng].tolist()
        cache[put] = raw
        pids = ids + 5000
        tier.offload_ragged(to_dev(cache, tdt), G, lens_dev(lengths), pids,
                            block_table=torch.tensor(put, dtype=torch.int32, device=DEV))
        dst = sentinel((ng + 5, G), tdt)
        back = rng.permutation(ng + 5)[:ng].tolist()
        tier.restore_blocks(pids, dst, torch.tensor(back, dtype=torch.int32, device=DEV))
        got = bits(dst)
        assert np.array_equal(got[back], want), "paged restore"
        assert (got[np.setdiff1d(np.arange(ng + 5), back)] == SENT16).all()
    finally:
        tier.close()


def test_tier_ragged_scheme_rules():
    G = 2048
    x = torch.randn(4, G, device=DEV).half()
    lens = lens_dev([100, 2048, 0, 64])
    tier = HostTier(16 << 20)
    try:
        tier.set_scheme(0)
        with pytest.raises(SpeckvError) as ei:
            tier.offload_ragged(x, G, lens, np.arange(4))
        assert ei.value.status == -4                               # SPECKV_ERR_INVAL
        # a block keeps the scheme it was stored under
        tier.set_scheme(4)
        tier.offload_ragged(x, G, lens, np.arange(4))
        tier.set_scheme(2)
        out = sentinel((4, G), F16)
        tier.restore(np.arange(4), G, torch.float16, out=out)
        raw = x.cpu().numpy()
        assert np.array_equal(bits(out), _roundtrip_want(raw, [100, 2048, 0, 64], G, F16, 4))
    finally:
        tier.close()
    with pytest.raises(SpeckvError) as ei:
        codec.compress_ragged(x, G, lens, scheme=0)
    assert ei.value.status == -4


# ---- 5. vLLM ----------------------------------------------------------------------------------------------------
def test_vllm_offload_kv_blocks_num_tokens():
    rng = np.random.default_rng(3)
    num_blocks, block_size, heads, dim = 10, 16, 8, 128    # a block = 16 tokens x 1024 elements = 16384
    G = block_size * heads * dim
    cache = torch.from_numpy(rng.standard_normal((num_blocks, block_size, heads, dim)).astype(np.float16) * 50).to(DEV)
    prefix = torch.from_numpy(rng.standard_normal((5, heads, dim)).astype(np.float16)).to(DEV)
    cache[2, :5] = prefix
    cache[6, :5] = prefix                                  # same 5 tokens, different stale tails
    cache[6, 5:] = float("nan")
    table = torch.tensor([2, 6, 4], dtype=torch.int32, device=DEV)
    num_tokens = [5, 5, 16]
    tier = HostTier(64 << 20)
    try:
        stored = []
        for i in range(3):   # one block per call: what each one stores
            CxlSpeckvKVAllocator.offload_kv_blocks(cache, table[i:i + 1], tier, num_tokens=num_tokens[i:i + 1])
            stored.append(tier.stats()["last_offload_stored_bytes"])
        assert stored[0] == stored[1]
        raw = cache.view(num_blocks, G).cpu().numpy()
        _, _, c = Port.compress_batch(np.ascontiguousarray(raw[2, :5 * heads * dim]), 5 * heads * dim, dtype=F16)
        assert stored[0] == (int(c[0]) + 15) // 16 * 16
        dst = sentinel((num_blocks, block_size, heads, dim), F16)
        back = torch.tensor([1, 8, 3], dtype=torch.int32, device=DEV)
        CxlSpeckvKVAllocator.restore_kv_blocks(dst, back, tier, block_ids=table.cpu().numpy().astype("uint64"))
        got = bits(dst.view(num_blocks, G))
        want = _roundtrip_want(raw[[2, 6, 4]], [5 * heads * dim, 5 * heads * dim, G], G, F16, 2)
        assert np.array_equal(got[[1, 8, 3]], want)
        assert np.array_equal(got[1], got[8])              # stale data never reached the tier
    finally:
        tier.close()
