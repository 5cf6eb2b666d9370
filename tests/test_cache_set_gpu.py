"""GPU parity tests of KV cache sets: one call for a request's blocks across all layers (speckv_ext_cache_set_create,
speckv_ext_compress_gather_set / _decompress_scatter_set, speckv_ext_tier_offload_set / _restore_set / _fetch_set,
KVCacheSet, CxlSpeckvKVAllocator.register_kv_caches / offload_request / restore_request).

The bar is the single-cache paged path run cache by cache (compress_gather / compress_ragged / decompress_scatter /
offload_blocks / restore_blocks / fetch with a block table), which the rest of the suite pins to the oracle: every
output is bit-equal to it.  A few groups are also compared with oracle.Port directly.  Blocks a call does not name
keep a sentinel."""
import numpy as np
import pytest
import torch

from oracle.oracle import Port
from tests.helpers import BF16, F16, F32

pytestmark = pytest.mark.gpu

import cxl_speckv_b200 as pkg  # noqa: E402
from cxl_speckv_b200 import SpeckvError, codec  # noqa: E402
from cxl_speckv_b200.codec import KVCacheSet  # noqa: E402
from cxl_speckv_b200.tier import HostTier  # noqa: E402
from cxl_speckv_b200.vllm_speckv_backend import CxlSpeckvKVAllocator  # noqa: E402

DEV = "cuda:0"
DTYPES = [torch.float16, torch.bfloat16, torch.float32]
CODE = {torch.float16: F16, torch.bfloat16: BF16, torch.float32: F32}
INT_VIEW = {torch.float16: torch.int16, torch.bfloat16: torch.int16, torch.float32: torch.int32}
SENT = {torch.float16: 0x7E01, torch.bfloat16: 0x7F81, torch.float32: 0x7FC00001}   # NaN payloads no decoder writes


def _bits(t):
    return t.view(INT_VIEW[t.dtype])


def _i32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(DEV)


def _i64(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(DEV)


class Caches:
    """n caches of nb blocks of G elements, `mult` caches interleaved per parent tensor: block b of cache c is row
    b * mult + c % mult of parent c // mult (mult 2 = vLLM's [num_blocks, 2, ...] layout, stride 2G).  With `shift`
    every base sits 8 bytes past a 16-byte boundary.  Block 0 of every cache is zero, block 1 holds long runs."""

    def __init__(self, n, nb, G, dtype, mult=1, seed=0, shift=False):
        self.n, self.nb, self.G, self.dtype, self.mult = n, nb, G, dtype, mult
        gen = torch.Generator(device=DEV).manual_seed(seed)
        n_par = -(-n // mult)
        per = nb * mult * G
        pad = 8 // (torch.finfo(dtype).bits // 8) if shift else 0
        self.flat = torch.empty(n_par * per + pad, dtype=dtype, device=DEV)
        self.flat[pad:] = torch.randn(n_par * per, generator=gen, device=DEV).to(dtype)
        self.parents = [self.flat[pad + p * per: pad + (p + 1) * per].view(nb * mult, G) for p in range(n_par)]
        self.caches = [self.parents[c // mult].view(nb, mult, G)[:, c % mult] for c in range(n)]
        for c in self.caches:
            c[0].zero_()
            c[1, : G // 2] = 0.5
            c[1, G // 2:] = -0.25

    def ref(self, c, blocks):
        """(single-cache tensor, its block numbers) of blocks `blocks` of cache c"""
        return self.parents[c // self.mult], blocks * self.mult + c % self.mult

    def fill(self, code):
        for p in self.parents:
            p.view(INT_VIEW[self.dtype]).fill_(code)


def _pairs(rng, n, nb, k, must=()):
    """k distinct (cache, block) pairs in a random order (not cache-major), the pairs `must` among them"""
    must = [c * nb + b for c, b in must]
    flat = rng.permutation(np.concatenate([must, rng.permutation(np.setdiff1d(np.arange(n * nb), must))[: k - len(must)]]))
    return (flat // nb).astype(np.int32), (flat % nb).astype(np.int32)


def _assert_same_container(a, b):
    assert torch.equal(a.comp_bytes, b.comp_bytes)
    assert torch.equal(a.scales.view(torch.int32), b.scales.view(torch.int32))
    comp = a.comp_bytes.cpu().numpy()
    pa, pb = a.payload.cpu().numpy(), b.payload.cpu().numpy()
    for g in range(comp.size):
        assert np.array_equal(pa[g, :comp[g]], pb[g, :comp[g]]), f"payload of group {g}"


def _ref_compress(cs, ci, bt, scheme, lens=None):
    """The single-cache path cache by cache, reassembled in the order of the set call's groups."""
    n = ci.size
    sb = codec.slot_bytes(cs.G, scheme)
    out = codec.CompressedKV(torch.zeros((n, sb), dtype=torch.uint8, device=DEV),
                             torch.zeros(n, dtype=torch.float32, device=DEV),
                             torch.zeros(n, dtype=torch.int32, device=DEV), cs.G, cs.dtype, scheme)
    for c in np.unique(ci):
        idx = np.nonzero(ci == c)[0]
        t, blocks = cs.ref(c, bt[idx])
        if lens is None:
            r = codec.compress_gather(t, _i32(blocks), scheme=scheme)
        else:
            r = codec.compress_ragged(t, cs.G, lens[_i64(idx)], block_table=_i32(blocks), scheme=scheme)
        ii = _i64(idx)
        out.payload[ii] = r.payload
        out.scales[ii] = r.scales
        out.comp_bytes[ii] = r.comp_bytes
    return out


def _oracle_sample(cs, ci, bt, c_set, scheme, groups):
    for g in groups:
        x = cs.caches[ci[g]][bt[g]]
        raw = x.view(torch.int16).cpu().numpy().view(np.uint16) if cs.dtype == torch.bfloat16 else x.cpu().numpy()
        payload, scales, comp = Port.compress_batch(raw, cs.G, dtype=CODE[cs.dtype], scheme=scheme)
        assert int(c_set.comp_bytes[g]) == int(comp[0]), f"oracle comp_bytes, group {g}"
        assert np.float32(c_set.scales[g].item()).view(np.uint32) == scales.view(np.uint32)[0], f"oracle scale, group {g}"
        assert np.array_equal(c_set.payload[g, :comp[0]].cpu().numpy(), payload[0, :comp[0]]), f"oracle payload, group {g}"


@pytest.mark.parametrize("G,nb", [(2048, 24), (16384, 8), (131072, 3), (1000, 16)])
@pytest.mark.parametrize("mult", [1, 2])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("scheme", [1, 2, 3, 4])
def test_codec_set_matches_per_cache(G, nb, mult, dtype, scheme):
    rng = np.random.default_rng(G + 7 * mult + scheme)
    n = 3 + (G + scheme) % 5                                                  # 3-7 caches
    cs = Caches(n, nb, G, dtype, mult, seed=G + scheme)
    cset = KVCacheSet(cs.caches)
    assert cset.block_stride == mult * G and len(cset) == n
    ci, bt = _pairs(rng, n, nb, (n * nb * 3) // 4, must=[(0, 0), (n - 1, 1)])   # a zero block and a long-run block
    c_set = codec.compress_gather_set(cset, _i32(ci), _i32(bt), scheme=scheme)
    _assert_same_container(c_set, _ref_compress(cs, ci, bt, scheme))
    _oracle_sample(cs, ci, bt, c_set, scheme, [int(np.nonzero((ci == 0) & (bt == 0))[0][0]),
                                               int(np.nonzero((ci == n - 1) & (bt == 1))[0][0]), ci.size - 1])

    # ragged lengths, 0 and G included
    lens = _i32(np.concatenate([[0, G], rng.integers(0, G + 1, ci.size - 2)]))
    r_set = codec.compress_gather_set(cset, _i32(ci), _i32(bt), lengths=lens, scheme=scheme)
    _assert_same_container(r_set, _ref_compress(cs, ci, bt, scheme, lens))

    # scatter back into sentinel-filled caches: the set form against decompress_scatter cache by cache
    src = rng.permutation(ci.size).astype(np.int32)
    oel = torch.zeros(ci.size, dtype=torch.int32, device=DEV)
    cs.fill(SENT[dtype])
    codec.decompress_scatter_set(c_set, cset, _i32(ci), _i32(bt), src_index=_i32(src), out_elems=oel)
    got = _bits(cs.flat).clone()
    cs.fill(SENT[dtype])
    for c in np.unique(ci):
        idx = np.nonzero(ci == c)[0]
        t, blocks = cs.ref(c, bt[idx])
        codec.decompress_scatter(c_set, t, _i32(blocks), src_index=_i32(src[idx]))
    assert torch.equal(got, _bits(cs.flat))
    assert (oel == G).all()


@pytest.mark.parametrize("G", [2048, 16384])
@pytest.mark.parametrize("scheme", [1, 2])
def test_unaligned_set_takes_generic_kernels(G, scheme):
    rng = np.random.default_rng(G)
    cs = Caches(4, 6, G, torch.float16, 1, seed=3, shift=True)
    assert cs.caches[0].data_ptr() % 16 == 8
    cset = KVCacheSet(cs.caches)
    ci, bt = _pairs(rng, 4, 6, 20)
    c_set = codec.compress_gather_set(cset, _i32(ci), _i32(bt), scheme=scheme)
    _assert_same_container(c_set, _ref_compress(cs, ci, bt, scheme))
    cs.fill(SENT[torch.float16])
    codec.decompress_scatter_set(c_set, cset, _i32(ci), _i32(bt))
    got = _bits(cs.flat).clone()
    cs.fill(SENT[torch.float16])
    for c in np.unique(ci):
        idx = np.nonzero(ci == c)[0]
        t, blocks = cs.ref(c, bt[idx])
        codec.decompress_scatter(c_set, t, _i32(blocks), src_index=_i32(idx))
    assert torch.equal(got, _bits(cs.flat))


def _tier_for(cs, factor=3):
    return HostTier(pool_bytes=int(cs.flat.numel() * cs.flat.element_size() * factor) + (8 << 20))


@pytest.mark.parametrize("G,nb", [(2048, 32), (16384, 8)])
@pytest.mark.parametrize("mult", [1, 2])
@pytest.mark.parametrize("ragged", [False, True])
def test_tier_set_round_trip_and_mixed_forms(G, nb, mult, ragged):
    rng = np.random.default_rng(G + mult + 10 * ragged)
    n = 5
    cs = Caches(n, nb, G, torch.float16, mult, seed=G + mult)
    cset = KVCacheSet(cs.caches)
    tier = _tier_for(cs)
    try:
        ci, bt = _pairs(rng, n, nb, n * nb // 2)
        ids = rng.permutation(1 << 20)[: ci.size].astype(np.uint64) + np.uint64(1 << 33)
        lens = _i32(np.concatenate([[0, G], rng.integers(0, G + 1, ci.size - 2)])) if ragged else None
        tier.offload_set(cset, _i32(ci), _i32(bt), ids, lengths=lens)
        st = tier.stats()
        assert st["blocks"] == ci.size
        want_raw = int(lens.sum()) * 2 if ragged else ci.size * G * 2
        assert st["bytes_offloaded_raw"] == want_raw
        # the same blocks through the single-cache forms, under other ids
        ids2 = ids + np.uint64(1 << 40)
        for c in np.unique(ci):
            idx = np.nonzero(ci == c)[0]
            t, blocks = cs.ref(c, bt[idx])
            if ragged:
                tier.offload_ragged(t, G, lens[_i64(idx)], ids2[idx], block_table=_i32(blocks))
            else:
                tier.offload_blocks(t, _i32(blocks), ids2[idx])
        st2 = tier.stats()
        assert st2["blocks"] == 2 * ci.size and st2["used_bytes"] == 2 * st["used_bytes"]
        assert st2["bytes_offloaded_stored"] == 2 * st["bytes_offloaded_stored"]

        def restore_all(by_set, which):
            cs.fill(SENT[torch.float16])
            if by_set:
                tier.restore_set(which, cset, _i32(ci), _i32(bt))
            else:
                for c in np.unique(ci):
                    idx = np.nonzero(ci == c)[0]
                    t, blocks = cs.ref(c, bt[idx])
                    tier.restore_blocks(which[idx], t, _i32(blocks))
            torch.cuda.synchronize()
            return _bits(cs.flat).clone()

        want = restore_all(False, ids2)
        assert torch.equal(restore_all(True, ids), want)       # set -> set
        assert torch.equal(restore_all(False, ids), want)      # set -> single-cache
        assert torch.equal(restore_all(True, ids2), want)      # single-cache -> set
        assert tier.stats()["bytes_restored_raw"] == 4 * want_raw

    finally:
        tier.close()


def test_tier_set_duplicate_and_reoffload_ids():
    G, nb, n = 2048, 8, 3
    cs = Caches(n, nb, G, torch.bfloat16, 1, seed=5)
    cset = KVCacheSet(cs.caches)
    tier = _tier_for(cs)
    try:
        def decoded(c, b):   # what a block decodes to (the codec is lossy)
            return codec.decompress(codec.compress_gather_set(cset, _i32([c]), _i32([b])))[0]

        ids = np.array([11, 12, 11], dtype=np.uint64)                           # id 11 twice: the later block wins
        tier.offload_set(cset, _i32([0, 1, 2]), _i32([3, 4, 5]), ids)
        assert tier.stats()["blocks"] == 2
        want = decoded(2, 5)
        tier.offload_set(cset, _i32([1]), _i32([6]), np.array([12], dtype=np.uint64))   # re-offload id 12
        want12 = decoded(1, 6)
        cs.fill(SENT[torch.bfloat16])
        tier.restore_set(np.array([11, 12], dtype=np.uint64), cset, _i32([0, 0]), _i32([0, 1]))
        assert torch.equal(_bits(cs.caches[0][0]), _bits(want)) and torch.equal(_bits(cs.caches[0][1]), _bits(want12))
        assert torch.equal(_bits(cs.caches[0][2]), torch.full_like(_bits(want), SENT[torch.bfloat16]))
        st = tier.stats()
        assert st["blocks"] == 2
    finally:
        tier.close()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("scheme", [2, 4])
def test_fetch_set_graph_across_directory_growth(dtype, scheme):
    G, nb, n = 2048, 16, 4
    rng = np.random.default_rng(scheme)
    cs = Caches(n, nb, G, dtype, 2, seed=scheme)
    cset = KVCacheSet(cs.caches)
    tier = _tier_for(cs, factor=80)
    s = torch.cuda.Stream()
    try:
        with torch.cuda.stream(s):
            tier.set_scheme(scheme)
            ci, bt = _pairs(rng, n, nb, 24)
            ids = np.arange(ci.size, dtype=np.uint64) * np.uint64(7919) + np.uint64(3)
            tier.offload_set(cset, _i32(ci), _i32(bt), ids)
            tier.enable_fetch()
            d_ids, d_ci, d_bt = _i64(ids), _i32(ci), _i32(bt)
            count = _i32([ci.size - 4])                                          # device count: the last 4 stay put
            oel = torch.zeros(ci.size, dtype=torch.int32, device=DEV)
            st = torch.zeros(ci.size, dtype=torch.uint8, device=DEV)
            tier.fetch_set(d_ids, cset, d_ci, d_bt, scheme=scheme, count=count, out_elems=oel, status=st)
            s.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                tier.fetch_set(d_ids, cset, d_ci, d_bt, scheme=scheme, count=count, out_elems=oel, status=st)
            more = np.arange(3000, dtype=np.uint64) + np.uint64(1 << 30)
            tier.offload(torch.randn(3000 * G, device=DEV).to(dtype), G, more)   # the directory grows
            cs.fill(SENT[dtype])
            oel.zero_()
            st.zero_()
            g.replay()
            s.synchronize()
            got = _bits(cs.flat).clone()
            # reference: fetch with a block table, cache by cache
            cs.fill(SENT[dtype])
            k = ci.size - 4
            for c in np.unique(ci[:k]):
                idx = np.nonzero(ci[:k] == c)[0]
                t, blocks = cs.ref(c, bt[idx])
                tier.fetch(_i64(ids[idx]), G, dtype, scheme=scheme, out=t, block_table=_i32(blocks))
            s.synchronize()
            assert torch.equal(got, _bits(cs.flat))
            assert st.cpu().numpy().tolist() == [1] * k + [0] * 4
            assert (oel[:k] == G).all() and (oel[k:] == 0).all()
    finally:
        tier.close()


def test_fetch_set_unserved_requests_keep_sentinel():
    G, nb, n = 16384, 6, 3
    cs = Caches(n, nb, G, torch.float16, 1, seed=9)
    cset = KVCacheSet(cs.caches)
    other = torch.randn((4, 2048), device=DEV).half()
    tier = _tier_for(cs)
    try:
        tier.offload_set(cset, _i32([0, 1, 2]), _i32([2, 3, 4]), np.array([1, 2, 3], dtype=np.uint64))
        tier.offload(other, 2048, np.array([50, 51, 52, 53], dtype=np.uint64))   # another geometry
        tier.enable_fetch()
        cs.fill(SENT[torch.float16])
        # served, unknown id, cache index out of range, another geometry, served
        ids = _i64([1, 999, 2, 50, 3])
        ci = _i32([0, 1, 7, 2, 2])
        bt = _i32([0, 1, 2, 3, 4])
        oel, st = tier.fetch_set(ids, cset, ci, bt)
        torch.cuda.synchronize()
        assert st.cpu().numpy().tolist() == [1, 0, 0, 0, 1]
        assert oel.cpu().numpy().tolist() == [G, 0, 0, 0, G]
        sent = torch.full((G,), SENT[torch.float16], dtype=torch.int16, device=DEV)
        for c, b in ((1, 1), (2, 3)):
            assert torch.equal(_bits(cs.caches[c][b]), sent)
        flat_sent = (_bits(cs.flat) == SENT[torch.float16]).view(n, nb, G).all(-1)
        want = torch.ones((n, nb), dtype=torch.bool, device=DEV)
        want[0, 0] = want[2, 4] = False
        assert torch.equal(flat_sent, want)
    finally:
        tier.close()


@pytest.mark.parametrize("layout", ["2nb", "nb2"])
@pytest.mark.parametrize("ragged", [False, True])
def test_allocator_register_offload_restore_request(layout, ragged):
    layers, nb, bs, heads, dim = 3, 12, 16, 8, 128
    shape = (2, nb, bs, heads, dim) if layout == "2nb" else (nb, 2, bs, heads, dim)
    gen = torch.Generator(device=DEV).manual_seed(1)
    kv = {f"model.layers.{i}.attn": torch.randn(shape, generator=gen, device=DEV).half() for i in range(layers)}
    alloc = CxlSpeckvKVAllocator(pkg.lib_path(), "cuda:0")
    try:
        _check_request_path(alloc, kv, layout, ragged, bs, heads, dim, layers)
    finally:
        alloc._speckv.finalize()


def _check_request_path(alloc, kv, layout, ragged, bs, heads, dim, layers):
    cset = alloc.register_kv_caches(kv)
    G = bs * heads * dim
    assert len(cset) == 2 * layers and cset.block_elems == G
    assert cset.block_stride == (G if layout == "2nb" else 2 * G)
    table = _i32([7, 2, 9, 4])
    num_tokens = [0, 16, 5, 11] if ragged else None
    tier = HostTier(pool_bytes=64 << 20)
    try:
        alloc.offload_request(table, tier, num_tokens=num_tokens)
        ids = alloc.request_block_ids(table)
        assert ids.shape == (2 * layers, 4) and int(ids[3, 2]) == (3 << 40) | 9
        # the per-layer path: offload_kv_blocks on every K / V view under the same ids, restored through it
        views = [v for kvt in kv.values() for v in ((kvt[0], kvt[1]) if layout == "2nb" else (kvt[:, 0], kvt[:, 1]))]
        want = []
        for c, v in enumerate(views):
            x = torch.empty_like(v, memory_format=torch.contiguous_format).copy_(v)
            CxlSpeckvKVAllocator.offload_kv_blocks(x, table, tier, block_ids=ids[c] + np.uint64(1 << 60),
                                                   num_tokens=num_tokens)
            x.view(torch.int16).fill_(SENT[torch.float16])
            CxlSpeckvKVAllocator.restore_kv_blocks(x, table, tier, block_ids=ids[c] + np.uint64(1 << 60))
            want.append(x)
        for t in kv.values():
            t.view(torch.int16).fill_(SENT[torch.float16])
        alloc.restore_request(table, tier)
        torch.cuda.synchronize()
        for c, v in enumerate(views):
            assert torch.equal(_bits(v), _bits(want[c])), f"cache {c}"
    finally:
        tier.close()


def test_set_argument_checks():
    cs = Caches(3, 4, 2048, torch.float16, 1)
    cset = KVCacheSet(cs.caches)
    ci, bt = _i32([0, 1]), _i32([0, 1])
    with pytest.raises(SpeckvError):
        codec.compress_gather_set(cset, ci, bt, scheme=0)                       # no gather form of the raw scheme
    c = codec.compress_gather_set(cset, ci, bt)
    with pytest.raises(SpeckvError):
        codec.decompress_scatter_set(codec.CompressedKV(c.payload, c.scales, c.comp_bytes, 2048, torch.float16, 0),
                                     cset, ci, bt)
    L = pkg.lib()
    h = cset.handle()
    assert L.speckv_ext_compress_gather_set(h, None, bt.data_ptr(), None, 2, c.payload.data_ptr(), c.payload.shape[1],
                                            c.scales.data_ptr(), c.comp_bytes.data_ptr(), 2, None) == pkg.SPECKV_ERR_INVAL
    assert L.speckv_ext_compress_gather_set(None, ci.data_ptr(), bt.data_ptr(), None, 2, c.payload.data_ptr(),
                                            c.payload.shape[1], c.scales.data_ptr(), c.comp_bytes.data_ptr(), 2,
                                            None) == pkg.SPECKV_ERR_INVAL
    assert L.speckv_ext_decompress_scatter_set(c.payload.data_ptr(), c.payload.shape[1], c.scales.data_ptr(),
                                               c.comp_bytes.data_ptr(), None, h, ci.data_ptr(), None, 2, None, 2,
                                               None) == pkg.SPECKV_ERR_INVAL
    # each rejected argument on its own; an empty call checks no index array, but the raw scheme is refused even then
    buf = dict(h=h, ci=ci.data_ptr(), bt=bt.data_ptr(), n=2, p=c.payload.data_ptr(), sb=c.payload.shape[1],
               s=c.scales.data_ptr(), cb=c.comp_bytes.data_ptr(), scheme=2)
    codec_calls = {
        "gather_set": lambda a: L.speckv_ext_compress_gather_set(a["h"], a["ci"], a["bt"], None, a["n"], a["p"], a["sb"],
                                                                 a["s"], a["cb"], a["scheme"], None),
        "scatter_set": lambda a: L.speckv_ext_decompress_scatter_set(a["p"], a["sb"], a["s"], a["cb"], None, a["h"],
                                                                     a["ci"], a["bt"], a["n"], None, a["scheme"], None),
    }
    for name, call in codec_calls.items():
        for bad_arg in [dict(h=None), dict(ci=None), dict(bt=None), dict(scheme=0), dict(scheme=5), dict(sb=16),
                        dict(p=None), dict(s=None), dict(cb=None), dict(p=c.payload.data_ptr() + 8)]:
            assert call({**buf, **bad_arg}) == pkg.SPECKV_ERR_INVAL, (name, bad_arg)
        assert call({**buf, "n": 0, "scheme": 0}) == pkg.SPECKV_ERR_INVAL, name
        assert call({**buf, "n": 0, "ci": None, "bt": None, "p": None, "s": None, "cb": None}) == pkg.SPECKV_OK, name
    lens = _i32([5, 7])
    with pytest.raises(TypeError):
        codec.compress_gather_set(cset, ci, bt, lengths=lens.long())
    with pytest.raises(ValueError):
        codec.compress_gather_set(cset, ci, bt, lengths=lens[:1])
    with pytest.raises(ValueError):
        codec.compress_gather_set(cset, ci[:1], bt)
    with pytest.raises(TypeError):
        codec.compress_gather_set(cs.caches, ci, bt)
    with pytest.raises(ValueError):
        codec.decompress_scatter_set(c, cset, ci, bt, src_index=_i32([0]))
    with pytest.raises(ValueError):
        codec.decompress_scatter_set(c, cset, ci[:1], bt[:1])
    tier = HostTier(pool_bytes=8 << 20)
    try:
        ids = np.array([1, 2], dtype=np.uint64)
        assert L.speckv_ext_tier_offload_set(tier._h, h, None, bt.data_ptr(), None, 2, ids.ctypes.data,
                                             None) == pkg.SPECKV_ERR_INVAL
        assert L.speckv_ext_tier_restore_set(tier._h, ids.ctypes.data, 2, h, ci.data_ptr(), None,
                                             None) == pkg.SPECKV_ERR_INVAL
        tbuf = dict(t=tier._h, h=h, ci=ci.data_ptr(), bt=bt.data_ptr(), n=2, ids=ids.ctypes.data)
        tier_calls = {
            "offload_set": lambda a: L.speckv_ext_tier_offload_set(a["t"], a["h"], a["ci"], a["bt"], None, a["n"],
                                                                   a["ids"], None),
            "restore_set": lambda a: L.speckv_ext_tier_restore_set(a["t"], a["ids"], a["n"], a["h"], a["ci"], a["bt"],
                                                                   None),
        }
        for name, call in tier_calls.items():
            for bad_arg in [dict(t=None), dict(h=None), dict(ci=None), dict(bt=None), dict(ids=None)]:
                assert call({**tbuf, **bad_arg}) == pkg.SPECKV_ERR_INVAL, (name, bad_arg)
            assert call({**tbuf, "n": 0, "ci": None, "bt": None}) == pkg.SPECKV_OK, name
        with pytest.raises(ValueError):
            tier.offload_set(cset, ci, bt, ids[:1])
        with pytest.raises(ValueError):
            tier.offload_set(cset, ci, bt, ids, lengths=lens[:1])
        with pytest.raises(ValueError):
            tier.offload_set(cset, ci, bt, ids, lengths=_i32([5, -1]))        # would store the whole block
        with pytest.raises(ValueError):
            tier.restore_set(ids[:1], cset, ci, bt)
        dids = torch.from_numpy(ids.astype(np.int64)).to(DEV)
        need = L.speckv_ext_tier_fetch_workspace_bytes(2, 2048)
        ws = torch.empty(need, dtype=torch.uint8, device=DEV)
        fbuf = dict(t=tier._h, ids=dids.data_ptr(), n=2, h=h, ci=ci.data_ptr(), bt=bt.data_ptr(), scheme=2,
                    ws=ws.data_ptr(), wsb=need)

        def fetch_set(a):
            return L.speckv_ext_tier_fetch_set(a["t"], a["ids"], None, a["n"], a["h"], a["ci"], a["bt"], a["scheme"],
                                               None, None, a["ws"], a["wsb"], None)

        assert fetch_set(fbuf) == pkg.SPECKV_ERR_INVAL                                # before enable_fetch
        tier.enable_fetch()
        for bad_arg in [dict(t=None), dict(h=None), dict(ci=None), dict(bt=None), dict(ids=None), dict(scheme=0),
                        dict(scheme=5), dict(ws=None), dict(ws=ws.data_ptr() + 8), dict(wsb=need - 1),
                        dict(n=1 << 31)]:
            assert fetch_set({**fbuf, **bad_arg}) == pkg.SPECKV_ERR_INVAL, bad_arg
        assert fetch_set({**fbuf, "n": 0, "ids": None, "ci": None, "bt": None, "ws": None}) == pkg.SPECKV_OK
        with pytest.raises(TypeError):
            tier.fetch_set(dids.int(), cset, ci, bt)
        with pytest.raises(TypeError):
            tier.fetch_set(dids, cset, ci[:1], bt)
        with pytest.raises(TypeError):
            tier.fetch_set(dids, cset, ci, bt.long())
        with pytest.raises(TypeError):
            tier.fetch_set(dids, cset, ci, bt, count=torch.ones(1, dtype=torch.int64, device=DEV))
        tier.set_scheme(0)
        with pytest.raises(SpeckvError):
            tier.offload_set(cset, ci, bt, ids)                                 # raw passthrough: no gather form
    finally:
        tier.close()
    import ctypes as C
    out = C.c_void_p()
    bases = (C.c_void_p * 1)(cs.caches[0].data_ptr())
    assert L.speckv_ext_cache_set_create(bases, 1, 2048, 1024, 0, C.byref(out)) == pkg.SPECKV_ERR_INVAL   # stride < block
    with pytest.raises(ValueError):
        KVCacheSet([cs.caches[0], cs.caches[1][:2]])
