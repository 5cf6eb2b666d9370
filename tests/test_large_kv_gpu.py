"""GPU parity tests of the codec and the host tier on KV caches past 4 GiB.

A vLLM paged KV cache fills most of the device, so the entry points that address cache blocks (paged gather /
scatter, ragged compress with a block table, the host tier's paged offload / restore / fetch) and the dense calls
that cover a whole cache work at element offsets past 2^31, byte offsets past 2^32 and slot containers larger than
4 GiB.  These tests run every such entry point there.  Only the groups under test travel to the host; the groups
are picked by where they sit:
  - the group that ends just below each boundary and the one that starts at or after it,
  - for a geometry that does not divide the boundary (G = 6000), the group that straddles it,
  - the last group, and a seeded sample.
Boundaries: 2^31 elements, 2^31 and 2^32 bytes of the input / output elements and of the slot container.  Every
assertion names the boundary its group sits at.

Bar: scales, comp_bytes, payload bytes [:comp_bytes], out_elems and decoded bits equal the oracle's
(oracle.oracle.Port) on exactly those groups; outputs go into sentinel-filled buffers, and a block a call must not
write keeps its sentinel.

The frozen API part: pool pages past 4 GiB of one speckv_alloc are stored in the host tier under their own ids
(PageTable::tier_key), so they neither replace another page's stored copy nor leave with another handle's blocks.

Each test checks the free device memory it needs first and skips, naming the amount, when it is not there.  Two
4 GiB buffers (a source cache and a sentinel destination) are shared by the tests of this file and released at
its end; the largest case adds a slot container of 4 GiB."""
import ctypes as C
import gc

import numpy as np
import pytest
import torch

from oracle.oracle import Port
from tests.helpers import BF16, F16, F32, bf16_from_f32, f32_bits

pytestmark = pytest.mark.gpu

import cxl_speckv_b200 as pkg  # noqa: E402
from cxl_speckv_b200 import codec  # noqa: E402
from cxl_speckv_b200.tier import HostTier  # noqa: E402
from cxl_speckv_b200.vllm_speckv_backend import CxlSpeckvKVAllocator  # noqa: E402
from tests.test_codec_paths_gpu import CLASSES, class_group  # noqa: E402

DEV = "cuda:0"
GIB = 1 << 30
E31 = 1 << 31                     # elements
B31, B32 = 1 << 31, 1 << 32       # bytes
BIG_BYTES = B32 + (2 << 20)       # the shared buffers: 4 GiB + 2 MiB
TORCH_DT = {F16: torch.float16, BF16: torch.bfloat16, F32: torch.float32}
ESZ = {F16: 2, BF16: 2, F32: 4}
DT_NAME = {F16: "f16", BF16: "bf16", F32: "f32"}
SENT16, SENT32 = 0x1234, 0x3F9E0419   # patterns no decode of these inputs produces by chance
SENT_WORD = 0x5A5A5A5A
GEOMETRIES = (131072, 2048, 16384, 6000)   # tuned R = 64, tuned R = 1 (pages), the vLLM block, generic


# ---- memory ------------------------------------------------------------------------------------------------------
class _Big:
    """The two shared 4 GiB buffers: `src` holds the cache under test (content keyed by (G, dtype)), `dst` is the
    sentinel destination of decodes."""
    src = None
    dst = None
    key = None
    marks = None

    @classmethod
    def held(cls):
        return sum(b.numel() for b in (cls.src, cls.dst) if b is not None)

    @classmethod
    def release(cls):
        cls.src = cls.dst = cls.key = cls.marks = None
        gc.collect()
        torch.cuda.empty_cache()


@pytest.fixture(scope="module", autouse=True)
def _release_buffers():
    yield
    _Big.release()


@pytest.fixture(autouse=True)
def _free_between_cases():
    yield
    gc.collect()
    torch.cuda.empty_cache()


def need(nbytes, what):
    """Skip unless nbytes of device memory are free (the shared buffers this file already holds count as free)."""
    free, _ = torch.cuda.mem_get_info()
    have = free + _Big.held()
    if have < nbytes:
        pytest.skip(f"{what} needs {nbytes / GIB:.1f} GiB of free device memory, {have / GIB:.1f} GiB available")


def _buffer(name):
    b = getattr(_Big, name)
    if b is None:
        b = torch.empty(BIG_BYTES, dtype=torch.uint8, device=DEV)
        setattr(_Big, name, b)
    return b


# ---- which groups ------------------------------------------------------------------------------------------------
def around(marks, bound_units, unit, n_groups, label):
    """Groups at a boundary bound_units (counted in `unit`s, the size of one group): the one ending just below, the
    one starting at or after it, and the one straddling it when the geometry does not divide it."""
    g, rem = divmod(bound_units, unit)
    picks = ((g - 1, "ends below"), (g, "straddles" if rem else "starts at"))
    if rem:
        picks += ((g + 1, "starts after"),)
    for gg, how in picks:
        if 0 <= gg < n_groups:
            marks.setdefault(gg, []).append(f"{how} {label}")


def element_marks(G, esz, n_groups):
    marks = {}
    around(marks, E31, G, n_groups, "2^31 elements")
    for b, name in ((B31, "2^31"), (B32, "2^32")):
        if b % esz == 0:
            around(marks, b // esz, G, n_groups, f"{name} bytes")
    return marks


def slot_marks(sb, n_groups):
    marks = {}
    for b, name in ((B31, "2^31"), (B32, "2^32")):
        around(marks, b, sb, n_groups, f"{name} container bytes")
    return marks


def finish_marks(marks, n_groups, seed, n_sample=3):
    marks = {g: list(v) for g, v in marks.items()}
    marks.setdefault(n_groups - 1, []).append("last")
    rng = np.random.default_rng(seed)
    for g in rng.choice(n_groups, n_sample, replace=False):
        marks.setdefault(int(g), []).append("sample")
    return dict(sorted(marks.items()))


def label(marks, g):
    return f"group {g} ({', '.join(marks[g])})"


# ---- device <-> host ---------------------------------------------------------------------------------------------
def raw_rows(t2d, groups, tdt):
    """The stored elements of rows `groups` of a [n, G] device tensor: np.float16 / bf16 bits (uint16) / np.float32."""
    rows = t2d[torch.as_tensor(np.asarray(groups, np.int64), device=DEV)]
    if tdt == BF16:
        return rows.view(torch.int16).cpu().numpy().view(np.uint16)
    return rows.cpu().numpy()


def bit_rows(t2d, groups, tdt):
    rows = t2d[torch.as_tensor(np.asarray(groups, np.int64), device=DEV)]
    if tdt == F32:
        return rows.view(torch.int32).cpu().numpy().view(np.uint32)
    return rows.view(torch.int16).cpu().numpy().view(np.uint16)


def to_dev(raw, tdt):
    raw = np.ascontiguousarray(raw)
    if tdt == BF16:
        return torch.from_numpy(raw.view(np.int16)).to(DEV).view(torch.bfloat16)
    return torch.from_numpy(raw).to(DEV)


def narrow(x, tdt):
    if tdt == F16:
        with np.errstate(over="ignore", invalid="ignore"):
            return x.astype(np.float16)
    if tdt == BF16:
        return bf16_from_f32(x.reshape(-1)).reshape(x.shape)
    return x.astype(np.float32)


def sent_value(tdt):
    return np.uint32(SENT32) if tdt == F32 else np.uint16(SENT16)


def fill_sentinel(t, tdt):
    (t.view(torch.int32) if tdt == F32 else t.view(torch.int16)).fill_(SENT32 if tdt == F32 else SENT16)
    return t


def sentinel(shape, tdt):
    return fill_sentinel(torch.empty(shape, dtype=TORCH_DT[tdt], device=DEV), tdt)


def changed_blocks(t2d, tdt, chunk=1 << 28):
    """Blocks of a sentinel-filled [n, G] tensor that hold anything else (chunked: no 4 GiB temporary)."""
    G = t2d.shape[1]
    w = t2d.view(torch.int32) if tdt == F32 else t2d.view(torch.int16)
    s = SENT32 if tdt == F32 else SENT16
    rows = max(1, chunk // G)
    out = []
    for r0 in range(0, t2d.shape[0], rows):
        hit = (w[r0:r0 + rows] != s).any(dim=1).nonzero().flatten()
        out.append(hit + r0)
    return set(torch.cat(out).cpu().tolist())


# ---- oracle ------------------------------------------------------------------------------------------------------
def oracle_encode(raw, G, tdt, scheme):
    """-> (payload [n, sb], scales, comp) of the groups in raw [n, G] (scheme 0: the raw passthrough)."""
    sb = codec.slot_bytes(G, scheme)
    if scheme == 0:
        n = raw.shape[0]
        payload = np.zeros((n, sb), np.uint8)
        payload[:, :2 * G] = np.ascontiguousarray(raw).view(np.uint8).reshape(n, 2 * G)
        return payload, np.ones(n, np.float32), np.full(n, 2 * G, np.uint32)
    return Port.compress_batch(np.ascontiguousarray(raw).reshape(-1), G, dtype=tdt, slot_bytes=sb, threads=8,
                               scheme=scheme)


def oracle_decode(payload, scales, comp, G, tdt, scheme):
    """-> (element bits [n, G] with everything past out_elems set to the sentinel, out_elems)."""
    if scheme == 0:
        n = payload.shape[0]
        want = payload[:, :2 * G].copy().view(np.uint16).reshape(n, G)
        return want, np.full(n, G, np.uint32)
    want, want_n = Port.decompress_batch(payload, scales, comp, G, tdt, threads=8, scheme=scheme)
    want = want.view(np.uint32 if tdt == F32 else np.uint16).reshape(-1, G)
    return np.where(np.arange(G)[None, :] < want_n[:, None], want, sent_value(tdt)), want_n


def oracle_prefix(raw, lengths, G, tdt, scheme):
    """Port on raw[i, :n_i]: (scale bits, comp_bytes, payloads) and the decode of each prefix, sentinel behind it."""
    sc, cb, pl = [], [], []
    dec = np.full((len(lengths), G), sent_value(tdt))
    for i, n in enumerate(lengths):
        n = min(n, G)
        if n == 0:
            sc.append(np.float32(1.0))
            cb.append(0)
            pl.append(np.zeros(0, np.uint8))
            continue
        p, s, c = Port.compress_batch(np.ascontiguousarray(raw[i, :n]), n, dtype=tdt, scheme=scheme)
        sc.append(s[0])
        cb.append(int(c[0]))
        pl.append(p[0, :c[0]].copy())
        d, _ = Port.decompress_batch(p, s, c, n, tdt, scheme=scheme)
        dec[i, :n] = d.view(np.uint32 if tdt == F32 else np.uint16).reshape(-1)
    return f32_bits(np.array(sc, np.float32)), np.array(cb, np.uint32), pl, dec


def assert_container(c, rows, want, tags):
    """Groups `rows` of the device container c equal the oracle's groups (want = payload, scales, comp)."""
    payload, scales, comp = want
    idx = torch.as_tensor(np.asarray(rows, np.int64), device=DEV)
    got_s = f32_bits(c.scales[idx].cpu().numpy())
    got_c = c.comp_bytes[idx].cpu().numpy().view(np.uint32)
    got_p = c.payload[idx].cpu().numpy()
    for i, tag in enumerate(tags):
        assert got_s[i] == f32_bits(scales)[i], (tag, "scale", hex(got_s[i]), hex(f32_bits(scales)[i]))
        assert got_c[i] == comp[i], (tag, "comp_bytes", int(got_c[i]), int(comp[i]))
        n = int(comp[i])
        bad = np.flatnonzero(got_p[i, :n] != payload[i, :n])
        assert bad.size == 0, (tag, "payload bytes differ from", int(bad[0]) if bad.size else None)


def assert_bits(got, want, tags):
    for i, tag in enumerate(tags):
        bad = np.flatnonzero(got[i] != want[i])
        assert bad.size == 0, (tag, f"{bad.size} elements differ, first at {int(bad[0]) if bad.size else None}",
                               hex(int(got[i][bad[0]])) if bad.size else None, hex(int(want[i][bad[0]])) if bad.size else None)


def assert_touched(t2d, tdt, expect, what):
    touched = changed_blocks(t2d, tdt)
    assert touched == set(expect), (what, "blocks written outside the table", sorted(touched - set(expect))[:8],
                                    "named blocks left untouched", sorted(set(expect) - touched)[:8])


# ---- the source cache --------------------------------------------------------------------------------------------
def source(G, tdt):
    """The shared source buffer as a [n_blocks, G] cache of tdt past 4 GiB: N(0, 1) everywhere, the blocks at the
    element boundaries hold the codec's group classes (runs, zero tails, inf, tiny, outliers, ...).
    -> (cache, element-boundary marks)."""
    esz = ESZ[tdt]
    nb = BIG_BYTES // (G * esz)
    buf = _buffer("src")
    cache = buf[: nb * G * esz].view(TORCH_DT[tdt]).view(nb, G)
    if _Big.key != (G, tdt):
        _Big.key = None
        torch.manual_seed(G * 7 + tdt)
        cache.normal_()
        marks = element_marks(G, esz, nb)
        rng = np.random.default_rng(G * 31 + tdt)
        groups = sorted(marks)
        x = np.stack([class_group(rng, CLASSES[i % len(CLASSES)], G, tdt if tdt != F32 else F16)
                      for i in range(len(groups))])
        cache[torch.as_tensor(groups, device=DEV)] = to_dev(narrow(x, tdt), tdt)
        _Big.key, _Big.marks = (G, tdt), marks
    return cache, _Big.marks


def destination(nb, G, tdt):
    """The shared destination buffer as a sentinel-filled [nb, G] cache of tdt."""
    esz = ESZ[tdt]
    t = _buffer("dst")[: nb * G * esz].view(TORCH_DT[tdt]).view(nb, G)
    return fill_sentinel(t, tdt)


def case_id(G, tdt, scheme):
    return f"G{G}-{DT_NAME[tdt]}-s{scheme}"


# ---- 1. dense: one call over more than 2^31 elements ---------------------------------------------------------------
DENSE = [(G, tdt, s) for G in GEOMETRIES for tdt in (F16, BF16, F32) for s in range(5) if not (s == 0 and tdt == F32)]


@pytest.mark.parametrize("G,tdt,scheme", DENSE, ids=[case_id(*c) for c in DENSE])
def test_dense_call_past_2e31_elements(G, tdt, scheme):
    """compress then decompress of one flat tensor of more than 2^31 elements (16-bit types) or 2^32 bytes (fp32),
    then decompress_indexed / decompress_routed of the boundary groups into a small output."""
    esz = ESZ[tdt]
    n_groups = (E31 if esz == 2 else B32 // esz) // G + 2
    sb = codec.slot_bytes(G, scheme)
    need(2 * BIG_BYTES + n_groups * sb + (64 << 20), "the dense case")
    cache, emarks = source(G, tdt)
    x = cache[:n_groups]
    assert x.numel() * esz > B32 - 1 and (esz == 4 or x.numel() > E31)
    marks = {g: v for g, v in emarks.items() if g < n_groups}
    for g, v in slot_marks(sb, n_groups).items():
        marks.setdefault(g, []).extend(v)
    marks = finish_marks(marks, n_groups, seed=G + scheme)
    groups = list(marks)
    tags = [f"{case_id(G, tdt, scheme)} {label(marks, g)}" for g in groups]
    raw = raw_rows(x, groups, tdt)
    want = oracle_encode(raw, G, tdt, scheme)
    want_bits, want_n = oracle_decode(*want, G, tdt, scheme)

    c = codec.compress(x.reshape(-1), G, scheme=scheme)
    assert c.payload.numel() == n_groups * sb
    assert_container(c, groups, want, [t + " compress" for t in tags])

    out = destination(n_groups, G, tdt)
    oel = torch.full((n_groups,), SENT_WORD, dtype=torch.int32, device=DEV)
    codec.decompress(c, out=out, out_elems=oel)
    got_n = oel[torch.as_tensor(groups, device=DEV)].cpu().numpy().view(np.uint32)
    assert np.array_equal(got_n, want_n), (tags, got_n, want_n)
    assert_bits(bit_rows(out, groups, tdt), want_bits, [t + " decompress" for t in tags])
    out = None

    # requests naming the boundary groups, shuffled, one of them twice, into a small sentinel output
    rng = np.random.default_rng(G * 5 + scheme)
    order = rng.permutation(len(groups))
    order = np.concatenate([order, order[:1]])
    src = torch.as_tensor(np.asarray(groups, np.int64)[order].astype(np.int32), device=DEV)
    small = sentinel((len(order), G), tdt)
    codec.decompress_indexed(c, src, out=small)
    assert_bits(bit_rows(small, range(len(order)), tdt), want_bits[order],
                [tags[i] + " decompress_indexed" for i in order])

    routed = sentinel((len(order) + 2, G), tdt)
    count = torch.tensor([len(order) - 1], dtype=torch.int32, device=DEV)
    srcr = torch.cat([src, torch.zeros(2, dtype=torch.int32, device=DEV)])
    codec.decompress_routed(c, srcr, count, out=routed)
    got = bit_rows(routed, range(len(order) + 2), tdt)
    assert_bits(got[:len(order) - 1], want_bits[order[:-1]], [tags[i] + " decompress_routed" for i in order[:-1]])
    assert (got[len(order) - 1:] == sent_value(tdt)).all(), (case_id(G, tdt, scheme), "routed wrote at or past the count")


# ---- 2. decode from slots past 4 GiB, every scheme ---------------------------------------------------------------
SLOTS = [(G, tdt, s) for G in (131072, 2048, 6000) for tdt in (F16, BF16, F32) for s in range(5)
         if not (s == 0 and tdt == F32)]


@pytest.mark.parametrize("G,tdt,scheme", SLOTS, ids=[case_id(*c) for c in SLOTS])
def test_indexed_and_routed_decode_from_slots_past_4gib(G, tdt, scheme):
    """A container of more than 4 GiB of slots (also under the codes-only schemes, whose dense container stays near
    2 GiB at 2^31 elements) holding the oracle's payloads at the slots around 2^31 and 2^32 bytes and the last one:
    decompress_indexed and decompress_routed of those slots into a small sentinel output."""
    sb = codec.slot_bytes(G, scheme)
    n_slots = B32 // sb + 3
    need(n_slots * sb + (64 << 20), "the slot container")
    marks = finish_marks(slot_marks(sb, n_slots), n_slots, seed=G * 3 + scheme, n_sample=2)
    groups = list(marks)
    tags = [f"{case_id(G, tdt, scheme)} slot {label(marks, g)}" for g in groups]
    rng = np.random.default_rng(G * 11 + scheme + 100 * tdt)
    x = np.stack([class_group(rng, CLASSES[i % len(CLASSES)], G, tdt if tdt != F32 else F16) for i in range(len(groups))])
    want = oracle_encode(narrow(x, tdt), G, tdt, scheme)
    want_bits, want_n = oracle_decode(*want, G, tdt, scheme)

    c = codec.CompressedKV(torch.empty((n_slots, sb), dtype=torch.uint8, device=DEV),
                           torch.ones(n_slots, dtype=torch.float32, device=DEV),
                           torch.zeros(n_slots, dtype=torch.int32, device=DEV), G, TORCH_DT[tdt], scheme)
    assert c.payload.numel() > B32
    idx = torch.as_tensor(groups, device=DEV)
    c.payload[idx] = torch.from_numpy(want[0]).to(DEV)
    c.scales[idx] = torch.from_numpy(want[1]).to(DEV)
    c.comp_bytes[idx] = torch.from_numpy(want[2].view(np.int32)).to(DEV)

    order = np.concatenate([np.arange(len(groups))[::-1], [0]])
    src = torch.as_tensor(np.asarray(groups, np.int64)[order].astype(np.int32), device=DEV)
    small = sentinel((len(order), G), tdt)
    codec.decompress_indexed(c, src, out=small)
    assert_bits(bit_rows(small, range(len(order)), tdt), want_bits[order], [tags[i] + " indexed" for i in order])

    routed = sentinel((len(order), G), tdt)
    count = torch.tensor([len(order) - 1], dtype=torch.int32, device=DEV)
    codec.decompress_routed(c, src, count, out=routed)
    got = bit_rows(routed, range(len(order)), tdt)
    assert_bits(got[:-1], want_bits[order[:-1]], [tags[i] + " routed" for i in order[:-1]])
    assert (got[-1] == sent_value(tdt)).all(), (case_id(G, tdt, scheme), "routed wrote past the count")


# ---- 3. paged: a cache past 4 GiB through a block table ------------------------------------------------------------
PAGED = [(G, tdt, s) for G in GEOMETRIES for tdt in (F16, BF16, F32) for s in (1, 2, 3, 4)]


def table_for(marks, nb, seed):
    """Every marked block plus a sample, shuffled, the first one named twice at the end -> (table, marks)."""
    marks = finish_marks(marks, nb, seed)
    rng = np.random.default_rng(seed)
    blocks = rng.permutation(np.asarray(list(marks), np.int64))
    return np.concatenate([blocks, blocks[:1]]), marks


def restore_targets(table, nb):
    """Distinct destination blocks for the entries of `table`: the same high blocks rotated by one (no block comes
    back where it was read), and for the duplicate entry the highest block the table does not name."""
    named = set(table.tolist())
    spare = next(b for b in range(nb - 1, 0, -1) if b not in named)
    return np.concatenate([np.roll(table[:-1], 1), [spare]])


def mixed_lengths(n, G):
    """0, a partial block and a whole one, in turn."""
    return [(0, G // 3 + 5, G)[i % 3] for i in range(n)]


@pytest.mark.parametrize("G,tdt,scheme", PAGED, ids=[case_id(*c) for c in PAGED])
def test_paged_cache_past_4gib(G, tdt, scheme):
    """compress_gather and compress_ragged (mixed lengths) through a block table naming the boundary blocks of a cache
    past 4 GiB; decompress_scatter of the oracle's container into those blocks of another such cache, which keeps
    its sentinel everywhere else."""
    esz = ESZ[tdt]
    need(2 * BIG_BYTES + (64 << 20), "the paged case")
    cache, emarks = source(G, tdt)
    nb = cache.shape[0]
    table, marks = table_for(emarks, nb, seed=G * 13 + scheme)
    tags = [f"{case_id(G, tdt, scheme)} block {label(marks, int(b))}" for b in table]
    raw = raw_rows(cache, table, tdt)
    want = oracle_encode(raw, G, tdt, scheme)
    tdev = torch.as_tensor(table.astype(np.int32), device=DEV)

    cg = codec.compress_gather(cache, tdev, scheme=scheme)
    assert_container(cg, range(len(table)), want, [t + " compress_gather" for t in tags])

    lengths = mixed_lengths(len(table), G)
    sbits, comp, pl, dec = oracle_prefix(raw, lengths, G, tdt, scheme)
    lens = torch.tensor(lengths, dtype=torch.int32, device=DEV)
    cr = codec.compress_ragged(cache.view(-1), G, lens, block_table=tdev, scheme=scheme)
    got_s = f32_bits(cr.scales.cpu().numpy())
    got_c = cr.comp_bytes.cpu().numpy().view(np.uint32)
    got_p = cr.payload.cpu().numpy()
    for i, tag in enumerate(tags):
        t = f"{tag} compress_ragged n={lengths[i]}"
        assert got_s[i] == sbits[i], (t, "scale")
        assert got_c[i] == comp[i], (t, "comp_bytes", int(got_c[i]), int(comp[i]))
        assert np.array_equal(got_p[i, :pl[i].size], pl[i]), (t, "payload")

    # scatter: request i decodes stored block i into destination block dst[i] (distinct blocks, shuffled again)
    dst_blocks = np.random.default_rng(G + scheme).permutation(np.unique(table))
    n = dst_blocks.size
    c = codec.CompressedKV(torch.from_numpy(want[0][:n]).to(DEV), torch.from_numpy(want[1][:n]).to(DEV),
                           torch.from_numpy(want[2][:n].view(np.int32)).to(DEV), G, TORCH_DT[tdt], scheme)
    want_bits, want_n = oracle_decode(want[0][:n], want[1][:n], want[2][:n], G, tdt, scheme)
    out = destination(nb, G, tdt)
    oel = torch.full((n,), SENT_WORD, dtype=torch.int32, device=DEV)
    codec.decompress_scatter(c, out, torch.as_tensor(dst_blocks.astype(np.int32), device=DEV), out_elems=oel)
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n), case_id(G, tdt, scheme)
    dtags = [f"{case_id(G, tdt, scheme)} decompress_scatter into block {label(marks, int(b))}" for b in dst_blocks]
    assert_bits(bit_rows(out, dst_blocks, tdt), want_bits, dtags)
    assert_touched(out, tdt, dst_blocks.tolist(), f"{case_id(G, tdt, scheme)} decompress_scatter")


# ---- 4. host tier over the same caches ---------------------------------------------------------------------------
@pytest.mark.parametrize("G,tdt,scheme", PAGED, ids=[case_id(*c) for c in PAGED])
def test_host_tier_past_4gib(G, tdt, scheme):
    """offload_blocks of the boundary blocks -> restore_blocks into other high blocks of a sentinel cache;
    offload_ragged through the table -> restore_blocks; fetch(block_table=...) scattering into high blocks."""
    esz = ESZ[tdt]
    need(2 * BIG_BYTES + (256 << 20), "the host-tier case")
    cache, emarks = source(G, tdt)
    nb = cache.shape[0]
    table, marks = table_for(emarks, nb, seed=G * 17 + scheme)
    raw = raw_rows(cache, table, tdt)
    want = oracle_encode(raw, G, tdt, scheme)
    want_bits, _ = oracle_decode(*want, G, tdt, scheme)
    tdev = torch.as_tensor(table.astype(np.int32), device=DEV)
    n = len(table)
    dst = restore_targets(table, nb)
    assert np.unique(dst).size == n
    ddev = torch.as_tensor(dst.astype(np.int32), device=DEV)
    tags = [f"{case_id(G, tdt, scheme)} block {label(marks, int(s))} -> {int(d)}" for s, d in zip(table, dst)]

    tier = HostTier(64 << 20)
    try:
        tier.set_scheme(scheme)
        tier.enable_fetch()
        ids = np.arange(n, dtype=np.uint64) + 1000
        tier.offload_blocks(cache, tdev, ids)
        assert tier.stats()["blocks"] == n
        out = destination(nb, G, tdt)
        tier.restore_blocks(ids, out, ddev)
        assert_bits(bit_rows(out, dst, tdt), want_bits, [t + " restore_blocks" for t in tags])
        assert_touched(out, tdt, dst.tolist(), f"{case_id(G, tdt, scheme)} restore_blocks")

        out = destination(nb, G, tdt)
        _, oel, status = tier.fetch(torch.as_tensor(ids.astype(np.int64), device=DEV), G, TORCH_DT[tdt],
                                    scheme=scheme, out=out, block_table=ddev)
        assert (status.cpu().numpy() == 1).all(), (case_id(G, tdt, scheme), "fetch status", status.cpu().numpy())
        assert (oel.cpu().numpy() == G).all(), (case_id(G, tdt, scheme), "fetch out_elems")
        assert_bits(bit_rows(out, dst, tdt), want_bits, [t + " fetch" for t in tags])
        assert_touched(out, tdt, dst.tolist(), f"{case_id(G, tdt, scheme)} fetch")

        lengths = mixed_lengths(n, G)
        _, _, _, dec = oracle_prefix(raw, lengths, G, tdt, scheme)
        rids = ids + 5000
        tier.offload_ragged(cache, G, torch.tensor(lengths, dtype=torch.int32, device=DEV), rids, block_table=tdev)
        out = destination(nb, G, tdt)
        tier.restore_blocks(rids, out, ddev)
        assert_bits(bit_rows(out, dst, tdt), dec, [f"{t} offload_ragged n={m}" for t, m in zip(tags, lengths)])
        assert_touched(out, tdt, [int(d) for d, m in zip(dst, lengths) if m], f"{case_id(G, tdt, scheme)} offload_ragged")
    finally:
        tier.close()


@pytest.mark.parametrize("scheme", [2, 4])
def test_allocator_kv_blocks_past_131072(scheme):
    """CxlSpeckvKVAllocator.offload_kv_blocks / restore_kv_blocks on a [num_blocks, 16, 8, 128] fp16 cache with
    num_blocks > 131072: block 65536 starts at 2^31 bytes, block 131072 at 2^31 elements; whole blocks and filled
    token counts."""
    G = 16 * 8 * 128
    need(2 * BIG_BYTES + (256 << 20), "the allocator case")
    cache, emarks = source(G, F16)
    nb = cache.shape[0]
    assert nb > 131072
    kv = cache.view(nb, 16, 8, 128)
    table, marks = table_for(emarks, nb, seed=scheme)
    assert {65535, 65536, 131071, 131072} <= set(table.tolist())
    n = len(table)
    raw = raw_rows(cache, table, F16)
    want_bits, _ = oracle_decode(*oracle_encode(raw, G, F16, scheme), G, F16, scheme)
    dst = restore_targets(table, nb)
    tags = [f"s{scheme} block {label(marks, int(s))} -> {int(d)}" for s, d in zip(table, dst)]
    tier = HostTier(64 << 20)
    try:
        tier.set_scheme(scheme)
        ids = np.arange(n, dtype=np.uint64) + 7
        CxlSpeckvKVAllocator.offload_kv_blocks(kv, torch.as_tensor(table.astype(np.int32), device=DEV), tier, block_ids=ids)
        out = destination(nb, G, F16)
        CxlSpeckvKVAllocator.restore_kv_blocks(out.view(nb, 16, 8, 128), torch.as_tensor(dst.astype(np.int32), device=DEV),
                                               tier, block_ids=ids)
        assert_bits(bit_rows(out, dst, F16), want_bits, [t + " offload_kv_blocks" for t in tags])
        assert_touched(out, F16, dst.tolist(), f"s{scheme} restore_kv_blocks")

        tokens = [(0, 5, 16)[i % 3] for i in range(n)]
        _, _, _, dec = oracle_prefix(raw, [t * 1024 for t in tokens], G, F16, scheme)
        rids = ids + 100
        CxlSpeckvKVAllocator.offload_kv_blocks(kv, torch.as_tensor(table.astype(np.int32), device=DEV), tier,
                                               block_ids=rids, num_tokens=tokens)
        out = destination(nb, G, F16)
        CxlSpeckvKVAllocator.restore_kv_blocks(out.view(nb, 16, 8, 128), torch.as_tensor(dst.astype(np.int32), device=DEV),
                                               tier, block_ids=rids)
        assert_bits(bit_rows(out, dst, F16), dec, [f"{t} num_tokens={k}" for t, k in zip(tags, tokens)])
        assert_touched(out, F16, [int(d) for d, k in zip(dst, tokens) if k], f"s{scheme} num_tokens restore")
    finally:
        tier.close()


# ---- 5. a tier fetch larger than one gather sweep ----------------------------------------------------------------
def test_tier_fetch_spans_several_gather_sweeps():
    """fetch_gather_kernel walks the staging range with a persistent grid of SMs x 4 CTAs x 32 KiB.  Fetch 320
    blocks of 131072 fp16 under scheme 4 (40 MiB of payload, more than two sweeps) and 320 pages under scheme 2:
    bit-equal to restore, spot-checked against the oracle."""
    sweep = torch.cuda.get_device_properties(0).multi_processor_count * 4 * 32 * 1024
    need(1 * GIB, "the tier fetch case")
    tier = HostTier(160 << 20)
    try:
        for G, scheme, base in ((131072, 4, 0), (2048, 2, 1 << 20)):
            n = 320
            torch.manual_seed(G + scheme)
            x = torch.randn(n, G, device=DEV).half()
            x[7, 1000:4000] = 0.5                      # a long run
            x[150, 20:40] = 0.0
            ids = np.arange(n, dtype=np.uint64) + base
            tier.set_scheme(scheme)
            tier.offload(x.reshape(-1), G, ids)
            tier.enable_fetch()
            stored = tier.stats()["used_bytes"]
            want = tier.restore(ids, G, torch.float16)
            out = sentinel((n, G), F16)
            _, oel, status = tier.fetch(torch.as_tensor(ids.astype(np.int64), device=DEV), G, torch.float16,
                                        scheme=scheme, out=out)
            torch.cuda.synchronize()
            tag = f"G={G} scheme={scheme}"
            assert (status.cpu().numpy() == 1).all() and (oel.cpu().numpy() == G).all(), tag
            assert torch.equal(out.view(torch.int16), want.view(torch.int16)), (tag, "fetch differs from restore")
            if G == 131072:
                assert stored >= 2 * sweep, (tag, stored, sweep)
            # blocks at the start, around each sweep boundary, and at the end of the staging range
            per = max(1, stored // n)
            spots = sorted({0, 7, 150, n - 1} | {min(n - 1, (k * sweep) // per) for k in (1, 2)})
            raw = x[torch.as_tensor(spots, device=DEV)].cpu().numpy()
            wb, _ = oracle_decode(*oracle_encode(raw, G, F16, scheme), G, F16, scheme)
            assert_bits(bit_rows(out, spots, F16), wb, [f"{tag} block {s}" for s in spots])
            tier.drop(ids)
    finally:
        tier.close()


# ---- 6. the frozen API: pool pages past 4 GiB of one allocation -----------------------------------------------------
PAGE = 4096
BIG_PAGES = (1 << 20) + 64                       # 4 GiB + 256 KiB


def _frozen_lib():
    L = pkg.lib()
    assert L.speckv_init(b"cuda:0") == 0
    return L


def _alloc(L, nbytes):
    h = C.c_uint64()
    assert L.speckv_alloc(nbytes, None, C.byref(h)) == 0
    return h.value


def _alloc_with_parity(L, nbytes, parity):
    """Allocate until the handle has the parity asked for (the others are freed again)."""
    for _ in range(4):
        h = _alloc(L, nbytes)
        if h % 2 == parity:
            return h
        assert L.speckv_free(h) == 0
    pytest.fail("no handle of the asked parity came up")


def _fill_pages(pool, pages, seed):
    """Distinct content per page: N(0, 1) scaled by a per-page factor, one page with a long run."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    v = pool.view(-1, PAGE // 2)
    for k, p in enumerate(pages):
        v[p] = (torch.randn(PAGE // 2, generator=g, device=DEV) * (k + 1)).half()
    v[pages[-1], 100:900] = 0.75


def _round_trip(pool, pages):
    """What each page looks like after the tier: decompress(compress(page)), the bar of the pool tests."""
    v = pool.view(-1, PAGE // 2)
    rows = v[torch.as_tensor(pages, device=DEV)].clone()
    return codec.decompress(codec.compress(rows.reshape(-1), PAGE // 2)).view(torch.int16)


def _page_bits(pool, p):
    return pool.view(-1, PAGE // 2)[p].view(torch.int16)


def _lookup_documented(L, h, n_pages):
    """speckv_ext_page_lookup keeps the reference's ids: page i of handle h is (h << 32) | (i << 12), which for
    i >= 2^20 reaches the handle bits.  The lookup of an address in page 2^20 therefore finds the entry only when
    (h << 32) | (1 << 32) is that address's page (h even); for h odd it reports a miss (0 / 0)."""
    tbl = torch.zeros(n_pages * 3, dtype=torch.int64, device=DEV)
    cnt = C.c_size_t()
    assert L.speckv_ext_page_table_export(h, tbl.data_ptr(), n_pages, C.byref(cnt), None) == 0
    rec = tbl.view(n_pages, 3)[(1 << 20) - 1:(1 << 20) + 2].cpu().numpy().view(np.uint64)
    for k, i in enumerate(((1 << 20) - 1, 1 << 20, (1 << 20) + 1)):
        assert int(rec[k, 0]) == ((h << 32) | (i << 12)) & 0xFFFFFFFFFFFFFFFF, ("virt_page_id of page", i)
        assert int(rec[k, 1]) == 0x4000000000 + (h << 20) + (i << 12), ("phys_page_id of page", i)
    va = np.array([(h << 32) + ((1 << 20) - 1) * PAGE + 17, (h << 32) + (1 << 20) * PAGE + 17], np.uint64)
    dva = torch.from_numpy(va.view(np.int64)).to(DEV)
    pa = torch.zeros(2, dtype=torch.int64, device=DEV)
    fl = torch.zeros(2, dtype=torch.int32, device=DEV)
    assert L.speckv_ext_page_lookup(tbl.data_ptr(), n_pages, h << 32, dva.data_ptr(), pa.data_ptr(), fl.data_ptr(),
                                    2, None) == 0
    got = pa.cpu().numpy().view(np.uint64)
    assert int(got[0]) == 0x4000000000 + (h << 20) + (((1 << 20) - 1) << 12) + 17   # below 2^20: found
    i = 1 << 20
    hit = ((h << 32) | (i << 12)) == (int(va[1]) & ~0xFFF)
    assert hit == (h % 2 == 0)
    assert int(got[1]) == (0x4000000000 + (h << 20) + (i << 12) + 17 if hit else 0), ("lookup of page 2^20", h)


def test_frozen_api_pages_past_4gib_odd_handle():
    """Odd handle h: page 2^20 has the reference id of page 0 of h, page 2^20 + 1 that of page 1.  All four pages
    offloaded, the pool zeroed: each must come back with its own content, and the tier must hold four blocks."""
    need(BIG_PAGES * PAGE + (512 << 20), "the frozen-API case")
    _Big.release()
    L = _frozen_lib()
    tier = HostTier(16 << 20)
    try:
        nbytes = BIG_PAGES * PAGE
        h = _alloc_with_parity(L, nbytes, 1)
        pool = torch.zeros(nbytes // 2, dtype=torch.float16, device=DEV)
        pages = [0, 1, 1 << 20, (1 << 20) + 1]
        _fill_pages(pool, pages, seed=h)
        want = _round_trip(pool, pages)
        assert L.speckv_ext_bind_pool(h, C.c_void_p(pool.data_ptr()), nbytes, tier._h) == 0
        assert L.speckv_ext_offload_pages(h, 0, 2, None) == 0
        assert L.speckv_ext_offload_pages(h, 1 << 20, 2, None) == 0
        pool.view(-1, PAGE // 2)[torch.as_tensor(pages, device=DEV)] = 0
        ptr = C.c_void_p()
        for k, p in enumerate(pages):
            if k % 2 == 0:
                assert L.speckv_access(h, p * PAGE + 8, 16, C.byref(ptr)) == 0, ("speckv_access of page", p)
                assert ptr.value == pool.data_ptr() + p * PAGE + 8
            else:
                assert L.speckv_ext_fetch_pages(h, p, 1, None) == 0, ("fetch_pages of page", p)
            torch.cuda.synchronize()
            assert torch.equal(_page_bits(pool, p), want[k]), (f"handle {h} (odd): page {p} restored other bits",
                                                              [torch.equal(_page_bits(pool, p), w) for w in want])
        assert tier.stats()["blocks"] == 4
        _lookup_documented(L, h, BIG_PAGES)
        assert L.speckv_free(h) == 0
        assert tier.stats()["blocks"] == 0
    finally:
        L.speckv_finalize()
        tier.close()


def test_frozen_api_pages_past_4gib_even_handle():
    """Even handle h followed by a small handle h + 1: page 2^20 of h has the reference id of page 0 of h + 1.
    Page 0 of h + 1 must restore its own content, and speckv_free(h) must leave its block in the tier."""
    need(BIG_PAGES * PAGE + (512 << 20), "the frozen-API case")
    _Big.release()
    L = _frozen_lib()
    tier = HostTier(16 << 20)
    try:
        nbytes = BIG_PAGES * PAGE
        h = _alloc_with_parity(L, nbytes, 0)
        h2 = _alloc(L, 16 * PAGE)
        assert h2 == h + 1, ("handles are not consecutive", h, h2)
        pool = torch.zeros(nbytes // 2, dtype=torch.float16, device=DEV)
        pool2 = torch.zeros(16 * PAGE // 2, dtype=torch.float16, device=DEV)
        _fill_pages(pool, [1 << 20], seed=3)
        _fill_pages(pool2, [0], seed=4)
        want_h = _round_trip(pool, [1 << 20])[0]
        want_h2 = _round_trip(pool2, [0])[0]
        assert not torch.equal(want_h, want_h2)
        orig_h = _page_bits(pool, 1 << 20).clone()
        orig_h2 = _page_bits(pool2, 0).clone()
        assert L.speckv_ext_bind_pool(h, C.c_void_p(pool.data_ptr()), nbytes, tier._h) == 0
        assert L.speckv_ext_bind_pool(h2, C.c_void_p(pool2.data_ptr()), 16 * PAGE, tier._h) == 0
        assert L.speckv_ext_offload_pages(h2, 0, 1, None) == 0
        assert L.speckv_ext_offload_pages(h, 1 << 20, 1, None) == 0
        pool.zero_()
        pool2.zero_()
        assert L.speckv_ext_fetch_pages(h2, 0, 1, None) == 0
        assert L.speckv_ext_fetch_pages(h, 1 << 20, 1, None) == 0
        torch.cuda.synchronize()
        assert torch.equal(_page_bits(pool2, 0), want_h2), \
            (f"handle {h2}: page 0 restored other bits", "page 2^20 of handle", h, torch.equal(_page_bits(pool2, 0), want_h))
        assert torch.equal(_page_bits(pool, 1 << 20), want_h), f"handle {h}: page 2^20 restored other bits"
        assert tier.stats()["blocks"] == 2
        _lookup_documented(L, h, BIG_PAGES)

        # offload again, then free the big handle: page 0 of h + 1 keeps its stored copy.  The pages get their
        # original content back first: a restored page is already quantised, and scheme 2's round trip is no
        # identity, so offloading it would store different bits
        _page_bits(pool, 1 << 20).copy_(orig_h)
        _page_bits(pool2, 0).copy_(orig_h2)
        assert L.speckv_ext_offload_pages(h2, 0, 1, None) == 0
        assert L.speckv_ext_offload_pages(h, 1 << 20, 1, None) == 0
        pool2.zero_()
        assert L.speckv_free(h) == 0
        assert tier.stats()["blocks"] == 1
        ptr = C.c_void_p()
        assert L.speckv_access(h2, 0, PAGE, C.byref(ptr)) == 0, f"handle {h2}: page 0 left the tier with handle {h}"
        torch.cuda.synchronize()
        assert torch.equal(_page_bits(pool2, 0), want_h2)
        assert L.speckv_free(h2) == 0
    finally:
        L.speckv_finalize()
        tier.close()
