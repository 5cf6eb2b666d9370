"""GPU parity tests of the codec's entry points, schemes and call sequences against the CPU oracle.

The plain compress -> decompress call under scheme 2 is pinned elsewhere (test_codec_gpu.py).  These tests cover
what the tier, the prefetcher and the vLLM backend call: the indexed, routed (request count on the device), paged
gather / scatter and packed-container forms, every storage scheme (1 codes, 2 the reference pipeline, 3 / 4 the
clamped extensions), and state the codec keeps per stream between calls (flag words, the run-expansion list and its
counters) under back-to-back calls, two streams and CUDA-graph replay.

Bar everywhere: scales, comp_bytes, payload bytes [:comp_bytes], out_elems and decoded bits equal the oracle's
(oracle.oracle.Port); outputs are views into sentinel-filled buffers, so what a call must not write is checked too."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.oracle import Port
from tests.helpers import BF16, F16, bf16_from_f32, f32_bits

pytestmark = pytest.mark.gpu

from cxl_speckv_b200 import codec  # noqa: E402
from cxl_speckv_b200._lib import lib  # noqa: E402

DEV = "cuda:0"
TORCH_DT = {F16: torch.float16, BF16: torch.bfloat16}
SENT = 0x1234          # 16-bit element sentinel (an ordinary fp16 / bf16 value no decode of these inputs produces by chance)
SENT_BYTE = 0xA5
SENT_WORD = 0x5A5A5A5A

# Decode path of a group under the tuned kernels (DESIGN.md section 4.1).  Nothing in the library reports the path a
# group took, so the batch builder below places groups by the rules that decide it:
#   normal     N(0,1): counts of 1 and rare 2s -> in-place expansion in the tuned kernel
#   runs300    constant runs of 300 elements: counts above 2 with non-zero values outgrow the in-place staging slack
#              -> flagged 2, run-expansion pass (decode_runs_region) in the second launch
#   smooth     a random walk (bench's smooth_fp16 generator): long runs of equal codes, under scheme 3 mostly
#              counts > 2 -> run expansion; under scheme 2 the wrapping codes break most runs (tuned in place)
#   zero_tail  N(0,1) up to a random fill level, zeros behind it: the boundary region is split, its zero-valued
#              tail written as a constant fill (tuned path)
#   zeros      an all-zero group: closed-form payload, decoded as one fill
#   inf        a +-inf in the group: infinite scale -> flagged 1, generic kernel (special values)
#   tiny       bf16 values around 1e-39 (max below the range the tuned compress covers) -> generic compress;
#              for fp16, denormals
#   outlier    KV-like: N(0,1) with two large outlier channels of a 128-wide head dim
#   oversized  N(0,1) whose stored comp_bytes is patched past the slot (decode side only, RLE schemes): the tuned
#              kernel leaves it to the generic kernel, which clamps the stream to the slot
CLASSES = ("normal", "runs300", "smooth", "zero_tail", "zeros", "inf", "tiny", "outlier", "oversized")


def walk(rng, G, step=0.01, length=1 << 20):
    """G consecutive elements of a random walk cumsum(step * N(0,1)) of `length` elements (bench.py's smooth_fp16
    step): a head channel drifting slowly along the sequence, cut into blocks.  The walk's value where the window
    starts is drawn directly, N(0, step^2 * start)."""
    start = int(rng.integers(0, max(1, length - G) + 1))
    x0 = step * np.sqrt(start) * rng.standard_normal()
    return (x0 + np.cumsum(step * rng.standard_normal(G))).astype(np.float32)


def class_group(rng, cls, G, tdt):
    x = rng.standard_normal(G).astype(np.float32)
    if cls == "runs300":
        x = np.repeat(x[:G // 300 + 1], 300)[:G]
    elif cls == "smooth":
        x = walk(rng, G)
    elif cls == "zero_tail":
        x[int(rng.integers(1, G)):] = 0.0
    elif cls == "zeros":
        x[:] = 0.0
    elif cls == "inf":
        x[int(rng.integers(0, G))] = np.inf if rng.random() < 0.5 else -np.inf
    elif cls == "tiny":
        x *= np.float32(1e-39 if tdt == BF16 else 1e-6)
    elif cls == "outlier":
        ch = np.arange(G) % 128
        x[(ch == 5) | (ch == 77)] *= np.float32(40.0)
    return x


def path_batch(rng, G, n_groups, tdt, classes=CLASSES, offset=0):
    """n_groups groups cycling through `classes` (starting at `offset`); returns (fp32 values, class per group)."""
    cls = [classes[(offset + i) % len(classes)] for i in range(n_groups)]
    return np.stack([class_group(rng, c, G, tdt) for c in cls]), cls


def narrow(x, tdt):
    """fp32 -> the stored 16-bit elements (np.float16, or bf16 bits as np.uint16)"""
    if tdt == F16:
        with np.errstate(over="ignore"):
            return x.astype(np.float16)
    return bf16_from_f32(x.reshape(-1)).reshape(x.shape)


def to_dev(raw, tdt):
    if tdt == BF16:
        return torch.from_numpy(np.ascontiguousarray(raw).view(np.int16)).to(DEV).view(torch.bfloat16)
    return torch.from_numpy(np.ascontiguousarray(raw)).to(DEV)


def bits(t):
    return t.view(torch.int16).cpu().numpy().view(np.uint16)


def sentinel_out(shape, tdt):
    return torch.full(shape, SENT, dtype=torch.int16, device=DEV).view(TORCH_DT[tdt])


def oracle_encode(raw, G, tdt, scheme):
    sb = codec.slot_bytes(G, scheme)
    return Port.compress_batch(raw.reshape(-1), G, dtype=tdt, slot_bytes=sb, threads=8, scheme=scheme)


def oracle_decode(payload, scales, comp, G, tdt, scheme):
    """Expected decode as 16-bit patterns with everything past out_elems set to SENT.  comp past the slot is clamped
    to it (the library decodes at most one slot; the oracle would read on into the next one)."""
    comp = np.minimum(comp, payload.shape[1]).astype(np.uint32)
    want, want_n = Port.decompress_batch(payload, scales, comp, G, tdt, threads=8, scheme=scheme)
    want = want.view(np.uint16).reshape(-1, G)
    return np.where(np.arange(G)[None, :] < want_n[:, None], want, np.uint16(SENT)), want_n


def assert_compressed(c, payload, scales, comp, tag, rows=None):
    """Device container c equals the oracle's (rows: which oracle group each stored group should be)."""
    if rows is not None:
        payload, scales, comp = payload[rows], scales[rows], comp[rows]
    assert np.array_equal(f32_bits(c.scales.cpu().numpy()), f32_bits(scales)), tag
    got_comp = c.comp_bytes.cpu().numpy().view(np.uint32)
    assert np.array_equal(got_comp, comp), (tag, np.flatnonzero(got_comp != comp)[:5])
    gp = c.payload.cpu().numpy()
    mask = np.arange(gp.shape[1])[None, :] < comp[:, None]
    bad = np.flatnonzero((np.where(mask, gp, 0) != np.where(mask, payload, 0)).any(axis=1))
    assert bad.size == 0, (tag, "payload differs in groups", bad[:5])


def assert_rows(got, want, tag):
    bad = np.argwhere(got != want)
    assert bad.size == 0, (tag, "mismatches", len(bad), "first (row, elem)", bad[0].tolist(),
                           hex(int(got[tuple(bad[0])])), hex(int(want[tuple(bad[0])])))


def container(payload, scales, comp, G, tdt, scheme):
    return codec.CompressedKV(torch.from_numpy(np.ascontiguousarray(payload)).to(DEV),
                              torch.from_numpy(np.ascontiguousarray(scales)).to(DEV),
                              torch.from_numpy(np.ascontiguousarray(comp, dtype=np.uint32).view(np.int32)).to(DEV),
                              G, TORCH_DT[tdt], scheme)


def regions(G):
    return G // 2048 if G % 2048 == 0 and (G // 2048) & (G // 2048 - 1) == 0 and G <= 128 * 2048 else 0


# ---- the indirection matrix -------------------------------------------------------------------------------------

@pytest.mark.parametrize("G,n_groups", [(2048, 72), (8192, 40), (32768, 24), (131072, 18), (6000, 40)])
@pytest.mark.parametrize("tdt", [F16, BF16])
@pytest.mark.parametrize("scheme", [1, 2, 3, 4])
def test_entry_points_match_the_oracle(G, n_groups, tdt, scheme):
    """Every group class through plain, indexed, scatter, routed and gather calls.  Requests repeat, reverse and
    name every class; scatter and routed outputs keep their sentinel where nothing may be written."""
    rng = np.random.default_rng(1000 * G + 10 * scheme + tdt)
    x, cls = path_batch(rng, G, n_groups, tdt)
    raw = narrow(x, tdt)
    tag = f"G={G} n={n_groups} dtype={tdt} scheme={scheme}"
    payload, scales, comp = oracle_encode(raw, G, tdt, scheme)
    sb = payload.shape[1]

    # plain compress, and the paged gather with a table that names some blocks twice
    cache = to_dev(raw, tdt)
    c = codec.compress(cache.reshape(-1), G, scheme=scheme)
    assert_compressed(c, payload, scales, comp, tag + " compress")
    table = np.concatenate([rng.permutation(n_groups), [0, n_groups - 1, 3, 3]]).astype(np.int32)
    cg = codec.compress_gather(cache, torch.from_numpy(table).to(DEV), scheme=scheme)
    assert_compressed(cg, payload, scales, comp, tag + " gather", rows=table)

    # decode side: the oracle's container, one group's size patched past its slot (RLE schemes)
    dcomp = comp.copy()
    if scheme in (2, 3):
        for g in (i for i, k in enumerate(cls) if k == "oversized"):
            dcomp[g] = sb + 32
    dc = container(payload, scales, dcomp, G, tdt, scheme)
    want, want_n = oracle_decode(payload, scales, dcomp, G, tdt, scheme)

    out = sentinel_out((n_groups, G), tdt)
    oel = torch.full((n_groups,), SENT_WORD, dtype=torch.int32, device=DEV)
    l0 = codec.stats()["kernel_launches"]
    codec.decompress(dc, out=out, out_elems=oel)
    torch.cuda.synchronize()
    assert codec.stats()["kernel_launches"] - l0 == (2 if regions(G) else 1), tag   # tuned kernel + flagged second pass
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n), tag
    assert_rows(bits(out), want, tag + " plain")

    # requests: half the blocks in reverse, then repeats, one block of every class among them
    src = np.concatenate([np.arange(n_groups)[::-1][:n_groups // 2], rng.integers(0, n_groups, n_groups - n_groups // 2)])
    for j, k in enumerate(CLASSES):
        src[n_groups // 2 + j] = cls.index(k)
    src = src.astype(np.int32)
    n_req = src.size
    srcd = torch.from_numpy(src).to(DEV)

    out = sentinel_out((n_req, G), tdt)
    codec.decompress_indexed(dc, srcd, out=out)
    assert_rows(bits(out), want[src], tag + " indexed")

    num_blocks = n_req + 7
    dst = rng.permutation(num_blocks)[:n_req].astype(np.int32)
    kv = sentinel_out((num_blocks, G), tdt)
    oel = torch.full((n_req + 4,), SENT_WORD, dtype=torch.int32, device=DEV)
    codec.decompress_scatter(dc, kv, torch.from_numpy(dst).to(DEV), srcd, out_elems=oel[2:2 + n_req])
    got_oel = oel.cpu().numpy().view(np.uint32)
    assert np.array_equal(got_oel[2:2 + n_req], want_n[src]), tag
    assert (got_oel[:2] == SENT_WORD).all() and (got_oel[2 + n_req:] == SENT_WORD).all(), tag
    expect = np.full((num_blocks, G), SENT, np.uint16)
    expect[dst] = want[src]
    assert_rows(bits(kv), expect, tag + " scatter")

    cap = n_req
    out = sentinel_out((cap, G), tdt)
    for count in (0, 1, cap - 1, cap, cap + 5):
        out.view(torch.int16).fill_(SENT)
        codec.decompress_routed(dc, srcd, torch.tensor([count], dtype=torch.int32, device=DEV), out)
        expect = np.full((cap, G), SENT, np.uint16)
        expect[:min(count, cap)] = want[src[:min(count, cap)]]
        assert_rows(bits(out), expect, f"{tag} routed count={count}")


# ---- packed host container --------------------------------------------------------------------------------------

@pytest.mark.parametrize("G", [2048, 32768, 6000])
@pytest.mark.parametrize("tdt", [F16, BF16])
@pytest.mark.parametrize("scheme", [1, 2, 3, 4])
def test_host_tier_restores_the_oracles_bits(G, tdt, scheme):
    """HostTier keeps blocks back to back in a pinned pool (slot_offsets on the decode side).  offload / restore and
    the paged offload_blocks / restore_blocks, over every group class, give what the oracle decodes."""
    from cxl_speckv_b200.tier import HostTier
    rng = np.random.default_rng(77 * G + 5 * scheme + tdt)
    n = max(24, min(96, (1 << 21) // G))
    classes = CLASSES[:-1]
    x, _ = path_batch(rng, G, n, tdt, classes)
    raw = narrow(x, tdt)
    payload, scales, comp = oracle_encode(raw, G, tdt, scheme)
    want, want_n = oracle_decode(payload, scales, comp, G, tdt, scheme)
    assert (want_n == G).all()
    tier = HostTier(pool_bytes=4 * n * G * 2 + (4 << 20))
    try:
        tier.set_scheme(scheme)
        xd = to_dev(raw, tdt)
        ids = np.arange(100, 100 + n, dtype=np.uint64)
        tier.offload(xd.reshape(-1), G, ids)
        order = rng.permutation(n)
        order[-3:] = (0, 0, n - 1)                    # repeats, as many requests as stored blocks
        y = tier.restore(ids[order], G, TORCH_DT[tdt], DEV)
        torch.cuda.synchronize()
        assert_rows(bits(y), want[order], f"restore G={G} scheme={scheme}")

        # paged: blocks of a cache named by a table go in under other ids, come back into other cache blocks
        num_blocks = n + 9
        cache = sentinel_out((num_blocks, G), tdt)
        cache[:n] = xd.view(n, G)
        table = rng.permutation(n).astype(np.int32)
        ids2 = np.arange(5000, 5000 + n, dtype=np.uint64)
        tier.offload_blocks(cache, torch.from_numpy(table).to(DEV), ids2)
        back = rng.permutation(n)
        dst = rng.permutation(num_blocks)[:n].astype(np.int32)
        kv = sentinel_out((num_blocks, G), tdt)
        tier.restore_blocks(ids2[back], kv, torch.from_numpy(dst).to(DEV))
        torch.cuda.synchronize()
        expect = np.full((num_blocks, G), SENT, np.uint16)
        expect[dst] = want[table[back]]
        assert_rows(bits(kv), expect, f"restore_blocks G={G} scheme={scheme}")
    finally:
        tier.close()


# ---- scheme 3 in its own regime -----------------------------------------------------------------------------------

@pytest.mark.parametrize("G", [2048 << k for k in range(8)] + [6000])
@pytest.mark.parametrize("tdt", [F16, BF16])
def test_scheme3_smooth_kv(G, tdt):
    """Random-walk KV (bench.py's smooth_fp16: cumsum(0.01 * N(0,1)) along 131072-element rows, cut into groups) and
    partially filled smooth blocks under the clamped RLE scheme: mostly counts > 2, i.e. the long-run emission and the
    run-expansion decode.  The ratio (16-bit bytes over payload bytes) above 2 shows the batch really is in that
    regime."""
    rng = np.random.default_rng(3 * G + tdt)
    n_groups = max(6, min(64, (4 << 20) // G))
    x = np.stack([walk(rng, G) for _ in range(n_groups)])
    levels = [1, 255, 2049, G // 2 + 7, G - 300, G - 1]
    for i, lvl in enumerate(levels):                  # partially filled blocks: smooth up to the level, zeros behind
        x[n_groups - 1 - i, min(lvl, G - 1):] = 0.0
    raw = narrow(x, tdt)
    payload, scales, comp = oracle_encode(raw, G, tdt, 3)
    assert 2.0 * G * n_groups / comp.sum() > 2.0
    c = codec.compress(to_dev(raw, tdt).reshape(-1), G, scheme=3)
    assert_compressed(c, payload, scales, comp, f"G={G}")
    want, want_n = oracle_decode(payload, scales, comp, G, tdt, 3)
    out = sentinel_out((n_groups, G), tdt)
    oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
    codec.decompress(c, out=out, out_elems=oel)
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n)
    assert_rows(bits(out), want, f"G={G}")


# ---- the short dequantiser's guard ------------------------------------------------------------------------------

def _short_form_differs(s, tdt):
    """For fp32 scales s: does q * RN(s / 127) round to other fp16 / bf16 bits than the reference (q / 127) * s for
    some code q?  numpy float32 arithmetic is IEEE round-to-nearest, as on the GPU (no contraction)."""
    q = np.arange(-128, 128, dtype=np.float32)[None, :]
    s = s[:, None]
    ref = (q / np.float32(127.0)) * s
    short = q * (s / np.float32(127.0))
    if tdt == F16:
        with np.errstate(over="ignore"):
            return (ref.astype(np.float16).view(np.uint16) != short.astype(np.float16).view(np.uint16)).any(axis=1)
    return (bf16_from_f32(ref.reshape(-1)) != bf16_from_f32(short.reshape(-1))).reshape(ref.shape).any(axis=1)


def failing_scales(tdt, k=6, seed=0):
    """k scales (over 2^-12 .. 2^8) for which the two dequantiser forms differ for some code."""
    rng = np.random.default_rng(seed + tdt)
    found = []
    for _ in range(64):
        s = (rng.uniform(1.0, 2.0, 1 << 16) * np.exp2(rng.integers(-12, 9, 1 << 16))).astype(np.float32)
        found.extend(s[_short_form_differs(s, tdt)][:k].tolist())
        if len(found) >= k:
            return np.array(found[:k], np.float32)
    raise AssertionError("no scale found where the short dequantiser differs")


@pytest.mark.parametrize("R", [8, 16, 128])
@pytest.mark.parametrize("tdt", [F16, BF16])
def test_short_dequantiser_guard(R, tdt):
    """The tuned decode (R >= 8) switches to q * RN(s / 127) only after checking all 256 codes for the group's scale.
    More than 99 % of scales pass, so ordinary data never reaches the fallback: these groups carry scales for which
    some code differs, and payloads that hit every code.  Codes-only payloads always take the reference form and
    serve as a control."""
    G = R * 2048
    scales = failing_scales(tdt)
    scales = np.concatenate([scales, -scales[:2], np.float32([1.0, 0.37])])     # plus two scales that pass
    n = scales.size
    rng = np.random.default_rng(R + tdt)
    sb = codec.slot_bytes(G)
    payload = np.zeros((n, sb), np.uint8)
    vals = rng.integers(0, 256, (n, G), dtype=np.uint8)
    vals[:, :256] = 1                                  # codes 1, 2, ..., 255, 0 up front, then a random walk
    payload[:, 0:2 * G:2] = vals
    payload[:, 1:2 * G:2] = 1
    comp = np.full(n, 2 * G, np.uint32)
    assert _short_form_differs(scales[:n - 2], tdt).all()
    want, want_n = oracle_decode(payload, scales, comp, G, tdt, 2)
    out = sentinel_out((n, G), tdt)
    oel = torch.zeros(n, dtype=torch.int32, device=DEV)
    codec.decompress(container(payload, scales, comp, G, tdt, 2), out=out, out_elems=oel)
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n)
    assert_rows(bits(out), want, f"rle R={R}")

    cb = codec.slot_bytes(G, 1)
    codes = np.zeros((n, cb), np.uint8)
    codes[:, :G] = vals
    codes[:, :256] = np.arange(256, dtype=np.uint8)
    ccomp = np.full(n, G, np.uint32)
    want, _ = oracle_decode(codes, scales, ccomp, G, tdt, 1)
    out = sentinel_out((n, G), tdt)
    codec.decompress(container(codes, scales, ccomp, G, tdt, 1), out=out)
    assert_rows(bits(out), want, f"codes R={R}")


# ---- buffer bounds ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("R,n_groups", [(1, 5), (2, 1), (2, 7), (2, 9), (8, 3)])
@pytest.mark.parametrize("scheme", [1, 2, 3])
def test_outputs_stay_inside_their_views(R, n_groups, scheme):
    """A CTA holds 16 / R groups; when n_groups is not a multiple of that, the tail CTA's idle warps must not write
    scales, comp_bytes, payload, out or out_elems of groups that do not exist.  Every output is a view into a larger
    sentinel-filled buffer; nothing outside the views may change."""
    G, tdt, pad = R * 2048, F16, 3
    rng = np.random.default_rng(R * 100 + n_groups + scheme)
    x, cls = path_batch(rng, G, n_groups, tdt, CLASSES[:-1], offset=n_groups)
    raw = narrow(x, tdt)
    payload, scales, comp = oracle_encode(raw, G, tdt, scheme)
    sb = payload.shape[1]
    pbig = torch.full(((n_groups + 2 * pad) * sb,), SENT_BYTE, dtype=torch.uint8, device=DEV)
    sbig = torch.full((n_groups + 8,), SENT_WORD, dtype=torch.int32, device=DEV)
    cbig = torch.full((n_groups + 8,), SENT_WORD, dtype=torch.int32, device=DEV)
    c = codec.CompressedKV(pbig[pad * sb:(pad + n_groups) * sb].view(n_groups, sb), sbig[4:4 + n_groups].view(torch.float32),
                           cbig[4:4 + n_groups], G, torch.float16, scheme)
    codec.compress(to_dev(raw, tdt).reshape(-1), G, scheme=scheme, out=c)
    assert_compressed(c, payload, scales, comp, "views")
    pb = pbig.cpu().numpy()
    assert (pb[:pad * sb] == SENT_BYTE).all() and (pb[(pad + n_groups) * sb:] == SENT_BYTE).all()
    for big in (sbig, cbig):
        b = big.cpu().numpy()
        assert (b[:4] == SENT_WORD).all() and (b[4 + n_groups:] == SENT_WORD).all()

    want, want_n = oracle_decode(payload, scales, comp, G, tdt, scheme)
    obig = torch.full(((n_groups + 2 * pad) * G,), SENT, dtype=torch.int16, device=DEV)
    ebig = torch.full((n_groups + 8,), SENT_WORD, dtype=torch.int32, device=DEV)
    out = obig[pad * G:(pad + n_groups) * G].view(torch.float16).view(n_groups, G)
    codec.decompress(c, out=out, out_elems=ebig[4:4 + n_groups])
    ob = obig.cpu().numpy().view(np.uint16)
    assert (ob[:pad * G] == SENT).all() and (ob[(pad + n_groups) * G:] == SENT).all()
    assert_rows(ob[pad * G:(pad + n_groups) * G].reshape(n_groups, G), want, "decode")
    e = ebig.cpu().numpy()
    assert np.array_equal(e[4:4 + n_groups].view(np.uint32), want_n)
    assert (e[:4] == SENT_WORD).all() and (e[4 + n_groups:] == SENT_WORD).all()


@pytest.mark.parametrize("G", [2048, 32768, 6000])
@pytest.mark.parametrize("extra", [16, 4096])
@pytest.mark.parametrize("scheme", [1, 2, 3])
def test_slot_stride_larger_than_the_minimum(G, extra, scheme):
    """Callers may lay slots out with a stride above speckv_ext_slot_bytes (bench.py's chunked calls, page-aligned
    pools).  Through the raw C calls: every group lands at its own stride, bytes of a slot past its 16-byte padded
    payload keep their contents, and the decode reads the same stride."""
    tdt = F16
    rng = np.random.default_rng(G + extra + scheme)
    n_groups = max(17, min(48, (1 << 21) // G))
    x, _ = path_batch(rng, G, n_groups, tdt, CLASSES[:-1])
    raw = narrow(x, tdt)
    payload, scales, comp = oracle_encode(raw, G, tdt, scheme)
    stride = payload.shape[1] + extra
    L = lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    xd = to_dev(raw, tdt).reshape(-1)
    pbig = torch.full(((n_groups + 1) * stride,), SENT_BYTE, dtype=torch.uint8, device=DEV)
    sc = torch.full((n_groups,), SENT_WORD, dtype=torch.int32, device=DEV)
    cb = torch.full((n_groups,), SENT_WORD, dtype=torch.int32, device=DEV)
    assert L.speckv_ext_compress(xd.data_ptr(), 0, G, n_groups, pbig.data_ptr(), stride, sc.data_ptr(), cb.data_ptr(),
                                 scheme, st) == 0
    assert np.array_equal(sc.cpu().numpy().view(np.uint32), f32_bits(scales))
    assert np.array_equal(cb.cpu().numpy().view(np.uint32), comp)
    pb = pbig.cpu().numpy()
    slots = pb[:n_groups * stride].reshape(n_groups, stride)
    for g in range(n_groups):
        assert np.array_equal(slots[g, :comp[g]], payload[g, :comp[g]]), g
        assert (slots[g, (int(comp[g]) + 15) // 16 * 16:] == SENT_BYTE).all(), (g, comp[g])
    assert (pb[n_groups * stride:] == SENT_BYTE).all()

    want, want_n = oracle_decode(slots, scales, comp, G, tdt, scheme)
    out = sentinel_out((n_groups + 1, G), tdt)
    oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
    assert L.speckv_ext_decompress(pbig.data_ptr(), stride, sc.data_ptr(), cb.data_ptr(), G, n_groups, 0, out.data_ptr(),
                                   oel.data_ptr(), scheme, st) == 0
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n)
    got = bits(out)
    assert_rows(got[:n_groups], want, "stride decode")
    assert (got[n_groups] == SENT).all()


# ---- calls in sequence, two streams, CUDA graphs ------------------------------------------------------------------

def _roundtrip_case(rng, G, n_groups, tdt, scheme, classes, offset=0):
    x, _ = path_batch(rng, G, n_groups, tdt, classes, offset)
    raw = narrow(x, tdt)
    payload, scales, comp = oracle_encode(raw, G, tdt, scheme)
    want, want_n = oracle_decode(payload, scales, comp, G, tdt, scheme)
    return raw, (payload, scales, comp, want, want_n)


def _check_roundtrip(c, out, oel, expect, tag):
    payload, scales, comp, want, want_n = expect
    assert_compressed(c, payload, scales, comp, tag)
    assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n), tag
    assert_rows(bits(out), want, tag)


RUNS = ("runs300", "smooth", "normal")            # a non-empty run-expansion list (under scheme 3)
PLAIN = ("normal", "zero_tail", "outlier", "zeros")
GENERIC = ("inf", "normal", "tiny", "runs300")


def test_back_to_back_calls_on_one_stream():
    """Eager calls without synchronisation, cycling R (64 -> 1 -> 16 -> 128) and the path mix: the per-stream scratch
    is resized and reused, and the run-list counters must be back at zero after a call with a non-empty list, one
    with none and one with generic groups alike."""
    rng = np.random.default_rng(64)
    steps = [(64, RUNS), (1, PLAIN), (16, GENERIC), (128, RUNS), (64, PLAIN), (1, RUNS), (16, RUNS), (128, GENERIC),
             (64, GENERIC), (1, GENERIC), (16, PLAIN), (128, PLAIN)]
    results = []
    for i, (R, mix) in enumerate(steps):
        G = R * 2048
        tdt = (F16, BF16)[i % 2]
        n_groups = max(3, min(40, (1 << 21) // G))
        raw, expect = _roundtrip_case(rng, G, n_groups, tdt, 3, mix, offset=i)
        c = codec.compress(to_dev(raw, tdt).reshape(-1), G, scheme=3)
        out = sentinel_out((n_groups, G), tdt)
        oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
        codec.decompress(c, out=out, out_elems=oel)
        results.append((c, out, oel, expect, f"step {i} R={R} {mix}"))
    torch.cuda.synchronize()
    for r in results:
        _check_roundtrip(*r)


def test_two_streams_alternating():
    """Two streams, each with its own geometry and scheme, calls alternating between them with no synchronisation:
    each stream's scratch is its own."""
    rng = np.random.default_rng(2)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    geo = [(16 * 2048, 12, F16, 3), (2048, 96, BF16, 2)]
    results = []
    for i in range(8):
        k = i % 2
        G, n_groups, tdt, scheme = geo[k]
        raw, expect = _roundtrip_case(rng, G, n_groups, tdt, scheme, (RUNS, PLAIN, GENERIC)[i % 3], offset=i)
        xd = to_dev(raw, tdt).reshape(-1)
        with torch.cuda.stream(streams[k]):
            streams[k].wait_stream(torch.cuda.default_stream())
            c = codec.compress(xd, G, scheme=scheme)
            out = sentinel_out((n_groups, G), tdt)
            oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
            codec.decompress(c, out=out, out_elems=oel)
        results.append((xd, c, out, oel, expect, f"call {i} stream {k}"))   # xd stays alive until the streams are done
    torch.cuda.synchronize()
    for r in results:
        _check_roundtrip(*r[1:])


@pytest.mark.parametrize("G,n_groups,scheme", [(2048, 64, 3), (16 * 2048, 12, 3), (64 * 2048, 6, 2), (6000, 20, 3)])
def test_graph_replay_with_new_contents(G, n_groups, scheme):
    """compress + decompress captured once on static buffers and replayed with new contents that move groups between
    paths (run list empty / non-empty, generic groups, zero groups): every replay equals the oracle.  The call runs
    eagerly on the capture stream first, so the per-stream scratch has its final size before the capture."""
    tdt = F16
    rng = np.random.default_rng(G + n_groups)
    sb = codec.slot_bytes(G, scheme)
    s = torch.cuda.Stream()
    xs = torch.zeros(n_groups * G, dtype=torch.float16, device=DEV)
    c = codec.CompressedKV(torch.zeros((n_groups, sb), dtype=torch.uint8, device=DEV),
                           torch.zeros(n_groups, dtype=torch.float32, device=DEV),
                           torch.zeros(n_groups, dtype=torch.int32, device=DEV), G, torch.float16, scheme)
    out = torch.zeros((n_groups, G), dtype=torch.float16, device=DEV)
    oel = torch.zeros(n_groups, dtype=torch.int32, device=DEV)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        codec.compress(xs, G, scheme=scheme, out=c)
        codec.decompress(c, out=out, out_elems=oel)
    s.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        codec.compress(xs, G, scheme=scheme, out=c)
        codec.decompress(c, out=out, out_elems=oel)
    mixes = [RUNS, PLAIN, GENERIC, CLASSES[:-1], RUNS, ("zeros",), GENERIC, ("normal",)]
    for i, mix in enumerate(mixes):
        raw, expect = _roundtrip_case(rng, G, n_groups, tdt, scheme, mix, offset=i)
        with torch.cuda.stream(s):
            xs.copy_(to_dev(raw, tdt).reshape(-1))
            out.view(torch.int16).fill_(SENT)
            graph.replay()
        s.synchronize()
        _check_roundtrip(c, out, oel, expect, f"replay {i} {mix}")


@pytest.mark.parametrize("G,scheme", [(2048, 2), (32768, 3), (32768, 1)])
def test_routed_graph_replay(G, scheme):
    """decompress_routed captured once; between replays the device-held request count and the block indices change
    (0, 1, cap - 1, cap, > cap requests).  Rows at or past the count keep their sentinel."""
    tdt = F16
    rng = np.random.default_rng(G * 3 + scheme)
    n_stored = max(16, min(80, (1 << 21) // G))
    x, _ = path_batch(rng, G, n_stored, tdt, CLASSES[:-1])
    raw = narrow(x, tdt)
    payload, scales, comp = oracle_encode(raw, G, tdt, scheme)
    want, _ = oracle_decode(payload, scales, comp, G, tdt, scheme)
    c = container(payload, scales, comp, G, tdt, scheme)
    cap = n_stored - 3
    bi = torch.zeros(cap, dtype=torch.int32, device=DEV)
    cnt = torch.zeros(1, dtype=torch.int32, device=DEV)
    out = sentinel_out((cap, G), tdt)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        codec.decompress_routed(c, bi, cnt, out)
    s.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        codec.decompress_routed(c, bi, cnt, out)
    for count in (cap, 0, 1, cap - 1, cap + 4, 7, cap):
        idx = rng.integers(0, n_stored, cap).astype(np.int32)
        with torch.cuda.stream(s):
            bi.copy_(torch.from_numpy(idx).to(DEV))
            cnt.fill_(count)
            out.view(torch.int16).fill_(SENT)
            graph.replay()
        s.synchronize()
        expect = np.full((cap, G), SENT, np.uint16)
        expect[:min(count, cap)] = want[idx[:min(count, cap)]]
        assert_rows(bits(out), expect, f"routed replay count={count}")


def test_randomised_entry_points():
    """tests/fuzz_codec.py paths mode for a few seconds: random schemes, entry points and KV-like value structures."""
    from tests import fuzz_codec
    fuzz_codec.main_paths(seconds=8.0, seed=21)
