"""Randomised differential run of the CUDA codec against the CPU oracle (test infrastructure, not collected by
pytest):  python tests/fuzz_codec.py [seconds] [seed]  |  decode [seconds] [seed]  |  paths [seconds] [seed]
Random geometries (tuned and generic kernels), dtypes and value distributions -- mixtures of noise, constant and
zero stretches of random lengths (around the 8-element lane chunk and the 255 cap), NaN / Inf / denormal
sprinkles, tiny and huge magnitudes -- compressed and decompressed on the GPU; sizes, scales, payload bytes,
decoded lengths and decoded bits must equal the oracle's."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from cxl_speckv_b200 import codec
from oracle.oracle import Port
from tests.helpers import BF16, F16, bf16_from_f32


def make(rng, n):
    x = rng.standard_normal(n).astype(np.float32) * np.float32(np.exp(rng.uniform(-3, 3)))
    kind = rng.integers(0, 6)
    if kind >= 1:                                   # stretches: constant / zero / slowly varying
        pos = 0
        while pos < n:
            seg = int(rng.choice([1, 2, 3, 7, 8, 9, 15, 16, 17, 254, 255, 256, 300, 511, 2047, 2048, 2049, 5000]))
            seg = max(1, int(seg * rng.uniform(0.5, 1.5))) if rng.random() < 0.3 else seg
            mode = rng.integers(0, 4)
            if mode == 0:
                x[pos:pos + seg] = x[pos]
            elif mode == 1:
                x[pos:pos + seg] = 0.0
            elif mode == 2 and kind >= 3:
                x[pos:pos + seg] = np.linspace(x[pos], x[pos] * 1.5, min(seg, n - pos), dtype=np.float32)
            pos += seg + int(rng.integers(0, 40 if kind < 5 else 4000))
    if rng.random() < 0.3:
        idx = rng.integers(0, n, max(1, n // 3000))
        x[idx] = rng.choice(np.array([np.nan, np.inf, -np.inf, 1e-8, -1e-8, 6e-8, 65504.0, -0.0], dtype=np.float32), idx.size)
    return x


def main(seconds=120.0, seed=0):
    rng = np.random.default_rng(seed)
    t_end = time.time() + seconds
    cases = 0
    while time.time() < t_end:
        tuned = rng.random() < 0.75
        if tuned:
            G = 2048 * int(2 ** rng.integers(0, 8))
        else:
            G = int(rng.integers(1, 20000))
        n_groups = int(max(1, min(64, rng.integers(1, max(2, (3 << 20) // G)))))
        dtype = F16 if rng.random() < 0.6 else BF16
        x = np.concatenate([make(rng, G) for _ in range(n_groups)])
        if dtype == BF16 and rng.random() < 0.3:
            x *= np.float32(np.exp(rng.uniform(-70, 80)))
        if dtype == F16:
            with np.errstate(over="ignore"):
                raw = x.astype(np.float16)
            xd = torch.from_numpy(raw).cuda()
        else:
            raw = bf16_from_f32(x)
            xd = torch.from_numpy(raw.astype(np.int16)).cuda().view(torch.bfloat16)
        if os.environ.get("FUZZ_VERBOSE"):
            print(f"case {cases}: G={G} n={n_groups} dtype={dtype}", file=sys.stderr, flush=True)
        c = codec.compress(xd, G)
        oel = torch.zeros(n_groups, dtype=torch.int32, device="cuda")
        y = codec.decompress(c, out_elems=oel)
        torch.cuda.synchronize()
        payload, scales, comp = Port.compress_batch(raw, G, dtype=dtype, threads=8)
        tag = f"case {cases}: G={G} n={n_groups} dtype={dtype} seed={seed}"
        assert np.array_equal(c.scales.cpu().numpy().view(np.uint32), scales.view(np.uint32)), tag
        assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp), tag
        gp = c.payload.cpu().numpy()
        for g in range(n_groups):
            assert np.array_equal(gp[g, :comp[g]], payload[g, :comp[g]]), (tag, g)
        want, want_n = Port.decompress_batch(payload, scales, comp, G, dtype, threads=8)
        assert np.array_equal(oel.cpu().numpy().view(np.uint32), want_n), tag
        got = y.view(torch.int16).cpu().numpy().view(np.uint16)
        wantb = want.view(np.uint16).reshape(n_groups, G)
        if not np.array_equal(got, wantb):
            bad = np.argwhere(got != wantb)
            g0, e0 = bad[0]
            print(tag, "mismatches:", len(bad), "first at group", g0, "elem", e0, "got", hex(got[g0, e0]), "want", hex(wantb[g0, e0]),
                  "scale bits", hex(int(scales.view(np.uint32)[g0])), "comp", comp[g0], "groups hit", sorted(set(bad[:, 0].tolist()))[:10],
                  "input around", raw.reshape(n_groups, G)[g0, max(0, e0 - 3):e0 + 3])
            raise AssertionError(tag)
        cases += 1
    print(f"fuzz ok: {cases} cases in {seconds:.0f} s (seed {seed}); {codec.stats()}")


def make_payload(rng, G, sb):
    """A payload the encoder may never produce: arbitrary values and counts, any length up to the slot."""
    style = rng.integers(0, 5)
    npairs = int(rng.integers(0, sb // 2 + 1)) if rng.random() < 0.5 else int(min(sb // 2, rng.integers(0, G + G // 8 + 2)))
    val = rng.integers(0, 256, npairs, dtype=np.uint8)
    if style == 0:
        cnt = np.ones(npairs, np.uint8)
    elif style == 1:
        cnt = rng.choice(np.array([0, 1, 1, 1, 1, 1, 1, 2, 2, 3, 255], np.uint8), npairs)
    elif style == 2:
        cnt = rng.integers(0, 256, npairs, dtype=np.uint8)
    elif style == 3:
        cnt = np.ones(npairs, np.uint8)
        if npairs:
            cnt[rng.integers(0, npairs, max(1, npairs // 200))] = rng.integers(0, 256, max(1, npairs // 200), dtype=np.uint8)
            val[rng.integers(0, npairs, npairs // 2)] = 0
    else:
        cnt = rng.integers(1, 3, npairs, dtype=np.uint8)
        val[:] = 0 if rng.random() < 0.5 else val
    p = np.stack([val, cnt], axis=1).reshape(-1)
    if rng.random() < 0.2:
        p = np.concatenate([p, rng.integers(0, 256, 1, dtype=np.uint8)])[:sb]     # trailing odd byte
    return p


def main_decode(seconds=60.0, seed=0):
    """Decode side alone: arbitrary payloads (zero counts, long counts, short and overlong streams, odd lengths,
    negative and tiny scales) at tuned and generic geometries against the oracle's decoder."""
    rng = np.random.default_rng(seed)
    t_end = time.time() + seconds
    cases = 0
    while time.time() < t_end:
        G = 2048 * int(2 ** rng.integers(0, 8)) if rng.random() < 0.8 else int(rng.integers(1, 20000))
        n_groups = int(max(1, min(48, rng.integers(1, max(2, (2 << 20) // G)))))
        dtype = F16 if rng.random() < 0.6 else BF16
        sb = codec.slot_bytes(G)
        payload = rng.integers(0, 256, (n_groups, sb), dtype=np.uint8)               # garbage behind every payload
        comp = np.zeros(n_groups, np.uint32)
        for g in range(n_groups):
            p = make_payload(rng, G, sb)
            payload[g, :p.size] = p
            comp[g] = p.size
        scales = (rng.standard_normal(n_groups) * np.exp(rng.uniform(-8, 8, n_groups))).astype(np.float32)
        if rng.random() < 0.3:
            k = rng.integers(0, n_groups)
            scales[k] = rng.choice(np.array([np.inf, -np.inf, np.nan, 0.0, -0.0, 1e-45, 3e38], dtype=np.float32))
        tdt = torch.float16 if dtype == F16 else torch.bfloat16
        c = codec.CompressedKV(torch.from_numpy(payload).cuda(), torch.from_numpy(scales).cuda(),
                               torch.from_numpy(comp.view(np.int32)).cuda(), G, tdt, 2)
        out = torch.full((n_groups, G), 0x1234, dtype=torch.int16, device="cuda").view(tdt)
        oel = torch.zeros(n_groups, dtype=torch.int32, device="cuda")
        codec.decompress(c, out=out, out_elems=oel)
        torch.cuda.synchronize()
        want, want_n = Port.decompress_batch(payload, scales, comp, G, dtype, threads=8)
        tag = f"decode case {cases}: G={G} n={n_groups} dtype={dtype} seed={seed}"
        got_n = oel.cpu().numpy().view(np.uint32)
        assert np.array_equal(got_n, want_n), (tag, got_n[:8], want_n[:8])
        got = out.view(torch.int16).cpu().numpy().view(np.uint16)
        wantb = want.view(np.uint16).reshape(n_groups, G)
        for g in range(n_groups):
            n = int(want_n[g])
            if not np.array_equal(got[g, :n], wantb[g, :n]):
                e = int(np.argmax(got[g, :n] != wantb[g, :n]))
                raise AssertionError((tag, "group", g, "elem", e, hex(got[g, e]), hex(wantb[g, e]), "comp", comp[g], "scale", scales[g]))
            assert (got[g, n:] == 0x1234).all(), (tag, "wrote past the decoded length", g)
        cases += 1
    print(f"decode fuzz ok: {cases} cases in {seconds:.0f} s (seed {seed})")


def make_kv(rng, n):
    """KV-like values: a window of a slow random walk (bench.py smooth_fp16), or N(0,1) with a few outlier channels
    of a 128-wide head dim; sometimes filled only up to a random token, zeros behind it."""
    if rng.random() < 0.5:                          # n steps of a 2^20-step walk, its start value drawn directly
        x0 = 0.01 * np.sqrt(rng.integers(0, 1 << 20)) * rng.standard_normal()
        x = (x0 + np.cumsum(0.01 * rng.standard_normal(n))).astype(np.float32)
    else:
        x = rng.standard_normal(n).astype(np.float32)
        ch = np.arange(n) % 128
        for c in rng.integers(0, 128, int(rng.integers(1, 5))):
            x[ch == c] *= np.float32(rng.uniform(5, 100))
    if rng.random() < 0.25:
        x[int(rng.integers(1, n + 1)):] = 0.0
    return x


ENTRIES = ("plain", "gather", "indexed", "routed", "scatter")


def main_paths(seconds=60.0, seed=0):
    """Every scheme through every entry point: plain compress / decompress, paged gather (a block table with
    repeats), indexed decode (requests with repeats), routed decode (request count on the device, 0 .. past the
    capacity) and paged scatter (src_index + permuted block table).  Sizes, scales, payload bytes, decoded lengths
    and decoded bits equal the oracle's; outputs nothing may write keep their sentinel."""
    rng = np.random.default_rng(seed)
    t_end = time.time() + seconds
    counts = {("scheme", s): 0 for s in (1, 2, 3, 4)}
    counts.update({("entry", e): 0 for e in ENTRIES})
    cases = 0
    S = 0x1234
    while time.time() < t_end:
        scheme = int(rng.integers(1, 5))
        entry = ENTRIES[int(rng.integers(0, len(ENTRIES)))]
        G = 2048 * int(2 ** rng.integers(0, 8)) if rng.random() < 0.75 else int(rng.integers(1, 20000))
        n_groups = int(max(1, min(64, rng.integers(1, max(2, (3 << 20) // G)))))
        dtype = F16 if rng.random() < 0.6 else BF16
        tdt = torch.float16 if dtype == F16 else torch.bfloat16
        x = np.concatenate([make_kv(rng, G) if rng.random() < 0.4 else make(rng, G) for _ in range(n_groups)])
        if dtype == BF16 and rng.random() < 0.2:
            with np.errstate(over="ignore"):
                x *= np.float32(np.exp(rng.uniform(-70, 80)))
        if dtype == F16:
            with np.errstate(over="ignore"):
                raw = x.astype(np.float16)
            xd = torch.from_numpy(raw).cuda()
        else:
            raw = bf16_from_f32(x)
            xd = torch.from_numpy(raw.astype(np.int16)).cuda().view(torch.bfloat16)
        tag = f"paths case {cases}: {entry} scheme={scheme} G={G} n={n_groups} dtype={dtype} seed={seed}"
        if os.environ.get("FUZZ_VERBOSE"):
            print(tag, file=sys.stderr, flush=True)
        sb = codec.slot_bytes(G, scheme)
        payload, scales, comp = Port.compress_batch(raw, G, dtype=dtype, slot_bytes=sb, threads=8, scheme=scheme)
        rows = np.arange(n_groups)
        if entry == "gather":
            rows = rng.integers(0, n_groups, int(rng.integers(1, n_groups + 4))).astype(np.int32)
            c = codec.compress_gather(xd.view(n_groups, G), torch.from_numpy(rows).cuda(), scheme=scheme)
        else:
            c = codec.compress(xd, G, scheme=scheme)
        assert np.array_equal(c.scales.cpu().numpy().view(np.uint32), scales[rows].view(np.uint32)), tag
        assert np.array_equal(c.comp_bytes.cpu().numpy().view(np.uint32), comp[rows]), tag
        gp = c.payload.cpu().numpy()
        for i, g in enumerate(rows):
            assert np.array_equal(gp[i, :comp[g]], payload[g, :comp[g]]), (tag, i)
        want, want_n = Port.decompress_batch(payload, scales, comp, G, dtype, threads=8, scheme=scheme)
        want = np.where(np.arange(G)[None, :] < want_n[:, None], want.view(np.uint16).reshape(n_groups, G), np.uint16(S))
        n_st = rows.size
        src = rng.integers(0, n_st, n_st).astype(np.int32)          # as many requests as stored blocks, with repeats
        if rng.random() < 0.5:
            src[: n_st // 2] = np.arange(n_st)[::-1][: n_st // 2]
        srcd = torch.from_numpy(src).cuda()
        oel = torch.full((n_st,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
        if entry in ("plain", "gather"):
            out = torch.full((n_st, G), S, dtype=torch.int16, device="cuda").view(tdt)
            codec.decompress(c, out=out, out_elems=oel)
            expect, expect_n = want[rows], want_n[rows]
        elif entry == "indexed":
            out = torch.full((n_st, G), S, dtype=torch.int16, device="cuda").view(tdt)
            codec.decompress_indexed(c, srcd, out=out)
            expect, expect_n = want[src], None
        elif entry == "routed":
            cnt = int(rng.choice([0, 1, max(0, n_st - 1), n_st, n_st + 3, int(rng.integers(0, n_st + 1))]))
            out = torch.full((n_st, G), S, dtype=torch.int16, device="cuda").view(tdt)
            codec.decompress_routed(c, srcd, torch.tensor([cnt], dtype=torch.int32, device="cuda"), out)
            expect, expect_n = np.full((n_st, G), S, np.uint16), None
            expect[:min(cnt, n_st)] = want[src[:min(cnt, n_st)]]
            tag += f" count={cnt}"
        else:
            nb = n_st + int(rng.integers(0, 9))
            dst = rng.permutation(nb)[:n_st].astype(np.int32)
            out = torch.full((nb, G), S, dtype=torch.int16, device="cuda").view(tdt)
            codec.decompress_scatter(c, out, torch.from_numpy(dst).cuda(), srcd, out_elems=oel)
            expect = np.full((nb, G), S, np.uint16)
            expect[dst] = want[src]
            expect_n = want_n[src]
        torch.cuda.synchronize()
        if expect_n is not None:
            assert np.array_equal(oel.cpu().numpy().view(np.uint32), expect_n), tag
        got = out.view(torch.int16).cpu().numpy().view(np.uint16)
        if not np.array_equal(got, expect):
            bad = np.argwhere(got != expect)
            r0, e0 = bad[0]
            raise AssertionError((tag, "mismatches", len(bad), "first at row", r0, "elem", e0, hex(got[r0, e0]),
                                  hex(expect[r0, e0]), "rows hit", sorted(set(bad[:, 0].tolist()))[:10]))
        counts[("scheme", scheme)] += 1
        counts[("entry", entry)] += 1
        cases += 1
    per = ", ".join(f"{k[0]} {k[1]}: {v}" for k, v in counts.items())
    print(f"paths fuzz ok: {cases} cases in {seconds:.0f} s (seed {seed}); {per}")
    return counts


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "decode":
        main_decode(float(sys.argv[2]) if len(sys.argv) > 2 else 60.0, int(sys.argv[3]) if len(sys.argv) > 3 else 0)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "paths":
        main_paths(float(sys.argv[2]) if len(sys.argv) > 2 else 60.0, int(sys.argv[3]) if len(sys.argv) > 3 else 0)
        sys.exit(0)
    main(float(sys.argv[1]) if len(sys.argv) > 1 else 120.0, int(sys.argv[2]) if len(sys.argv) > 2 else 0)
