"""Ragged (filled-prefix) compress against whole-block compress on the same tensors.

python profiles/ragged_bench.py [--iters N] [--out FILE]

fp16 N(0,1) KV blocks of G = 131072 (2560 groups: the 1024-token x 128-dim headline launch), 16384 and 2048 elements
(the same 640 MiB each).  Every block holds `fill` of its tokens (128 elements each) and garbage behind them (N(0,1)
x 1000: the stale K/V of an earlier request in a reused block).  Fills: 1.0, 0.5, uniform random in whole tokens,
1 token.  Per case: ragged and dense compress time (CUDA events, mean over the timed calls), KV GB/s counted on the
bytes each call encodes (valid bytes for ragged, whole blocks for dense), decode time of the ragged and the dense
container under schemes 2 and 4, and the compression ratio (valid fp16 bytes / payload bytes).  A seeded sample of
groups is checked against the oracle on their prefix before anything is timed.  The input (640 MiB) is larger than
the L2, so every call reads it from HBM.  Prints the card name and its power limit with the results."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cxl_speckv_b200 import codec  # noqa: E402
from oracle.oracle import Port  # noqa: E402

TOKEN = 128
GEOMETRIES = ((131072, 2560), (16384, 20480), (2048, 163840))
FILLS = ("1.0", "0.5", "random", "1tok")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def lengths_for(fill, G, n, gen):
    tokens = G // TOKEN
    if fill == "1.0":
        t = torch.full((n,), tokens)
    elif fill == "0.5":
        t = torch.full((n,), tokens // 2)
    elif fill == "random":
        t = torch.randint(1, tokens + 1, (n,), generator=gen)
    else:
        t = torch.ones(n, dtype=torch.int64)
    return (t * TOKEN).to(torch.int32)


def timed(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e-3   # seconds per call


def check_sample(x, lens, c, G, scheme, gen, k=6):
    idx = torch.randint(0, x.shape[0], (k,), generator=gen).tolist()
    for g in idx:
        n = int(lens[g])
        raw = x[g, :n].cpu().numpy()
        p, s, cb = Port.compress_batch(raw, n, scheme=scheme)
        assert int(c.comp_bytes[g]) == int(cb[0]), ("comp_bytes", G, g)
        assert np.float32(c.scales[g].item()).view(np.uint32) == s[0].view(np.uint32), ("scale", G, g)
        assert np.array_equal(c.payload[g, :cb[0]].cpu().numpy(), p[0, :cb[0]]), ("payload", G, g)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "ragged_bench needs a CUDA device"
    gen = torch.Generator().manual_seed(1234)
    rows = []
    info = {"card": card(), "torch": torch.__version__}
    print(json.dumps(info), flush=True)
    for G, n in GEOMETRIES:
        torch.manual_seed(G)
        x = torch.randn(n, G, device="cuda").half()
        garbage = (torch.randn(n, G, device="cuda") * 1000).half()
        for fill in FILLS:
            lens = lengths_for(fill, G, n, gen)
            ld = lens.to("cuda")
            col = torch.arange(G, device="cuda")[None, :]
            xb = torch.where(col < ld[:, None].long(), x, garbage)
            valid = int(lens.to(torch.int64).sum()) * 2
            row = {"G": G, "groups": n, "fill": fill, "valid_bytes": valid, "dense_bytes": n * G * 2}
            for scheme in (2, 4):
                cr = codec.compress_ragged(xb, G, ld, scheme=scheme)
                cd = codec.compress(xb, G, scheme=scheme)
                torch.cuda.synchronize()
                check_sample(xb, lens, cr, G, scheme, gen)
                tr = timed(lambda: codec.compress_ragged(xb, G, ld, scheme=scheme, out=cr), args.iters)
                td = timed(lambda: codec.compress(xb, G, scheme=scheme, out=cd), args.iters)
                yr = torch.empty_like(xb)
                yd = torch.empty_like(xb)
                dr = timed(lambda: codec.decompress(cr, out=yr), args.iters)
                dd = timed(lambda: codec.decompress(cd, out=yd), args.iters)
                comp = int(cr.comp_bytes.to(torch.int64).sum())
                row[f"s{scheme}"] = {
                    "compress_ragged_ms": tr * 1e3, "compress_dense_ms": td * 1e3,
                    "compress_ragged_gbs": valid / tr / 1e9, "compress_dense_gbs": n * G * 2 / td / 1e9,
                    "decode_ragged_ms": dr * 1e3, "decode_dense_ms": dd * 1e3,
                    "decode_ragged_gbs": valid / dr / 1e9, "decode_dense_gbs": n * G * 2 / dd / 1e9,
                    "ratio_ragged": valid / max(comp, 1),
                }
                del cr, cd, yr, yd
            print(json.dumps(row), flush=True)
            rows.append(row)
        del x, garbage, xb
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"info": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
