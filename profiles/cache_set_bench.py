"""One request's KV across all layers: one KV-cache-set call against the per-layer loop of single-cache calls.

Shape: Llama-2-70B KV on one GPU -- 80 layers x K|V = 160 paged caches in vLLM's FlashAttention layout
([2, num_blocks, 16, 8, 128] fp16 per layer, a block of 16 tokens x 8 KV heads x 128 = 16384 elements), blocks
N(0,1), enough blocks for the largest request.  Requests of 512, 4096 and 32768 tokens, shuffled block tables,
schemes 2 (the reference's delta + RLE) and 4 (clamped INT8 codes).

Per request and scheme:
  offload   HostTier.offload_set (one call)      vs 160 x offload_blocks        host wall time, best of --reps
  restore   HostTier.restore_set (one call)      vs 160 x restore_blocks        host wall time, best of --reps
  fetch     one fetch_set in a CUDA graph        vs 160 fetch calls in one graph  CUDA events, best of --reps replays
  ceiling   one plain cudaMemcpyAsync of the same stored bytes between pinned host memory and HBM (D2H for the
            offload, H2D for restore and fetch), best of 10, in the same run
Before anything is timed, every output is checked bit for bit against the per-layer path: the set offload's records
restore (through the loop) to the same bits as the loop's records, and set restore / set fetch write the same bits
as loop restore / loop fetch.  Prints one JSON line per case and writes them all to --out; records the card's name
and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cxl_speckv_b200.codec import KVCacheSet  # noqa: E402
from cxl_speckv_b200.tier import HostTier  # noqa: E402

DEV = "cuda:0"
LAYERS, BS, HEADS, DIM = 80, 16, 8, 128
G = BS * HEADS * DIM
SENT = 0x7E01   # an fp16 NaN pattern no decoder writes


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.draw,clocks.sm,temperature.gpu",
                            "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def wall(fn, reps):
    best = float("inf")
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    return best


def replay_time(g, stream, reps):
    best = float("inf")
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            a.record(stream)
            g.replay()
            b.record(stream)
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) * 1e-3)
    return best


def copy_ceiling(nbytes, reps=10):
    """Best of `reps` plain copies of nbytes each way between pinned host memory and HBM: (d2h s, h2d s)."""
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dev = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    out = []
    for dst, src in ((host, dev), (dev, host)):
        best = float("inf")
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            dst.copy_(src, non_blocking=True)
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b) * 1e-3)
        out.append(best)
    del host, dev
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tokens", default="512,4096,32768")
    ap.add_argument("--schemes", default="2,4")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    tokens = [int(t) for t in args.tokens.split(",")]
    schemes = [int(s) for s in args.schemes.split(",")]
    info = {"card (name, power limit, draw, sm clock, temp)": card(), "caches": 2 * LAYERS, "block_elems": G,
            "dtype": "fp16 N(0,1)", "layout": "[2, num_blocks, 16, 8, 128] per layer"}
    print(json.dumps(info), flush=True)

    nb = max(tokens) // BS + 64
    gen = torch.Generator(device=DEV).manual_seed(0)
    kv = []
    for _ in range(LAYERS):
        t = torch.empty((2, nb, BS, HEADS, DIM), dtype=torch.float16, device=DEV)
        t.normal_(generator=gen)
        kv.append(t)
    views = [t[k] for t in kv for k in (0, 1)]   # cache 2 * layer + k
    cset = KVCacheSet(views)
    stream = torch.cuda.Stream()
    rows = []
    rng = np.random.default_rng(1)
    for ntok in tokens:
        n = ntok // BS
        table_np = rng.permutation(nb)[:n].astype(np.int32)
        table = torch.from_numpy(table_np).to(DEV)
        ci, blocks = cset.groups(table)
        nc = len(views)
        ids = ((np.arange(nc, dtype=np.uint64)[:, None] << np.uint64(40)) | table_np.astype(np.uint64)[None, :])
        loop_ids = ids | np.uint64(1 << 62)
        flat_ids = ids.reshape(-1)
        d_ids = torch.from_numpy(flat_ids.astype(np.int64)).to(DEV)
        raw = nc * n * G * 2
        for scheme in schemes:
            tier = HostTier(pool_bytes=int(2.2 * raw) + (64 << 20))
            tier.set_scheme(scheme)
            snap = None
            try:
                def off_set():
                    tier.offload_set(cset, ci, blocks, flat_ids)

                def off_loop(which=ids):
                    for c in range(nc):
                        tier.offload_blocks(views[c], table, which[c])

                def res_set():
                    tier.restore_set(flat_ids, cset, ci, blocks)

                def res_loop(which=ids):
                    for c in range(nc):
                        tier.restore_blocks(which[c], views[c], table)

                def req_bits():
                    return torch.stack([v[table.long()] for v in views]).view(torch.int16)

                def clear():
                    for v in views:
                        v.view(torch.int16)[table.long()] = SENT

                # ---- bit-exactness against the per-layer loop ----
                off_set()
                stored = tier.stats()["last_offload_stored_bytes"]
                off_loop(loop_ids)
                clear()
                res_loop(loop_ids)
                snap = req_bits()                      # loop offload -> loop restore
                clear()
                res_loop(ids)                          # set offload -> loop restore
                ok_offload = torch.equal(req_bits(), snap)
                clear()
                res_set()
                ok_restore = torch.equal(req_bits(), snap)
                tier.drop(loop_ids.reshape(-1))
                tier.enable_fetch()
                oel = torch.zeros(n * nc, dtype=torch.int32, device=DEV)
                st = torch.zeros(n * nc, dtype=torch.uint8, device=DEV)
                d_loop = [d_ids[c * n:(c + 1) * n] for c in range(nc)]
                oel_l = [oel[c * n:(c + 1) * n] for c in range(nc)]
                st_l = [st[c * n:(c + 1) * n] for c in range(nc)]

                def fetch_set():
                    tier.fetch_set(d_ids, cset, ci, blocks, scheme=scheme, out_elems=oel, status=st)

                def fetch_loop():
                    for c in range(nc):
                        tier.fetch(d_loop[c], G, torch.float16, scheme=scheme, out=views[c], block_table=table,
                                   out_elems=oel_l[c], status=st_l[c])

                graphs = {}
                for name, fn in (("set", fetch_set), ("loop", fetch_loop)):
                    with torch.cuda.stream(stream):
                        fn()
                        stream.synchronize()
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g, stream=stream):
                            fn()
                    graphs[name] = g
                ok_fetch = True
                for name in ("set", "loop"):
                    clear()
                    st.zero_()
                    torch.cuda.synchronize()
                    with torch.cuda.stream(stream):
                        graphs[name].replay()
                    stream.synchronize()
                    ok_fetch &= torch.equal(req_bits(), snap) and bool((st == 1).all())
                del snap
                snap = None
                if not (ok_offload and ok_restore and ok_fetch):
                    raise SystemExit(f"set and loop differ: tokens {ntok}, scheme {scheme}: "
                                     f"offload {ok_offload} restore {ok_restore} fetch {ok_fetch}")

                # ---- timing ----
                t = {
                    "offload_set": wall(off_set, args.reps), "offload_loop": wall(off_loop, args.reps),
                    "restore_set": wall(res_set, args.reps), "restore_loop": wall(res_loop, args.reps),
                    "fetch_set": replay_time(graphs["set"], stream, args.reps),
                    "fetch_loop": replay_time(graphs["loop"], stream, args.reps),
                }
                d2h, h2d = copy_ceiling(stored)
                row = {"tokens": ntok, "scheme": scheme, "caches": nc, "blocks": n * nc, "raw_bytes": raw,
                       "stored_bytes": stored, "bit_exact_vs_loop": True,
                       "ceiling_d2h_ms": d2h * 1e3, "ceiling_h2d_ms": h2d * 1e3}
                for op, ceil in (("offload", d2h), ("restore", h2d), ("fetch", h2d)):
                    row[f"{op}_set_ms"] = t[f"{op}_set"] * 1e3
                    row[f"{op}_loop_ms"] = t[f"{op}_loop"] * 1e3
                    row[f"{op}_speedup"] = t[f"{op}_loop"] / t[f"{op}_set"]
                    row[f"{op}_set_of_ceiling"] = ceil / t[f"{op}_set"]
                    row[f"{op}_loop_of_ceiling"] = ceil / t[f"{op}_loop"]
                rows.append(row)
                print(json.dumps(row), flush=True)
                del graphs
            finally:
                tier.close()
                torch.cuda.synchronize()
    info["card after (name, power limit, draw, sm clock, temp)"] = card()
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"info": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
