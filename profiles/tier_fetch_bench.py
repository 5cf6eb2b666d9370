"""Device-side tier fetch (HostTier.fetch) against the host-driven restore of the same ids.

python profiles/tier_fetch_bench.py [--iters N] [--out FILE]

Workloads (fp16 N(0,1) blocks, stored in a HostTier, ids fetched in shuffled order):
  a  1024 blocks of 131072 elements under scheme 4 (~128 KiB stored each) and scheme 2 (~256 KiB each)
  b  32768 pages of 2048 elements under scheme 2 (the 4 KiB page geometry), scattered into a paged cache
  c  small batches: 16 blocks of 131072, 64 pages of 2048 (where the host round trip matters most)
  d  a prefetch step from the tier: 256 sequences, k = 4, 4096 stored blocks of 131072 (bench.py cfg5's shape);
     emit -> route -> ids -> fetch as one CUDA graph against emit -> route -> decompress_routed from an HBM container
Per workload: fetch time per call eager and graph-replayed (CUDA events, mean over the timed calls), stored bytes moved
over PCIe per second, the ceiling (one plain host-to-device cudaMemcpyAsync of the same number of bytes out of pinned
host memory, best of 10, same run) and the wall time of the host-driven restore of the same ids.  Before anything is
timed, every timed output is checked bit for bit against HostTier.restore / restore_blocks of the same ids.  Outputs
of (a) and (b) are 256 MiB and 128 MiB, larger than the L2.  Prints the card name and its power limit with the results."""
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

from cxl_speckv_b200 import codec, prefetch  # noqa: E402
from cxl_speckv_b200.tier import HostTier  # noqa: E402

DEV = "cuda:0"


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def timed(fn, iters, stream):
    with torch.cuda.stream(stream):
        for _ in range(3):
            fn()
        stream.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(iters):
            fn()
        b.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e-3   # seconds per call


def graph_of(fn, stream):
    with torch.cuda.stream(stream):
        fn()
        stream.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            fn()
    return g


_CEIL = {}


def ceiling(nbytes, reps=10):
    """Best of `reps` plain H2D copies of nbytes from pinned host memory (seconds)."""
    if nbytes not in _CEIL:
        src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        dst = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
        best = float("inf")
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            dst.copy_(src, non_blocking=True)
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b) * 1e-3)
        _CEIL[nbytes] = best
    return _CEIL[nbytes]


def restore_wall(fn, reps=5):
    best = float("inf")
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    return best


def bits(t):
    return t.view(torch.int16)


def case(name, tier, ids, G, scheme, iters, stream, cache=None, table=None):
    """Fetch ids (numpy uint64) into a dense output, or into `cache` through `table`; check, then time."""
    n = len(ids)
    d_ids = torch.from_numpy(ids.view(np.int64)).to(DEV)
    out = cache if cache is not None else torch.empty((n, G), dtype=torch.float16, device=DEV)
    oel = torch.empty(n, dtype=torch.int32, device=DEV)
    st = torch.empty(n, dtype=torch.uint8, device=DEV)

    def fetch():
        tier.fetch(d_ids, G, torch.float16, scheme=scheme, out=out, block_table=table, out_elems=oel, status=st)

    if cache is not None:
        ref_cache = torch.empty_like(cache)
        restore = lambda: tier.restore_blocks(ids, ref_cache, table)   # noqa: E731
    else:
        ref = torch.empty((n, G), dtype=torch.float16, device=DEV)
        restore = lambda: tier.restore(ids, G, torch.float16, out=ref)   # noqa: E731
    if cache is not None:
        ref_cache.copy_(cache)
    restore()
    stored = tier.stats()["last_restore_stored_bytes"]
    with torch.cuda.stream(stream):
        fetch()
    torch.cuda.synchronize()
    assert bool((st == 1).all()), name
    assert torch.equal(bits(out), bits(ref_cache if cache is not None else ref)), name + ": fetch differs from restore"
    t_eager = timed(fetch, iters, stream)
    g = graph_of(fetch, stream)
    t_graph = timed(g.replay, iters, stream)
    torch.cuda.synchronize()
    assert torch.equal(bits(out), bits(ref_cache if cache is not None else ref)), name + ": graph replay differs"
    t_restore = restore_wall(restore)
    t_ceil = ceiling(stored)
    row = {"workload": name, "blocks": n, "G": G, "scheme": scheme, "stored_bytes": stored,
           "fetch_eager_ms": t_eager * 1e3, "fetch_graph_ms": t_graph * 1e3,
           "fetch_stored_GBps": stored / t_graph / 1e9, "fetch_eager_stored_GBps": stored / t_eager / 1e9,
           "ceiling_copy_ms": t_ceil * 1e3, "ceiling_GBps": stored / t_ceil / 1e9,
           "frac_of_ceiling": t_ceil / t_graph, "restore_wall_ms": t_restore * 1e3,
           "restore_stored_GBps": stored / t_restore / 1e9, "fetch_vs_restore_speedup": t_restore / t_graph}
    print(json.dumps(row), flush=True)
    return row


def step_case(iters, stream):
    """(d): the cfg5 prefetch step with its predicted blocks fetched from the tier vs decoded from an HBM container."""
    G, n_blocks, batch, k, base = 131072, 4096, 256, 4, 1 << 40
    rng = np.random.default_rng(1)
    emb = ((rng.random((32000, 64), dtype=np.float32) - 0.5) * 0.1).astype(np.float32)
    wout = ((rng.random((32000, 128), dtype=np.float32) - 0.5) * 0.1).astype(np.float32)
    prefetch.load_predictor(emb, wout)
    toks = torch.from_numpy(np.random.default_rng(7).integers(0, 32000, (batch, 16)).astype(np.int32)).to(DEV)
    x = torch.empty(n_blocks * G, device=DEV, dtype=torch.float16).normal_()
    c = codec.compress(x, G)
    tier = HostTier(pool_bytes=int(n_blocks * G * 2 * 1.1) + (64 << 20))
    tier.offload(x, G, np.arange(n_blocks, dtype=np.uint64) + np.uint64(base))
    tier.enable_fetch()
    del x
    cap = batch * k
    table = torch.zeros((prefetch.table_records(batch, k), prefetch.REQUEST_BYTES), dtype=torch.uint8, device=DEV)
    block_index = torch.zeros(cap, dtype=torch.int32, device=DEV)
    count = torch.zeros(1, dtype=torch.int32, device=DEV)
    ids = torch.zeros(cap, dtype=torch.int64, device=DEV)
    out_t = torch.empty((cap, G), dtype=torch.float16, device=DEV)
    out_h = torch.empty((cap, G), dtype=torch.float16, device=DEV)
    oel = torch.empty(cap, dtype=torch.int32, device=DEV)
    st = torch.empty(cap, dtype=torch.uint8, device=DEV)

    def route():
        prefetch.emit(toks, k=k, layer_id=0, timestamp=1, table=table)
        prefetch.route(table, 1, cap, n_blocks, 1, 0, block_index=block_index, count=count)

    def step_tier():
        route()
        torch.add(block_index.long(), base, out=ids)
        tier.fetch(ids, G, torch.float16, out=out_t, count=count, out_elems=oel, status=st)

    def step_hbm():
        route()
        codec.decompress_routed(c, block_index, count, out_h)

    g_t, g_h = graph_of(step_tier, stream), graph_of(step_hbm, stream)
    g_t.replay()
    g_h.replay()
    torch.cuda.synchronize()
    n = int(count.item())
    want = tier.restore(ids[:n].cpu().numpy().astype(np.uint64), G, torch.float16)
    stored = tier.stats()["last_restore_stored_bytes"]
    assert torch.equal(bits(out_t[:n]), bits(want)), "step: tier fetch differs from restore"
    assert torch.equal(bits(out_h[:n]), bits(want)), "step: HBM decode differs from restore"
    t_tier = timed(g_t.replay, iters, stream)
    t_hbm = timed(g_h.replay, iters, stream)
    t_ceil = ceiling(stored)
    row = {"workload": "d: cfg5 step, 256 seq x k=4, 4096 stored blocks of 131072 fp16, scheme 2",
           "blocks_fetched": n, "stored_bytes": stored, "step_tier_graph_ms": t_tier * 1e3,
           "step_hbm_graph_ms": t_hbm * 1e3, "pcie_bound_ms": t_ceil * 1e3, "step_over_pcie_bound": t_tier / t_ceil,
           "fetch_stored_GBps": stored / t_tier / 1e9}
    print(json.dumps(row), flush=True)
    tier.close()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default="abcd")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tier_fetch_bench needs a CUDA device"
    info = {"card": card(), "torch": torch.__version__}
    print(json.dumps(info), flush=True)
    stream = torch.cuda.Stream()
    rng = np.random.default_rng(5)
    rows = []
    if "a" in args.only or "c" in args.only:
        G, n = 131072, 1024
        x = torch.randn(n * G, device=DEV).half()
        ids = np.arange(n, dtype=np.uint64) * np.uint64(131) + np.uint64(7)
        for scheme in (4, 2):
            tier = HostTier(pool_bytes=int(n * G * 2 * 1.1) + (64 << 20))
            tier.set_scheme(scheme)
            tier.offload(x, G, ids)
            tier.enable_fetch()
            sel = ids[rng.permutation(n)]
            if "a" in args.only:
                rows.append(case(f"a: 1024 blocks of 131072, scheme {scheme}", tier, sel, G, scheme, args.iters, stream))
            if "c" in args.only and scheme == 2:
                rows.append(case("c: 16 blocks of 131072, scheme 2", tier, sel[:16], G, scheme, args.iters * 10, stream))
            tier.close()
        del x
    if "b" in args.only or "c" in args.only:
        G, n = 2048, 32768
        x = torch.randn(n * G, device=DEV).half()
        ids = np.arange(n, dtype=np.uint64) << np.uint64(12)
        tier = HostTier(pool_bytes=int(n * G * 2 * 1.3) + (64 << 20))
        tier.offload(x, G, ids)
        tier.enable_fetch()
        sel = ids[rng.permutation(n)]
        cache = torch.zeros((n, G), dtype=torch.float16, device=DEV)
        table = torch.from_numpy(rng.permutation(n).astype(np.int32)).to(DEV)
        if "b" in args.only:
            rows.append(case("b: 32768 pages of 2048 into a paged cache, scheme 2", tier, sel, G, 2, args.iters, stream,
                             cache=cache, table=table))
        if "c" in args.only:
            rows.append(case("c: 64 pages of 2048, scheme 2", tier, sel[:64], G, 2, args.iters * 10, stream,
                             cache=cache, table=table[:64].contiguous()))
        tier.close()
        del x, cache
    if "d" in args.only:
        rows.append(step_case(args.iters, stream))
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"info": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
