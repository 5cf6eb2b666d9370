#!/usr/bin/env python
"""bench.py -- KV block codec throughput on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path

One "step" = one pass of the hot path over one batch of synthetic KV: every group of the
workload is compressed (scale -> wrapped int8 -> delta -> byte-pair RLE) and then
decompressed again.  `value` = uncompressed fp16 KV bytes that made the round trip per
second, whole job (all ranks), inputs resident in HBM.  `e2e` = the same metric through the
host-buffer C ABI (speckv_ext_compress_host / _decompress_host) with the H2D / D2H copies
inside the timed region, next to the plain-memcpy ceiling of the same bytes.

Headline workload (BASELINE.json configs[2], the shape the north-star target is quoted on):
  cfg3  Llama-2-70B GQA KV, 80 L x 2 x 8 KVH x 8K ctx: 10240 groups of 1024 tok x 128 d
        = 2.5 GiB fp16, layers split 80/N contiguously across the ranks (STRONG scaling;
        at N = 1 the whole tensor on one GPU)
Sub-records in `aux` (same run, same ranks):
  cfg2  Llama-2-7B KV, batch 32 x 4K ctx PER GPU: 262144 groups = 64 GiB per GPU (weak scaling)
  cfg5  batch-256 decode: LSTM prefetch scoring + request exchange + routed decompress
  tier  cfg4 (Llama-3-8B 32K ctx as 4 KiB pages): translate, offload -> restore through the
        pinned host pool, PCIe GB/s
  ratios  per value distribution / scheme: ratio, MSE, codec GB/s and fraction of the HBM peak
One process per GPU (torchrun), no data-path collective; at N > 1 the only exchanges are NCCL
all-gathers of metadata (per-group page-table records; PrefetchRequest tables in cfg5).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

G_BLOCK = 131072          # 1024 tokens x 128 dims: one (layer, head, K|V) block
METRIC = "kv_compress_decompress_roundtrip_throughput"
UNIT = "GB/s"             # 1e9 bytes of uncompressed fp16 KV per second


def workload_spec(name: str, world: int, rank: int, scale: float):
    """-> dict(label, group_elems, n_groups (this rank), chunk_groups, scaling)"""
    if name == "cfg2":
        layers, per_layer = 32, 2 * 32 * 32 * 4          # K|V x heads x batch x (4096/1024)
        layers = max(1, int(round(layers * scale)))
        return dict(label=f"cfg2: Llama-2-7B KV, batch 32 x 4K ctx per GPU ({layers} layers x {per_layer} blocks of 1024x128 fp16)",
                    group_elems=G_BLOCK, n_groups=layers * per_layer, chunk_groups=per_layer, scaling="weak",
                    global_batch=32 * world)
    if name == "cfg3":
        layers, per_layer = 80, 2 * 8 * 8                # K|V x KV heads x (8192/1024)
        mine = range(rank * layers // world, (rank + 1) * layers // world)      # contiguous 80 / N layers per rank
        return dict(label=f"cfg3: Llama-2-70B GQA KV, 80 L x 8 KVH x 8K ctx, layers sharded {layers}/{world}",
                    group_elems=G_BLOCK, n_groups=len(mine) * per_layer, chunk_groups=per_layer * 20, scaling="strong",
                    global_batch=1)
    if name == "cfg4p":
        layers, per_layer = 32, 2 * 8 * 32768 * 128 // 2048
        layers = max(1, int(round(layers * scale)))
        return dict(label=f"cfg4p: Llama-3-8B 32K ctx paged KV, {layers} layers x {per_layer} page groups of 2048 fp16",
                    group_elems=2048, n_groups=layers * per_layer, chunk_groups=per_layer, scaling="weak",
                    global_batch=world)
    raise SystemExit(f"unknown workload {name}")


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel_key: str):
    """DRAM bytes per group of 131072 fp16 elements from the committed ncu --set full capture of the kernel
    (profiles/ncu_traffic.json: {"compress": {"dram_bytes_per_group": .., "source": "<capture, head, date>"}, ..})."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            r = json.load(f).get(kernel_key)
        return r if isinstance(r, dict) and "dram_bytes_per_group" in r else None
    except Exception:
        return None


# speckv_comp_scheme_t (host/include/speckv.h:59-63) + the extension ids of include/speckv_ext.h (non-wrapping quantiser)
SCHEME_IDS = {"fp16": 0, "int8": 1, "int8_delta_rle": 2, "int8_clamp_delta_rle": 3, "int8_clamp": 4}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.05):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8)): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._halt.wait(self.period)

    def mark(self):
        """the timed region starts now: samples from here on are counted separately"""
        self.marked_at = len(self.samples)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        timed = sorted(self.samples[getattr(self, "marked_at", 0):])
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s),
                "samples_in_timed_region": len(timed), "sm_mhz_timed_region": (timed[len(timed) // 2] if timed else None),
                "window": "warm-up steps (same kernels, back to back) + timed region"}


# --------------------------------------------------------------------------------------
# reference arm: the reference's own C++ engine (oracle/_ref) on the host cores
# --------------------------------------------------------------------------------------
def cpu_roundtrip_rate(group_elems: int, budget_s: float, threads: int, seed: int = 1234):
    """Times the reference CPU path (oracle/_ref when it was built here, else the C port) on a
    bounded sample of the workload: round trip of `n` groups of N(0,1) fp16.  -> dict"""
    import numpy as np
    from oracle.oracle import Port, Ref

    rng = np.random.default_rng(seed)
    kind = "reference" if Ref.available() else "port"

    def run(x16, ngroups):
        t0 = time.perf_counter()
        if kind == "reference":
            Ref.roundtrip_batch(x16, 0, group_elems, threads)
        else:
            payload, scales, comp = Port.compress_batch(x16, group_elems, threads=threads)
            Port.decompress_batch(payload, scales, comp, group_elems, 0, threads=threads)
        return time.perf_counter() - t0

    probe_groups = max(threads, 8) if group_elems >= 65536 else max(threads * 16, 256)
    xp = rng.standard_normal(probe_groups * group_elems).astype(np.float16)
    run(xp, probe_groups)                                    # warm-up (page faults, thread start)
    t_probe = run(xp, probe_groups)
    # one pass over <= 512 MiB of KV, repeated until the time budget is used
    cap = max(probe_groups, (512 << 20) // (group_elems * 2))
    n = int(max(probe_groups, min(probe_groups * budget_s / max(t_probe, 1e-6), cap)))
    n = (n // threads) * threads or threads
    x = rng.standard_normal(n * group_elems).astype(np.float16)
    dt, reps = 0.0, 0
    while dt < budget_s and reps < 1000:
        dt += run(x, n)
        reps += 1
    gbs = reps * n * group_elems * 2 / dt / 1e9
    return {"value": gbs, "unit": UNIT, "cores": threads, "kind": kind, "seconds": dt,
            "sample": f"{reps} x {n} groups of {group_elems} fp16 N(0,1) elements ({n * group_elems * 2 / 2**20:.0f} MiB per pass), "
                      f"compress+decompress round trip, {threads} threads, {dt:.1f} s"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    spec = workload_spec(args.workload, world, 0, args.scale)
    threads = os.cpu_count() or 1
    per_step_budget = max(2.0, min(10.0, 90.0 / max(1, args.steps + args.warmup)))
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_roundtrip_rate(spec["group_elems"], per_step_budget, threads, seed=1234 + i)
        if i >= args.warmup:
            vals.append(r)
    tot_bytes = sum(v["value"] * v["seconds"] for v in vals)
    tot_s = sum(v["seconds"] for v in vals)
    value = tot_bytes / tot_s
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / len(vals),
            "higher_is_better": True, "scaling": spec["scaling"], "vs_baseline": None, "dtype": "f32+i8",
            "data": "synthetic N(0,1) fp16 KV (numpy default_rng)",
            "config": {"workload": spec["label"], "group_elems": spec["group_elems"],
                       "note": "reference CPU engine (FPGACacheEngine::compress/decompress) on host cores; "
                               "each step is a bounded sample of the workload"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": vals[-1]["kind"],
                             "sample": vals[-1]["sample"]},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------
# CUDA arm
# --------------------------------------------------------------------------------------
def bind_to_gpu_cpus(local_rank):
    """Pin this rank to the host cores NVML lists as local to its GPU, so that the pinned host
    buffers of the e2e leg are allocated on the GPU's own NUMA node (matters at 8 ranks per box).
    Returns the previous affinity so that the CPU baseline can take all cores back."""
    before = os.sched_getaffinity(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(before) + 64) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1} & before
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass
    return before


class Env:
    """What every leg of the CUDA arm needs: torch, the process group, the library."""

    def __init__(self, args, rank, world, local_rank):
        import torch
        import torch.distributed as dist

        import cxl_speckv_b200 as pkg

        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback "
                             "(use --impl reference for the CPU baseline)")
        self.args, self.rank, self.world, self.local_rank = args, rank, world, local_rank
        self.torch, self.dist = torch, dist
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        if world > 1:
            import datetime
            dist.init_process_group("nccl", device_id=self.dev, timeout=datetime.timedelta(seconds=180))
        self.L = pkg.lib()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, vals, op="max"):
        """list of floats -> the same list reduced over the ranks"""
        t = self.torch.tensor(vals, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return t.tolist()

    def gather_floats(self, v):
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [float(v)]
        out = self.torch.empty(self.world, dtype=self.torch.float64, device=self.dev)
        self.dist.all_gather_into_tensor(out, t)
        return out.tolist()


DUMP_BYTES_MAX = 64 << 20
DUMP_GROUPS_MAX = 1 << 20          # per-group records (20 B each) beyond this are a seeded sample


def dump_outputs(dump_dir, env, first_held, payload, scales, comp, out):
    """Writes what the round trip hands its caller after the last timed step, as .npy files that two builds can be
    compared by: the scale and compressed size of every group (of a seeded sample of DUMP_GROUPS_MAX groups beyond
    that, group_index names them), and for 16 groups picked with a fixed seed their payload (the first comp_bytes of
    the slot, the rest zero) and their decoded values.  float32 / float64, at most DUMP_BYTES_MAX in all."""
    import numpy as np

    torch = env.torch
    n = comp.numel()
    held = n - first_held                                    # groups whose decode `out` still holds, from row 0
    pick = np.sort(np.random.default_rng(0).choice(held, min(16, held), replace=False))
    rows = torch.from_numpy(pick).to(out.device)
    groups = pick + first_held
    comp_h = comp.cpu().numpy()
    pay = payload.index_select(0, rows + first_held).cpu().numpy()
    pay = np.where(np.arange(pay.shape[1])[None, :] < comp_h[groups][:, None], pay, 0)
    every = np.arange(n) if n <= DUMP_GROUPS_MAX else np.sort(np.random.default_rng(1).choice(n, DUMP_GROUPS_MAX, replace=False))
    arrays = {"group_index": every.astype(np.float64),
              "scales": scales[torch.from_numpy(every).to(scales.device)].cpu().numpy().astype(np.float32),
              "comp_bytes": comp_h[every].astype(np.float64),
              "sample_groups": groups.astype(np.float64), "payload_sample": pay.astype(np.float32),
              "decoded_sample": out.index_select(0, rows).float().cpu().numpy()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES_MAX, f"--dump-outputs: {total} bytes exceed {DUMP_BYTES_MAX}"
    os.makedirs(dump_dir, exist_ok=True)
    suffix = f"_rank{env.rank}" if env.world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(dump_dir, f"{name}{suffix}.npy"), a)


def codec_roundtrip(env, spec, steps, warmup, use_graph, sample_clocks=False, scheme=2, dump_dir=None):
    """K timed steps of: compress every group of this rank's shard -> (N > 1: all-gather of the page-table
    metadata on a side stream, overlapped) -> decompress every group.  Device-resident inputs.
    -> dict with the whole-job value, the per-phase times (CUDA events on the launching stream) and the roofline.
    dump_dir: where to write the last timed step's outputs (dump_outputs)."""
    import ctypes as C

    torch, dist, L, dev, world = env.torch, env.dist, env.L, env.dev, env.world
    from cxl_speckv_b200 import codec

    G, n_groups, cg = spec["group_elems"], spec["n_groups"], spec["chunk_groups"]
    sb = codec.slot_bytes(G, scheme)
    n_chunks = (n_groups + cg - 1) // cg
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + env.rank)
    x = torch.empty(n_groups * G, dtype=torch.float16, device=dev)
    for c0 in range(0, n_groups, cg):
        c1 = min(n_groups, c0 + cg)
        x[c0 * G:c1 * G].normal_(generator=gen)
    payload = torch.empty((n_groups, sb), dtype=torch.uint8, device=dev)
    scales = torch.empty(n_groups, dtype=torch.float32, device=dev)
    comp = torch.empty(n_groups, dtype=torch.int32, device=dev)
    out_groups = n_groups if n_groups * G * 2 <= (4 << 30) else min(cg, n_groups)   # whole shard, or one launch chunk
    out = torch.empty((out_groups, G), dtype=torch.float16, device=dev)
    gathered = torch.empty(world * n_groups, dtype=torch.int32, device=dev) if world > 1 else None
    main = torch.cuda.Stream(device=dev)
    side = torch.cuda.Stream(device=dev) if world > 1 else None

    def compress_all():
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        for c0 in range(0, n_groups, cg):
            n = min(cg, n_groups - c0)
            rc = L.speckv_ext_compress(x.data_ptr() + c0 * G * 2, 0, G, n, payload.data_ptr() + c0 * sb, sb,
                                       scales.data_ptr() + c0 * 4, comp.data_ptr() + c0 * 4, scheme, st)
            assert rc == 0, rc

    def decompress_all():
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        for c0 in range(0, n_groups, cg):
            n = min(cg, n_groups - c0)
            o = out.data_ptr() + (c0 * G * 2 if out_groups == n_groups else 0)
            rc = L.speckv_ext_decompress(payload.data_ptr() + c0 * sb, sb, scales.data_ptr() + c0 * 4,
                                         comp.data_ptr() + c0 * 4, G, n, 0, o, None, scheme, st)
            assert rc == 0, rc

    graphs = None
    with torch.cuda.stream(main):
        s0 = codec.stats()["kernel_launches"]
        compress_all()
        decompress_all()                                    # also sizes the per-stream scratch before any capture
        launches_per_step = codec.stats()["kernel_launches"] - s0
        main.synchronize()
        if use_graph:
            try:
                graphs = (torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph())
                with torch.cuda.graph(graphs[0], stream=main):
                    compress_all()
                with torch.cuda.graph(graphs[1], stream=main):
                    decompress_all()
            except Exception as e:                          # noqa: BLE001 -- eager launches are the same kernels
                graphs = None
                spec = dict(spec, graph_error=str(e)[:200])
                torch.cuda.synchronize()

    def step(ev=None):
        if ev:
            ev[0].record(main)
        graphs[0].replay() if graphs else compress_all()
        if ev:
            ev[1].record(main)
        if world > 1:                                       # page-table metadata exchange, overlapped with the decode
            side.wait_stream(main)
            with torch.cuda.stream(side):
                dist.all_gather_into_tensor(gathered, comp)
        graphs[1].replay() if graphs else decompress_all()
        if ev:
            ev[2].record(main)
        if world > 1:
            main.wait_stream(side)                          # the next step rewrites comp

    sampler = None
    with torch.cuda.stream(main):
        # NVML answers in ~5-10 ms, the timed region at N = 8 lasts ~6 ms: the sampler runs from the first warm-up step
        # (the same kernels, back to back) to the end of the timed region and marks the samples taken inside it
        if sample_clocks:
            sampler = ClockSampler(env.local_rank, period=0.002)
            sampler.start()
        # >= W warm-up steps, then as many more as fill ~0.25 s (clocks are up before the timed region); the number is
        # agreed between the ranks -- every step holds a collective
        n_warm = max(warmup, 3)
        for _ in range(n_warm):
            step()                                          # includes one-time costs (NCCL connection set-up)
        main.synchronize()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record(main)
        for _ in range(3):
            step()
        w1.record(main)
        main.synchronize()
        n_warm += 3
        per_step_ms, = env.reduce([w0.elapsed_time(w1) / 3])
        extra = int(min(2000, max(0.0, 250.0 / max(per_step_ms, 1e-3) - n_warm)))
        for i in range(extra):
            step()
            if i % 16 == 15:
                main.synchronize()
        n_warm += extra
        env.barrier()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        if sampler:
            sampler.mark()
        t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        env.barrier()
        t_start.record(main)
        for i in range(steps):
            step(evs[i])
        t_end.record(main)
        env.barrier()
    clocks = sampler.stop() if sampler else None
    elapsed_ms = t_start.elapsed_time(t_end)
    t_comp = sum(e[0].elapsed_time(e[1]) for e in evs) / steps
    t_dec = sum(e[1].elapsed_time(e[2]) for e in evs) / steps
    elapsed_max, = env.reduce([elapsed_ms])
    per_rank_ms = env.gather_floats(elapsed_ms / steps)
    kv_bytes = n_groups * G * 2
    comp_total = int(comp.to(torch.int64).sum().item())
    kv_all, comp_all, groups_all = env.reduce([kv_bytes, comp_total, n_groups], "sum")
    ms_per_step = elapsed_max / steps
    value = kv_all / (ms_per_step * 1e-3) / 1e9

    # correctness of what was timed: the round trip of the first groups equals the library's one-shot path
    chk = min(n_groups, 8)
    ref = codec.decompress(codec.compress(x[:chk * G], G, scheme=scheme))
    assert torch.equal(ref.view(torch.int16), out[:chk].view(torch.int16)) or out_groups != n_groups, "bench output differs"
    if dump_dir:
        # with one launch chunk of output buffer, `out` holds the last chunk's decode
        first_held = 0 if out_groups == n_groups else (n_groups - 1) // cg * cg
        dump_outputs(dump_dir, env, first_held, payload, scales, comp, out)

    peak, peak_src = hbm_peak()
    alg_comp = 2 * G * n_groups + comp_total + 12 * n_groups       # 2n read + c write + 12 B header per group
    alg_dec = comp_total + 12 * n_groups + 2 * G * n_groups        # c + header read, 2n write
    comp_gbs = alg_comp / (t_comp * 1e-3) / 1e9
    dec_gbs = alg_dec / (t_dec * 1e-3) / 1e9
    dom = "compress" if t_comp >= t_dec else "decompress"
    tr = ncu_traffic(dom)
    roofline = {"bound": "hbm", "kernel": f"kv_{dom} ({dom}_fast_kernel)", "achieved": comp_gbs if dom == "compress" else dec_gbs,
                "peak": peak, "unit": "GB/s", "frac": (comp_gbs if dom == "compress" else dec_gbs) / peak, "peak_source": peak_src,
                "traffic": (tr["dram_bytes_per_group"] * min(cg, n_groups)) if tr else None,
                "traffic_source": tr.get("source") if tr else None,
                "algorithmic_bytes_per_launch": (alg_comp if dom == "compress" else alg_dec) / n_chunks,
                "ms_per_launch": (t_comp if dom == "compress" else t_dec) / n_chunks, "launches_per_phase": n_chunks,
                "timing": "CUDA events on the launching stream around each phase of every timed step (this rank)",
                "compress": {"GB/s": comp_gbs, "frac": comp_gbs / peak, "ms_per_step": t_comp,
                             "kv_GB/s": kv_bytes / (t_comp * 1e-3) / 1e9},
                "decompress": {"GB/s": dec_gbs, "frac": dec_gbs / peak, "ms_per_step": t_dec,
                               "kv_GB/s": kv_bytes / (t_dec * 1e-3) / 1e9},
                "roundtrip_frac": (alg_comp + alg_dec) / ((t_comp + t_dec) * 1e-3) / 1e9 / peak,
                "frac_of_nominal_8TBs": (comp_gbs if dom == "compress" else dec_gbs) / 8000.0}
    res = {"value": value, "ms_per_step": ms_per_step, "per_gpu_value": value / world, "per_rank_ms_per_step": per_rank_ms,
           "kv_bytes_per_step_total": int(kv_all), "groups_total": int(groups_all), "groups_per_rank": n_groups,
           "launch_chunk_groups": min(cg, n_groups), "warmup_steps_run": n_warm, "graph": bool(graphs), "graph_error": spec.get("graph_error"),
           "gpu_launches": int(launches_per_step) * steps,
           "compression_ratio": {"vs_fp16": kv_all / comp_all, "vs_fp32_reference_accounting": 2 * kv_all / comp_all},
           "roofline": roofline, "clocks": clocks}
    res["_x"] = x                                              # the e2e leg reuses the shard
    del payload, out, gathered
    return res


def pcie_ceiling(env, h_src, h_dst, passes, reps=4):
    """The e2e leg's copy schedule without its kernels: for every pass (h2d bytes, d2h bytes) the bytes move in 64 MiB
    pieces round-robin over three streams, H2D then D2H per piece, plain cudaMemcpyAsync from / to the SAME pinned
    buffers the e2e leg uses, every rank at the same time.  -> best seconds over `reps` (max over ranks per rep)."""
    torch, dev = env.torch, env.dev
    piece = 64 << 20
    streams = [torch.cuda.Stream(device=dev) for _ in range(3)]
    dbuf = [torch.empty(piece, dtype=torch.uint8, device=dev) for _ in range(3)]

    def one():
        i = 0
        for up, down in passes:
            n_pieces = max((up + piece - 1) // piece, (down + piece - 1) // piece)
            for j in range(n_pieces):
                k = i % 3
                i += 1
                with torch.cuda.stream(streams[k]):
                    a, b = j * piece, min(up, (j + 1) * piece)
                    if b > a:
                        dbuf[k][:b - a].copy_(h_src[a:b], non_blocking=True)
                    a, b = j * piece, min(down, (j + 1) * piece)
                    if b > a:
                        h_dst[a:b].copy_(dbuf[k][:b - a], non_blocking=True)
        torch.cuda.synchronize()

    one()
    best = None
    for _ in range(reps):
        env.barrier()
        t0 = time.perf_counter()
        one()
        dt, = env.reduce([time.perf_counter() - t0])
        best = dt if best is None else min(best, dt)
    return best


def e2e_leg(env, spec, x, steps, scheme=2):
    """The same round trip through the host-buffer C ABI: pinned host in -> payload in host memory -> host out,
    every H2D / D2H copy inside the timed region; next to it the plain-memcpy ceiling of the same bytes."""
    import ctypes as C

    import numpy as np

    torch, L, dev = env.torch, env.L, env.dev
    from cxl_speckv_b200 import codec

    G = spec["group_elems"]
    sb = codec.slot_bytes(G, scheme)
    ng = min(spec["n_groups"], max(1, int(env.args.e2e_mib * 2**20) // (G * 2)))
    nb_in, nb_pay = ng * G * 2, ng * sb
    ptrs = [L.speckv_ext_host_alloc(n) for n in (nb_in, nb_pay, nb_in, ng * 4, ng * 4)]
    assert all(ptrs), "pinned host allocation failed"
    h_in, h_pay, h_out, h_sc, h_cb = ptrs
    x_host = x[:ng * G].cpu().numpy()
    C.memmove(h_in, x_host.ctypes.data, nb_in)
    del x_host

    def e2e_step():
        rc = L.speckv_ext_compress_host(h_in, 0, G, ng, h_pay, sb, h_sc, h_cb, scheme)
        assert rc == 0, rc
        rc = L.speckv_ext_decompress_host(h_pay, sb, h_sc, h_cb, G, ng, 0, h_out, None, scheme)
        assert rc == 0, rc

    e2e_step()
    n_steps = max(1, min(steps, 5))
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(n_steps):
        e2e_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    dt, = env.reduce([dt])
    tot_in, = env.reduce([float(nb_in)], "sum")
    cb = np.ctypeslib.as_array(C.cast(h_cb, C.POINTER(C.c_uint32)), shape=(ng,))
    moved_pay = int(cb.astype(np.int64).sum())               # the host API ships comp_bytes of every slot, not the slot
    h2d, d2h = nb_in + moved_pay + 8 * ng, moved_pay + 8 * ng + nb_in
    # the host path must reproduce the device path bit for bit
    y = np.ctypeslib.as_array(C.cast(h_out, C.POINTER(C.c_uint16)), shape=(ng * G,))
    k = min(ng, 64)
    want = codec.decompress(codec.compress(x[:k * G], G, scheme=scheme))
    assert np.array_equal(y[:k * G], want.view(torch.int16).cpu().numpy().view(np.uint16).ravel()), "e2e output differs"
    # plain-copy ceiling on the same pinned buffers: pass 1 = compress_host's copies, pass 2 = decompress_host's
    as_t = lambda p, n: torch.from_numpy(np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n,)))
    t_ceil = pcie_ceiling(env, as_t(h_in, nb_in), as_t(h_out, nb_in), [(nb_in, moved_pay), (moved_pay, nb_in)])
    for p in ptrs:
        L.speckv_ext_host_free(p)
    traffic = (h2d + d2h) * env.world
    return {"value": tot_in * n_steps / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "steps": n_steps, "api": "speckv_ext_compress_host + speckv_ext_decompress_host (pinned host buffers)",
            "sample": f"{ng} groups ({nb_in / 2**20:.0f} MiB fp16) per rank per step",
            "pcie_traffic_GBs": traffic * n_steps / dt / 1e9,
            "pcie_ceiling_GBs": traffic / t_ceil / 1e9,
            "pcie_ceiling": "the same copy schedule without the kernels: plain cudaMemcpyAsync of the step's H2D / D2H bytes in 64 MiB pieces over 3 streams, same pinned buffers, all ranks concurrently, best of 4",
            "frac_of_ceiling": (t_ceil * n_steps) / dt}


def aux_cfg5(env, use_graph):
    """Batch-256 decode step (BASELINE config 5): LSTM prefetch scoring (k = 4) with residency filter and
    PrefetchRequest emission on the device -> N > 1: NCCL all-gather of the request tables (the only collective)
    -> device-side routing to the owning rank -> decompress of the predicted blocks with a device-side count.
    No host synchronisation inside a step; the step is one CUDA graph where the capture allows it."""
    import numpy as np

    torch, dist, dev, world, rank = env.torch, env.dist, env.dev, env.world, env.rank
    from cxl_speckv_b200 import codec, prefetch

    rng = np.random.default_rng(1)
    emb = ((rng.random((32000, 64), dtype=np.float32) - 0.5) * 0.1).astype(np.float32)
    wout = ((rng.random((32000, 128), dtype=np.float32) - 0.5) * 0.1).astype(np.float32)
    prefetch.load_predictor(emb, wout)
    batch, k = 256, 4
    all_toks = np.random.default_rng(7).integers(0, 32000, (batch, 16)).astype(np.int32)
    per = (batch + world - 1) // world
    toks = torch.from_numpy(all_toks[rank * per:(rank + 1) * per]).to(dev)
    G, n_blocks = G_BLOCK, 4096                                   # 1 GiB of stored blocks in all, contiguous ranges per rank
    per_blocks = (n_blocks + world - 1) // world
    local_blocks = max(0, min(per_blocks, n_blocks - rank * per_blocks))
    x = torch.empty(local_blocks * G, device=dev, dtype=torch.float16).normal_()
    c = codec.compress(x, G)
    cap = per * k                                                 # requests per table
    table = torch.zeros((prefetch.table_records(per, k), prefetch.REQUEST_BYTES), dtype=torch.uint8, device=dev)
    tables = torch.zeros((world,) + tuple(table.shape), dtype=torch.uint8, device=dev) if world > 1 else table
    block_index = torch.zeros(world * cap, dtype=torch.int32, device=dev)
    count = torch.zeros(1, dtype=torch.int32, device=dev)
    out = torch.empty((world * cap, G), dtype=torch.float16, device=dev)   # worst case: every prediction lands here
    main = torch.cuda.Stream(device=dev)

    def score_part():
        prefetch.emit(toks, k=k, layer_id=0, timestamp=1, table=table)

    def decode_part():
        prefetch.route(tables, world, cap, n_blocks, world, rank, block_index=block_index, count=count)
        codec.decompress_routed(c, block_index, count, out)

    def exchange():
        if world > 1:
            dist.all_gather_into_tensor(tables.view(-1), table.view(-1))

    def eager_step():
        score_part()
        exchange()
        decode_part()

    graph, graph_note = None, None
    with torch.cuda.stream(main):
        for _ in range(3):
            eager_step()
        main.synchronize()
        if use_graph:
            try:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=main):
                    eager_step()
            except Exception as e:                               # noqa: BLE001
                graph, graph_note = None, str(e)[:200]
                torch.cuda.synchronize()
        step = graph.replay if graph else eager_step
        for _ in range(3):
            step()
        env.barrier()
        reps = 20
        a, m, b = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record(main)
        for _ in range(reps):
            score_part()
        m.record(main)
        for _ in range(reps):
            step()
        b.record(main)
        env.barrier()
    n_dec = int(count.item())
    # what was decoded is what the requests name
    bi = block_index[:n_dec].long()
    full = codec.decompress(c)
    assert torch.equal(out[:n_dec].view(torch.int16), full[bi].view(torch.int16)), "cfg5: routed decode differs"
    t_score, t_step = env.reduce([a.elapsed_time(m) / reps, m.elapsed_time(b) / reps])
    n_all, = env.reduce([float(n_dec)], "sum")
    return {"workload": "cfg5: 256 sequences x 16-token history, vocab 32000, k=4 -> 1024 predicted blocks of 1024x128 fp16, "
                        f"sequences and stored blocks split over {world} GPU(s)",
            "n_gpus": world, "score_ms": t_score, "step_ms": t_step, "step": "emit (score + residency filter + request records)"
            " -> all-gather of request tables -> route -> routed decompress", "graph": bool(graph), "graph_error": graph_note,
            "blocks_decoded_per_step": n_all, "step_seq_per_s": batch / t_step * 1e3,
            "decoded_kv_GB/s": n_all * G * 2 / (t_step * 1e-3) / 1e9, "reference_cpu_ms_per_sequence": 17.8,
            "exchange": "none (1 GPU)" if world == 1 else f"NCCL all-gather of {world} tables x {1 + cap} PrefetchRequest records (32 B)"}


def aux_tier(env):
    """BASELINE config 4 data path: Llama-3-8B 32K-context KV as 4 KiB pages, address translation + page-table
    lookup for every page, offload -> restore through the pinned host pool (PCIe GB/s of stored bytes)."""
    import ctypes as C

    import numpy as np

    torch, L, dev = env.torch, env.L, env.dev
    from cxl_speckv_b200 import codec
    from cxl_speckv_b200.tier import HostTier

    layers = max(1, int(round(32 * env.args.tier_scale)))
    G, pages = 2048, layers * 2 * 8 * 32768 * 128 // 2048
    gen = torch.Generator(device=dev)
    gen.manual_seed(4321 + env.rank)
    x = torch.empty(pages * G, dtype=torch.float16, device=dev).normal_(generator=gen)

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    assert L.speckv_init(f"cuda:{env.local_rank}".encode()) == 0
    h = C.c_uint64()
    assert L.speckv_alloc(pages * 4096, None, C.byref(h)) == 0
    tbl = torch.empty(pages * 3, dtype=torch.int64, device=dev)
    cnt = C.c_size_t()
    assert L.speckv_ext_page_table_export(h.value, tbl.data_ptr(), pages, C.byref(cnt), None) == 0
    va = (torch.arange(pages, dtype=torch.int64, device=dev) << 12) + (h.value << 32) + 0x123
    pa = torch.empty_like(va)
    fl = torch.empty(pages, dtype=torch.int32, device=dev)
    t_tr = timed(lambda: codec.translate(va, out=pa))
    t_lk = timed(lambda: L.speckv_ext_page_lookup(tbl.data_ptr(), pages, h.value << 32, va.data_ptr(), pa.data_ptr(), fl.data_ptr(), pages, None))
    assert int(pa[5].item()) == 0x4000000000 + (h.value << 20) + (5 << 12) + 0x123
    L.speckv_finalize()
    del tbl, va, pa, fl

    tier = HostTier(int(pages * G * 2 * 1.02) + (64 << 20))
    ids = np.arange(pages, dtype=np.uint64) << np.uint64(12)
    warm = min(pages, 65536)
    tier.offload(x[:warm * G], G, ids[:warm])
    tier.drop(ids[:warm])
    env.barrier()
    t0 = time.perf_counter()
    tier.offload(x, G, ids)
    torch.cuda.synchronize()
    t_off = time.perf_counter() - t0
    st_off = tier.stats()
    out = torch.empty((pages, G), dtype=torch.float16, device=dev)
    tier.restore(ids[:warm], G, torch.float16, out=out[:warm])
    env.barrier()
    t0 = time.perf_counter()
    tier.restore(ids, G, torch.float16, out=out)
    torch.cuda.synchronize()
    t_res = time.perf_counter() - t0
    st = tier.stats()
    k = min(pages, 4096)
    want = codec.decompress(codec.compress(x[:k * G], G))
    assert torch.equal(out[:k].view(torch.int16), want.view(torch.int16)), "tier: restored pages differ"
    tier.close()
    t_off_max, t_res_max = env.reduce([t_off, t_res])
    stored, = env.reduce([float(st_off["last_offload_stored_bytes"])], "sum")
    restored, = env.reduce([float(st["last_restore_stored_bytes"])], "sum")
    kv_all = pages * G * 2 * env.world
    return {"workload": f"cfg4: Llama-3-8B 32K ctx paged KV per GPU, {layers} layers, {pages} pages of 4 KiB, offload -> restore through the pinned host pool",
            "n_gpus": env.world, "translate_Gaddr_per_s": pages / t_tr / 1e6, "translate_GB/s": pages * 16 / t_tr / 1e6,
            "page_lookup_Gaddr_per_s": pages / t_lk / 1e6,
            "offload": {"s": t_off_max, "stored_bytes": stored, "pcie_GB/s": stored / t_off_max / 1e9, "kv_GB/s": kv_all / t_off_max / 1e9},
            "restore": {"s": t_res_max, "stored_bytes": restored, "pcie_GB/s": restored / t_res_max / 1e9, "kv_GB/s": kv_all / t_res_max / 1e9},
            "pcie_GB/s_per_gpu": {"offload": stored / t_off_max / 1e9 / env.world, "restore": restored / t_res_max / 1e9 / env.world},
            "verified": "restored pages == device compress -> decompress, bit for bit"}


def aux_ratios(env, n_groups=4096, reps=8):
    """Compression ratio, reconstruction error and codec throughput per value distribution (SURVEY.md section 8d)
    and per scheme; rank 0 only."""
    torch, dev = env.torch, env.dev
    from cxl_speckv_b200 import codec

    G = G_BLOCK
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)
    base = torch.empty(n_groups * G, dtype=torch.float16, device=dev).normal_(generator=gen)
    peak, _ = hbm_peak()
    dists = {
        "normal_fp16": (base, 2),
        "normal_bf16": (base.to(torch.bfloat16), 2),
        "zeros_fp16": (torch.zeros_like(base), 2),
        "runs300_fp16": (base[: (n_groups * G + 299) // 300].repeat_interleave(300)[: n_groups * G].contiguous(), 2),
        "zero_tail60_fp16": (torch.where((torch.arange(G, device=dev) < int(G * 0.4)).repeat(n_groups), base, torch.zeros_like(base)), 2),
        "smooth_fp16": ((torch.cumsum(base.float().view(n_groups, G) * 0.01, 1)).to(torch.float16).view(-1), 2),
        "normal_fp16_int8": (base, 1),
        "normal_fp16_fp16": (base, 0),
    }
    for name, sid in SCHEME_IDS.items():
        if sid > 2:
            dists[f"normal_fp16_{name}"] = (base, sid)
            dists[f"smooth_fp16_{name}"] = (dists["smooth_fp16"][0], sid)
    res = {}
    for name, (x, scheme) in dists.items():
        try:
            c = codec.compress(x, G, scheme=scheme)
            y = codec.decompress(c)
            torch.cuda.synchronize()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
            for _ in range(reps):
                codec.compress(x, G, scheme=scheme, out=c)
            ev[1].record()
            for _ in range(reps):
                codec.decompress(c, out=y)
            ev[2].record()
            torch.cuda.synchronize()
            tc, td = ev[0].elapsed_time(ev[1]) / reps, ev[1].elapsed_time(ev[2]) / reps
            cb = float(c.comp_bytes.to(torch.int64).sum().item())
            raw = n_groups * G * 2
            mse = ((y.float() - x.view(n_groups, G).float()) ** 2).mean().item()
            res[name] = {"scheme": scheme, "ratio_vs_fp16": raw / cb, "ratio_fp32_reference_accounting": 2 * raw / cb,
                         "compress_kv_GB/s": raw / tc / 1e6, "decompress_kv_GB/s": raw / td / 1e6,
                         "compress_algorithmic_GB/s": (raw + cb) / tc / 1e6, "decompress_algorithmic_GB/s": (raw + cb) / td / 1e6,
                         "compress_frac_of_peak": (raw + cb) / tc / 1e6 / peak, "decompress_frac_of_peak": (raw + cb) / td / 1e6 / peak,
                         "roundtrip_mse": mse}
            del c, y
        except Exception as e:                                   # noqa: BLE001
            res[name] = {"error": str(e)[:200]}
    return {"workload": f"{n_groups} groups of 1024x128 per distribution ({n_groups * G * 2 >> 20} MiB of KV per call, {reps} calls "
                        "per direction through the library API, CUDA events around them)", "distributions": res}


_T0 = time.perf_counter()


def log(rank, msg):
    if rank == 0:
        print(f"[bench {time.perf_counter() - _T0:7.2f}s] {msg}", file=sys.stderr, flush=True)


def run_cuda(args, rank, world, local_rank):
    all_cpus = bind_to_gpu_cpus(local_rank)
    env = Env(args, rank, world, local_rank)
    torch = env.torch
    use_graph = not args.no_graph
    spec = workload_spec(args.workload, world, rank, args.scale)
    log(rank, f"headline {args.workload} x{world} ...")
    head = codec_roundtrip(env, spec, args.steps, args.warmup, use_graph, sample_clocks=True, dump_dir=args.dump_outputs)
    x = head.pop("_x")
    e2e = None
    if not args.no_e2e:
        log(rank, "e2e ...")
        e2e = e2e_leg(env, spec, x, args.steps)
    del x
    torch.cuda.empty_cache()

    aux = {}
    wanted = [a for a in args.aux.split(",") if a and a != "none"]

    def leg(name, fn):
        env.barrier()
        log(rank, f"aux.{name} ...")
        t0 = time.perf_counter()
        try:
            r = fn()
        except Exception as e:                                   # noqa: BLE001 -- an auxiliary record must not cost the headline
            r = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
        if isinstance(r, dict):
            r["wall_s"] = round(time.perf_counter() - t0, 2)
        aux[name] = r
        torch.cuda.empty_cache()

    if "cfg2" in wanted and args.workload != "cfg2":
        def cfg2():
            s2 = workload_spec("cfg2", world, rank, args.aux_scale)
            r = codec_roundtrip(env, s2, max(1, min(args.steps, 4)), 3, use_graph, sample_clocks=True)
            r.pop("_x")
            return dict(r, workload=s2["label"], scaling="weak", unit=UNIT)
        leg("cfg2", cfg2)
    if "schemes" in wanted:
        def schemes():
            # the same shard under the other schemes: 1 = the reference's codes only, 3 / 4 = the non-wrapping quantiser
            # (extension ids; NOT reference behaviour) with and without delta + RLE
            out = {}
            for name in ("int8", "int8_clamp_delta_rle", "int8_clamp"):
                r = codec_roundtrip(env, spec, max(1, min(args.steps, 5)), 3, use_graph, scheme=SCHEME_IDS[name])
                xs = r.pop("_x")
                rec = {"scheme_id": SCHEME_IDS[name], "value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"],
                       "compression_ratio_vs_fp16": r["compression_ratio"]["vs_fp16"],
                       "compress_frac_of_peak": r["roofline"]["compress"]["frac"], "decompress_frac_of_peak": r["roofline"]["decompress"]["frac"],
                       "compress_kv_GB/s": r["roofline"]["compress"]["kv_GB/s"], "decompress_kv_GB/s": r["roofline"]["decompress"]["kv_GB/s"]}
                if name == "int8_clamp" and not args.no_e2e:
                    e = e2e_leg(env, spec, xs, args.steps, scheme=SCHEME_IDS[name])
                    rec["e2e"] = {k: e[k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "pcie_traffic_GBs", "frac_of_ceiling")}
                del xs
                out[name] = rec
                env.torch.cuda.empty_cache()
            return {"workload": spec["label"], "schemes": out,
                    "note": "int8 = the reference's quantiser alone (wrapping codes, MSE ~ the data); the clamp schemes are this "
                            "library's extension ids 3 / 4 (s = max|x|, non-wrapping; aux.ratios gives their MSE)"}
        leg("schemes", schemes)
    if "cfg5" in wanted:
        leg("cfg5", lambda: aux_cfg5(env, use_graph))
    if "tier" in wanted:
        leg("tier", lambda: aux_tier(env))
    if "ratios" in wanted:
        leg("ratios", lambda: aux_ratios(env) if rank == 0 else None)    # every rank enters the leg (it starts with a barrier)
        env.barrier()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        log(rank, "cpu baseline ...")
        os.sched_setaffinity(0, all_cpus)
        cpu = cpu_roundtrip_rate(spec["group_elems"], args.cpu_seconds, os.cpu_count() or 1)
        cpu.pop("seconds", None)

    if rank == 0:
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "warmup_steps_run": head["warmup_steps_run"], "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": spec["scaling"], "vs_baseline": None, "dtype": "f32+i8",
                "data": "synthetic N(0,1) fp16 KV (torch seed 1234+rank)",
                "config": {"workload": spec["label"], "group_elems": spec["group_elems"], "groups_per_rank": head["groups_per_rank"],
                           "groups_total": head["groups_total"], "kv_bytes_per_step_total": head["kv_bytes_per_step_total"],
                           "launch_chunk_groups": head["launch_chunk_groups"], "global_batch": spec["global_batch"],
                           "parallelism": (f"layers split {world} ways (contiguous), no data-path collective; NCCL all-gather of the "
                                           "page-table metadata on a side stream" if world > 1 else "single GPU"),
                           "cuda_graph": head["graph"],
                           "cache": "each step streams this rank's shard (input + payload + output > L2) once per direction; no flush needed"},
                "per_gpu_value": head["per_gpu_value"], "per_rank_ms_per_step": head["per_rank_ms_per_step"],
                "compression_ratio": head["compression_ratio"], "clocks": head["clocks"], "e2e": e2e,
                "gpu_launches": head["gpu_launches"], "roofline": head["roofline"], "cpu_baseline": cpu, "aux": aux}
        print(json.dumps(line), flush=True)
    if world > 1:
        env.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg2", "cfg3", "cfg4p"], help="headline workload")
    ap.add_argument("--aux", default="cfg2,schemes,cfg5,tier,ratios", help="comma list of sub-records to add (or 'none')")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the headline workload's layers (debug only; cfg2 / cfg4p)")
    ap.add_argument("--aux-scale", type=float, default=1.0, help="fraction of aux.cfg2's layers (debug only)")
    ap.add_argument("--tier-scale", type=float, default=1.0, help="fraction of aux.tier's layers (debug only)")
    ap.add_argument("--e2e-mib", type=float, default=2560.0, help="host-buffer sample per rank per e2e step (MiB of fp16 KV)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="CUDA path only (--impl cuda): write the headline round trip's "
                    "outputs of its last timed step to DIR/<name>.npy (scales and sizes of every group, payload and "
                    "decoded values of 16 seeded groups; at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the CUDA path's outputs")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_cuda(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
