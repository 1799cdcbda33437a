#!/usr/bin/env python
"""bench.py — segment transform throughput (BASELINE.json metric) on N B200s, one process per GPU.

A "step" = one pass of the hot path over one synthetic segment (default: 1 GiB, 4 MiB chunks, Zstd + AES-256-GCM,
i.e. BASELINE.json configs[3], which is the configuration the metric is quoted on and fits one GPU).
  value   device-resident: the segment is already in HBM, output slots stay in HBM (CUDA events, max over ranks)
  e2e     the reference-facing C-ABI call tsgpu_transform with HOST (pinned) buffers: H2D + kernels + D2H timed
  roofline  dominant kernel: algorithmic bytes / CUDA-event duration of that kernel vs MEASURED_PEAKS.json
  cpu_baseline  the oracle (libzstd + OpenSSL stand-in for zstd-jni + JCE, see oracle/tsoracle.h) on host cores
`--impl reference` times that CPU path with all host threads on the same config (rank 0 only).
Weak scaling: every rank transforms its own segment; value = total original bytes / max-over-ranks time.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GIB = float(1 << 30)
MIB = 1 << 20
METRIC = "segment_transform_GiB_per_s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="tsgpu", choices=["tsgpu", "reference"])
    ap.add_argument("--workload", default="zstd+aes", choices=["zstd+aes", "aes", "zstd", "none"])
    ap.add_argument("--corpus", default="K", choices=["K", "R", "Z"])
    ap.add_argument("--segment-mib", type=int, default=1024)
    ap.add_argument("--chunk-mib", type=int, default=4)
    ap.add_argument("--cpu-sample-mib", type=int, default=0, help="0 = auto (aim for ~10 s of CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--zstd-mode", default="speed", choices=["speed", "dense"],
                    help="speed: independent 8 KiB blocks (default, TSGPU_FLAG_ZSTD); dense: 64 KiB regions, shared tables "
                         "(TSGPU_FLAG_ZSTD | TSGPU_FLAG_ZSTD_DENSE) — denser, slower, byte-identical frames on every run")
    ap.add_argument("--direction", default="transform", choices=["transform", "fetch"],
                    help="fetch = BASELINE configs[4]: ranged fetchLogSegment, 16 MiB windows of a 1 GiB segment")
    ap.add_argument("--frames", default="own", choices=["own", "libzstd"],
                    help="fetch only: who wrote the segment (libzstd = the reference's writer, via the CPU arm)")
    ap.add_argument("--window-mib", type=int, default=16)
    ap.add_argument("--config", type=int, default=None, choices=[0, 1, 2, 3, 4],
                    help="shorthand for BASELINE.json configs[N] (0: 256 MiB no transform, 1: zstd, 2: aes, 3: zstd+aes, 4: ranged fetch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_transform_outputs)")
    a = ap.parse_args()
    if a.config is not None:
        if a.config == 0:
            a.workload, a.segment_mib = "none", 256
        elif a.config == 4:
            a.workload, a.direction = "zstd+aes", "fetch"
        else:
            a.workload = {1: "zstd", 2: "aes", 3: "zstd+aes"}[a.config]
    if a.dump_outputs and (a.impl != "tsgpu" or a.direction != "transform" or a.workload == "none"):
        ap.error("--dump-outputs covers the GPU transform path only (--impl tsgpu, --direction transform, a transforming workload)")
    return a


def flags_of(workload, mode="speed"):
    f = {"zstd+aes": 3, "aes": 2, "zstd": 1, "none": 0}[workload]
    return f | (4 if (f & 1) and mode == "dense" else 0)


def config_index(args):
    if args.direction == "fetch":
        return 4
    return {"zstd+aes": 3, "aes": 2, "zstd": 1, "none": 0}[args.workload]


def config_of(args, n_gpus):
    return {
        "workload": "%s%d MiB segment per GPU, %d MiB chunks, %s, corpus %s (BASELINE configs[%d])" % (
            ("ranged fetch of %d MiB windows (%s-written frames) from a " % (args.window_mib, args.frames)) if args.direction == "fetch" else "",
            args.segment_mib, args.chunk_mib, args.workload, args.corpus, config_index(args)),
        "segment_bytes": args.segment_mib * MIB, "chunk_bytes": args.chunk_mib * MIB,
        "transform": args.workload, "corpus": args.corpus, "zstd_mode": args.zstd_mode if "zstd" in args.workload else None,
        "parallelism": "segments sharded across %d GPU(s), no data-path collective" % n_gpus,
        "l2_policy": "inputs (segment >= 1 GiB) larger than the 126 MB L2; no explicit flush",
    }


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []          # (arrival time, csv line)
        self.proc = None
        self.t0 = self.t1 = None

    def begin(self):
        self.t0 = time.monotonic()

    def end(self):
        self.t1 = time.monotonic()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        # samples that arrived inside the timed region; if the region was shorter than the sampling period, the samples
        # taken under the same load right before it (warm-up runs the identical step) are used and counted separately
        inside = [r for (t, r) in self.rows if self.t0 is not None and self.t0 <= t <= (self.t1 or t)]
        rows = inside if inside else [r for (t, r) in self.rows][-5:]
        sm, mx, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_inside_timed_region": len(inside)}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_segment(args, segment_id):
    from tsgpu import corpus
    return corpus.gen_segment(args.corpus, segment_id, args.segment_mib * MIB, args.chunk_mib * MIB)


# ------------------------------------------------------------------------------------------ CPU arm (oracle)
def cpu_transform_chunks(ora, flags, src, cs, key, aad, ivs, lo, hi):
    """virtual chunks [lo, hi) through the oracle's chain, one chunk at a time like the reference's pull pipeline;
    virtual chunk v is chunk v mod nch of the sample (several passes over the sample keep every worker busy)"""
    n = src.size
    nch = max(1, (n + cs - 1) // cs)
    out = 0
    for v in range(lo, hi):
        i = v % nch
        a, b = i * cs, min(n, (i + 1) * cs)
        t, sizes = ora.transform_segment(flags, src[a:b], cs, key, aad, ivs[12 * i:12 * i + 12])
        out += sizes[0]
    return out


_POOL_STATE = {}


def _pool_job(r):
    st = _POOL_STATE
    c0 = time.process_time()
    if st.get("objects") is not None:            # fetch direction: decrypt + decompress chunk by chunk (DefaultChunkManager.getChunk)
        objs = st["objects"]
        for v in range(r[0], r[1]):
            t = objs[v % len(objs)]
            st["ora"].detransform_chunks(st["flags"], t, [t.size], st["cs"], st["key"], st["aad"])
    else:
        cpu_transform_chunks(st["ora"], st["flags"], st["src"], st["cs"], st["key"], st["aad"], st["ivs"], r[0], r[1])
    return time.process_time() - c0


class CpuArm:
    """The oracle's chain over the first `sample_bytes` of a segment on `threads` host cores.  threads > 1 uses
    forked worker processes kept alive across steps (per-chunk contexts and buffers are freshly allocated, as in
    the reference; separate address spaces keep page-fault handling off one mm lock, and warm-up passes populate
    the forked page tables before anything is timed).  Every worker gets at least `min_chunks_per_worker` chunks
    per step (the sample is passed over several times if needed) so that dispatch latency does not dominate."""

    def __init__(self, args, flags, src, threads, sample_bytes, min_chunks_per_worker=1, fetch=False):
        from oracle import oracle as ora
        from tsgpu import corpus
        self.cs = args.chunk_mib * MIB
        self.nch = max(1, min(src.size, sample_bytes) // self.cs)
        key, aad, ivs = corpus.fixed_key_material(self.nch)
        objects = None
        if fetch:                                # the reference-written chunks to be fetched (produced before anything is timed)
            objects = []
            for i in range(self.nch):
                t, _ = ora.transform_segment(flags & 3, src[i * self.cs:(i + 1) * self.cs], self.cs, key, aad, ivs[12 * i:12 * i + 12])
                objects.append(np.array(t, copy=True))
        self.rounds = max(1, -(-min_chunks_per_worker * threads // self.nch)) if threads > 1 else 1
        total = self.nch * self.rounds
        per = (total + threads - 1) // threads
        self.ranges = [(k * per, min(total, (k + 1) * per)) for k in range(threads) if k * per < total]
        flags &= 3                                # the CPU chain has one compressor: libzstd level 3
        _POOL_STATE.update(ora=ora, flags=flags, src=src[:self.nch * self.cs], cs=self.cs, key=key, aad=aad, ivs=ivs, objects=objects)
        self.pool = None
        self.cpu_seconds = 0.0
        if len(self.ranges) > 1:
            import multiprocessing as mp
            self.pool = mp.get_context("fork").Pool(len(self.ranges))

    @property
    def cores(self):
        return len(self.ranges)

    def step(self):
        """one pass; returns (bytes, seconds)"""
        t0 = time.perf_counter()
        if self.pool is None:
            cpu = [_pool_job(self.ranges[0])]
        else:
            cpu = self.pool.map(_pool_job, self.ranges, chunksize=1)
        dt = time.perf_counter() - t0
        self.cpu_seconds += float(sum(cpu))
        return self.nch * self.rounds * self.cs, dt

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as ora
    flags = flags_of(args.workload, args.zstd_mode)
    threads = os.cpu_count() or 1
    # a bounded sample of the same workload: the first sample_mib of the segment, all host cores
    sample_mib = args.cpu_sample_mib or min(args.segment_mib, 64 * threads)
    seg_args = argparse.Namespace(**vars(args))
    seg_args.segment_mib = sample_mib
    src = make_segment(seg_args, 0)
    arm = CpuArm(args, flags, src, threads, src.size, min_chunks_per_worker=8, fetch=args.direction == "fetch")
    for _ in range(max(1, args.warmup)):
        arm.step()
    arm.cpu_seconds = 0.0
    t_tot, b_tot = 0.0, 0
    for _ in range(args.steps):
        nbytes, dt = arm.step()
        t_tot += dt; b_tot += nbytes
    used = arm.cores
    busy = arm.cpu_seconds / t_tot if t_tot > 0 else 0.0      # CPU-seconds burnt per wall second = cores actually granted
    rounds = arm.rounds
    arm.close()
    val = b_tot / GIB / t_tot
    line = {
        "metric": "ranged_fetch_GiB_per_s" if args.direction == "fetch" else METRIC, "value": val, "unit": "GiB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * t_tot / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "impl": "reference", "config": config_of(args, args.gpus),
        "cpu_baseline": {"value": val, "unit": "GiB/s", "cores": used, "kind": "port",
                         "effective_cores": round(busy, 1),
                         "sample": "first %d MiB of the segment, %d pass(es) per step, on %d worker processes (%.1f CPU-seconds "
                                   "consumed per wall second: what the host actually granted); libzstd %s level 3 + OpenSSL "
                                   "EVP AES-256-GCM standing in for zstd-jni 1.5.6-9 + SunJCE (no JVM in the image)" % (
                                       sample_mib, rounds, used, busy, ora.lib().ora_zstd_version().decode())},
        "e2e": {"value": val, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------ fetch direction (configs[4])
def fetch_windows(nch, wch):
    """first chunk of each window: start, middle, end of the segment, then a sweep (SURVEY.md §8d C5)"""
    firsts = [0, nch // 2, nch - wch] + [(k * 37) % (nch - wch + 1) for k in range(1, 14)]
    seen, out = set(), []
    for f in firsts:                                   # (a window as large as the segment — the bulk decode line — has one position)
        f = min(f, nch - wch)
        if f not in seen:
            seen.add(f); out.append(f)
    return out


def make_object(args, flags, src_np, ctx_host, key, aad, ivs):
    """the uploaded .log object of the segment and its chunk sizes, written by this library or by the reference's
    writer (libzstd level 3 + JCE stand-in: the CPU arm — used only to PRODUCE a reference-written object, never timed)"""
    cs = args.chunk_mib * MIB
    if args.frames == "own":
        return ctx_host.transform(flags, src_np, cs, key, aad, ivs)
    from oracle import oracle as ora
    return ora.transform_segment(flags & 3, src_np, cs, key, aad, ivs)


def main_fetch(args):
    """BASELINE configs[4]: ranged fetchLogSegment — decrypt + decompress the chunks covering a 16 MiB window of a 1 GiB
    segment.  A step = one window.  value: transformed chunks resident in HBM (detransform_device, CUDA events);
    e2e: tsgpu_detransform with host buffers (H2D of the transformed chunks, kernels, D2H of the window)."""
    import torch
    import torch.distributed as dist
    import tsgpu
    from tsgpu import corpus
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl tsgpu needs a GPU: libtsgpu has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    bind_to_gpu_numa_node(torch, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    flags = flags_of(args.workload, args.zstd_mode)
    seg, cs = args.segment_mib * MIB, args.chunk_mib * MIB
    nch, wch = seg // cs, max(1, args.window_mib // args.chunk_mib)
    key, aad, ivs = corpus.fixed_key_material(nch)
    src_np = make_segment(args, rank)
    hctx = tsgpu.Context(max_chunk_bytes=cs, max_batch=max(wch + 1, 4), devices=[local])
    obj, tsz = make_object(args, flags, src_np, hctx, key, aad, ivs)
    pos = np.concatenate([[0], np.cumsum(np.asarray(tsz, dtype=np.int64))])
    ctx = tsgpu.Context(max_chunk_bytes=cs, max_batch=wch, devices=[local])
    stride = ctx.slot_stride(flags, cs)
    firsts = fetch_windows(nch, wch)
    # device-resident: every window's chunks sit in slots
    wins = []
    for f in firsts:
        slots = np.zeros(wch * stride, dtype=np.uint8)
        for k in range(wch):
            slots[k * stride + 4:k * stride + 4 + tsz[f + k]] = obj[pos[f + k]:pos[f + k + 1]]
        wins.append((torch.from_numpy(slots).to(dev), torch.tensor(tsz[f:f + wch], dtype=torch.int32, device=dev)))
    d_dst = torch.zeros(wch * cs, dtype=torch.uint8, device=dev)
    d_osz = torch.zeros(wch, dtype=torch.int32, device=dev); d_st = torch.zeros(wch, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 * MIB, dtype=torch.uint8, device=dev)      # > 126 MB L2: written between timed windows

    def step_device(i):
        d_slots, d_sizes = wins[i % len(wins)]
        ctx.detransform_device(flags, d_slots.data_ptr(), stride, d_sizes.data_ptr(), wch, cs, key, aad, d_dst.data_ptr(),
                               d_osz.data_ptr(), d_st.data_ptr(), stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        step_device(i)
    barrier()
    l0 = ctx.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    sampler.begin()
    ok = True
    for i in range(args.steps):
        flush.fill_(i & 255)                                              # L2 flush, outside the per-step events
        evs[i][0].record()
        step_device(i)
        evs[i][1].record()
        evs[i][1].synchronize()
        f = firsts[i % len(firsts)]
        ok = ok and int(d_st.abs().sum().item()) == 0
    barrier()
    sampler.end()
    ok = ok and bool(np.array_equal(d_dst.cpu().numpy(), src_np[f * cs:(f + wch) * cs]))      # last window, checked after timing
    ms = sum(a.elapsed_time(b) for a, b in evs)
    launches = ctx.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    win_bytes = wch * cs
    value = world * win_bytes * args.steps / GIB / (ms_max / 1000.0)

    ctx.profile_enable(True)
    step_device(0)
    rep = ctx.profile_report()
    ctx.profile_enable(False)
    kernels = {k: {"launches": v["launches"], "ms": v["ms"]} for k, v in rep.items()} if rep else None
    roofline = None
    if rep:
        name, rec = max(rep.items(), key=lambda kv: kv[1]["ms"])
        ms_k = rec["ms"] / rec["launches"]
        tbytes = int(sum(tsz[firsts[0]:firsts[0] + wch]))
        alg = tbytes + win_bytes                                          # transformed in + original out (SURVEY.md §8d)
        peak, how = load_peaks()
        roofline = {"bound": "hbm", "kernel": name, "achieved": alg / 1e9 / (ms_k / 1000.0), "peak": peak, "unit": "GB/s",
                    "frac": alg / 1e9 / (ms_k / 1000.0) / peak, "traffic": None, "peak_source": how,
                    "algorithmic_bytes_per_launch": alg, "kernel_ms": ms_k}

    e2e = None
    if not args.no_e2e:
        h_out = torch.empty(win_bytes, dtype=torch.uint8).pin_memory()
        h_in = torch.empty(int(max(pos[f + wch] - pos[f] for f in firsts)) + 64, dtype=torch.uint8).pin_memory()
        out_np, in_np = h_out.numpy(), h_in.numpy()
        def step_host(i):
            f = firsts[i % len(firsts)]
            n = int(pos[f + wch] - pos[f])
            in_np[:n] = obj[pos[f]:pos[f + wch]]                          # the bytes of the ranged GET, landing in pinned memory
            hctx.detransform(flags, in_np[:n], tsz[f:f + wch], win_bytes, key, aad, dst=out_np)
            return f, n
        for i in range(max(1, args.warmup)):
            step_host(i)
        barrier()
        h2d = 0
        t0 = time.perf_counter()
        for i in range(args.steps):
            f, n = step_host(i); h2d += n
        dt = time.perf_counter() - t0
        ok = ok and bool(np.array_equal(out_np, src_np[f * cs:(f + wch) * cs]))
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * win_bytes * args.steps / GIB / float(tt.item()), "unit": "GiB/s",
               "ms_per_window": 1000.0 * float(tt.item()) / args.steps,
               "h2d_bytes_per_step": h2d // args.steps, "d2h_bytes_per_step": win_bytes,
               "timer": "host wall clock around tsgpu_detransform (it synchronises internally), max over ranks"}
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import oracle as ora
        f = firsts[0]
        part = obj[pos[f]:pos[f + wch]]
        ora.detransform_chunks(flags & 3, part, tsz[f:f + wch], win_bytes, key, aad)
        t0 = time.perf_counter(); reps = 0
        while time.perf_counter() - t0 < 5.0:
            ora.detransform_chunks(flags & 3, part, tsz[f:f + wch], win_bytes, key, aad); reps += 1
        dtc = (time.perf_counter() - t0) / reps
        cpu = {"value": win_bytes / GIB / dtc, "unit": "GiB/s", "cores": 1, "kind": "port", "ms_per_window": 1000.0 * dtc,
               "sample": "%d x one %d MiB window, chunk-sequential on 1 thread like DefaultChunkManager.getChunk; libzstd %s + "
                         "OpenSSL EVP standing in for zstd-jni + SunJCE" % (reps, args.window_mib, ora.lib().ora_zstd_version().decode())}
    if rank == 0:
        print(json.dumps({
            "metric": "ranged_fetch_GiB_per_s", "value": value, "unit": "GiB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": dict(config_of(args, world),
                l2_policy="256 MiB written between timed windows (L2 flush), outside the per-window events"),
            "frames_written_by": args.frames, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "roofline": roofline, "cpu_baseline": cpu, "kernels_ms_per_step": kernels, "verified": {"windows_bit_exact": bool(ok)}}))
    if not ok:
        raise SystemExit("bench.py: a fetched window differs from the segment")
    ctx.close(); hctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------ configs[0]: ChunkIndex plumbing
def main_plumbing(args):
    """BASELINE configs[0]: 256 MiB segment, no compression / encryption (TransformFinisher's no-transform fast path,
    TransformFinisher.java:124-140): the bytes pass through unchanged, the fixed ChunkIndex is computed arithmetically and
    serialised.  The reference runs this on the CPU and so does the library (flags == 0 never touches the GPU), so this
    line has gpu_launches 0 by design; it exists so that every BASELINE config has a driver-runnable line."""
    import tsgpu
    from tsgpu import binding
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    seg, cs = args.segment_mib * MIB, args.chunk_mib * MIB
    src = make_segment(args, 0)
    ctx = tsgpu.Context(max_chunk_bytes=cs, max_batch=4)
    dst = np.empty(seg + 64, dtype=np.uint8)
    def step():
        out, sizes = ctx.transform(0, src, cs, dst=dst)
        js = binding.chunk_index_json(cs, seg, cs, sizes[-1])
        return out, sizes, js
    for _ in range(max(1, args.warmup)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out, sizes, js = step()
    dt = time.perf_counter() - t0
    ok = bool(np.array_equal(out, src)) and js == ('{"type":"fixed","originalChunkSize":%d,"originalFileSize":%d,'
                                                   '"transformedChunkSize":%d,"finalTransformedChunkSize":%d}' % (cs, seg, cs, cs))
    v = seg * args.steps / GIB / dt
    print(json.dumps({"metric": METRIC, "value": v, "unit": "GiB/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "u8", "data": "synthetic", "config": config_of(args, 1),
                      "e2e": {"value": v, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0, "note": "no-transform fast path: host memcpy + ChunkIndex arithmetic, no GPU work by design",
                      "chunk_index": js, "verified": {"bytes_unchanged_and_index_json": ok}}))
    ctx.close()
    return 0 if ok else 1


# ------------------------------------------------------------------------------------------ GPU arm
def bind_to_gpu_numa_node(torch, index):
    """Pin this rank to the CPUs next to its GPU so the pinned staging buffers are first-touched on the local NUMA
    node (matters for the PCIe-bound e2e number when 8 ranks share one host).  Best effort: any failure is ignored."""
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        cpus = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
    except Exception:
        pass


DUMP_BUDGET = 60_000_000        # bytes of .npy payload: --dump-outputs stays under 64 MB whatever the segment size


def dump_transform_outputs(path, d_slots, d_sizes, stride, nch):
    """Writes what a caller of transform_device receives, so that two builds can be compared output for output:
      transformed_sizes.npy  float64 [nch]     every chunk's transformed size (d_sizes)
      sample_chunk_ids.npy   float64 [k]       a fixed, seeded sample of chunk indices (k from the budget and the slot size)
      sample_chunks.npy      float32 [k, w]    those chunks' transformed bytes (the slot past SLOT_HEAD), zero past the chunk's end
    The sample depends only on the shape arguments, never on what the path computed."""
    from tsgpu import binding
    os.makedirs(path, exist_ok=True)
    sizes = d_sizes.cpu().numpy().astype(np.int64)
    width = stride - binding.SLOT_HEAD
    cols = min(width, (DUMP_BUDGET - 16 * nch) // 4)
    k = max(1, min(nch, (DUMP_BUDGET - 16 * nch) // (4 * cols)))
    ids = np.sort(np.random.default_rng(20240).choice(nch, k, replace=False))
    chunks = np.zeros((k, cols), dtype=np.float32)
    for j, i in enumerate(ids):
        n = min(int(sizes[i]), cols)
        a = int(i) * stride + binding.SLOT_HEAD
        chunks[j, :n] = d_slots[a:a + n].cpu().numpy()
    np.save(os.path.join(path, "transformed_sizes.npy"), sizes.astype(np.float64))
    np.save(os.path.join(path, "sample_chunk_ids.npy"), ids.astype(np.float64))
    np.save(os.path.join(path, "sample_chunks.npy"), chunks)


def main_tsgpu(args):
    import torch
    import torch.distributed as dist
    import tsgpu
    from tsgpu import corpus

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl tsgpu needs a GPU: libtsgpu has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    bind_to_gpu_numa_node(torch, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    flags = flags_of(args.workload, args.zstd_mode)
    seg, cs = args.segment_mib * MIB, args.chunk_mib * MIB
    nch = seg // cs
    key, aad, ivs = corpus.fixed_key_material(nch)

    src_np = make_segment(args, rank)
    h_src = torch.empty(seg, dtype=torch.uint8).pin_memory()
    h_src.numpy()[:] = src_np
    d_src = h_src.to(dev, non_blocking=True)
    ctx = tsgpu.Context(max_chunk_bytes=cs, max_batch=nch, devices=[local])
    stride = ctx.slot_stride(flags, cs)
    d_slots = torch.empty(nch * stride, dtype=torch.uint8, device=dev)
    d_sizes = torch.zeros(nch, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step_device():
        ctx.transform_device(flags, d_src.data_ptr(), seg, cs, key, aad, ivs, d_slots.data_ptr(), stride,
                             d_sizes.data_ptr(), stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: device-resident, CUDA events on the launching stream
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                    # started before warm-up so nvidia-smi is already streaming
    for _ in range(args.warmup):
        step_device()
    barrier()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.begin()
    e0.record()
    for _ in range(args.steps):
        step_device()
    e1.record()
    barrier()
    sampler.end()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_transform_outputs(args.dump_outputs, d_slots, d_sizes, stride, nch)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * seg * args.steps / GIB / (ms_max / 1000.0)
    sizes = d_sizes.cpu().numpy().astype(np.int64)
    transformed_total = int(sizes.sum())

    # ---- verify what was timed (after the timed region): the slots the LAST timed step left behind go back through the
    # device detransform and must equal the segment byte for byte; a seeded sample of chunks is also decoded by the CPU
    # chain (libzstd + OpenSSL) in the cpu_baseline leg below
    verified = None
    if not args.no_verify:
        d_back = torch.zeros(seg, dtype=torch.uint8, device=dev)
        d_osz = torch.zeros(nch, dtype=torch.int32, device=dev)
        d_stat = torch.full((nch,), 9, dtype=torch.int32, device=dev)
        ctx.detransform_device(flags, d_slots.data_ptr(), stride, d_sizes.data_ptr(), nch, cs, key, aad, d_back.data_ptr(),
                               d_osz.data_ptr(), d_stat.data_ptr(), stream)
        torch.cuda.synchronize()
        ok = bool(torch.equal(d_back, d_src)) and int(d_stat.abs().sum().item()) == 0 and \
            d_osz.cpu().numpy().tolist() == [min(cs, seg - i * cs) for i in range(nch)]
        verified = {"device_roundtrip_whole_segment": ok}
        del d_back
        if not ok:
            raise SystemExit("bench.py: the timed step's output does not detransform back to the input")

    # ---- roofline: per-kernel CUDA-event timing, separate steps so the events do not perturb `value`
    roofline, kernels = None, None
    ctx.profile_enable(True)
    for _ in range(max(1, min(args.steps, 3))):
        step_device()
    rep = ctx.profile_report()
    ctx.profile_enable(False)
    psteps = max(1, min(args.steps, 3))
    if rep:
        kernels = {k: {"launches": v["launches"] // psteps, "ms": v["ms"] / psteps} for k, v in rep.items()}
        top = max(rep.items(), key=lambda kv: kv[1]["ms"])
        name, ms_k = top[0], top[1]["ms"] / top[1]["launches"]
        # algorithmic bytes of the dominant kernel per launch (DESIGN.md "Kernels"): the bytes it must read + write
        if name.startswith("zstd_compress") or name.startswith("zstd_enc"):
            frame_total = transformed_total - (28 * nch if flags & 2 else 0)
            alg = seg + frame_total
        elif name.startswith("gcm_main"):
            payload = transformed_total - 28 * nch
            alg = 2 * payload
        else:
            alg = seg + transformed_total
        peak, how = load_peaks()
        achieved = alg / 1e9 / (ms_k / 1000.0)
        traffic, traffic_capture = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                # keys are kernel names ("zstd_enc_blocks"); values {"bytes": per-launch DRAM read + write, "capture": file}
                tj = json.load(open(tpath))
                ent = tj.get(name, tj.get(name.rsplit("_", 1)[0]))
                here = "%s|%s|%s|%d" % (args.workload, args.zstd_mode, args.corpus, args.segment_mib)
                if isinstance(ent, dict) and ent.get("bench_config") == here:      # only a capture taken at THIS configuration
                    traffic, traffic_capture = ent.get("bytes"), ent.get("capture")
            except Exception:
                traffic = None
        roofline = {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "peak_source": how,
                    "traffic_source": None if traffic is None else
                    "STATIC: dram__bytes_read.sum + dram__bytes_write.sum of one launch at this configuration from the ncu --set "
                    "full capture %s (not measured in this run)" % traffic_capture,
                    "algorithmic_bytes_per_launch": alg, "kernel_ms": ms_k,
                    "note": "integer/LDS-bound kernels: see DESIGN.md for the ALU/shared-memory ceilings"}

    # ---- e2e: the host-buffer C-ABI call (pinned src/dst), H2D + kernels + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        ectx = tsgpu.Context(max_chunk_bytes=cs, max_batch=4, devices=[local])
        cap = int(ectx.lib.tsgpu_transform_bound(flags, seg, cs)) + 64
        h_dst = torch.empty(cap, dtype=torch.uint8).pin_memory()
        dst_np = h_dst.numpy()
        out_sizes = None
        for _ in range(max(1, args.warmup)):
            _, out_sizes = ectx.transform(flags, src_np if False else h_src.numpy(), cs, key, aad, ivs, dst=dst_np)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            _, out_sizes = ectx.transform(flags, h_src.numpy(), cs, key, aad, ivs, dst=dst_np)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt_max = float(tt.item())
        e2e = {"value": world * seg * args.steps / GIB / dt_max, "unit": "GiB/s",
               "h2d_bytes_per_step": seg, "d2h_bytes_per_step": int(sum(out_sizes)),
               "timer": "host wall clock around tsgpu_transform (it synchronises internally), max over ranks"}
        ectx.close()

    # ---- cpu_baseline: the oracle on this box's host cores, rank 0, bounded sample
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import oracle as ora
        probe = CpuArm(args, flags, src_np, 1, 2 * cs)
        probe.step()
        pb, pdt = probe.step()
        probe_v = pb / GIB / pdt
        target_s = 10.0
        sample = args.cpu_sample_mib * MIB if args.cpu_sample_mib else int(min(seg, max(4 * cs, probe_v * GIB * target_s)))
        sample = (sample // cs) * cs
        arm = CpuArm(args, flags, src_np, 1, sample)
        nbytes, dt = arm.step()
        v = nbytes / GIB / dt
        # Kafka's copier pool: T = min(nproc, 10) segments in flight (README.md:221 of the reference), one chain per thread
        T = min(os.cpu_count() or 1, 10)
        pool = None
        if T > 1:
            parm = CpuArm(args, flags, src_np, T, min(seg, 8 * T * cs), min_chunks_per_worker=4)
            parm.step()
            parm.cpu_seconds = 0.0
            pb2, pdt2 = parm.step()
            pool = {"value": pb2 / GIB / pdt2, "unit": "GiB/s", "cores": parm.cores,
                    "effective_cores": round(parm.cpu_seconds / pdt2, 1) if pdt2 > 0 else None,
                    "sample": "T = min(nproc, 10) = %d worker processes, %d MiB per step" % (parm.cores, pb2 // MIB)}
            parm.close()
        if verified is not None:
            # the checker: a seeded sample of the last timed step's chunks decoded by libzstd + OpenSSL
            rng = np.random.default_rng(11)
            pick = sorted(set([0, nch - 1] + rng.choice(nch, min(nch, 6), replace=False).tolist()))
            slots_np = d_slots.cpu().numpy().reshape(nch, stride)
            sz_now = d_sizes.cpu().numpy().astype(np.int64)      # the slots as they are now (profiling steps re-ran the path)
            good = True
            for i in pick:
                t = slots_np[i, 4:4 + int(sz_now[i])]
                back, osz = ora.detransform_chunks(flags & 3, t, [int(sz_now[i])], cs, key, aad)
                good = good and np.array_equal(back, src_np[i * cs:(i + 1) * cs])
            verified["cpu_chain_decodes_sample_chunks"] = {"chunks": pick, "ok": bool(good)}
            if not good:
                raise SystemExit("bench.py: libzstd + OpenSSL do not decode the timed step's output")
        cpu = {"value": v, "unit": "GiB/s", "cores": 1, "kind": "port", "copier_pool": pool,
               "sample": "first %d MiB of the same segment, chunk-sequential on 1 thread (the reference's per-segment "
                         "pipeline is single-threaded); libzstd %s level 3 + OpenSSL EVP AES-256-GCM standing in for "
                         "zstd-jni 1.5.6-9 + SunJCE; %.1f s" % (nbytes // MIB, ora.lib().ora_zstd_version().decode(), dt)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": config_of(args, world),
            "compression_ratio": seg / max(1, transformed_total - (28 * nch if flags & 2 else 0)) if flags & 1 else None,
            "transformed_bytes_per_segment": transformed_total,
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "cpu_baseline": cpu, "kernels_ms_per_step": kernels, "verified": verified,
        }
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        sys.exit(main_reference(a))
    if a.workload == "none":
        sys.exit(main_plumbing(a))
    sys.exit(main_fetch(a) if a.direction == "fetch" else main_tsgpu(a))
