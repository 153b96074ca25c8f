#!/usr/bin/env python
"""bench.py - headline metric of BASELINE.json: input MB/s of the zultra compression hot path on N B200s.

One "step" = one pass of the whole pipeline (suffix array + LCP, match lists, block split, optimal parse, Huffman,
bit emission) over the workload.  N=1 workload: configs[1] of BASELINE.json, a synthetic 100 000 000 B
enwik8-shaped XML/wiki text, deflate format, default 1 MiB max-block (96 blocks).
  value      MB/s (10^6 B/s) with the input already resident in HBM (zultra_cuda_compress_blocks_device), timed
             with CUDA events, max over ranks
  e2e        same metric through the public zultra_memory_compress call with pinned HOST buffers, H2D/D2H inside;
             at N > 1 that one call (ZULTRA_CUDA_DEVICES=N, made by rank 0) drives all N GPUs and returns ONE stitched
             host buffer - shard DMA, bit-offset scan and boundary merge are all inside the timed region
  roofline   dominant kernel: algorithmic bytes / its average CUDA-event duration vs the measured HBM copy peak
  match_finder   second half of BASELINE.json's metric: input GB/s of the stages S1-S3 + M1 (suffix array, LCP, match lists)
  strong     the north-star scaling configs at their stated sizes, STRONG scaling: mix1g (1 GiB, config 4) and mozilla51m
             (config 3) split over the N GPUs, with per-rank {compute, all_gather, emit, gather, merge} ms
  cpu_baseline   the reference's own CPU code (oracle/_ref) on a bounded sample, one thread; its output is kept and
             must equal the CUDA path's stream for the same bytes
Parity gate before any number counts: the complete stream of every configuration must equal the unmodified reference's
(sha256 in tests/golden/config_golden.npz, made by tests/golden/make_config_golden.py where the reference compiles).
--impl reference times the reference CPU implementation on the host cores instead (no GPU work).
--dump-outputs DIR writes the stream of the last timed step (see dump_outputs) so that two builds can be compared
output for output; the inputs are generated from fixed seeds, so the same arguments give the same inputs.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "input MB/s (zultra compression hot path, byte-identical to CPU zultra)"   # both arms report this metric
BLOCK = 1 << 20
WORKLOADS = {
    "enwik100m": dict(size=100_000_000, flags=0, fmt="deflate", gen="enwik"),
    "mozilla51m": dict(size=51_220_480, flags=2, fmt="gzip", gen="mozilla"),
    "mix1g": dict(size=1 << 30, flags=2, fmt="gzip", gen="mix"),
}
# algorithmic bytes per unit for the kernels that can dominate (DESIGN.md section 5)
KERNEL_BYTES = {
    "mf_build_walk": ("per block byte: 4 B SA|LCP word in (x1.031 window) + 32 B match list out", lambda n, P: 4.0 * P + 32.0 * n),
    "mf_tile_filter": ("per window position: 4 B word read + 4 B tile word written", lambda n, P: 8.0 * P),
    "parse_dp": ("per block byte and pass: 32 B match list + 1 B text read, 4 B choice written; 4 passes", lambda n, P: 4 * 37.0 * n),
    "rs_scatter": ("per sorted element and pass: 12 B key+index read, 12 B written", lambda n, P: 24.0 * P),
    "rs_hist": ("per sorted element and pass: 8 B key read", lambda n, P: 8.0 * P),
    "lcp_pack": ("per window position: 4 B SA read, 1 B text, 4 B word written", lambda n, P: 9.0 * P),
}


def gen_workload(name, size=None, seg=0):
    """Segment `seg` of a workload (segment 0 is the configuration itself; further segments, other seeds, make up the
    N x larger stream of a weak-scaling run).  Cached under /tmp; written atomically since ranks may race."""
    from zultra_b200 import synth
    w = WORKLOADS[name]
    n = size or w["size"]
    cache = os.path.join("/tmp", "zb_%s_%d_s%d.npy" % (name, n, seg))
    if os.path.exists(cache):
        return np.load(cache, mmap_mode="r" if n >= (256 << 20) else None)
    fn = getattr(synth, w["gen"])
    d = fn(n) if seg == 0 else fn(n, seed=0x5A170100 + 1009 * seg)
    try:
        tmp = cache + ".%d.tmp.npy" % os.getpid()
        np.save(tmp, d)
        os.replace(tmp, cache)
    except OSError:
        pass
    return d


def stream_range(name, size, lo, hi):
    """Bytes [lo, hi) of the stream made of consecutive segments of `size` bytes each."""
    parts = []
    for sg in range(lo // size, (max(lo, hi - 1)) // size + 1):
        d = gen_workload(name, size, sg)
        a, b = max(lo, sg * size) - sg * size, min(hi, (sg + 1) * size) - sg * size
        if b > a:
            parts.append(d[a:b])
    return np.concatenate(parts) if len(parts) != 1 else np.ascontiguousarray(parts[0])


def ncu_traffic(kernel):
    """dram bytes per launch of `kernel` from the committed ncu --set full capture of this workload (profiles/), or None."""
    try:
        j = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        return j.get(kernel)
    except (OSError, ValueError):
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe).  The sampler is started
    before the warm-up (nvidia-smi needs a few hundred ms to deliver its first row); every row is stamped on arrival and only
    rows that fall inside [mark_begin, mark_end] are reported (all rows under load if the region was shorter than a period)."""

    def __init__(self, index=0):
        self.rows, self.p, self.index, self.t0, self.t1 = [], None, index, None, None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index),
                                       "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                                       "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)   # let the row sampled at the end of the region arrive
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.p.kill()
        inside = [r for (t, r) in self.rows if self.t0 is not None and self.t0 <= t <= (self.t1 or t) + 0.06]
        rows = inside if inside else [r for (t, r) in self.rows if self.t0 is None or t >= self.t0 - 1.0]
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(rows)}


def cpu_reference_timing(data, flags, threads, slice_bytes, keep=False):
    """Reference CPU code (oracle/_ref): `threads` workers, each compressing its own slice of the workload with the stock
    zultra_memory_compress.  Returns (MB/s aggregate, seconds, description[, streams])."""
    import refharness
    if not os.path.exists(refharness.REF_SO):
        return (None, None, "oracle/_ref missing") + ((None,) if keep else ())
    lib = C.CDLL(refharness.REF_SO)
    lib.zultra_memory_compress.restype = C.c_size_t
    lib.zultra_memory_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_uint, C.c_uint]
    lib.zultra_memory_bound.restype = C.c_size_t
    lib.zultra_memory_bound.argtypes = [C.c_size_t, C.c_uint, C.c_uint]
    slices = [np.ascontiguousarray(data[i * slice_bytes:(i + 1) * slice_bytes]) for i in range(threads)]
    slices = [s for s in slices if len(s)]
    outs = [np.empty(lib.zultra_memory_bound(len(s), flags, 0), dtype=np.uint8) for s in slices]
    sizes = [0] * len(slices)

    def work(i):
        sizes[i] = lib.zultra_memory_compress(slices[i].ctypes.data, len(slices[i]), outs[i].ctypes.data, len(outs[i]), flags, 0)

    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(len(slices))]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    total = sum(len(s) for s in slices)
    r = (total / dt / 1e6, dt, "%d thread(s) x %d B slices of the workload, stock zultra_memory_compress" % (len(slices), slice_bytes))
    return r + ([o[:k].tobytes() for o, k in zip(outs, sizes)],) if keep else r


def config_of(name, n, world, weak):
    """The `config` object of the JSON line - the same for both arms (the reference arm times the reference on this config)."""
    w = WORKLOADS[name]
    return {"workload": name if not weak else "%s x %d (one stream of %d segments of the configuration's shape)" % (name, world, world),
            "bytes": int(n), "format": w["fmt"], "max_block": BLOCK, "blocks": int((n + BLOCK - 1) // BLOCK),
            "parallelism": "1 GPU, whole stream per call" if world == 1 else "round-robin chunks of max-blocks over %d GPUs (each with its 32 KiB history), NCCL only for the 8-phase maps and the shard bitstreams" % world,
            "l2": "256 MiB flush write between iterations"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    name = args.workload
    w = WORKLOADS[name]
    data = gen_workload(name, args.size)
    world = max(1, world)
    weak = world > 1 and name == "enwik100m"
    cores = max(1, min(os.cpu_count() or 1, 64))
    slice_bytes = 2 << 20
    vals = []
    for it in range(args.warmup + args.steps):
        v, dt, sample = cpu_reference_timing(data[(it * cores * slice_bytes) % max(1, len(data) - cores * slice_bytes):], w["flags"], cores, slice_bytes)
        if v is None:
            print(json.dumps({"impl": "reference", "unavailable": sample}))
            return
        if it >= args.warmup:
            vals.append((v, dt))
    v = sum(x[0] for x in vals) / len(vals)
    ms = 1000.0 * sum(x[1] for x in vals) / len(vals)
    n = int(len(data)) * (world if weak else 1)
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": round(v, 3), "unit": "MB/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                      "config": config_of(name, n, world, weak),
                      "cpu_baseline": {"value": round(v, 3), "unit": "MB/s", "cores": cores, "kind": "reference",
                                       "sample": sample + "; every step = each host thread compresses one 2 MiB slice of segment 0 of this config"},
                      "e2e": {"value": round(v, 3), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def golden():
    try:
        return np.load(os.path.join(ROOT, "tests", "golden", "config_golden.npz"))
    except OSError:
        return None


def verify_stream(name, weak, data, stream, flags):
    """Parity gate.  Returns the `verified` string; raises if the stream is not the reference's."""
    import hashlib
    import zlib
    g = golden()
    if not weak and g is not None and name + "/out_sha" in g and hashlib.sha256(data).digest() == g[name + "/in_sha"].tobytes():
        assert hashlib.sha256(stream).digest() == g[name + "/out_sha"].tobytes(), "%s: stream differs from the reference's (tests/golden/config_golden.npz)" % name
        return "sha256(complete stream) == unmodified reference's stream for this config (tests/golden/config_golden.npz)"
    assert zlib.decompress(stream, {0: -15, 1: 15, 2: 31}[flags]) == bytes(data), "output does not inflate to the input"
    # no golden vector for this stream: its leading max-blocks must equal the reference run on the same leading bytes here
    import refharness
    if os.path.exists(refharness.REF_SO):
        k = 3 << 20
        want = refharness.Ref().compress(np.frombuffer(bytes(data[:k]), dtype=np.uint8), flags=flags)
        body = len(want) - {0: 0, 1: 4, 2: 8}[flags]
        same = 0
        lim = min(body, len(stream))
        a, b = np.frombuffer(want[:lim], dtype=np.uint8), np.frombuffer(stream[:lim], dtype=np.uint8)
        diff = np.nonzero(a != b)[0]
        same = int(diff[0]) if len(diff) else lim
        assert same >= body - (1 << 20) - 4096, "leading max-blocks differ from oracle/_ref at byte %d" % same   # all but the last block (BFINAL, flush)
        return "inflate(stream) == input; first 2 max-blocks == oracle/_ref run on the same bytes in this run"
    return "inflate(stream) == input"


DUMP_SAMPLE = 4 << 20     # stream bytes kept by --dump-outputs: 16 MB of float32 values + 32 MB of float64 positions


def dump_outputs(out_dir, stream, checksum):
    """The complete framed stream a caller of the timed path receives, as .npy files under out_dir:
      stream.npy         its bytes as float32 - all of them, or DUMP_SAMPLE bytes at positions drawn with a fixed seed
      stream_index.npy   the positions of those bytes in the stream (float64)
      stream_sha256.npy  the 32 bytes of sha256 of the whole stream (float32), so that every byte is compared
      checksum.npy       [stream length in bytes, adler32 / crc32 of the input the path returned] (float64)"""
    import hashlib
    os.makedirs(out_dir, exist_ok=True)
    b = np.frombuffer(stream, dtype=np.uint8)
    if len(b) <= DUMP_SAMPLE:
        idx = np.arange(len(b))
    else:
        idx = np.sort(np.random.default_rng(0x5A17D).choice(len(b), DUMP_SAMPLE, replace=False))
    np.save(os.path.join(out_dir, "stream.npy"), b[idx].astype(np.float32))
    np.save(os.path.join(out_dir, "stream_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "stream_sha256.npy"), np.frombuffer(hashlib.sha256(stream).digest(), dtype=np.uint8).astype(np.float32))
    np.save(os.path.join(out_dir, "checksum.npy"), np.array([len(b), checksum], dtype=np.float64))


def run_workload(args, name, weak, steps, warmup, env, headline):
    """One workload on all ranks.  Returns the result dict on rank 0 (None elsewhere)."""
    torch, dist, z, L, rank, world, local = env["torch"], env["dist"], env["z"], env["L"], env["rank"], env["world"], env["local"]
    from bench_shard import ShardRunner
    w = WORKLOADS[name]
    seg_size = (args.size if headline and args.size else None) or w["size"]
    nseg = world if weak else 1
    n = seg_size * nseg
    # segments are generated once per box (cached under /tmp), spread over the ranks
    for sg in range(nseg):
        if sg % world == rank:
            gen_workload(name, seg_size, sg)
    if dist is not None:
        dist.barrier()
    ctx = z.CudaCtx(local)
    runner = ShardRunner(z, ctx, lambda lo, hi: stream_range(name, seg_size, lo, hi), n, w["flags"], BLOCK, rank, world, dist, torch)
    data = stream_range(name, seg_size, 0, n) if rank == 0 else None
    flush = env["flush"]

    def step(profile):
        flush.fill_(1)   # L2 flush between iterations
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        L.zultra_cuda_profile(1 if profile else 0)
        ms = runner.step_device()
        L.zultra_cuda_profile(0)
        return ms

    for _ in range(warmup):
        step(False)
    times, l0 = [], L.zultra_cuda_launch_count()
    bsum = {}
    if headline and env.get("sampler"):
        env["sampler"].mark_begin()
    for _ in range(steps):
        times.append(step(headline and not args.no_profile))
        for k, v in runner.breakdown.items():
            bsum[k] = bsum.get(k, 0.0) + v / steps
    if headline and env.get("sampler"):
        env["sampler"].mark_end()
    launches = L.zultra_cuda_launch_count() - l0
    verified, stream_sha = None, None
    if rank == 0:      # the stream of the last timed step
        import hashlib
        stream = runner.final_stream()
        verified = verify_stream(name, weak, data, stream, w["flags"])
        stream_sha = hashlib.sha256(stream).hexdigest()
        if headline and args.dump_outputs:
            dump_outputs(args.dump_outputs, stream, runner.checksum)
    t = torch.tensor([sum(times)], dtype=torch.float64, device="cuda")
    lt = torch.tensor([float(launches)], dtype=torch.float64, device="cuda")
    per_rank = None
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        rows = [None] * world
        dist.all_gather_object(rows, {k: round(v, 3) for k, v in bsum.items()})
        per_rank = rows
    ms_per_step = float(t.item()) / steps
    stages = ctx.timings()
    counters = ctx.counters()
    # ---- end to end through the public API: pinned (and pageable) host buffers, ONE call for the whole stream on all GPUs ----
    e2e = None
    if rank == 0:
        os.environ["ZULTRA_CUDA_DEVICES"] = str(world)
        os.environ["ZULTRA_CUDA_DEVICE"] = str(local)
        hin = torch.from_numpy(np.ascontiguousarray(data)).pin_memory()
        cap = L.zultra_memory_bound(n, w["flags"], BLOCK)
        hout = torch.empty(cap, dtype=torch.uint8).pin_memory()
        ts, r = [], 0
        for it in range(2 + max(1, steps)):      # 2 untimed: the pooled contexts of the public API allocate their device buffers on first use
            t0 = time.perf_counter()
            r = L.zultra_memory_compress(C.c_void_p(hin.data_ptr()), n, C.c_void_p(hout.data_ptr()), cap, w["flags"], BLOCK)
            assert r != C.c_size_t(-1).value, "zultra_memory_compress failed"
            if it >= 2:
                ts.append(time.perf_counter() - t0)
        assert hout[:r].numpy().tobytes() == stream, "public-API stream differs from the device-resident path's"
        e2e_ms = 1e3 * sum(ts) / len(ts)
        e2e = {"value": round(n / (e2e_ms / 1e3) / 1e6, 2), "unit": "MB/s", "h2d_bytes_per_step": int(n + 32768 * max(0, len(runner.plan) - 1)), "d2h_bytes_per_step": int(r),
               "ms_per_step": round(e2e_ms, 3), "call": "zultra_memory_compress, pinned host in -> one stitched host buffer out, ZULTRA_CUDA_DEVICES=%d" % world}
        if headline or world == 1:      # a drop-in caller has pageable memory: report that too
            pin = np.array(data, copy=True); pout = np.empty(cap, dtype=np.uint8)
            tp = []
            for it in range(2):
                t0 = time.perf_counter()
                r2 = L.zultra_memory_compress(pin.ctypes.data, n, pout.ctypes.data, cap, w["flags"], BLOCK)
                tp.append(time.perf_counter() - t0)
            assert r2 == r
            e2e["pageable_value"] = round(n / min(tp) / 1e6, 2)
        del hin, hout
        L.zultra_cuda_release_cached()
        os.environ.pop("ZULTRA_CUDA_DEVICES", None)
    if dist is not None:      # the other ranks wait on the host (an NCCL barrier would spin on their GPUs while rank 0 uses them)
        store = dist.distributed_c10d._get_default_store()
        key = "zb_e2e_done_%s_%d" % (name, env.setdefault("seq", 0))
        env["seq"] += 1
        if rank == 0:
            store.set(key, "1")
        else:
            store.wait([key])
        dist.barrier()
    out = None
    if rank == 0:
        comp = [r.get("compute", 0.0) for r in per_rank] if per_rank else [bsum.get("compute", 0.0)]
        out = {"value": round(n / (ms_per_step / 1e3) / 1e6, 2), "unit": "MB/s", "ms_per_step": round(ms_per_step, 3), "steps": steps, "warmup": warmup,
               "scaling": "weak" if (weak or world == 1) else "strong", "config": config_of(name, n, world, weak), "e2e": e2e,
               "gpu_launches": int(lt.item()), "per_rank_ms": per_rank if per_rank else [{k: round(v, 3) for k, v in bsum.items()}],
               "rank_compute_ms_max": round(max(comp), 3), "rank_compute_ms_min": round(min(comp), 3),
               "limiting_step": None, "stages_ms": {k: round(v, 3) for k, v in stages.items()}, "counters": counters,
               "compressed_bytes": runner.last_out_bytes, "stream_sha256": stream_sha, "verified": verified}
        if per_rank:
            tot = {k: max(r.get(k, 0.0) for r in per_rank) for k in ("compute", "all_gather", "emit", "gather", "merge")}
            k = max(tot, key=tot.get)
            out["limiting_step"] = "%s (%.1f ms on the slowest rank; all_gather also absorbs the wait for the slowest rank's compute)" % (k, tot[k])
        out["_n"], out["_stages"], out["_runner_plan"] = n, stages, (1 if runner.single else len(runner.plan))
    ctx.close()
    del runner
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="enwik100m")
    ap.add_argument("--size", type=int, default=None)
    ap.add_argument("--scaling", default="auto", choices=["auto", "weak", "strong"], help="N > 1: weak = one stream of N x the configuration (default for enwik100m), strong = the configuration split N ways")
    ap.add_argument("--strong", default="mozilla51m,mix1g", help="comma list of configurations also timed with strong scaling (reported under `strong`); empty = none")
    ap.add_argument("--strong-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true", help="no per-kernel CUDA events in the timed steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the stream of the last timed step of the headline workload to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.strong_steps < 1:
        ap.error("--steps and --strong-steps must be at least 1, --warmup at least 0")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import zultra_b200 as z
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    name = args.workload
    w = WORKLOADS[name]
    # weak scaling (default for the headline workload): the job is ONE stream of N segments of the configuration's size;
    # strong: the configuration itself split N ways
    weak = world > 1 and (args.scaling == "weak" or (args.scaling == "auto" and name == "enwik100m"))
    L = z.load()
    env = dict(torch=torch, dist=dist, z=z, L=L, rank=rank, world=world, local=local, flush=torch.empty(256 << 20, dtype=torch.uint8, device="cuda"))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        env["sampler"] = sampler
    head = run_workload(args, name, weak, args.steps, args.warmup, env, True)
    clocks = sampler.stop() if rank == 0 else None
    names = C.create_string_buffer(32 * 256); kms = (C.c_float * 256)(); kcnt = (C.c_int * 256)()
    nk = L.zultra_cuda_profile_collect(names, kms, kcnt, 256)
    ktab = sorted([(names.raw[32 * i:32 * i + 32].split(b"\0")[0].decode(), kms[i], kcnt[i]) for i in range(nk)], key=lambda r: -r[1])
    strong = {}
    for sname in [x for x in args.strong.split(",") if x and x != name and x in WORKLOADS]:
        r = run_workload(args, sname, False, args.strong_steps, 1, env, False)
        if r is not None:
            for k in ("_n", "_stages", "_runner_plan"):
                r.pop(k, None)
            strong[sname] = r
    out = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        n = head.pop("_n"); stages = head.pop("_stages"); nchunks = head.pop("_runner_plan")
        n_local = n // world
        P_local = n_local + (n_local // BLOCK) * 32768
        top = next((r for r in ktab if r[0] in KERNEL_BYTES), ktab[0] if ktab else ("none", 0.0, 1))
        desc, fn = KERNEL_BYTES.get(top[0], ("unknown", lambda a, b: 0.0))
        alg_bytes_per_step = fn(n_local, P_local)
        per_launch_ms = top[1] / max(1, top[2])
        launches_per_step = top[2] / args.steps
        achieved = (alg_bytes_per_step / launches_per_step) / (per_launch_ms / 1e3) / 1e9 if per_launch_ms > 0 else 0.0
        mf_ms = stages.get("sa_lcp", 0.0) + stages.get("match", 0.0)
        mf_gbs = n_local / (mf_ms / 1e3) / 1e9 if mf_ms > 0 else 0.0
        out = {"metric": METRIC, "value": head["value"], "unit": "MB/s",
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
               "scaling": head["scaling"], "vs_baseline": None, "dtype": "u8", "data": "synthetic",
               "config": head["config"], "clocks": clocks, "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
               "roofline": {"bound": "hbm", "kernel": top[0], "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 5),
                            "traffic": ncu_traffic(top[0]), "traffic_source": "profiles/ncu_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch, enwik100m at N=1)",
                            "algorithmic_bytes": desc, "kernel_ms_per_step": round(top[1] / args.steps, 3),
                            "kernel_share_of_step": round(top[1] / max(1e-9, sum(r[1] for r in ktab)), 4), "kernel_share_basis": "sum of all kernel durations on rank 0",
                            "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if peaks else "fallback 6.65 TB/s"},
               "match_finder": {"value": round(mf_gbs, 3), "unit": "GB/s", "ms_per_step": round(mf_ms, 3), "stages": "suffix array + LCP (S1-S3) and match lists (M1), rank 0, device-resident",
                                "algorithmic_bytes_per_input_byte": 41.3, "frac": round(41.3 * mf_gbs / peak, 5)},
               "stages_ms": head["stages_ms"],
               "kernels_ms_per_step": {r[0]: round(r[1] / args.steps, 3) for r in ktab[:48]},
               "per_rank_ms": head["per_rank_ms"], "rank_compute_ms_max": head["rank_compute_ms_max"], "rank_compute_ms_min": head["rank_compute_ms_min"],
               "limiting_step": head["limiting_step"], "chunks": nchunks,
               "counters": head["counters"], "compressed_bytes": head["compressed_bytes"], "stream_sha256": head["stream_sha256"], "verified": head["verified"],
               "strong": strong}
        if not args.no_cpu_baseline and world == 1:
            data = gen_workload(name, args.size)
            k = 24 << 20
            v, dt, sample, streams = cpu_reference_timing(data, w["flags"], 1, k, keep=True)
            if v is not None:
                got = z.memory_compress(np.ascontiguousarray(data[:k]), w["flags"], BLOCK)
                assert got == streams[0], "CUDA stream of the first 24 MiB differs from the reference's (oracle/_ref, this run)"
                out["cpu_baseline"] = {"value": round(v, 3), "unit": "MB/s", "cores": 1, "kind": "reference",
                                       "sample": "first 24 MiB of the workload, " + sample + ", %.1f s; its output == the CUDA path's stream for the same bytes" % dt}
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
