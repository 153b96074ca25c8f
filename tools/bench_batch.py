#!/usr/bin/env python
"""Config 5 of BASELINE.json: a batch of independent 4-64 KB payloads (PNG-IDAT / HTTP-body shaped), one zlib stream each,
through zultra_cuda_memory_compress_batch.  Host buffers in, host buffers out; the argument arrays and the output buffers are
built ONCE (a C caller keeps its buffers too) and only the C call is timed.  Reports MB/s for pageable and page-locked
caller memory, per-stage ms, and checks EVERY stream against the unmodified reference: the sha256 prefixes of
tests/golden/config_golden.npz when the batch is the configuration's own 100 000 payloads, else oracle/_ref run here.

--dict-bytes K: the same payloads also go through zultra_cuda_memory_compress_batch_dict with a K-byte preset dictionary
sampled from the text pool of the payloads (synth.batch_dictionary), and the result gets a "dictionary" section with the
same figures plus the device time of the input assembly kernel.  Every dictionary stream is checked against the plain-C
oracle (tests/oracle_py.py) on all host cores before anything is printed."""
import argparse
import ctypes as C
import hashlib
import json
import multiprocessing
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402


class BatchArgs:
    """ctypes argument block over ONE input slab and ONE output slab (pageable numpy or page-locked torch memory)."""

    def __init__(self, L, payloads, flags, pinned, extra=0):
        n = len(payloads)
        sizes = np.array([len(p) for p in payloads], dtype=np.int64)
        caps = np.array([L.zultra_memory_bound(int(s), flags, 0) + extra for s in sizes], dtype=np.int64)
        ioff = np.concatenate(([0], np.cumsum(sizes)))
        ooff = np.concatenate(([0], np.cumsum(caps)))
        if pinned:
            import torch
            self._ti = torch.empty(int(ioff[-1]), dtype=torch.uint8).pin_memory()
            self._to = torch.empty(int(ooff[-1]), dtype=torch.uint8).pin_memory()
            self.inp, self.out = self._ti.numpy(), self._to.numpy()
        else:
            self.inp, self.out = np.empty(int(ioff[-1]), dtype=np.uint8), np.zeros(int(ooff[-1]), dtype=np.uint8)
        for p, o in zip(payloads, ioff[:-1]):
            self.inp[o:o + len(p)] = p
        ib, ob = self.inp.ctypes.data, self.out.ctypes.data
        self.n, self.sizes, self.ooff = n, sizes, ooff
        self.in_ptrs = (C.c_void_p * n)(*[ib + int(o) for o in ioff[:-1]])
        self.in_sizes = (C.c_size_t * n)(*[int(s) for s in sizes])
        self.out_ptrs = (C.c_void_p * n)(*[ob + int(o) for o in ooff[:-1]])
        self.out_caps = (C.c_size_t * n)(*[int(c) for c in caps])
        self.out_sizes = (C.c_size_t * n)()

    def stream(self, i):
        return self.out[int(self.ooff[i]):int(self.ooff[i]) + int(self.out_sizes[i])].tobytes()


def load_payloads(count, lo, hi):
    """synth.batch, kept in the temporary directory so that alternating runs of two builds in one session generate it once."""
    from zultra_b200 import synth
    path = os.path.join(tempfile.gettempdir(), "zultra_bench_batch_%d_%d_%d.npz" % (count, lo, hi))
    if os.path.exists(path):
        f = np.load(path)
        return np.split(f["data"], np.cumsum(f["sizes"])[:-1])
    payloads = synth.batch(count, lo=lo, hi=hi)
    tmp = path + ".%d.tmp.npz" % os.getpid()
    np.savez(tmp, data=np.concatenate(payloads), sizes=np.array([len(p) for p in payloads], dtype=np.int64))
    os.replace(tmp, path)
    return payloads


_CHECK = {}


def _oracle_mismatches(lo_hi):
    """Streams in [lo, hi) whose dictionary output differs from the oracle (a forked worker: inherits _CHECK)."""
    import oracle_py
    a, payloads, dic = _CHECK["args"], _CHECK["payloads"], _CHECK["dic"]
    return [i for i in range(*lo_hi) if a.stream(i) != oracle_py.compress(payloads[i], 1, dic=dic)]


def run_mode(L, ctx, payloads, steps, dic, res, verify):
    """Time the call for pageable and pinned caller memory; stage ms, counters and the check from the pageable run."""
    total = sum(len(p) for p in payloads)
    extra = 4 if dic is not None else 0      # zlib DICTID, not counted by zultra_memory_bound
    dptr, dlen = (dic.ctypes.data, len(dic)) if dic is not None else (None, 0)

    def call(a):
        if dic is None:
            return L.zultra_cuda_memory_compress_batch(ctx.p, a.in_ptrs, a.in_sizes, a.out_ptrs, a.out_caps, a.out_sizes, a.n, 1, 0)
        return L.zultra_cuda_memory_compress_batch_dict(ctx.p, a.in_ptrs, a.in_sizes, a.out_ptrs, a.out_caps, a.out_sizes, a.n, 1, 0, dptr, dlen)
    for mode in ("pageable", "pinned"):
        a = BatchArgs(L, payloads, 1, mode == "pinned", extra)
        ts = []
        for it in range(1 + steps):      # first call: the context sizes its device buffers
            t0 = time.perf_counter()
            rc = call(a)
            assert rc == 0, rc
            if it:
                ts.append(time.perf_counter() - t0)
        res["MB/s_host_to_host_" + mode] = round(total / min(ts) / 1e6, 1)
        res["ms_" + mode] = round(1e3 * min(ts), 1)
        if mode == "pageable":
            res["stages_ms"] = {k: round(v, 1) for k, v in ctx.timings().items()}
            res["counters"] = ctx.counters()
            res["verified"] = verify(a)
            res["compressed_bytes"] = int(sum(int(x) for x in a.out_sizes))
            if dic is not None:      # device time of the assembly kernel, from one more call with per-kernel events on
                L.zultra_cuda_profile(1)
                L.zultra_cuda_profile_collect(None, None, None, 0)
                assert call(a) == 0
                names, ms, cnt = C.create_string_buffer(32 * 256), (C.c_float * 256)(), (C.c_int * 256)()
                k = L.zultra_cuda_profile_collect(names, ms, cnt, 256)
                L.zultra_cuda_profile(0)
                rows = {names.raw[32 * i:32 * i + 32].split(b"\0")[0].decode(): (float(ms[i]), int(cnt[i])) for i in range(k)}
                t, c = rows.get("batch_assemble", (0.0, 0))
                res["batch_assemble_ms"] = round(t, 2)
                res["batch_assemble_launches"] = c
        del a


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--count", type=int, default=10000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--lo", type=int, default=4096, help="smallest payload, bytes")
    ap.add_argument("--hi", type=int, default=65536, help="largest payload, bytes")
    ap.add_argument("--dict-bytes", type=int, default=0, help="also compress the payloads against a preset dictionary of this size")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import zultra_b200 as z
    from zultra_b200 import synth
    L = z.load()
    t0 = time.time()
    payloads = load_payloads(args.count, args.lo, args.hi)
    total = sum(len(p) for p in payloads)
    gen_s = time.time() - t0
    ctx = z.CudaCtx()
    res = {"workload": "batch (config 5)", "payloads": args.count, "bytes": total, "format": "zlib", "generate_s": round(gen_s, 1)}
    if (args.lo, args.hi) != (4096, 65536):
        res["payload_bytes"] = [args.lo, args.hi]

    def verify_plain(a):
        """every stream against the reference"""
        gpath = os.path.join(ROOT, "tests", "golden", "config_golden.npz")
        g = np.load(gpath) if os.path.exists(gpath) else None
        if args.count == 100000 and (args.lo, args.hi) == (4096, 65536) and g is not None and "batch100k/out_group" in g:
            # the golden keeps, per group of 1000 payloads, the sha256 over (length, 8-byte sha256 prefix) of every stream
            want = g["batch100k/out_group"]
            for lo in range(0, a.n, 1000):
                rec = b"".join(len(s).to_bytes(4, "little") + hashlib.sha256(s).digest()[:8] for s in (a.stream(i) for i in range(lo, min(a.n, lo + 1000))))
                assert hashlib.sha256(rec).digest() == want[lo // 1000].tobytes(), "a stream in %d..%d differs from the reference" % (lo, lo + 999)
            return "all %d streams == unmodified reference (tests/golden/config_golden.npz)" % a.n
        import refharness
        k = min(a.n, 500)
        if os.path.exists(refharness.REF_SO):
            ref = refharness.Ref()
            for i in range(k):
                assert a.stream(i) == ref.compress(payloads[i], flags=1), i
            return "first %d streams == oracle/_ref in this run" % k
        return None

    run_mode(L, ctx, payloads, args.steps, None, res, verify_plain)
    if args.dict_bytes > 0:
        import oracle_py
        dic = synth.batch_dictionary(args.dict_bytes)
        d = {"dict_bytes": args.dict_bytes}

        def verify_dict(a):
            """every stream against the plain-C oracle with the same dictionary, on all host cores (processes: the oracle keeps
            state in globals)"""
            t0 = time.time()
            oracle_py.lib()
            _CHECK.update(args=a, payloads=payloads, dic=dic)
            nproc = os.cpu_count() or 1
            with multiprocessing.get_context("fork").Pool(nproc) as pool:
                bad = sum(pool.map(_oracle_mismatches, [(i, min(a.n, i + 256)) for i in range(0, a.n, 256)]), [])
            _CHECK.clear()
            assert not bad, "dictionary streams differ from the oracle: %s" % bad[:10]
            return "all %d streams == plain-C oracle with the dictionary (%d processes, %.0f s)" % (a.n, nproc, time.time() - t0)
        run_mode(L, ctx, payloads, args.steps, dic, d, verify_dict)
        d["ratio_gain"] = round(res["compressed_bytes"] / d["compressed_bytes"], 4)
        res["dictionary"] = d
    print(json.dumps(res))
    if args.out:
        with open(args.out, "a") as f:
            f.write(json.dumps(res) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
