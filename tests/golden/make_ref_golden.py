"""Generates tests/golden/ref_golden.npz: fingerprints (sha256 + length) of the reference outputs that the larger parity
tests compare with, so that they need no reference build.

    python tests/golden/make_ref_golden.py

The streams come from the plain-C oracle (oracle/zultra_oracle.c), which restates the reference and is held to it by
golden_v1.npz; the CUDA path equalled the compiled reference on every one of these inputs.  Stored:
  <key of cases.ref_streams()>   the stream (or its body without header and trailer) of that input
  stage<i>/<field>               stage dumps of cases.stage_windows()[i]: sub-block count, split ends, static/dynamic
                                 decision and costs, code lengths, parse, body bits (values as int64); SA|LCP words, match lists
  batch600_s4242/zlib            one fingerprint per payload of synth.batch(600, seed=4242)
"""
import os
import sys
from multiprocessing import Pool

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
import cases  # noqa: E402
import oracle_py  # noqa: E402

HDR = {0: 0, 1: 2, 2: 10}
FTR = {0: 0, 1: 4, 2: 8}


def one_stream(key):
    fn, flags, block, part = cases.ref_streams()[key]
    out = oracle_py.compress(fn(), flags, block)
    if part == "body":
        out = out[HDR[flags]:len(out) - FTR[flags]]
    return {key: cases.fingerprint(out)}


def stages(i):
    win, hist = cases.stage_windows()[i]
    _, d = oracle_py.compress(win[hist:], 0, dic=win[:hist] if hist else None, dump=True)
    got = dict(n=np.array([len(d["end"])]), split=d["end"], dyn=d["dyn"], sc=d["sc"], dc=d["dc"], ll=d["ll"], ol=d["ol"],
               best=d["best"][hist:len(win)], bits=d["bits"], sa_lcp=oracle_py.sa_lcp(win), match=oracle_py.matches(win, hist))
    return {"stage%d/%s" % (i, k): cases.fingerprint(v) for k, v in got.items()}


def batch():
    from zultra_b200 import synth
    return {"batch600_s4242/zlib": np.stack([cases.fingerprint(oracle_py.compress(p, 1)) for p in synth.batch(600, seed=4242)])}


def main():
    oracle_py.lib()      # builds oracle/libzultra_oracle.so once, before the workers load it
    keys = sorted(cases.ref_streams(), key=lambda k: -len(k))
    out = {}
    with Pool(os.cpu_count() or 1) as pool:
        jobs = [pool.apply_async(one_stream, (k,)) for k in keys]
        jobs += [pool.apply_async(stages, (i,)) for i in range(len(cases.stage_windows()))]
        jobs.append(pool.apply_async(batch))
        for j in jobs:
            out.update(j.get())
    np.savez_compressed(os.path.join(HERE, "ref_golden.npz"), **out)
    print("wrote", len(out), "entries")


if __name__ == "__main__":
    main()
