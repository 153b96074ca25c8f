"""Seeded parity inputs shared by the golden generators, the CPU tests and the GPU tests."""
import hashlib
import os

import numpy as np

from zultra_b200 import synth

REF_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_golden.npz")
FMT = {0: "deflate", 1: "zlib", 2: "gzip"}


def small_cases():
    """name -> uint8 array; every case finishes in well under a second on the reference."""
    rng = np.random.default_rng(7)
    c = {}
    c["js48k"] = synth.js48k()
    c["enwik200k"] = synth.enwik(200000)
    c["moz300k"] = synth.mozilla(300000)
    c["zeros100k"] = np.zeros(100000, dtype=np.uint8)
    c["period7"] = np.tile(np.frombuffer(b"abcdefg", dtype=np.uint8), 20000)
    c["random64k"] = rng.integers(0, 256, size=65536).astype(np.uint8)
    c["alpha2"] = rng.integers(0, 2, size=100000).astype(np.uint8)
    c["alpha3"] = rng.integers(0, 3, size=60000).astype(np.uint8)
    c["one"] = np.array([65], dtype=np.uint8)
    c["abc"] = np.frombuffer(b"abc", dtype=np.uint8).copy()
    c["aaaaa"] = np.frombuffer(b"aaaaa", dtype=np.uint8).copy()
    for a, p in [(1, 0.5), (2, 0.9), (15, 0.5), (96, 0.99), (256, 0.0), (256, 0.995)]:
        c["lz_a%d_p%g" % (a, p)] = synth.lz_selftest(40000, 123 + a, a, p)
    c["rows1000"] = np.tile(rng.integers(0, 256, size=1000).astype(np.uint8), 90)
    c["utf16"] = np.stack([synth.enwik(40000, seed=5), np.zeros(40000, dtype=np.uint8)], axis=1).reshape(-1)
    return c


def multi_block_cases():
    """(name, data, block_size) exercising several max-blocks, history overlap and bit-phase carry."""
    return [
        ("enwik2.5M_b1M", synth.enwik(2500000, seed=21), 0),
        ("moz700k_b32k", synth.mozilla(700000, seed=9), 32768),
        ("moz3.2M_b1M", synth.mozilla(3200000, seed=11), 0),
        ("exact2_b64k", synth.enwik(131072, seed=3), 65536),
        ("mix1.5M_b256k", synth.mix(1500000, seed=4, seg_lo=100000, seg_hi=400000), 262144),
        ("rand+text_b2M", np.concatenate([np.random.default_rng(3).integers(0, 256, size=300000).astype(np.uint8), synth.enwik(400000, seed=8)]), 2097152),
    ]


def mixed(seed):
    """Text, random bytes, binary and a zero run: 2.7 MB with stored, static and dynamic sub-blocks."""
    rng = np.random.default_rng(seed)
    return np.concatenate([synth.enwik(700000, seed=seed), rng.integers(0, 256, size=300000).astype(np.uint8), synth.mozilla(900000, seed=seed + 1),
                           np.zeros(200000, dtype=np.uint8), rng.integers(0, 256, size=150000).astype(np.uint8), synth.enwik(450000, seed=seed + 2)])


def lanes_input():
    rng = np.random.default_rng(5)
    return np.concatenate([synth.enwik(700000, seed=31), rng.integers(0, 256, size=300000).astype(np.uint8), synth.mozilla(900000, seed=32),
                           rng.integers(0, 256, size=150000).astype(np.uint8), synth.enwik(450000, seed=33)])


def runs_and_periodic():
    """Byte runs of every length, short records and long periodic repeats."""
    rng = np.random.default_rng(17)
    parts = []
    for _ in range(60):
        run = int(np.exp(rng.uniform(np.log(16), np.log(200000))))
        parts.append(np.full(run, int(rng.choice([0, 0xFF, 0x41])), dtype=np.uint8))
        parts.append(rng.integers(0, 256, size=int(rng.integers(1, 300))).astype(np.uint8))
    rec = np.zeros((40000, 16), dtype=np.uint8)
    rec[:, 0:4] = (np.arange(40000, dtype=np.uint32) + 77).astype("<u4").view(np.uint8).reshape(-1, 4)
    rec[:, 8] = rng.integers(0, 4, size=40000)
    parts.append(rec.reshape(-1))
    parts.append(np.tile(rng.integers(0, 256, size=300).astype(np.uint8), 1500))
    parts.append(np.tile(np.frombuffer(b"ab", dtype=np.uint8), 150000))
    parts.append(synth.enwik(300000, seed=41))
    parts.append(np.zeros(700000, dtype=np.uint8))
    return np.concatenate(parts)


def one_shot_320_blocks():
    """10 MiB: 320 max-blocks of 32768 bytes, more than one 256-block engine call."""
    rng = np.random.default_rng(11)
    return np.concatenate([synth.enwik(3 << 20, seed=51), rng.integers(0, 256, size=1 << 20).astype(np.uint8), synth.mozilla(6 << 20, seed=52)])


def parse_chunk_input(cd):
    return synth.mix(6 << 20, seed=300 + cd, seg_lo=400000, seg_hi=2 << 20)


PARSE_CHUNKS = [704, 960, 1856, 2048, 64, 128, 200, 320, 512]


def stage_windows():
    """(window, history bytes) of the wider stage comparison."""
    rng = np.random.default_rng(5)
    return [(synth.enwik(400000, seed=41), 32768), (synth.mozilla(500000, seed=42), 32768), (synth.mozilla(200000, seed=43), 1000),
            (np.concatenate([np.zeros(70000, dtype=np.uint8), rng.integers(0, 4, size=50000).astype(np.uint8)]), 0)]


STAGE_FIELDS = ("n", "split", "dyn", "sc", "dc", "ll", "ol", "best", "bits")


def ref_streams():
    """key -> (input, flags, max-block, part) of every reference output the tests compare with beyond golden_v1.npz.
    `input` is a function returning the bytes; part "body" is the stream without its zlib/gzip header and trailer,
    which is what zultra_cuda_compress_blocks returns."""
    s = {}

    def add(name, fn, flags, block=0, part="stream"):
        s["%s/%s/b%d%s" % (name, FMT[flags], block, "/body" if part == "body" else "")] = (fn, flags, block, part)

    add("moz200k_s9", lambda: synth.mozilla(200000, seed=9), 0, 32768)
    for i in (1, 2, 4):
        name, _, block = multi_block_cases()[i]
        add(name, lambda i=i: multi_block_cases()[i][1], 0, block)
    for flags in (0, 2):
        add("mix5M_s100", lambda: synth.mix(5 << 20, seed=100, seg_lo=300000, seg_hi=2 << 20), flags)
    add("runs", runs_and_periodic, 0)
    add("runs", runs_and_periodic, 2, 262144)
    for block in (262144, 131072, 65536):
        for flags in (0, 1, 2):
            add("lanes", lanes_input, flags, block, "body")
    for flags in (0, 1, 2):
        add("oneshot10M", one_shot_320_blocks, flags, 32768)
    for cd in sorted(PARSE_CHUNKS):
        add("parse_chunk_cd%d" % cd, lambda cd=cd: parse_chunk_input(cd), 2, 0, "body")
    add("mix10M_s77", lambda: synth.mix(10 << 20, seed=77, seg_lo=1 << 20, seg_hi=3 << 20), 0)
    for seed, block in ((73, 131072), (74, 65536), (75, 262144)):
        for flags in (0, 2):
            add("mixed%d" % seed, lambda seed=seed: mixed(seed), flags, block, "body")
    for block in (65536, 262144):
        for flags in (0, 1, 2):
            add("mixed91", lambda: mixed(91), flags, block, "body")
    add("mix24M_s123", lambda: synth.mix(24 << 20, seed=123, seg_lo=1 << 20, seg_hi=5 << 20), 2)
    add("moz1.5M_s13", lambda: synth.mozilla(1500000, seed=13), 2)
    return s


def fingerprint(b):
    """sha256 + 8-byte length of a stream, or of an integer array's values."""
    if isinstance(b, np.ndarray):
        b = np.ascontiguousarray(b, dtype=np.int64).tobytes()
    return np.frombuffer(hashlib.sha256(b).digest() + len(b).to_bytes(8, "little"), dtype=np.uint8)


_REF = None


def ref_fp(key):
    """Stored fingerprint of the reference's output `key` (tests/golden/ref_golden.npz, made by make_ref_golden.py)."""
    global _REF
    if _REF is None:
        _REF = np.load(REF_GOLDEN)
    return _REF[key]


def same_as_ref(key, b):
    return np.array_equal(fingerprint(b), ref_fp(key))
