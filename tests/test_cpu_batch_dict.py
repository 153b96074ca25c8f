"""CPU-only: the dictionary batch path of the engine (zultra_cuda_memory_compress_batch_dict) in the host build (tests/emu).
Payloads cross to the device packed behind ONE copy of the dictionary and stage_assemble lays out [dictionary tail | payload]
per stream; every raw deflate bitstream must equal the plain-C oracle compressing that payload with the same dictionary."""
import ctypes as C
import os
import subprocess
import zlib

import numpy as np
import pytest

import oracle_py
import refharness
from zultra_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(refharness.EMU_SO):
        subprocess.check_call(["make", "-C", ROOT, "emu"])
    L = C.CDLL(refharness.EMU_SO)
    L.emu_batch_dict.restype = C.c_long
    L.emu_batch_dict.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.c_uint,
                                 C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p]
    return L


def batch_dict(L, payloads, dic, block=32768, flags=0):
    """-> [(raw deflate bytes, checksum)] per payload, from one engine call of the host build."""
    arrs = [np.ascontiguousarray(p, dtype=np.uint8) for p in payloads]
    d = np.ascontiguousarray(dic if dic is not None else np.zeros(0), dtype=np.uint8)
    n = len(arrs)
    ptrs = (C.c_void_p * n)(*[a.ctypes.data for a in arrs]); sizes = (C.c_size_t * n)(*[len(a) for a in arrs])
    cap = sum(len(a) + len(a) // 4 + 4096 for a in arrs)
    out = np.zeros(cap, dtype=np.uint8)
    off = (C.c_size_t * n)(); bits = (C.c_ulonglong * n)(); cks = (C.c_uint * n)()
    rc = L.emu_batch_dict(n, ptrs, sizes, d.ctypes.data if len(d) else None, len(d), block, flags, out.ctypes.data, cap, off, bits, cks)
    assert rc >= 0, rc
    return [(out[off[i]:off[i] + (bits[i] + 7) // 8].tobytes(), cks[i]) for i in range(n)]


def _dictionary(size):
    return synth.enwik(size, seed=4100 + size)


def _payloads(dic):
    text = synth.enwik(120000, seed=4242)
    tail = dic[-32768:]
    return [
        text[:1],                                   # one byte
        text[1000:6000],                            # an HTTP-body shaped text
        synth.batch(2, seed=7, lo=3000, hi=6000)[0],  # a PNG-IDAT shaped payload
        tail[: min(len(tail), 2000)].copy(),        # a copy of the dictionary's tail: matches at the longest distances
        text[20000:60000],                          # two 32 KiB max-blocks: the second one's history is the payload's own
    ]


@pytest.mark.parametrize("dict_size", [1, 300, 32768, 40000])
def test_batch_dict_matches_oracle(lib, dict_size):
    dic = _dictionary(dict_size)
    payloads = _payloads(dic)
    got = batch_dict(lib, payloads, dic, block=32768)
    for i, (p, (raw, _)) in enumerate(zip(payloads, got)):
        assert raw == oracle_py.compress(p, 0, block=32768, dic=dic), "stream %d" % i
        d = zlib.decompressobj(-15, zdict=dic.tobytes()[-32768:])
        assert d.decompress(raw) == p.tobytes(), "stream %d" % i


def test_batch_dict_tiny_streams_share_assembly_vectors(lib):
    """Streams of 2-4 assembled bytes: many streams meet inside one 16-byte vector of the assembly pass."""
    dic = _dictionary(1)
    rng = np.random.default_rng(5)
    payloads = [rng.integers(0, 256, size=int(rng.integers(1, 4)), dtype=np.uint8) for _ in range(60)]
    got = batch_dict(lib, payloads, dic)
    for i, (p, (raw, _)) in enumerate(zip(payloads, got)):
        assert raw == oracle_py.compress(p, 0, block=32768, dic=dic), "stream %d" % i


@pytest.mark.parametrize("flags", [1, 2])
def test_batch_dict_checksum_covers_the_payload_only(lib, flags):
    dic = _dictionary(32768)
    payloads = _payloads(dic)
    got = batch_dict(lib, payloads, dic, flags=flags)
    for p, (_, ck) in zip(payloads, got):
        want = zlib.adler32(p.tobytes()) if flags == 1 else zlib.crc32(p.tobytes())
        assert ck == want


def test_batch_without_dictionary_matches_oracle(lib):
    payloads = _payloads(_dictionary(300))
    got = batch_dict(lib, payloads, None)
    for p, (raw, _) in zip(payloads, got):
        assert raw == oracle_py.compress(p, 0, block=32768)
