"""GPU: the batch call with a shared preset dictionary (zultra_cuda_memory_compress_batch_dict, CudaCtx.memory_compress_batch(...,
dictionary=...)).  Stream i must be the bytes of zultra_stream_init + zultra_stream_set_dictionary + compress(FINALIZE) of payload i.
Expected outputs come from the plain-C oracle (tests/oracle_py.py), which the `dict/zlib` golden vector pins to the reference."""
import ctypes as C
import multiprocessing
import os
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle_py
from zultra_b200 import synth

pytestmark = pytest.mark.gpu
BAD = C.c_size_t(-1).value
DICT_SIZES = [1, 258, 32767, 32768, 32769, 100000]


@pytest.fixture(scope="module")
def z():
    import zultra_b200
    return zultra_b200


@pytest.fixture(scope="module")
def cx(z):
    c = z.CudaCtx()
    yield c
    c.close()


def _dictionary(size):
    return synth.enwik(size, seed=9000 + size % 997)


def _payloads(dic):
    """1-3 byte payloads, batch-shaped payloads, a copy of the dictionary's tail (matches at distance 32768 for a full tail),
    random bytes (stored blocks) and payloads of 2 and 3 max-blocks of 32 KiB."""
    rng = np.random.default_rng(len(dic))
    text = synth.enwik(110000, seed=77)
    return [b"a", b"\x00\x01", b"xyz"] + synth.batch(6, seed=31, lo=4096, hi=16384) + [
        dic[-32768:].copy(),
        rng.integers(0, 256, size=9000, dtype=np.uint8),
        text[:70000],
        text[5000:105000],
    ]


def _oracle_one(job):
    p, flags, block, dic = job
    return oracle_py.compress(p, flags, block=block, dic=dic)


def _oracle(payloads, flags, block, dic):
    """The oracle keeps state in globals (qsort comparators): one process per worker, never threads."""
    with multiprocessing.get_context("fork").Pool(min(8, os.cpu_count() or 1)) as pool:
        return pool.map(_oracle_one, [(p, flags, block, dic) for p in payloads])


def _call(z, ctx, payloads, flags, block, dic, caps):
    """Direct C call: returns (rc, outputs or None per stream)."""
    L = z.load()
    n = len(payloads)
    arrs = [np.ascontiguousarray(np.frombuffer(p, dtype=np.uint8) if isinstance(p, bytes) else p, dtype=np.uint8) for p in payloads]
    outs = [np.empty(max(c, 1), dtype=np.uint8) for c in caps]
    inp = (C.c_void_p * n)(*[a.ctypes.data for a in arrs]); ins = (C.c_size_t * n)(*[len(a) for a in arrs])
    outp = (C.c_void_p * n)(*[o.ctypes.data for o in outs]); oc = (C.c_size_t * n)(*caps); osz = (C.c_size_t * n)()
    rc = L.zultra_cuda_memory_compress_batch_dict(ctx.p, inp, ins, outp, oc, osz, n, flags, block,
                                                  dic.ctypes.data if dic is not None else None, len(dic) if dic is not None else 0)
    return rc, [None if osz[i] == BAD else outs[i][:osz[i]].tobytes() for i in range(n)]


@pytest.mark.parametrize("dict_size", DICT_SIZES)
@pytest.mark.parametrize("block", [32768, 0])
@pytest.mark.parametrize("flags", [0, 1, 2])
def test_batch_dict_equals_oracle(cx, flags, block, dict_size):
    dic = _dictionary(dict_size)
    payloads = _payloads(dic)
    got = cx.memory_compress_batch(payloads, flags, block, dictionary=dic)
    want = _oracle(payloads, flags, block, dic)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g is not None and g == w, "stream %d (%d bytes)" % (i, len(payloads[i]))


@pytest.mark.parametrize("flags", [0, 1, 2])
def test_batch_dict_equals_streaming_api(z, cx, flags):
    dic = _dictionary(40000)
    payloads = _payloads(dic)[2:8]
    got = cx.memory_compress_batch(payloads, flags, 32768, dictionary=dic)
    for p, g in zip(payloads, got):
        s = z.Stream(flags, 32768)
        assert s.set_dictionary(dic) == 0
        st, out = s.compress(p, z.ZULTRA_FINALIZE)
        s.end()
        assert st == z.ZULTRA_STREAM_END and g == out


def test_batch_dict_round_trip(cx):
    dic = _dictionary(32768)
    payloads = _payloads(dic)
    for p, out in zip(payloads, cx.memory_compress_batch(payloads, 1, 0, dictionary=dic)):
        raw = bytes(p) if isinstance(p, bytes) else p.tobytes()
        assert out[:2] == b"\x78\xf9" and int.from_bytes(out[2:6], "big") == zlib.adler32(dic.tobytes())
        d = zlib.decompressobj(zdict=dic.tobytes())
        assert d.decompress(out) == raw and d.eof
        assert int.from_bytes(out[-4:], "big") == zlib.adler32(raw)      # trailer: the payload only
    for p, out in zip(payloads, cx.memory_compress_batch(payloads, 0, 0, dictionary=dic)):
        d = zlib.decompressobj(-15, zdict=dic.tobytes())
        assert d.decompress(out) == (bytes(p) if isinstance(p, bytes) else p.tobytes())


def test_no_dictionary_is_todays_batch(z, cx):
    payloads = synth.batch(30, seed=123)
    for flags in (0, 1, 2):
        plain = cx.memory_compress_batch(payloads, flags)
        assert cx.memory_compress_batch(payloads, flags, dictionary=b"") == plain
        caps = [z.memory_bound(len(p), flags, 0) for p in payloads]
        rc, got = _call(z, cx, payloads, flags, 0, None, caps)
        assert rc == 0 and got == plain


def test_errors(z, cx):
    dic = _dictionary(32768)
    payloads = [synth.enwik(5000, seed=1), np.zeros(0, dtype=np.uint8), synth.enwik(7000, seed=2)]
    out = cx.memory_compress_batch(payloads, 1, dictionary=dic)
    assert out[1] is None and out[0] is not None and out[2] is not None
    # a cap of exactly the stream's size (DICTID included) is enough; one byte less fails that stream only
    caps = [len(out[0]), 16, len(out[2]) - 1]
    rc, got = _call(z, cx, payloads, 1, 0, dic, caps)
    assert rc == 0 and got[0] == out[0] and got[1] is None and got[2] is None
    # zultra_memory_bound does not count the 4 DICTID bytes: memory_compress_batch adds them to its capacities
    stored = np.random.default_rng(3).integers(0, 256, size=5000, dtype=np.uint8)
    bound = z.memory_bound(len(stored), 1, 0)
    full = cx.memory_compress_batch([stored], 1, dictionary=dic)[0]
    assert full is not None and len(full) <= bound + 4
    rc, got = _call(z, cx, [stored], 1, 0, dic, [len(full) - 4])
    assert rc == 0 and got == [None]
    # argument errors come back before any work
    L = z.load()
    n = 1
    a = np.ascontiguousarray(payloads[0]); o = np.empty(100000, dtype=np.uint8)
    inp = (C.c_void_p * n)(a.ctypes.data); ins = (C.c_size_t * n)(len(a)); outp = (C.c_void_p * n)(o.ctypes.data)
    oc = (C.c_size_t * n)(len(o)); osz = (C.c_size_t * n)(12345)
    assert L.zultra_cuda_memory_compress_batch_dict(cx.p, inp, ins, outp, oc, osz, n, 1, 0, dic.ctypes.data, -1) == -12
    assert L.zultra_cuda_memory_compress_batch_dict(cx.p, inp, ins, outp, oc, osz, n, 1, 0, None, 10) == -12
    assert osz[0] == 12345


def test_sub_batch_split_by_dictionary_history(cx):
    """14 000 payloads of 32 KiB: 459 MB of payload fit one sub-batch (768 MiB of window bytes) without a dictionary, but with
    32 KiB of dictionary history per stream the windows take 918 MB and the call splits after stream 12286."""
    dic = _dictionary(32768)
    payloads = synth.batch(14000, seed=2024, lo=32768, hi=32768)
    outs = cx.memory_compress_batch(payloads, 1, dictionary=dic)
    assert cx.counters()["windows"] < len(payloads)      # the last sub-batch is not the whole call
    zd = dic.tobytes()

    def inflate(i):
        d = zlib.decompressobj(zdict=zd)
        return d.decompress(outs[i]) == payloads[i].tobytes()
    with ThreadPoolExecutor(8) as ex:
        assert all(ex.map(inflate, range(len(payloads))))
    near = list(range(12187, 12387))
    want = _oracle([payloads[i] for i in near], 1, 0, dic)
    for i, w in zip(near, want):
        assert outs[i] == w, "stream %d" % i
