"""Suffix-sort group boundaries: tied groups of up to 32 suffixes (ZB_SA_LOCAL in zb_pipeline.h) are ordered by their
next 8 bytes in place, larger ones and members still tied after those bytes go through the doubling rounds.  The exact
SA|LCP words and the compressed streams are compared with the plain-C oracle on inputs aimed at those boundaries."""
import zlib

import numpy as np
import pytest

import oracle_py
from zultra_b200 import synth

LOCAL = 32
TAG = np.frombuffer(b"\x01\x02\x03\x04\x05\x06\x07", dtype=np.uint8)   # 7 bytes = the initial key of a one-window batch


def _group_window(count, seed, n=40000):
    """Random bytes >= 16 with `count` copies of TAG: the only group tied on its first 7 bytes has `count` members.  Half of
    the copies share their next 12 bytes (still tied after the local key), a few share 3, one ends the window 3 bytes
    after the tag and one ends with the tag itself (suffixes that end inside the compared bytes)."""
    rng = np.random.default_rng(seed)
    w = rng.integers(16, 256, n, dtype=np.uint8)
    common = rng.integers(16, 256, 12, dtype=np.uint8)
    pos = np.sort(rng.choice(np.arange(64, n - 200, 40), count - 2, replace=False))
    for k, p in enumerate(pos):
        w[p:p + 7] = TAG
        if k % 2 == 0:
            w[p + 7:p + 19] = common
        elif k % 5 == 1:
            w[p + 7:p + 10] = common[:3]
    w[n - 10:n - 3] = TAG
    w = np.concatenate([w, TAG])
    return w


def _padding_window(seed, n=30000):
    """Zero bytes: a suffix that ends short of the 7-byte key, or inside the next 8 bytes, ties with longer ones followed by
    zeros and sorts before them.  The bytes 1 and 2 occur only in the 15 placed copies of (1, 2, zeros...)."""
    rng = np.random.default_rng(seed)
    w = rng.choice(np.array([0, 0, 0, 3, 4, 5], dtype=np.uint8), n)
    for k, p in enumerate(range(100, n - 100, 2003)):
        tail = (0,) * 20 if k % 3 == 0 else (0,) * 9 + (3,) if k % 3 == 1 else (0,) * 7 + (4,)
        w[p:p + 2 + len(tail)] = (1, 2) + tail
    w[-5:] = (1, 2, 0, 0, 0)
    return w


def _windows():
    yield "group32", _group_window(LOCAL, 1)
    yield "group33", _group_window(LOCAL + 1, 2)
    yield "group31", _group_window(LOCAL - 1, 3)
    yield "padding", _padding_window(4)
    yield "one_byte", np.full(70000, 97, dtype=np.uint8)
    yield "period5", np.tile(np.frombuffer(b"abcab", dtype=np.uint8), 14000)
    yield "period3_noise", np.where(np.arange(60000) % 4099 == 0, 120, np.tile(np.frombuffer(b"xyz", dtype=np.uint8), 20000)).astype(np.uint8)
    yield "text", synth.js48k()[:40000]


CASES = list(_windows())


@pytest.mark.parametrize("name,win", CASES, ids=[c[0] for c in CASES])
def test_emulated_stream_vs_oracle(emu, name, win):
    """The host build of the same per-suffix code: deflate stream equals the oracle's, and so does the suffix array where
    no two suffixes agree on 258 bytes (compression leaves the order of those open)."""
    out, bits, d = emu.compress(win, dump=True)
    assert out == oracle_py.compress(win, 0), name
    if name.startswith(("group", "padding")):
        assert np.array_equal(d["sa_lcp"][:len(win)], oracle_py.sa_lcp(win)), name
    assert zlib.decompress(out, -15) == win.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("name,win", CASES, ids=[c[0] for c in CASES])
def test_exact_sa_lcp_vs_oracle(ctx, name, win):
    assert np.array_equal(ctx.window_sa_lcp(win), oracle_py.sa_lcp(win)), name


@pytest.mark.gpu
@pytest.mark.parametrize("name,win", CASES, ids=[c[0] for c in CASES])
def test_default_stream_vs_oracle(name, win):
    import zultra_b200 as z
    for flags in (0, 1):
        out = z.memory_compress(win, flags)
        assert out == oracle_py.compress(win, flags), (name, flags)


@pytest.mark.gpu
def test_many_window_batch_vs_oracle(ctx):
    """3000 payloads: 12 window bits leave 6 bytes of initial key, and many tiny windows of one repeated byte."""
    rng = np.random.default_rng(11)
    src = synth.js48k()
    payloads = []
    for k in range(3000):
        n = int(rng.integers(1, 300))
        if k % 3 == 0:
            payloads.append(np.full(n, 65 + k % 7, dtype=np.uint8))
        else:
            o = int(rng.integers(0, len(src) - n))
            payloads.append(np.ascontiguousarray(src[o:o + n]))
    outs = ctx.memory_compress_batch(payloads, 1)
    for p, o in zip(payloads, outs):
        assert o == oracle_py.compress(p, 1)
