"""Cutting a window's suffix list into its units of 32768 main + 32768 look-back positions (unit_dist_k in zb_prims.cu).  A
unit's list carries, for every member, the minimum LCP since the unit's previous member, which may lie in an earlier 32-entry
block, more than 128 blocks back, or in an earlier 4096-rank segment.  The match lists and the compressed streams of windows
aimed at those cases are compared with the plain-C oracle."""
import ctypes as C

import numpy as np
import pytest

import oracle_py
from zultra_b200 import synth

UNIT = 32768


def _runs(rng, n):
    """Runs of 'a' (258-byte LCPs inside them) between short stretches of bytes 1..60 (LCP 0 at the run ends)."""
    parts, k = [], 0
    while k < n:
        r = int(rng.integers(500, 1500))
        s = int(rng.integers(50, 200))
        parts += [np.full(r, 97, np.uint8), rng.integers(1, 61, s, dtype=np.uint8)]
        k += r + s
    return np.concatenate(parts)[:n]


def _mixed_window(seed, tail):
    """Two units of bytes 200..255, which sort after everything else: their units have no member in most segments, and the
    unit that straddles them and the text after them has a gap of thousands of ranks.  Then two units of text, two of byte
    runs and a last unit of `tail` positions."""
    rng = np.random.default_rng(seed)
    text = np.resize(synth.js48k(), 2 * UNIT)
    return np.concatenate([rng.integers(200, 256, 2 * UNIT, dtype=np.uint8), text, _runs(rng, 2 * UNIT), text[:tail]])


def _oracle_matches(win, hist):
    """oracle_py.matches with the pointers passed whole: arrays this large are mapped above 4 GB."""
    out = np.zeros(((len(win) - hist) * 8, 2), dtype=np.uint16)
    oracle_py.lib().zo_window_matches(C.c_void_p(win.ctypes.data), hist, len(win), C.c_void_p(out.ctypes.data))
    return out


# text_h32k is a full-size window of 32 units: consecutive members of a unit are about 16 ranks apart, often more than a block.
CASES = [("mixed_h0", _mixed_window(1, 5000), 0), ("mixed_h32k", _mixed_window(2, 700), UNIT), ("text_h32k", synth.enwik(33 * UNIT, seed=3), UNIT)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,win,hist", CASES, ids=[c[0] for c in CASES])
def test_window_matches_vs_oracle(ctx, name, win, hist):
    want = _oracle_matches(win, hist)
    for tile in (0, 4096):
        assert np.array_equal(ctx.window_matches(win, hist, tile=tile), want), (name, tile)


@pytest.mark.gpu
@pytest.mark.parametrize("name,win,hist", CASES, ids=[c[0] for c in CASES])
def test_stream_vs_oracle(name, win, hist):
    import zultra_b200 as z
    assert z.memory_compress(win, 0) == oracle_py.compress(win, 0), name


@pytest.mark.gpu
def test_one_unit_windows_batch_vs_oracle(ctx):
    """Payloads of one unit each, up to 5 segments long, among tiny ones."""
    rng = np.random.default_rng(5)
    src = synth.js48k()
    payloads = []
    for k in range(200):
        n = int(rng.integers(1, 20000)) if k % 4 else int(rng.integers(1, 64))
        o = int(rng.integers(0, len(src) - n))
        payloads.append(np.ascontiguousarray(src[o:o + n]) if k % 5 else _runs(rng, n))
    outs = ctx.memory_compress_batch(payloads, 1)
    for p, o in zip(payloads, outs):
        assert o == oracle_py.compress(p, 1)
