"""CPU-only tests: the checkers against the golden vectors, the host-emulated pipeline logic against the reference's
outputs, and the C-ABI surface of the built library."""
import ctypes as C
import hashlib
import os
import re
import zlib

import numpy as np
import pytest

import cases
import refharness
from zultra_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "golden_v1.npz"))


def _gold_ok(key, data):
    g = GOLD[key].tobytes()
    return hashlib.sha256(data).digest() == g[:32] and len(data) == int.from_bytes(g[32:], "little")


def test_reference_build_reproduces_golden(ref):
    """The golden file is what oracle/_ref produces (guards against a stale fixture)."""
    c = cases.small_cases()
    for name in ("js48k", "moz300k", "random64k", "abc"):
        for flags, fmt in ((0, "deflate"), (1, "zlib"), (2, "gzip")):
            assert _gold_ok("%s/%s" % (name, fmt), ref.compress(c[name], flags=flags))


@pytest.mark.parametrize("name", list(cases.small_cases().keys()))
def test_emulated_pipeline_vs_golden(emu, name):
    """Same per-task code the GPU runs, executed in a host loop (tests/emu): deflate stream equals the golden vector."""
    data = cases.small_cases()[name]
    out, bits, d = emu.compress(data, dump=True)
    assert _gold_ok("%s/deflate" % name, out)
    assert zlib.decompress(out, -15) == data.tobytes()
    assert d["crc"] == zlib.crc32(data.tobytes())
    assert (d["sub"][:, 7] >> 8).max() == 0   # the reference's undefined length-limit corner (huffencoder.c:334) never reached


def test_emulated_stages_vs_golden(emu):
    w1 = synth.js48k()[:12000]
    w2 = synth.mozilla(60000, seed=77)
    for tag, win, hist in (("stage_js12k", w1, 0), ("stage_moz60k_h32k", w2, 32768)):
        for tile in (0, 512, 4096):
            out, bits, d = emu.compress(win[hist:], hist=win[:hist] if hist else None, dump=True, tile=tile, finalize=0)
            assert np.array_equal(d["sa_lcp"][:len(win)], GOLD[tag + "/sa_lcp"])
            assert np.array_equal(d["match"][hist * 8:len(win) * 8], GOLD[tag + "/match"])
            assert np.array_equal(d["sub"][:, 2], GOLD[tag + "/split"]) and np.array_equal(d["sub"][:, 3], GOLD[tag + "/dyn"])
            assert np.array_equal(d["ll"], GOLD[tag + "/ll"]) and np.array_equal(d["ol"], GOLD[tag + "/ol"])
            assert np.array_equal(d["sub"][:, 6], GOLD[tag + "/bits"])
            assert np.array_equal(d["best"][hist:len(win)], GOLD[tag + "/best"])


def test_emulated_multi_block_and_phase_carry(emu):
    data = synth.mozilla(200000, seed=9)
    key = "moz200k_s9/deflate/b32768"
    out, bits, _ = emu.compress(data, block=32768)
    assert cases.same_as_ref(key, out)
    # two engine calls with the bit phase carried over, as the stream state machine does
    a, abits, _ = emu.compress(data[:98304], block=32768, finalize=0)
    b, bbits, _ = emu.compress(data[98304:], hist=data[98304 - 32768:98304], block=32768, finalize=1, in_bits=abits & 7)
    joined = bytearray(a[: abits >> 3])
    first = (a[abits >> 3] if abits & 7 else 0) | b[0]
    joined += bytes([first]) + b[1:]
    assert cases.same_as_ref(key, bytes(joined))


def test_c_abi_exports_every_declared_symbol():
    import zultra_b200
    path = zultra_b200.lib_path()
    assert os.path.exists(path), "build the library first (make)"
    L = C.CDLL(path)
    names = set()
    for h in ("libzultra.h", "zultra_cuda.h"):
        txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", h)).read(), flags=re.S)
        names |= set(re.findall(r"\b(zultra_[a-z0-9_]+)\s*\(", txt))
    assert len(names) >= 25
    for n in sorted(names):
        assert hasattr(L, n), n


def test_no_gpu_means_error_not_fallback():
    """Without a CUDA device the API must fail; it must never produce output by other means."""
    import zultra_b200 as z
    L = z.load()
    L.zultra_cuda_device_count.restype = C.c_int
    if L.zultra_cuda_device_count() > 0:
        pytest.skip("a GPU is present")
    assert z.memory_compress(b"some input bytes", 1) is None
    with pytest.raises(RuntimeError):
        z.Stream(1)
    with pytest.raises(RuntimeError):
        z.CudaCtx()


def test_host_framing_matches_zlib():
    import zultra_b200 as z
    L = z.load()
    L.zultra_frame_update_checksum.restype = C.c_uint
    L.zultra_frame_update_checksum.argtypes = [C.c_uint, C.c_void_p, C.c_size_t, C.c_uint]
    d = synth.mozilla(100001, seed=2).tobytes()
    assert L.zultra_frame_update_checksum(1, d, len(d), 1) == zlib.adler32(d)
    assert L.zultra_frame_update_checksum(0, d, len(d), 2) == zlib.crc32(d)
    buf = (C.c_ubyte * 16)()
    assert L.zultra_frame_encode_header(buf, 16, 1, None, 0) == 2 and bytes(buf[:2]) == b"\x78\xda"
    assert L.zultra_frame_encode_header(buf, 16, 2, None, 0) == 10 and bytes(buf[:10]) == b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x02\xff"
    assert L.zultra_frame_encode_header(buf, 16, 1, d, 100) == 6 and bytes(buf[:2]) == b"\x78\xf9"
    assert int.from_bytes(bytes(buf[2:6]), "big") == zlib.adler32(d[:100])


def test_synthetic_generators_are_deterministic():
    assert hashlib.sha256(synth.js48k().tobytes()).hexdigest() == hashlib.sha256(synth.js48k().tobytes()).hexdigest()
    assert len(synth.js48k()) == 48944 and len(synth.enwik(100001)) == 100001 and len(synth.mozilla(123457)) == 123457
    assert len(synth.batch(5)) == 5


# ---------------------------------------------------------------- the plain-C oracle (oracle/zultra_oracle.c) ----------------------------------------------------------------
import oracle_py  # noqa: E402


@pytest.mark.parametrize("name", list(cases.small_cases().keys()))
def test_oracle_vs_golden(name):
    """Pins the oracle: its output equals the reference's golden output for every format."""
    data = cases.small_cases()[name]
    for flags, fmt in ((0, "deflate"), (1, "zlib"), (2, "gzip")):
        assert _gold_ok("%s/%s" % (name, fmt), oracle_py.compress(data, flags))


def test_oracle_stages_vs_golden():
    w1 = synth.js48k()[:12000]
    w2 = synth.mozilla(60000, seed=77)
    for tag, win, hist in (("stage_js12k", w1, 0), ("stage_moz60k_h32k", w2, 32768)):
        assert np.array_equal(oracle_py.sa_lcp(win), GOLD[tag + "/sa_lcp"])
        assert np.array_equal(oracle_py.matches(win, hist), GOLD[tag + "/match"])
    out, d = oracle_py.compress(w1, 0, dump=True)
    tag = "stage_js12k"
    assert np.array_equal(d["end"], GOLD[tag + "/split"]) and np.array_equal(d["dyn"], GOLD[tag + "/dyn"])
    assert np.array_equal(d["ll"], GOLD[tag + "/ll"]) and np.array_equal(d["ol"], GOLD[tag + "/ol"]) and np.array_equal(d["bits"], GOLD[tag + "/bits"])
    assert np.array_equal(d["best"][:len(w1)], GOLD[tag + "/best"])


def test_oracle_multi_block_dictionary_and_errors():
    name, data, block = cases.multi_block_cases()[1]
    assert _gold_ok("%s/gzip" % name, oracle_py.compress(data, 2, block))
    dic = synth.enwik(20000, seed=31)
    body = synth.enwik(90000, seed=32)
    assert _gold_ok("dict/zlib", oracle_py.compress(body, 1, dic=dic))
    assert oracle_py.compress(np.zeros(0, dtype=np.uint8), 1) is None
    big = synth.mix(1500000, seed=4, seg_lo=100000, seg_hi=400000)
    assert cases.same_as_ref("mix1.5M_b256k/deflate/b262144", oracle_py.compress(big, 0, 262144))


@pytest.mark.parametrize("name", ["js48k", "moz300k", "zeros100k", "period7", "lz_a96_p0.99", "lz_a2_p0.9", "rows1000", "utf16", "alpha2"])
def test_emulated_compact_candidate_records_vs_golden(emu, name, monkeypatch):
    """The compact candidate records of the parse kernel (zb_cand_pack / zb_dp_eval, zb_core.h: leave-alone matches first,
    short matches shortest-first, one shared prefix-minimum sweep, choice words resolved through the match list), run chunk
    by chunk in the host build: same deflate stream as the golden vector."""
    monkeypatch.setenv("ZB_EMU_DP_LEAN", "1")
    data = cases.small_cases()[name]
    out, bits, d = emu.compress(data)
    assert _gold_ok("%s/deflate" % name, out)


def test_emulated_compact_candidate_records_multi_block(emu, monkeypatch):
    """Same, over several max-blocks with history, sub-block splits and clamped matches at sub-block ends."""
    monkeypatch.setenv("ZB_EMU_DP_LEAN", "1")
    for name, data, block in cases.multi_block_cases()[1:3]:
        out, bits, _ = emu.compress(data, block=block or (1 << 20))
        assert cases.same_as_ref("%s/deflate/b%d" % (name, block), out), name


@pytest.mark.parametrize("cd,lean", [(64, "0"), (320, "1"), (128, "0")])
def test_emulated_adaptive_warmup_vs_golden(emu, monkeypatch, cd, lean):
    """Adaptive warm-up of the chunked parse (zb_pipeline.h stage_parse, D2): a chunk is verified over, and warmed up above,
    only the costs its own candidates reach (need(c) = max(reach(c), need(c - 1) - CD) for chunks shorter than the 258-position
    horizon).  Host build, chunk lengths below, at and above the horizon, both recurrence forms: same stream as the golden
    vectors, on text, binaries, byte runs and short-period data."""
    monkeypatch.setenv("ZB_EMU_PARSE_CD", str(cd))
    if lean == "1":
        monkeypatch.setenv("ZB_EMU_DP_LEAN", "1")
    for name in ("js48k", "moz300k", "enwik200k", "rows1000") + (("period7",) if cd >= 320 else ()):      # (the host repair loop is slow on short-period data with short chunks)
        data = cases.small_cases()[name]
        out, bits, _ = emu.compress(data)
        assert _gold_ok("%s/deflate" % name, out), (name, cd, lean)
