"""GPU parity tests: the CUDA path, called through the C-ABI / libzultra API, against
(1) the committed golden vectors produced by the reference, (2) fingerprints of the reference's outputs on larger
inputs (tests/golden/ref_golden.npz), (3) size-independent properties (inflate round trip, checksums) at larger sizes.
Bit-exact everywhere: this path is integer/byte work."""
import hashlib
import os
import subprocess
import zlib

import numpy as np
import pytest

import cases
from zultra_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "golden_v1.npz"))


def _gold(key, data):
    g = GOLD[key].tobytes()
    assert hashlib.sha256(data).digest() == g[:32] and len(data) == int.from_bytes(g[32:], "little"), key


def _inflate(b, flags):
    return zlib.decompress(b, -15 if flags == 0 else (15 if flags == 1 else 31))


@pytest.fixture(scope="module")
def z():
    import zultra_b200
    return zultra_b200


def test_library_loaded_is_native(z):
    L = z.load()
    assert os.path.realpath(L._name) == os.path.realpath(z.lib_path())
    ctx = z.CudaCtx()
    ctx.close()


def test_stage_sa_lcp_and_matches_vs_golden(ctx):
    w1 = synth.js48k()[:12000]
    w2 = synth.mozilla(60000, seed=77)
    for tag, win, hist in (("stage_js12k", w1, 0), ("stage_moz60k_h32k", w2, 32768)):
        assert np.array_equal(ctx.window_sa_lcp(win), GOLD[tag + "/sa_lcp"]), tag
        for tile in (0, 512, 4096):
            assert np.array_equal(ctx.window_matches(win, hist, tile=tile), GOLD[tag + "/match"]), (tag, tile)
        st = ctx.block_stages(win, hist)
        assert np.array_equal(st["info"][:, 1], GOLD[tag + "/split"])
        assert np.array_equal(st["info"][:, 2], GOLD[tag + "/dyn"])
        assert np.array_equal(st["ll"], GOLD[tag + "/ll"]) and np.array_equal(st["ol"], GOLD[tag + "/ol"])
        assert np.array_equal(st["info"][:, 5], GOLD[tag + "/bits"])
        assert np.array_equal(st["best"][hist:], GOLD[tag + "/best"])


@pytest.mark.parametrize("name", list(cases.small_cases().keys()))
def test_small_cases_all_formats_vs_golden(z, name):
    data = cases.small_cases()[name]
    for flags, fmt in ((0, "deflate"), (1, "zlib"), (2, "gzip")):
        out = z.memory_compress(data, flags)
        assert out is not None
        _gold("%s/%s" % (name, fmt), out)
        assert _inflate(out, flags) == data.tobytes()


@pytest.mark.parametrize("idx", range(len(cases.multi_block_cases())))
def test_multi_block_vs_golden(z, idx):
    name, data, block = cases.multi_block_cases()[idx]
    out = z.memory_compress(data, 2, block)
    _gold("%s/gzip" % name, out)
    assert _inflate(out, 2) == data.tobytes()


def test_stages_vs_compiled_reference(ctx):
    """Wider stage diff against the reference's stage dumps: SA|LCP words, match lists, splits, static/dynamic decision
    and costs, code lengths, parse, body bits."""
    for i, (win, hist) in enumerate(cases.stage_windows()):
        a = ctx.block_stages(win, hist)
        got = dict(n=np.array([a["n"]]), split=a["info"][:, 1], dyn=a["info"][:, 2], sc=a["info"][:, 3], dc=a["info"][:, 4], ll=a["ll"], ol=a["ol"],
                   best=a["best"][hist:], bits=a["info"][:, 5], sa_lcp=ctx.window_sa_lcp(win), match=ctx.window_matches(win, hist))
        for k, v in got.items():
            assert np.array_equal(cases.fingerprint(v), cases.ref_fp("stage%d/%s" % (i, k))), (i, hist, k)


def test_streaming_api_equals_one_shot(z):
    data = synth.mix(3 * 1048576 + 12345, seed=12, seg_lo=200000, seg_hi=900000)
    one = z.memory_compress(data, 1)
    os.environ["ZULTRA_CUDA_BATCH_BLOCKS"] = "1"
    try:
        s = z.Stream(1)
        got = []
        raw = data.tobytes()
        for o in range(0, len(raw), 100000):
            chunk = raw[o:o + 100000]
            st, b = s.compress(chunk, z.ZULTRA_FINALIZE if o + 100000 >= len(raw) else z.ZULTRA_CONTINUE)
            assert st in (z.ZULTRA_OK, z.ZULTRA_STREAM_END)
            got.append(b)
        assert st == z.ZULTRA_STREAM_END
        assert s.s.total_in == len(raw) and s.s.adler == zlib.adler32(raw)
        st2, _ = s.compress(b"", z.ZULTRA_FINALIZE)
        assert st2 == -5   # ZULTRA_ERROR_COMPRESSION once the stream ended (libzultra.c:204)
        s.end()
    finally:
        del os.environ["ZULTRA_CUDA_BATCH_BLOCKS"]
    assert b"".join(got) == one
    assert zlib.decompress(one) == raw


def test_dictionary_stream_vs_golden(z):
    dic = synth.enwik(20000, seed=31)
    body = synth.enwik(90000, seed=32)
    s = z.Stream(1)
    assert s.set_dictionary(dic) == 0
    st, out = s.compress(body, z.ZULTRA_FINALIZE)
    assert st == z.ZULTRA_STREAM_END
    assert s.set_dictionary(dic) == -5
    s.end()
    _gold("dict/zlib", out)
    d = zlib.decompressobj(zdict=dic.tobytes())
    assert d.decompress(out) == body.tobytes()


def test_error_conventions(z):
    assert z.memory_compress(b"", 1) is None                      # empty input -> (size_t)-1 (libzultra.c:275,617)
    assert z.memory_compress(synth.enwik(50000), 1, out_cap=100) is None   # output too small -> (size_t)-1
    assert z.memory_bound(1000, 2, 0) == 10 + 1 * 6 * 64 + 1000 + 1 + 8


def test_batch_equals_one_shot(z):
    payloads = synth.batch(40, seed=77)
    outs = z.memory_compress_batch(payloads, 1)
    for p, o in zip(payloads, outs):
        assert o is not None and zlib.decompress(o) == p.tobytes()
    for p, o in list(zip(payloads, outs))[:6]:
        assert o == z.memory_compress(p, 1)


def test_large_roundtrip_properties(z):
    """16 MiB: inflate round trip + trailers (size-independent properties; no stored reference output)."""
    data = synth.mix(16 << 20, seed=99, seg_lo=1 << 20, seg_hi=4 << 20)
    out = z.memory_compress(data, 2)
    raw = data.tobytes()
    assert zlib.decompress(out, 31) == raw
    assert out[-8:-4] == zlib.crc32(raw).to_bytes(4, "little") and out[-4:] == (len(raw) & 0xffffffff).to_bytes(4, "little")


def test_large_vs_compiled_reference(z):
    data = synth.mix(5 << 20, seed=100, seg_lo=300000, seg_hi=2 << 20)
    for flags in (0, 2):
        assert cases.same_as_ref("mix5M_s100/%s/b0" % cases.FMT[flags], z.memory_compress(data, flags)), flags


def test_runs_and_periodic_vs_compiled_reference(z):
    """Byte runs and long periodic repeats: the parse does not re-synchronise there, so these inputs go through the
    chain repair (zb_parse_fix_k), including its scan path for blocks made of literals and far leave-alone matches."""
    data = cases.runs_and_periodic()
    for flags, block in ((0, 0), (2, 262144)):
        assert cases.same_as_ref("runs/%s/b%d" % (cases.FMT[flags], block), z.memory_compress(data, flags, block)), flags


def test_compress_blocks_vs_compiled_reference(z):
    """Several max-blocks in one zultra_cuda_compress_blocks call: the stream must equal the reference byte for byte,
    including stored sub-blocks whose size depends on the entering bit phase, a history that is not contiguous with the
    data, an entering bit count and the running checksum."""
    data = cases.lanes_input()
    for block in (262144, 131072, 65536):
        c = z.CudaCtx()
        try:
            for flags in (0, 1, 2):
                got, bits, ck = c.compress_blocks(data, block=block, finalize=1, flags=flags)
                assert cases.same_as_ref("lanes/%s/b%d/body" % (cases.FMT[flags], block), got), (block, flags)
                if flags == 1:
                    assert ck == zlib.adler32(data.tobytes())
                if flags == 2:
                    assert ck == zlib.crc32(data.tobytes())
            # second half of a stream: separate history buffer, 5 pending bits
            cut = 4 * block
            a, abits, ack = c.compress_blocks(data[:cut], block=block, finalize=0, flags=2)
            b, bbits, bck = c.compress_blocks(data[cut:], hist=data[cut - 32768:cut].copy(), block=block, finalize=1, in_bits=abits & 7, flags=2, checksum=ack)
            joined = bytearray(a)
            if abits & 7:
                joined[-1] |= b[0]
                joined += b[1:]
            else:
                joined += b
            assert cases.same_as_ref("lanes/gzip/b%d/body" % block, bytes(joined)) and bck == zlib.crc32(data.tobytes())
        finally:
            c.close()


def test_cli_drop_in(z, tmp_path):
    cli = os.path.join(ROOT, "zultra_b200", "zultra")
    src = tmp_path / "in.bin"
    data = synth.js48k()
    src.write_bytes(data.tobytes())
    for flag, f in (("-zlib", 1), ("-gzip", 2), ("-deflate", 0)):
        dst = tmp_path / ("out" + flag)
        r = subprocess.run([cli, flag, "-c", str(src), str(dst)], capture_output=True)
        assert r.returncode == 0, r.stderr
        _gold("js48k/%s" % flag[1:], dst.read_bytes())
    assert subprocess.run([cli, "-d", str(src), str(tmp_path / "x")]).returncode == 100
    assert subprocess.run([cli, "-gzip", "-D", str(src), str(src), str(tmp_path / "x")], capture_output=True).returncode == 100
    big = tmp_path / "big.bin"
    big.write_bytes(synth.mozilla(1500000, seed=13).tobytes())
    subprocess.check_call([cli, str(big), str(tmp_path / "a.gz")], stdout=subprocess.DEVNULL)
    assert cases.same_as_ref("moz1.5M_s13/gzip/b0", (tmp_path / "a.gz").read_bytes())
    assert subprocess.run([cli, "-quicktest"], capture_output=True).returncode == 0
