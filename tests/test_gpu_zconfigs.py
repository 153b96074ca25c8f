"""GPU parity AT THE STATED CONFIG SIZES of BASELINE.json (VERDICT r1 "what's weak" 1-2): the CUDA path against
  (1) tests/golden/config_golden.npz - sha256 of the unmodified reference's complete streams for js48k / enwik100m /
      mozilla51m / mix1g and of every one of the 100 000 batch payloads (made by tests/golden/make_config_golden.py
      where the reference compiles), and
  (2) fingerprints of the reference's outputs (tests/golden/ref_golden.npz) for the paths whose code changes with size:
      the 256-block batch boundary of the one-shot call, forced parse chunk lengths, multi-wave tile lists, the batch API.
Bit-exact everywhere (integer / byte work)."""
import hashlib
import os
import zlib

import numpy as np
import pytest

import cases
from zultra_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD_PATH = os.path.join(ROOT, "tests", "golden", "config_golden.npz")
CFG = {"js48k": ("js48k", 48944, 1), "enwik100m": ("enwik", 100_000_000, 0), "mozilla51m": ("mozilla", 51_220_480, 2), "mix1g": ("mix", 1 << 30, 2)}
CHUNK = 4 << 20
BATCH_GROUP = 1000


def batch_record(stream):
    """What the batch golden keeps of one stream: its length (4 bytes, little-endian) and the first 8 bytes of its sha256."""
    return len(stream).to_bytes(4, "little") + hashlib.sha256(stream).digest()[:8]


@pytest.fixture(scope="module")
def z():
    import zultra_b200
    return zultra_b200


@pytest.fixture(scope="module")
def gold():
    if not os.path.exists(GOLD_PATH):
        pytest.skip("tests/golden/config_golden.npz missing")
    return np.load(GOLD_PATH)


def _workload(name):
    """Same /tmp cache as bench.py (the 1 GiB stream takes over a minute to generate)."""
    import bench
    gen, size, flags = CFG[name]
    if name == "js48k":
        return synth.js48k(), flags
    return bench.gen_workload(name), flags


def _check_stream(gold, name, data, out):
    if name + "/out_sha" not in gold:
        pytest.skip("no golden entry for " + name)
    assert hashlib.sha256(data.tobytes()).digest() == gold[name + "/in_sha"].tobytes(), "synthetic input differs from the one the golden vector was made from"
    assert out is not None
    if hashlib.sha256(out).digest() != gold[name + "/out_sha"].tobytes():
        ch = gold[name + "/chunks"]
        bad = [i for i in range(len(ch)) if hashlib.sha256(out[i * CHUNK:(i + 1) * CHUNK]).digest()[:8] != ch[i].tobytes()]
        raise AssertionError("%s: stream differs from the reference: len %d vs %d, first differing 4 MiB piece %s" % (name, len(out), int(gold[name + "/out_len"][0]), bad[:1]))


@pytest.mark.parametrize("name", ["js48k", "enwik100m", "mozilla51m"])
def test_config_full_stream_vs_reference_golden(z, gold, name):
    """C1-C3: the complete stream of the configuration == the reference's (sha256 of the whole output)."""
    data, flags = _workload(name)
    out = z.memory_compress(data, flags)
    _check_stream(gold, name, data, out)


def test_config_mix1g_full_stream_vs_reference_golden(z, gold):
    """C4: 1 GiB through zultra_memory_compress (4 engine calls of 256 blocks, bit phase carried) == the reference."""
    data, flags = _workload("mix1g")
    out = z.memory_compress(data, flags)
    _check_stream(gold, "mix1g", data, out)
    assert out[-4:] == (len(data) & 0xffffffff).to_bytes(4, "little")


def test_config_batch100k_vs_reference_golden(z, gold):
    """C5: all 100 000 payloads through zultra_cuda_memory_compress_batch, every stream == the reference's (length and
    sha256 of every stream, folded per group of 1000 payloads)."""
    if "batch100k/out_group" not in gold:
        pytest.skip("no golden entry for batch100k")
    pay = synth.batch(100000)
    want, win = gold["batch100k/out_group"], gold["batch100k/in_sha8_997"]
    ctx = z.CudaCtx()
    try:
        step = 20000
        for lo in range(0, len(pay), step):
            part = pay[lo:lo + step]
            outs = ctx.memory_compress_batch(part, 1)
            for i, p in enumerate(part):
                k = lo + i
                if k % 997 == 0:
                    assert hashlib.sha256(p.tobytes()).digest()[:8] == win[k // 997].tobytes(), "payload %d differs from the golden generator's" % k
            assert all(o is not None for o in outs)
            for g in range(0, len(part), BATCH_GROUP):
                h = hashlib.sha256(b"".join(batch_record(o) for o in outs[g:g + BATCH_GROUP])).digest()
                assert h == want[(lo + g) // BATCH_GROUP].tobytes(), "a payload in %d..%d differs from the reference" % (lo + g, lo + g + BATCH_GROUP - 1)
    finally:
        ctx.close()


def test_batch_api_vs_compiled_reference(z):
    """600 batch-shaped payloads (PNG-IDAT / HTTP body) through the batch API == the reference, stream by stream."""
    pay = synth.batch(600, seed=4242)
    want = cases.ref_fp("batch600_s4242/zlib")
    got = z.memory_compress_batch(pay, 1)
    assert len(got) == len(want)
    for k, a in enumerate(got):
        assert a is not None and np.array_equal(cases.fingerprint(a), want[k]), k


def test_one_shot_across_256_block_batches_vs_compiled_reference(z):
    """10 MiB at max-block 32768 = 320 blocks: zultra_memory_compress cuts it into two engine calls and carries the pending
    bits of the last byte across (csrc/host/libzultra.c); the joined stream must equal the reference's."""
    data = cases.one_shot_320_blocks()
    assert len(data) // 32768 > 256
    for flags in (0, 1, 2):
        assert cases.same_as_ref("oneshot10M/%s/b32768" % cases.FMT[flags], z.memory_compress(data, flags, 32768)), flags


@pytest.mark.parametrize("cd,name", [(cd, "mix6M") for cd in cases.PARSE_CHUNKS] + [(128, "mixed91"), (512, "mixed91")])
def test_forced_parse_chunk_vs_compiled_reference(z, monkeypatch, cd, name):
    """The parse chunk length is chosen from the batch size (960 at 100 MB, up to 1856 for 256-block batches, 128 for small
    inputs): force the lengths the configurations use on an input the reference finishes in seconds.  The adaptive warm-up
    follows what a chunk's candidates reach (its warm-up and the verified part of its signature); chunks shorter than the
    258-position horizon take the propagated form need(c) = max(reach(c), need(c - 1) - CD).  Two lengths also run over
    64 KiB max-blocks of the mixed stream, whose zero run and random stretches go through the repair chains."""
    monkeypatch.setenv("ZULTRA_CUDA_PARSE_CD", str(cd))
    if name == "mixed91":
        data, block, key = cases.mixed(91), 65536, "mixed91/gzip/b65536/body"
    else:
        data, block, key = cases.parse_chunk_input(cd), 0, "parse_chunk_cd%d/gzip/b0/body" % cd
    c = z.CudaCtx()
    try:
        got, bits, ck = c.compress_blocks(data, block=block, finalize=1, flags=2)
    finally:
        c.close()
    assert cases.same_as_ref(key, got) and ck == zlib.crc32(data.tobytes())


def test_multi_wave_tile_lists_vs_compiled_reference(z, monkeypatch):
    """More than 16384 match-finder tiles in one call (only > 128 MiB inputs reach that with the default tile): forced with
    512-position tiles on 10 MiB."""
    monkeypatch.setenv("ZULTRA_CUDA_TILE", "512")
    data = synth.mix(10 << 20, seed=77, seg_lo=1 << 20, seg_hi=3 << 20)
    c = z.CudaCtx()
    try:
        got, bits, ck = c.compress_blocks(data, finalize=1, flags=0)
        assert c.counters()["r7"] > 16384
    finally:
        c.close()
    assert cases.same_as_ref("mix10M_s77/deflate/b0", got)


def test_stream_api_large_single_call_vs_golden(z, gold):
    """ADVICE r1: one zultra_stream_compress(FINALIZE) call holding the whole 100 MB must be cut into bounded engine calls
    (not one unbounded launch) and still produce the reference's stream."""
    data, flags = _workload("enwik100m")
    s = z.Stream(flags)
    st, out = s.compress(data, z.ZULTRA_FINALIZE, out_chunk=8 << 20)
    s.end()
    assert st == z.ZULTRA_STREAM_END
    _check_stream(gold, "enwik100m", data, out)
