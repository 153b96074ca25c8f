"""GPU tests of the multi-GPU path (SURVEY 8(e), VERDICT r1 J3/J5): round-robin chunks, per-chunk phase maps, bit-offset
stitch.  The single-device tests drive the chunk C-ABI with two contexts on one GPU standing in for two ranks; the
multi-device tests (skipped on a 1-GPU box) go through the library's own in-process path - zultra_cuda_ctx_set_devices /
ZULTRA_CUDA_DEVICES behind zultra_cuda_compress_blocks, zultra_memory_compress, the streaming API and the CLI.
Everything is compared byte for byte with the reference's outputs (fingerprints in tests/golden/ref_golden.npz)."""
import os
import subprocess
import zlib

import numpy as np
import pytest

import cases
from zultra_b200 import shard, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def z():
    import zultra_b200
    return zultra_b200


def _ngpu(z):
    return z.load().zultra_cuda_device_count()


@pytest.mark.parametrize("world,block,g", [(2, 131072, 2), (3, 65536, 1), (4, 262144, 1)])
def test_chunk_abi_two_contexts_stitch_vs_compiled_reference(z, world, block, g):
    """zultra_cuda_chunks_prepare / _emit / zultra_cuda_stitch_device: `world` contexts on this GPU play the ranks."""
    import torch
    data = cases.mixed(71 + world)
    dev_in = torch.from_numpy(data).cuda()
    plan = shard.plan_chunks(len(data), block, world, g=g)
    ctxs = [z.CudaCtx() for _ in range(world)]
    try:
        for flags in (0, 2):
            maps, cks = [None] * len(plan), [None] * len(plan)
            mine = [[j for j, c in enumerate(plan) if c[2] == r] for r in range(world)]
            for r in range(world):
                chunks = [(plan[j][0] - min(plan[j][0], 32768), min(plan[j][0], 32768), plan[j][1] - plan[j][0], 1 if plan[j][1] >= len(data) else 0) for j in mine[r]]
                m, c = ctxs[r].chunks_prepare(dev_in.data_ptr(), chunks, block=block, flags=flags)
                for i, j in enumerate(mine[r]):
                    maps[j], cks[j] = m[i], c[i]
            offs, nbits, total = shard.compose(maps)
            src, dbit, nb = [], [], []
            for r in range(world):
                ptr, off, bits = ctxs[r].chunks_emit([offs[j] & 7 for j in mine[r]])
                for i, j in enumerate(mine[r]):
                    assert bits[i] - (offs[j] & 7) == nbits[j]
                    src.append(ptr + off[i]); dbit.append(offs[j]); nb.append(nbits[j])
            dst = torch.zeros((total + 7) // 8 + 8, dtype=torch.uint8, device="cuda")
            ctxs[0].stitch_device(dst.data_ptr(), src, dbit, nb)
            got = dst[: (total + 7) // 8].cpu().numpy().tobytes()
            assert cases.same_as_ref("mixed%d/%s/b%d/body" % (71 + world, cases.FMT[flags], block), got), (world, block, flags)
            ck = cks[0]
            for j in range(1, len(plan)):
                ck = z.load().zultra_cuda_checksum_combine(flags, ck, cks[j], plan[j][1] - plan[j][0])
            if flags == 2:
                assert ck == zlib.crc32(data.tobytes())
    finally:
        for c in ctxs:
            c.close()


def test_stitch_device_random_parts(z):
    """The stitch kernel against shard.merge (numpy) on random parts with every phase and tiny sizes."""
    import torch
    rng = np.random.default_rng(3)
    nbits = [int(x) for x in rng.integers(1, 4000, size=40)] + [1, 7, 8, 9, 31, 32, 33, 100000]
    offs, pos = [], int(rng.integers(0, 8))
    start = pos
    for b in nbits:
        offs.append(pos); pos += b
    bufs = []
    for o, b in zip(offs, nbits):
        ph = o & 7
        nby = (ph + b + 7) // 8
        v = rng.integers(0, 256, size=nby).astype(np.uint8)
        v[0] &= (0xff << ph) & 0xff
        tail = (ph + b) & 7
        if tail:
            v[-1] &= (1 << tail) - 1
        bufs.append(v)
    want = shard.merge([b.tobytes() for b in bufs], offs, nbits, pos)
    devs = [torch.from_numpy(np.concatenate([b, np.zeros(8, dtype=np.uint8)])).cuda() for b in bufs]
    dst = torch.zeros((pos + 7) // 8 + 8, dtype=torch.uint8, device="cuda")
    c = z.CudaCtx()
    try:
        c.stitch_device(dst.data_ptr(), [d.data_ptr() for d in devs], offs, nbits)
    finally:
        c.close()
    assert dst[: (pos + 7) // 8].cpu().numpy().tobytes() == want and start < 8


def test_multi_device_compress_blocks_vs_compiled_reference(z):
    """The in-library multi-GPU path on every device count the box has."""
    n = _ngpu(z)
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    data = cases.mixed(91)
    for ndev in sorted({2, min(n, 3), n}):
        for block in (65536, 262144):
            c = z.CudaCtx(0)
            try:
                assert c.set_devices(ndev) == ndev
                for flags in (0, 1, 2):
                    got, bits, ck = c.compress_blocks(data, block=block, finalize=1, flags=flags)
                    assert c.counters()["devices"] == ndev
                    assert cases.same_as_ref("mixed91/%s/b%d/body" % (cases.FMT[flags], block), got), (ndev, block, flags)
                    if flags == 1:
                        assert ck == zlib.adler32(data.tobytes())
                    if flags == 2:
                        assert ck == zlib.crc32(data.tobytes())
                # second half of a stream: separate history buffer, pending bits, running checksum
                cut = 6 * block
                a, abits, ack = c.compress_blocks(data[:cut], block=block, finalize=0, flags=2)
                b, bbits, bck = c.compress_blocks(data[cut:], hist=data[cut - 32768:cut].copy(), block=block, finalize=1, in_bits=abits & 7, flags=2, checksum=ack)
                joined = bytearray(a)
                if abits & 7:
                    joined[-1] |= b[0]
                    joined += b[1:]
                else:
                    joined += b
                assert cases.same_as_ref("mixed91/gzip/b%d/body" % block, bytes(joined)) and bck == zlib.crc32(data.tobytes())
            finally:
                c.close()


def test_multi_device_public_api_and_cli_vs_compiled_reference(z, monkeypatch, tmp_path):
    """ZULTRA_CUDA_DEVICES: zultra_memory_compress, the streaming API and the CLI on all GPUs == the reference."""
    n = _ngpu(z)
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    monkeypatch.setenv("ZULTRA_CUDA_DEVICES", str(n))
    data = synth.mix(24 << 20, seed=123, seg_lo=1 << 20, seg_hi=5 << 20)
    key = "mix24M_s123/gzip/b0"
    assert cases.same_as_ref(key, z.memory_compress(data, 2))
    monkeypatch.setenv("ZULTRA_CUDA_BATCH_BLOCKS", "8")
    s = z.Stream(2)
    raw = data.tobytes()
    got = []
    for o in range(0, len(raw), 3000000):
        st, b = s.compress(raw[o:o + 3000000], z.ZULTRA_FINALIZE if o + 3000000 >= len(raw) else z.ZULTRA_CONTINUE)
        assert st in (z.ZULTRA_OK, z.ZULTRA_STREAM_END)
        got.append(b)
    s.end()
    assert st == z.ZULTRA_STREAM_END and cases.same_as_ref(key, b"".join(got))
    src = tmp_path / "in.bin"
    src.write_bytes(raw)
    cli = os.path.join(ROOT, "zultra_b200", "zultra")
    env = dict(os.environ, ZULTRA_CUDA_TRACE="1")
    r = subprocess.run([cli, str(src), str(tmp_path / "out.gz")], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, env=env, check=True)
    assert cases.same_as_ref(key, (tmp_path / "out.gz").read_bytes())
    assert b"devices %d" % n in r.stderr, r.stderr[-400:]      # the CLI really spread the stream over all GPUs
