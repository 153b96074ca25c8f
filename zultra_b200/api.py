"""ctypes mirror of the libzultra.h API (reference libzultra.h:54-157) and of the CUDA C-ABI (zultra_cuda.h).

Same names and argument meaning as the C API.  Nothing here computes: every call goes into
libzultra_b200.so, which fails if its CUDA device is missing - there is no CPU path to fall back to.
"""
import ctypes as C
import os

import numpy as np

ZULTRA_FLAG_DEFLATE_FRAMING, ZULTRA_FLAG_ZLIB_FRAMING, ZULTRA_FLAG_GZIP_FRAMING = 0, 1, 2
ZULTRA_CONTINUE, ZULTRA_FINALIZE = 0, 1
ZULTRA_OK, ZULTRA_STREAM_END = 0, 1
ZULTRA_ERROR_SRC, ZULTRA_ERROR_DST, ZULTRA_ERROR_DICTIONARY, ZULTRA_ERROR_MEMORY, ZULTRA_ERROR_COMPRESSION = -1, -2, -3, -4, -5

_ALLOC = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_uint, C.c_uint)
_FREE = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p)


class zultra_stream_t(C.Structure):
    """Field order/types of reference libzultra.h:78-93."""
    _fields_ = [("next_in", C.c_void_p), ("avail_in", C.c_size_t), ("total_in", C.c_ulonglong),
                ("next_out", C.c_void_p), ("avail_out", C.c_size_t), ("total_out", C.c_ulonglong),
                ("zalloc", C.c_void_p), ("zfree", C.c_void_p), ("opaque", C.c_void_p),
                ("state", C.c_void_p), ("adler", C.c_uint)]


def lib_path():
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "libzultra_b200.so")


_lib = None


def load():
    """Load the native library; raises if it has not been built (run `make` or __graft_entry__.build())."""
    global _lib
    if _lib is None:
        p = lib_path()
        if not os.path.exists(p):
            raise RuntimeError("zultra_b200: native library %s is missing - build it with `make`; there is no Python/CPU fallback" % p)
        L = C.CDLL(p)
        L.zultra_memory_bound.restype = C.c_size_t
        L.zultra_memory_bound.argtypes = [C.c_size_t, C.c_uint, C.c_uint]
        L.zultra_memory_compress.restype = C.c_size_t
        L.zultra_memory_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_uint, C.c_uint]
        L.zultra_stream_init.argtypes = [C.c_void_p, C.c_uint, C.c_uint]
        L.zultra_stream_set_dictionary.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.zultra_stream_compress.argtypes = [C.c_void_p, C.c_int]
        L.zultra_stream_end.argtypes = [C.c_void_p]
        L.zultra_stream_end.restype = None
        L.zultra_cuda_ctx_create.argtypes = [C.c_void_p, C.c_int]
        L.zultra_cuda_ctx_destroy.argtypes = [C.c_void_p]
        L.zultra_cuda_ctx_destroy.restype = None
        L.zultra_cuda_compress_blocks.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_uint, C.c_int, C.c_uint, C.c_uint,
                                                  C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.zultra_cuda_compress_blocks_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_int, C.c_uint, C.c_void_p,
                                                         C.c_void_p, C.c_size_t, C.c_void_p]
        L.zultra_cuda_shard_prepare.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_uint, C.c_int, C.c_uint, C.c_void_p, C.c_void_p]
        L.zultra_cuda_shard_emit.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_size_t, C.c_void_p]
        L.zultra_cuda_checksum_combine.restype = C.c_uint
        L.zultra_cuda_checksum_combine.argtypes = [C.c_uint, C.c_uint, C.c_uint, C.c_ulonglong]
        L.zultra_cuda_memory_compress_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_uint]
        L.zultra_cuda_memory_compress_batch_dict.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_uint,
                                                             C.c_void_p, C.c_int]
        L.zultra_cuda_window_sa_lcp.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.zultra_cuda_window_matches.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint]
        L.zultra_cuda_block_stages.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.zultra_cuda_checksum_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_void_p]
        L.zultra_cuda_ctx_set_devices.argtypes = [C.c_void_p, C.c_int]
        L.zultra_cuda_chunks_prepare.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p]
        L.zultra_cuda_chunks_emit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.zultra_cuda_stitch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.zultra_cuda_profile.argtypes = [C.c_int]
        L.zultra_cuda_launch_count.restype = C.c_longlong
        L.zultra_cuda_profile_collect.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.zultra_cuda_last_timings.argtypes = [C.c_void_p, C.c_void_p]
        L.zultra_cuda_last_counters.argtypes = [C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _u8(a):
    return np.ascontiguousarray(np.frombuffer(a, dtype=np.uint8) if isinstance(a, (bytes, bytearray, memoryview)) else a, dtype=np.uint8)


def memory_bound(n, flags=0, block=0):
    return load().zultra_memory_bound(n, flags, block)


def memory_compress(data, flags=ZULTRA_FLAG_DEFLATE_FRAMING, block=0, out_cap=None):
    """zultra_memory_compress (libzultra.c:601): returns the compressed bytes, or None where the C API returns (size_t)-1."""
    L = load()
    d = _u8(data)
    cap = L.zultra_memory_bound(len(d), flags, block) if out_cap is None else out_cap
    out = np.empty(max(cap, 1), dtype=np.uint8)
    n = L.zultra_memory_compress(d.ctypes.data, len(d), out.ctypes.data, cap, flags, block)
    if n == C.c_size_t(-1).value:
        return None
    return out[:n].tobytes()


class Stream:
    """zultra_stream_t wrapper: init / set_dictionary / compress / end (libzultra.c:82,177,200,521)."""

    def __init__(self, flags=0, block=0):
        self.L = load()
        self.s = zultra_stream_t()
        st = self.L.zultra_stream_init(C.byref(self.s), flags, block)
        if st != ZULTRA_OK:
            raise RuntimeError("zultra_stream_init failed: %d" % st)
        self._keep = []

    def set_dictionary(self, d):
        d = _u8(d)
        self._keep.append(d)
        return self.L.zultra_stream_set_dictionary(C.byref(self.s), d.ctypes.data, len(d))

    def compress(self, data, finalize, out_chunk=16384):
        """Feed `data`; returns (status, bytes produced), calling zultra_stream_compress until avail_out is left over."""
        d = _u8(data)
        self.s.next_in = d.ctypes.data if len(d) else None
        self.s.avail_in = len(d)
        buf = np.empty(out_chunk, dtype=np.uint8)
        chunks = []
        while True:
            self.s.next_out = buf.ctypes.data
            self.s.avail_out = out_chunk
            st = self.L.zultra_stream_compress(C.byref(self.s), finalize)
            if st not in (ZULTRA_OK, ZULTRA_STREAM_END):
                return st, b"".join(chunks)
            chunks.append(buf[: out_chunk - self.s.avail_out].tobytes())
            if self.s.avail_out != 0:
                break
        return st, b"".join(chunks)

    def end(self):
        self.L.zultra_stream_end(C.byref(self.s))


class CudaCtx:
    """zultra_cuda_ctx_t: direct access to the CUDA C-ABI (stage dumps, device-resident compression, timings)."""

    def __init__(self, device=-1):
        self.L = load()
        self.p = C.c_void_p()
        rc = self.L.zultra_cuda_ctx_create(C.byref(self.p), device)
        if rc != 0:
            raise RuntimeError("zultra_cuda_ctx_create failed (%d): no usable CUDA device" % rc)

    def close(self):
        if self.p:
            self.L.zultra_cuda_ctx_destroy(self.p)
            self.p = C.c_void_p()

    def compress_blocks(self, data, hist=None, block=0, finalize=1, in_bits=0, flags=0, checksum=None):
        d = _u8(data)
        h = _u8(hist) if hist is not None and len(hist) else None
        cap = len(d) + len(d) // 8 + 65536
        out = np.empty(cap, dtype=np.uint8)
        bits = C.c_ulonglong(0)
        ck = C.c_uint((1 if flags == 1 else 0) if checksum is None else checksum)
        rc = self.L.zultra_cuda_compress_blocks(self.p, h.ctypes.data if h is not None else None, len(h) if h is not None else 0, d.ctypes.data, len(d),
                                                block, finalize, in_bits, flags, C.byref(ck), out.ctypes.data, cap, C.byref(bits))
        if rc != 0:
            raise RuntimeError("zultra_cuda_compress_blocks failed: %d" % rc)
        return out[: (bits.value + 7) // 8].tobytes(), bits.value, ck.value

    def compress_blocks_device(self, dev_in_ptr, n, dev_out_ptr, out_cap, block=0, finalize=1, flags=0):
        bits = C.c_ulonglong(0)
        ck = C.c_uint(1 if flags == 1 else 0)
        rc = self.L.zultra_cuda_compress_blocks_device(self.p, dev_in_ptr, n, block, finalize, flags, C.byref(ck), dev_out_ptr, out_cap, C.byref(bits))
        if rc != 0:
            raise RuntimeError("zultra_cuda_compress_blocks_device failed: %d" % rc)
        return bits.value, ck.value

    def shard_prepare(self, dev_in_ptr, hist, n, block=0, finalize=0, flags=0):
        """Phase-independent part of a shard; returns (bits for entering phases 0..7, checksum of the shard bytes)."""
        bits = (C.c_ulonglong * 8)()
        ck = C.c_uint(1 if flags == 1 else 0)
        rc = self.L.zultra_cuda_shard_prepare(self.p, dev_in_ptr, hist, n, block, finalize, flags, C.byref(ck), bits)
        if rc != 0:
            raise RuntimeError("zultra_cuda_shard_prepare failed: %d" % rc)
        return [int(b) for b in bits], ck.value

    def shard_emit(self, in_bits, dev_out_ptr, out_cap):
        bits = C.c_ulonglong(0)
        rc = self.L.zultra_cuda_shard_emit(self.p, in_bits, dev_out_ptr, out_cap, C.byref(bits))
        if rc != 0:
            raise RuntimeError("zultra_cuda_shard_emit failed: %d" % rc)
        return bits.value

    def set_devices(self, n):
        """Spread every compress_blocks call of this context over n devices (zultra_cuda_ctx_set_devices); returns the count used."""
        return self.L.zultra_cuda_ctx_set_devices(self.p, n)

    def chunks_prepare(self, dev_in_ptr, chunks, block=0, flags=0):
        """chunks: [(offset of the chunk's history start in the resident buffer, history bytes, chunk bytes, finalize)].
        Returns (maps [n][8], checksums [n])."""
        n = len(chunks)
        off = (C.c_size_t * n)(*[c[0] for c in chunks]); hist = (C.c_int * n)(*[c[1] for c in chunks])
        ln = (C.c_size_t * n)(*[c[2] for c in chunks]); fin = (C.c_int * n)(*[c[3] for c in chunks])
        cks = (C.c_uint * n)(); maps = (C.c_ulonglong * (8 * n))()
        rc = self.L.zultra_cuda_chunks_prepare(self.p, dev_in_ptr, n, off, hist, ln, fin, block, flags, cks, maps)
        if rc != 0:
            raise RuntimeError("zultra_cuda_chunks_prepare failed: %d" % rc)
        return [[int(maps[8 * i + p]) for p in range(8)] for i in range(n)], [int(c) for c in cks]

    def chunks_emit(self, in_bits):
        """Emit the prepared chunks at their entering phases; returns (device pointer, byte offsets [n], bits [n])."""
        n = len(in_bits)
        ib = (C.c_uint * n)(*in_bits); off = (C.c_size_t * n)(); bits = (C.c_ulonglong * n)(); ptr = C.c_void_p()
        rc = self.L.zultra_cuda_chunks_emit(self.p, ib, C.byref(ptr), off, bits)
        if rc != 0:
            raise RuntimeError("zultra_cuda_chunks_emit failed: %d" % rc)
        return ptr.value, [int(o) for o in off], [int(b) for b in bits]

    def stitch_device(self, dev_dst_ptr, src_ptrs, dst_bits, nbits):
        n = len(src_ptrs)
        sp = (C.c_void_p * n)(*src_ptrs); db = (C.c_ulonglong * n)(*dst_bits); nb = (C.c_ulonglong * n)(*nbits)
        rc = self.L.zultra_cuda_stitch_device(self.p, dev_dst_ptr, n, sp, db, nb)
        if rc != 0:
            raise RuntimeError("zultra_cuda_stitch_device failed: %d" % rc)

    def window_sa_lcp(self, win):
        w = _u8(win)
        out = np.zeros(len(w), dtype=np.uint32)
        rc = self.L.zultra_cuda_window_sa_lcp(self.p, w.ctypes.data, len(w), out.ctypes.data)
        if rc != 0:
            raise RuntimeError("zultra_cuda_window_sa_lcp failed: %d" % rc)
        return out

    def window_matches(self, win, hist, tile=0):
        w = _u8(win)
        out = np.zeros(((len(w) - hist) * 8, 2), dtype=np.uint16)
        rc = self.L.zultra_cuda_window_matches(self.p, w.ctypes.data, hist, len(w), out.ctypes.data, tile)
        if rc != 0:
            raise RuntimeError("zultra_cuda_window_matches failed: %d" % rc)
        return out

    def block_stages(self, win, hist):
        w = _u8(win)
        info = np.zeros((64, 8), dtype=np.int32); ll = np.zeros((64, 288), dtype=np.int32); ol = np.zeros((64, 32), dtype=np.int32)
        best = np.zeros((len(w), 2), dtype=np.uint16)
        k = self.L.zultra_cuda_block_stages(self.p, w.ctypes.data, hist, len(w), info.ctypes.data, ll.ctypes.data, ol.ctypes.data, best.ctypes.data)
        if k < 0:
            raise RuntimeError("zultra_cuda_block_stages failed: %d" % k)
        return dict(n=k, info=info[:k], ll=ll[:k], ol=ol[:k], best=best)

    def timings(self):
        ms = (C.c_float * 8)()
        self.L.zultra_cuda_last_timings(self.p, ms)
        return dict(zip(["h2d", "sa_lcp", "match", "greedy_split", "parse", "emit", "d2h", "total"], [float(x) for x in ms]))

    def counters(self):
        v = (C.c_longlong * 8)()
        self.L.zultra_cuda_last_counters(self.p, v)
        return dict(zip(["windows", "sub_blocks", "sa_rounds", "parse_redo", "launches", "r5", "devices", "r7"], [int(x) for x in v]))

    def memory_compress_batch(self, payloads, flags=ZULTRA_FLAG_ZLIB_FRAMING, block=0, dictionary=None):
        """One stream per payload; None where the C call reports (size_t)-1.  With `dictionary`, every payload is compressed
        against that preset dictionary (zultra_cuda_memory_compress_batch_dict), as a Stream with set_dictionary would."""
        n = len(payloads)
        arrs = [_u8(p) for p in payloads]
        d = _u8(dictionary) if dictionary is not None else None
        # zlib framing with a dictionary: the 4-byte DICTID, which zultra_memory_bound does not count (neither does the reference's)
        dictid = 4 if d is not None and len(d) and (flags & 3) == ZULTRA_FLAG_ZLIB_FRAMING else 0
        caps = [memory_bound(len(a), flags, block) + dictid for a in arrs]
        outs = [np.empty(c, dtype=np.uint8) for c in caps]
        inp = (C.c_void_p * n)(*[a.ctypes.data for a in arrs]); ins = (C.c_size_t * n)(*[len(a) for a in arrs])
        outp = (C.c_void_p * n)(*[o.ctypes.data for o in outs]); oc = (C.c_size_t * n)(*caps); osz = (C.c_size_t * n)()
        if d is None:
            rc = self.L.zultra_cuda_memory_compress_batch(self.p, inp, ins, outp, oc, osz, n, flags, block)
        else:
            rc = self.L.zultra_cuda_memory_compress_batch_dict(self.p, inp, ins, outp, oc, osz, n, flags, block, d.ctypes.data if len(d) else None, len(d))
        if rc != 0:
            raise RuntimeError("zultra_cuda_memory_compress_batch%s failed: %d" % ("" if d is None else "_dict", rc))
        bad = C.c_size_t(-1).value
        return [None if osz[i] == bad else outs[i][: osz[i]].tobytes() for i in range(n)]


def memory_compress_batch(payloads, flags=ZULTRA_FLAG_ZLIB_FRAMING, block=0, device=-1, dictionary=None):
    ctx = CudaCtx(device)
    try:
        return ctx.memory_compress_batch(payloads, flags, block, dictionary=dictionary)
    finally:
        ctx.close()
