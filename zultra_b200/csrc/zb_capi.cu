/*
 * zb_capi.cu - the C-ABI of include/zultra_cuda.h over the CUDA pipeline.
 */
#include "zb_engine.h"
#include "../../include/zultra_cuda.h"
#include <new>
#include <mutex>
#include <thread>


struct zultra_cuda_ctx_s {
   int device;
   int broken = 0;      /* a CUDA call or allocation failed in this context: it is destroyed, never pooled again */
   unsigned tile = 0;
   ZbPipe pipe;
   float ms[8];
   long long counters[8];
   std::vector<uint8_t> out;
   /* several devices behind one context (zultra_cuda_ctx_set_devices): peers[k - 1] is the context on device (device + k) % count */
   int ndev = 1;
   std::vector<zultra_cuda_ctx_s *> peers;
   int nchunks = 0;      /* chunks of the last zultra_cuda_chunks_prepare */
};

/* ZULTRA_CUDA_TRACE=1: timestamps (ms since the first traced event of the process) of the API's milestones on stderr */
static void zb_trace(const char *what, const float *ms = 0) {
   static const int on = getenv("ZULTRA_CUDA_TRACE") ? atoi(getenv("ZULTRA_CUDA_TRACE")) : 0;
   if (!on) return;
   static const double t0 = zb_now_ms();
   if (ms) fprintf(stderr, "[zb %9.2f ms] %s: h2d %.2f sa %.2f match %.2f split %.2f parse %.2f emit %.2f d2h %.2f total %.2f\n", zb_now_ms() - t0, what, ms[0], ms[1], ms[2], ms[3], ms[4], ms[5], ms[6], ms[7]);
   else fprintf(stderr, "[zb %9.2f ms] %s\n", zb_now_ms() - t0, what);
}

extern "C" void zultra_cuda_trace(const char *what) { zb_trace(what ? what : ""); }

static int ctx_enter(zultra_cuda_ctx_t *c) {
   if (!c) return ZULTRA_CUDA_ERR_ARG;
   if (cudaSetDevice(c->device) != cudaSuccess) return ZULTRA_CUDA_ERR_CUDA;
   g_zb_cuda_error = 0;
   return 0;
}
static int ctx_leave(zultra_cuda_ctx_t *c, int rc) {
   if (g_zb_cuda_error) { cudaGetLastError(); c->broken = 1; return ZULTRA_CUDA_ERR_CUDA; }
   cudaError_t e = cudaGetLastError();
   if (e != cudaSuccess) { fprintf(stderr, "zultra-b200: CUDA error %s\n", cudaGetErrorString(e)); c->broken = 1; return ZULTRA_CUDA_ERR_CUDA; }
   if (rc == ZULTRA_CUDA_ERR_CUDA) c->broken = 1;
   return rc;
}
static void fill_counters(zultra_cuda_ctx_t *c, long long launches0) {
   ZbPipe &p = c->pipe;
   c->counters[0] = p.nwin; c->counters[1] = p.nsub; c->counters[2] = p.stat_sa_rounds;
   c->counters[4] = g_zb_launches - launches0;
   c->counters[3] = p.stat_redo; c->counters[7] = p.stat_tiles;
}

extern "C" {

int zultra_cuda_device_count(void) {
   int n = 0;
   if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
   return n;
}

int zultra_cuda_ctx_create(zultra_cuda_ctx_t **pp, int device) {
   if (!pp) return ZULTRA_CUDA_ERR_ARG;
   *pp = 0;
   zb_trace("ctx_create: begin");
   int n = zultra_cuda_device_count();
   zb_trace("ctx_create: device count known (driver initialised)");
   if (n <= 0) return ZULTRA_CUDA_ERR_NODEVICE;
   if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
   if (device >= n) return ZULTRA_CUDA_ERR_NODEVICE;
   if (cudaSetDevice(device) != cudaSuccess) return ZULTRA_CUDA_ERR_CUDA;
   zultra_cuda_ctx_t *c = new (std::nothrow) zultra_cuda_ctx_t();
   if (!c) return ZULTRA_CUDA_ERR_ARG;
   c->device = device;
   c->pipe.device = device;
   memset(c->ms, 0, sizeof(c->ms)); memset(c->counters, 0, sizeof(c->counters));
   if (cudaStreamCreateWithFlags(&c->pipe.st, cudaStreamNonBlocking) != cudaSuccess) { delete c; return ZULTRA_CUDA_ERR_CUDA; }
   zb_trace("ctx_create: stream created (primary context up)");
   {  /* test hooks: chunk and tile lengths of large inputs on small ones (never change the output) */
      const char *e;
      if ((e = getenv("ZULTRA_CUDA_PARSE_CD")) && atoi(e) >= 64) c->pipe.parse_cd = atoi(e);
      if ((e = getenv("ZULTRA_CUDA_TILE")) && atoi(e) >= 256) c->tile = (unsigned)atoi(e);
   }
   *pp = c;
   return 0;
}

void zultra_cuda_ctx_destroy(zultra_cuda_ctx_t *c) {
   if (!c) return;
   cudaSetDevice(c->device);
   for (size_t i = 0; i < c->peers.size(); i++) zultra_cuda_ctx_destroy(c->peers[i]);
   cudaSetDevice(c->device);
   c->pipe.release_all();
   cudaStreamDestroy(c->pipe.st);
   delete c;
}

static int run_one(zultra_cuda_ctx_t *c, const ZbStreamIn &s, unsigned block, ZbRunOpts &o, std::vector<ZbStreamRes> &res) {
   long long l0 = g_zb_launches;
   zb_memset(c->pipe.st, 0, 0, 0);
   c->pipe.counters.need(64);
   zb_memset(c->pipe.st, c->pipe.counters.p, 0, 64 * 4);
   cudaEvent_t e0, e1;
   cudaEventCreate(&e0); cudaEventCreate(&e1);
   cudaEventRecord(e0, c->pipe.st);
   if (!o.tile_main) o.tile_main = c->tile;
   c->pipe.stat_redo = 0;
   int rc = zb_run_batch(c->pipe, &s, 1, block, c->out, res, o);
   cudaEventRecord(e1, c->pipe.st);
   cudaEventSynchronize(e1);
   memcpy(c->ms, o.ms, sizeof(c->ms));
   { float t = 0; if (cudaEventElapsedTime(&t, e0, e1) == cudaSuccess) c->ms[7] = t; }   /* device-side total, CUDA events on the launching stream */
   cudaEventDestroy(e0); cudaEventDestroy(e1);
   fill_counters(c, l0);
   return rc;
}

/* ============================================================ several GPUs behind one call ============================================================
 * A call = consecutive max-blocks of one stream (host memory in, host memory out).  The range is cut into CHUNKS of a few
 * max-blocks, dealt round-robin to the devices: every device gets a sample of the whole range, so a stream whose cost per
 * byte varies along its length (text next to binaries next to byte runs) still loads all devices evenly, without a cost
 * model.  A chunk is a shard in the sense of zultra_cuda_shard_prepare: its own 32 KiB of preceding input as history,
 * everything up to the sub-block sizes independent of the entering bit phase.  Per device ONE pipeline pass over all its
 * chunks (they are streams of one batch), driven by its own host thread:
 *   1. DMA of every chunk [history | bytes] straight from the caller's buffer, pipeline up to the sub-block sizes,
 *      an 8-entry phase map and a checksum per chunk;
 *   2. (host) the maps compose left to right into every chunk's entering phase and absolute bit offset - the bit-offset
 *      scan of the stitch (tests/test_cpu_shards.py checks this algebra against the reference);
 *   3. emission for the true phases, then every chunk's bytes go by DMA from its device straight to their byte offset in
 *      the caller's output buffer; the byte a chunk shares with its predecessor is OR-merged on the host.
 * No device-to-device traffic at all: the shard bitstreams meet in host memory, where the caller wants them.
 * Replaces the per-block loop of libzultra.c:269-438 across devices. */
static zultra_cuda_ctx_t *multi_dev_ctx(zultra_cuda_ctx_t *c, int k) {
   if (k == 0) return c;
   int count = zultra_cuda_device_count();
   while ((int)c->peers.size() < k) {
      zultra_cuda_ctx_t *q = 0;
      const int dev = (c->device + (int)c->peers.size() + 1) % count;
      if (zultra_cuda_ctx_create(&q, dev)) return 0;
      q->pipe.parse_cd = c->pipe.parse_cd; q->tile = c->tile;
      c->peers.push_back(q);
   }
   return c->peers[k - 1];
}

static size_t multi_chunk_blocks(size_t nblocks, int ndev) {
   size_t g = nblocks / ((size_t)ndev * 4);
   return g < 1 ? 1 : (g > 8 ? 8 : g);
}

static int run_multi(zultra_cuda_ctx_t *c, int ndev, const uint8_t *host_hist, int hist_size, const uint8_t *host_in, size_t n, unsigned block, int finalize,
                     unsigned in_bits, unsigned flags, unsigned *checksum, uint8_t *host_out, size_t out_cap, unsigned long long *out_bits) {
   const long long l0 = g_zb_launches;
   const int kind = (flags & 2) ? 2 : ((flags & 1) ? 1 : 0);
   const size_t nblocks = (n + block - 1) / block, G = multi_chunk_blocks(nblocks, ndev), nchunk = (nblocks + G - 1) / G;
   struct Chunk { size_t lo, hi; int dev, idx; unsigned ck; unsigned long long map[8], abs_bits, bits; size_t out_off; uint32_t first_word; };
   struct Dev { zultra_cuda_ctx_t *q; std::vector<int> chunks; int rc; ZbRunOpts o; };
   std::vector<Chunk> ch(nchunk);
   std::vector<Dev> D(ndev);
   for (int k = 0; k < ndev; k++) { D[k].q = multi_dev_ctx(c, k); D[k].rc = 0; if (!D[k].q) return ZULTRA_CUDA_ERR_CUDA; }
   for (size_t j = 0; j < nchunk; j++) {
      ch[j].lo = j * G * block; ch[j].hi = std::min(n, (j + 1) * G * block); ch[j].dev = (int)(j % ndev); ch[j].idx = (int)D[ch[j].dev].chunks.size();
      D[ch[j].dev].chunks.push_back((int)j);
   }
   ZbTimer tot;
   auto prepare = [&](int k) {
      Dev &d = D[k];
      if (d.chunks.empty()) return;
      g_zb_cuda_error = 0;
      if (cudaSetDevice(d.q->device) != cudaSuccess) { d.rc = -3; return; }
      std::vector<ZbStreamIn> s(d.chunks.size());
      for (size_t i = 0; i < d.chunks.size(); i++) {
         const Chunk &x = ch[d.chunks[i]];
         const bool first = d.chunks[i] == 0;
         const uint32_t h = first ? (uint32_t)hist_size : (uint32_t)ZB_HISTORY;
         ZbStreamIn t = {host_in + x.lo, x.hi - x.lo, first ? host_hist : host_in + x.lo - h, h, (finalize && x.hi == n) ? 1 : 0, 0,
                         kind == 1 ? 1u : 0u /* every chunk from the initial value; folded into the running checksum below */, 0};
         s[i] = t;
      }
      d.o = ZbRunOpts();
      d.o.phase = 1; d.o.checksum_kind = kind; d.o.tile_main = c->tile; d.o.direct_h2d = 1;
      d.q->pipe.counters.need(64);
      zb_memset(d.q->pipe.st, d.q->pipe.counters.p, 0, 64 * 4);
      d.q->pipe.stat_redo = 0;
      std::vector<ZbStreamRes> res;
      d.rc = zb_run_batch(d.q->pipe, s.data(), (int)s.size(), block, d.q->out, res, d.o);
      if (zb_failed()) d.rc = -3;
      if (d.rc) { d.q->broken = 1; return; }
      for (size_t i = 0; i < d.chunks.size(); i++) {
         Chunk &x = ch[d.chunks[i]];
         memcpy(x.map, d.o.phase_maps.data() + 8 * i, sizeof(x.map));
         x.ck = res[i].checksum;
      }
   };
   {
      std::vector<std::thread> th;
      for (int k = 1; k < ndev; k++) th.emplace_back(prepare, k);
      prepare(0);
      for (size_t i = 0; i < th.size(); i++) th[i].join();
   }
   for (int k = 0; k < ndev; k++) if (D[k].rc) return ZULTRA_CUDA_ERR_CUDA;
   /* the bit-offset scan */
   unsigned long long pos = in_bits;
   for (size_t j = 0; j < nchunk; j++) { ch[j].abs_bits = pos; pos += ch[j].map[pos & 7] - (pos & 7); }
   const size_t nb_total = (size_t)((pos + 7) / 8);
   if (nb_total > out_cap) return ZULTRA_CUDA_ERR_DST;
   const float t_prep = tot.lap();
   auto emit = [&](int k) {
      Dev &d = D[k];
      if (d.chunks.empty()) return;
      g_zb_cuda_error = 0;
      if (cudaSetDevice(d.q->device) != cudaSuccess) { d.rc = -3; return; }
      const size_t m = d.chunks.size();
      std::vector<unsigned> ib(m); std::vector<size_t> off(m); std::vector<unsigned long long> bits(m);
      for (size_t i = 0; i < m; i++) ib[i] = (unsigned)(ch[d.chunks[i]].abs_bits & 7);
      d.rc = zb_finish_chunks(d.q->pipe, ib.data(), off.data(), bits.data());
      if (d.rc) { d.q->broken = 1; return; }
      const uint8_t *ob = (const uint8_t *)d.q->pipe.out.p;
      for (size_t i = 0; i < m; i++) {
         Chunk &x = ch[d.chunks[i]];
         x.bits = bits[i]; x.out_off = off[i];
         const size_t nb = (size_t)((bits[i] + 7) / 8), at = (size_t)(x.abs_bits >> 3);
         /* a chunk entered at phase p != 0 shares its first byte with its predecessor: that byte is merged on the host below
            (the very first chunk's pending bits belong to the caller, its low bits are zero here) */
         const size_t skip = (ib[i] != 0 && d.chunks[i] != 0) ? 1 : 0;
         if (skip) zb_d2h(d.q->pipe.st, &x.first_word, ob + off[i], 4);
         if (nb > skip) zb_d2h(d.q->pipe.st, host_out + at + skip, ob + off[i] + skip, nb - skip);
      }
      zb_sync(d.q->pipe.st);
      if (zb_failed()) { d.rc = -3; d.q->broken = 1; }
   };
   {
      std::vector<std::thread> th;
      for (int k = 1; k < ndev; k++) th.emplace_back(emit, k);
      emit(0);
      for (size_t i = 0; i < th.size(); i++) th[i].join();
   }
   for (int k = 0; k < ndev; k++) if (D[k].rc) return ZULTRA_CUDA_ERR_CUDA;
   for (size_t j = 1; j < nchunk; j++) if (ch[j].abs_bits & 7) host_out[ch[j].abs_bits >> 3] |= (uint8_t)(ch[j].first_word & 0xffu);
   *out_bits = pos;
   if (checksum) {
      unsigned ck = *checksum;
      for (size_t j = 0; j < nchunk; j++) ck = zultra_cuda_checksum_combine(flags, ck, ch[j].ck, ch[j].hi - ch[j].lo);
      *checksum = ck;
   }
   memset(c->ms, 0, sizeof(c->ms)); memset(c->counters, 0, sizeof(c->counters));
   for (int k = 0; k < ndev; k++) {
      if (D[k].chunks.empty()) continue;
      ZbPipe &p = D[k].q->pipe;
      for (int i = 0; i < 7; i++) c->ms[i] = std::max(c->ms[i], D[k].o.ms[i]);
      c->counters[0] += p.nwin; c->counters[1] += p.nsub; c->counters[2] = std::max<long long>(c->counters[2], p.stat_sa_rounds);
      c->counters[3] += p.stat_redo; c->counters[7] += p.stat_tiles;
   }
   c->ms[6] = tot.lap(); c->ms[7] = t_prep + c->ms[6];
   c->counters[4] = g_zb_launches - l0; c->counters[6] = ndev;
   return 0;
}

static unsigned clamp_block(unsigned b) {
   if (!b) b = 1048576;
   if (b < 32768) b = 32768;
   if (b > 2097152) b = 2097152;
   return b;
}

int zultra_cuda_compress_blocks(zultra_cuda_ctx_t *c, const unsigned char *hist, int hist_size, const unsigned char *in, size_t n,
                                unsigned int block, int finalize, unsigned int in_bits, unsigned int flags, unsigned int *checksum,
                                unsigned char *out, size_t out_cap, unsigned long long *out_bits) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   if (!in || !out || !out_bits || in_bits > 7 || hist_size < 0 || hist_size > ZB_HISTORY) return ZULTRA_CUDA_ERR_ARG;
   if (c->ndev > 1 && n > clamp_block(block)) {      /* at least two max-blocks: spread them over the context's devices */
      const size_t nblocks = (n + clamp_block(block) - 1) / clamp_block(block);
      const int nd = (int)std::min<size_t>((size_t)c->ndev, nblocks);
      rc = run_multi(c, nd, hist, hist_size, in, n, clamp_block(block), finalize, in_bits, flags, checksum, out, out_cap, out_bits);
      cudaSetDevice(c->device);
      { char msg[64]; snprintf(msg, sizeof msg, "compress_blocks: end, devices %d", nd); zb_trace(msg, c->ms); }
      return ctx_leave(c, rc);
   }
   ZbStreamIn s = {in, n, hist, (uint32_t)hist_size, finalize, in_bits, checksum ? *checksum : 0};
   ZbRunOpts o;
   o.checksum_kind = (flags & 2) ? 2 : ((flags & 1) ? 1 : 0);
   o.host_out = out; o.host_out_cap = out_cap;
   std::vector<ZbStreamRes> res;
   zb_trace("compress_blocks: begin");
   rc = run_one(c, s, clamp_block(block), o, res);
   zb_trace("compress_blocks: end", c->ms);
   if (rc == 0) { *out_bits = res[0].total_bits; if (checksum) *checksum = res[0].checksum; }
   else rc = rc == -2 ? ZULTRA_CUDA_ERR_DST : ZULTRA_CUDA_ERR_CUDA;
   return ctx_leave(c, rc);
}

int zultra_cuda_shard_prepare(zultra_cuda_ctx_t *c, const void *dev_in, int hist_size, size_t n, unsigned int block, int finalize, unsigned int flags,
                              unsigned int *checksum, unsigned long long *phase_bits8) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   if (!dev_in || !phase_bits8 || hist_size < 0 || hist_size > ZB_HISTORY) return ZULTRA_CUDA_ERR_ARG;
   ZbStreamIn s = {0, n, 0, (uint32_t)hist_size, finalize, 0, checksum ? *checksum : 0};
   ZbRunOpts o;
   o.dev_in = (const uint8_t *)dev_in; o.phase = 1;
   o.checksum_kind = (flags & 2) ? 2 : ((flags & 1) ? 1 : 0);
   std::vector<ZbStreamRes> res;
   rc = run_one(c, s, clamp_block(block), o, res);
   if (rc == 0) { memcpy(phase_bits8, o.phase_bits, sizeof(o.phase_bits)); if (checksum) *checksum = res[0].checksum; }
   return ctx_leave(c, rc ? ZULTRA_CUDA_ERR_CUDA : 0);
}

int zultra_cuda_shard_emit(zultra_cuda_ctx_t *c, unsigned int in_bits, void *dev_out, size_t out_cap, unsigned long long *out_bits) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   if (!dev_out || !out_bits || in_bits > 7) return ZULTRA_CUDA_ERR_ARG;
   long long l0 = g_zb_launches;
   rc = zb_finish_shard(c->pipe, in_bits, (uint8_t *)dev_out, out_cap, out_bits);
   c->counters[4] += g_zb_launches - l0;
   return ctx_leave(c, rc == -2 ? ZULTRA_CUDA_ERR_DST : (rc ? ZULTRA_CUDA_ERR_CUDA : 0));
}

unsigned int zultra_cuda_checksum_combine(unsigned int flags, unsigned int ck1, unsigned int ck2, unsigned long long len2) {
   if (flags & 2) return zb_crc32_combine(ck1, ck2, len2);
   if (flags & 1) {   /* adler32 of A||B from adler(A), adler(B) (B started from 1), len(B) */
      const unsigned long long BASE = 65521;
      unsigned long long rem = len2 % BASE, sum1 = ck1 & 0xffff, sum2 = (rem * sum1) % BASE;
      sum1 += (ck2 & 0xffff) + BASE - 1;
      sum2 += ((ck1 >> 16) & 0xffff) + ((ck2 >> 16) & 0xffff) + BASE - rem;
      if (sum1 >= BASE) sum1 -= BASE;
      if (sum1 >= BASE) sum1 -= BASE;
      if (sum2 >= (BASE << 1)) sum2 -= (BASE << 1);
      if (sum2 >= BASE) sum2 -= BASE;
      return (unsigned int)(sum1 | (sum2 << 16));
   }
   return 0;
}

int zultra_cuda_compress_blocks_device(zultra_cuda_ctx_t *c, const void *dev_in, size_t n, unsigned int block, int finalize,
                                       unsigned int flags, unsigned int *checksum, void *dev_out, size_t out_cap, unsigned long long *out_bits) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   if (!dev_in || !dev_out || !out_bits) return ZULTRA_CUDA_ERR_ARG;
   ZbStreamIn s = {0, n, 0, 0, finalize, 0, checksum ? *checksum : 0};
   ZbRunOpts o;
   o.dev_in = (const uint8_t *)dev_in; o.dev_out = (uint8_t *)dev_out; o.dev_out_cap = out_cap;
   o.checksum_kind = (flags & 2) ? 2 : ((flags & 1) ? 1 : 0);
   std::vector<ZbStreamRes> res;
   rc = run_one(c, s, clamp_block(block), o, res);
   if (rc == 0) { *out_bits = res[0].total_bits; if (checksum) *checksum = res[0].checksum; }
   else rc = rc == -2 ? ZULTRA_CUDA_ERR_DST : ZULTRA_CUDA_ERR_CUDA;
   return ctx_leave(c, rc);
}

int zultra_cuda_ctx_set_devices(zultra_cuda_ctx_t *c, int n) {
   if (!c) return ZULTRA_CUDA_ERR_ARG;
   const int count = zultra_cuda_device_count();
   if (n < 1) n = 1;
   if (n > count) n = count;
   c->ndev = n;
   return n;
}

/* ---- several chunks of one device-resident buffer per call (one process per GPU: bench.py under torchrun) ---- */
int zultra_cuda_chunks_prepare(zultra_cuda_ctx_t *c, const void *dev_in, int nchunks, const size_t *chunk_off, const int *chunk_hist, const size_t *chunk_len,
                               const int *chunk_final, unsigned int block, unsigned int flags, unsigned int *cks, unsigned long long *maps8) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   if (!dev_in || nchunks <= 0 || !chunk_off || !chunk_hist || !chunk_len || !maps8) return ZULTRA_CUDA_ERR_ARG;
   const int kind = (flags & 2) ? 2 : ((flags & 1) ? 1 : 0);
   std::vector<ZbStreamIn> s((size_t)nchunks);
   for (int i = 0; i < nchunks; i++) {
      if (chunk_hist[i] < 0 || chunk_hist[i] > ZB_HISTORY || !chunk_len[i]) return ZULTRA_CUDA_ERR_ARG;
      ZbStreamIn t = {0, chunk_len[i], 0, (uint32_t)chunk_hist[i], chunk_final ? chunk_final[i] : 0, 0, kind == 1 ? 1u : 0u, chunk_off[i]};
      s[i] = t;
   }
   const long long l0 = g_zb_launches;
   ZbRunOpts o;
   o.dev_in = (const uint8_t *)dev_in; o.dev_offsets = 1; o.phase = 1; o.checksum_kind = kind; o.tile_main = c->tile;
   c->pipe.counters.need(64);
   zb_memset(c->pipe.st, c->pipe.counters.p, 0, 64 * 4);
   c->pipe.stat_redo = 0;
   std::vector<ZbStreamRes> res;
   rc = zb_run_batch(c->pipe, s.data(), nchunks, clamp_block(block), c->out, res, o);
   memcpy(c->ms, o.ms, sizeof(c->ms));
   fill_counters(c, l0);
   if (rc == 0) {
      memcpy(maps8, o.phase_maps.data(), sizeof(unsigned long long) * 8 * (size_t)nchunks);
      if (cks) for (int i = 0; i < nchunks; i++) cks[i] = res[i].checksum;
      c->nchunks = nchunks;
   }
   return ctx_leave(c, rc ? ZULTRA_CUDA_ERR_CUDA : 0);
}

int zultra_cuda_chunks_emit(zultra_cuda_ctx_t *c, const unsigned int *in_bits, void **dev_out, size_t *out_off, unsigned long long *out_bits) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   if (!in_bits || !dev_out || !out_off || !out_bits || c->nchunks <= 0 || (int)c->pipe.plan.size() != c->nchunks) return ZULTRA_CUDA_ERR_ARG;
   const long long l0 = g_zb_launches;
   rc = zb_finish_chunks(c->pipe, in_bits, out_off, out_bits);
   *dev_out = c->pipe.out.p;
   c->counters[4] += g_zb_launches - l0;
   return ctx_leave(c, rc ? ZULTRA_CUDA_ERR_CUDA : 0);
}

/* The stitch on one device: part i = src[i][0 .. ceil((phase_i + nbits_i) / 8)) bytes, its first bit at phase_i = dst_bit[i] & 7 of
   its first byte (the bits below are zero), goes to byte dst_bit[i] >> 3 of dst; bytes two parts share are OR-merged.  dst must be
   zero where parts meet: the caller clears it before the call.  Grid: y = part, x strides over the aligned 32-bit words of the
   part's destination span; a word comes out of two aligned source words and a funnel shift, interior words are plain stores,
   the first and last word of a part go through atomicOr.  Every source span is followed by >= 8 readable zero bytes (the
   pipeline's output spans are; zultra_cuda.h states it for other callers). */
struct ZbStitchPart { const uint8_t *src; unsigned long long dst_bit, nbits; };
__global__ void __launch_bounds__(256) zb_stitch_k(uint32_t *dst, const ZbStitchPart *parts) {
   const ZbStitchPart p = parts[blockIdx.y];
   const unsigned long long b0 = p.dst_bit >> 3, nb = ((p.dst_bit & 7) + p.nbits + 7) >> 3;
   if (!nb) return;
   const unsigned long long w0 = b0 >> 2, nwords = ((b0 + nb + 3) >> 2) - w0;
   for (unsigned long long j = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; j < nwords; j += (unsigned long long)gridDim.x * blockDim.x) {
      const long long s0 = (long long)((w0 + j) << 2) - (long long)b0;      /* source byte that lands in byte 0 of this word (< 0 only for j = 0) */
      uint32_t v;
      if (s0 >= 0 && (unsigned long long)s0 + 4 <= nb) {
         const uintptr_t a = (uintptr_t)(p.src + s0);
         const uint32_t *pa = (const uint32_t *)(a & ~(uintptr_t)3);
         v = (a & 3) ? __funnelshift_r(pa[0], pa[1], (uint32_t)(a & 3) << 3) : pa[0];
      } else {
         v = 0;
#pragma unroll
         for (int k = 0; k < 4; k++) { const long long q = s0 + k; if (q >= 0 && (unsigned long long)q < nb) v |= (uint32_t)p.src[q] << (8 * k); }
      }
      if (!v) continue;
      if (s0 < 1 || (unsigned long long)s0 + 4 >= nb) atomicOr(dst + w0 + j, v); else dst[w0 + j] = v;      /* an edge word may share bytes with a neighbouring part */
   }
}

int zultra_cuda_stitch_device(zultra_cuda_ctx_t *c, void *dev_dst, int nparts, const void *const *dev_src, const unsigned long long *dst_bit, const unsigned long long *nbits) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   if (!dev_dst || nparts <= 0 || nparts > 65535 || !dev_src || !dst_bit || !nbits || ((uintptr_t)dev_dst & 3)) return ZULTRA_CUDA_ERR_ARG;
   std::vector<ZbStitchPart> h((size_t)nparts);
   unsigned long long maxwords = 0;
   for (int i = 0; i < nparts; i++) {
      h[i].src = (const uint8_t *)dev_src[i]; h[i].dst_bit = dst_bit[i]; h[i].nbits = nbits[i];
      maxwords = std::max(maxwords, (((dst_bit[i] & 7) + nbits[i] + 7) >> 5) + 2);
   }
   c->pipe.ck_rng.need(((size_t)nparts * sizeof(ZbStitchPart) + 7) / 8);
   if (zb_failed()) return ctx_leave(c, ZULTRA_CUDA_ERR_CUDA);
   zb_h2d(c->pipe.st, c->pipe.ck_rng.p, h.data(), h.size() * sizeof(ZbStitchPart));
   const unsigned gx = (unsigned)std::min<unsigned long long>(std::max<unsigned long long>((maxwords + 1023) / 1024, 1), 4096);
   zb_stitch_k<<<dim3(gx, (unsigned)nparts), 256, 0, c->pipe.st>>>((uint32_t *)dev_dst, (const ZbStitchPart *)c->pipe.ck_rng.p);
   zb_count_launch(1);
   ZB_CUDA_CHECK(cudaGetLastError());
   zb_sync(c->pipe.st);
   return ctx_leave(c, 0);
}

/* ---- context pool: contexts (device buffers, stream) are expensive to build; the libzultra front end borrows them ---- */
static std::mutex g_pool_mu;
static std::vector<zultra_cuda_ctx_t *> g_pool;

int zultra_cuda_ctx_acquire(zultra_cuda_ctx_t **pp, int device) {
   if (!pp) return ZULTRA_CUDA_ERR_ARG;
   if (device < 0) { if (zultra_cuda_device_count() <= 0) return ZULTRA_CUDA_ERR_NODEVICE; if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
   {
      std::lock_guard<std::mutex> g(g_pool_mu);
      for (size_t i = 0; i < g_pool.size(); i++)
         if (g_pool[i]->device == device) { *pp = g_pool[i]; g_pool.erase(g_pool.begin() + i); return 0; }
   }
   return zultra_cuda_ctx_create(pp, device);
}
void zultra_cuda_ctx_release(zultra_cuda_ctx_t *c) {
   if (!c) return;
   if (c->broken) { zultra_cuda_ctx_destroy(c); return; }
   std::lock_guard<std::mutex> g(g_pool_mu);
   if (g_pool.size() < 16) g_pool.push_back(c); else zultra_cuda_ctx_destroy(c);
}
void zultra_cuda_release_cached(void) {
   std::lock_guard<std::mutex> g(g_pool_mu);
   for (size_t i = 0; i < g_pool.size(); i++) zultra_cuda_ctx_destroy(g_pool[i]);
   g_pool.clear();
}

/* frame bytes written on the host side of the batch call (frame.c:387-452, :509-547) */
static size_t put_header(unsigned char *o, unsigned flags) {
   if (flags & 2) { const unsigned char h[10] = {0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 2, 255}; memcpy(o, h, 10); return 10; }
   if (flags & 1) { o[0] = 0x78; o[1] = 0xda; return 2; }
   return 0;
}
static size_t put_footer(unsigned char *o, unsigned flags, unsigned ck, unsigned long long n) {
   if (flags & 2) { for (int i = 0; i < 4; i++) { o[i] = (unsigned char)(ck >> (8 * i)); o[4 + i] = (unsigned char)(n >> (8 * i)); } return 8; }
   if (flags & 1) { for (int i = 0; i < 4; i++) o[i] = (unsigned char)(ck >> (8 * (3 - i))); return 4; }
   return 0;
}

int zultra_cuda_memory_compress_batch(zultra_cuda_ctx_t *c, const unsigned char *const *in, const size_t *in_sizes, unsigned char *const *outp,
                                      const size_t *out_caps, size_t *out_sizes, size_t nstreams, unsigned int flags, unsigned int block) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   block = clamp_block(block);
   long long l0 = g_zb_launches;
   const unsigned hdr = (flags & 2) ? 10 : ((flags & 1) ? 2 : 0), ftr = (flags & 2) ? 8 : ((flags & 1) ? 4 : 0);
   float ms[8] = {0};
   size_t i0 = 0;
   while (i0 < nstreams) {
      /* sub-batch: bounded positions */
      size_t i1 = i0, bytes = 0;
      std::vector<ZbStreamIn> s;
      while (i1 < nstreams && (i1 == i0 || bytes + in_sizes[i1] + ((in_sizes[i1] / block) * ZB_HISTORY) < ((size_t)768 << 20))) {
         if (in_sizes[i1] > 0) {   /* empty input yields (size_t)-1 like the reference (libzultra.c:275,617) */
            ZbStreamIn t = {in[i1], in_sizes[i1], 0, 0, 1, 0, (flags & 2) ? 0u : 1u};
            s.push_back(t);
            bytes += in_sizes[i1] + (in_sizes[i1] / block) * ZB_HISTORY;
         }
         i1++;
      }
      std::vector<ZbStreamRes> res;
      ZbRunOpts o;
      o.checksum_kind = (flags & 2) ? 2 : ((flags & 1) ? 1 : 0);
      o.want_out_ptr = 1;
      c->pipe.counters.need(64);
      zb_memset(c->pipe.st, c->pipe.counters.p, 0, 64 * 4);
      if (!s.empty() && zb_run_batch(c->pipe, s.data(), (int)s.size(), block, c->out, res, o)) return ctx_leave(c, ZULTRA_CUDA_ERR_CUDA);
      const uint8_t *obase = o.out_ptr ? o.out_ptr : c->out.data();
      for (int k = 0; k < 8; k++) ms[k] += o.ms[k];
      {  /* frame every stream into its caller buffer: 4 host threads for large batches (150 MB of output is 20 ms of one core's memcpy) */
         std::vector<size_t> kof(i1 - i0 + 1, 0);
         for (size_t i = i0; i < i1; i++) kof[i - i0 + 1] = kof[i - i0] + (in_sizes[i] ? 1 : 0);
         auto frame = [&](size_t a, size_t b) {
            for (size_t i = a; i < b; i++) {
               if (in_sizes[i] == 0) { out_sizes[i] = (size_t)-1; continue; }
               const size_t k = kof[i - i0];
               const size_t nb = (size_t)((res[k].total_bits + 7) / 8);
               if (hdr + nb + ftr > out_caps[i]) out_sizes[i] = (size_t)-1;
               else {
                  size_t w = put_header(outp[i], flags);
                  memcpy(outp[i] + w, obase + res[k].out_off, nb); w += nb;
                  w += put_footer(outp[i] + w, flags, res[k].checksum, in_sizes[i]);
                  out_sizes[i] = w;
               }
            }
         };
         const size_t cnt = i1 - i0;
         if (cnt < 2048) frame(i0, i1);
         else {
            std::thread th[3];
            for (int q = 0; q < 3; q++) th[q] = std::thread(frame, i0 + cnt * (size_t)(q + 1) / 4, i0 + cnt * (size_t)(q + 2) / 4);
            frame(i0, i0 + cnt / 4);
            for (int q = 0; q < 3; q++) th[q].join();
         }
      }
      i0 = i1;
   }
   memcpy(c->ms, ms, sizeof(ms));
   fill_counters(c, l0);
   return ctx_leave(c, 0);
}

int zultra_cuda_checksum_device(zultra_cuda_ctx_t *c, const void *dev, size_t n, unsigned int flags, unsigned int *ck) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   const int kind = (flags & 2) ? 2 : ((flags & 1) ? 1 : 0);
   if (!kind) { *ck = 0; return 0; }
   c->pipe.in_ptr = (const uint8_t *)dev;
   std::vector<uint64_t> off(1, 0), len(1, n); std::vector<uint32_t> sums;
   c->pipe.stage_checksum(kind, off, len, sums, *ck);
   *ck = sums[0];
   return ctx_leave(c, 0);
}

int zultra_cuda_window_sa_lcp(zultra_cuda_ctx_t *c, const unsigned char *win, int n, unsigned int *words) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   ZbStreamIn s = {win, (size_t)n, 0, 0, 1, 0, 0};
   ZbRunOpts o; ZbDump d; o.dump = &d; o.stop_after = 1;
   std::vector<ZbStreamRes> res;
   c->pipe.sa_exact = true;                          /* the parity artefact is the exact suffix array */
   rc = run_one(c, s, 2097152u + 65536u, o, res);   /* one window: block size above any window */
   c->pipe.sa_exact = false;
   if (rc == 0) memcpy(words, d.sa_lcp.data(), (size_t)n * 4);
   return ctx_leave(c, rc ? ZULTRA_CUDA_ERR_CUDA : 0);
}

int zultra_cuda_window_matches(zultra_cuda_ctx_t *c, const unsigned char *win, int hist, int n, unsigned short *matches, unsigned int tile) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   ZbStreamIn s = {win + hist, (size_t)(n - hist), win, (uint32_t)hist, 1, 0, 0};
   ZbRunOpts o; ZbDump d; o.dump = &d; o.stop_after = 2; o.tile_main = tile;
   std::vector<ZbStreamRes> res;
   rc = run_one(c, s, 2097152u + 65536u, o, res);
   if (rc == 0) memcpy(matches, d.match.data() + (size_t)hist * 8, (size_t)(n - hist) * 8 * sizeof(zb_match_t));
   return ctx_leave(c, rc ? ZULTRA_CUDA_ERR_CUDA : 0);
}

int zultra_cuda_block_stages(zultra_cuda_ctx_t *c, const unsigned char *win, int hist, int n, int *info, int *lit_len, int *off_len, unsigned short *best) {
   int rc = ctx_enter(c);
   if (rc) return rc;
   ZbStreamIn s = {win + hist, (size_t)(n - hist), win, (uint32_t)hist, 0, 0, 0};
   ZbRunOpts o; ZbDump d; o.dump = &d;
   std::vector<ZbStreamRes> res;
   rc = run_one(c, s, 2097152u + 65536u, o, res);
   if (rc) return ctx_leave(c, ZULTRA_CUDA_ERR_CUDA);
   for (size_t i = 0; i < d.sub.size(); i++) {
      const ZbSub &b = d.sub[i];
      int *q = info + 8 * i;
      q[0] = b.ps; q[1] = b.pe; q[2] = b.is_dyn; q[3] = b.static_cost; q[4] = b.dynamic_cost; q[5] = b.body_bits; q[6] = b.stored; q[7] = b.mask | (b.ub_hit << 8);
      for (int j = 0; j < 288; j++) lit_len[288 * i + j] = d.tabs[i].llen[j];
      for (int j = 0; j < 32; j++) off_len[32 * i + j] = d.tabs[i].olen[j];
   }
   if (best) memcpy(best, d.best.data(), (size_t)n * sizeof(zb_match_t));
   return ctx_leave(c, (int)d.sub.size());
}

long long zultra_cuda_launch_count(void) { return __atomic_load_n(&g_zb_launches, __ATOMIC_RELAXED); }
int zultra_cuda_last_timings(zultra_cuda_ctx_t *c, float *ms) { if (!c) return ZULTRA_CUDA_ERR_ARG; memcpy(ms, c->ms, sizeof(c->ms)); return 0; }
int zultra_cuda_last_counters(zultra_cuda_ctx_t *c, long long *v) { if (!c) return ZULTRA_CUDA_ERR_ARG; memcpy(v, c->counters, sizeof(c->counters)); return 0; }

}
