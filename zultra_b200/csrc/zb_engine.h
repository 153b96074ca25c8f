/*
 * zb_engine.h - host-side driver of one batch: builds the window list for a set of streams, runs the
 * pipeline stages and brings the stitched bitstreams back.
 */
#ifndef ZB_ENGINE_H
#define ZB_ENGINE_H
#include "zb_pipeline.h"
#include <chrono>
#include <thread>
#include <vector>

struct ZbStreamIn {
   const uint8_t *data; size_t n;          /* bytes to compress in this call (whole max-blocks except possibly the last) */
   const uint8_t *hist; uint32_t hist_len; /* <= 32768 bytes preceding data (previous block tail or preset dictionary) */
   int finalize;                           /* 1: the last window is the end of the stream (BFINAL) */
   uint32_t in_bits;                       /* bits already pending in the current output byte (0..7) */
   uint32_t checksum;                      /* running checksum in */
   size_t dev_off;                         /* with ZbRunOpts::dev_in and dev_offsets: where this stream's [history | data] starts in the resident buffer */
};
struct ZbStreamRes { uint64_t total_bits; size_t out_off; int err; uint32_t checksum; };

struct ZbDump {   /* optional stage dumps for tests (host copies) */
   std::vector<uint32_t> sa_lcp; std::vector<zb_match_t> match; std::vector<ZbSub> sub; std::vector<ZbSubTabs> tabs; std::vector<zb_match_t> best;
   std::vector<uint32_t> wbase;
};

struct ZbRunOpts {
   uint32_t tile_main = 0;
   int checksum_kind = 0;          /* 0 none, 1 Adler-32, 2 CRC-32 (frame.c:473) */
   const uint8_t *dev_in = 0;      /* single stream already in device memory: [hist_len history bytes | data] */
   int dev_offsets = 0;            /* dev_in holds several streams (chunks of one resident buffer): ZbStreamIn::dev_off locates each */
   int direct_h2d = 0;             /* several streams from host memory, each [history | data] contiguous there: one DMA per stream straight from the
                                      caller's buffer instead of gathering them into page-locked staging first */
   int shared_hist = 0;            /* several streams from host memory with the SAME history (s[i].hist and hist_len equal: a preset
                                      dictionary): gather and send the history once and the payloads packed, then build every
                                      stream's [history | data] on the device (stage_assemble) */
   int phase = 3;                  /* 1 = stop after the phase-independent part (shards), 2 = only finish, 3 = both */
   unsigned long long phase_bits[8] = {0, 0, 0, 0, 0, 0, 0, 0};
   std::vector<unsigned long long> phase_maps;   /* phase 1: 8 entries per stream (phase_bits = those of stream 0) */
   uint8_t *dev_out = 0; size_t dev_out_cap = 0;   /* leave the bitstream of stream 0 in device memory instead of copying back */
   uint8_t *host_out = 0; size_t host_out_cap = 0; /* single stream: copy the bitstream straight into the caller's buffer (no staging vector) */
   int want_out_ptr = 0;           /* several streams: leave the bitstreams in the pipe's page-locked buffer; res[i].out_off is relative to out_ptr */
   const uint8_t *out_ptr = 0;
   ZbDump *dump = 0;
   int stop_after = 99;            /* 1 = SA, 2 = match (stage dumps) */
   float ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};   /* h2d, sa, match, greedy+split, parse, emit, d2h, total */
};

/* main positions per match-finder tile: as large as shared memory allows (amortises the 32768 look-back entries every
   tile loads) while still giving every SM several tiles */
static inline uint32_t zb_pick_tile(size_t total) {
   uint32_t t = 16384;
   while (t > 512 && total / t < 600) t >>= 1;
   return t;
}

static inline double zb_now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
struct ZbTimer {
   std::chrono::steady_clock::time_point t0;
   ZbTimer() : t0(std::chrono::steady_clock::now()) {}
   float lap() { auto t = std::chrono::steady_clock::now(); float ms = std::chrono::duration<float, std::milli>(t - t0).count(); t0 = t; return ms; }
};

/* Returns 0 on success.  out receives, per stream, ceil(total_bits/8) bytes at res[i].out_off; the pending bits of the
   first byte are zero (the caller ORs its carried partial byte in). */
static inline int zb_run_batch(ZbPipe &p, const ZbStreamIn *s, int ns, uint32_t block_size, std::vector<uint8_t> &out,
                               std::vector<ZbStreamRes> &res, ZbRunOpts &o) {
   std::vector<ZbWinDesc> wins;
   std::vector<ZbStreamOut> so(ns);
   std::vector<uint64_t> ck_off(ns), ck_len(ns);
   size_t in_bytes = 0;
   for (int i = 0; i < ns; i++) in_bytes += s[i].hist_len + s[i].n;
   if (in_bytes >= ((size_t)1 << 31)) return -1;
   /* shared history: the staged input is [history | payload 0 | payload 1 | ...] (stage_assemble expands it on the device) */
   const bool shared = o.shared_hist && !o.dev_in && ns > 0;
   const uint32_t sh_len = shared ? s[0].hist_len : 0;
   for (int i = 0; i < ns && shared; i++) if (s[i].hist_len != sh_len || s[i].hist != s[0].hist) return -1;
   size_t stage_bytes = shared ? sh_len : in_bytes;
   for (int i = 0; i < ns && shared; i++) stage_bytes += s[i].n;
   ZbTimer tm, tot;
   /* copy straight from the caller's buffer when [history | data] is contiguous there; otherwise gather the streams into
      page-locked memory (several host threads: a single memcpy stream does not keep up with the DMA that follows) */
   const bool single_direct = (ns == 1 && !o.dev_in && !shared && (s[0].hist_len == 0 || s[0].hist + s[0].hist_len == s[0].data));
   bool multi_direct = ns > 1 && !o.dev_in && !shared && o.direct_h2d;
   for (int i = 0; i < ns && multi_direct; i++) if (s[i].hist_len && s[i].hist + s[i].hist_len != s[i].data) multi_direct = false;
   uint8_t *stage = 0;
   bool staged_to_device = false, pipe_fail = false;      /* the gather threads already sent the staged input to the device */
   if (!o.dev_in && !single_direct && !multi_direct) {
      p.hin.need(stage_bytes + 16);
      stage = p.hin.p;
      if (!stage || zb_failed()) return -3;
      std::vector<size_t> offs(ns + 1, sh_len);      /* where stream i's staged bytes start */
      for (int i = 0; i < ns; i++) offs[i + 1] = offs[i] + (shared ? 0 : s[i].hist_len) + s[i].n;
      const int nth = stage_bytes > ((size_t)8 << 20) ? 4 : 1;
#ifndef ZB_EMU
      /* large batches: every gathering thread sends what it has gathered to the device in 4 MiB pieces on its own stream, so the
         DMA runs under the remaining memcpys instead of after them (347 MB of small streams: 25 ms of gather + DMA -> the longer of the two) */
      const bool piped = nth > 1 && p.stager.init();
      ZbBuf<uint8_t> &dev_stage = shared ? p.pk : p.in;
      if (piped) { dev_stage.need(stage_bytes + 16); if (zb_failed()) return -3; staged_to_device = true; }
#else
      const bool piped = false;
#endif
      auto gather = [&](int a, int b, int lane) {
         size_t sent = a == 0 ? 0 : (a < ns ? offs[a] : stage_bytes);
         if (shared && a == 0 && b > 0) memcpy(stage, s[0].hist, sh_len);      /* the history once, ahead of the first payload */
         for (int i = a; i < b; i++) {
            const size_t h = shared ? 0 : s[i].hist_len;
            if (h) memcpy(stage + offs[i], s[i].hist, h);
            memcpy(stage + offs[i] + h, s[i].data, s[i].n);
#ifndef ZB_EMU
            if (piped && (offs[i + 1] - sent >= ((size_t)4 << 20) || i + 1 == b)) {
               cudaMemcpyAsync(dev_stage.p + sent, stage + sent, offs[i + 1] - sent, cudaMemcpyHostToDevice, p.stager.st[lane]);
               sent = offs[i + 1];
            }
#endif
         }
#ifndef ZB_EMU
         if (piped) { cudaSetDevice(p.device); if (cudaStreamSynchronize(p.stager.st[lane]) != cudaSuccess) pipe_fail = true; }
#endif
         (void)lane; (void)sent;
      };
      if (nth == 1) gather(0, ns, 0);
      else {
         std::vector<std::thread> th;
         int a = 0;
         for (int k = 0; k < nth; k++) {   /* equal byte shares */
            int b = a;
            while (b < ns && (k == nth - 1 || offs[b] < stage_bytes / nth * (k + 1))) b++;
            th.emplace_back(gather, a, b, k);
            a = b;
         }
         for (auto &t : th) t.join();
      }
   }
   size_t off = 0, total_block = 0;
   for (int i = 0; i < ns; i++) {
      memset(&so[i], 0, sizeof(ZbStreamOut));
      so[i].first_win = (uint32_t)wins.size();
      so[i].in_bits = s[i].in_bits;
      if (o.dev_in && o.dev_offsets) off = s[i].dev_off;
      ck_off[i] = off + s[i].hist_len; ck_len[i] = s[i].n;
      size_t done = 0; uint32_t k = 0;
      while (done < s[i].n) {
         ZbWinDesc d; memset(&d, 0, sizeof(d));
         size_t blk = std::min((size_t)block_size, s[i].n - done);
         d.hist = k == 0 ? s[i].hist_len : ZB_HISTORY;
         d.in_off = (uint32_t)(off + s[i].hist_len + done - d.hist);
         d.len = d.hist + (uint32_t)blk;
         d.stream = (uint32_t)i;
         done += blk; k++;
         d.last = (done == s[i].n && s[i].finalize) ? 1 : 0;
         wins.push_back(d);
      }
      so[i].nwin = k;
      off += s[i].hist_len + s[i].n;
      total_block += s[i].n;
   }
   res.assign(ns, ZbStreamRes());
   for (int i = 0; i < ns; i++) res[i].checksum = s[i].checksum;
   if (wins.empty()) { out.clear(); return 0; }
   if (pipe_fail) return -3;
   p.setup(wins, o.dev_in ? o.dev_in : (single_direct ? s[0].data - s[0].hist_len : ((staged_to_device || shared) ? (const uint8_t *)0 : stage)), in_bytes, o.dev_in != 0);
   if (multi_direct && !zb_failed()) {      /* setup allocated the device input (no source given): one DMA per stream */
      size_t at = 0;
      for (int i = 0; i < ns; i++) { zb_h2d(p.st, p.in.p + at, s[i].data - s[i].hist_len, s[i].hist_len + s[i].n); at += s[i].hist_len + s[i].n; }
   }
   if (shared && !zb_failed()) {      /* the packed input (already on the device when the gather sent it) -> [history | data] per stream */
      if (!staged_to_device) { p.pk.need(stage_bytes + 16); if (zb_failed()) return -3; zb_h2d(p.st, p.pk.p, stage, stage_bytes); }
      std::vector<uint32_t> tab(2 * (size_t)ns + 2);
      size_t a = 0, q = sh_len;
      for (int i = 0; i < ns; i++) { tab[2 * i] = (uint32_t)a; tab[2 * i + 1] = (uint32_t)q; a += sh_len + s[i].n; q += s[i].n; }
      tab[2 * (size_t)ns] = (uint32_t)a; tab[2 * (size_t)ns + 1] = (uint32_t)q;
      p.stage_assemble(tab, sh_len, in_bytes);
   }
   zb_sync(p.st); o.ms[0] = tm.lap();
   if (zb_failed()) return -3;      /* allocation or copy failed: nothing has been launched on missing buffers */
   p.stage_sa();
   zb_sync(p.st); o.ms[1] = tm.lap();
   if (zb_failed()) return -3;
   if (o.stop_after >= 2) {
      p.stage_match(o.tile_main ? o.tile_main : zb_pick_tile(total_block));
      zb_sync(p.st); o.ms[2] = tm.lap();
      if (zb_failed()) return -3;
   }
   if (o.stop_after >= 3) {
      p.stage_greedy();
      if (zb_failed()) return -3;
      p.stage_split();
      zb_sync(p.st); o.ms[3] = tm.lap();
      if (zb_failed()) return -3;
      p.stage_parse();
      zb_sync(p.st); o.ms[4] = tm.lap();
      if (zb_failed()) return -3;
      p.stage_emit_prepare();
      if (zb_failed()) return -3;
      if (o.phase == 1) {   /* shard(s): report the size for every entering phase and wait for zb_finish_shard / zb_finish_chunks */
         if (o.checksum_kind) {
            std::vector<uint32_t> sums;
            if (ns == 1) { p.stage_checksum(o.checksum_kind, ck_off, ck_len, sums, s[0].checksum); res[0].checksum = sums[0]; }
            else {      /* every stream from the initial value; the caller folds them with zultra_cuda_checksum_combine */
               p.stage_checksum(o.checksum_kind, ck_off, ck_len, sums, 0);
               for (int i = 0; i < ns; i++) res[i].checksum = sums[i];
            }
         }
         p.plan = so;
         o.phase_maps.assign((size_t)ns * 8, 0);
         p.phase_maps(so, o.phase_maps.data());
         memcpy(o.phase_bits, o.phase_maps.data(), sizeof(o.phase_bits));
         zb_sync(p.st); o.ms[5] = tm.lap(); o.ms[7] = tot.lap();
         return zb_failed() ? -3 : 0;
      }
      p.stage_emit_finish(so);
      if (zb_failed()) return -3;
      if (o.checksum_kind) {
         std::vector<uint32_t> sums;
         if (ns == 1) { p.stage_checksum(o.checksum_kind, ck_off, ck_len, sums, s[0].checksum); res[0].checksum = sums[0]; }
         else { p.stage_checksum(o.checksum_kind, ck_off, ck_len, sums, 0); for (int i = 0; i < ns; i++) res[i].checksum = sums[i]; }
      }
      zb_sync(p.st); o.ms[5] = tm.lap();
      size_t ob = 0;
      for (int i = 0; i < ns; i++) { res[i].total_bits = p.h_sout[i].total_bits; res[i].out_off = ob; res[i].err = 0; ob += (size_t)((p.h_sout[i].total_bits + 7) / 8); }
      if (o.dev_out) {
         const size_t nb = (size_t)((p.h_sout[0].total_bits + 7) / 8);
         if (nb > o.dev_out_cap) return -2;
         zb_d2d(p.st, o.dev_out, p.out.p + p.h_sout[0].out_word_off, nb);
         zb_sync(p.st);
         out.clear();
      } else {
         size_t total_words = 0;
         for (int i = 0; i < ns; i++) total_words = std::max<size_t>(total_words, p.h_sout[i].out_word_off + (p.h_sout[i].total_bits + 31) / 32);
         if (ns == 1 && o.host_out) {   /* straight into the caller's buffer */
            if (ob > o.host_out_cap) return -2;
#ifndef ZB_EMU
            if (ob >= ((size_t)8 << 20) && ZbStager::pageable(o.host_out)) { zb_sync(p.st); if (!p.stager.copy(1, p.out.p, o.host_out, ob, p.device)) return -3; }
            else
#endif
            zb_d2h(p.st, o.host_out, p.out.p, ob);
            zb_sync(p.st);
            out.clear();
         } else if (ns == 1) {   /* straight into the result vector */
            out.resize(total_words * 4 + 4);
            zb_d2h(p.st, out.data(), p.out.p, total_words * 4);
            zb_sync(p.st);
            out.resize(ob);
         } else {
            p.hout.need(total_words * 4 + 16);
            if (!p.hout.p || zb_failed()) return -3;
            zb_d2h(p.st, p.hout.p, p.out.p, total_words * 4);
            zb_sync(p.st);
            if (o.want_out_ptr) {   /* the caller copies each stream out of the page-locked buffer itself */
               o.out_ptr = p.hout.p;
               for (int i = 0; i < ns; i++) res[i].out_off = (size_t)p.h_sout[i].out_word_off * 4;
               out.clear();
            } else {
               out.resize(ob);
               for (int i = 0; i < ns; i++)
                  memcpy(out.data() + res[i].out_off, p.hout.p + (size_t)p.h_sout[i].out_word_off * 4, (size_t)((p.h_sout[i].total_bits + 7) / 8));
            }
         }
      }
      o.ms[6] = tm.lap();
   }
   o.ms[7] = tot.lap();
   if (o.dump) {
      ZbDump *dump = o.dump;
      dump->wbase = p.h_wbase;
      dump->sa_lcp.resize(p.P); zb_d2h(p.st, dump->sa_lcp.data(), p.sa_lcp.p, (size_t)p.P * 4);
      if (o.stop_after >= 2) { dump->match.resize((size_t)p.P * 8); zb_d2h(p.st, dump->match.data(), p.match.p, (size_t)p.P * 8 * sizeof(zb_match_t)); }
      if (o.stop_after >= 3) {
         dump->best.resize(p.P); zb_d2h(p.st, dump->best.data(), p.best.p, (size_t)p.P * sizeof(zb_match_t));
         dump->sub.resize(p.nsub); zb_d2h(p.st, dump->sub.data(), p.sub.p, sizeof(ZbSub) * p.nsub);
         dump->tabs.resize(p.nsub); zb_d2h(p.st, dump->tabs.data(), p.tabs.p, sizeof(ZbSubTabs) * p.nsub);
      }
      zb_sync(p.st);
   }
   return 0;
}
/* second half of a sharded call: the entering bit phase is now known */
static inline int zb_finish_shard(ZbPipe &p, uint32_t in_bits, uint8_t *dev_out, size_t dev_out_cap, unsigned long long *total_bits) {
   std::vector<ZbStreamOut> so(1);
   memset(&so[0], 0, sizeof(ZbStreamOut));
   so[0].first_win = 0; so[0].nwin = (uint32_t)p.nwin; so[0].in_bits = in_bits;
   p.stage_emit_finish(so);
   const size_t nb = (size_t)((p.h_sout[0].total_bits + 7) / 8);
   if (nb > dev_out_cap) return -2;
   zb_d2d(p.st, dev_out, p.out.p + p.h_sout[0].out_word_off, nb);
   zb_sync(p.st);
   *total_bits = p.h_sout[0].total_bits;
   return 0;
}
/* second half for several chunks prepared in one call: in_bits[i] = entering phase of chunk i; the bitstreams stay in the
   pipe's output buffer, chunk i at byte offset out_off[i] (word aligned), bits[i] = its bits including the entering ones */
static inline int zb_finish_chunks(ZbPipe &p, const unsigned *in_bits, size_t *out_off, unsigned long long *bits) {
   std::vector<ZbStreamOut> so = p.plan;
   for (size_t i = 0; i < so.size(); i++) so[i].in_bits = in_bits[i];
   p.stage_emit_finish(so);
   zb_sync(p.st);
   if (zb_failed()) return -3;
   for (size_t i = 0; i < so.size(); i++) { out_off[i] = (size_t)p.h_sout[i].out_word_off * 4; bits[i] = p.h_sout[i].total_bits; }
   return 0;
}
#endif
