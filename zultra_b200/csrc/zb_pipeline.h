/*
 * zb_pipeline.h - the batch compression pipeline: suffix array + LCP -> match lists -> block split ->
 * optimal parse -> Huffman tables -> bit emission, for a batch of independent windows.
 *
 * One source, two builds: nvcc (product, every task is a GPU thread) and g++ -DZB_EMU (tests/emu, host
 * loop) - see zb_rt.h.  All state lives in device buffers owned by ZbPipe.
 *
 * Vocabulary (follows the reference): a WINDOW is one max-block plus its <=32 KB history
 * (libzultra.c:287); a SUB-BLOCK is one deflate block produced by the splitter (blockdeflate.c:800);
 * a STREAM is one zlib/gzip/deflate output (one zultra_stream_t).  Windows of one stream are consecutive.
 */
#ifndef ZB_PIPELINE_H
#define ZB_PIPELINE_H
#include "zb_rt.h"
#include <vector>
#include <algorithm>
#ifndef ZB_EMU
#include <cuda_pipeline.h>
#endif

#ifndef ZB_CG
#define ZB_CG 1024        /* positions per greedy-path chunk */
#endif
#ifndef ZB_CP
#define ZB_CP 1024        /* positions per parsed-path chunk */
#endif
#define ZB_CD 2048        /* positions per parse (DP) chunk */
#define ZB_WU 384         /* parse warm-up positions past the chunk end (>= 258; text re-synchronises well within it, the rest is repaired) */
#define ZB_TOKI 256       /* tokens per prefix-histogram interval */
#define ZB_NH 320         /* 288 lit/len + 32 distance counters */
#define ZB_MAXSB 64       /* sub-blocks per window */
#define ZB_MAXNODES 64    /* splitter nodes per window per level (<= 32 used) */
#define ZB_MF_TILE_MAX 16384  /* main positions per match-finder tile: the list of 32768 + 16384 suffixes (4 bytes each) + the rank of every main position (2 bytes) = 224 KB of the 227 KB of shared memory */

struct ZbWinDesc {
   uint32_t in_off;   /* offset of the window's first byte (history start) in the device input */
   uint32_t hist;     /* history bytes in front of the block */
   uint32_t len;      /* hist + block bytes */
   uint32_t stream;   /* stream index */
   uint32_t last;     /* 1 = last window of its stream AND the stream is being finalized */
   uint32_t pad[3];
};

/* splitter node (one recursion frame of blockdeflate.c:634) */
struct ZbNode {
   uint32_t win, depth;
   uint32_t ts, te;          /* token range on the window's greedy path */
   uint32_t ps, pe;          /* position range (window coordinates) */
   uint32_t t0, nchk;        /* token count at the first check point, number of check points */
   uint32_t chk_base;        /* first check record */
   int32_t total_cost;
   int32_t best_delta; uint32_t best_tok;  /* chosen split (token count relative to ts), 0 = none */
   uint32_t pad[4];
};

/* one deflate sub-block */
struct ZbSub {
   uint32_t win, idx_in_win;
   uint32_t ps, pe;          /* position range, window coordinates */
   uint32_t ts, te;          /* greedy token range */
   int32_t is_dyn, static_cost, dynamic_cost;
   uint32_t dchunk_base, ndchunk;   /* parse chunks */
   uint32_t pchunk_base, npchunk;   /* path chunks */
   int32_t mask, nl, no, ncl;       /* RLE mask, HLIT+257, HDIST+1, HCLEN+4 */
   int32_t hdr_bits;                /* bits of the table description (after the 3 block header bits) */
   int32_t body_bits;               /* hdr_bits + token bits + EOB, i.e. what zultra_block_deflate writes */
   int32_t stored;                  /* decided by the stitch scan */
   int32_t final_bit;
   uint64_t bit_off;                /* absolute bit offset of the sub-block's 3 header bits in its stream's output */
   int32_t ub_hit; int32_t pad;
};

struct ZbSubTabs {
   int lcnt[ZB_NLIT], ocnt[ZB_NOFF];
   int llen[ZB_NLIT], olen[ZB_NOFF];
   uint16_t lcode[ZB_NLIT], ocode[ZB_NOFF];
   int cllen[ZB_NCL]; uint16_t clcode[ZB_NCL];
   alignas(16) uint8_t cl[ZB_NLIT + ZB_NOFF]; int mask_cost[20];   /* cl: 16-byte aligned, the mask search copies it with vector loads */
   ZbCostTab cost;
};

struct ZbStreamOut {
   uint64_t out_word_off;   /* first 32-bit word of this stream's output area */
   uint64_t in_bits;        /* bits already pending in the first byte (entering phase 0..7) */
   uint64_t total_bits;     /* result: bits written including in_bits */
   uint32_t first_win, nwin;
   uint32_t err, pad;
};

/* histogram contribution of one greedy token */
ZB_HD void zb_tok_count(const uint8_t *T, uint32_t p, uint32_t len, uint32_t off, int *lc, int *oc, int sign) {
   if (len >= ZB_MIN_MATCH) { lc[zb_len_sym(len - ZB_MIN_MATCH)] += sign; oc[zb_off_sym(off)] += sign; }
   else lc[T[p]] += sign;
}

/* Warm-up of a parse chunk whose candidates read at most `reach` positions past its end: the full warm-up ZB_WU is the
   258-position horizon plus a settling margin; the same margin above `reach` (stage_parse, D2). */
static_assert(ZB_WU > ZB_MAX_MATCH, "the adaptive warm-up needs a settling margin above the 258-position horizon");
ZB_HD int zb_warmup_len(int reach) {
   const int w = reach + (ZB_WU - ZB_MAX_MATCH);
   return w < ZB_WU ? w : ZB_WU;
}

template <class T> struct ZbBuf {
   T *p = 0; size_t cap = 0;
   void need(size_t n) { if (n > cap) { zb_dev_free(p); size_t c = n + n / 8 + 64; p = (T *)zb_dev_alloc(c * sizeof(T)); cap = p ? c : 0; } }
   void release() { zb_dev_free(p); p = 0; cap = 0; }
};

struct ZbHostBuf {   /* grow-only page-locked host buffer */
   uint8_t *p = 0; size_t cap = 0;
   void need(size_t n) { if (n > cap) { zb_host_free(p); size_t c = n + n / 8 + 4096; p = (uint8_t *)zb_host_alloc(c); cap = p ? c : 0; } }
   void release() { zb_host_free(p); p = 0; cap = 0; }
};

#ifndef ZB_EMU
/* Host <-> device copies of PAGEABLE caller memory.  cudaMemcpyAsync on unregistered memory goes through the driver's own
   bounce buffers on the calling thread: ~11 GB/s up and ~4.4 GB/s down on the B200 box, i.e. 9 + 11 ms of a 100 MB one-shot
   call whose device work is 73 ms.  Here the range is cut into 4 lanes, each with its own host thread, CUDA stream and a pair
   of page-locked 4 MiB buffers: memcpy and DMA of consecutive pieces overlap inside a lane, and the lanes' memcpys run side
   by side.  Page-locked (or registered) caller memory is copied directly, as before. */
#include <thread>
struct ZbStager {
   enum { LANES = 4, PIECE = 4 << 20 };
   uint8_t *buf = 0; cudaStream_t st[LANES]; cudaEvent_t ev[LANES][2]; bool ready = false;
   bool init() {
      if (ready) return true;
      if (cudaHostAlloc((void **)&buf, (size_t)LANES * 2 * PIECE, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); buf = 0; return false; }
      for (int l = 0; l < LANES; l++) { cudaStreamCreateWithFlags(&st[l], cudaStreamNonBlocking); cudaEventCreateWithFlags(&ev[l][0], cudaEventDisableTiming); cudaEventCreateWithFlags(&ev[l][1], cudaEventDisableTiming); }
      ready = true;
      return true;
   }
   void release() { if (!ready) return; for (int l = 0; l < LANES; l++) { cudaStreamDestroy(st[l]); cudaEventDestroy(ev[l][0]); cudaEventDestroy(ev[l][1]); } cudaFreeHost(buf); buf = 0; ready = false; }
   static bool pageable(const void *p) {
      cudaPointerAttributes a;
      if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
      return a.type == cudaMemoryTypeUnregistered;
   }
   /* dir 0: host -> device, 1: device -> host.  Synchronous: returns when all bytes have arrived.  Returns false on a CUDA error. */
   bool copy(int dir, void *dev, void *host, size_t n, int device) {
      if (!init()) return false;
      bool ok[LANES];
      auto lane = [&](int l) {
         ok[l] = true;
         if (cudaSetDevice(device) != cudaSuccess) { ok[l] = false; return; }
         const size_t per = ((n + LANES - 1) / LANES + 255) & ~(size_t)255, lo = std::min(n, (size_t)l * per), hi = std::min(n, lo + per);
         uint8_t *b[2] = {buf + (size_t)(2 * l) * PIECE, buf + (size_t)(2 * l + 1) * PIECE};
         size_t pend_off[2] = {0, 0}, pend_len[2] = {0, 0};
         int k = 0;
         for (size_t off = lo; off < hi; off += PIECE, k ^= 1) {
            const size_t len = std::min((size_t)PIECE, hi - off);
            if (dir == 0) {
               if (cudaEventSynchronize(ev[l][k]) != cudaSuccess) ok[l] = false;      /* the DMA that last read this buffer */
               memcpy(b[k], (const uint8_t *)host + off, len);
               if (cudaMemcpyAsync((uint8_t *)dev + off, b[k], len, cudaMemcpyHostToDevice, st[l]) != cudaSuccess) ok[l] = false;
               cudaEventRecord(ev[l][k], st[l]);
            } else {
               if (pend_len[k]) { if (cudaEventSynchronize(ev[l][k]) != cudaSuccess) ok[l] = false; memcpy((uint8_t *)host + pend_off[k], b[k], pend_len[k]); }
               if (cudaMemcpyAsync(b[k], (const uint8_t *)dev + off, len, cudaMemcpyDeviceToHost, st[l]) != cudaSuccess) ok[l] = false;
               cudaEventRecord(ev[l][k], st[l]);
               pend_off[k] = off; pend_len[k] = len;
            }
         }
         if (dir == 1) for (int q = 0; q < 2; q++, k ^= 1) if (pend_len[k]) { if (cudaEventSynchronize(ev[l][k]) != cudaSuccess) ok[l] = false; memcpy((uint8_t *)host + pend_off[k], b[k], pend_len[k]); pend_len[k] = 0; }
         if (cudaStreamSynchronize(st[l]) != cudaSuccess) ok[l] = false;
      };
      std::thread th[LANES - 1];
      for (int l = 1; l < LANES; l++) th[l - 1] = std::thread(lane, l);
      lane(0);
      for (int l = 1; l < LANES; l++) th[l - 1].join();
      for (int l = 0; l < LANES; l++) if (!ok[l]) { cudaGetLastError(); return false; }
      return true;
   }
};
#endif

struct ZbPipe {
   zb_stream_t st;
   ZbHostBuf hin, hout;         /* staging of multi-stream batches */
#ifndef ZB_EMU
   ZbStager stager;             /* pageable caller memory: multi-lane staged copies */
   int device = 0;
#endif
   /* batch description */
   int nwin = 0, nstream = 0;
   uint32_t P = 0;              /* total window positions */
   std::vector<ZbWinDesc> h_win;
   std::vector<uint32_t> h_wbase;
   ZbBuf<ZbWinDesc> win; ZbBuf<uint32_t> wbase;
   ZbBuf<uint8_t> in;           /* device input (owned copy) */
   const uint8_t *in_ptr = 0;   /* input actually used by the stages (in.p or a caller's device buffer) */
   ZbBuf<uint8_t> pk; ZbBuf<uint32_t> asm_tab;   /* shared-history batches: packed input and its stream table (stage_assemble) */
   /* suffix array stage */
   ZbBuf<uint64_t> keyA, keyB; ZbBuf<uint32_t> valA, valB, rank, sa, actA, actB, tmpA, tmpB, scratch;
   ZbBuf<uint32_t> sa_lcp;      /* packed SA|LCP words, rank order, per window at wbase[w] */
   ZbBuf<uint32_t> counters;    /* misc device counters */
   /* match finder */
   ZbBuf<ZbTileDesc> tiles, units, groups; ZbBuf<uint32_t> tile_iv, tile_pd, tile_cnt, tile_q, unit_words, unit_cnt, group_words, group_cnt, filt_seg;
   ZbBuf<zb_match_t> match; ZbBuf<uint16_t> glen, goff;
   /* greedy path */
   ZbBuf<uint16_t> exitoff, exitc; ZbBuf<uint32_t> gentry, gtokcnt, gtokbase, tokpos, wtok; /* wtok[w] = tokens of window w; base in wtokbase */
   ZbBuf<uint32_t> wtokbase, wintbase; ZbBuf<int> ph; /* prefix histograms [interval][ZB_NH] */
   std::vector<uint32_t> h_gchunk_first; ZbBuf<uint32_t> gchunk_first, gchunk_win;
   /* splitter */
   ZbBuf<ZbNode> nodesA, nodesB; ZbBuf<int> nodehist; ZbBuf<uint16_t> chk_stat; ZbBuf<uint8_t> chk_flag; ZbBuf<int> chk_delta; ZbBuf<uint32_t> chk_node;
   ZbBuf<uint32_t> wsplit; ZbBuf<uint32_t> wnsplit, wsubcnt, wsubbase;
   /* sub-blocks */
   ZbBuf<ZbSub> sub; ZbBuf<ZbSubTabs> tabs; ZbBuf<uint32_t> dchunk_sub, pchunk_sub;
   ZbBuf<zb_match_t> best; ZbBuf<int16_t> sig_true, sig_warm, sig_new; ZbBuf<uint8_t> dok; ZbBuf<uint32_t> dbad;
   ZbBuf<uint32_t> pentry, pbits, cand /* 16-byte candidate records, zb_cand_pack */; ZbBuf<uint16_t> dpfar;   /* dpfar: cost rows of the thread-per-chunk parse kernel */
   int cp = ZB_CP;          /* positions per parsed-path chunk of this batch (stage_parse decides: shorter for small batches) */
   ZbBuf<int> dreach;       /* per parse chunk: how far past its end its candidates read (0..258), stage_parse */
   /* output */
   ZbBuf<uint32_t> out; ZbBuf<ZbStreamOut> sout;
   std::vector<ZbStreamOut> h_sout;
   int nsub = 0;
   /* stats */
   bool sa_exact = false;       /* run the suffix sort to the end (stage dumps); see stage_sa */
   int parse_cd = 0;            /* parse chunk (0 = by batch size, see stage_parse) */
   int stat_sa_rounds = 0, stat_redo = 0, stat_ub = 0, stat_tiles = 0;
   double t_stage[8];

   void release_all();
   /* stages */
   void setup(const std::vector<ZbWinDesc> &wins, const uint8_t *h_in, size_t in_bytes, bool in_is_device);
   void stage_assemble(const std::vector<uint32_t> &tab, uint32_t hist_len, size_t in_bytes);
   void stage_sa();
   void stage_match(uint32_t tile_main);
   void stage_greedy();
   void stage_split();
   void stage_parse();
   void stage_emit(const std::vector<ZbStreamOut> &streams) { stage_emit_prepare(); stage_emit_finish(streams); }
   void stage_emit_prepare();                                   /* path, token bits, sub-block sizes: independent of the bit phase */
   void stage_emit_finish(const std::vector<ZbStreamOut> &streams);   /* stitch scan for the entering phase, then emission */
   void phase_maps(const std::vector<ZbStreamOut> &streams, unsigned long long *bits_out);   /* per stream: total bits for each entering phase 0..7 */
   std::vector<ZbStreamOut> plan;   /* streams of a prepared (phase 1) batch, for the emit call that follows */
   /* checksum partials of byte ranges of the device input: kind 1 = Adler-32, 2 = CRC-32 */
   ZbBuf<uint32_t> ck_tab, ck_part; ZbBuf<uint64_t> ck_rng; bool ck_tab_ready = false;
   void stage_checksum(int kind, const std::vector<uint64_t> &range_off, const std::vector<uint64_t> &range_len, std::vector<uint32_t> &sums, uint32_t init_first);
};

/* window lookup for a global position index */
ZB_HD int zb_find_win(const uint32_t *wbase, int nwin, uint32_t g) {
   int lo = 0, hi = nwin - 1;
   while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (wbase[mid] <= g) lo = mid; else hi = mid - 1; }
   return lo;
}

inline void ZbPipe::setup(const std::vector<ZbWinDesc> &wins, const uint8_t *h_in, size_t in_bytes, bool in_is_device) {
   h_win = wins; nwin = (int)wins.size();
   h_wbase.assign(nwin + 1, 0);
   for (int w = 0; w < nwin; w++) h_wbase[w + 1] = h_wbase[w] + wins[w].len;
   P = h_wbase[nwin];
   win.need(nwin); wbase.need(nwin + 1); counters.need(64);
   if (!in_is_device) in.need(in_bytes + 16);
   if (zb_failed()) return;
   zb_h2d(st, win.p, h_win.data(), sizeof(ZbWinDesc) * nwin);
   zb_h2d(st, wbase.p, h_wbase.data(), 4 * (nwin + 1));
   if (in_is_device) in_ptr = h_in;
   else {
      if (h_in) {
#ifndef ZB_EMU
         if (in_bytes >= ((size_t)8 << 20) && ZbStager::pageable(h_in)) { zb_sync(st); if (!stager.copy(0, in.p, (void *)h_in, in_bytes, device)) zb_cuda_fail(cudaErrorUnknown); }
         else
#endif
         zb_h2d(st, in.p, h_in, in_bytes);
      }
      in_ptr = in.p;
   }
}

/* ============================================================ shared-history input assembly ============================================================
 * A batch whose streams all start from the same history (a preset dictionary, zultra_cuda_memory_compress_batch_dict) crosses
 * the bus packed: pk = [history (hl bytes) | payload 0 | payload 1 | ...], the history once.  This pass writes the layout the
 * stages read, [history | payload i] for every stream back to back in `in`, so the history is copied on the device and not on
 * the host or the bus.  tab: {start in `in`, start of the payload in pk} per stream, then {total bytes, packed bytes}.
 * One task per aligned 16 bytes of `in`: a task whose 16 bytes come from one run of pk (all but about two per stream) reads
 * five aligned words, funnel-shifts them and stores one vector; a task across the history/payload seam or a stream end goes
 * byte by byte.  Bytes past the total are written as zero (the buffer has 16 bytes of slack).
 */
inline void ZbPipe::stage_assemble(const std::vector<uint32_t> &h_tab, uint32_t hl, size_t in_bytes) {
   const int ns = (int)h_tab.size() / 2 - 1;
   asm_tab.need(h_tab.size());
   if (zb_failed()) return;
   zb_h2d(st, asm_tab.p, h_tab.data(), h_tab.size() * 4);
   const uint32_t *tab = asm_tab.p; const uint8_t *src = pk.p; uint8_t *dst = in.p; const uint32_t total = (uint32_t)in_bytes;
   zb_tag("batch_assemble");
   zb_launch(st, (long)((in_bytes + 15) / 16), ZB_LAMBDA(long x) {
      const uint32_t b0 = (uint32_t)x * 16u;
      int lo = 0, hi = ns - 1;      /* the stream holding byte b0 */
      while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (tab[2 * mid] <= b0) lo = mid; else hi = mid - 1; }
      const uint32_t r = b0 - tab[2 * lo];
      const uint32_t s0 = r < hl ? r : tab[2 * lo + 1] + (r - hl);
      const uint32_t run = r < hl ? hl - r : tab[2 * lo + 2] - b0;      /* bytes from s0 on that are contiguous in pk */
      uint32_t w[4];
      if (run >= 16) {
         const uint32_t *q = (const uint32_t *)(src + (s0 & ~3u)), sh = (s0 & 3u) * 8u;
         uint32_t v[5];
#pragma unroll
         for (int k = 0; k < 5; k++) v[k] = q[k];
#pragma unroll
         for (int k = 0; k < 4; k++) w[k] = (uint32_t)((((uint64_t)v[k + 1] << 32) | v[k]) >> sh);
      } else {
         w[0] = w[1] = w[2] = w[3] = 0;
         for (uint32_t j = 0, i = (uint32_t)lo; j < 16; j++) {
            const uint32_t b = b0 + j;
            if (b >= total) break;
            while (b >= tab[2 * i + 2]) i++;
            const uint32_t q = b - tab[2 * i];
            w[j >> 2] |= (uint32_t)src[q < hl ? q : tab[2 * i + 1] + (q - hl)] << (8 * (j & 3));
         }
      }
#ifdef __CUDA_ARCH__
      *(uint4 *)(dst + b0) = make_uint4(w[0], w[1], w[2], w[3]);
#else
      memcpy(dst + b0, w, 16);
#endif
   }, 256);
}

/* ============================================================ suffix array + LCP ============================================================
 * Replaces divsufsort_build_array (divsufsort.c:377) and the PLCP/LCP/pack steps of matchfinder.c:57-90.
 * Prefix doubling: sort all suffixes of all windows by (window, first nb bytes), order every tied group of at most
 * ZB_SA_LOCAL suffixes by its next 8 bytes in place (zb_sa_key), then repeatedly sort the still-tied groups by the rank of
 * the suffix h positions further on.  A suffix that runs off its window end is smaller than any longer suffix it is a
 * prefix of (no sentinel; the reference's order, SURVEY A-20).
 */
#define ZB_SA_LOCAL 32    /* tied groups up to this size are ordered by their members' text, each member counting the ones before it */

/* Order key of the suffix at window offset i (window of len bytes, text t) among suffixes that agree on their first d
   bytes, zero-padded past the window end: the next 8 bytes big-endian, zero-padded (w), then min(suffix length, d + 9)
   (tl).  A suffix ending inside the 8 bytes sorts before every longer one it is a prefix of, the shorter first; two
   different suffixes of one window with equal keys both run on past d + 8 bytes and agree on all of them.  d >= 3. */
ZB_HD void zb_sa_key(const uint8_t *t, uint32_t i, uint32_t len, uint32_t d, uint64_t &w, uint32_t &tl) {
   const uint32_t rem = len - i;
   tl = rem < d + 9 ? rem : d + 9;
#ifdef __CUDA_ARCH__
   if ((uint64_t)i + d + 12 <= len) {   /* three aligned words, all inside the window (d >= 3: none starts before the input) */
      const uintptr_t a = (uintptr_t)(t + i + d);
      const uint32_t *pa = (const uint32_t *)(a & ~(uintptr_t)3);
      const uint32_t sh = (uint32_t)(a & 3) << 3;
      const uint32_t x0 = __funnelshift_r(pa[0], pa[1], sh), x1 = __funnelshift_r(pa[1], pa[2], sh);
      w = ((uint64_t)__byte_perm(x0, 0, 0x0123) << 32) | __byte_perm(x1, 0, 0x0123);
      return;
   }
#endif
   uint64_t x = 0;
   for (uint32_t b = 0; b < 8; b++) x = (x << 8) | ((uint64_t)i + d + b < len ? t[i + d + b] : 0u);
   w = x;
}

inline void ZbPipe::stage_sa() {
   const long n = P;
   keyA.need(n); keyB.need(n); valA.need(n); valB.need(n); rank.need(n); sa.need(n); actA.need(n); actB.need(n); tmpA.need(n + 1); tmpB.need(n + 1);
   sa_lcp.need(n);
   scratch.need(zb_sort_scratch_words(n) + zb_scan_scratch_words(n) + 64);
   if (zb_failed()) return;      /* fail fast: no launch ever sees a missing buffer (zb_run_batch reports the error) */
   int wb = 0; while ((1L << wb) < nwin) wb++;
   int nbytes = (64 - wb) / 8; if (nbytes > 7) nbytes = 7;
   const uint8_t *T = in_ptr; const ZbWinDesc *wd = win.p; const uint32_t *wbs = wbase.p; const int nw = nwin;
   uint64_t *kA = keyA.p; uint32_t *vA = valA.p;
   zb_tag("sa_keys");
   zb_launch(st, n, ZB_LAMBDA(long g) {
      int w = zb_find_win(wbs, nw, (uint32_t)g);
      uint32_t i = (uint32_t)g - wbs[w], len = wd[w].len;
      const uint8_t *t = T + wd[w].in_off;
      uint64_t k = 0;
      for (int b = 0; b < nbytes; b++) k = (k << 8) | (i + b < len ? t[i + b] : 0);
      kA[g] = ((uint64_t)w << (8 * nbytes)) | k;
      vA[g] = (uint32_t)g;
   }, 256);
   zb_sort_pairs(st, keyA.p, valA.p, keyB.p, valB.p, n, 0, 8 * nbytes + wb, scratch.p);
   /* initial groups.  Each suffix finds its group [gh, ge) in the sorted keys: a singleton is final; a member of a group of
      at most ZB_SA_LOCAL counts the members whose key (zb_sa_key, 8 more bytes) is smaller, and the equal ones ahead of it,
      which gives its slot and its rank (the slot of its first equal member); members of larger groups stay in place with
      the group's first slot as rank.  head[j] = 1 marks slot j as still tied: all of a large group, members of a small one
      with an equal key.  Every rank is the slot of the first suffix that agrees with it on at least nbytes bytes. */
   uint32_t *head = tmpA.p, *grp = tmpB.p, *rk = rank.p, *SA = sa.p, *act = actA.p, *act2 = actB.p, *cnt = counters.p;
   const int kbits = 8 * nbytes;
   zb_tag("sa_group");
   zb_launch(st, n, ZB_LAMBDA(long jl) {
      const uint32_t j = (uint32_t)jl;
      const uint64_t key = kA[j];
      /* first member: gallop back, then bisect (lo < gh: kA[lo] differs or lo = -1) */
      uint32_t gh = j, step = 1;
      while (gh >= step && kA[gh - step] == key) { gh -= step; step <<= 1; }
      long lo = gh >= step ? (long)(gh - step) : -1L;
      while ((long)gh - lo > 1) { const uint32_t mid = (uint32_t)((lo + (long)gh) >> 1); if (kA[mid] == key) gh = mid; else lo = mid; }
      const uint32_t g = vA[j];
      if ((long)gh + ZB_SA_LOCAL < n && kA[gh + ZB_SA_LOCAL] == key) { SA[j] = g; rk[g] = gh; head[j] = 1u; return; }
      uint32_t ge = j + 1;
      while ((long)ge < n && kA[ge] == key) ge++;
      if (ge - gh == 1) { SA[j] = g; rk[g] = j; head[j] = 0u; return; }
      const int w = (int)(key >> kbits);
      const uint32_t base = wbs[w], len = wd[w].len;
      const uint8_t *t = T + wd[w].in_off;
      uint64_t kw; uint32_t kt;
      zb_sa_key(t, g - base, len, (uint32_t)nbytes, kw, kt);
      uint32_t less = 0, eq_before = 0, eq = 0;
      for (uint32_t y = gh; y < ge; y++) {
         if (y == j) continue;
         uint64_t yw; uint32_t yt;
         zb_sa_key(t, vA[y] - base, len, (uint32_t)nbytes, yw, yt);
         if (yw < kw || (yw == kw && yt < kt)) less++;
         else if (yw == kw && yt == kt) { eq++; if (y < j) eq_before++; }
      }
      const uint32_t p = gh + less + eq_before;
      SA[p] = g; rk[g] = gh + less; head[p] = eq ? 1u : 0u;
   }, 256);
   zb_exclusive_sum(st, head, grp, n, cnt, scratch.p);
   zb_launch(st, n, ZB_LAMBDA(long j) { if (head[j]) act[grp[j]] = (uint32_t)j; }, 256);
   uint32_t m = 0;
   zb_d2h(st, &m, cnt, 4); zb_sync(st);
   int rank_bits = 1; while ((1L << rank_bits) < n) rank_bits++;
   uint64_t *kB = keyB.p; uint32_t *vB = valB.p;
   stat_sa_rounds = 0;
   uint32_t maxwin = 0;
   for (int w = 0; w < nwin; w++) maxwin = std::max(maxwin, h_win[w].len);
   int r2_bits = 1; while ((1L << r2_bits) < (long)maxwin + 512) r2_bits++;
   const bool packed_keys = !sa_exact;      /* the exact sort doubles h past 512 and keeps the flag-bit form below */
   /* Rounds needed: all of them for the exact suffix array (the SA|LCP parity artefact, zultra_cuda_window_sa_lcp); for
      compression only until every suffix is ordered by its first 258 bytes - the match lists depend on the order only through
      min(lcp, 258) (matchfinder.c:85-88), how suffixes that agree on 258 bytes or more are ordered among themselves changes no
      clamped LCP and no record.  A 64 KiB byte run needs 14 rounds for its exact order and 6 for this. */
   for (uint32_t h = (uint32_t)nbytes; m > 0 && (sa_exact || h < ZB_MAX_MATCH); h <<= 1) {
      stat_sa_rounds++;
      const long mm = m;
      /* key = (current rank, rank of the suffix h further; suffixes running off the window sort first, shorter first) */
      zb_tag("sa_round_keys");
      if (packed_keys) {
         /* compression mode (h <= 258 < 512): a suffix running off its window gets wend - g (1..h), one inside rank + 512, so the
            second key fits r2_bits and the pair is ONE contiguous key: 6 radix passes for 100 MB instead of 3 + 4 */
         zb_launch(st, mm, ZB_LAMBDA(long a) {
            uint32_t j = act[a], g = SA[j];
            int w = zb_find_win(wbs, nw, g);
            uint32_t wend = wbs[w + 1];
            uint32_t r2;
            if ((uint64_t)g + h < wend) r2 = (rk[g + h] - wbs[w]) + 512u;
            else r2 = wend - g;
            kA[a] = ((uint64_t)rk[g] << r2_bits) | r2;
            vA[a] = g;
         }, 256);
         zb_sort_pairs(st, keyA.p, valA.p, keyB.p, valB.p, mm, 0, r2_bits + rank_bits, scratch.p);
      } else {
      zb_launch(st, mm, ZB_LAMBDA(long a) {
         uint32_t j = act[a], g = SA[j];
         int w = zb_find_win(wbs, nw, g);
         uint32_t wend = wbs[w + 1];
         uint32_t r2;
         if ((uint64_t)g + h < wend) r2 = (rk[g + h] - wbs[w]) + (1u << 22);
         else r2 = wend - g;
         kA[a] = ((uint64_t)rk[g] << 32) | r2;
         vA[a] = g;
      }, 256);
      zb_sort_pairs(st, keyA.p, valA.p, keyB.p, valB.p, mm, 0, 23, scratch.p);
      zb_sort_pairs(st, keyA.p, valA.p, keyB.p, valB.p, mm, 32, 32 + rank_bits, scratch.p);
      }
      zb_launch(st, mm, ZB_LAMBDA(long a) { head[a] = (a == 0 || kA[a] != kA[a - 1]) ? (uint32_t)a : 0u; SA[act[a]] = vA[a]; }, 256);
      zb_inclusive_max(st, head, grp, mm, scratch.p);
      zb_launch(st, mm, ZB_LAMBDA(long a) {
         const uint32_t ga = grp[a];
         rk[vA[a]] = act[ga];
         bool is_head = ga == (uint32_t)a;
         bool next_head = (a + 1 == mm) || grp[a + 1] == (uint32_t)(a + 1);
         head[a] = (is_head && next_head) ? 0u : 1u;
      }, 256);
      zb_exclusive_sum(st, head, (uint32_t *)kB, mm, cnt, scratch.p);
      {
         const uint32_t *dst = (const uint32_t *)kB;
         zb_launch(st, mm, ZB_LAMBDA(long a) { if (head[a]) act2[dst[a]] = act[a]; }, 256);
      }
      zb_d2h(st, &m, cnt, 4); zb_sync(st);
      std::swap(act, act2);
      (void)vB;
      if (h > (1u << 23)) break; /* cannot happen: windows are < 2^22 */
   }
   /* LCP with the previous suffix of the same window, clamped as matchfinder.c:81-90, packed pos | lcp << 22 */
   uint32_t *out = sa_lcp.p;
   zb_tag("lcp_pack");
   zb_launch(st, n, ZB_LAMBDA(long j) {
      uint32_t g = SA[j];
      int w = zb_find_win(wbs, nw, (uint32_t)j);
      uint32_t base = wbs[w], len = wd[w].len;
      uint32_t i = g - base;
      uint32_t l = 0;
      if ((uint32_t)j != base) {
         uint32_t q = SA[j - 1] - base;
         const uint8_t *t = T + wd[w].in_off;
         uint32_t lim = len - (i > q ? i : q);
         if (lim > ZB_MAX_MATCH) lim = ZB_MAX_MATCH;
#ifdef __CUDA_ARCH__
         /* four bytes per step out of aligned words (two loads a side): every step is a dependent round trip to L2, so
            fewer, wider steps.  Only while both 8-byte spans lie inside the input (the first 3 bytes of the buffer and the
            tail of the window go bytewise). */
         if (wd[w].in_off + (i < q ? i : q) >= 4) {
            while (l + 8 <= lim) {
               const uintptr_t a = (uintptr_t)(t + i + l), b = (uintptr_t)(t + q + l);
               const uint32_t *pa = (const uint32_t *)(a & ~(uintptr_t)3), *pb = (const uint32_t *)(b & ~(uintptr_t)3);
               const uint32_t x = __funnelshift_r(pa[0], pa[1], (uint32_t)(a & 3) << 3) ^ __funnelshift_r(pb[0], pb[1], (uint32_t)(b & 3) << 3);
               if (x) { l += (uint32_t)(__ffs((int)x) - 1) >> 3; lim = l; break; }
               l += 4;
            }
         }
#endif
         while (l < lim && t[i + l] == t[q + l]) l++;
         if (l < ZB_MIN_MATCH) l = 0;
      }
      out[j] = i | (l << ZB_POS_BITS);
   }, 256);
}

/* ============================================================ match finder ============================================================ */
#ifndef ZB_EMU
/* Match lists, kernel A.  CTA per tile: the tile's suffix list (<= 32768 + T words) and the rank of every main position live
   in shared memory.  Walk lengths are heavy-tailed, so lanes do not own fixed positions: a lane that finishes fetches the next
   main position from a shared counter and all 32 lanes keep stepping (same arithmetic as the rank walk of zb_mf_scan, kept
   as a resumable state).  Records go straight to global memory as they are found.  A position whose walk reaches the
   text-walk condition is handed to kernel B through a per-tile queue in global memory: three words
   {m | nm << 14 | moved << 18 | lvl << 19, bound | (i - 1 - best) << 9, first record}. */
#define ZB_MF_THREADS 1024
__global__ void __launch_bounds__(ZB_MF_THREADS) zb_mf_scan_k(const ZbTileDesc *td, int first, const uint32_t *unit_words, const uint32_t *unit_cnt, uint32_t *queues, size_t qstride,
                                                              size_t stride, uint32_t *qcnt, zb_match_t *mt, uint16_t *gl, uint16_t *go, const uint32_t *wbs, uint32_t tile_main,
                                                              int ts_min, int ts_mul) {
   extern __shared__ __align__(16) uint32_t zb_smw[];
   __shared__ uint32_t next_m, nq, wcnt[32], wtail[32];
   const int k = blockIdx.x;
   const ZbTileDesc t = td[first + k];
   const uint32_t nlook = t.m0 - t.lo, nmain = t.hi - t.m0;
   uint32_t *words = zb_smw + 1;          /* words[-1] and words[n] are LCP-0 sentinels: no bounds tests in the walk */
   uint16_t *rom = (uint16_t *)(zb_smw + stride + 2);
   uint32_t *queue = queues + (size_t)k * qstride;
   /* The tile's suffix list is filtered out of its unit's list while it is loaded (the last filter level, fused): rank order
      kept, the LCP min-reduced over the skipped entries.  1024 entries per step: ballot compaction and a segmented shuffle
      min-scan inside each warp, counts and trailing minima of the 32 warps combined through shared memory. */
   int n = 0;
   {
      const uint32_t *src = unit_words + t.src_base;
      const uint32_t nsrc = unit_cnt[t.src_cnt_idx];
      const uint32_t lo_rel = t.lo - t.src_lo, span = t.hi - t.lo;
      const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
      const uint32_t lt = (1u << lane) - 1u;
      uint32_t count = 0, carry = 0x1ffu;
      /* 4 x 1024 entries are in flight per thread group: the loads of the next group are issued before this one is processed */
      uint32_t wn[4];
#pragma unroll
      for (int j = 0; j < 4; j++) { const uint32_t r = (uint32_t)j * ZB_MF_THREADS + threadIdx.x; wn[j] = r < nsrc ? __ldg(src + r) : 0u; }
      for (uint32_t g0 = 0; g0 < nsrc; g0 += 4 * ZB_MF_THREADS) {
      uint32_t wc[4];
#pragma unroll
      for (int j = 0; j < 4; j++) { wc[j] = wn[j]; const uint32_t r = g0 + (uint32_t)(4 + j) * ZB_MF_THREADS + threadIdx.x; wn[j] = r < nsrc ? __ldg(src + r) : 0u; }
#pragma unroll
      for (int j = 0; j < 4; j++) {
         const uint32_t r0 = g0 + (uint32_t)j * ZB_MF_THREADS;
         if (r0 >= nsrc) break;
         const uint32_t r = r0 + threadIdx.x;
         const bool valid = r < nsrc;
         const uint32_t w = wc[j];
         const uint32_t pos = (w & ZB_POS_MASK) - lo_rel;
         uint32_t v = valid ? ((w >> ZB_POS_BITS) & 0x1ffu) : 0x1ffu;
         const bool keep = valid && pos < span;
         const uint32_t kmask = __ballot_sync(0xffffffffu, keep);
         const uint32_t below = kmask & lt;
         const int start = below ? (32 - __clz((int)below)) : 0;
#pragma unroll
         for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, v, d);
            if (lane >= start + d) v = min(v, o);
         }
         const uint32_t v31 = __shfl_sync(0xffffffffu, v, 31);
         if (lane == 0) { wcnt[warp] = __popc(kmask); wtail[warp] = ((kmask >> 31) ? 0x1ffu : v31) | (kmask ? 0x10000u : 0u); }
         __syncthreads();
         /* every warp: exclusive count of the warps before it, the minimum carried into it, and the step's totals */
         const uint32_t cx = wcnt[lane], tx = wtail[lane];
         uint32_t inc = cx;
#pragma unroll
         for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
         const uint32_t prefix = __shfl_sync(0xffffffffu, inc - cx, warp), total = __shfl_sync(0xffffffffu, inc, 31);
         const uint32_t hasmask = __ballot_sync(0xffffffffu, (tx >> 16) & 1u);
         const uint32_t hb = hasmask & ((1u << warp) - 1u);
         const int lo_u = hb ? 31 - __clz((int)hb) : 0;
         uint32_t cin = __reduce_min_sync(0xffffffffu, (lane >= lo_u && lane < warp) ? (tx & 0xffffu) : 0x1ffu);
         if (!hb) cin = min(cin, carry);
         const int lo_2 = hasmask ? 31 - __clz((int)hasmask) : 0;
         uint32_t cnew = __reduce_min_sync(0xffffffffu, lane >= lo_2 ? (tx & 0xffffu) : 0x1ffu);
         if (!hasmask) cnew = min(cnew, carry);
         if (start == 0) v = min(v, cin);
         if (keep) {
            const uint32_t at = count + prefix + __popc(below);
            words[at] = pos | (v << ZB_POS_BITS);
            if (pos >= nlook) rom[pos - nlook] = (uint16_t)at;
         }
         count += total; carry = cnew;
         __syncthreads();
      }
      }
      n = (int)count;
   }
   if (threadIdx.x == 0) { next_m = 0; nq = 0; zb_smw[0] = 0; words[n] = 0; }
   __syncthreads();
   const uint32_t gbase = wbs[t.win];
   const int lane = threadIdx.x & 31;
   bool busy = false, drained = false, moved = false;
   uint32_t m = 0, lL = 0, lR = 0, lvl = 0, maxlen = 0, rec0 = 0, rec1 = 0;
   int i = 0, L = 0, R = 0, best = -1, nm = 0, steps = 0, gap = 0, thr = 0;
   uint32_t *dst = 0;
   /* the first two records of a position stay in registers (most positions have no more) and leave with one 8-byte store when
      the walk ends; further records go straight to their slot */
#define ZB_MF_EMIT(v_) do { uint32_t v__ = (v_); if ((v__ & 0xffffu) > maxlen) v__ = (v__ & 0xffff0000u) | maxlen; \
      if (nm == 0) rec0 = v__; else if (nm == 1) rec1 = v__; else dst[nm] = v__; nm++; } while (0)
   /* the rank walk hands over to the text walk (kernel B) once steps >= ts_min and gap = i - 1 - best <= ts_mul * steps; the
      product is kept as a running sum (thr), the gap changes only when `best` moves */
   for (;;) {
      {  /* positions are handed out warp by warp: one shared-memory atomic for all lanes that need one */
         const uint32_t need = __ballot_sync(0xffffffffu, !busy && !drained);
         if (need) {
            uint32_t base = 0;
            if (lane == __ffs((int)need) - 1) base = atomicAdd(&next_m, (uint32_t)__popc(need));
            base = __shfl_sync(0xffffffffu, base, __ffs((int)need) - 1);
            if (!busy && !drained) {
               m = base + (uint32_t)__popc(need & ((1u << lane) - 1u));
               if (m >= nmain) drained = true;
               else {
                  busy = true;
                  const int r = (int)rom[m];
                  i = (int)(nlook + m);
                  L = r - 1; R = r + 1;
                  lL = words[r] >> ZB_POS_BITS;     /* words[0] has LCP 0 */
                  lR = words[R] >> ZB_POS_BITS;     /* words[n] = 0 */
                  best = (i > ZB_MAX_OFFSET ? i - ZB_MAX_OFFSET : 0) - 1;   /* p > best also enforces the 32768 limit */
                  nm = 0; lvl = 0; moved = false; steps = 0; rec0 = 0; rec1 = 0;
                  gap = i - 1 - best; thr = 0;
                  maxlen = t.wlen - (t.m0 + m);     /* matchfinder.c:276-280 (LAST_LITERALS = 0) */
                  dst = (uint32_t *)(mt + ((size_t)(gbase + t.m0 + m) << 3));
               }
            }
         }
      }
      if (__all_sync(0xffffffffu, !busy)) break;      /* every lane is drained */
      bool fin = false;
      if (busy) {
#pragma unroll 1
         for (int step = 0; step < 8; step++) {
            const uint32_t l = lL > lR ? lL : lR;
            if (l < lvl && moved) {
               ZB_MF_EMIT(lvl | ((uint32_t)(i - best) << 16));
               moved = false;
               if (nm == ZB_NMATCH) { fin = true; break; }
            }
            if (l < ZB_MIN_MATCH) { fin = true; break; }
            if (steps >= ts_min && gap <= thr) {   /* the rest is cheaper read from the text: kernel B */
               const uint32_t at = atomicAdd(&nq, 1u);
               if (nm == 1) dst[0] = rec0; else if (nm >= 2) *(uint2 *)dst = make_uint2(rec0, rec1);      /* kernel B fills the slots from nm on */
               queue[3 * at] = m | ((uint32_t)nm << 14) | ((moved ? 1u : 0u) << 18) | (lvl << 19);
               queue[3 * at + 1] = l | ((uint32_t)(i - 1 - best) << 9);
               queue[3 * at + 2] = rec0;
               busy = false;
               break;
            }
            lvl = l; steps++; thr += ts_mul;
            /* one step to the side with the larger running LCP, without a branch (the two sides would split the warp): the
               left side's new LCP is in the word it consumes, the right side's in the word after it (never read past the
               list: with R at the end sentinel lR is 0 and the left side is taken) */
            /* equal running LCPs (both clamped at 258 inside a long byte run or periodic stretch): alternate, so that the side
               holding the EARLIER positions is reached at once - always preferring one side walked thousands of later
               positions of the run before the text-walk hand-over (45 % of all rank steps on the mozilla-shaped config) */
            const bool goL = lL > lR || (lL == lR && (steps & 1));
            const int at = goL ? L : R;
            const uint32_t w = words[at], w2 = words[at + 1];
            const uint32_t wl = (goL ? w : w2) >> ZB_POS_BITS;
            L -= goL ? 1 : 0; R += goL ? 0 : 1;
            const uint32_t side = goL ? lL : lR;
            const uint32_t nl = wl < side ? wl : side;
            lL = goL ? nl : lL; lR = goL ? lR : nl;
            const int p = (int)(w & ZB_POS_MASK);
            if (p < i && p > best) {
               best = p; moved = true;
               if (best == i - 1) { ZB_MF_EMIT(lvl | (1u << 16)); fin = true; break; }
               gap = i - 1 - best;
            }
         }
      }
      if (fin) {
         /* slots 0 and 1 from the registers, the unused ones zeroed (matchfinder.c:271-274) */
         *(uint2 *)dst = make_uint2(rec0, nm >= 2 ? rec1 : 0u);
         if (nm <= 2) { *(uint2 *)(dst + 2) = make_uint2(0u, 0u); *(uint4 *)(dst + 4) = make_uint4(0u, 0u, 0u, 0u); }
         else for (int z = nm; z < ZB_NMATCH; z++) dst[z] = 0u;
         const uint32_t p = t.m0 + m;
         const uint32_t l0 = rec0 & 0xffffu;
         gl[gbase + p] = l0 >= ZB_MIN_MATCH ? (uint16_t)l0 : (uint16_t)1;
         go[gbase + p] = l0 >= ZB_MIN_MATCH ? (uint16_t)(rec0 >> 16) : (uint16_t)0;
         busy = false;
      }
   }
#undef ZB_MF_EMIT
   __syncthreads();
   if (threadIdx.x == 0) qcnt[k] = nq;
}

/* Match lists, kernel B: the text walk of zb_mf_scan for the positions kernel A queued, one WARP per position.  The tile's
   text is in shared memory; the 32 lanes test 32 positions j of (best, i) per step for the 3-byte prefix, candidates are
   compared 32 bytes at a time, nearest first.  Control flow is warp-uniform. */
#define ZB_MT_THREADS 512      /* at most; 256 for tiles of <= 8192 main positions */
__global__ void __launch_bounds__(ZB_MT_THREADS) zb_mf_text_k(const ZbTileDesc *td, int first, const uint32_t *lists, size_t stride, const uint32_t *qcnt,
                                                              zb_match_t *mt, uint16_t *gl, uint16_t *go, const uint32_t *wbs, const ZbWinDesc *wd, const uint8_t *T) {
   extern __shared__ __align__(16) uint32_t zb_smw[];
   __shared__ uint32_t next_q;
   __shared__ __align__(8) uint64_t txt_bar;
   const int k = blockIdx.x;
   const uint32_t nq = qcnt[k];
   if (nq == 0) return;
   const ZbTileDesc t = td[first + k];
   const uint32_t nlook = t.m0 - t.lo;
   const uint32_t *queue = lists + (size_t)k * stride;
   /* The tile's text comes in as ONE bulk copy (TMA, cp.async.bulk): global -> shared without passing through registers, one
      thread issues it and an mbarrier counts the bytes in.  Source, destination and size of a bulk copy are multiples of 16, so
      the shared copy sits at the same offset modulo 16 as the source (`delta`), the whole 16-byte pieces go by TMA and the
      ragged head and tail (< 16 bytes each) bytewise.  All text indices below carry `delta`. */
   const uint8_t *tsrc = T + wd[t.win].in_off + t.lo;
   const uint32_t delta = (uint32_t)((uintptr_t)tsrc & 15u);
   uint8_t *txt = (uint8_t *)zb_smw;            /* txt[delta + x] = window byte t.lo + x */
   {
      uint32_t ntxt = t.hi - t.lo + ZB_MAX_MATCH;
      if (ntxt > t.wlen - t.lo) ntxt = t.wlen - t.lo;
      uint32_t head = (16u - delta) & 15u; if (head > ntxt) head = ntxt;
      const uint32_t bulk = (ntxt - head) & ~15u;
      const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&txt_bar);
      if (threadIdx.x == 0) {
         asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar));
         asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      /* the async proxy sees the initialised barrier */
         if (bulk) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bulk) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"((uint32_t)__cvta_generic_to_shared(txt + delta + head)), "l"(tsrc + head), "r"(bulk), "r"(bar) : "memory");
         }
      }
      for (uint32_t e = threadIdx.x; e < head; e += blockDim.x) txt[delta + e] = tsrc[e];
      for (uint32_t e = head + bulk + threadIdx.x; e < ntxt; e += blockDim.x) txt[delta + e] = tsrc[e];
      __syncthreads();      /* the barrier's initialisation is visible to every thread before any of them polls it */
      if (bulk) {
         uint32_t ok = 0;
         while (!ok) asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(bar) : "memory");
      }
   }
   if (threadIdx.x == 0) next_q = 0;
   __syncthreads();
   const uint32_t gbase = wbs[t.win];
   const int lane = threadIdx.x & 31;
   /* tasks are taken 32 at a time: one atomic and one coalesced load of the 32 records per batch, the three words of each
      task then come out of the lanes' registers by shuffle (a fetch per task was a sixth of this kernel's instructions) */
   for (;;) {
      uint32_t e0 = 0;
      if (lane == 0) e0 = atomicAdd(&next_q, 32u);
      e0 = __shfl_sync(0xffffffffu, e0, 0);
      if (e0 >= nq) break;
      const uint32_t nhere = nq - e0 < 32u ? nq - e0 : 32u;
      uint32_t r0 = 0, r1 = 0, r2 = 0;
      if ((uint32_t)lane < nhere) { const uint32_t *qe = queue + 3 * (size_t)(e0 + lane); r0 = __ldg(qe); r1 = __ldg(qe + 1); r2 = __ldg(qe + 2); }
      for (uint32_t tix = 0; tix < nhere; tix++) {
      const uint32_t c0 = __shfl_sync(0xffffffffu, r0, (int)tix), c1 = __shfl_sync(0xffffffffu, r1, (int)tix), c2 = __shfl_sync(0xffffffffu, r2, (int)tix);
      const uint32_t m = c0 & 0x3fffu, lvl = c0 >> 19, bound = c1 & 0x1ffu;
      const int nm = (int)((c0 >> 14) & 15u);
      const bool moved = (c0 >> 18) & 1u;
      const int i = (int)(nlook + m + delta);
      const int best = i - 1 - (int)(c1 >> 9);
      const uint32_t k3 = (uint32_t)txt[i] | ((uint32_t)txt[i + 1] << 8) | ((uint32_t)txt[i + 2] << 16);
      /* record number d (in order of discovery = increasing length) is kept by lane d % 32; only the last 8 can survive */
      uint32_t myrec = 0, curmax = 0;
      int nd = 0;
      bool done = false;
      /* one candidate jh (nearest first): its match length against i, 32 bytes per ballot, kept when strictly longer */
#define ZB_MT_TRY(jh_)                                                                                              \
      {                                                                                                             \
         const int jh = (jh_);                                                                                      \
         uint32_t len = bound;                                                                                      \
         for (uint32_t o = ZB_MIN_MATCH; o < bound; o += 32) {                                                      \
            const uint32_t xo = o + (uint32_t)lane;                                                                 \
            const bool neq = xo < bound && txt[jh + xo] != txt[i + xo];                                             \
            const uint32_t mm = __ballot_sync(0xffffffffu, neq);                                                    \
            if (mm) { len = o + (uint32_t)(__ffs((int)mm) - 1); break; }                                            \
         }                                                                                                          \
         if (len > curmax) {                                                                                        \
            if (lane == (nd & 31)) myrec = len | ((uint32_t)(i - jh) << 16);                                        \
            nd++;                                                                                                   \
            curmax = len;                                                                                           \
            if (len == bound) done = true;                                                                          \
         }                                                                                                          \
      }
      if (i - 1 - best <= 64) {
         /* short interval (batches of small streams: most of them): one position per lane and step */
         for (int jb = i - 1; jb > best && !done; jb -= 32) {
            const int j = jb - lane;
            bool hit = false;
            if (j > best) {   /* bytes j..j+2 out of the two aligned words around them (the buffer is padded by a word) */
               const uint32_t w0 = zb_smw[j >> 2], w1 = zb_smw[(j >> 2) + 1];
               hit = (__funnelshift_r(w0, w1, (uint32_t)(j & 3) << 3) & 0xffffffu) == k3;
            }
            uint32_t hits = __ballot_sync(0xffffffffu, hit);
            while (hits && !done) {
               const int h = __ffs((int)hits) - 1;
               hits &= hits - 1u;
               ZB_MT_TRY(jb - h)
            }
         }
      } else {
      /* 128 positions per step: lane L tests the four positions q + 3 .. q (q = jb - 4 L - 3, a multiple of 4) out of the two
         aligned words at q; bit s of its nibble = position jb - 4 L - s hit.  Hits are then taken nearest first: lanes in order,
         bits of a lane's nibble in order.  The first step starts at the aligned group holding i - 1; positions >= i and <= best
         are masked out. */
      for (int jb = (i - 1) | 3; jb > best && !done; jb -= 128) {
         const int q = jb - 4 * lane - 3;
         uint32_t nib = 0;
         if (q + 3 > best) {
            const uint32_t w0 = zb_smw[q >> 2], w1 = zb_smw[(q >> 2) + 1];
            nib = ((((__funnelshift_r(w0, w1, 24) ^ k3) & 0xffffffu) == 0u) ? 1u : 0u) | ((((__funnelshift_r(w0, w1, 16) ^ k3) & 0xffffffu) == 0u) ? 2u : 0u) |
                  ((((w0 >> 8) ^ k3) == 0u) ? 4u : 0u) | ((((w0 ^ k3) & 0xffffffu) == 0u) ? 8u : 0u);
            const int hi_s = q + 3 - best;       /* s < hi_s: position above best */
            if (hi_s < 4) nib &= (1u << hi_s) - 1u;
            const int lo_s = q + 4 - i;          /* s >= lo_s: position below i (first step only; at most 3) */
            if (lo_s > 0) nib &= ~((1u << lo_s) - 1u);
         }
         uint32_t any = __ballot_sync(0xffffffffu, nib != 0u);
         while (any && !done) {
            const int hl = __ffs((int)any) - 1;
            any &= any - 1u;
            uint32_t nb = __shfl_sync(0xffffffffu, nib, hl);
            while (nb && !done) {
               const int sb = __ffs((int)nb) - 1;
               nb &= nb - 1u;
               ZB_MT_TRY(jb - 4 * hl - sb)
            }
         }
      }
      }
#undef ZB_MT_TRY
      /* slots nm.. of the record: [pending record of the rank walk, unless a nearer position reached the same level] then
         the text-walk records, longest first; lane z writes slot z */
      const uint32_t p = t.m0 + m;
      const uint32_t maxlen = t.wlen - p;
      const int nt = nd < ZB_NMATCH ? nd : ZB_NMATCH;
      const bool pend = moved && !(nt && curmax == lvl);
      const int z = lane - nm - (pend ? 1 : 0);      /* this lane's slot takes the z-th longest text-walk record: discovery nd - 1 - z */
      const uint32_t got = __shfl_sync(0xffffffffu, myrec, (nd - 1 - z) & 31);
      uint32_t v = 0;
      if (pend && lane == nm) v = lvl | (((c1 >> 9) + 1u) << 16);
      if (z >= 0 && z < nt) v = got;
      if ((v & 0xffffu) > maxlen) v = (v & 0xffff0000u) | maxlen;
      uint32_t *dst = (uint32_t *)(mt + ((size_t)(gbase + p) << 3));
      if (lane >= nm && lane < ZB_NMATCH) dst[lane] = v;
      const uint32_t first_rec = nm ? c2 : __shfl_sync(0xffffffffu, v, 0);
      if (lane == 0) {
         const uint32_t l0 = first_rec & 0xffffu;
         gl[gbase + p] = l0 >= ZB_MIN_MATCH ? (uint16_t)l0 : (uint16_t)1;
         go[gbase + p] = l0 >= ZB_MIN_MATCH ? (uint16_t)(first_rec >> 16) : (uint16_t)0;
      }
      }
   }
}
#endif

inline void ZbPipe::stage_match(uint32_t tile_main) {
   /* Filter levels, each cutting the list of the level above down to a position range (rank order kept, LCPs min-reduced):
      [groups of 8 units, only for windows of more than 4 units ->] units: 32768 main positions + the 32768 before them ->
      tiles: tile_main main positions (a divisor of 32768) + look-back.  The group level keeps the total streamed volume near
      7 words per window position instead of 33. */
   if (tile_main > ZB_MF_TILE_MAX) tile_main = ZB_MF_TILE_MAX;
   while (ZB_MAX_OFFSET % tile_main) tile_main >>= 1;
   {  /* batches of small streams (windows of a few tiles at most): the larger tile only costs occupancy there */
      uint32_t mx = 0;
      for (int w = 0; w < nwin; w++) mx = std::max(mx, h_win[w].len);
      if (mx <= 4 * ZB_MAX_OFFSET && tile_main > 8192) tile_main = 8192;
   }
   const uint32_t GU = 8, gspan = GU * ZB_MAX_OFFSET;
   uint32_t maxlen = 0;
   for (int w = 0; w < nwin; w++) maxlen = std::max(maxlen, h_win[w].len);
   const bool use_groups = maxlen > 4 * ZB_MAX_OFFSET;
   const size_t gstride = (size_t)(GU + 1) * ZB_MAX_OFFSET;
   std::vector<ZbTileDesc> hg, hu, ht;
   for (int w = 0; w < nwin; w++) {
      const ZbWinDesc &d = h_win[w];
      for (uint32_t u0 = d.hist; u0 < d.len; u0 += ZB_MAX_OFFSET) {
         ZbTileDesc u; memset(&u, 0, sizeof(u));
         u.win = (uint32_t)w; u.m0 = u0; u.hi = std::min(d.len, u0 + ZB_MAX_OFFSET);
         u.lo = u0 > ZB_MAX_OFFSET ? u0 - ZB_MAX_OFFSET : 0;
         u.src_base = h_wbase[w]; u.src_n = d.len; u.src_lo = 0; u.src_cnt_idx = -1; u.wlen = d.len;
         if (use_groups) {
            if ((u0 - d.hist) % gspan == 0) {
               ZbTileDesc g = u;
               g.hi = std::min(d.len, u0 + gspan);
               hg.push_back(g);
            }
            const int gi = (int)hg.size() - 1;
            u.src_base = (uint64_t)gi * gstride; u.src_n = 0; u.src_lo = hg[gi].lo; u.src_cnt_idx = gi;
         }
         const int ui = (int)hu.size();
         hu.push_back(u);
         for (uint32_t m0 = u0; m0 < u.hi; m0 += tile_main) {
            ZbTileDesc t; memset(&t, 0, sizeof(t));
            t.win = (uint32_t)w; t.m0 = m0; t.hi = std::min(u.hi, m0 + tile_main);
            t.lo = m0 > ZB_MAX_OFFSET ? m0 - ZB_MAX_OFFSET : 0;
            t.src_base = (uint64_t)ui * (2 * ZB_MAX_OFFSET); t.src_n = 0; t.src_lo = u.lo; t.src_cnt_idx = ui; t.wlen = d.len;
            ht.push_back(t);
         }
      }
   }
   const int ngroup = (int)hg.size(), nunit = (int)hu.size(), ntile = (int)ht.size();
   units.need(nunit); tiles.need(ntile);
   zb_h2d(st, units.p, hu.data(), sizeof(ZbTileDesc) * nunit);
   zb_h2d(st, tiles.p, ht.data(), sizeof(ZbTileDesc) * ntile);
   match.need((size_t)P * ZB_NMATCH); glen.need(P); goff.need(P);
   if (zb_failed()) return;
   unit_words.need((size_t)nunit * (2 * ZB_MAX_OFFSET)); unit_cnt.need(nunit);
   auto segs_for = [](size_t n) { size_t k = (n + 8191) / 8192; return (int)(k < 1 ? 1 : (k > 64 ? 64 : k)); };
   const int wave_tiles = std::min(ntile, 16384);
   const int seg_g = segs_for(maxlen), seg_u = segs_for(use_groups ? gstride : maxlen), seg_t = segs_for(2 * ZB_MAX_OFFSET);
   filt_seg.need(2 * std::max((size_t)ngroup * seg_g, std::max((size_t)nunit * seg_u, (size_t)wave_tiles * seg_t)) + 64);
#ifndef ZB_EMU
   {  /* window lists -> unit lists: one stable partition per window (zb_unit_distribute) */
      std::vector<ZbDistWin> hd(nwin);
      uint32_t ub = 0, sb2 = 0, numax = 1;
      for (int w = 0; w < nwin; w++) {
         const ZbWinDesc &d = h_win[w];
         ZbDistWin x; memset(&x, 0, sizeof(x));
         x.sa_base = h_wbase[w]; x.len = d.len; x.hist = d.hist; x.unit_base = ub; x.seg_base = sb2;
         x.nu = (d.len - d.hist + ZB_MAX_OFFSET - 1) / ZB_MAX_OFFSET;
         ub += x.nu; sb2 += (d.len + 4095) / 4096; numax = std::max(numax, x.nu);
         hd[w] = x;
      }
      groups.need((sizeof(ZbDistWin) * (size_t)nwin + sizeof(ZbTileDesc) - 1) / sizeof(ZbTileDesc) + 1);      /* (the group descriptors' buffer, unused in this build) */
      filt_seg.need(2 * (size_t)sb2 * numax + 64);
      if (zb_failed() || (int)ub != nunit) { if ((int)ub != nunit) zb_cuda_fail(cudaErrorUnknown); return; }
      zb_h2d(st, groups.p, hd.data(), sizeof(ZbDistWin) * nwin);
      zb_unit_distribute(st, sa_lcp.p, (const ZbDistWin *)groups.p, nwin, (int)sb2, nunit, (int)numax, filt_seg.p, unit_words.p, unit_cnt.p);
   }
#else
   if (use_groups) {
      groups.need(ngroup); group_words.need((size_t)ngroup * gstride); group_cnt.need(ngroup);
      zb_h2d(st, groups.p, hg.data(), sizeof(ZbTileDesc) * ngroup);
      zb_tile_filter(st, sa_lcp.p, 0, groups.p, ngroup, 0, group_words.p, gstride, group_cnt.p, seg_g, filt_seg.p);
      zb_tile_filter(st, group_words.p, group_cnt.p, units.p, nunit, 0, unit_words.p, 2 * ZB_MAX_OFFSET, unit_cnt.p, seg_u, filt_seg.p);
   } else {
      zb_tile_filter(st, sa_lcp.p, 0, units.p, nunit, 0, unit_words.p, 2 * ZB_MAX_OFFSET, unit_cnt.p, seg_u, filt_seg.p);
   }
#endif
   const size_t stride = ZB_MAX_OFFSET + tile_main;
   const int wave = 16384;
   const int nw_tiles = std::min(ntile, wave);
#ifdef ZB_EMU
   tile_iv.need((size_t)nw_tiles * stride); tile_cnt.need(nw_tiles);
#else
   const size_t qstride = 3 * (size_t)tile_main;      /* text-walk queue of a tile: 3 words per main position at most */
   tile_iv.need((size_t)nw_tiles * qstride); tile_cnt.need(nw_tiles);
#endif
   const ZbTileDesc *td = tiles.p; uint32_t *ivb = tile_iv.p, *tc = tile_cnt.p;
   zb_match_t *mt = match.p; uint16_t *gl = glen.p, *go = goff.p; const uint32_t *wbs = wbase.p;
   stat_tiles = ntile;
#ifndef ZB_EMU
   const size_t smem = (stride + 2) * 4 + (size_t)tile_main * 2;
   const size_t smem_txt = (stride + ZB_MAX_MATCH + 16 + 7) & ~(size_t)3;      /* + the source's offset modulo 16 (zb_mf_text_k) */
   const ZbWinDesc *wdp = win.p; const uint8_t *Tp = in_ptr;
   tile_q.need(nw_tiles);
   if (zb_failed()) return;
   uint32_t *tq = tile_q.p;
   {  /* the limit is a per-function global: always the largest configuration, so concurrent host threads cannot undercut each other */
      const size_t smax = ((size_t)ZB_MAX_OFFSET + ZB_MF_TILE_MAX + 2) * 4 + (size_t)ZB_MF_TILE_MAX * 2;
      ZB_CUDA_CHECK(cudaFuncSetAttribute(zb_mf_scan_k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smax));
      ZB_CUDA_CHECK(cudaFuncSetAttribute(zb_mf_text_k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(((size_t)ZB_MAX_OFFSET + ZB_MF_TILE_MAX + ZB_MAX_MATCH + 16 + 7) & ~(size_t)3)));
   }
#else
   tile_pd.need((size_t)nw_tiles * tile_main);
   uint32_t *pdb = tile_pd.p; const ZbWinDesc *wdp = win.p; const uint8_t *Tp = in_ptr;
#endif
   for (int first = 0; first < ntile; first += wave) {
      const int cnt = std::min(wave, ntile - first);
#ifdef ZB_EMU
      zb_tile_filter(st, unit_words.p, unit_cnt.p, tiles.p, cnt, first, tile_iv.p, stride, tile_cnt.p, seg_t, filt_seg.p);
#endif
#ifndef ZB_EMU
      if (g_zb_prof_on) { zb_tag("mf_scan"); zb_prof_begin(0, st); }
      /* ZB_TS_MIN / ZB_TS_MUL go in as arguments: compiled in as constants the kernel ran 3 % slower on B200 */
      zb_mf_scan_k<<<cnt, ZB_MF_THREADS, smem, st>>>(td, first, unit_words.p, unit_cnt.p, ivb, qstride, stride, tq, mt, gl, go, wbs, tile_main, ZB_TS_MIN, ZB_TS_MUL);
      if (g_zb_prof_on) zb_prof_end(st);
      if (g_zb_prof_on) { zb_tag("mf_text"); zb_prof_begin(0, st); }
      /* a 16384-position tile has twice the queue and 49 KB of text (4 CTAs per SM): twice the warps per CTA keep the SM as full */
      zb_mf_text_k<<<cnt, tile_main > 8192 ? 512 : 256, smem_txt, st>>>(td, first, ivb, qstride, tq, mt, gl, go, wbs, wdp, Tp);
      if (g_zb_prof_on) zb_prof_end(st);
      zb_count_launch(2);
      ZB_CUDA_CHECK(cudaGetLastError());
#else
      /* host build: same per-position scan, lists in ordinary memory */
      zb_launch(st, cnt, ZB_LAMBDA(long k) {
         const ZbTileDesc t = td[first + k];
         const uint32_t *words = ivb + (size_t)k * stride; uint32_t *rom = pdb + (size_t)k * tile_main;
         const uint32_t nlook = t.m0 - t.lo;
         for (uint32_t e = 0; e < tc[k]; e++) { uint32_t p = words[e] & ZB_POS_MASK; if (p >= nlook) rom[p - nlook] = e; }
      });
      zb_launch(st, (long)cnt * tile_main, ZB_LAMBDA(long x) {
         const int k = (int)(x / tile_main); const uint32_t m = (uint32_t)(x % tile_main);
         const ZbTileDesc t = td[first + k];
         if (m >= t.hi - t.m0) return;
         const uint32_t *words = ivb + (size_t)k * stride; const uint32_t *rom = pdb + (size_t)k * tile_main;
         const uint32_t nlook = t.m0 - t.lo, p = t.m0 + m, gbase = wbs[t.win];
         zb_match_t o[ZB_NMATCH];
         const int nm = zb_mf_scan(words, (int)tc[k], (int)rom[m], nlook + m, Tp + wdp[t.win].in_off + t.lo, o);
         const uint32_t maxlen = t.wlen - p;
         zb_match_t *dst = mt + ((size_t)(gbase + p) << 3);
         for (int q = 0; q < ZB_NMATCH; q++) {
            zb_match_t v; v.length = 0; v.offset = 0;
            if (q < nm) { v = o[q]; if (v.length > maxlen) v.length = (uint16_t)maxlen; }
            dst[q] = v;
         }
         const uint16_t l0 = dst[0].length;
         gl[gbase + p] = l0 >= ZB_MIN_MATCH ? l0 : (uint16_t)1;
         go[gbase + p] = l0 >= ZB_MIN_MATCH ? dst[0].offset : (uint16_t)0;
      });
#endif
   }
}

#ifndef ZB_EMU
/* ---- path marking: where the token chain that enters a 1024-position chunk leaves it ----
 * A chain p -> p + len(p) can only enter a chunk within its first 258 positions, so per chunk a row of 258 exit offsets is
 * all the hop needs.  Sweep: one thread per chunk, backwards; the exit offsets of the positions behind (<= 258) sit in a
 * shared-memory ring ([slot][thread]: conflict-free), lengths are read 16 bytes at a time.  MODE 0: greedy path, lengths
 * from glen (u16), chunks per window.  MODE 1: chosen path, lengths from best[] (< 3 counts as a literal), chunks per
 * sub-block; pass >= 0 skips static sub-blocks after the first pass.  The length is the low 9 bits of the word in both the parse
 * kernel's choice format (k | sym << 9 | m << 14) and the final {length, offset} format. */
#define ZB_SW_THREADS 64
#define ZB_SW_RING 288
#define ZB_EXROW 264          /* u16 per chunk row: 258 used, 528 bytes = 33 x 16 */
template <int MODE>
__global__ void __launch_bounds__(ZB_SW_THREADS) zb_sweep_k(long nchunk, const ZbWinDesc *wd, const uint32_t *wbs, const uint32_t *gcf, int nw, uint32_t *gcw,
                                                            const uint16_t *gl, const ZbSub *sb, const uint32_t *pcs, int pass, const zb_match_t *bm, uint16_t *exc,
                                                            uint32_t cpv /* MODE 1: positions per path chunk (ZbPipe::cp) */) {
   __shared__ uint16_t ring_s[ZB_SW_RING * ZB_SW_THREADS];
   const long c = (long)blockIdx.x * ZB_SW_THREADS + threadIdx.x;
   if (c >= nchunk) return;
   uint32_t lo, hi, gb;
   if (MODE == 0) {
      const int w = zb_find_win(gcf, nw, (uint32_t)c);
      gcw[c] = (uint32_t)w;
      lo = wd[w].hist + (uint32_t)(c - gcf[w]) * ZB_CG;
      hi = lo + ZB_CG < wd[w].len ? lo + ZB_CG : wd[w].len;
      gb = wbs[w];
   } else {
      const ZbSub s = sb[pcs[c]];
      if (pass > 0 && !s.is_dyn) return;
      const uint32_t k = (uint32_t)c - s.pchunk_base;
      gb = wbs[s.win];
      lo = s.ps + k * cpv; hi = lo + cpv < s.pe ? lo + cpv : s.pe;
   }
   uint16_t *ring = ring_s + threadIdx.x;
   uint16_t *row = exc + (size_t)c * ZB_EXROW;
   int idx = (int)((hi - 1 - lo) % ZB_SW_RING) + 1;     /* slot of position p is (p - lo) % ZB_SW_RING; idx = slot(p) + 1 before the step */
   uint32_t p = hi;
#define ZB_SW_STEP(len_) do { \
      uint32_t l_ = (len_);      /* evaluated before p moves: the scalar callers index with p - 1 */ \
      p--; idx--; if (idx < 0) idx += ZB_SW_RING; \
      if (MODE == 1 && l_ < ZB_MIN_MATCH) l_ = 1; \
      const uint32_t j_ = p + l_; \
      uint32_t e_; \
      if (j_ >= hi) e_ = j_ - hi; else { int i2_ = idx + (int)l_; if (i2_ >= ZB_SW_RING) i2_ -= ZB_SW_RING; e_ = ring[i2_ * ZB_SW_THREADS]; } \
      ring[idx * ZB_SW_THREADS] = (uint16_t)e_; \
      if (p - lo < 258u) row[p - lo] = (uint16_t)e_; \
   } while (0)
   if (MODE == 0) {
      /* the 16-byte groups are fetched two ahead into three registers used in rotation (no copies: a register move would
         wait for the load it forwards): the steps are a dependent chain through the ring, a load consumed at once would put
         a DRAM round trip on it every few steps */
      while (p > lo && ((gb + p) & 7u)) ZB_SW_STEP(gl[gb + p - 1]);
      const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
#define ZB_SW_LD0(k_) (p >= lo + (k_) ? __ldg((const uint4 *)(gl + gb + p - (k_))) : z4)
#define ZB_SW_PROC0(v) do { ZB_SW_STEP((v).w >> 16); ZB_SW_STEP((v).w & 0xffffu); ZB_SW_STEP((v).z >> 16); ZB_SW_STEP((v).z & 0xffffu); \
                            ZB_SW_STEP((v).y >> 16); ZB_SW_STEP((v).y & 0xffffu); ZB_SW_STEP((v).x >> 16); ZB_SW_STEP((v).x & 0xffffu); } while (0)
      uint4 va = ZB_SW_LD0(8), vb = ZB_SW_LD0(16), vc = ZB_SW_LD0(24);
      for (;;) {
         if (p < lo + 8) break; ZB_SW_PROC0(va); va = ZB_SW_LD0(24);
         if (p < lo + 8) break; ZB_SW_PROC0(vb); vb = ZB_SW_LD0(24);
         if (p < lo + 8) break; ZB_SW_PROC0(vc); vc = ZB_SW_LD0(24);
      }
#undef ZB_SW_LD0
#undef ZB_SW_PROC0
      while (p > lo) ZB_SW_STEP(gl[gb + p - 1]);
   } else {
      while (p > lo && ((gb + p) & 3u)) ZB_SW_STEP(bm[gb + p - 1].length & 0x1ffu);
      const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
#define ZB_SW_LD1(k_) (p >= lo + (k_) ? *(const uint4 *)(bm + gb + p - (k_)) : z4)
#define ZB_SW_PROC1(v) do { ZB_SW_STEP((v).w & 0x1ffu); ZB_SW_STEP((v).z & 0x1ffu); ZB_SW_STEP((v).y & 0x1ffu); ZB_SW_STEP((v).x & 0x1ffu); } while (0)
      uint4 va = ZB_SW_LD1(4), vb = ZB_SW_LD1(8), vc = ZB_SW_LD1(12);
      for (;;) {
         if (p < lo + 4) break; ZB_SW_PROC1(va); va = ZB_SW_LD1(12);
         if (p < lo + 4) break; ZB_SW_PROC1(vb); vb = ZB_SW_LD1(12);
         if (p < lo + 4) break; ZB_SW_PROC1(vc); vc = ZB_SW_LD1(12);
      }
#undef ZB_SW_LD1
#undef ZB_SW_PROC1
      while (p > lo) ZB_SW_STEP(bm[gb + p - 1].length & 0x1ffu);
   }
#undef ZB_SW_STEP
}

/* Hop: one warp per window (MODE 0) or sub-block (MODE 1) follows the chain from chunk to chunk; the rows of the next 8
   chunks are fetched into shared memory (cp.async, double buffered) while lane 0 walks the current 8.  MODE 1 also starts
   the pass's fresh histogram (blockdeflate.c:887-891; EOB counted here) when pass >= 0. */
#define ZB_HOP_G 8
template <int MODE>
__global__ void __launch_bounds__(32) zb_hop_k(int nunits, const ZbWinDesc *wd, const uint32_t *gcf, const ZbSub *sb, ZbSubTabs *tb, int pass, const uint16_t *exc, uint32_t *ent, uint32_t cpv) {
   __shared__ __align__(16) uint16_t buf[2][ZB_HOP_G][ZB_EXROW];
   const int x = blockIdx.x, lane = threadIdx.x;
   if (x >= nunits) return;
   uint32_t start, end, cbase, nchunk, clen;
   if (MODE == 0) { start = wd[x].hist; end = wd[x].len; cbase = gcf[x]; nchunk = gcf[x + 1] - gcf[x]; clen = ZB_CG; }
   else {
      const ZbSub s = sb[x];
      if (pass > 0 && !s.is_dyn) return;
      start = s.ps; end = s.pe; cbase = s.pchunk_base; nchunk = s.npchunk; clen = cpv;
      if (pass >= 0 && s.is_dyn) {
         ZbSubTabs &t = tb[x];
         for (int i = lane; i < ZB_NLIT; i += 32) t.lcnt[i] = i == ZB_EOB ? 1 : 0;
         if (lane < ZB_NOFF) t.ocnt[lane] = 0;
      }
   }
   const uint16_t *rows = exc + (size_t)cbase * ZB_EXROW;
   const int per = ZB_EXROW * 2 / 16;      /* 16-byte pieces per row */
   auto fetch = [&](uint32_t g0, int b) {
      const uint32_t ng = nchunk - g0 < ZB_HOP_G ? nchunk - g0 : ZB_HOP_G;
      for (int q = lane; q < (int)ng * per; q += 32)
         __pipeline_memcpy_async((char *)&buf[b][0][0] + (size_t)q * 16, (const char *)(rows + (size_t)g0 * ZB_EXROW) + (size_t)q * 16, 16);
      __pipeline_commit();
   };
   uint32_t e = start;
   if (nchunk) fetch(0, 0);
   int b = 0;
   for (uint32_t g0 = 0; g0 < nchunk; g0 += ZB_HOP_G, b ^= 1) {
      if (g0 + ZB_HOP_G < nchunk) { fetch(g0 + ZB_HOP_G, b ^ 1); __pipeline_wait_prior(1); }
      else __pipeline_wait_prior(0);
      __syncwarp();
      if (lane == 0) {
         const uint32_t ng = nchunk - g0 < ZB_HOP_G ? nchunk - g0 : ZB_HOP_G;
         for (uint32_t k = 0; k < ng; k++) {
            const uint32_t lo = start + (g0 + k) * clen, hi = lo + clen < end ? lo + clen : end;
            ent[cbase + g0 + k] = e;
            if (e < hi) e = hi + buf[b][k][e - lo];
         }
      }
      e = __shfl_sync(0xffffffffu, e, 0);
      __syncwarp();
   }
}
#endif

/* ============================================================ greedy path ============================================================
 * The greedy parse of blockdeflate.c:333-361 / :684-703 takes match[i][0] whenever its length is >= 3.  All
 * greedy walks inside a window are segments of the one path from the block start (SURVEY A-14), so the path
 * is materialised once: exit offsets per chunk (backward sweep), a serial hop over chunk entries per window,
 * then the token list, and prefix histograms every ZB_TOKI tokens.
 */
inline void ZbPipe::stage_greedy() {
   h_gchunk_first.assign(nwin + 1, 0);
   for (int w = 0; w < nwin; w++) h_gchunk_first[w + 1] = h_gchunk_first[w] + (h_win[w].len - h_win[w].hist + ZB_CG - 1) / ZB_CG;
   const long nch = h_gchunk_first[nwin];
   gchunk_first.need(nwin + 1); gchunk_win.need(nch);
   zb_h2d(st, gchunk_first.p, h_gchunk_first.data(), 4 * (nwin + 1));
#ifdef ZB_EMU
   exitoff.need(P);
#endif
   gentry.need(nch + 1); gtokcnt.need(nch + 1); gtokbase.need(nch + 1); tokpos.need(P);
   wtokbase.need(nwin + 1); wintbase.need(nwin + 1);
#ifndef ZB_EMU
   exitc.need((size_t)(nch + 1) * ZB_EXROW);
#endif
   if (zb_failed()) return;
   const ZbWinDesc *wd = win.p; const uint32_t *wbs = wbase.p, *gcf = gchunk_first.p; const int nw = nwin;
   uint32_t *gcw = gchunk_win.p; uint16_t *ex = exitoff.p; const uint16_t *gl = glen.p;
   uint32_t *ent = gentry.p, *tcnt = gtokcnt.p, *tbase = gtokbase.p, *tp = tokpos.p;
#ifndef ZB_EMU
   if (nch > 0) {
      if (g_zb_prof_on) { zb_tag("path_sweep"); zb_prof_begin(0, st); }
      zb_sweep_k<0><<<(unsigned)((nch + ZB_SW_THREADS - 1) / ZB_SW_THREADS), ZB_SW_THREADS, 0, st>>>(nch, wd, wbs, gcf, nw, gcw, gl, 0, 0, -1, 0, exitc.p, ZB_CG);
      if (g_zb_prof_on) zb_prof_end(st);
      if (g_zb_prof_on) { zb_tag("path_hop"); zb_prof_begin(0, st); }
      zb_hop_k<0><<<nwin, 32, 0, st>>>(nwin, wd, gcf, 0, 0, -1, exitc.p, ent, ZB_CG);
      if (g_zb_prof_on) zb_prof_end(st);
      zb_count_launch(2);
      ZB_CUDA_CHECK(cudaGetLastError());
   }
   (void)ex;
#else
   zb_launch(st, nch, ZB_LAMBDA(long c) {
      int w = zb_find_win(gcf, nw, (uint32_t)c);
      gcw[c] = (uint32_t)w;
      const uint32_t lo = wd[w].hist + (uint32_t)(c - gcf[w]) * ZB_CG;
      const uint32_t hi = lo + ZB_CG < wd[w].len ? lo + ZB_CG : wd[w].len;
      const uint32_t gb = wbs[w];
      for (uint32_t p = hi; p-- > lo;) {
         uint32_t j = p + gl[gb + p];
         ex[gb + p] = (uint16_t)(j >= hi ? j - hi : ex[gb + j]);
      }
   });
   zb_launch(st, nwin, ZB_LAMBDA(long w) {
      uint32_t e = wd[w].hist;
      const uint32_t gb = wbs[w];
      for (uint32_t c = gcf[w]; c < gcf[w + 1]; c++) {
         ent[c] = e;
         const uint32_t lo = wd[w].hist + (c - gcf[w]) * ZB_CG;
         const uint32_t hi = lo + ZB_CG < wd[w].len ? lo + ZB_CG : wd[w].len;
         if (e < hi) e = hi + ex[gb + e];
      }
   });
#endif
   zb_launch(st, nch, ZB_LAMBDA(long c) {
      const uint32_t w = gcw[c];
      const uint32_t lo = wd[w].hist + (uint32_t)(c - gcf[w]) * ZB_CG;
      const uint32_t hi = lo + ZB_CG < wd[w].len ? lo + ZB_CG : wd[w].len;
      const uint32_t gb = wbs[w];
      uint32_t n = 0;
      for (uint32_t p = ent[c]; p < hi; p += gl[gb + p]) n++;
      tcnt[c] = n;
   });
   scratch.need(zb_scan_scratch_words(nch + 1) + 64);
   zb_exclusive_sum(st, tcnt, tbase, nch, counters.p, scratch.p);
   zb_launch(st, nch, ZB_LAMBDA(long c) {
      const uint32_t w = gcw[c];
      const uint32_t lo = wd[w].hist + (uint32_t)(c - gcf[w]) * ZB_CG;
      const uint32_t hi = lo + ZB_CG < wd[w].len ? lo + ZB_CG : wd[w].len;
      const uint32_t gb = wbs[w];
      uint32_t k = tbase[c];
      for (uint32_t p = ent[c]; p < hi; p += gl[gb + p]) tp[k++] = p;
   });
   /* per-window token base / count, prefix-histogram interval base */
   uint32_t *wtb = wtokbase.p, *wib = wintbase.p, *cn = counters.p;
   zb_launch(st, 1, ZB_LAMBDA(long) {
      uint32_t ib = 0;
      for (int w = 0; w < nw; w++) {
         uint32_t b = tbase[gcf[w]];
         uint32_t e = (w + 1 < nw) ? tbase[gcf[w + 1]] : cn[0];
         wtb[w] = b; wib[w] = ib;
         ib += (e - b) / ZB_TOKI + 1;   /* prefix rows 0..floor(ntok/ZB_TOKI) */
         if (w + 1 == nw) { wtb[nw] = e; wib[nw] = ib; }
      }
   });
   std::vector<uint32_t> h_wib(nwin + 1);
   zb_d2h(st, h_wib.data(), wib, 4 * (nwin + 1)); zb_sync(st);
   const long nint = h_wib[nwin];
   ph.need((size_t)nint * ZB_NH);
   if (zb_failed()) return;
   int *PH = ph.p; const uint8_t *T = in_ptr; const uint16_t *go = goff.p;
   /* per-interval histograms: row k+1 of a window = histogram of tokens [k*ZB_TOKI, (k+1)*ZB_TOKI) */
   zb_launch(st, nint, ZB_LAMBDA(long r) {
      int w = zb_find_win(wib, nw, (uint32_t)r);
      uint32_t k = (uint32_t)r - wib[w];
      int *row = PH + (size_t)r * ZB_NH;
      for (int i = 0; i < ZB_NH; i++) row[i] = 0;
      if (k == 0) return;
      const uint32_t gb = wbs[w];
      const uint8_t *t = T + wd[w].in_off;
      const uint32_t t1 = wtb[w] + (k - 1) * ZB_TOKI, t2 = t1 + ZB_TOKI;
      uint32_t q = t1;
#ifdef __CUDA_ARCH__
      for (; q + 8 <= t2; q += 8) {      /* the loads of 8 tokens level by level (see ZbGreedyView::add_tokens) */
         uint32_t p[8], l[8], o[8], c[8];
#pragma unroll
         for (int j = 0; j < 8; j++) p[j] = tp[q + j];
#pragma unroll
         for (int j = 0; j < 8; j++) { l[j] = gl[gb + p[j]]; o[j] = go[gb + p[j]]; c[j] = t[p[j]]; }
#pragma unroll
         for (int j = 0; j < 8; j++) {
            if (l[j] >= ZB_MIN_MATCH) { row[zb_len_sym(l[j] - ZB_MIN_MATCH)] += 1; row[ZB_NLIT + zb_off_sym(o[j])] += 1; }
            else row[c[j]] += 1;
         }
      }
#endif
      for (; q < t2; q++) {
         uint32_t p = tp[q];
         uint32_t l = gl[gb + p];
         zb_tok_count(t, p, l, go[gb + p], row, row + ZB_NLIT, 1);
      }
   });
   /* prefix sums down the rows of each window, one task per (window, bin) */
   zb_launch(st, (long)nwin * ZB_NH, ZB_LAMBDA(long x) {
      const int w = (int)(x / ZB_NH), b = (int)(x % ZB_NH);
      int acc = 0;
      uint32_t r = wib[w];
      const uint32_t r1 = wib[w + 1];
      for (; r + 8 <= r1; r += 8) {       /* 8 rows' loads in flight, then the running sums */
         int v[8];
#pragma unroll
         for (int j = 0; j < 8; j++) v[j] = PH[(size_t)(r + j) * ZB_NH + b];
#pragma unroll
         for (int j = 0; j < 8; j++) { acc += v[j]; PH[(size_t)(r + j) * ZB_NH + b] = acc; }
      }
      for (; r < r1; r++) { acc += PH[(size_t)r * ZB_NH + b]; PH[(size_t)r * ZB_NH + b] = acc; }
   });
}

/* histogram of greedy tokens [t1, t2) (window-relative token indices) of window w into h[ZB_NH] (overwritten) */
struct ZbGreedyView {
   const int *PH; const uint32_t *wib, *wtb, *tp, *wbs; const uint16_t *gl, *go; const uint8_t *T; const ZbWinDesc *wd;
   ZB_HD void add_tokens(int w, uint32_t t1, uint32_t t2, int *h, int sign) const {
      const uint32_t gb = wbs[w]; const uint8_t *t = T + wd[w].in_off;
      uint32_t q = wtb[w] + t1;
      const uint32_t q1 = wtb[w] + t2;
#ifdef __CUDA_ARCH__
      /* one thread walks up to 2 x 255 edge tokens, three dependent loads each: batches of 8 with the loads of a level issued
         together, so a batch costs three memory round trips instead of twenty-four */
      for (; q + 8 <= q1; q += 8) {
         uint32_t p[8], l[8], o[8], c[8];
#pragma unroll
         for (int j = 0; j < 8; j++) p[j] = tp[q + j];
#pragma unroll
         for (int j = 0; j < 8; j++) { l[j] = gl[gb + p[j]]; o[j] = go[gb + p[j]]; c[j] = t[p[j]]; }
#pragma unroll
         for (int j = 0; j < 8; j++) {
            if (l[j] >= ZB_MIN_MATCH) { h[zb_len_sym(l[j] - ZB_MIN_MATCH)] += sign; h[ZB_NLIT + zb_off_sym(o[j])] += sign; }
            else h[c[j]] += sign;
         }
      }
#endif
      for (; q < q1; q++) {
         uint32_t p = tp[q];
         zb_tok_count(t, p, gl[gb + p], go[gb + p], h, h + ZB_NLIT, sign);
      }
   }
   ZB_HD void range_hist(int w, uint32_t t1, uint32_t t2, int *h) const {
      const uint32_t k1 = (t1 + ZB_TOKI - 1) / ZB_TOKI, k2 = t2 / ZB_TOKI;
      if (k1 <= k2) {
         const int *a = PH + (size_t)(wib[w] + k1) * ZB_NH, *b = PH + (size_t)(wib[w] + k2) * ZB_NH;
         for (int i = 0; i < ZB_NH; i++) h[i] = b[i] - a[i];
         add_tokens(w, t1, k1 * ZB_TOKI, h, 1);
         add_tokens(w, k2 * ZB_TOKI, t2, h, 1);
      } else {
         for (int i = 0; i < ZB_NH; i++) h[i] = 0;
         add_tokens(w, t1, t2, h, 1);
      }
   }
   /* token index (window-relative) of the token starting at position p (p must be on the path) */
   ZB_HD uint32_t tok_of_pos(int w, uint32_t p, uint32_t ntok) const {
      uint32_t lo = 0, hi = ntok;
      const uint32_t *a = tp + wtb[w];
      while (lo < hi) { uint32_t mid = (lo + hi) >> 1; if (a[mid] < p) lo = mid + 1; else hi = mid; }
      return lo;
   }
};

#ifndef ZB_EMU
/* Splitter drift test (blockdeflate.c:706-721), one warp per node: lane k of a round owns check point base + k; the 18-bin
   running statistics before it are a warp prefix sum of the per-interval statistics (same unsigned 32-bit arithmetic as the
   reference's sequential accumulation, SURVEY A-15). */
__global__ void __launch_bounds__(128) zb_split_drift_k(const ZbNode *cur, int ncur, const uint16_t *cs, uint8_t *cf) {
   const int lane = threadIdx.x & 31;
   const int x = blockIdx.x * 4 + (threadIdx.x >> 5);
   if (x >= ncur) return;
   const ZbNode nd = cur[x];
   uint32_t carry[18];
#pragma unroll
   for (int j = 0; j < 18; j++) carry[j] = 0;
   for (uint32_t base = 0; base < nd.nchk; base += 32) {
      const uint32_t k = base + lane;
      const bool valid = k < nd.nchk;
      const uint16_t *ns = cs + (size_t)(nd.chk_base + (valid ? k : 0)) * 18;
      uint32_t own[18], stat[18], nstat = 0;
#pragma unroll
      for (int j = 0; j < 18; j++) {
         own[j] = valid ? (uint32_t)ns[j] : 0u;
         uint32_t inc = own[j];
#pragma unroll
         for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
         stat[j] = carry[j] + inc - own[j];
         nstat += stat[j];
         carry[j] += __shfl_sync(0xffffffffu, inc, 31);
      }
      if (valid) {
         const uint32_t nnew = k == 0 ? nd.t0 : 256;
         uint8_t flag = 0;
         if (nstat) {
            uint32_t tot = 0;
#pragma unroll
            for (int j = 0; j < 18; j++) {
               const uint32_t e = stat[j] * nnew, a = own[j] * nstat;
               tot += e > a ? e - a : a - e;
            }
            if ((tot / nnew) >= (nstat * 45 / 100)) flag = 1;
         }
         cf[nd.chk_base + k] = flag;
      }
   }
}
#endif

#ifndef ZB_EMU
#include "zb_warp.h"
#define ZB_WT 128                 /* threads per CTA of the warp-per-task kernels: 4 tasks */

/* splitter S1 (blockdeflate.c:646-667): one warp per node - greedy histogram of the node, its cost estimate, check-point layout */
__global__ void __launch_bounds__(ZB_WT) zb_split_nodes_k(ZbNode *cur, int ncur, int *nh, ZbGreedyView gv) {
   __shared__ ZbWarpScratch ws[ZB_WT / 32];
   const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
   const int x = blockIdx.x * (ZB_WT / 32) + wi;
   if (x >= ncur) return;
   ZbWarpScratch &s = ws[wi];
   ZbNode nd = cur[x];
   nd.nchk = 0; nd.best_tok = 0; nd.best_delta = 0; nd.t0 = 0;
   if (nd.pe - nd.ps >= 8192) {
      zbw_range_hist(gv, (int)nd.win, nd.ts, nd.te, s.h, lane);
      if (lane == 0) s.h[ZB_EOB] += 1;
      __syncwarp();
      int *h = nh + (size_t)x * ZB_NH;
      for (int i = lane; i < ZB_NH; i += 32) h[i] = s.h[i];
      zbw_lengths(s.h, ZB_NLIT, s.llen, s, lane);
      zbw_lengths(s.h + ZB_NLIT, ZB_NOFF, s.olen, s, lane);
      nd.total_cost = zbw_dynamic_cost(s.h, s.llen, s.h + ZB_NLIT, s.olen, s, lane);
      /* first check: >= 256 tokens and >= 512 bytes consumed (blockdeflate.c:705), then every 256 tokens */
      const uint32_t ntok = nd.te - nd.ts;
      const uint32_t *a = gv.tp + gv.wtb[nd.win] + nd.ts;
      uint32_t t0 = 256;
      while (t0 <= ntok) {
         const uint32_t endpos = t0 < ntok ? a[t0] : nd.pe;
         if (endpos - nd.ps >= 512) break;
         t0++;
      }
      if (t0 <= ntok) { nd.t0 = t0; nd.nchk = (ntok - t0) / 256 + 1; }
   }
   if (lane == 0) cur[x] = nd;
}

/* splitter S4 (blockdeflate.c:724-757): one warp per side of a drift-flagged candidate */
__global__ void __launch_bounds__(ZB_WT) zb_split_eval_k(const ZbNode *cur, long ntask, const uint8_t *cf, const uint32_t *cnode, const int *nh, int *cdl, ZbGreedyView gv) {
   __shared__ ZbWarpScratch ws[ZB_WT / 32];
   const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
   const long y = (long)blockIdx.x * (ZB_WT / 32) + wi;
   if (y >= ntask) return;
   const long c = y >> 1; const int right_side = (int)(y & 1);
   if (!cf[c]) { if (lane == 0) cdl[y] = -1; return; }
   ZbWarpScratch &s = ws[wi];
   const uint32_t x = cnode[c];
   const ZbNode nd = cur[x];
   const uint32_t k = (uint32_t)c - nd.chk_base;   /* k >= 1 here */
   const uint32_t tsplit = nd.t0 + 256 * (k - 1);   /* tokens left of the split */
   zbw_range_hist(gv, (int)nd.win, nd.ts, nd.ts + tsplit, s.h, lane);
   if (right_side) {
      const int *tot = nh + (size_t)x * ZB_NH;
      for (int i = lane; i < ZB_NH; i += 32) s.h[i] = tot[i] - s.h[i];
   }
   __syncwarp();
   if (lane == 0) s.h[ZB_EOB] = 1;
   __syncwarp();
   zbw_lengths(s.h, ZB_NLIT, s.llen, s, lane);
   zbw_lengths(s.h + ZB_NLIT, ZB_NOFF, s.olen, s, lane);
   const int cost = zbw_dynamic_cost(s.h, s.llen, s.h + ZB_NLIT, s.olen, s, lane);
   if (lane == 0) cdl[y] = cost;
}

/* D1: greedy histogram, static-vs-dynamic decision (libzultra.c:317-324), first tables (blockdeflate.c:863-869): one warp per sub-block */
__global__ void __launch_bounds__(ZB_WT) zb_sub_init_k(ZbSub *sb, ZbSubTabs *tb, int ns, ZbGreedyView gv) {
   __shared__ ZbWarpScratch ws[ZB_WT / 32];
   const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
   const int x = blockIdx.x * (ZB_WT / 32) + wi;
   if (x >= ns) return;
   ZbWarpScratch &s = ws[wi];
   ZbSub sub = sb[x]; ZbSubTabs &t = tb[x];
   zbw_range_hist(gv, (int)sub.win, sub.ts, sub.te, s.h, lane);
   if (lane == 0) s.h[ZB_EOB] += 1;
   __syncwarp();
   {  /* zb_static_cost */
      int c = 0;
      for (int i = lane; i < 286; i += 32) c += s.h[i] * (zb_static_lit_len(i) + (i >= 257 ? zb_lensym_extra(i - 257) : 0));
      if (lane < ZB_NOFF) c += s.h[ZB_NLIT + lane] * (5 + zb_offsym_extra(lane));
      sub.static_cost = zbw_sum(c) + 3;
   }
   zbw_lengths(s.h, ZB_NLIT, s.llen, s, lane);
   zbw_lengths(s.h + ZB_NLIT, ZB_NOFF, s.olen, s, lane);
   sub.dynamic_cost = zbw_dynamic_cost(s.h, s.llen, s.h + ZB_NLIT, s.olen, s, lane);
   sub.is_dyn = sub.static_cost <= sub.dynamic_cost ? 0 : 1;
   sub.ub_hit = 0;
   if (sub.is_dyn) {
      int ub = 0;
      zbw_build(s.h, ZB_NLIT, 15, s.llen, s, &ub, lane);
      zbw_build(s.h + ZB_NLIT, ZB_NOFF, 15, s.olen, s, &ub, lane);
      sub.ub_hit = __shfl_sync(ZBW_FULL, ub, 0);
      for (int i = lane; i < ZB_NLIT; i += 32) t.llen[i] = s.llen[i];
      if (lane < ZB_NOFF) t.olen[lane] = s.olen[lane];
      zbw_make_costtab(s.llen, s.olen, true, t.cost, lane);      /* blockdeflate.c:873-881 */
   } else {
      for (int i = lane; i < ZB_NLIT; i += 32) { t.llen[i] = zb_static_lit_len(i); s.llen[i] = zb_static_lit_len(i); }   /* blockdeflate.c:839-849 */
      if (lane < ZB_NOFF) { t.olen[lane] = 5; s.olen[lane] = 5; }
      __syncwarp();
      zbw_make_costtab(s.llen, s.olen, false, t.cost, lane);
   }
   if (lane == 0) sb[x] = sub;
}

/* D7: rebuild the tables from the pass's histogram (blockdeflate.c:893-919): one warp per sub-block */
__global__ void __launch_bounds__(ZB_WT) zb_sub_tables_k(ZbSub *sb, ZbSubTabs *tb, int ns, int pass) {
   __shared__ ZbWarpScratch ws[ZB_WT / 32];
   const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
   const int x = blockIdx.x * (ZB_WT / 32) + wi;
   if (x >= ns) return;
   if (!sb[x].is_dyn) return;
   ZbWarpScratch &s = ws[wi];
   ZbSubTabs &t = tb[x];
   if (pass == 3 && lane == 0) {   /* always describe at least two distance codes (blockdeflate.c:893-913) */
      int nz = 0;
      for (int i = 0; nz < 2 && i < ZB_NOFF - 2; i++) if (t.ocnt[i]) nz++;
      if (nz == 0) t.ocnt[0] = t.ocnt[1] = 1;
      else if (nz == 1) { if (t.ocnt[0]) t.ocnt[1] = 1; else t.ocnt[0] = 1; }
   }
   __syncwarp();
   for (int i = lane; i < ZB_NLIT; i += 32) s.h[i] = t.lcnt[i];
   if (lane < ZB_NOFF) s.h[ZB_NLIT + lane] = t.ocnt[lane];
   __syncwarp();
   int ub = 0;
   zbw_build(s.h, ZB_NLIT, 15, s.llen, s, &ub, lane);
   zbw_build(s.h + ZB_NLIT, ZB_NOFF, 15, s.olen, s, &ub, lane);
   for (int i = lane; i < ZB_NLIT; i += 32) t.llen[i] = s.llen[i];
   if (lane < ZB_NOFF) t.olen[lane] = s.olen[lane];
   zbw_make_costtab(s.llen, s.olen, pass < 3, t.cost, lane);      /* final lengths as they are: the post-optimiser and the emitter use them */
   if (lane == 0 && ub) sb[x].ub_hit = 1;
}
/* F1a: RLE smoothing trial (blockdeflate.c:926-945) and the code-length sequence to be described: one warp per sub-block */
__global__ void __launch_bounds__(ZB_WT) zb_sub_smooth_k(ZbSub *sb, ZbSubTabs *tb, int ns) {
   __shared__ ZbWarpScratch ws[ZB_WT / 32];
   const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
   const int x = blockIdx.x * (ZB_WT / 32) + wi;
   if (x >= ns) return;
   ZbWarpScratch &s = ws[wi];
   ZbSub sub = sb[x]; ZbSubTabs &t = tb[x];
   if (!sub.is_dyn) {
      sub.nl = 288; sub.no = 32; sub.ncl = 0; sub.mask = 0; sub.hdr_bits = 0;
      if (lane == 0) sb[x] = sub;
      return;
   }
   for (int i = lane; i < ZB_NLIT; i += 32) { s.llen[i] = t.llen[i]; s.h[i] = t.lcnt[i]; s.olen[i] = i < ZB_NOFF ? t.olen[i] : 0; }
   if (lane < ZB_NOFF) s.h[ZB_NLIT + lane] = t.ocnt[lane];
   __syncwarp();
   const int cur_cost = zbw_dynamic_cost(s.h, s.llen, s.h + ZB_NLIT, s.olen, s, lane);
   if (lane == 0) {      /* zultra_huffman_encoder_optimize_for_rle: two short sequential scans */
      zb_smooth_counts(ZB_NLIT, s.h, s.sc.cl);
      zb_smooth_counts(ZB_NOFF, s.h + ZB_NLIT, s.sc.cl);
   }
   __syncwarp();
   int ub = 0;
   zbw_build(s.h, ZB_NLIT, 15, s.llen, s, &ub, lane);
   zbw_build(s.h + ZB_NLIT, ZB_NOFF, 15, s.olen, s, &ub, lane);
   const int opt_cost = zbw_dynamic_cost(s.h, s.llen, s.h + ZB_NLIT, s.olen, s, lane);
   if (opt_cost < cur_cost) {      /* the smoothed counts stay in the encoder (SURVEY A-7) */
      for (int i = lane; i < ZB_NLIT; i += 32) { t.lcnt[i] = s.h[i]; t.llen[i] = s.llen[i]; }
      if (lane < ZB_NOFF) { t.ocnt[lane] = s.h[ZB_NLIT + lane]; t.olen[lane] = s.olen[lane]; }
      if (__shfl_sync(ZBW_FULL, ub, 0)) sub.ub_hit = 1;
   } else {
      for (int i = lane; i < ZB_NLIT; i += 32) s.llen[i] = t.llen[i];
      if (lane < ZB_NOFF) s.olen[lane] = t.olen[lane];
   }
   __syncwarp();
   int nl = 257, no = 1;
   { const int i = 256 + lane; const uint32_t mk = __ballot_sync(ZBW_FULL, i >= 257 && s.llen[i] != 0); if (mk) nl = 256 + 32 - __clz((int)mk); }
   { const uint32_t mk = __ballot_sync(ZBW_FULL, lane >= 1 && s.olen[lane] != 0); if (mk) no = 32 - __clz((int)mk); }
   sub.nl = nl; sub.no = no;
   for (int i = lane; i < nl; i += 32) t.cl[i] = (uint8_t)s.llen[i];
   for (int i = lane; i < no; i += 32) t.cl[nl + i] = (uint8_t)s.olen[i];
   if (lane == 0) sb[x] = sub;
}
#endif

/* ============================================================ block splitter ============================================================
 * zultra_compressor_split_subblock_recursive (blockdeflate.c:634-786), one recursion level per round.
 */
inline void ZbPipe::stage_split() {
   const int maxnodes = nwin * 32;
   nodesA.need(maxnodes); nodesB.need(maxnodes); nodehist.need((size_t)maxnodes * ZB_NH);
   wsplit.need((size_t)nwin * ZB_MAXSB); wnsplit.need(nwin);
   sub.need((size_t)nwin * ZB_MAXSB); tabs.need((size_t)nwin * ZB_MAXSB); wsubcnt.need(nwin + 1); wsubbase.need(nwin + 1);
   if (zb_failed()) return;
   zb_memset(st, wnsplit.p, 0, 4 * nwin);
   ZbGreedyView gv = {ph.p, wintbase.p, wtokbase.p, tokpos.p, wbase.p, glen.p, goff.p, in_ptr, win.p};
   const ZbWinDesc *wd = win.p; const uint32_t *wtb = wtokbase.p;
   ZbNode *cur = nodesA.p, *nxt = nodesB.p;
   int *nh = nodehist.p; uint32_t *cn = counters.p;
   const int nw = nwin;
   zb_launch(st, nwin, ZB_LAMBDA(long w) {
      ZbNode nd; memset(&nd, 0, sizeof(nd));
      nd.win = (uint32_t)w; nd.depth = 0; nd.ts = 0; nd.te = wtb[w + 1] - wtb[w]; nd.ps = wd[w].hist; nd.pe = wd[w].len;
      cur[w] = nd;
   });
   int ncur = nwin;
   for (int depth = 0; depth < 6 && ncur > 0; depth++) {
      /* S1: node totals, check-point layout */
#ifndef ZB_EMU
      if (g_zb_prof_on) { zb_tag("split_nodes"); zb_prof_begin(0, st); }
      zb_split_nodes_k<<<(unsigned)((ncur + ZB_WT / 32 - 1) / (ZB_WT / 32)), ZB_WT, 0, st>>>(cur, ncur, nh, gv);
      if (g_zb_prof_on) zb_prof_end(st);
      zb_count_launch(1);
      ZB_CUDA_CHECK(cudaGetLastError());
#else
      zb_launch(st, ncur, ZB_LAMBDA(long x) {
         ZbNode nd = cur[x];
         nd.nchk = 0; nd.best_tok = 0; nd.best_delta = 0; nd.t0 = 0;
         if (nd.pe - nd.ps >= 8192) {
            int *h = nh + (size_t)x * ZB_NH;
            gv.range_hist((int)nd.win, nd.ts, nd.te, h);
            h[ZB_EOB] += 1;
            ZbScratch s; int llen[ZB_NLIT], olen[ZB_NLIT];
            zb_huff_lengths(h, ZB_NLIT, llen, s.key);
            zb_huff_lengths(h + ZB_NLIT, ZB_NOFF, olen, s.key);
            nd.total_cost = zb_dynamic_cost(h, llen, h + ZB_NLIT, olen, s);
            /* first check: >= 256 tokens and >= 512 bytes consumed (blockdeflate.c:705), then every 256 tokens */
            const uint32_t ntok = nd.te - nd.ts;
            const uint32_t *a = gv.tp + gv.wtb[nd.win] + nd.ts;
            uint32_t t0 = 256;
            while (t0 <= ntok) {
               uint32_t endpos = t0 < ntok ? a[t0] : nd.pe;
               if (endpos - nd.ps >= 512) break;
               t0++;
            }
            if (t0 <= ntok) { nd.t0 = t0; nd.nchk = (ntok - t0) / 256 + 1; }
         }
         cur[x] = nd;
      });
#endif
      /* check record bases (serial, few nodes) */
      zb_launch(st, 1, ZB_LAMBDA(long) {
         uint32_t b = 0;
         for (int x = 0; x < ncur; x++) { cur[x].chk_base = b; b += cur[x].nchk; }
         cn[1] = b;
      });
      uint32_t nchk = 0;
      zb_d2h(st, &nchk, cn + 1, 4); zb_sync(st);
      int nnext = 0;
      if (nchk > 0) {
         chk_stat.need((size_t)nchk * 18); chk_flag.need(nchk); chk_delta.need(2 * (size_t)nchk); chk_node.need(nchk);
         if (zb_failed()) return;
         uint16_t *cs = chk_stat.p; uint8_t *cf = chk_flag.p; int *cdl = chk_delta.p; uint32_t *cnode = chk_node.p;
         /* node of every check point: the last node whose base is <= c and that has check points (bases ascend with the node index) */
         zb_launch(st, nchk, ZB_LAMBDA(long c) {
            int lo = 0, hi = ncur - 1;
            while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (cur[mid].chk_base <= (uint32_t)c) lo = mid; else hi = mid - 1; }
            while (cur[lo].nchk == 0) lo--;      /* nodes without check points share the base of the next one */
            cnode[c] = (uint32_t)lo;
         }, 256);
         /* S2: 18-bin statistics of each check interval (blockdeflate.c:686-703) */
         zb_launch(st, nchk, ZB_LAMBDA(long c) {
            const ZbNode nd = cur[cnode[c]];
            const uint32_t k = (uint32_t)c - nd.chk_base;
            const uint32_t t1 = k == 0 ? 0 : nd.t0 + 256 * (k - 1), t2 = nd.t0 + 256 * k;
            /* the 18 counters (each <= 512: an interval is 256 tokens, the first one at most 512 - 512 bytes are consumed by then)
               packed four to a 64-bit word and bumped by a shifted add: an indexed local array would live in local memory */
            uint64_t w0 = 0, w1 = 0, w2 = 0, w3 = 0, w4 = 0;
            const uint32_t gb = gv.wbs[nd.win]; const uint8_t *t = gv.T + gv.wd[nd.win].in_off;
            const uint32_t *a = gv.tp + gv.wtb[nd.win] + nd.ts;
            for (uint32_t q = t1; q < t2; q++) {
               const uint32_t p = a[q], l = gv.gl[gb + p];
               uint32_t idx;
               if (l >= ZB_MIN_MATCH) idx = l >= 9 ? 17u : 16u;
               else { const uint32_t b = t[p]; idx = ((b >> 4) & 0xcu) | (b & 3u); }
               const uint64_t one = (uint64_t)1 << ((idx & 3u) * 16u);
               const uint32_t wsel = idx >> 2;
               w0 += wsel == 0 ? one : 0; w1 += wsel == 1 ? one : 0; w2 += wsel == 2 ? one : 0; w3 += wsel == 3 ? one : 0; w4 += wsel == 4 ? one : 0;
            }
            uint16_t *dst = cs + (size_t)c * 18;
            for (int i = 0; i < 4; i++) { dst[i] = (uint16_t)(w0 >> (16 * i)); dst[4 + i] = (uint16_t)(w1 >> (16 * i)); dst[8 + i] = (uint16_t)(w2 >> (16 * i)); dst[12 + i] = (uint16_t)(w3 >> (16 * i)); }
            dst[16] = (uint16_t)w4; dst[17] = (uint16_t)(w4 >> 16);
         });
         /* S3: drift test per check point (blockdeflate.c:706-721, unsigned arithmetic) */
#ifndef ZB_EMU
         if (g_zb_prof_on) { zb_tag("split_drift"); zb_prof_begin(0, st); }
         zb_split_drift_k<<<(unsigned)((ncur + 3) / 4), 128, 0, st>>>(cur, ncur, cs, cf);
         if (g_zb_prof_on) zb_prof_end(st);
         zb_count_launch(1);
         ZB_CUDA_CHECK(cudaGetLastError());
#else
         zb_launch(st, ncur, ZB_LAMBDA(long x) {
            const ZbNode nd = cur[x];
            uint32_t stat[18], nstat = 0;
            for (int i = 0; i < 18; i++) stat[i] = 0;
            for (uint32_t k = 0; k < nd.nchk; k++) {
               const uint16_t *ns = cs + (size_t)(nd.chk_base + k) * 18;
               const uint32_t nnew = k == 0 ? nd.t0 : 256;
               uint8_t flag = 0;
               if (nstat) {
                  uint32_t tot = 0;
                  for (int j = 0; j < 18; j++) {
                     uint32_t e = stat[j] * nnew, a = (uint32_t)ns[j] * nstat;
                     tot += e > a ? e - a : a - e;
                  }
                  if ((tot / nnew) >= (nstat * 45 / 100)) flag = 1;   /* nLastGoodSplitIdx >= 0 holds from the 2nd check on */
               }
               cf[nd.chk_base + k] = flag;
               for (int j = 0; j < 18; j++) { nstat += ns[j]; stat[j] += ns[j]; }
            }
         });
#endif
         /* S4: cost delta of splitting at the PREVIOUS check point (blockdeflate.c:724-757) */
#ifndef ZB_EMU
         if (g_zb_prof_on) { zb_tag("split_eval"); zb_prof_begin(0, st); }
         zb_split_eval_k<<<(unsigned)((2L * nchk + ZB_WT / 32 - 1) / (ZB_WT / 32)), ZB_WT, 0, st>>>(cur, 2L * nchk, cf, cnode, nh, cdl, gv);
         if (g_zb_prof_on) zb_prof_end(st);
         zb_count_launch(1);
         ZB_CUDA_CHECK(cudaGetLastError());
#else
         zb_tag("split_eval");
         zb_launch(st, 2L * nchk, ZB_LAMBDA(long y) {      /* one task per side of a candidate: the two are independent */
            const long c = y >> 1; const int right_side = (int)(y & 1);
            cdl[y] = -1;
            if (!cf[c]) return;
            const uint32_t x = cnode[c];
            const ZbNode nd = cur[x];
            const uint32_t k = (uint32_t)c - nd.chk_base;   /* k >= 1 here */
            const uint32_t tsplit = nd.t0 + 256 * (k - 1);   /* tokens left of the split */
            int h[ZB_NH];
            gv.range_hist((int)nd.win, nd.ts, nd.ts + tsplit, h);
            if (right_side) {
               const int *tot = nh + (size_t)x * ZB_NH;
               for (int i = 0; i < ZB_NH; i++) h[i] = tot[i] - h[i];
            }
            h[ZB_EOB] = 1;
            ZbScratch s; int llen[ZB_NLIT], olen[ZB_NLIT];
            zb_huff_lengths(h, ZB_NLIT, llen, s.key);
            zb_huff_lengths(h + ZB_NLIT, ZB_NOFF, olen, s.key);
            cdl[y] = zb_dynamic_cost(h, llen, h + ZB_NLIT, olen, s);
         }, 64);
#endif
         /* S5: best candidate per node (first maximum, delta >= 0), emit children */
         zb_memset(st, cn + 2, 0, 4);
         uint32_t *wsp = wsplit.p, *wns = wnsplit.p;
         zb_launch(st, ncur, ZB_LAMBDA(long x) {
            ZbNode nd = cur[x];
            int best = -1; uint32_t bestk = 0;
            for (uint32_t k = 1; k < nd.nchk; k++) {
               if (!cf[nd.chk_base + k]) continue;
               int d = nd.total_cost - (cdl[2 * (nd.chk_base + k)] + cdl[2 * (nd.chk_base + k) + 1]);
               if (d >= 0 && (best < 0 || best < d)) { if (best < 0 || best < d) { best = d; bestk = k; } }
            }
            if (best >= 0) {
               const uint32_t tsplit = nd.t0 + 256 * (bestk - 1);
               const uint32_t *a = gv.tp + gv.wtb[nd.win] + nd.ts;
               const uint32_t psplit = a[tsplit];
               uint32_t slot = zb_atomic_add(wns + nd.win, 1u);
               wsp[(size_t)nd.win * ZB_MAXSB + slot] = psplit;
               if (nd.depth + 1 < 6) {   /* deeper frames return at once (blockdeflate.c:646) */
                  uint32_t o = zb_atomic_add(cn + 2, 2u);
                  ZbNode l = nd, r = nd;
                  l.depth = r.depth = nd.depth + 1;
                  l.te = nd.ts + tsplit; l.pe = psplit;
                  r.ts = nd.ts + tsplit; r.ps = psplit;
                  nxt[o] = l; nxt[o + 1] = r;
               }
            }
         });
         uint32_t nn = 0;
         zb_d2h(st, &nn, cn + 2, 4); zb_sync(st);
         nnext = (int)nn;
      }
      std::swap(cur, nxt);
      ncur = nnext;
   }
   /* sub-block list, in stream order */
   ZbSub *sb = sub.p; uint32_t *wsp = wsplit.p, *wns = wnsplit.p;
   /* per window: sort its split offsets and count its sub-blocks; exclusive sum -> first sub-block of every window; per
      window again: fill its sub-blocks (windows are independent, only the numbering runs through them) */
   uint32_t *wsc = wsubcnt.p, *wsbase = wsubbase.p;
   zb_launch(st, nw, ZB_LAMBDA(long w) {
      uint32_t *sp = wsp + (size_t)w * ZB_MAXSB;
      const uint32_t ns = wns[w];
      for (uint32_t i = 1; i < ns; i++) { uint32_t v = sp[i]; uint32_t j = i; while (j > 0 && sp[j - 1] > v) { sp[j] = sp[j - 1]; j--; } sp[j] = v; }
      wsc[w] = ns + 1;
   });
   zb_exclusive_sum(st, wsc, wsbase, nw, cn + 3, scratch.p);
   zb_launch(st, nw, ZB_LAMBDA(long w) {
      const uint32_t *sp = wsp + (size_t)w * ZB_MAXSB;
      const uint32_t ns = wns[w];
      uint32_t n = wsbase[w];
      uint32_t start = wd[w].hist;
      const uint32_t ntok = wtb[w + 1] - wtb[w];
      uint32_t ts = gv.tok_of_pos((int)w, start, ntok);
      for (uint32_t i = 0; i <= ns; i++) {
         uint32_t end = i < ns ? sp[i] : wd[w].len;
         ZbSub s; memset(&s, 0, sizeof(s));
         s.win = (uint32_t)w; s.idx_in_win = i; s.ps = start; s.pe = end;
         s.ts = ts; s.te = end < wd[w].len ? gv.tok_of_pos((int)w, end, ntok) : ntok;
         sb[n++] = s;
         start = end; ts = s.te;
      }
   });
   uint32_t ns = 0;
   zb_d2h(st, &ns, cn + 3, 4); zb_sync(st);
   nsub = (int)ns;
}

/* ============================================================ optimal parse ============================================================ */

/* walk the chosen path of one path-chunk: calls f(p, len, off) for every token starting in [entry, hi) */
template <class F>
ZB_HD void zb_walk_best(const zb_match_t *best, uint32_t entry, uint32_t hi, F &f) {
   for (uint32_t p = entry; p < hi;) {
      zb_match_t m = best[p];
      if (m.length >= ZB_MIN_MATCH) { f(p, (uint32_t)m.length, (uint32_t)m.offset); p += m.length; }
      else { f(p, 0u, 0u); p++; }
   }
}

#ifndef ZB_EMU
/* ---- candidate records: once per batch, one thread per position of every sub-block (zb_cand_pack, zb_core.h) ---- */
__global__ void __launch_bounds__(256) zb_cand_k(long npch, const ZbSub *sb, const uint32_t *pcs, const uint32_t *wbs, const zb_match_t *mt, uint4 *cand, uint32_t cpv) {
   const long c = blockIdx.x;
   if (c >= npch) return;
   const ZbSub s = sb[pcs[c]];
   const uint32_t k = (uint32_t)c - s.pchunk_base, gb = wbs[s.win];
   const uint32_t lo = s.ps + k * cpv, hi = lo + cpv < s.pe ? lo + cpv : s.pe;
   for (uint32_t p = lo + threadIdx.x; p < hi; p += 256) {
      const ZbMatchRec rec = zb_load_rec(mt + ((size_t)gb << 3), (int)p);
      const ZbCand cd = zb_cand_pack(rec, (int)(s.pe - p));
      cand[gb + p] = make_uint4(cd.w[0], cd.w[1], cd.w[2], cd.w[3]);
   }
}

/* after the last pass: choice words -> {length, offset} (private.h:59), the offset fetched from the match list */
__global__ void __launch_bounds__(256) zb_choice_k(long npch, const ZbSub *sb, const uint32_t *pcs, const uint32_t *wbs, const zb_match_t *mt, uint32_t *bm, uint32_t cpv) {
   const long c = blockIdx.x;
   if (c >= npch) return;
   const ZbSub s = sb[pcs[c]];
   const uint32_t k = (uint32_t)c - s.pchunk_base, gb = wbs[s.win];
   const uint32_t lo = s.ps + k * cpv, hi = lo + cpv < s.pe ? lo + cpv : s.pe;
   for (uint32_t p = lo + threadIdx.x; p < hi; p += 256) {
      const uint32_t w = bm[gb + p];
      uint32_t v = 0;
      if (w) v = (w & 511u) | ((uint32_t)mt[((size_t)(gb + p) << 3) + (w >> 14)].offset << 16);
      bm[gb + p] = v;
   }
}

/* ---- chunked backward recurrence, one thread per parse chunk (32 independent chunks per warp) ----
 * Every thread is one long dependent chain, so the kernel lives on instruction count and occupancy.  Per position a thread
 * reads a 16-byte candidate record (zb_cand_pack) and the literal byte, both fetched a position ahead; the costs of the last
 * 64 positions sit in a shared-memory ring ([slot][thread] u16: a warp's accesses fall into distinct banks up to the 2-way
 * u16 pairing) - short matches (< 40) only look 39 positions ahead - and every cost is also streamed to a global scratch row
 * ([step][thread], so a warp's store is one 64-byte line) from which the rare far reads of leave-alone matches (>= 40: one
 * cost, up to 258 ahead) and the two 259-entry signatures are taken.  A chunk starts from cost 0 and a step adds at most 15
 * bits, so with CD + ZB_WU <= 4368 steps the u16 costs never wrap and are compared as plain integers.
 * The candidate lengths of all short matches of a position share ONE prefix-minimum sweep: key = (cost[i + k] + lencost(k))
 * << 6 | 63 - k, one multiply-add and one minimum per length (the length cost and the tie-break come pre-combined out of a
 * per-sub-block table), the sweep pausing at every match's length to price that match.
 * Bit-cost tables: the CTA's 128 chunks belong to consecutive sub-blocks; their tables are copied to shared memory, one slot
 * each (the host sizes the dynamic shared memory by the largest number of sub-blocks any CTA spans - batches of small streams
 * span a dozen), and every lane uses the slot of its own sub-block. */
#define ZB_DP_THREADS 128
#define ZB_NR 64              /* near ring entries */
struct ZbDpTab { uint8_t lit[256]; uint8_t len[256]; uint8_t off[32]; uint32_t lenkey[40]; };   /* lenkey[k - 3] = lencost(k) << 6 | 63 - k */

/* the 259 relative costs at `pos0` (the signature two neighbouring chunks are compared by), read back from the scratch row:
   position p was done at step from - 1 - p; positions at and above `from` are the zero guess */
__device__ __forceinline__ void zb_dp_signature(int16_t *__restrict__ dst, size_t SS, const uint16_t *__restrict__ far0, int pos0, int from, int end, int t, uint32_t cprev, bool warm,
                                                const int qmax /* entries 0..qmax are written (the verify step reads no others of a warm signature) */,
                                                const int NT = ZB_DP_THREADS /* elements between consecutive steps of the cost row */) {
   /* loads batched 8 deep: each is an L2 round trip, and nothing else of this thread is in flight here */
   for (int q0 = 0; q0 <= qmax; q0 += 8) {
      uint32_t v[8];
#pragma unroll
      for (int j = 0; j < 8; j++) { const int tt = t - 1 - (q0 + j); v[j] = (tt >= 0 && q0 + j <= ZB_MAX_MATCH) ? (uint32_t)far0[(size_t)tt * NT] : 0u; }
#pragma unroll
      for (int j = 0; j < 8; j++) {
         const int q = q0 + j;
         const bool in = warm ? (pos0 + q <= end && pos0 + q <= from) : (pos0 + q <= end);
         if (q <= ZB_MAX_MATCH) dst[(size_t)q * SS] = in ? (int16_t)(uint16_t)(v[j] - cprev) : (int16_t)0;
      }
   }
}

/* positions [lo, from) of one chunk, descending; t = step of position from - 1 on entry.  All per-step addresses are running
   pointers (the cost row advances by one row, the records / text / choices retreat by one element, the ring slot by one slot
   modulo 64): the loop is instruction bound, and 64-bit address arithmetic from the position index was a fifth of it. */
__device__ __forceinline__ void zb_dp_range(const uint8_t *__restrict__ T, const uint4 *__restrict__ cand, const ZbDpTab *__restrict__ tab, int lo, int from,
                                            uint32_t *__restrict__ choice, uint16_t *ring0, uint16_t *far0, int &t_io, uint32_t &cprev_io, const bool KEEP) {
   const int NT = ZB_DP_THREADS;
   if (from - 1 < lo) return;
   int t = t_io;
   uint32_t cprev = cprev_io;                 /* cost of position i + 1 */
   const uint4 *pc = cand + (from - 1);
   const uint8_t *pt = T + (from - 1);
   uint32_t *pch = choice + (from - 1);
   uint16_t *pf = far0 + (size_t)t * NT;
   uint4 nxt = __ldg(pc);
   uint32_t nlit = *pt;
   const uint32_t *lenkey = tab->lenkey;
   uint32_t slot = (uint32_t)t & (ZB_NR - 1);  /* ring slot of the position being done */
   for (int n = from - lo; n > 0; n--, t++, pf += NT, pch--) {
      uint4 rec = nxt;
      const uint32_t lit = nlit;
      pc--; pt--;
      if (n > 1) { nxt = __ldg(pc); nlit = *pt; }
      uint32_t bestc = cprev + tab->lit[lit];
      uint32_t bestw = 0;
      if (rec.x) {
         uint32_t btla = 0xffffffffu, bwla = 0, bts = 0xffffffffu, bws = 0, curmin = 0xffffffffu, mla = 0;
         int k = ZB_MIN_MATCH;
         const int q = (int)((slot - ZB_MIN_MATCH) & (ZB_NR - 1));   /* slot of i + 3 (a slot not written yet reads as the zero guess) */
         const uint16_t *pr = ring0 + q * NT;                       /* slot of i + k, moving down by NT per k */
         int kw = k + q + 1;                                        /* first k whose slot wraps */
         uint32_t e = rec.x & 0xffffu;
#pragma unroll 1
         do {
            const uint32_t offc = tab->off[e & 31u];
            if (e & 0x8000u) {      /* leave-alone match: its one length */
               const int ml = (int)((e >> 5) & 511u);
               const int lidx = ml >= ZB_MIN_MATCH ? ml - ZB_MIN_MATCH : 255;
               uint32_t cv;
               if (ml < ZB_NR) cv = ring0[((slot - (uint32_t)ml) & (ZB_NR - 1)) * NT];
               else cv = t >= ml ? (uint32_t)*(pf - (size_t)ml * NT) : 0u;      /* the row of step t - ml */
               const uint32_t total = (uint32_t)tab->len[lidx] + offc + cv;
               if (total < btla) { btla = total; bwla = (uint32_t)ml | ((e & 31u) << 9) | (mla << 14); }
               mla++;
            } else {                /* short match: extend the shared sweep to its length, then price it */
               const int ml = (int)((e >> 5) & 63u);
               while (k <= ml) {
                  const int kstop = ml < kw - 1 ? ml : kw - 1;
#pragma unroll 2
                  for (; k <= kstop; k++, pr -= NT) {
                     const uint32_t key = ((uint32_t)*pr << 6) + lenkey[k - ZB_MIN_MATCH];
                     curmin = key < curmin ? key : curmin;
                  }
                  if (k == kw) { pr += ZB_NR * NT; kw += ZB_NR; }
               }
               const uint32_t total = (curmin >> 6) + offc;
               if (total <= bts) { bts = total; bws = (63u - (curmin & 63u)) | ((e & 31u) << 9) | (((e >> 11) & 7u) << 14); }
            }
            /* next entry: the record shifts down by 16 bits */
            rec.x = __funnelshift_r(rec.x, rec.y, 16); rec.y = __funnelshift_r(rec.y, rec.z, 16); rec.z = __funnelshift_r(rec.z, rec.w, 16); rec.w >>= 16;
            e = rec.x & 0xffffu;
         } while (e);
         if (bts < btla) { btla = bts; bwla = bws; }
         if (btla < bestc) { bestc = btla; bestw = bwla; }
      }
      ring0[slot * NT] = (uint16_t)bestc;
      *pf = (uint16_t)bestc;
      slot = (slot + 1) & (ZB_NR - 1);
      cprev = bestc;
      if (KEEP) *pch = bestw;
   }
   t_io = t; cprev_io = cprev;
}

/* unroll 2 of the sweep at 7 CTAs per SM (62 registers) measured fastest on B200 */
__global__ void __launch_bounds__(ZB_DP_THREADS, 7) zb_parse_dp_k(const ZbSub *sb, const ZbSubTabs *tb, const uint32_t *dcs, long ndch, int pass, const ZbWinDesc *wd,
                                                            const uint32_t *wbs, const uint8_t *T, const uint4 *cand, uint32_t *bm, int16_t *sgt, int16_t *sgw,
                                                            size_t SS, uint16_t *far, int CD, int nslot, const int *reach) {
   extern __shared__ __align__(16) uint8_t zb_dp_sm[];
   uint16_t *ring_s = (uint16_t *)zb_dp_sm;                                   /* [ZB_NR][ZB_DP_THREADS] */
   ZbDpTab *tab_s = (ZbDpTab *)(zb_dp_sm + ZB_NR * ZB_DP_THREADS * 2);        /* [nslot] */
   const long c0 = (long)blockIdx.x * ZB_DP_THREADS, c = c0 + threadIdx.x;
   const long clast = (c0 + ZB_DP_THREADS < ndch ? c0 + ZB_DP_THREADS : ndch) - 1;
   const uint32_t x0 = dcs[c0], x1 = dcs[clast];
   int ns = (int)(x1 - x0) + 1; if (ns > nslot) ns = nslot;                   /* never more than nslot (the host sized it by the maximum) */
   for (int sl = 0; sl < ns; sl++) {
      const uint32_t *src = (const uint32_t *)&tb[x0 + sl].cost; uint32_t *dstw = (uint32_t *)&tab_s[sl];
      for (int e = threadIdx.x; e < (int)(sizeof(ZbCostTab) / 4); e += ZB_DP_THREADS) dstw[e] = src[e];
      if (threadIdx.x < 40) { const int k = ZB_MIN_MATCH + threadIdx.x; tab_s[sl].lenkey[threadIdx.x] = ((uint32_t)tb[x0 + sl].cost.len[threadIdx.x] << 6) | (uint32_t)(63 - (k < 63 ? k : 63)); }
   }
   uint16_t *ring0 = ring_s + threadIdx.x;
   for (int e = 0; e < ZB_NR; e++) ring0[e * ZB_DP_THREADS] = 0;
   __syncthreads();
   if (c >= ndch) return;
   const uint32_t x = dcs[c];
   const ZbSub s = sb[x];
   if (pass > 0 && !s.is_dyn) return;
   const ZbDpTab *tab = &tab_s[x - x0];
   const uint32_t k = (uint32_t)c - s.dchunk_base;
   const uint32_t gb = wbs[s.win];
   const uint8_t *t = T + wd[s.win].in_off;
   const int lo = (int)(s.ps + k * CD);
   const int hi = (int)(lo + CD < (int)s.pe ? lo + CD : (int)s.pe);
   const int end = (int)s.pe;
   /* adaptive warm-up: the chunk only reads costs up to `reach` positions past its end, so only those have to be right, and
      the warm-up is the settling margin above THEM instead of above the full 258-position horizon */
   const int rc = reach[c];
   int from = hi + zb_warmup_len(rc); if (from > end) from = end;
   uint16_t *far0 = far + (size_t)blockIdx.x * (size_t)(CD + ZB_WU) * ZB_DP_THREADS + threadIdx.x;
   int16_t *sw = sgw + (size_t)c, *sg = sgt + (size_t)c;
   int step = 0; uint32_t cprev = 0;
   /* warm-up [hi, from) then the chunk [lo, hi): ONE copy of the recurrence (the two phases as iterations of a loop that is
      not unrolled) - the kernel is instruction-issue bound and its code should stay inside the I-cache */
#pragma unroll 1
   for (int phase = 0; phase < 2; phase++) {
      zb_dp_range(t, cand + gb, tab, phase ? lo : hi, phase ? hi : from, bm + gb, ring0, far0, step, cprev, phase != 0);
      zb_dp_signature(phase ? sg : sw, SS, far0, phase ? lo : hi, from, end, step, cprev, phase == 0, phase ? ZB_MAX_MATCH : rc);
   }
}

/* ---- repair of wrong chunks: the same recurrence, ONE WARP per chain ----
 * Chunks whose warm-up did not re-synchronise (byte runs, periodic records: the state never forgets the phase it was
 * started with) have to be redone from their right neighbour's true costs, one after the other.  That is a serial chain,
 * so what matters is the latency of one position, not throughput: a warp owns the chain, its 260-entry cost ring lives in
 * shared memory, lanes 0..7 decode one match of the position each, the candidate lengths k = 3.. of the short matches are
 * spread over the 32 lanes and reduced with redux.sync (min), one reduction per (step, match).  Key = cost << 6 | (63 - k)
 * so that the larger k wins ties - the first one met going down from the match length, as the reference's loop does
 * (blockdeflate.c:292-312); matches are then combined in index order on strictly lower cost, literal first.  Control flow
 * is uniform across the warp.  ~20x lower latency per position than the thread-per-chunk kernel. */
#define ZB_DW_THREADS 128
#define ZB_DW_WARPS (ZB_DW_THREADS / 32)
#define ZB_DW_INF 0x7fffffffu
#define ZB_DW_FAR_INF 0x3fffffff

#define ZB_DW_RING 576         /* costs of the last 576 positions: 259 for the recurrence, 517 + a block for the run shortcut below */
struct ZbDwShared {            /* per warp */
   uint16_t ring[ZB_DW_RING];
   uint32_t info[32][ZB_NMATCH + 1];  /* decoded matches of the 32 positions of the current block (+1: bank spread) */
   uint32_t meta[32];                 /* M | K << 4 | literal cost << 16 */
   ZbCostTab tab;                     /* the sub-block's bit costs */
   uint32_t pch[ZB_MAX_MATCH + 2];    /* byte-run shortcut: the 258 choice words one period of the run repeats (ZbDwUni::aE anchors them) */
};

/* Positions [lo, from) of one sub-block, descending.  Per block of 32 positions the lanes first decode one position each, in
   parallel and off the serial chain: valid-match count M, longest short length K, and per match a word
   {clamped length (9 bits) | leave-alone flag | fixed cost (6 bits: offset cost, plus the length cost for a leave-alone
   match) | offset (16 bits)}.  What stays serial per position is: ring reads, one redux per short match, a few compares,
   one ring write. */
/* Byte runs.  Inside a long run every position has the same match record and the same literal, so the recurrence is a fixed map
   applied over and over: once the 259 relative costs at a position equal those 258 positions above it (the length of the run's
   one match), every choice below repeats the choice 258 above and every cost is that cost plus a constant, for as long as the
   records stay the same.  The walker tracks the stretch of identical records it is in (whole blocks of 32), tests that
   periodicity once the stretch is 517 positions long, and from then on copies 32 choices per step instead of scanning them -
   a 64 KiB run of a mozilla-shaped input is one serial chain of 128 chunks, and this chain is what the repair's time is. */
struct ZbDwUni { uint4 ra, rb; uint32_t rl, delta; int len, top; bool periodic; int aE; bool a_valid; };   /* pch[j] = choice of position aE + 1 + j, while a_valid */

__device__ __forceinline__ void zb_dw_run(const uint8_t *__restrict__ t, const zb_match_t *__restrict__ match, int lo, int from, int end,
                                          zb_match_t *__restrict__ best, ZbDwShared &sh, int &slot, ZbDwUni &U, const int lane,
                                          const int pf_lo /* first position of the sub-block: L2 prefetches may run ahead of this chunk into the next ones of the chain */) {
   int s = slot;
   if (from <= lo) return;
   uint16_t *ring = sh.ring;
   const ZbCostTab &tab = sh.tab;
   /* length costs of the candidate lengths this lane evaluates: k = 3 + lane and k = 35 + lane */
   const int lcA = (int)tab.len[lane];
   const int lcB = lane < 5 ? (int)tab.len[32 + lane] : 0;
   /* records are fetched a block of 32 positions ahead (DRAM latency is several positions long): lane x holds position i0 - x */
   uint4 na = make_uint4(0u, 0u, 0u, 0u), nb = na; uint32_t nl = 0;
   {
      const int p = from - 1 - lane;
      if (p >= lo) { const uint4 *q = (const uint4 *)(match + ((size_t)p << 3)); na = __ldg(q); nb = __ldg(q + 1); nl = t[p]; }
   }
   uint32_t base = ring[s];       /* cost of the position above the next one to do: carried in a register */
   bool far_ok = true; int farE = ZB_DW_FAR_INF, lita = 0; uint32_t farw = 0u;
   /* after a block done the long way: count it into the stretch of identical records and, once the stretch spans 517 positions
      (none of them clamped by the sub-block end), test whether the cost window has become 258-periodic: cost[ib + q] -
      cost[ib + 258 + q] the same for q = 0..258, ib = the block's lowest position (slot s) */
#define ZB_DW_STRETCH() do { \
      if (cont || (U.len == 0 && U.top == i0)) U.len += nb_pos; \
      if (U.len >= 2 * ZB_MAX_MATCH + 1 && !U.periodic && end - U.top >= ZB_MAX_MATCH) { \
         __syncwarp(); \
         int s258_ = s - ZB_MAX_MATCH; if (s258_ < 0) s258_ += ZB_DW_RING; \
         const uint32_t d_ = ((uint32_t)ring[s] - (uint32_t)ring[s258_]) & 0xffffu; \
         bool ok_ = true; \
         for (int q_ = lane; q_ <= ZB_MAX_MATCH; q_ += 32) { \
            int x_ = s - q_; if (x_ < 0) x_ += ZB_DW_RING; \
            int y_ = x_ - ZB_MAX_MATCH; if (y_ < 0) y_ += ZB_DW_RING; \
            if ((((uint32_t)ring[x_] - (uint32_t)ring[y_]) & 0xffffu) != d_) ok_ = false; \
         } \
         if (__all_sync(0xffffffffu, ok_)) { U.periodic = true; U.delta = d_; U.a_valid = false; } \
      } \
   } while (0)
   for (int i0 = from - 1; i0 >= lo;) {      /* every path below steps i0 itself */
      __syncwarp();
      const int nb_pos = i0 - lo + 1 < 32 ? i0 - lo + 1 : 32;
      bool cont;      /* this block consists of copies of ONE record, the same as the stretch before it */
      {
         const uint4 a0 = make_uint4(__shfl_sync(0xffffffffu, na.x, 0), __shfl_sync(0xffffffffu, na.y, 0), __shfl_sync(0xffffffffu, na.z, 0), __shfl_sync(0xffffffffu, na.w, 0));
         const uint4 b0 = make_uint4(__shfl_sync(0xffffffffu, nb.x, 0), __shfl_sync(0xffffffffu, nb.y, 0), __shfl_sync(0xffffffffu, nb.z, 0), __shfl_sync(0xffffffffu, nb.w, 0));
         const uint32_t l0 = __shfl_sync(0xffffffffu, nl, 0);
         const bool mine = lane >= nb_pos || (na.x == a0.x && na.y == a0.y && na.z == a0.z && na.w == a0.w && nb.x == b0.x && nb.y == b0.y && nb.z == b0.z && nb.w == b0.w && nl == l0);
         const bool uniform = __all_sync(0xffffffffu, mine);
         cont = uniform && U.len > 0 && a0.x == U.ra.x && a0.y == U.ra.y && a0.z == U.ra.z && a0.w == U.ra.w && b0.x == U.rb.x && b0.y == U.rb.y && b0.z == U.rb.z && b0.w == U.rb.w && l0 == U.rl;
         if (!uniform) { U.len = 0; U.periodic = false; U.a_valid = false; }
         else if (!cont) { U.ra = a0; U.rb = b0; U.rl = l0; U.len = 0; U.top = i0; U.periodic = false; U.a_valid = false; }
      }
      if (U.periodic && cont) {
         /* The run shortcut, four blocks (128 positions) a round while the chunk has them.  Inside the periodic stretch every
            choice is the choice 258 above it, i.e. one of the 258 choice words above the place the shortcut first applied: they
            are read once into shared memory (pch), so a round reads nothing it has just written - only the records, to see
            that the run goes on, and those are loaded ONE ROUND AHEAD (and pulled into L2 a kilobyte ahead): the chain no
            longer waits for a memory round trip per round (it did: ~1.5 us per 128 positions, 0.8 ms for a 64 KiB run). */
         bool wide = false;
         if (i0 - 127 >= lo) {
            if (!U.a_valid) {
               for (int j = lane; j < ZB_MAX_MATCH; j += 32) sh.pch[j] = ((const uint32_t *)best)[i0 + 1 + j];
               U.aE = i0; U.a_valid = true;
               __syncwarp();
            }
            uint4 ca[3], cb[3]; uint32_t cl[3];
#pragma unroll
            for (int k = 0; k < 3; k++) {
               const int p = i0 - 32 * (k + 1) - lane;
               const uint4 *q = (const uint4 *)(match + ((size_t)p << 3));
               ca[k] = __ldg(q); cb[k] = __ldg(q + 1); cl[k] = t[p];
            }
            while (i0 - 127 >= lo) {
               uint4 ya[4], yb[4]; uint32_t yl[4];      /* the next round's records */
#pragma unroll
               for (int k = 0; k < 4; k++) {
                  const int p = i0 - 128 - 32 * k - lane;
                  ya[k] = make_uint4(0u, 0u, 0u, 0u); yb[k] = ya[k]; yl[k] = 0;
                  if (p >= lo) { const uint4 *q = (const uint4 *)(match + ((size_t)p << 3)); ya[k] = __ldg(q); yb[k] = __ldg(q + 1); yl[k] = t[p]; }
               }
#pragma unroll
               for (int k = 0; k < 4; k++) {
                  const int pf = i0 - 1024 - 32 * k - lane;
                  if (pf >= pf_lo) asm volatile("prefetch.global.L2 [%0];" :: "l"(match + ((size_t)pf << 3)));
               }
               bool okb = na.x == U.ra.x && na.y == U.ra.y && na.z == U.ra.z && na.w == U.ra.w && nb.x == U.rb.x && nb.y == U.rb.y && nb.z == U.rb.z && nb.w == U.rb.w && nl == U.rl;
#pragma unroll
               for (int k = 0; k < 3; k++)
                  okb = okb && ca[k].x == U.ra.x && ca[k].y == U.ra.y && ca[k].z == U.ra.z && ca[k].w == U.ra.w && cb[k].x == U.rb.x && cb[k].y == U.rb.y && cb[k].z == U.rb.z && cb[k].w == U.rb.w && cl[k] == U.rl;
               if (!__all_sync(0xffffffffu, okb)) break;      /* the single-block logic below takes it from here (this block is still `cont`) */
#pragma unroll
               for (int k = 0; k < 4; k++) {
                  int sl = s + 1 + 32 * k + lane; if (sl >= ZB_DW_RING) sl -= ZB_DW_RING;
                  int sh258 = sl - ZB_MAX_MATCH; if (sh258 < 0) sh258 += ZB_DW_RING;
                  ring[sl] = (uint16_t)((uint32_t)ring[sh258] + U.delta);
                  const int i = i0 - 32 * k - lane;
                  ((uint32_t *)best)[i] = sh.pch[ZB_MAX_MATCH - 1 - (U.aE - i) % ZB_MAX_MATCH];
               }
               wide = true;
               i0 -= 128;
               s += 128; if (s >= ZB_DW_RING) s -= ZB_DW_RING;
               U.len += 128;
               na = ya[0]; nb = yb[0]; nl = yl[0];
#pragma unroll
               for (int k = 0; k < 3; k++) { ca[k] = ya[k + 1]; cb[k] = yb[k + 1]; cl[k] = yl[k + 1]; }
               __syncwarp();
               base = ring[s];
            }
         }
         if (wide) continue;      /* a fresh look at the block now at i0 (its records are loaded) */
      }
      if (U.periodic && cont) {
         /* the run shortcut: choice and cost of position i = those of position i + 258 (+ delta) */
         if (lane < nb_pos) {
            const int i = i0 - lane;
            int sl = s + 1 + lane; if (sl >= ZB_DW_RING) sl -= ZB_DW_RING;
            int sh258 = sl - ZB_MAX_MATCH; if (sh258 < 0) sh258 += ZB_DW_RING;
            ring[sl] = (uint16_t)((uint32_t)ring[sh258] + U.delta);
            ((uint32_t *)best)[i] = ((const uint32_t *)best)[i + ZB_MAX_MATCH];
         }
         {
            const int p = i0 - 32 - lane;
            if (p >= lo) { const uint4 *q = (const uint4 *)(match + ((size_t)p << 3)); na = __ldg(q); nb = __ldg(q + 1); nl = t[p]; }
         }
         s += nb_pos; if (s >= ZB_DW_RING) s -= ZB_DW_RING;
         __syncwarp();
         base = ring[s];
         U.len += nb_pos;
         i0 -= 32;
         continue;
      }
      {  /* decode position i0 - lane */
         const int i = i0 - lane;
         const uint32_t w[ZB_NMATCH] = {na.x, na.y, na.z, na.w, nb.x, nb.y, nb.z, nb.w};
         far_ok = true; farE = ZB_DW_FAR_INF; farw = 0u;
         const int rem = end - i;
         int M = 0, K = 0;
#pragma unroll
         for (int m = 0; m < ZB_NMATCH; m++) {
            const int len0 = (int)(w[m] & 0xffffu), off0 = (int)(w[m] >> 16);
            uint32_t inf = 0;
            if (M == m && len0 >= ZB_MIN_MATCH && i >= lo) {
               M = m + 1;
               const int ml = len0 < rem ? len0 : rem;
               const bool lg = len0 >= ZB_LEAVE_ALONE;
               const uint32_t osym = (uint32_t)zb_off_sym((uint32_t)off0);
               int fixed = (int)tab.off[osym];
               if (lg) { int lidx = ml - ZB_MIN_MATCH; if (lidx < 0 || lidx > 255) lidx = 255; fixed += (int)tab.len[lidx]; }
               else if (ml > K) K = ml;
               inf = (uint32_t)ml | ((lg ? 1u : 0u) << 9) | ((uint32_t)fixed << 10) | (osym << 16) | ((uint32_t)m << 21);      /* bits 16..: what the choice word needs */
               /* far candidate: a leave-alone match that lands past the block's top position is already final */
               if (lg && ml > lane) {
                  int idx = s - (ml - 1 - lane); if (idx < 0) idx += ZB_DW_RING;
                  const int total = fixed + (int)(int16_t)(uint16_t)((uint32_t)ring[idx] - base);
                  if (total < farE) { farE = total; farw = (uint32_t)ml | (osym << 9) | ((uint32_t)m << 14); }
               } else far_ok = false;
            }
            sh.info[lane][m] = inf;
         }
         lita = (int)tab.lit[nl & 0xffu];
         sh.meta[lane] = (uint32_t)M | ((uint32_t)K << 4) | ((uint32_t)lita << 16);
         if (i < lo) { lita = 0; farE = ZB_DW_FAR_INF; }
      }
      {
         const int p = i0 - 32 - lane;
         if (p >= lo) { const uint4 *q = (const uint4 *)(match + ((size_t)p << 3)); na = __ldg(q); nb = __ldg(q + 1); nl = t[p]; }
         /* a scan block is over long before a DRAM round trip: the records of the blocks further ahead are pulled into L2 now,
            so that the register prefetch above only ever waits for L2 */
         const int pf = i0 - 32 * 6 - lane;
         if (pf >= pf_lo) asm volatile("prefetch.global.L2 [%0];" :: "l"(match + ((size_t)pf << 3)));
         if (lane == 0 && pf >= pf_lo + 31) asm volatile("prefetch.global.L2 [%0];" :: "l"(t + pf - 31));
      }
      __syncwarp();
      uint32_t outw = 0;      /* lane x keeps the choice of position i0 - x: one coalesced store per block */
      if (__all_sync(0xffffffffu, far_ok)) {
         /* Every candidate of every position of the block is either its literal or a leave-alone match landing above the
            block (byte runs, long periodic repeats - exactly the data that does not re-synchronise).  Position i0 - x then maps
            the cost c above it to min(c + lit, far): these maps compose ((A, B) : c -> min(c + A, B)), so the 32 positions are
            one warp scan instead of 32 serial steps.  Costs are relative to `base` = cost[i0 + 1]. */
         int A = lita, B = farE;
#pragma unroll
         for (int d = 1; d < 32; d <<= 1) {
            const int pa = __shfl_up_sync(0xffffffffu, A, d), pb = __shfl_up_sync(0xffffffffu, B, d);
            if (lane >= d) { const int nbv = pb + A; B = nbv < B ? nbv : B; A = pa + A; }
         }
         const int r = A < B ? A : B;                    /* cost[i0 - lane] - base */
         int cin = __shfl_up_sync(0xffffffffu, r, 1); if (lane == 0) cin = 0;
         if (farE < cin + lita) outw = farw;             /* literal first, a match only on strictly lower cost */
         if (lane < nb_pos) {
            int sl = s + 1 + lane; if (sl >= ZB_DW_RING) sl -= ZB_DW_RING;
            ring[sl] = (uint16_t)(base + (uint32_t)r);
            ((uint32_t *)best)[i0 - lane] = outw;
         }
         base = (base + (uint32_t)__shfl_sync(0xffffffffu, r, nb_pos - 1)) & 0xffffu;
         s += nb_pos; if (s >= ZB_DW_RING) s -= ZB_DW_RING;
         ZB_DW_STRETCH();
         i0 -= 32;
         continue;
      }
      /* what the lanes decoded for the block's positions is read one position ahead: the position's own chain (ring reads,
         pricing, one reduction, ring write) then starts with its inputs already in registers */
      uint32_t meta_n = sh.meta[0], infs_n[ZB_NMATCH];
#pragma unroll
      for (int m = 0; m < ZB_NMATCH; m++) infs_n[m] = sh.info[0][m];
      for (int x = 0; x < nb_pos; x++) {
         const uint32_t meta = meta_n;
         uint32_t infs[ZB_NMATCH];
#pragma unroll
         for (int m = 0; m < ZB_NMATCH; m++) infs[m] = infs_n[m];
         {
            const int xn = x + 1 < 32 ? x + 1 : 31;
            meta_n = sh.meta[xn];
#pragma unroll
            for (int m = 0; m < ZB_NMATCH; m++) infs_n[m] = sh.info[xn][m];
         }
         const int M = (int)(meta & 15u), K = (int)((meta >> 4) & 0xfffu);
         const int s1 = s;                           /* slot of i+1 */
         s = s1 + 1; if (s >= ZB_DW_RING) s -= ZB_DW_RING;
         int bestc = (int)(meta >> 16), bl = 0, bo = 0;
         if (M) {
            /* ONE reduction per position: lane L prices the candidate lengths k = 3 + L and 35 + L of every short match that is
               long enough, lane m the one length of leave-alone match m; key = (cost << 9) | (m << 6) | (63 - k), so the minimum is
               the cheapest candidate, among equals the earliest match, then its longest length - the reference's order
               (blockdeflate.c:272-312).  (A reduction per match made a position with 8 matches cost 800 cycles.) */
            uint32_t valA = ZB_DW_INF, valB = ZB_DW_INF;      /* cost[i + k] - cost[i + 1] + lencost(k) + 8192 */
            const int k = ZB_MIN_MATCH + lane, k2 = k + 32;
            if (k <= K) {
               int idx = s1 - (k - 1); if (idx < 0) idx += ZB_DW_RING;
               valA = (uint32_t)((int)(int16_t)(uint16_t)((uint32_t)ring[idx] - base) + lcA + 8192);
            }
            if (k2 <= K) {
               int idx = s1 - (k2 - 1); if (idx < 0) idx += ZB_DW_RING;
               valB = (uint32_t)((int)(int16_t)(uint16_t)((uint32_t)ring[idx] - base) + lcB + 8192);
            }
            uint32_t key = 0xffffffffu;
#pragma unroll
            for (int m = 0; m < ZB_NMATCH; m++) {
               if (m >= M) break;                /* M is warp-uniform */
               const uint32_t inf = infs[m];
               const int mlm = (int)(inf & 511u);
               const uint32_t fixed = (inf >> 10) & 63u;
               if ((inf >> 9) & 1u) {   /* >= 40: only the full (clamped) length, even below 3 (SURVEY A-3) */
                  if (lane == m) {
                     int idx = s1 - (mlm - 1); if (idx < 0) idx += ZB_DW_RING;
                     const uint32_t cv = mlm == 1 ? base : (uint32_t)ring[idx];     /* cost[i+1] is the register copy */
                     const uint32_t c = ((uint32_t)((int)fixed + (int)(int16_t)(uint16_t)(cv - base) + 8192) << 9) | ((uint32_t)m << 6);
                     key = c < key ? c : key;
                  }
               } else {
                  if (k <= mlm) { const uint32_t c = ((valA + fixed) << 9) | ((uint32_t)m << 6) | (uint32_t)(63 - k); key = c < key ? c : key; }
                  if (k2 <= mlm) { const uint32_t c = ((valB + fixed) << 9) | ((uint32_t)m << 6) | (uint32_t)(63 - k2); key = c < key ? c : key; }
               }
            }
            key = __reduce_min_sync(0xffffffffu, key);
            if (key != 0xffffffffu) {
               const int total = (int)(key >> 9) - 8192;
               if (total < bestc) {
                  const uint32_t inf = sh.info[x][(key >> 6) & 7u];      /* (a dynamic pick out of infs[] would go through local memory) */
                  bestc = total;
                  bl = ((inf >> 9) & 1u) ? (int)(inf & 511u) : 63 - (int)(key & 63u);
                  bo = (int)(inf >> 16);
               }
            }
         }
         base = (base + (uint32_t)bestc) & 0xffffu;
         if (lane == 0) ring[s] = (uint16_t)base;
         if (lane == x) outw = bl ? ((uint32_t)bl | (((uint32_t)bo & 31u) << 9) | (((uint32_t)bo >> 5) << 14)) : 0u;      /* choice word, as zb_parse_dp_k writes it */
         __syncwarp();
      }
      if (lane < nb_pos) ((uint32_t *)best)[i0 - lane] = outw;
      ZB_DW_STRETCH();
      i0 -= 32;
   }
#undef ZB_DW_STRETCH
   slot = s;
}

/* One warp per run of wrong chunks.  The warp of the run's rightmost chunk (its right neighbour is right) starts from that
   neighbour's true costs and walks left chunk after chunk, carrying the ring; past the run it goes on for as long as the
   chunk it enters had assumed other costs than the ones now known, and stops at a chunk another warp owns.  The caller
   verifies again afterwards, so a race with a neighbouring run costs a round, never correctness. */
__global__ void __launch_bounds__(ZB_DW_THREADS) zb_parse_fix_k(const ZbSub *sb, const ZbSubTabs *tb, const uint32_t *dcs, const uint32_t *badlist, int nbad, const uint8_t *ok,
                                                                const ZbWinDesc *wd, const uint32_t *wbs, const uint8_t *T, const zb_match_t *mt, zb_match_t *bm,
                                                                int16_t *sgt, int16_t *sgw, size_t SS, int CD, const int *reach) {
   __shared__ ZbDwShared sh_all[ZB_DW_WARPS];
   const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
   const long g = (long)blockIdx.x * ZB_DW_WARPS + wi;
   ZbDwShared &sh = sh_all[wi];
   uint16_t *ring = sh.ring;
   if (g >= nbad) return;
   long c = badlist[g];
   if (!ok[c + 1]) return;       /* not the head of its run: the head's warp will come through */
   const uint32_t x = dcs[c];
   const ZbSub s = sb[x];
   const uint32_t gb = wbs[s.win];
   const uint8_t *t = T + wd[s.win].in_off;
   const zb_match_t *m0 = mt + ((size_t)gb << 3);
   zb_match_t *b0 = bm + gb;
   const int end = (int)s.pe;
   int slot = 0;
   ZbDwUni U; U.ra = make_uint4(0u, 0u, 0u, 0u); U.rb = U.ra; U.rl = 0; U.delta = 0; U.len = 0; U.top = -1; U.periodic = false; U.aE = 0; U.a_valid = false;
   {
      const uint32_t *src = (const uint32_t *)&tb[x].cost; uint32_t *dstw = (uint32_t *)&sh.tab;
      for (int e = lane; e < (int)(sizeof(ZbCostTab) / 4); e += 32) dstw[e] = src[e];
      const int16_t *b = sgt + (size_t)(c + 1);
      int16_t *sw = sgw + (size_t)c;
      for (int e = lane; e < ZB_DW_RING; e += 32) ring[e] = 0;
      __syncwarp();
      for (int e = lane; e <= ZB_MAX_MATCH; e += 32) { int sl = slot - e; if (sl < 0) sl += ZB_DW_RING; const int16_t v = b[(size_t)e * SS]; ring[sl] = (uint16_t)v; sw[(size_t)e * SS] = v; }
   }
   __syncwarp();
   for (;;) {
      const int lo = (int)(s.ps + ((uint32_t)c - s.dchunk_base) * CD), hi = lo + CD;
      const bool has_nx = (uint32_t)c != s.dchunk_base;
      const uint8_t ok_c = ok[c], ok_nx = has_nx ? ok[c - 1] : (uint8_t)0;      /* asked for before the chunk's walk, there after it */
      zb_dw_run(t, m0, lo, hi, end, b0, sh, slot, U, lane, (int)s.ps);
      /* this chunk's true costs at its start */
      const uint16_t b = ring[slot];
      int16_t *sg = sgt + (size_t)c;
      for (int e = lane; e <= ZB_MAX_MATCH; e += 32) {
         int sl = slot - e; if (sl < 0) sl += ZB_DW_RING;
         sg[(size_t)e * SS] = (lo + e <= end) ? (int16_t)(uint16_t)(ring[sl] - b) : (int16_t)0;
      }
      if (!has_nx) break;
      const long nx = c - 1;
      if (!ok_nx && ok_c) break;   /* c had been right, so nx heads a run of its own: another warp owns it */
      int16_t *sw = sgw + (size_t)nx;
      if (ok_nx) {      /* (inside a run of wrong chunks nx is redone whatever it had assumed: no reason to wait for its 259 loads) */
         bool same = true;
         const int lim = reach[nx];      /* nx reads no cost further out (adaptive warm-up, stage_parse) */
         int16_t got[(ZB_MAX_MATCH + 32) / 32];
#pragma unroll
         for (int j = 0; j < (ZB_MAX_MATCH + 32) / 32; j++) { const int e = lane + 32 * j; got[j] = e <= lim ? sw[(size_t)e * SS] : (int16_t)0; }      /* all in flight together */
#pragma unroll
         for (int j = 0; j < (ZB_MAX_MATCH + 32) / 32; j++) {
            const int e = lane + 32 * j;
            if (e <= lim) {
               int sl = slot - e; if (sl < 0) sl += ZB_DW_RING;
               const int16_t v = (lo + e <= end) ? (int16_t)(uint16_t)(ring[sl] - b) : (int16_t)0;
               if (got[j] != v) same = false;
            }
         }
         if (__all_sync(0xffffffffu, same)) break;      /* nx was computed from exactly these costs: the run ends here */
      }
      for (int e = lane; e <= ZB_MAX_MATCH; e += 32) {   /* what chunk nx is now computed from */
         int sl = slot - e; if (sl < 0) sl += ZB_DW_RING;
         sw[(size_t)e * SS] = (lo + e <= end) ? (int16_t)(uint16_t)(ring[sl] - b) : (int16_t)0;
      }
      c = nx;
      __syncwarp();
   }
}
#endif

#ifndef ZB_EMU
/* Histogram along the chosen path (blockdeflate.c:371-400), one thread per path-chunk: the counts of a CTA's chunks are
   gathered in a shared-memory histogram of the CTA's first sub-block and flushed once (hot symbols would otherwise be one
   global atomic per token); a chunk of another sub-block (one CTA per sub-block boundary) counts straight into global memory. */
#define ZB_PH_THREADS 128
__global__ void __launch_bounds__(ZB_PH_THREADS) zb_path_hist_k(long npch, const ZbSub *sb, ZbSubTabs *tb, const uint32_t *pcs, const ZbWinDesc *wd, const uint32_t *wbs,
                                                                const uint8_t *T, const zb_match_t *bm, const uint32_t *pen, uint32_t cpv) {
   __shared__ int hl[ZB_NLIT], ho[ZB_NOFF];
   const long c0 = (long)blockIdx.x * ZB_PH_THREADS, c = c0 + threadIdx.x;
   const uint32_t x0 = pcs[c0];
   for (int e = threadIdx.x; e < ZB_NLIT; e += ZB_PH_THREADS) hl[e] = 0;
   if (threadIdx.x < ZB_NOFF) ho[threadIdx.x] = 0;
   __syncthreads();
   if (c < npch) {
      const uint32_t x = pcs[c];
      const ZbSub s = sb[x];
      if (s.is_dyn) {
         const uint32_t k = (uint32_t)c - s.pchunk_base, gb = wbs[s.win];
         const uint32_t lo = s.ps + k * cpv, hi = lo + cpv < s.pe ? lo + cpv : s.pe;
         const uint8_t *t = T + wd[s.win].in_off;
         int *lc = x == x0 ? hl : tb[x].lcnt, *oc = x == x0 ? ho : tb[x].ocnt;
         /* The path is a pointer chase (the next token starts where this one ends); followed load by load it is one DRAM
            round trip per token.  Instead the chunk's choices are streamed 16 bytes at a time, two groups ahead, through
            three registers used in rotation, and the positions that are not token starts are skipped. */
         const uint32_t *bw = (const uint32_t *)bm + gb;
         int next = (int)pen[c];
         const int hi_i = (int)hi, wlen = (int)wd[s.win].len;
         const long toff = (long)wd[s.win].in_off;
         int g = next - (int)((gb + (uint32_t)next) & 3u);   /* group start: (gb + g) % 4 == 0; may lie before the window (g < 0), never before the array */
         /* the 4 text bytes of a group, fetched with it (a literal's symbol must not be one more dependent load): two aligned
            words and a funnel shift where both lie inside the input, guarded byte loads at the edges */
         auto text4 = [&](int q) -> uint32_t {
            if (q >= hi_i) return 0u;
            if (toff + q >= 4 && q + 8 <= wlen) {
               const uintptr_t a = (uintptr_t)(t + q);
               const uint32_t *pa = (const uint32_t *)(a & ~(uintptr_t)3);
               return __funnelshift_r(pa[0], pa[1], (uint32_t)(a & 3) << 3);
            }
            uint32_t w = 0;
            for (int j = 0; j < 4; j++) if (q + j >= 0 && q + j < wlen) w |= (uint32_t)t[q + j] << (8 * j);
            return w;
         };
#define ZB_PH_LD(k_) (g + (k_) < hi_i ? *(const uint4 *)(bw + g + (k_)) : make_uint4(0u, 0u, 0u, 0u))
#define ZB_PH_ONE(w_, j_, tw_) do { const int pp_ = g + (j_); if (pp_ == next && pp_ < hi_i) { const uint32_t ln_ = (w_) & 0x1ffu;      /* choice word: k | sym << 9 | m << 14 */ \
            if (ln_ >= ZB_MIN_MATCH) { atomicAdd(lc + zb_len_sym(ln_ - ZB_MIN_MATCH), 1); atomicAdd(oc + (((w_) >> 9) & 31u), 1); next += (int)ln_; } \
            else { atomicAdd(lc + (((tw_) >> (8 * (j_))) & 0xffu), 1); next++; } } } while (0)
#define ZB_PH_PROC(v, tw_) do { ZB_PH_ONE((v).x, 0, tw_); ZB_PH_ONE((v).y, 1, tw_); ZB_PH_ONE((v).z, 2, tw_); ZB_PH_ONE((v).w, 3, tw_); g += 4; } while (0)
         uint4 va = ZB_PH_LD(0), vb = ZB_PH_LD(4), vc = ZB_PH_LD(8);
         uint32_t ta = text4(g), tb2 = text4(g + 4), tc = text4(g + 8);
         for (;;) {
            if (g >= hi_i) break; ZB_PH_PROC(va, ta); va = ZB_PH_LD(8); ta = text4(g + 8);
            if (g >= hi_i) break; ZB_PH_PROC(vb, tb2); vb = ZB_PH_LD(8); tb2 = text4(g + 8);
            if (g >= hi_i) break; ZB_PH_PROC(vc, tc); vc = ZB_PH_LD(8); tc = text4(g + 8);
         }
#undef ZB_PH_LD
#undef ZB_PH_ONE
#undef ZB_PH_PROC
      }
   }
   __syncthreads();
   if (!sb[x0].is_dyn) return;
   for (int e = threadIdx.x; e < ZB_NLIT; e += ZB_PH_THREADS) if (hl[e]) atomicAdd(tb[x0].lcnt + e, hl[e]);
   if (threadIdx.x < ZB_NOFF && ho[threadIdx.x]) atomicAdd(tb[x0].ocnt + threadIdx.x, ho[threadIdx.x]);
}
#endif

inline void ZbPipe::stage_parse() {
   /* One thread per chunk: the chunk count is the parallelism.  ZB_CD positions per chunk when that still gives ~40 K chunks,
      shorter chunks (more warm-up overhead, shorter serial chains) for small batches such as one GPU's shard of a stream. */
   /* (the thread-per-chunk kernel can keep 1152 chunks resident per SM; measured with the adaptive warm-up, it is fastest at
      ~0.65 of that - 960 positions per chunk on the 100 MB text, 512 on the 51 MB binaries: fewer warps fight for the
      shared-memory ring, and longer chunks carry less warm-up - and much slower just above one full wave) */
   int cd_auto = (int)(((long)P / ((long)zb_sm_count() * 720) + 32) / 64 * 64);
   /* the path chunks (sweep, histogram, token bits, emission: one thread walks a chunk) are half as long for small batches, where
      the walk of one chunk is the whole kernel's time (48 KB stream: path_hist 0.90 -> 0.45 ms); big batches have chunks to spare
      and the sweep's per-chunk overhead makes the short form slower there */
   cp = P <= (1L << 20) ? ZB_CP / 2 : ZB_CP;
   const uint32_t CPv = (uint32_t)cp;
   if (cd_auto < 128) cd_auto = 128;      /* small inputs (one 48 KB stream, a GPU's share of a strongly scaled 51 MB): short chunks = short serial chains, the warm-up then dominates a chunk */
   if (cd_auto > ZB_CD) cd_auto = ZB_CD;
   int CD = parse_cd ? parse_cd : cd_auto; if (CD > 2048) CD = 2048;      /* CD + ZB_WU <= 4368: u16 costs cannot wrap (zb_parse_dp_k) */
   const int ns = nsub;
   ZbSub *sb = sub.p; ZbSubTabs *tb = tabs.p; uint32_t *cn = counters.p;
   ZbGreedyView gv = {ph.p, wintbase.p, wtokbase.p, tokpos.p, wbase.p, glen.p, goff.p, in_ptr, win.p};
   /* D1: greedy histogram, static-vs-dynamic decision (libzultra.c:317-324), first tables (blockdeflate.c:863-869) */
#ifndef ZB_EMU
   if (ns > 0) {
      if (g_zb_prof_on) { zb_tag("sub_init"); zb_prof_begin(0, st); }
      zb_sub_init_k<<<(unsigned)((ns + ZB_WT / 32 - 1) / (ZB_WT / 32)), ZB_WT, 0, st>>>(sb, tb, ns, gv);
      if (g_zb_prof_on) zb_prof_end(st);
      zb_count_launch(1);
      ZB_CUDA_CHECK(cudaGetLastError());
   }
#else
   zb_launch(st, ns, ZB_LAMBDA(long x) {
      ZbSub s = sb[x]; ZbSubTabs &t = tb[x];
      int h[ZB_NH];
      gv.range_hist((int)s.win, s.ts, s.te, h);
      h[ZB_EOB] += 1;
      ZbScratch sc;
      s.static_cost = zb_static_cost(h, h + ZB_NLIT);
      zb_huff_lengths(h, ZB_NLIT, t.llen, sc.key);
      int olen288[ZB_NLIT];
      zb_huff_lengths(h + ZB_NLIT, ZB_NOFF, olen288, sc.key);
      s.dynamic_cost = zb_dynamic_cost(h, t.llen, h + ZB_NLIT, olen288, sc);
      s.is_dyn = s.static_cost <= s.dynamic_cost ? 0 : 1;
      s.ub_hit = 0;
      if (s.is_dyn) {
         zb_huff_build(h, ZB_NLIT, 15, t.llen, 0, sc.key, sc.order, &s.ub_hit);
         zb_huff_build(h + ZB_NLIT, ZB_NOFF, 15, olen288, 0, sc.key, sc.order, &s.ub_hit);
         for (int i = 0; i < ZB_NOFF; i++) t.olen[i] = olen288[i];
         int ll[ZB_NLIT], ol[ZB_NOFF];
         for (int i = 0; i < ZB_NLIT; i++) ll[i] = t.llen[i] ? t.llen[i] : 9;   /* blockdeflate.c:873-881 */
         for (int i = 0; i < ZB_NOFF; i++) ol[i] = t.olen[i] ? t.olen[i] : 6;
         zb_make_costtab(ll, ol, t.cost);
      } else {
         for (int i = 0; i < ZB_NLIT; i++) t.llen[i] = zb_static_lit_len(i);   /* blockdeflate.c:839-849 */
         for (int i = 0; i < ZB_NOFF; i++) t.olen[i] = 5;
         zb_make_costtab(t.llen, t.olen, t.cost);
      }
      sb[x] = s;
   }, 64);
#endif
   /* chunk lists */
   zb_launch(st, 1, ZB_LAMBDA(long) {
      uint32_t d = 0, p = 0;
      uint32_t curg = 0xffffffffu, cnt = 0, mx = 1;      /* most sub-blocks any group of 128 parse chunks (one CTA of zb_parse_dp_k) touches */
      for (int x = 0; x < ns; x++) {
         uint32_t size = sb[x].pe - sb[x].ps;
         const uint32_t nd = (size + CD - 1) / CD;
         sb[x].dchunk_base = d; sb[x].ndchunk = nd;
         if (nd) {
            const uint32_t g0 = d >> 7, g1 = (d + nd - 1) >> 7;
            if (g0 == curg) cnt++; else { curg = g0; cnt = 1; }
            if (cnt > mx) mx = cnt;
            if (g1 != g0) { curg = g1; cnt = 1; }
         }
         d += nd;
         sb[x].pchunk_base = p; sb[x].npchunk = (size + CPv - 1) / CPv; p += sb[x].npchunk;
      }
      cn[4] = d; cn[5] = p; cn[6] = mx;
   });
   uint32_t hc[3];
   zb_d2h(st, hc, cn + 4, 12); zb_sync(st);
   const long ndch = hc[0], npch = hc[1];
   dchunk_sub.need(ndch + 1); pchunk_sub.need(npch + 1); best.need(P);
#ifndef ZB_EMU
   cand.need((size_t)P * 4);
#endif
   sig_true.need((size_t)(ndch + 1) * 260); sig_warm.need((size_t)(ndch + 1) * 260); sig_new.need((size_t)(ndch + 1) * 260); dok.need(ndch + 1); dbad.need(ndch + 1);
   pentry.need(npch + 1); pbits.need(npch + 1);
#ifndef ZB_EMU
   exitc.need((size_t)(npch + 1) * ZB_EXROW);
   dpfar.need((size_t)((ndch + ZB_DP_THREADS - 1) / ZB_DP_THREADS) * (size_t)(CD + ZB_WU + 8) * ZB_DP_THREADS + 64);
#endif
   if (zb_failed()) return;
   uint32_t *dcs = dchunk_sub.p, *pcs = pchunk_sub.p;
   zb_launch(st, ns, ZB_LAMBDA(long x) {
      for (uint32_t k = 0; k < sb[x].ndchunk; k++) dcs[sb[x].dchunk_base + k] = (uint32_t)x;
      for (uint32_t k = 0; k < sb[x].npchunk; k++) pcs[sb[x].pchunk_base + k] = (uint32_t)x;
   });
   const ZbWinDesc *wd = win.p; const uint32_t *wbs = wbase.p; const uint8_t *T = in_ptr;
   const zb_match_t *mt = match.p; zb_match_t *bm = best.p;
   /* Adaptive warm-up (round 2).  A chunk reads costs past its end only through the candidates of its last positions: `reach`
      = max over its positions p of p + (longest candidate length of p) - chunk end, 0..258.  The chunk is right iff the relative
      costs at its end .. end + reach are (all it ever reads), so only those entries of the two signatures are compared and the
      warm-up is the settling margin above them, not above the full 258-position horizon: ~130 instead of 384 positions on text,
      where the reach is a handful of positions (99th percentile 28).  With chunks shorter than the horizon (small inputs: CD =
      128) a chunk's left neighbours read THROUGH it into its warm-up zone, so what a chunk needs right is
      need(c) = max(reach(c), need(c - 1) - CD) - then every entry any comparison or repair start ever uses is either inside a
      verified chunk or inside the verified part of a warm-up zone (induction from the exact last chunk of the sub-block).
      The lists do not change over the passes: once per batch, 8 tasks of 33 positions per chunk. */
   int *rch = 0;
   if (ndch > 0) {
      dreach.need(2 * (size_t)ndch + 2);
      if (zb_failed()) return;
      int *need = dreach.p;
      rch = dreach.p + ndch + 1;      /* raw reach first, need() derived from it below */
      zb_memset(st, rch, 0, (size_t)ndch * 4);
      zb_tag("parse_reach");
      zb_launch(st, ndch * 8, ZB_LAMBDA(long x) {
         const long c = x >> 3; const int part = (int)(x & 7);
         const ZbSub sx = sb[dcs[c]];
         const uint32_t k = (uint32_t)c - sx.dchunk_base;
         if (k + 1 >= sx.ndchunk) return;      /* the last chunk of a sub-block starts from the exact end */
         const int lo = (int)(sx.ps + k * CD), hi = lo + CD;
         const zb_match_t *m0 = mt + ((size_t)wbs[sx.win] << 3);
         int best_r = 0;
         for (int p = hi - 1 - part * 33, e = 0; e < 33 && p >= lo && hi - p <= ZB_MAX_MATCH; e++, p--) {
            const ZbCand cd = zb_cand_pack(zb_load_rec(m0, p), (int)sx.pe - p);
            int ml = 0;
            for (int z = 0; z < ZB_NMATCH; z++) {
               const uint32_t ent = (cd.w[z >> 1] >> (16 * (z & 1))) & 0xffffu;
               if (!ent) break;
               const int l = (ent & 0x8000u) ? (int)((ent >> 5) & 511u) : (int)((ent >> 5) & 63u);
               ml = l > ml ? l : ml;
            }
            const int r = p + ml - hi;
            best_r = r > best_r ? r : best_r;
         }
         if (best_r > ZB_MAX_MATCH) best_r = ZB_MAX_MATCH;
         if (best_r > 0) zb_atomic_max(rch + c, best_r);
      }, 256);
      {
         const int *raw = rch;
         zb_launch(st, ndch, ZB_LAMBDA(long c) {
            const ZbSub sx = sb[dcs[c]];
            int nd = raw[c];
            for (long j = 1; j * CD < ZB_MAX_MATCH && c - j >= (long)sx.dchunk_base; j++) { const int r = raw[c - j] - (int)j * CD; nd = r > nd ? r : nd; }
            need[c] = nd;
         }, 256);
      }
      rch = need;
   }
#ifndef ZB_EMU
   /* candidate records (once: the match lists do not change over the passes) and the parse kernel's shared memory */
   const int dp_nslot = (int)(hc[2] < 1 ? 1 : (hc[2] > ZB_DP_THREADS ? ZB_DP_THREADS : hc[2]));
   const size_t dp_smem = (size_t)ZB_NR * ZB_DP_THREADS * 2 + (size_t)dp_nslot * sizeof(ZbDpTab);
   {  /* the limit is a per-function global: always the largest configuration, so concurrent host threads cannot undercut each other */
      const size_t smax = (size_t)ZB_NR * ZB_DP_THREADS * 2 + (size_t)ZB_DP_THREADS * sizeof(ZbDpTab);
      ZB_CUDA_CHECK(cudaFuncSetAttribute(zb_parse_dp_k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smax));
   }
   if (npch > 0) {
      if (g_zb_prof_on) { zb_tag("parse_cand"); zb_prof_begin(0, st); }
      zb_cand_k<<<(unsigned)npch, 256, 0, st>>>(npch, sb, pcs, wbs, mt, (uint4 *)cand.p, CPv);
      if (g_zb_prof_on) zb_prof_end(st);
      zb_count_launch(1);
      ZB_CUDA_CHECK(cudaGetLastError());
   }
#endif
   const size_t SS = (size_t)ndch + 1;   /* signatures are stored [entry][chunk]: neighbouring chunks' accesses coalesce */
   int16_t *sgt = sig_true.p, *sgw = sig_warm.p, *sgn = sig_new.p; uint8_t *ok = dok.p; uint32_t *bad = dbad.p; (void)sgn;
   uint16_t *ex = exitoff.p; uint32_t *pen = pentry.p;

   for (int pass = 0; pass < 4; pass++) {
      /* D2: chunked backward recurrence.  Chunk k of a sub-block covers [ps + k*CD, ..).  Every chunk but the last
         starts up to ZB_WU positions past its end from an all-zero cost guess; the relative costs it sees at its own end
         (sig_warm) are later compared with what the next chunk really computed there (sig_true). */
#ifndef ZB_EMU
      if (ndch > 0) {
         if (g_zb_prof_on) { zb_tag("parse_dp"); zb_prof_begin(0, st); }
         zb_parse_dp_k<<<(unsigned)((ndch + ZB_DP_THREADS - 1) / ZB_DP_THREADS), ZB_DP_THREADS, dp_smem, st>>>(sb, tb, dcs, ndch, pass, wd, wbs, T, (const uint4 *)cand.p, (uint32_t *)bm,
                                                                                                       sgt, sgw, SS, dpfar.p, CD, dp_nslot, rch);
         if (g_zb_prof_on) zb_prof_end(st);
         zb_count_launch(1);
         ZB_CUDA_CHECK(cudaGetLastError());
      }
#else
      zb_tag("parse_dp");
      const bool emu_lean = getenv("ZB_EMU_DP_LEAN") != 0;    /* host build only: run the chunks through the compact candidate records (zb_cand_pack / zb_dp_eval), as zb_parse_dp_k does */
      zb_launch(st, ndch, ZB_LAMBDA(long c) {
         const ZbSub s = sb[dcs[c]];
         if (pass > 0 && !s.is_dyn) return;
         if (emu_lean) {
            const uint32_t kc = (uint32_t)c - s.dchunk_base;
            const uint32_t gb = wbs[s.win];
            const uint8_t *t = T + wd[s.win].in_off;
            const zb_match_t *m0 = mt + ((size_t)gb << 3);
            const int lo = (int)(s.ps + kc * CD);
            const int hi = (int)(lo + CD < (int)s.pe ? lo + CD : (int)s.pe);
            const int end = (int)s.pe;
            int from = hi + zb_warmup_len(rch[c]); if (from > end) from = end;
            const ZbCostTab &ct = tb[dcs[c]].cost;
            std::vector<uint32_t> v((size_t)(from - lo) + 1, 0u);      /* cost of step tt (position from - 1 - tt) */
            uint32_t cprev = 0;
            int tt = 0;
            for (int i = from - 1; i >= lo; i--, tt++) {
               const ZbCand cd = zb_cand_pack(zb_load_rec(m0, i), end - i);
               auto costat = [&](int k) -> uint32_t { const int q = tt - k; return q >= 0 ? v[(size_t)q] : 0u; };
               uint32_t ch = 0;
               const uint32_t cc = zb_dp_eval(cd, ct.lit[t[i]], cprev, ct, costat, &ch);
               if (cc > 0xffffu) { fprintf(stderr, "dp cost overflow\n"); abort(); }
               v[(size_t)tt] = cc; cprev = cc;
               if (i < hi) {      /* the choice word, resolved the way zb_choice_k does */
                  zb_match_t b; b.length = 0; b.offset = 0;
                  if (ch) { b.length = (uint16_t)(ch & 511u); b.offset = m0[((size_t)i << 3) + (ch >> 14)].offset;
                            if ((uint32_t)zb_off_sym(b.offset) != ((ch >> 9) & 31u)) { fprintf(stderr, "choice symbol mismatch\n"); abort(); } }
                  bm[gb + i] = b;
               }
            }
            const int tw = from - hi, tall = from - lo;
            const uint32_t bw_ = tw > 0 ? v[(size_t)tw - 1] : 0u, bt_ = tall > 0 ? v[(size_t)tall - 1] : 0u;
            int16_t *sw = sgw + (size_t)c, *sg = sgt + (size_t)c;
            for (int q = 0; q <= ZB_MAX_MATCH; q++) {
               const uint32_t vw = tw - 1 - q >= 0 ? v[(size_t)(tw - 1 - q)] : 0u, vt = tall - 1 - q >= 0 ? v[(size_t)(tall - 1 - q)] : 0u;
               sw[(size_t)q * SS] = (hi + q <= end && hi + q <= from) ? (int16_t)(uint16_t)(vw - bw_) : (int16_t)0;
               sg[(size_t)q * SS] = (lo + q <= end) ? (int16_t)(uint16_t)(vt - bt_) : (int16_t)0;
            }
            return;
         }
         const uint32_t k = (uint32_t)c - s.dchunk_base;
         const uint32_t gb = wbs[s.win];
         const uint8_t *t = T + wd[s.win].in_off;
         const int lo = (int)(s.ps + k * CD);
         const int hi = (int)(lo + CD < (int)s.pe ? lo + CD : (int)s.pe);
         const int end = (int)s.pe;
         int from = hi + zb_warmup_len(rch[c]); if (from > end) from = end;
         ZbRingLocal ring;
         for (int i = 0; i < ZB_RING; i++) ring.v[i] = 0;
         int slot = 0;
         const ZbCostTab &ct = tb[dcs[c]].cost;
         if (from > hi) zb_parse_range(t, mt + ((size_t)gb << 3), ct, hi, from, end, hi, bm + gb, ring, slot);
         /* warm-up view of the window [hi, hi+258] */
         {
            int16_t *sw = sgw + (size_t)c;
            const uint16_t b = ring.get(slot);
            for (int q = 0; q <= ZB_MAX_MATCH; q++) {
               int sl = slot - q; if (sl < 0) sl += ZB_RING;
               sw[(size_t)q * SS] = (hi + q <= end && hi + q <= from) ? (int16_t)(uint16_t)(ring.get(sl) - b) : (int16_t)0;
            }
         }
         zb_parse_range(t, mt + ((size_t)gb << 3), ct, lo, hi, end, hi, bm + gb, ring, slot);
         {
            int16_t *sg = sgt + (size_t)c;
            const uint16_t b = ring.get(slot);
            for (int q = 0; q <= ZB_MAX_MATCH; q++) {
               int sl = slot - q; if (sl < 0) sl += ZB_RING;
               sg[(size_t)q * SS] = (lo + q <= end) ? (int16_t)(uint16_t)(ring.get(sl) - b) : (int16_t)0;
            }
         }
      }, 64);
#endif
      /* D3/D4: verify and repair.  A chunk is right iff the relative costs its warm-up saw over the 259-position horizon
         at its end equal what its right neighbour really computed there, and the neighbour is right.  Rounds: every chunk
         is compared with its neighbour's current costs; every chunk that disagrees is recomputed IN PARALLEL from the
         neighbour's costs; repeat until nothing disagrees.  By induction from the (exact) last chunk of each sub-block the
         fixed point is the sequential result; the number of rounds is the longest run of consecutive wrong chunks
         (non-resynchronising data such as long byte runs), independent chains repair concurrently. */
      for (;;) {
         zb_memset(st, cn + 7, 0, 4);
         zb_tag("parse_verify");
         zb_launch(st, ndch, ZB_LAMBDA(long c) {
            const ZbSub s = sb[dcs[c]];
            uint8_t good = 1;
            const uint32_t k = (uint32_t)c - s.dchunk_base;
            if (!(pass > 0 && !s.is_dyn) && k + 1 < s.ndchunk) {
               const int16_t *a = sgw + (size_t)c, *b = sgt + (size_t)(c + 1);
               const int lim = rch[c];      /* the chunk reads no cost further out */
               for (int q = 0; q <= lim && good; q++) if (a[(size_t)q * SS] != b[(size_t)q * SS]) good = 0;
            }
            ok[c] = good;
            if (!good) { const int at = zb_atomic_add((int *)cn + 7, 1); bad[at] = (uint32_t)c; }
         });
         uint32_t nbad = 0;
         zb_d2h(st, &nbad, cn + 7, 4); zb_sync(st);
         if (!nbad) break;
         stat_redo += (int)nbad;
#ifndef ZB_EMU
         if (g_zb_prof_on) { zb_tag("parse_repair"); zb_prof_begin(0, st); }
         zb_parse_fix_k<<<(unsigned)((nbad + ZB_DW_WARPS - 1) / ZB_DW_WARPS), ZB_DW_THREADS, 0, st>>>(sb, tb, dcs, bad, (int)nbad, ok, wd, wbs, T, mt, bm, sgt, sgw, SS, CD, rch);
         if (g_zb_prof_on) zb_prof_end(st);
         zb_count_launch(1);
         ZB_CUDA_CHECK(cudaGetLastError());
#else
         zb_tag("parse_repair");
         zb_launch(st, ndch, ZB_LAMBDA(long c) {
            if (ok[c]) return;
            const uint32_t x = dcs[c];
            const ZbSub s = sb[x];
            const uint32_t k = (uint32_t)c - s.dchunk_base;
            const uint32_t gb = wbs[s.win];
            const uint8_t *t = T + wd[s.win].in_off;
            const int end = (int)s.pe;
            const ZbCostTab &ct = tb[x].cost;
            const int lo = (int)(s.ps + k * CD), hi = lo + CD;
            ZbRingLocal ring;
            const int16_t *b = sgt + (size_t)(c + 1);
            int16_t *sw = sgw + (size_t)c;
            int slot = 0;
            for (int q = 0; q <= ZB_MAX_MATCH; q++) { int sl = slot - q; if (sl < 0) sl += ZB_RING; ring.v[sl] = (uint16_t)b[(size_t)q * SS]; sw[(size_t)q * SS] = b[(size_t)q * SS]; }
            zb_parse_range(t, mt + ((size_t)gb << 3), ct, lo, hi, end, hi, bm + gb, ring, slot);
            /* the new costs at this chunk's start go to a staging row: neighbours still read the old row this round */
            int16_t *sg = sgn + (size_t)c;
            const uint16_t b0 = ring.get(slot);
            for (int q = 0; q <= ZB_MAX_MATCH; q++) {
               int sl = slot - q; if (sl < 0) sl += ZB_RING;
               sg[(size_t)q * SS] = (lo + q <= end) ? (int16_t)(uint16_t)(ring.get(sl) - b0) : (int16_t)0;
            }
         }, 32);
         zb_launch(st, ndch, ZB_LAMBDA(long c) {
            if (ok[c]) return;
            int16_t *sg = sgt + (size_t)c; const int16_t *sn = sgn + (size_t)c;
            for (int q = 0; q <= ZB_MAX_MATCH; q++) sg[(size_t)q * SS] = sn[(size_t)q * SS];
         });
#endif
      }
      /* D5: chosen path: exit offsets per path-chunk, serial hop per sub-block */
#ifndef ZB_EMU
      if (npch > 0) {
         if (g_zb_prof_on) { zb_tag("path_sweep"); zb_prof_begin(0, st); }
         zb_sweep_k<1><<<(unsigned)((npch + ZB_SW_THREADS - 1) / ZB_SW_THREADS), ZB_SW_THREADS, 0, st>>>(npch, wd, wbs, 0, 0, 0, 0, sb, pcs, pass, bm, exitc.p, CPv);
         if (g_zb_prof_on) zb_prof_end(st);
         if (g_zb_prof_on) { zb_tag("path_hop"); zb_prof_begin(0, st); }
         zb_hop_k<1><<<ns, 32, 0, st>>>(ns, wd, 0, sb, tb, pass, exitc.p, pen, CPv);
         if (g_zb_prof_on) zb_prof_end(st);
         zb_count_launch(2);
         ZB_CUDA_CHECK(cudaGetLastError());
      }
      (void)ex;
#else
      zb_launch(st, npch, ZB_LAMBDA(long c) {
         const ZbSub s = sb[pcs[c]];
         if (pass > 0 && !s.is_dyn) return;
         const uint32_t k = (uint32_t)c - s.pchunk_base, gb = wbs[s.win];
         const uint32_t lo = s.ps + k * CPv, hi = lo + CPv < s.pe ? lo + CPv : s.pe;
         for (uint32_t p = hi; p-- > lo;) {
            uint32_t l = bm[gb + p].length; if (l < ZB_MIN_MATCH) l = 1;
            uint32_t j = p + l;
            ex[gb + p] = (uint16_t)(j >= hi ? j - hi : ex[gb + j]);
         }
      });
      zb_launch(st, ns, ZB_LAMBDA(long x) {
         const ZbSub s = sb[x];
         if (pass > 0 && !s.is_dyn) return;
         const uint32_t gb = wbs[s.win];
         uint32_t e = s.ps;
         for (uint32_t k = 0; k < s.npchunk; k++) {
            const uint32_t lo = s.ps + k * CPv, hi = lo + CPv < s.pe ? lo + CPv : s.pe;
            pen[s.pchunk_base + k] = e;
            if (e < hi) e = hi + ex[gb + e];
         }
         /* fresh histogram for this pass (blockdeflate.c:887-891); EOB counted here */
         if (s.is_dyn) {
            ZbSubTabs &t = tb[x];
            for (int i = 0; i < ZB_NLIT; i++) t.lcnt[i] = 0;
            for (int i = 0; i < ZB_NOFF; i++) t.ocnt[i] = 0;
            t.lcnt[ZB_EOB] = 1;
         }
      });
#endif
      /* D6: histogram along the chosen path (blockdeflate.c:371-400) */
#ifndef ZB_EMU
      if (npch > 0) {
         if (g_zb_prof_on) { zb_tag("path_hist"); zb_prof_begin(0, st); }
         zb_path_hist_k<<<(unsigned)((npch + ZB_PH_THREADS - 1) / ZB_PH_THREADS), ZB_PH_THREADS, 0, st>>>(npch, sb, tb, pcs, wd, wbs, T, bm, pen, CPv);
         if (g_zb_prof_on) zb_prof_end(st);
         zb_count_launch(1);
         ZB_CUDA_CHECK(cudaGetLastError());
      }
#else
      zb_launch(st, npch, ZB_LAMBDA(long c) {
         const uint32_t x = pcs[c];
         const ZbSub s = sb[x];
         if (!s.is_dyn) return;
         const uint32_t k = (uint32_t)c - s.pchunk_base, gb = wbs[s.win];
         const uint32_t lo = s.ps + k * CPv, hi = lo + CPv < s.pe ? lo + CPv : s.pe;
         const uint8_t *t = T + wd[s.win].in_off;
         int *lc = tb[x].lcnt, *oc = tb[x].ocnt;
         for (uint32_t p = pen[c]; p < hi;) {
            zb_match_t m = bm[gb + p];
            if (m.length >= ZB_MIN_MATCH) { zb_atomic_add(lc + zb_len_sym(m.length - ZB_MIN_MATCH), 1); zb_atomic_add(oc + zb_off_sym(m.offset), 1); p += m.length; }
            else { zb_atomic_add(lc + t[p], 1); p++; }
         }
      });
#endif
      /* D7: rebuild tables (blockdeflate.c:893-919) */
#ifndef ZB_EMU
      if (ns > 0) {
         if (g_zb_prof_on) { zb_tag("sub_tables"); zb_prof_begin(0, st); }
         zb_sub_tables_k<<<(unsigned)((ns + ZB_WT / 32 - 1) / (ZB_WT / 32)), ZB_WT, 0, st>>>(sb, tb, ns, pass);
         if (g_zb_prof_on) zb_prof_end(st);
         zb_count_launch(1);
         ZB_CUDA_CHECK(cudaGetLastError());
      }
#else
      zb_launch(st, ns, ZB_LAMBDA(long x) {
         ZbSub s = sb[x];
         if (!s.is_dyn) return;
         ZbSubTabs &t = tb[x];
         if (pass == 3) {   /* always describe at least two distance codes (blockdeflate.c:893-913) */
            int nz = 0;
            for (int i = 0; nz < 2 && i < ZB_NOFF - 2; i++) if (t.ocnt[i]) nz++;
            if (nz == 0) t.ocnt[0] = t.ocnt[1] = 1;
            else if (nz == 1) { if (t.ocnt[0]) t.ocnt[1] = 1; else t.ocnt[0] = 1; }
         }
         ZbScratch sc; int olen288[ZB_NLIT];
         zb_huff_build(t.lcnt, ZB_NLIT, 15, t.llen, 0, sc.key, sc.order, &s.ub_hit);
         zb_huff_build(t.ocnt, ZB_NOFF, 15, olen288, 0, sc.key, sc.order, &s.ub_hit);
         for (int i = 0; i < ZB_NOFF; i++) t.olen[i] = olen288[i];
         if (pass < 3) {
            int ll[ZB_NLIT], ol[ZB_NOFF];
            for (int i = 0; i < ZB_NLIT; i++) ll[i] = t.llen[i] ? t.llen[i] : 9;
            for (int i = 0; i < ZB_NOFF; i++) ol[i] = t.olen[i] ? t.olen[i] : 6;
            zb_make_costtab(ll, ol, t.cost);
         } else {
            zb_make_costtab(t.llen, t.olen, t.cost);   /* final lengths: used by the post-optimiser and the emitter */
         }
         sb[x] = s;
      }, 64);
#endif
   }
#ifndef ZB_EMU
   if (npch > 0) {      /* choice words -> {length, offset} */
      if (g_zb_prof_on) { zb_tag("parse_choice"); zb_prof_begin(0, st); }
      zb_choice_k<<<(unsigned)npch, 256, 0, st>>>(npch, sb, pcs, wbs, mt, (uint32_t *)bm, CPv);
      if (g_zb_prof_on) zb_prof_end(st);
      zb_count_launch(1);
      ZB_CUDA_CHECK(cudaGetLastError());
   }
#endif
   /* P7: matches that are cheaper as literals (blockdeflate.c:410-458), dynamic sub-blocks only */
   zb_launch(st, npch, ZB_LAMBDA(long c) {
      const uint32_t x = pcs[c];
      const ZbSub s = sb[x];
      if (!s.is_dyn) return;
      const uint32_t k = (uint32_t)c - s.pchunk_base, gb = wbs[s.win];
      const uint32_t lo = s.ps + k * CPv, hi = lo + CPv < s.pe ? lo + CPv : s.pe;
      const uint8_t *t = T + wd[s.win].in_off;
      const ZbCostTab &ct = tb[x].cost;
      for (uint32_t p = pen[c]; p < hi;) {
         zb_match_t m = bm[gb + p];
         if (m.length >= ZB_MIN_MATCH) {
            const uint32_t mc = (uint32_t)ct.len[m.length - ZB_MIN_MATCH] + ct.off[zb_off_sym(m.offset)];
            uint32_t lc = 0; bool all = true;
            for (uint32_t j = 0; j < m.length && lc < mc; j++) {
               uint32_t c1 = ct.lit[t[p + j]];
               if (c1 == 0) { all = false; break; }
               lc += c1;
            }
            if (all && lc < mc) for (uint32_t j = 0; j < m.length; j++) bm[gb + p + j].length = 0;
            p += m.length;
         } else p++;
      }
   });
   /* F1a: RLE smoothing trial (blockdeflate.c:926-945); the code-length sequence to be described */
#ifndef ZB_EMU
   if (ns > 0) {
      if (g_zb_prof_on) { zb_tag("sub_smooth"); zb_prof_begin(0, st); }
      zb_sub_smooth_k<<<(unsigned)((ns + ZB_WT / 32 - 1) / (ZB_WT / 32)), ZB_WT, 0, st>>>(sb, tb, ns);
      if (g_zb_prof_on) zb_prof_end(st);
      zb_count_launch(1);
      ZB_CUDA_CHECK(cudaGetLastError());
   }
#else
   zb_launch(st, ns, ZB_LAMBDA(long x) {
      ZbSub s = sb[x]; ZbSubTabs &t = tb[x];
      ZbScratch sc;
      if (s.is_dyn) {
         int oc288[ZB_NLIT], ol288[ZB_NLIT];
         for (int i = 0; i < ZB_NLIT; i++) { oc288[i] = i < ZB_NOFF ? t.ocnt[i] : 0; ol288[i] = i < ZB_NOFF ? t.olen[i] : 0; }
         const int cur_cost = zb_dynamic_cost(t.lcnt, t.llen, oc288, ol288, sc);
         int lc2[ZB_NLIT], oc2[ZB_NLIT], ll2[ZB_NLIT], ol2[ZB_NLIT];
         uint8_t good[ZB_NLIT];
         for (int i = 0; i < ZB_NLIT; i++) { lc2[i] = t.lcnt[i]; oc2[i] = oc288[i]; }
         zb_smooth_counts(ZB_NLIT, lc2, good);
         zb_smooth_counts(ZB_NOFF, oc2, good);
         int ub = 0;
         zb_huff_build(lc2, ZB_NLIT, 15, ll2, 0, sc.key, sc.order, &ub);
         zb_huff_build(oc2, ZB_NOFF, 15, ol2, 0, sc.key, sc.order, &ub);
         const int opt_cost = zb_dynamic_cost(lc2, ll2, oc2, ol2, sc);
         if (opt_cost < cur_cost) {
            for (int i = 0; i < ZB_NLIT; i++) { t.lcnt[i] = lc2[i]; t.llen[i] = ll2[i]; }
            for (int i = 0; i < ZB_NOFF; i++) { t.ocnt[i] = oc2[i]; t.olen[i] = ol2[i]; }
            s.ub_hit |= ub;
         }
         s.nl = zb_defined_count(t.llen, ZB_NLIT, 257);
         int ol32[ZB_NOFF]; for (int i = 0; i < ZB_NOFF; i++) ol32[i] = t.olen[i];
         s.no = zb_defined_count(ol32, ZB_NOFF, 1);
         for (int i = 0; i < s.nl; i++) t.cl[i] = (uint8_t)t.llen[i];
         for (int i = 0; i < s.no; i++) t.cl[s.nl + i] = (uint8_t)t.olen[i];
      } else {
         s.nl = 288; s.no = 32; s.ncl = 0; s.mask = 0; s.hdr_bits = 0;
      }
      sb[x] = s;
   }, 64);
#endif
   /* F1b: the 20 RLE masks {0..7, 9, 11, .., 31} in parallel (blockdeflate.c:958-974) */
   zb_launch(st, (long)ns * 20, ZB_LAMBDA(long y) {
      const long x = y / 20; const int mi = (int)(y % 20);
      const ZbSub s = sb[x]; ZbSubTabs &t = tb[x];
      if (!s.is_dyn) return;
      const int mask = mi < 8 ? mi : 9 + 2 * (mi - 8);
      int clcnt[ZB_NCL], cllen[ZB_NLIT]; uint32_t key[ZB_NLIT]; int16_t order[ZB_NLIT]; int ub = 0;
      /* private copy of the code-length sequence (20 vector loads): the two scans read it byte by byte in dependent steps */
      alignas(16) uint8_t cll[ZB_NLIT + ZB_NOFF];
      { struct V16 { uint32_t a, b, c, d; }; struct alignas(16) A16 { V16 v; };
        for (int e = 0; e < (ZB_NLIT + ZB_NOFF) / 16; e++) ((A16 *)cll)[e] = ((const A16 *)t.cl)[e]; }
      for (int i = 0; i < ZB_NCL; i++) clcnt[i] = 0;
      ZbRleCount cv = {clcnt};
      zb_rle_scan(cll, s.nl + s.no, (unsigned)mask, cv);
      zb_huff_build(clcnt, ZB_NCL, 7, cllen, 0, key, order, &ub);
      ZbRleSize sv = {cllen, 0};
      zb_rle_scan(cll, s.nl + s.no, (unsigned)mask, sv);
      t.mask_cost[mi] = sv.bits | (ub << 30);
   }, 64);
   /* F1c: pick the mask (later one wins ties, :966), final code-length code, codewords, header size */
   zb_launch(st, ns, ZB_LAMBDA(long x) {
      ZbSub s = sb[x]; ZbSubTabs &t = tb[x];
      if (s.is_dyn) {
         int bestmi = -1, bestcost = 0;
         for (int mi = 0; mi < 20; mi++) {
            const int c = t.mask_cost[mi] & 0x3fffffff;
            if (t.mask_cost[mi] >> 30) s.ub_hit = 1;
            if (bestmi == -1 || bestcost >= c) { bestmi = mi; bestcost = c; }
         }
         const int bestmask = bestmi < 8 ? bestmi : 9 + 2 * (bestmi - 8);
         int clcnt[ZB_NCL], cllen[ZB_NLIT]; uint32_t key[ZB_NLIT]; int16_t order[ZB_NLIT];
         for (int i = 0; i < ZB_NCL; i++) clcnt[i] = 0;
         ZbRleCount cv = {clcnt};
         zb_rle_scan(t.cl, s.nl + s.no, (unsigned)bestmask, cv);
         zb_huff_build(clcnt, ZB_NCL, 7, cllen, t.clcode, key, order, &s.ub_hit);
         for (int i = 0; i < ZB_NCL; i++) t.cllen[i] = cllen[i];
         s.mask = bestmask;
         s.ncl = zb_raw_table_size(cllen);
         s.hdr_bits = 14 + 3 * s.ncl + bestcost;
         if (s.nl > 286 || s.no > 30) s.hdr_bits = -1;   /* blockdeflate.c:981-983: block_deflate fails -> stored */
      }
      {
         int16_t order[ZB_NLIT];
         int n = zb_order_by_len(t.llen, ZB_NLIT, order);
         zb_huff_codes(t.llen, order, n, t.lcode);
         int ol[ZB_NOFF]; for (int i = 0; i < ZB_NOFF; i++) ol[i] = t.olen[i];
         n = zb_order_by_len(ol, ZB_NOFF, order);
         zb_huff_codes(ol, order, n, t.ocode);
         zb_make_costtab(t.llen, ol, t.cost);
      }
      sb[x] = s;
   }, 64);
}

/* ============================================================ emission ============================================================
 * Token bits per path-chunk, per sub-block totals, then one serial scan per stream that reproduces the bit
 * writer's arithmetic of libzultra.c:327-398 (entering bit phase, stored-block fallback on BYTE deltas), then
 * every chunk writes its tokens at its absolute bit offset.
 */
inline void ZbPipe::stage_emit_prepare() {
   const uint32_t CPv = (uint32_t)cp;
   const int ns = nsub;
   ZbSub *sb = sub.p; ZbSubTabs *tb = tabs.p; uint32_t *cn = counters.p;
   const ZbWinDesc *wd = win.p; const uint32_t *wbs = wbase.p; const uint8_t *T = in_ptr;
   zb_match_t *bm = best.p; uint16_t *ex = exitoff.p; uint32_t *pen = pentry.p, *pb = pbits.p, *pcs = pchunk_sub.p;
   long npch = 0;
   {
      uint32_t v; zb_d2h(st, &v, cn + 5, 4); zb_sync(st); npch = v;
   }
   /* path again (the post-optimiser turned some matches into literals) */
#ifndef ZB_EMU
   if (npch > 0) {
      if (g_zb_prof_on) { zb_tag("path_sweep"); zb_prof_begin(0, st); }
      zb_sweep_k<1><<<(unsigned)((npch + ZB_SW_THREADS - 1) / ZB_SW_THREADS), ZB_SW_THREADS, 0, st>>>(npch, wd, wbs, 0, 0, 0, 0, sb, pcs, -1, bm, exitc.p, CPv);
      if (g_zb_prof_on) zb_prof_end(st);
      if (g_zb_prof_on) { zb_tag("path_hop"); zb_prof_begin(0, st); }
      zb_hop_k<1><<<ns, 32, 0, st>>>(ns, wd, 0, sb, tb, -1, exitc.p, pen, CPv);
      if (g_zb_prof_on) zb_prof_end(st);
      zb_count_launch(2);
      ZB_CUDA_CHECK(cudaGetLastError());
   }
   (void)ex;
#else
   zb_launch(st, npch, ZB_LAMBDA(long c) {
      const ZbSub s = sb[pcs[c]];
      const uint32_t k = (uint32_t)c - s.pchunk_base, gb = wbs[s.win];
      const uint32_t lo = s.ps + k * CPv, hi = lo + CPv < s.pe ? lo + CPv : s.pe;
      for (uint32_t p = hi; p-- > lo;) {
         uint32_t l = bm[gb + p].length; if (l < ZB_MIN_MATCH) l = 1;
         uint32_t j = p + l;
         ex[gb + p] = (uint16_t)(j >= hi ? j - hi : ex[gb + j]);
      }
   });
   zb_launch(st, ns, ZB_LAMBDA(long x) {
      const ZbSub s = sb[x];
      const uint32_t gb = wbs[s.win];
      uint32_t e = s.ps;
      for (uint32_t k = 0; k < s.npchunk; k++) {
         const uint32_t lo = s.ps + k * CPv, hi = lo + CPv < s.pe ? lo + CPv : s.pe;
         pen[s.pchunk_base + k] = e;
         if (e < hi) e = hi + ex[gb + e];
      }
   });
#endif
   /* E1: token bits per chunk */
   zb_launch(st, npch, ZB_LAMBDA(long c) {
      const uint32_t x = pcs[c];
      const ZbSub s = sb[x];
      const uint32_t k = (uint32_t)c - s.pchunk_base, gb = wbs[s.win];
      const uint32_t lo = s.ps + k * CPv, hi = lo + CPv < s.pe ? lo + CPv : s.pe;
      const uint8_t *t = T + wd[s.win].in_off;
      const ZbCostTab &ct = tb[x].cost;
      uint32_t bits = 0;
      for (uint32_t p = pen[c]; p < hi;) {
         zb_match_t m = bm[gb + p];
         if (m.length >= ZB_MIN_MATCH) { bits += (uint32_t)ct.len[m.length - ZB_MIN_MATCH] + ct.off[zb_off_sym(m.offset)]; p += m.length; }
         else { bits += ct.lit[t[p]]; p++; }
      }
      pb[c] = bits;
   });
   /* E2: per sub-block: chunk bit offsets (exclusive scan) and body size */
   zb_launch(st, ns, ZB_LAMBDA(long x) {
      ZbSub s = sb[x];
      uint32_t acc = 0;
      for (uint32_t k = 0; k < s.npchunk; k++) { uint32_t v = pb[s.pchunk_base + k]; pb[s.pchunk_base + k] = acc; acc += v; }
      s.body_bits = s.hdr_bits < 0 ? -1 : (int32_t)(s.hdr_bits + acc + tb[x].llen[ZB_EOB]);
      sb[x] = s;
   });
}

/* The stitch arithmetic of libzultra.c:327-398 on the host, for all 8 entering bit phases (multi-GPU: a shard learns its
   phase from the shards before it; everything up to here is phase independent). */
inline void ZbPipe::phase_maps(const std::vector<ZbStreamOut> &streams, unsigned long long *bits_out) {
   std::vector<ZbSub> hs(nsub);
   zb_d2h(st, hs.data(), sub.p, sizeof(ZbSub) * nsub); zb_sync(st);
   int x0 = 0;      /* sub-blocks are in window order and streams own consecutive windows */
   for (size_t q = 0; q < streams.size(); q++) {
      const uint32_t first_win = streams[q].first_win, nw = streams[q].nwin;
      while (x0 < nsub && hs[x0].win < first_win) x0++;
      int x1 = x0;
      while (x1 < nsub && hs[x1].win < first_win + nw) x1++;
      for (int ph = 0; ph < 8; ph++) {
         unsigned long long bit = (unsigned long long)ph;
         for (int x = x0; x < x1; x++) {
            const ZbSub &s = hs[x];
            const uint32_t size = s.pe - s.ps;
            bool stored = s.body_bits < 0;
            if (!stored) { const unsigned long long a = (bit + 3) >> 3, b = (bit + 3 + (unsigned long long)s.body_bits) >> 3; if (b - a > size) stored = true; }
            if (!stored) bit += 3 + (unsigned long long)s.body_bits;
            else { uint32_t rem = size; while (rem) { uint32_t n = rem > 65535 ? 65535 : rem; bit += 3; bit = (bit + 7) & ~7ull; bit += 32 + 8ull * n; rem -= n; } }
         }
         bits_out[8 * q + ph] = bit;
      }
      x0 = x1;
   }
}

inline void ZbPipe::stage_emit_finish(const std::vector<ZbStreamOut> &streams) {
   const uint32_t CPv = (uint32_t)cp;
   const int ns = nsub;
   ZbSub *sb = sub.p; ZbSubTabs *tb = tabs.p; uint32_t *cn = counters.p;
   const ZbWinDesc *wd = win.p; const uint32_t *wbs = wbase.p; const uint8_t *T = in_ptr;
   zb_match_t *bm = best.p; uint32_t *pen = pentry.p, *pb = pbits.p, *pcs = pchunk_sub.p;
   long npch = 0;
   {
      uint32_t v; zb_d2h(st, &v, cn + 5, 4); zb_sync(st); npch = v;
   }
   (void)tb; (void)T; (void)bm; (void)pen; (void)pb; (void)pcs; (void)wbs;
   /* E3: stitch scan, one task per stream */
   const int nstr = (int)streams.size();
   h_sout = streams; nstream = nstr;
   sout.need(nstr);
   if (zb_failed()) return;
   zb_h2d(st, sout.p, h_sout.data(), sizeof(ZbStreamOut) * nstr);
   ZbStreamOut *so = sout.p;
   /* sub-blocks are in window order; find each stream's first sub-block by scanning (serial, small) */
   zb_launch(st, nstr, ZB_LAMBDA(long q) {
      ZbStreamOut o = so[q];
      uint64_t bit = o.in_bits;
      /* locate first sub-block of window first_win by binary search on win */
      int lo = 0, hi = ns;
      while (lo < hi) { int mid = (lo + hi) >> 1; if (sb[mid].win < o.first_win) lo = mid + 1; else hi = mid; }
      for (int x = lo; x < ns && sb[x].win < o.first_win + o.nwin; x++) {
         ZbSub s = sb[x];
         const uint32_t size = s.pe - s.ps;
         const bool last_sub = (x + 1 == ns) || sb[x + 1].win != s.win;
         s.final_bit = (wd[s.win].last && last_sub) ? 1 : 0;
         s.bit_off = bit;
         bool stored = s.body_bits < 0;
         if (!stored) {
            const uint64_t a = (bit + 3) >> 3, b = (bit + 3 + (uint64_t)s.body_bits) >> 3;
            if (b - a > size) stored = true;   /* libzultra.c:345-347 */
         }
         s.stored = stored ? 1 : 0;
         if (!stored) bit += 3 + (uint64_t)s.body_bits;
         else {
            uint32_t rem = size;
            while (rem) {   /* libzultra.c:354-397 */
               uint32_t n = rem > 65535 ? 65535 : rem;
               bit += 3; bit = (bit + 7) & ~7ull; bit += 32 + 8ull * n;
               rem -= n;
            }
         }
         sb[x] = s;
      }
      o.total_bits = bit;
      so[q] = o;
   });
   zb_d2h(st, h_sout.data(), so, sizeof(ZbStreamOut) * nstr); zb_sync(st);
   /* output area: every stream gets a zeroed, word-aligned span */
   uint64_t w = 0;
   for (int q = 0; q < nstr; q++) { h_sout[q].out_word_off = w; w += (h_sout[q].total_bits + 31) / 32 + 2; }
   out.need(w + 4);
   if (zb_failed()) return;
   zb_memset(st, out.p, 0, (w + 4) * 4);
   zb_h2d(st, so, h_sout.data(), sizeof(ZbStreamOut) * nstr);
   uint32_t *ow = out.p;
   /* E4: tokens */
   zb_tag("emit_tokens");
   zb_launch(st, npch, ZB_LAMBDA(long c) {
      const uint32_t x = pcs[c];
      const ZbSub s = sb[x];
      if (s.stored) return;
      const uint32_t k = (uint32_t)c - s.pchunk_base, gb = wbs[s.win];
      const uint32_t lo = s.ps + k * CPv, hi = lo + CPv < s.pe ? lo + CPv : s.pe;
      const uint8_t *t = T + wd[s.win].in_off;
      const ZbSubTabs &tt = tb[x];
      ZbBitSink sink;
      sink.init(ow + so[wd[s.win].stream].out_word_off, s.bit_off + 3 + (uint64_t)s.hdr_bits + pb[c]);
      for (uint32_t p = pen[c]; p < hi;) {
         zb_match_t m = bm[gb + p];
         if (m.length >= ZB_MIN_MATCH) {
            const uint32_t li = m.length - ZB_MIN_MATCH;
            const int lsym = zb_len_sym(li), leb = zb_len_extra_bits(li);
            sink.put(tt.lcode[lsym], tt.llen[lsym]);
            if (leb) sink.put(li & ((1u << leb) - 1u), leb);
            const int osym = zb_off_sym(m.offset), oeb = zb_off_extra_bits(m.offset);
            sink.put(tt.ocode[osym], tt.olen[osym]);
            if (oeb) sink.put((m.offset - 1u) & ((1u << oeb) - 1u), oeb);
            p += m.length;
         } else { sink.put(tt.lcode[t[p]], tt.llen[t[p]]); p++; }
      }
      if (k + 1 == s.npchunk) sink.put(tt.lcode[ZB_EOB], tt.llen[ZB_EOB]);
      sink.finish();
   });
   /* E5: block headers and table descriptions, or stored-block headers */
   zb_launch(st, ns, ZB_LAMBDA(long x) {
      const ZbSub s = sb[x];
      const ZbSubTabs &tt = tb[x];
      uint32_t *base = ow + so[wd[s.win].stream].out_word_off;
      ZbBitSink sink;
      sink.init(base, s.bit_off);
      if (!s.stored) {
         sink.put((uint32_t)s.final_bit, 1);
         sink.put(1u + (uint32_t)s.is_dyn, 2);
         if (s.is_dyn) {
            sink.put((uint32_t)(s.nl - 257), 5); sink.put((uint32_t)(s.no - 1), 5); sink.put((uint32_t)(s.ncl - 4), 4);
            for (int i = 0; i < s.ncl; i++) sink.put((uint32_t)tt.cllen[zb_clorder(i)], 3);
            uint8_t cl[ZB_NLIT + ZB_NOFF];
            for (int i = 0; i < s.nl; i++) cl[i] = (uint8_t)tt.llen[i];
            for (int i = 0; i < s.no; i++) cl[s.nl + i] = (uint8_t)tt.olen[i];
            struct W { ZbBitSink *k; const ZbSubTabs *t;
               ZB_HD void sym(int y) { k->put(t->clcode[y], t->cllen[y]); }
               ZB_HD void rep(int y, int ev, int eb) { k->put(t->clcode[y], t->cllen[y]); k->put((uint32_t)ev, eb); } } wv = {&sink, &tt};
            zb_rle_scan(cl, s.nl + s.no, (unsigned)s.mask, wv);
         }
         sink.finish();
      } else {
         uint64_t bit = s.bit_off;
         uint32_t rem = s.pe - s.ps;
         uint8_t *bytes = (uint8_t *)base;
         while (rem) {
            const uint32_t n = rem > 65535 ? 65535 : rem;
            const uint32_t fin = (rem > 65535) ? 0u : (uint32_t)s.final_bit;
            ZbBitSink hs; hs.init(base, bit); hs.put(fin, 1); hs.put(0, 2); hs.finish();
            bit += 3; bit = (bit + 7) & ~7ull;
            /* LEN / NLEN: bytes of their own, but their word may hold a neighbour's bits */
            ZbBitSink ls; ls.init(base, bit); ls.put(n & 0xffffu, 16); ls.put((n ^ 0xffffu) & 0xffffu, 16); ls.finish();
            bit += 32 + 8ull * n;
            rem -= n;
         }
         (void)bytes;
      }
   });
   /* E6: stored payload bytes (libzultra.c:385-390), one task per path chunk of a stored sub-block.  Payload of stored
      chunk j (65535 bytes each) starts 5 bytes later than the previous one; the first starts after the padded header. */
   zb_tag("emit_stored");
   zb_launch(st, npch, ZB_LAMBDA(long c) {
      const uint32_t x = pcs[c];
      const ZbSub s = sb[x];
      if (!s.stored) return;
      const uint32_t k = (uint32_t)c - s.pchunk_base;
      const uint32_t lo = s.ps + k * CPv, hi = lo + CPv < s.pe ? lo + CPv : s.pe;
      uint8_t *bytes = (uint8_t *)(ow + so[wd[s.win].stream].out_word_off);
      const uint8_t *t = T + wd[s.win].in_off;
      const uint64_t first_payload = ((s.bit_off + 3 + 7) >> 3) + 4;
      for (uint32_t p = lo; p < hi; p++) {
         const uint32_t q = p - s.ps;
         bytes[first_payload + q + 5ull * (q / 65535u)] = t[p];
      }
   });
}

inline void ZbPipe::release_all() {
#ifndef ZB_EMU
   stager.release();
#endif
   win.release(); wbase.release(); in.release(); pk.release(); asm_tab.release(); keyA.release(); keyB.release(); valA.release(); valB.release(); rank.release(); sa.release();
   actA.release(); actB.release(); tmpA.release(); tmpB.release(); scratch.release(); sa_lcp.release(); counters.release(); tiles.release();
   tile_iv.release(); tile_pd.release(); tile_cnt.release(); tile_q.release(); groups.release(); group_words.release(); group_cnt.release(); filt_seg.release(); units.release(); unit_words.release(); unit_cnt.release(); match.release(); glen.release(); goff.release(); exitoff.release(); exitc.release(); gentry.release();
   gtokcnt.release(); gtokbase.release(); tokpos.release(); wtok.release(); wtokbase.release(); wintbase.release(); ph.release();
   gchunk_first.release(); gchunk_win.release(); nodesA.release(); nodesB.release(); nodehist.release(); chk_stat.release(); chk_flag.release();
   chk_delta.release(); chk_node.release(); wsplit.release(); wnsplit.release(); sub.release(); tabs.release(); dchunk_sub.release(); pchunk_sub.release();
   best.release(); sig_true.release(); sig_warm.release(); sig_new.release(); dok.release(); dbad.release(); pentry.release(); pbits.release(); cand.release(); dpfar.release(); hin.release(); hout.release(); wsubcnt.release(); wsubbase.release(); out.release(); sout.release();
}


/* ============================================================ checksums ============================================================
 * frame.c:74 (Adler-32) and frame.c:324 (CRC-32), computed where the data already is.  One task per 4 KiB chunk
 * produces a partial; the host folds the partials with the usual combine algebra.
 */
#define ZB_CK_CHUNK 4096
static inline uint32_t zb_gf2_times(const uint32_t *mat, uint32_t vec) { uint32_t s = 0; for (int i = 0; vec; vec >>= 1, i++) if (vec & 1) s ^= mat[i]; return s; }
static inline void zb_gf2_square(uint32_t *sq, const uint32_t *mat) { for (int i = 0; i < 32; i++) sq[i] = zb_gf2_times(mat, mat[i]); }
/* crc of A||B from crc(A), crc(B), len(B): apply len(B) zero bytes to crc(A) */
static inline uint32_t zb_crc32_combine(uint32_t c1, uint32_t c2, uint64_t len2) {
   if (!len2) return c1;
   uint32_t even[32], odd[32];
   odd[0] = 0xedb88320u;
   uint32_t row = 1;
   for (int i = 1; i < 32; i++) { odd[i] = row; row <<= 1; }
   zb_gf2_square(even, odd);
   zb_gf2_square(odd, even);
   do {
      zb_gf2_square(even, odd);
      if (len2 & 1) c1 = zb_gf2_times(even, c1);
      len2 >>= 1;
      if (!len2) break;
      zb_gf2_square(odd, even);
      if (len2 & 1) c1 = zb_gf2_times(odd, c1);
      len2 >>= 1;
   } while (len2);
   return c1 ^ c2;
}

inline void ZbPipe::stage_checksum(int kind, const std::vector<uint64_t> &range_off, const std::vector<uint64_t> &range_len, std::vector<uint32_t> &sums, uint32_t init_first) {
   const int nr = (int)range_off.size();
   sums.assign(nr, kind == 1 ? 1u : 0u);
   if (nr == 0) return;
   if (nr == 1) sums[0] = init_first;
   std::vector<uint64_t> h(2 * (size_t)nr + 1);
   uint64_t nchunk = 0;
   for (int i = 0; i < nr; i++) { h[2 * i] = range_off[i]; h[2 * i + 1] = nchunk; nchunk += (range_len[i] + ZB_CK_CHUNK - 1) / ZB_CK_CHUNK; }
   h[2 * (size_t)nr] = nchunk;
   if (nchunk == 0) return;
   ck_rng.need(3 * (size_t)nr + 2);
   std::vector<uint64_t> hh(3 * (size_t)nr);
   for (int i = 0; i < nr; i++) { hh[3 * i] = h[2 * i + 1]; hh[3 * i + 1] = range_off[i]; hh[3 * i + 2] = range_len[i]; }
   zb_h2d(st, ck_rng.p, hh.data(), hh.size() * 8);
   if (!ck_tab_ready) {
      uint32_t tab[256];
      for (uint32_t i = 0; i < 256; i++) { uint32_t c = i; for (int k = 0; k < 8; k++) c = (c >> 1) ^ ((c & 1) ? 0xedb88320u : 0u); tab[i] = c; }
      ck_tab.need(256);
      zb_h2d(st, ck_tab.p, tab, sizeof(tab)); zb_sync(st);
      ck_tab_ready = true;
   }
   ck_part.need(2 * nchunk);
   const uint64_t *rg = ck_rng.p; const uint32_t *tab = ck_tab.p; uint32_t *part = ck_part.p; const uint8_t *T = in_ptr;
   zb_launch(st, (long)nchunk, ZB_LAMBDA(long c) {
      int lo = 0, hi = nr - 1;
      while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (rg[3 * mid] <= (uint64_t)c) lo = mid; else hi = mid - 1; }
      const uint64_t k = (uint64_t)c - rg[3 * lo];
      const uint8_t *p = T + rg[3 * lo + 1] + k * ZB_CK_CHUNK;
      uint64_t rem = rg[3 * lo + 2] - k * ZB_CK_CHUNK;
      const uint32_t L = rem > ZB_CK_CHUNK ? ZB_CK_CHUNK : (uint32_t)rem;
      if (kind == 1) {
         uint32_t a = 0, b = 0;
         for (uint32_t i = 0; i < L; i++) { uint32_t v = p[i]; a += v; b += (L - i) * v; }
         part[2 * c] = a % 65521u; part[2 * c + 1] = b % 65521u;
      } else {
         uint32_t crc = 0xffffffffu;
         for (uint32_t i = 0; i < L; i++) crc = tab[(crc ^ p[i]) & 255u] ^ (crc >> 8);
         part[2 * c] = ~crc; part[2 * c + 1] = L;
      }
   });
   std::vector<uint32_t> hp(2 * nchunk);
   zb_d2h(st, hp.data(), part, hp.size() * 4); zb_sync(st);
   /* fixed-length CRC operator for full chunks */
   uint32_t op[32];
   if (kind == 2) for (int i = 0; i < 32; i++) op[i] = zb_crc32_combine(1u << i, 0, ZB_CK_CHUNK);
   for (int i = 0; i < nr; i++) {
      const uint64_t c0 = h[2 * i + 1], c1 = h[2 * i + 3 > 2 * (size_t)nr ? 2 * (size_t)nr : 2 * i + 3];
      if (kind == 1) {
         uint64_t s1 = sums[i] & 0xffff, s2 = (sums[i] >> 16) & 0xffff, left = range_len[i];
         for (uint64_t c = c0; c < c1; c++) {
            const uint64_t L = left > ZB_CK_CHUNK ? ZB_CK_CHUNK : left;
            s2 = (s2 + L * s1 + hp[2 * c + 1]) % 65521u;
            s1 = (s1 + hp[2 * c]) % 65521u;
            left -= L;
         }
         sums[i] = (uint32_t)(s1 | (s2 << 16));
      } else {
         uint32_t crc = sums[i];
         for (uint64_t c = c0; c < c1; c++) {
            const uint32_t L = hp[2 * c + 1];
            crc = (L == ZB_CK_CHUNK ? zb_gf2_times(op, crc) : zb_crc32_combine(crc, 0, L)) ^ hp[2 * c];
         }
         sums[i] = crc;
      }
   }
}

#endif
