/*
 * zb_prims.cu - cooperative sm_100a primitives: stable LSD radix sort (8-bit digits, warp-match ranking,
 * shared-memory histograms), device-wide scans (warp-shuffle), and the warp-per-tile suffix filter.
 *
 * These replace what libdivsufsort does on the CPU (reference divsufsort.c / sssort.c / trsort.c build the
 * suffix array with induced copying; here it is radix sort + prefix doubling, see zb_pipeline.h) and feed
 * the tile match finder.
 */
#include "zb_rt.h"

void zb_cuda_fail(cudaError_t e) {
   (void)e;
   /* no CPU fallback: a CUDA failure is fatal for the engine call; the pipeline stops at the next stage boundary
      (zb_failed) and the C-ABI layer reports it.  The flag belongs to the calling host thread: concurrent streams / lanes
      cannot clear or read each other's errors. */
   g_zb_cuda_error = 1;
}
thread_local int g_zb_cuda_error = 0;
long long g_zb_launches = 0;

/* ---- per-kernel timing ---- */
#include <vector>
#include <string>
#include <map>
#include <mutex>
int g_zb_prof_on = 0;
struct ZbProfRec { std::string tag; cudaEvent_t a, b; };
static std::vector<ZbProfRec> g_prof;
static std::mutex g_prof_mu;
/* several host threads (one per lane, zb_capi.cu) launch concurrently: the pending tag / record are per thread */
static thread_local const char *g_next_tag = 0;
static thread_local ZbProfRec g_cur;
void zb_tag(const char *tag) { g_next_tag = tag; }
void zb_prof_begin(int line, cudaStream_t st) {
   if (g_next_tag) g_cur.tag = g_next_tag; else { char b[32]; snprintf(b, sizeof b, "L%d", line); g_cur.tag = b; }
   g_next_tag = 0;
   cudaEventCreate(&g_cur.a); cudaEventCreate(&g_cur.b);
   cudaEventRecord(g_cur.a, st);
}
void zb_prof_end(cudaStream_t st) {
   cudaEventRecord(g_cur.b, st);
   std::lock_guard<std::mutex> g(g_prof_mu);
   g_prof.push_back(g_cur);
}
/* aggregate and clear; writes up to cap rows: name (32 bytes each), total ms, launches */
extern "C" int zultra_cuda_profile_collect(char *names, float *ms, int *counts, int cap) {
   std::map<std::string, std::pair<float, int> > agg;
   cudaDeviceSynchronize();
   for (size_t i = 0; i < g_prof.size(); i++) {
      float t = 0;
      cudaEventElapsedTime(&t, g_prof[i].a, g_prof[i].b);
      agg[g_prof[i].tag].first += t; agg[g_prof[i].tag].second += 1;
      cudaEventDestroy(g_prof[i].a); cudaEventDestroy(g_prof[i].b);
   }
   g_prof.clear();
   int n = 0;
   for (std::map<std::string, std::pair<float, int> >::iterator it = agg.begin(); it != agg.end() && n < cap; ++it, ++n) {
      snprintf(names + 32 * n, 32, "%s", it->first.c_str());
      ms[n] = it->second.first; counts[n] = it->second.second;
   }
   return n;
}
extern "C" void zultra_cuda_profile(int on) { g_zb_prof_on = on; }
#define PROF_K(tag, st) do { if (g_zb_prof_on) { zb_tag(tag); zb_prof_begin(0, st); } } while (0)
#define PROF_E(st) do { if (g_zb_prof_on) zb_prof_end(st); } while (0)

void *zb_dev_alloc(size_t n) {
   void *p = 0;
   cudaError_t e = cudaMalloc(&p, n ? n : 256);
   if (e != cudaSuccess) { fprintf(stderr, "zultra-b200: cudaMalloc(%zu) failed: %s\n", n, cudaGetErrorString(e)); g_zb_cuda_error = 1; return 0; }
   return p;
}
void zb_dev_free(void *p) { if (p) cudaFree(p); }

/* ------------------------------------------------------------------ scans ------------------------------------------------------------------ */

#define SCAN_THREADS 256
#define SCAN_ITEMS 8
#define SCAN_TILE (SCAN_THREADS * SCAN_ITEMS)

struct OpSum { __device__ static uint32_t id() { return 0; } __device__ static uint32_t op(uint32_t a, uint32_t b) { return a + b; } };
struct OpMax { __device__ static uint32_t id() { return 0; } __device__ static uint32_t op(uint32_t a, uint32_t b) { return a > b ? a : b; } };

/* block-wide exclusive scan of one value per thread; returns exclusive prefix, *total = block total (all threads) */
template <class Op>
__device__ __forceinline__ uint32_t block_exclusive(uint32_t v, uint32_t *total) {
   __shared__ uint32_t wsum[SCAN_THREADS / 32];
   __shared__ uint32_t wtot;
   const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
   uint32_t inc = v;
#pragma unroll
   for (int d = 1; d < 32; d <<= 1) {
      uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc = Op::op(inc, o);
   }
   if (lane == 31) wsum[warp] = inc;
   __syncthreads();
   if (warp == 0) {
      uint32_t w = lane < SCAN_THREADS / 32 ? wsum[lane] : Op::id();
      uint32_t winc = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
         uint32_t o = __shfl_up_sync(0xffffffffu, winc, d);
         if (lane >= d) winc = Op::op(winc, o);
      }
      uint32_t wexc = __shfl_up_sync(0xffffffffu, winc, 1);
      if (lane == 0) wexc = Op::id();
      if (lane < SCAN_THREADS / 32) wsum[lane] = wexc;
      if (lane == SCAN_THREADS / 32 - 1) wtot = winc;
   }
   __syncthreads();
   uint32_t exc = __shfl_up_sync(0xffffffffu, inc, 1);
   if (lane == 0) exc = Op::id();
   exc = Op::op(exc, wsum[warp]);
   *total = wtot;
   __syncthreads();
   return exc;
}

template <class Op>
__global__ void __launch_bounds__(SCAN_THREADS) scan_reduce_k(const uint32_t *in, uint32_t *partial, long n) {
   const long base = (long)blockIdx.x * SCAN_TILE + (long)threadIdx.x * SCAN_ITEMS;
   uint32_t acc = Op::id();
#pragma unroll
   for (int k = 0; k < SCAN_ITEMS; k++) if (base + k < n) acc = Op::op(acc, in[base + k]);
   uint32_t tot;
   block_exclusive<Op>(acc, &tot);
   if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}

/* out = scan(in) seeded with prefix[blockIdx] (or identity if prefix == 0); optionally writes the grand total */
template <class Op, bool INCLUSIVE>
__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_k(const uint32_t *in, uint32_t *out, const uint32_t *prefix, long n, uint32_t *total_dev) {
   const long base = (long)blockIdx.x * SCAN_TILE + (long)threadIdx.x * SCAN_ITEMS;
   uint32_t v[SCAN_ITEMS];
   uint32_t acc = Op::id();
#pragma unroll
   for (int k = 0; k < SCAN_ITEMS; k++) { v[k] = (base + k < n) ? in[base + k] : Op::id(); acc = Op::op(acc, v[k]); }
   uint32_t tot;
   uint32_t exc = block_exclusive<Op>(acc, &tot);
   uint32_t seed = prefix ? prefix[blockIdx.x] : Op::id();
   exc = Op::op(exc, seed);
#pragma unroll
   for (int k = 0; k < SCAN_ITEMS; k++) {
      uint32_t inc = Op::op(exc, v[k]);
      if (base + k < n) out[base + k] = INCLUSIVE ? inc : exc;
      exc = inc;
   }
   if (total_dev && blockIdx.x == gridDim.x - 1 && threadIdx.x == SCAN_THREADS - 1) *total_dev = exc;
}

size_t zb_scan_scratch_words(long n) {
   size_t tot = 0;
   long m = n;
   while (m > SCAN_TILE) { m = (m + SCAN_TILE - 1) / SCAN_TILE; tot += (size_t)((m + 63) & ~63L); }
   return tot + 64;
}

template <class Op, bool INCLUSIVE>
static void scan_impl(cudaStream_t st, const uint32_t *in, uint32_t *out, long n, uint32_t *total_dev, uint32_t *scratch) {
   if (n <= 0) { if (total_dev) ZB_CUDA_CHECK(cudaMemsetAsync(total_dev, 0, 4, st)); return; }
   long nb = (n + SCAN_TILE - 1) / SCAN_TILE;
   if (nb == 1) {
      scan_apply_k<Op, INCLUSIVE><<<1, SCAN_THREADS, 0, st>>>(in, out, 0, n, total_dev);
      zb_count_launch(1);
   } else {
      scan_reduce_k<Op><<<(unsigned)nb, SCAN_THREADS, 0, st>>>(in, scratch, n);
      scan_impl<Op, false>(st, scratch, scratch, nb, 0, scratch + ((nb + 63) & ~63L));
      scan_apply_k<Op, INCLUSIVE><<<(unsigned)nb, SCAN_THREADS, 0, st>>>(in, out, scratch, n, total_dev);
      zb_count_launch(2);
   }
   ZB_CUDA_CHECK(cudaGetLastError());
}

void zb_exclusive_sum(zb_stream_t st, const uint32_t *in, uint32_t *out, long n, uint32_t *total_dev, uint32_t *scratch) {
   scan_impl<OpSum, false>(st, in, out, n, total_dev, scratch);
}
void zb_inclusive_max(zb_stream_t st, const uint32_t *in, uint32_t *out, long n, uint32_t *scratch) {
   scan_impl<OpMax, true>(st, in, out, n, 0, scratch);
}

/* --------------------------------------------------------------- radix sort --------------------------------------------------------------- */

#define RS_THREADS 256
#define RS_ITEMS 8
#define RS_TILE (RS_THREADS * RS_ITEMS)
#define RS_WARPS (RS_THREADS / 32)

__global__ void __launch_bounds__(RS_THREADS) rs_hist_k(const uint64_t *keys, long n, int shift, uint32_t mask, uint32_t *hist, int ntiles) {
   __shared__ uint32_t h[256];
   h[threadIdx.x] = 0;
   __syncthreads();
   const long base = (long)blockIdx.x * RS_TILE;
#pragma unroll
   for (int k = 0; k < RS_ITEMS; k++) {
      long idx = base + k * RS_THREADS + threadIdx.x;
      if (idx < n) atomicAdd(&h[(uint32_t)(keys[idx] >> shift) & mask], 1u);
   }
   __syncthreads();
   hist[(size_t)threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}

/* One tile (2048 pairs) per CTA: rank every pair inside the tile (warp-level match.any, per-warp digit counters), move the
   pairs to their tile-local sorted place in shared memory, then write them out: pairs of one digit are consecutive there,
   so the global stores go out in runs instead of 32 scattered 8-byte writes per warp (the L2 sector rate was the limit). */
__global__ void __launch_bounds__(RS_THREADS) rs_scatter_k(const uint64_t *kin, const uint32_t *vin, uint64_t *kout, uint32_t *vout, long n,
                                                          int shift, uint32_t mask, const uint32_t *hist_scanned, int ntiles) {
   __shared__ uint32_t cnt[RS_WARPS][256];
   __shared__ uint32_t gbase[256];      /* global start of this tile's run of digit d, minus the run's tile-local start */
   __shared__ uint32_t dstart[256];
   __shared__ uint64_t skey[RS_TILE];
   __shared__ uint32_t sval[RS_TILE];
   __shared__ uint32_t wsum[RS_WARPS];
   const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
   for (int w = 0; w < RS_WARPS; w++) cnt[w][tid] = 0;
   const uint32_t gb = hist_scanned[(size_t)tid * ntiles + blockIdx.x];
   __syncthreads();
   const long base = (long)blockIdx.x * RS_TILE + (long)warp * (32 * RS_ITEMS);
   uint64_t key[RS_ITEMS];
   uint32_t val[RS_ITEMS], rk[RS_ITEMS];
   const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
   for (int k = 0; k < RS_ITEMS; k++) {
      const long idx = base + k * 32 + lane;
      const bool valid = idx < n;
      key[k] = valid ? kin[idx] : 0;
      val[k] = valid ? vin[idx] : 0;
   }
#pragma unroll
   for (int k = 0; k < RS_ITEMS; k++) {
      const long idx = base + k * 32 + lane;
      const bool valid = idx < n;
      const uint32_t d = valid ? ((uint32_t)(key[k] >> shift) & mask) : 0xffffffffu;
      const uint32_t peers = __match_any_sync(0xffffffffu, d);
      const uint32_t pre = __popc(peers & lt);
      const int leader = __ffs(peers) - 1;
      uint32_t old = 0;
      if (valid && lane == leader) { old = cnt[warp][d]; cnt[warp][d] = old + __popc(peers); }
      old = __shfl_sync(0xffffffffu, old, leader);
      rk[k] = old + pre;
      __syncwarp();
   }
   __syncthreads();
   /* digit tid: exclusive prefix over the warps, tile total, then exclusive scan of the totals over the digits */
   uint32_t tot = 0;
#pragma unroll
   for (int w = 0; w < RS_WARPS; w++) { uint32_t t = cnt[w][tid]; cnt[w][tid] = tot; tot += t; }
   uint32_t inc = tot;
#pragma unroll
   for (int d = 1; d < 32; d <<= 1) { uint32_t o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
   if (lane == 31) wsum[warp] = inc;
   __syncthreads();
   uint32_t woff = 0;
#pragma unroll
   for (int w = 0; w < RS_WARPS; w++) if (w < warp) woff += wsum[w];
   const uint32_t ds = woff + inc - tot;
   dstart[tid] = ds;
   gbase[tid] = gb - ds;
   __syncthreads();
#pragma unroll
   for (int k = 0; k < RS_ITEMS; k++) {
      const long idx = base + k * 32 + lane;
      if (idx < n) {
         const uint32_t d = (uint32_t)(key[k] >> shift) & mask;
         const uint32_t lp = dstart[d] + cnt[warp][d] + rk[k];
         skey[lp] = key[k]; sval[lp] = val[k];
      }
   }
   __syncthreads();
   const long tile_n = n - (long)blockIdx.x * RS_TILE < RS_TILE ? n - (long)blockIdx.x * RS_TILE : RS_TILE;
#pragma unroll
   for (int k = 0; k < RS_ITEMS; k++) {
      const int e = k * RS_THREADS + tid;
      if (e < tile_n) {
         const uint64_t kk = skey[e];
         const uint32_t d = (uint32_t)(kk >> shift) & mask;
         const size_t dst = (size_t)(uint32_t)(gbase[d] + (uint32_t)e);   /* 32-bit wrap: gbase holds start - local start */
         kout[dst] = kk;
         vout[dst] = sval[e];
      }
   }
}

size_t zb_sort_scratch_words(long n) {
   long ntiles = (n + RS_TILE - 1) / RS_TILE;
   if (ntiles < 1) ntiles = 1;
   return (size_t)256 * ntiles + zb_scan_scratch_words(256 * ntiles) + 64;
}

void zb_sort_pairs(zb_stream_t st, uint64_t *keys, uint32_t *vals, uint64_t *keys_tmp, uint32_t *vals_tmp, long n, int bit_lo, int bit_hi, uint32_t *scratch) {
   if (n <= 1 || bit_hi <= bit_lo) return;
   const int ntiles = (int)((n + RS_TILE - 1) / RS_TILE);
   uint32_t *hist = scratch;
   uint32_t *scan_scratch = scratch + (size_t)256 * ntiles;
   uint64_t *kin = keys, *kout = keys_tmp;
   uint32_t *vin = vals, *vout = vals_tmp;
   int npass = 0;
   for (int shift = bit_lo; shift < bit_hi; shift += 8, npass++) {
      const int w = (bit_hi - shift) < 8 ? (bit_hi - shift) : 8;
      const uint32_t mask = (1u << w) - 1u;
      PROF_K("rs_hist", st);
      rs_hist_k<<<ntiles, RS_THREADS, 0, st>>>(kin, n, shift, mask, hist, ntiles);
      PROF_E(st);
      scan_impl<OpSum, false>(st, hist, hist, (long)256 * ntiles, 0, scan_scratch);
      PROF_K("rs_scatter", st);
      rs_scatter_k<<<ntiles, RS_THREADS, 0, st>>>(kin, vin, kout, vout, n, shift, mask, hist, ntiles);
      PROF_E(st);
      zb_count_launch(2);
      uint64_t *tk = kin; kin = kout; kout = tk;
      uint32_t *tv = vin; vin = vout; vout = tv;
   }
   ZB_CUDA_CHECK(cudaGetLastError());
   if (npass & 1) { /* result sits in the tmp buffers */
      ZB_CUDA_CHECK(cudaMemcpyAsync(keys, keys_tmp, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
      ZB_CUDA_CHECK(cudaMemcpyAsync(vals, vals_tmp, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
   }
}

/* --------------------------------------------------------------- unit distribution --------------------------------------------------------------- */

/* A list filter (round 1; the host build still has one, tests/emu) gives every consumer its own pass over the producer's list; for the first cut - a window's suffix list
   (~1.08 M words) into its ~33 units of 32768 main + 32768 look-back positions - that was 26 words streamed per window position
   over two levels.  Every position belongs to at most TWO units (the one it is a main position of, and the next one, whose
   look-back it is in), so the cut is a stable partition: the window's list is read in segments of 4096 ranks, twice
   (count, then scatter), and every entry is routed to its units.  The LCP an entry gets in a unit's list is the minimum of the
   window LCPs after the unit's previous member up to the entry itself.  The count pass keeps per unit only its number of entries
   (warp-aggregated shared counters), its last member (atomicMax) and the minimum LCP after that member; across segments these are
   chained by a small per-unit scan.  The scatter pass keeps a 4096-bit membership bitmap per unit: popcounts give an entry's rank
   among the unit's entries of the segment, the highest set bit below it in its 32-entry word its predecessor there.  A warp
   handles exactly one such word (32 consecutive ranks) at a time and holds its LCPs in registers, so a gap minimum inside the
   word is two shuffles of a sparse table over the lanes; a gap that starts in an earlier word is the minimum up to the word,
   which a per-unit scan over the words computes once per segment (from in-block suffix minima and block minima, seeded with the
   minimum carried in from earlier segments).  Same lists, bit for bit, as filtering the window list for every unit separately. */
#define DS_SEG 4096
#define DS_THREADS 256
#define DS_WORDS (DS_SEG / 32)
#define DS_BROW (DS_WORDS + 1)      /* bitmap row stride in words, prefix row stride in u16 pairs: rows of different units start in different banks
                                       (the lanes of a warp look at the SAME word index of DIFFERENT units: unpadded, a 32-way bank conflict per access) */
#define DS_PROW (DS_WORDS + 2)
#define DS_SROW 33                  /* suffix-minimum row stride in u16: the word scan reads a different block's row in every lane, and rows of 32 would put
                                       every other lane in the same bank */

__device__ __forceinline__ int ds_find_win(const ZbDistWin *dw, int nwin, uint32_t seg) {
   int lo = 0, hi = nwin - 1;
   while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (dw[mid].seg_base <= seg) lo = mid; else hi = mid - 1; }
   return lo;
}

/* min(l[a .. lane]) over the lanes of a warp, a <= lane, where win[j] = min(l[lane - 2^j + 1 .. lane]) (cut at lane 0): the two
   windows of length 2^j, j = floor(log2(lane - a + 1)), ending at lane and starting at a cover the range.  All lanes call it. */
__device__ __forceinline__ uint32_t ds_lane_range_min(const uint32_t (&win)[6], int a, int lane) {
   const int k = 31 - __clz(lane - a + 1);
   uint32_t m = 0;
#pragma unroll
   for (int j = 0; j < 6; j++) {
      const uint32_t o = __shfl_sync(0xffffffffu, win[j], (a + (1 << j) - 1) & 31);
      if (j == k) m = min(win[j], o);
   }
   return m;
}

template <bool SCATTER>
__global__ void __launch_bounds__(DS_THREADS) unit_dist_k(const uint32_t *sa_lcp, const ZbDistWin *dw, int nwin, int nu_max, uint32_t *segrec, uint32_t *unit_words) {
   extern __shared__ uint32_t ds_sm[];
   uint16_t *smin = (uint16_t *)ds_sm;                           /* [DS_WORDS][DS_SROW] minimum of lcp[i .. end of i's block] */
   uint16_t *bmin = smin + DS_WORDS * DS_SROW;                   /* [DS_WORDS] minimum of every 32-entry block */
   uint32_t *ucnt = (uint32_t *)(bmin + DS_WORDS);               /* [nu + 1] entries per unit; SCATTER: turned into where each unit's entries start in `stage` */
   int *ulast = (int *)(ucnt + nu_max + 1);                      /* [nu] count pass: rank of the unit's last member */
   uint32_t *bm = (uint32_t *)(ulast + nu_max);                  /* [nu][DS_WORDS] SCATTER: membership bitmaps */
   uint16_t *pre = (uint16_t *)(bm + (size_t)nu_max * DS_BROW);  /* [nu][DS_WORDS] SCATTER: members before each word */
   uint16_t *gap = pre + (size_t)nu_max * DS_PROW;               /* [nu][DS_WORDS] SCATTER: minimum LCP after the last member before each word, up to the word */
   uint32_t *stage = (uint32_t *)(gap + (size_t)nu_max * DS_PROW); /* [2 * DS_SEG] SCATTER: the segment's output, unit by unit, so that it leaves in runs */
   const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
   const int w = ds_find_win(dw, nwin, blockIdx.x);
   const ZbDistWin W = dw[w];
   const uint32_t seg = blockIdx.x - W.seg_base, r0 = seg * DS_SEG;
   const uint32_t nr = W.len - r0 < DS_SEG ? W.len - r0 : DS_SEG;
   const int nu = (int)W.nu;
   {  /* A CTA lives for one load round trip plus a little work, and only a few fit an SM: pull the words of the CTA that will run
         ~1024 segments from now (16 MB further on in the same array) into L2, one 128-byte line per thread.  The address is
         exact inside a window and a few ranks off across a window end - it is only a hint. */
      const size_t tot = (size_t)dw[nwin - 1].sa_base + dw[nwin - 1].len;
      const size_t pf = (size_t)W.sa_base + r0 + (size_t)1024 * DS_SEG + (size_t)tid * 32;
      if (tid < DS_SEG / 32 && pf < tot) asm volatile("prefetch.global.L2 [%0];" :: "l"(sa_lcp + pf));
   }
   if (nu == 1) {      /* a window of one unit (batches of small streams): its list IS the unit's list */
      if (!SCATTER) { if (tid == 0) { segrec[(size_t)blockIdx.x * nu_max * 2] = nr; segrec[(size_t)blockIdx.x * nu_max * 2 + 1] = 0x1ffu | 0x10000u; } }
      else for (uint32_t idx = tid; idx < nr; idx += DS_THREADS) unit_words[(size_t)W.unit_base * (2 * ZB_MAX_OFFSET) + r0 + idx] = __ldg(sa_lcp + W.sa_base + r0 + idx);
      return;
   }
   uint32_t wv[DS_SEG / DS_THREADS];
   /* all 16 loads of a thread first, in flight together (interleaved with the shared-memory atomics below they went out one
      at a time: 57 % of the kernel's samples sat on the first use of the loaded word) */
#pragma unroll
   for (int k = 0; k < DS_SEG / DS_THREADS; k++) {
      const uint32_t idx = (uint32_t)k * DS_THREADS + tid;
      wv[k] = idx < nr ? __ldg(sa_lcp + W.sa_base + r0 + idx) : (0x1ffu << ZB_POS_BITS);
   }
   if (SCATTER) { for (int e = tid; e < nu * DS_BROW; e += DS_THREADS) bm[e] = 0; }
   else { for (int u = tid; u < nu; u += DS_THREADS) { ucnt[u] = 0; ulast[u] = -1; } }
   __syncthreads();
   /* entry idx = k * DS_THREADS + tid: warp `warp` holds block idx >> 5 whole, lane = idx & 31 */
#pragma unroll
   for (int k = 0; k < DS_SEG / DS_THREADS; k++) {
      const uint32_t idx = (uint32_t)k * DS_THREADS + tid;
      const uint32_t v = wv[k], p = v & ZB_POS_MASK;
      const int ua = p < W.hist ? 0 : (int)((p - W.hist) >> 15);
      const bool in = idx < nr, dual = p >= W.hist && ua + 1 < nu;
      if (SCATTER) {
         if (in) {
            atomicOr(bm + ua * DS_BROW + (idx >> 5), 1u << lane);
            if (dual) atomicOr(bm + (ua + 1) * DS_BROW + (idx >> 5), 1u << lane);
         }
      } else {
#pragma unroll
         for (int q = 0; q < 2; q++) {
            const int u = in && (q == 0 || dual) ? ua + q : -1;
            const uint32_t peers = __match_any_sync(0xffffffffu, (uint32_t)u);
            if (u >= 0 && lane == 31 - __clz((int)peers)) { atomicAdd(ucnt + u, (uint32_t)__popc(peers)); atomicMax(ulast + u, (int)idx); }
         }
      }
      uint32_t s = (v >> ZB_POS_BITS) & 0x1ffu;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_down_sync(0xffffffffu, s, d); if (lane + d < 32) s = min(s, o); }
      smin[(idx >> 5) * DS_SROW + lane] = (uint16_t)s;
      if (lane == 0) bmin[idx >> 5] = (uint16_t)s;
   }
   __syncthreads();
   uint32_t *rec = segrec + (size_t)blockIdx.x * nu_max * 2;
   if (!SCATTER) {
      /* per unit: entries in this segment, and the minimum LCP after its last entry (over the whole segment if it has none) */
      for (int u = warp; u < nu; u += DS_THREADS / 32) {
         const int last = ulast[u], from = last + 1, fb = (from + 31) >> 5;
         uint32_t m = lane == 0 && (from & 31) ? (uint32_t)smin[(from >> 5) * DS_SROW + (from & 31)] : 0x1ffu;
         for (int bb = fb + lane; bb < DS_WORDS; bb += 32) m = min(m, (uint32_t)bmin[bb]);
         m = __reduce_min_sync(0xffffffffu, m);
         if (lane == 0) { rec[2 * u] = ucnt[u]; rec[2 * u + 1] = m | (last >= 0 ? 0x10000u : 0u); }
      }
      return;
   }
   /* per unit and bitmap word: set bits before the word, and the minimum LCP from after the unit's last member before the word
      (from the segment start, seeded with the minimum carried in, if there is none) up to the word's start.  A word with members
      restarts that minimum at the LCPs after its last member, a word without continues it with its block minimum. */
   for (int u = warp; u < nu; u += DS_THREADS / 32) {
      const uint32_t *b = bm + u * DS_BROW;
      uint32_t run = 0, gin = rec[2 * u + 1];
#pragma unroll
      for (int j = 0; j < DS_WORDS / 32; j++) {
         const int wd = j * 32 + lane;
         const uint32_t x = b[wd];
         const uint32_t c = (uint32_t)__popc(x);
         uint32_t inc = c;
#pragma unroll
         for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
         pre[u * DS_PROW + wd] = (uint16_t)(run + inc - c);
         run += __shfl_sync(0xffffffffu, inc, 31);
         const int t = 32 - __clz((int)x);      /* first offset after the word's last member */
         uint32_t f = x != 0, g = x == 0 ? (uint32_t)bmin[wd] : t < 32 ? (uint32_t)smin[wd * DS_SROW + t] : 0x1ffu;
#pragma unroll
         for (int d = 1; d < 32; d <<= 1) {
            const uint32_t fo = __shfl_up_sync(0xffffffffu, f, d), go = __shfl_up_sync(0xffffffffu, g, d);
            if (lane >= d) { if (!f) g = min(g, go); f |= fo; }
         }
         const uint32_t incl = f ? g : min(gin, g);
         const uint32_t excl = __shfl_up_sync(0xffffffffu, incl, 1);
         gap[u * DS_PROW + wd] = (uint16_t)(lane == 0 ? gin : excl);
         gin = __shfl_sync(0xffffffffu, incl, 31);
      }
      if (lane == 0) ucnt[u + 1] = run;      /* the unit's count, turned into a start below */
   }
   __syncthreads();
   if (tid == 0) { uint32_t acc = 0; ucnt[0] = 0; for (int u = 0; u < nu; u++) { const uint32_t c = ucnt[u + 1]; ucnt[u + 1] = acc + c; acc += c; } }
   __syncthreads();
#pragma unroll
   for (int k = 0; k < DS_SEG / DS_THREADS; k++) {
      const uint32_t idx = (uint32_t)k * DS_THREADS + tid, wi = idx >> 5;
      const uint32_t v = wv[k], p = v & ZB_POS_MASK;
      const int ua = p < W.hist ? 0 : (int)((p - W.hist) >> 15);
      const bool in = idx < nr, dual = p >= W.hist && ua + 1 < nu;
      uint32_t win[6];
      win[0] = (v >> ZB_POS_BITS) & 0x1ffu;
#pragma unroll
      for (int j = 1; j < 6; j++) { const uint32_t o = __shfl_up_sync(0xffffffffu, win[j - 1], 1 << (j - 1)); win[j] = lane >= (1 << (j - 1)) ? min(win[j - 1], o) : win[j - 1]; }
#pragma unroll
      for (int q = 0; q < 2; q++) {
         const bool on = in && (q == 0 || dual);
         const int u = ua + q;
         uint32_t rank = 0, g = 0x1ffu;
         int a = lane;
         if (on) {
            const uint32_t below = bm[u * DS_BROW + wi] & ((1u << lane) - 1u);
            rank = (uint32_t)pre[u * DS_PROW + wi] + (uint32_t)__popc(below);
            /* minimum of lcp[prev + 1 .. idx]: inside the word after a predecessor there, else from the word's start on top of the gap before it */
            if (below) a = 32 - __clz((int)below);
            else { a = 0; g = gap[u * DS_PROW + wi]; }
         }
         const uint32_t m = min(g, ds_lane_range_min(win, a, lane));
         if (on) {
            /* unit u of this window: main positions from hist + u * 32768, look-back 32768 before them */
            const uint32_t m0 = W.hist + (uint32_t)u * ZB_MAX_OFFSET, ulo = m0 > ZB_MAX_OFFSET ? m0 - ZB_MAX_OFFSET : 0;
            stage[ucnt[u] + rank] = (p - ulo) | (m << ZB_POS_BITS);
         }
      }
   }
   __syncthreads();
   for (int u = warp; u < nu; u += DS_THREADS / 32) {      /* a unit's entries of this segment are one run of its list */
      const uint32_t a = ucnt[u], n = ucnt[u + 1] - a;
      uint32_t *dst = unit_words + (size_t)(W.unit_base + u) * (2 * ZB_MAX_OFFSET) + rec[2 * u];
      for (uint32_t j = lane; j < n; j += 32) dst[j] = stage[a + j];
   }
}

/* per (window, unit): counts -> offsets, trailing minima -> carried-in minima, over the window's segments */
__global__ void unit_dist_offsets_k(const ZbDistWin *dw, int nwin, int nu_max, uint32_t *segrec, uint32_t *unit_cnt, int total_units) {
   const int g = blockIdx.x * blockDim.x + threadIdx.x;
   if (g >= total_units) return;
   int lo = 0, hi = nwin - 1;
   while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (dw[mid].unit_base <= (uint32_t)g) lo = mid; else hi = mid - 1; }
   const ZbDistWin W = dw[lo];
   const int u = g - (int)W.unit_base;
   const uint32_t nseg = (W.len + DS_SEG - 1) / DS_SEG;
   uint32_t acc = 0, carry = 0x1ffu;
   for (uint32_t sg = 0; sg < nseg; sg++) {
      uint32_t *rec = segrec + ((size_t)(W.seg_base + sg) * nu_max + u) * 2;
      const uint32_t c = rec[0], th = rec[1];
      rec[0] = acc; rec[1] = carry;
      acc += c;
      const uint32_t tl = th & 0xffffu;
      carry = (th >> 16) ? tl : (tl < carry ? tl : carry);
   }
   unit_cnt[g] = acc;
}

void zb_unit_distribute(zb_stream_t st, const uint32_t *sa_lcp, const ZbDistWin *dw, int nwin, int nseg_total, int total_units, int nu_max, uint32_t *segrec,
                        uint32_t *unit_words, uint32_t *unit_cnt) {
   if (nseg_total <= 0 || total_units <= 0) return;
   const size_t smem_count = (size_t)DS_WORDS * DS_SROW * 2 + DS_WORDS * 2 + ((size_t)nu_max + 1) * 4 + (size_t)nu_max * 4;
   const size_t smem = smem_count + (size_t)nu_max * DS_BROW * 4 + (size_t)nu_max * DS_PROW * 2 * 2 + 2 * DS_SEG * 4;
   ZB_CUDA_CHECK(cudaFuncSetAttribute(unit_dist_k<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_count));
   ZB_CUDA_CHECK(cudaFuncSetAttribute(unit_dist_k<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
   PROF_K("mf_unit_dist", st);
   unit_dist_k<false><<<nseg_total, DS_THREADS, smem_count, st>>>(sa_lcp, dw, nwin, nu_max, segrec, unit_words);      /* the count pass has no bitmaps and no staging area */
   unit_dist_offsets_k<<<(total_units + 127) / 128, 128, 0, st>>>(dw, nwin, nu_max, segrec, unit_cnt, total_units);
   unit_dist_k<true><<<nseg_total, DS_THREADS, smem, st>>>(sa_lcp, dw, nwin, nu_max, segrec, unit_words);
   PROF_E(st);
   zb_count_launch(3);
   ZB_CUDA_CHECK(cudaGetLastError());
}
