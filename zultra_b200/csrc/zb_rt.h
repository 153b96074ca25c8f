/*
 * zb_rt.h - tiny runtime layer under the pipeline: device memory, task launch, atomics, and the
 * cooperative primitives (radix sort, scans, tile filter) the pipeline calls.
 *
 * Product build (nvcc, ZB_EMU undefined): everything runs on the GPU; a missing device is a hard error.
 * Test build (g++ -DZB_EMU, tests/emu only): tasks run in a host loop so the per-task logic can be diffed
 * against the reference without a GPU.  The product library never contains this mode.
 */
#ifndef ZB_RT_H
#define ZB_RT_H
#include <stdint.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "zb_core.h"

#ifdef ZB_EMU
/* ---------------- host emulation (tests only) ---------------- */
typedef int zb_stream_t;
#define ZB_LAMBDA [=]
#define ZB_DEV
template <class F> static inline void zb_launch_(int, zb_stream_t, long n, F f, int = 128) { for (long i = 0; i < n; i++) f(i); }
static inline void zb_tag(const char *) {}
static inline void *zb_dev_alloc(size_t n) { void *p = malloc(n ? n : 1); if (!p) { fprintf(stderr, "emu alloc fail\n"); abort(); } return p; }
static inline void zb_dev_free(void *p) { free(p); }
static inline void *zb_host_alloc(size_t n) { return malloc(n ? n : 1); }
static inline void zb_host_free(void *p) { free(p); }
static inline void zb_memset(zb_stream_t, void *p, int v, size_t n) { memset(p, v, n); }
static inline void zb_h2d(zb_stream_t, void *d, const void *h, size_t n) { memcpy(d, h, n); }
static inline void zb_d2h(zb_stream_t, void *h, const void *d, size_t n) { memcpy(h, d, n); }
static inline void zb_d2d(zb_stream_t, void *d, const void *s, size_t n) { memcpy(d, s, n); }
static inline void zb_sync(zb_stream_t) {}
static inline int zb_atomic_add(int *p, int v) { int o = *p; *p += v; return o; }
static inline unsigned zb_atomic_add(unsigned *p, unsigned v) { unsigned o = *p; *p += v; return o; }
static inline int zb_atomic_max(int *p, int v) { int o = *p; if (v > o) *p = v; return o; }
static inline unsigned zb_atomic_or(unsigned *p, unsigned v) { unsigned o = *p; *p |= v; return o; }
static inline int zb_sm_count() { return 148; }
static inline bool zb_failed() { return false; }
#else
/* ---------------- CUDA ---------------- */
#include <cuda_runtime.h>
typedef cudaStream_t zb_stream_t;
#define ZB_LAMBDA [=] __device__
#define ZB_DEV __device__
#define ZB_CUDA_CHECK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "zultra-b200: CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); zb_cuda_fail(e_); } } while (0)
void zb_cuda_fail(cudaError_t e);
extern thread_local int g_zb_cuda_error;   /* set by a failed CUDA call / allocation on this host thread (zb_prims.cu) */
static inline bool zb_failed() { return g_zb_cuda_error != 0; }
extern long long g_zb_launches;   /* kernels launched by this library (bench.py reports it); several host threads count */
static inline void zb_count_launch(int n) { __atomic_fetch_add(&g_zb_launches, (long long)n, __ATOMIC_RELAXED); }
template <class F> __global__ void zb_task_kernel(long n, F f) {
   long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
   if (i < n) f(i);
}
/* optional per-kernel timing (CUDA events on the launching stream), enabled by zultra_cuda_profile() */
extern int g_zb_prof_on;
void zb_tag(const char *tag);                                /* name the next launch */
void zb_prof_begin(int line, cudaStream_t st);
void zb_prof_end(cudaStream_t st);
template <class F> static inline void zb_launch_(int line, zb_stream_t st, long n, F f, int blk = 128) {
   if (n <= 0) { zb_tag(0); return; }
   /* few tasks are the serial per-sub-block / per-node ones (Huffman builds, splitter scans): give each its own warp, so that
      32 unrelated control flows do not serialise inside one, and its own SM share instead of crowding two SMs */
   if (n <= 4096) blk = 1;
   if (g_zb_prof_on) zb_prof_begin(line, st);
   zb_task_kernel<<<(unsigned)((n + blk - 1) / blk), blk, 0, st>>>(n, f);
   if (g_zb_prof_on) zb_prof_end(st);
   zb_count_launch(1);
   ZB_CUDA_CHECK(cudaGetLastError());
}
void *zb_dev_alloc(size_t n);
void zb_dev_free(void *p);
/* page-locked host staging memory (multi-stream batches are gathered into / scattered out of it around one DMA each way) */
static inline void *zb_host_alloc(size_t n) { void *p = 0; ZB_CUDA_CHECK(cudaHostAlloc(&p, n ? n : 1, cudaHostAllocDefault)); return p; }
static inline void zb_host_free(void *p) { if (p) cudaFreeHost(p); }
static inline void zb_memset(zb_stream_t st, void *p, int v, size_t n) { if (n) ZB_CUDA_CHECK(cudaMemsetAsync(p, v, n, st)); }
static inline void zb_h2d(zb_stream_t st, void *d, const void *h, size_t n) { if (n) ZB_CUDA_CHECK(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, st)); }
static inline void zb_d2h(zb_stream_t st, void *h, const void *d, size_t n) { if (n) ZB_CUDA_CHECK(cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, st)); }
static inline void zb_d2d(zb_stream_t st, void *d, const void *s, size_t n) { if (n) ZB_CUDA_CHECK(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToDevice, st)); }
static inline void zb_sync(zb_stream_t st) { ZB_CUDA_CHECK(cudaStreamSynchronize(st)); }
static inline int zb_sm_count() {   /* SMs of the current device (B200: 148) */
   int dev = 0, n = 0;
   if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
   return n;
}
__device__ __forceinline__ int zb_atomic_add(int *p, int v) { return atomicAdd(p, v); }
__device__ __forceinline__ unsigned zb_atomic_add(unsigned *p, unsigned v) { return atomicAdd(p, v); }
__device__ __forceinline__ int zb_atomic_max(int *p, int v) { return atomicMax(p, v); }
__device__ __forceinline__ unsigned zb_atomic_or(unsigned *p, unsigned v) { return atomicOr(p, v); }
#endif

#define zb_launch(...) zb_launch_(__LINE__, __VA_ARGS__)

/* ---- cooperative primitives (zb_prims.cu on the GPU, zb_prims_emu.cpp in the test build) ---- */

/* stable LSD radix sort of (key,val) pairs on key bits [lo,hi); result ends in keys/vals (tmp are scratch) */
void zb_sort_pairs(zb_stream_t st, uint64_t *keys, uint32_t *vals, uint64_t *keys_tmp, uint32_t *vals_tmp, long n, int bit_lo, int bit_hi,
                   uint32_t *scratch /* >= zb_sort_scratch_words(n) */);
size_t zb_sort_scratch_words(long n);
/* out[i] = sum_{j<i} in[j]; returns nothing, total written to *total_dev (device ptr, may be null). in==out allowed */
void zb_exclusive_sum(zb_stream_t st, const uint32_t *in, uint32_t *out, long n, uint32_t *total_dev, uint32_t *scratch /* >= zb_scan_scratch_words(n) */);
/* out[i] = max_{j<=i} in[j] */
void zb_inclusive_max(zb_stream_t st, const uint32_t *in, uint32_t *out, long n, uint32_t *scratch);
size_t zb_scan_scratch_words(long n);

/*
 * Tile filter: for each tile t, stream a list of packed pos|lcp<<22 words in suffix-array order (src + src_base,
 * src_n words, or src_cnt[src_cnt_idx] words when src_cnt_idx >= 0; positions in the list are relative to src_lo),
 * keep the suffixes whose window position lies in [lo, hi), min-reduce the LCP over skipped entries, and write
 * (pos-lo)|lcp<<22 words to out + t*stride (count to cnt[t]).  Used twice: window -> 64 Ki-position units -> tiles.
 */
struct ZbTileDesc { uint32_t win; uint32_t lo, m0, hi; uint64_t src_base; uint32_t src_n; uint32_t src_lo; int32_t src_cnt_idx; uint32_t wlen; };
void zb_tile_filter(zb_stream_t st, const uint32_t *src, const uint32_t *src_cnt, const ZbTileDesc *tiles, int ntiles, int first_tile, uint32_t *out, size_t stride, uint32_t *cnt,
                    int nseg /* warps per tile: the source list is cut into that many segments */, uint32_t *seg_scratch /* >= 2 * ntiles * nseg words */);

/*
 * Unit distribution (CUDA build): the cut of every window's suffix list into its units (32768 main positions + the 32768 before
 * them) as ONE stable partition - see zb_prims.cu.  dw: one descriptor per window (device memory); unit u of a window covers
 * main positions [hist + u * 32768, ..) and writes its list to unit_words + (unit_base + u) * 65536, its length to unit_cnt.
 */
struct ZbDistWin { uint32_t sa_base, len, hist, unit_base, nu, seg_base, pad[2]; };
#ifndef ZB_EMU
void zb_unit_distribute(zb_stream_t st, const uint32_t *sa_lcp, const ZbDistWin *dw, int nwin, int nseg_total, int total_units, int nu_max,
                        uint32_t *segrec /* >= 2 * nseg_total * nu_max words */, uint32_t *unit_words, uint32_t *unit_cnt);
#endif

#endif
