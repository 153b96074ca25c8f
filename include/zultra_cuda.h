/*
 * zultra_cuda.h - the thin C-ABI between the C host library (libzultra API, stream state machine, CLI) and
 * the CUDA pipeline.  Plain pointers and sizes only.  Each entry point names the reference code it replaces.
 * All functions return 0 on success and a negative value on failure (no device, CUDA error, output too small);
 * nothing here ever computes on the CPU instead.
 */
#ifndef ZULTRA_CUDA_H
#define ZULTRA_CUDA_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct zultra_cuda_ctx_s zultra_cuda_ctx_t;

#define ZULTRA_CUDA_ERR_NODEVICE (-10)
#define ZULTRA_CUDA_ERR_CUDA     (-11)
#define ZULTRA_CUDA_ERR_DST      (-2)
#define ZULTRA_CUDA_ERR_ARG      (-12)

/* Context = one CUDA device + stream + scratch buffers (replaces the per-stream arrays allocated at
   libzultra.c:135-147 and the divsufsort context, divsufsort.c:340).  device < 0 selects the current device. */
int zultra_cuda_ctx_create(zultra_cuda_ctx_t **ppCtx, int nDevice);
void zultra_cuda_ctx_destroy(zultra_cuda_ctx_t *pCtx);
int zultra_cuda_device_count(void);
/* Borrow / return a pooled context (keeps device buffers alive between zultra_memory_compress calls). */
int zultra_cuda_ctx_acquire(zultra_cuda_ctx_t **ppCtx, int nDevice);
void zultra_cuda_ctx_release(zultra_cuda_ctx_t *pCtx);
void zultra_cuda_release_cached(void);

/*
 * Compress consecutive max-blocks of ONE stream: the body of the per-block loop at libzultra.c:269-438
 * (zultra_build_suffix_array, zultra_skip_matches, zultra_find_all_matches, zultra_block_split, the
 * static/dynamic decision, zultra_block_deflate, stored fallback).
 *   pHistory/nHistorySize  up to 32768 bytes that precede pInData (tail of the previous block, or the preset dictionary)
 *   pInData/nInDataSize    whole max-blocks; only the last one may be short
 *   nDoFinalize            non-zero: the last block ends the stream (BFINAL on its last sub-block, libzultra.c:328)
 *   nInBitCount            bits already pending in the stream's current output byte (the bit writer state that
 *                          persists across blocks, libzultra.c:427-434); the caller keeps that byte and ORs
 *                          pOutData[0] into it
 *   nFlags/pnChecksum      ZULTRA_FLAG_xxx framing; *pnChecksum is the running Adler-32/CRC-32 of the stream and is
 *                          advanced over pInData on the device (zultra_frame_update_checksum, libzultra.c:279)
 *   pOutData               receives ceil(total_bits/8) bytes; bit 0 of byte 0 is stream bit -nInBitCount
 *   *pnOutBitCount         total bits in pOutData including the nInBitCount leading pending bits
 */
int zultra_cuda_compress_blocks(zultra_cuda_ctx_t *pCtx, const unsigned char *pHistory, int nHistorySize,
                                const unsigned char *pInData, size_t nInDataSize, unsigned int nMaxBlockSize, int nDoFinalize,
                                unsigned int nInBitCount, unsigned int nFlags, unsigned int *pnChecksum,
                                unsigned char *pOutData, size_t nMaxOutDataSize, unsigned long long *pnOutBitCount);

/* Same, input already resident in device memory and output left there (benchmarks: HBM-resident timing). */
int zultra_cuda_compress_blocks_device(zultra_cuda_ctx_t *pCtx, const void *pDevInData, size_t nInDataSize, unsigned int nMaxBlockSize,
                                       int nDoFinalize, unsigned int nFlags, unsigned int *pnChecksum,
                                       void *pDevOutData, size_t nMaxOutDataSize, unsigned long long *pnOutBitCount);

/*
 * Sharded operation (multi-GPU): a shard = a contiguous range of max-blocks of one stream on one device, its input
 * resident as [nHistorySize bytes preceding the shard | shard bytes].  Everything except the final placement of bits is
 * independent of the entering bit phase, so shard_prepare runs the pipeline and reports the shard's total size in bits
 * for each of the 8 possible entering phases (the stored-block decision of libzultra.c:345-347 depends on the phase);
 * once the phases of the preceding shards are known, shard_emit writes the shard's bitstream for its true phase.
 * *pnChecksum (shard_prepare) receives the checksum of the shard's own bytes started from the initial value given;
 * zultra_cuda_checksum_combine folds shard checksums in order.
 */
int zultra_cuda_shard_prepare(zultra_cuda_ctx_t *pCtx, const void *pDevInData, int nHistorySize, size_t nInDataSize, unsigned int nMaxBlockSize,
                              int nDoFinalize, unsigned int nFlags, unsigned int *pnChecksum, unsigned long long *pnPhaseBits8);
int zultra_cuda_shard_emit(zultra_cuda_ctx_t *pCtx, unsigned int nInBitCount, void *pDevOutData, size_t nMaxOutDataSize, unsigned long long *pnOutBitCount);
unsigned int zultra_cuda_checksum_combine(unsigned int nFlags, unsigned int nChecksum1, unsigned int nChecksum2, unsigned long long nLength2);

/*
 * Several GPUs behind one context (SURVEY 8(b) extension ii; north_star "sharded across the GPUs of one 8xB200 box").  After
 * zultra_cuda_ctx_set_devices(ctx, n) every zultra_cuda_compress_blocks call on that context with at least two max-blocks
 * spreads them over devices device .. device+n-1 (mod the device count): chunks of a few max-blocks dealt round-robin, one
 * host thread and pipeline per device, phase maps composed on the host, every chunk's bytes copied from its device straight
 * to their byte offset in pOutData.  The libzultra front end sets this from ZULTRA_CUDA_DEVICES, so zultra_memory_compress,
 * the streaming API and the CLI use n GPUs.  Returns the device count actually used.  (Per-block loop: libzultra.c:269-438.)
 */
int zultra_cuda_ctx_set_devices(zultra_cuda_ctx_t *pCtx, int nDevices);

/*
 * One process per GPU (bench.py under torchrun): the same chunk scheme with the exchange left to the caller (NCCL).
 * chunks_prepare: nChunks chunks of ONE device-resident buffer, chunk i = [pnChunkHistory[i] bytes of preceding input |
 * pnChunkSize[i] bytes] starting at byte pnChunkOffset[i]; returns an 8-entry phase map (pnPhaseBits8 + 8 i) and the
 * checksum of the chunk's own bytes from the initial value, per chunk.  chunks_emit: entering phase per chunk (from the
 * composed maps of ALL ranks); leaves chunk i's bitstream at *ppDevOut + pnOutOffset[i] (device memory owned by the context,
 * valid until its next call), pnOutBits[i] bits including the entering ones.  stitch_device (the gathering rank): OR-merges
 * parts at their absolute bit offsets into a zeroed device buffer - the "shift and concatenate" of the stitch; every source
 * part must be followed by at least 8 readable zero bytes (the spans zultra_cuda_chunks_emit leaves are).
 */
int zultra_cuda_chunks_prepare(zultra_cuda_ctx_t *pCtx, const void *pDevInData, int nChunks, const size_t *pnChunkOffset, const int *pnChunkHistory,
                               const size_t *pnChunkSize, const int *pnChunkFinalize, unsigned int nMaxBlockSize, unsigned int nFlags,
                               unsigned int *pnChecksums, unsigned long long *pnPhaseBits8);
int zultra_cuda_chunks_emit(zultra_cuda_ctx_t *pCtx, const unsigned int *pnInBitCounts, void **ppDevOut, size_t *pnOutOffset, unsigned long long *pnOutBits);
int zultra_cuda_stitch_device(zultra_cuda_ctx_t *pCtx, void *pDevDst, int nParts, const void *const *ppDevSrc, const unsigned long long *pnDstBitOffset,
                              const unsigned long long *pnBits);

/* Batch of independent streams, each equal to zultra_memory_compress(p, n, .., nFlags, nMaxBlockSize) (config 5 of
   BASELINE.json; an extension, not in the reference).  pnOutSizes[i] = (size_t)-1 on per-stream failure. */
int zultra_cuda_memory_compress_batch(zultra_cuda_ctx_t *pCtx, const unsigned char *const *ppInData, const size_t *pnInSizes,
                                      unsigned char *const *ppOutData, const size_t *pnMaxOutSizes, size_t *pnOutSizes, size_t nStreams,
                                      unsigned int nFlags, unsigned int nMaxBlockSize);

/* Checksums on the device for device-resident input (frame.c:74 Adler-32, frame.c:324 CRC-32). */
int zultra_cuda_checksum_device(zultra_cuda_ctx_t *pCtx, const void *pDevData, size_t nSize, unsigned int nFlags, unsigned int *pnChecksum);

/* ---- stage dumps for the parity tests (window = history + block bytes, as matchfinder.c:49 sees it) ---- */
/* packed SA|LCP words as they stand after matchfinder.c:90 */
int zultra_cuda_window_sa_lcp(zultra_cuda_ctx_t *pCtx, const unsigned char *pWindow, int nWindowSize, unsigned int *pOutWords);
/* match[(i - nHistory) * 8 + m] = {u16 length, u16 offset} as after zultra_find_all_matches (matchfinder.c:262) */
int zultra_cuda_window_matches(zultra_cuda_ctx_t *pCtx, const unsigned char *pWindow, int nHistory, int nWindowSize, unsigned short *pOutMatches,
                               unsigned int nTileSize);
/* per sub-block results of zultra_block_split / the decision at libzultra.c:317-324 / zultra_block_deflate:
   pInfo: 8 ints per sub-block {start, end, is_dynamic, static_cost, dynamic_cost, body_bits, stored, rle_mask};
   pLitLen 288 / pOffLen 32 ints per sub-block; pBest nWindowSize entries {u16 length,u16 offset}.  Returns sub-block count. */
int zultra_cuda_block_stages(zultra_cuda_ctx_t *pCtx, const unsigned char *pWindow, int nHistory, int nWindowSize,
                             int *pInfo, int *pLitLen, int *pOffLen, unsigned short *pBest);

/* milliseconds spent per stage in the last compress call: {h2d, sa+lcp, match, greedy+split, parse, emit, d2h, total} */
int zultra_cuda_last_timings(zultra_cuda_ctx_t *pCtx, float *pMs8);
/* counters of the last call: {windows, sub-blocks, suffix-sort rounds, parse chunks redone, kernel launches, 0 (unused),
   devices of the last call spread over several devices (0 before the first), match-finder tiles} */
int zultra_cuda_last_counters(zultra_cuda_ctx_t *pCtx, long long *pCounters8);

/* kernels this library has launched in this process so far (all contexts, all host threads) */
long long zultra_cuda_launch_count(void);
/* ZULTRA_CUDA_TRACE=1: one more line "[zb <ms since the first traced event>] what" on stderr (the host library and the tool mark
   their own milestones with it); a no-op otherwise */
void zultra_cuda_trace(const char *pszWhat);

/* per-kernel CUDA-event timing: zultra_cuda_profile(1) turns it on; collect returns rows {32-byte name, total ms, launches} and clears */
void zultra_cuda_profile(int nOn);
int zultra_cuda_profile_collect(char *pNames, float *pMs, int *pCounts, int nMaxRows);

#ifdef __cplusplus
}
#endif
#endif
