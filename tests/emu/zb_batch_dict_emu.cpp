/* Host build of the pipeline (tests only): the dictionary batch path, a C entry point for ctypes. */
#include "zb_engine.h"

extern "C" {
/* batch of streams against one preset dictionary, host build of the zultra_cuda_memory_compress_batch_dict engine call: the
   dictionary's last <= 32768 bytes are every stream's first history, the payloads go packed through stage_assemble.  Stream i's
   raw deflate bitstream lands at out + out_off[i] (out_bits[i] bits), cks[i] = its checksum (flags as in the C-ABI). */
long emu_batch_dict(int ns, const uint8_t *const *data, const size_t *n, const uint8_t *dict, int dict_size, unsigned block_size, unsigned flags,
                    uint8_t *out, long cap, size_t *out_off, unsigned long long *out_bits, unsigned *cks) {
   ZbPipe p; p.st = 0;
   const int kind = (flags & 2) ? 2 : ((flags & 1) ? 1 : 0);
   const uint32_t dk = dict_size > 0 ? (uint32_t)std::min(dict_size, ZB_HISTORY) : 0u;
   std::vector<ZbStreamIn> s((size_t)ns);
   for (int i = 0; i < ns; i++) { ZbStreamIn t = {data[i], n[i], dk ? dict + (dict_size - (int)dk) : 0, dk, 1, 0, kind == 1 ? 1u : 0u}; s[i] = t; }
   std::vector<uint8_t> o; std::vector<ZbStreamRes> r;
   ZbRunOpts opt; opt.checksum_kind = kind; opt.shared_hist = dk ? 1 : 0;
   if (zb_run_batch(p, s.data(), ns, block_size, o, r, opt)) return -1;
   if ((long)o.size() > cap) return -2;
   memcpy(out, o.data(), o.size());
   for (int i = 0; i < ns; i++) { out_off[i] = r[i].out_off; out_bits[i] = r[i].total_bits; cks[i] = r[i].checksum; }
   p.release_all();
   return (long)o.size();
}
}
