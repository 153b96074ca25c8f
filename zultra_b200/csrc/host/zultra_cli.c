/*
 * zultra_cli.c - command-line tool of zultra-b200, a drop-in for the reference `zultra` tool
 * (tool/zultra.c:778-935): same flags (-z -d -c -cbench -test -quicktest -D<file> -v -deflate -gzip -zlib),
 * gzip framing by default, -D only with -zlib, exit code 100 on any error, 16 KiB streaming chunks.
 * Verification (-c, -test) inflates with the system zlib, as the reference does with its vendored copy.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/time.h>
#include <unistd.h>
#include <zlib.h>
#include "libzultra.h"
#include "zultra_cuda.h"

#define OPT_VERBOSE 1
#define FMT_DEFLATE 2
#define FMT_ZLIB 4
#define FMT_GZIP 8
#define FMT_MASK 14
#define CHUNK 16384

static long long g_t0;
static long long now_us(void) { struct timeval t; gettimeofday(&t, NULL); return (long long)t.tv_sec * 1000000LL + t.tv_usec; }
static unsigned int lib_flags(unsigned int opt) { return (opt & FMT_ZLIB) ? ZULTRA_FLAG_ZLIB_FRAMING : ((opt & FMT_GZIP) ? ZULTRA_FLAG_GZIP_FRAMING : 0); }

static void report(zultra_status_t st, const char *in, const char *out, const char *dict) {
   switch (st) {
   case ZULTRA_ERROR_SRC: fprintf(stderr, "error reading '%s'\n", in); break;
   case ZULTRA_ERROR_DST: fprintf(stderr, "error writing '%s'\n", out); break;
   case ZULTRA_ERROR_DICTIONARY: fprintf(stderr, "error reading dictionary '%s'\n", dict); break;
   case ZULTRA_ERROR_MEMORY: fprintf(stderr, "'%s': out of memory\n", in); break;
   case ZULTRA_ERROR_COMPRESSION: fprintf(stderr, "'%s': internal compression error\n", in); break;
   case ZULTRA_OK: fprintf(stderr, "'%s': unfinished compression\n", in); break;
   case ZULTRA_STREAM_END: break;
   default: fprintf(stderr, "unknown compression error %d\n", (int)st); break;
   }
}

static int do_compress(const char *in, const char *out, const char *dictfile, unsigned int opt) {
   FILE *fi = NULL, *fo = NULL;
   unsigned char *ib = NULL, *ob = NULL;
   void *dict = NULL; int dict_size = 0;
   zultra_stream_t s;
   zultra_status_t st = ZULTRA_OK;
   int flush = 0;
   long long t0 = now_us();
   memset(&s, 0, sizeof(s));
   fi = fopen(in, "rb"); if (!fi) st = ZULTRA_ERROR_SRC;
   if (!st) { fo = fopen(out, "wb"); if (!fo) st = ZULTRA_ERROR_DST; }
   if (!st) st = zultra_dictionary_load(dictfile, &dict, &dict_size);
   if (!st) { ib = (unsigned char *)malloc(CHUNK); ob = (unsigned char *)malloc(CHUNK); if (!ib || !ob) st = ZULTRA_ERROR_MEMORY; }
   if (!st) st = zultra_stream_init(&s, lib_flags(opt), 0);
   zultra_cuda_trace("cli: stream initialised");
   if (!st && dict) st = zultra_stream_set_dictionary(&s, dict, dict_size);
   while (!flush && !st) {
      int progress = 0;
      s.avail_in = fread(ib, 1, CHUNK, fi);
      if (ferror(fi)) { st = ZULTRA_ERROR_SRC; break; }
      flush = feof(fi) ? ZULTRA_FINALIZE : ZULTRA_CONTINUE;
      s.next_in = ib;
      do {
         size_t n;
         s.avail_out = CHUNK; s.next_out = ob;
         st = zultra_stream_compress(&s, flush);
         if (st != ZULTRA_OK && st != ZULTRA_STREAM_END) break;
         n = CHUNK - s.avail_out;
         if (n) progress = 1;
         if (fwrite(ob, 1, n, fo) != n || ferror(fo)) { st = ZULTRA_ERROR_DST; break; }
      } while (s.avail_out == 0);
      if ((st == ZULTRA_OK || st == ZULTRA_STREAM_END) && s.avail_in != 0) st = ZULTRA_ERROR_COMPRESSION;
      if ((st == ZULTRA_OK || st == ZULTRA_STREAM_END) && !flush && progress && s.total_in && s.total_out >= 1024) {
         fprintf(stdout, "\r%lld => %lld (%g %%)     \b\b\b\b\b", (long long)s.total_in, (long long)s.total_out, (double)(s.total_out * 100.0 / s.total_in));
         fflush(stdout);
      }
      if (st == ZULTRA_STREAM_END && !flush) st = ZULTRA_ERROR_COMPRESSION;
      if (st == ZULTRA_OK && !flush) continue;
      if (st == ZULTRA_OK && flush) break;
   }
   {
      unsigned long long tin = s.total_in, tout = s.total_out;
      zultra_cuda_trace("cli: last byte written");
      zultra_stream_end(&s);
      free(ob); free(ib);
      zultra_dictionary_free(&dict);
      if (fo) fclose(fo);
      if (fi) fclose(fi);
      zultra_cuda_trace("cli: files closed");
      if (st != ZULTRA_STREAM_END) { report(st, in, out, dictfile); return 100; }
      if ((opt & OPT_VERBOSE) && tin && tout) {
         double dt = (double)(now_us() - t0) / 1000000.0;
         fprintf(stdout, "\rCompressed '%s' in %g seconds, %.02g Mb/s, %lld into %lld bytes ==> %g %%\n", in, dt, ((double)tin / 1048576.0) / dt,
                 (long long)tin, (long long)tout, (double)(tout * 100.0 / tin));
      }
   }
   return 0;
}

/* inflate `comp` (any framing) and compare with `orig` */
static int inflate_matches(const unsigned char *comp, size_t ncomp, const unsigned char *orig, size_t norig, unsigned int opt, const void *dict, int dict_size) {
   z_stream z;
   unsigned char *buf = (unsigned char *)malloc(norig + 16);
   int rc, ok;
   if (!buf) return 0;
   memset(&z, 0, sizeof(z));
   if (inflateInit2(&z, (opt & FMT_DEFLATE) ? -15 : ((opt & FMT_GZIP) ? 16 + 15 : 15)) != Z_OK) { free(buf); return 0; }
   z.next_in = (Bytef *)comp; z.avail_in = (uInt)ncomp; z.next_out = buf; z.avail_out = (uInt)(norig + 16);
   rc = inflate(&z, Z_FINISH);
   if (rc == Z_NEED_DICT && dict) { inflateSetDictionary(&z, (const Bytef *)dict, (uInt)dict_size); rc = inflate(&z, Z_FINISH); }
   ok = (rc == Z_STREAM_END && z.total_out == norig && !memcmp(buf, orig, norig));
   inflateEnd(&z);
   free(buf);
   return ok;
}

static unsigned char *read_file(const char *name, size_t *n) {
   FILE *f = fopen(name, "rb");
   unsigned char *b;
   long sz;
   if (!f) return NULL;
   fseek(f, 0, SEEK_END); sz = ftell(f); fseek(f, 0, SEEK_SET);
   b = (unsigned char *)malloc((size_t)sz + 1);
   if (b && fread(b, 1, (size_t)sz, f) != (size_t)sz) { free(b); b = NULL; }
   fclose(f);
   *n = (size_t)sz;
   return b;
}

static int do_compare(const char *comp, const char *orig, const char *dictfile, unsigned int opt) {
   size_t nc = 0, no = 0;
   unsigned char *c = read_file(comp, &nc), *o = read_file(orig, &no);
   void *dict = NULL; int dict_size = 0, ok = 0;
   long long t0 = now_us();
   if (c && o && zultra_dictionary_load(dictfile, &dict, &dict_size) == ZULTRA_OK) ok = inflate_matches(c, nc, o, no, opt, dict, dict_size);
   zultra_dictionary_free(&dict);
   free(c); free(o);
   if (!ok) { fprintf(stderr, "error comparing compressed file '%s' with original '%s'\n", comp, orig); return 100; }
   if (opt & OPT_VERBOSE) fprintf(stdout, "Compared '%s' in %g seconds\n", comp, (double)(now_us() - t0) / 1000000.0);
   return 0;
}

static int do_cbench(const char *in, const char *out, unsigned int opt) {
   size_t n = 0, cap, best_n = 0;
   unsigned char *data = read_file(in, &n), *buf;
   long long best = -1;
   int i;
   FILE *f;
   if (!data) { fprintf(stderr, "error reading '%s'\n", in); return 100; }
   cap = zultra_memory_bound(n, lib_flags(opt), 0);
   buf = (unsigned char *)malloc(cap + 2048);
   if (!buf) { free(data); return 100; }
   for (i = 0; i < 5; i++) {
      long long t0, dt;
      size_t r;
      memset(buf, 0x55, 1024); memset(buf + 1024 + cap, 0xaa, 1024);   /* guard bytes (tool/zultra.c:708-752) */
      t0 = now_us();
      r = zultra_memory_compress(data, n, buf + 1024, cap, lib_flags(opt), 0);
      dt = now_us() - t0;
      if (r == (size_t)-1) { fprintf(stderr, "compression error\n"); free(buf); free(data); return 100; }
      {
         size_t k;
         for (k = 0; k < 1024; k++) if (buf[k] != 0x55 || buf[1024 + cap + k] != 0xaa) { fprintf(stderr, "buffer overrun\n"); free(buf); free(data); return 100; }
      }
      if (best < 0 || dt < best) best = dt;
      best_n = r;
   }
   f = fopen(out, "wb");
   if (f) { fwrite(buf + 1024, 1, best_n, f); fclose(f); }
   fprintf(stdout, "compressed size: %lld bytes\n", (long long)best_n);
   fprintf(stdout, "compression time: %lld microseconds (%g Mb/s)\n", best, ((double)n / 1048576.0) / ((double)best / 1000000.0));
   free(buf); free(data);
   return 0;
}

/* self-test data of the reference's shape (tool/zultra.c:425-463): random literals mixed with copies */
static size_t gen_data(unsigned char *b, size_t n, unsigned int seed, int nsyms, float match_prob) {
   size_t i = 0;
   int mp = (int)((float)RAND_MAX * match_prob);
   srand(seed);
   if (n) b[i++] = (unsigned char)(rand() % nsyms);
   while (i < n) {
      if (rand() > mp) b[i++] = (unsigned char)(rand() % nsyms);
      else {
         size_t len = 3 + (size_t)(rand() & 1023), off = 1 + (size_t)rand() % (i > 32768 ? 32768 : i);
         while (len-- && i < n) { b[i] = b[i - off]; i++; }
      }
   }
   return n;
}

static int do_self_test(int quick) {
   static const int syms[12] = {1, 2, 3, 15, 30, 56, 96, 137, 178, 191, 255, 256};
   size_t maxn = quick ? 4096 : 131072, n;
   unsigned char *data = (unsigned char *)malloc(maxn), *comp;
   size_t cap = zultra_memory_bound(maxn, ZULTRA_FLAG_ZLIB_FRAMING, 0);
   unsigned int seed = 123;
   int s, p, fails = 0, tests = 0;
   comp = (unsigned char *)malloc(cap);
   if (!data || !comp) return 100;
   /* too-small output buffers must fail cleanly (tool/zultra.c:521-524) */
   for (s = 0; s < 12; s++) {
      gen_data(data, 4096, seed++, syms[s], 0.5f);
      if (zultra_memory_compress(data, 4096, comp, 8, ZULTRA_FLAG_ZLIB_FRAMING, 0) != (size_t)-1) { fprintf(stderr, "small-buffer test %d failed\n", s); fails++; }
      tests++;
   }
   for (n = quick ? maxn : 16384; n <= maxn; n *= 2)
      for (s = 0; s < 12; s++)
         for (p = 0; p <= (quick ? 2 : 4); p++) {
            static const float probs[5] = {0.0f, 0.5f, 0.9f, 0.99f, 0.995f};
            size_t r;
            gen_data(data, n, seed++, syms[s], probs[p]);
            r = zultra_memory_compress(data, n, comp, cap, ZULTRA_FLAG_ZLIB_FRAMING, 0);
            tests++;
            if (r == (size_t)-1 || !inflate_matches(comp, r, data, n, FMT_ZLIB, NULL, 0)) { fprintf(stderr, "self-test failed: size %lld symbols %d prob %g\n", (long long)n, syms[s], probs[p]); fails++; }
         }
   free(comp); free(data);
   fprintf(stdout, "%d tests, %d failed\n", tests, fails);
   return fails ? 100 : 0;
}

int main(int argc, char **argv) {
   const char *in = NULL, *out = NULL, *dict = NULL;
   int bad = 0, have_cmd = 0, verify = 0, i;
   char cmd = 'z';
   unsigned int opt = 0;
   g_t0 = now_us();
   /* the tool drives ZULTRA_CUDA_DEVICES GPUs (default one): unless the caller chose, expose only those to the CUDA runtime,
      whose start-up otherwise initialises every device of the box (seconds on an 8-GPU node, for a tool that may compress 48 KB) */
   {
      const char *e = getenv("ZULTRA_CUDA_DEVICES");
      int n = (e && atoi(e) > 1) ? atoi(e) : 1, k;
      char list[128]; size_t at = 0;
      if (n > 16) n = 16;
      for (k = 0; k < n && at + 4 < sizeof(list); k++) at += (size_t)snprintf(list + at, sizeof(list) - at, k ? ",%d" : "%d", k);
      setenv("CUDA_VISIBLE_DEVICES", list, 0);
   }
   for (i = 1; i < argc; i++) {
      const char *a = argv[i];
      if (!strcmp(a, "-d") || !strcmp(a, "-z") || !strcmp(a, "-cbench") || !strcmp(a, "-test") || !strcmp(a, "-quicktest")) {
         if (have_cmd) bad = 1;
         have_cmd = 1;
         cmd = !strcmp(a, "-d") ? 'd' : !strcmp(a, "-z") ? 'z' : !strcmp(a, "-cbench") ? 'B' : !strcmp(a, "-test") ? 't' : 'T';
      } else if (!strcmp(a, "-c")) { if (verify) bad = 1; verify = 1; }
      else if (!strcmp(a, "-D")) { if (!dict && i + 1 < argc) dict = argv[++i]; else bad = 1; }
      else if (!strncmp(a, "-D", 2)) { if (!dict) dict = a + 2; else bad = 1; }
      else if (!strcmp(a, "-v")) { if (opt & OPT_VERBOSE) bad = 1; opt |= OPT_VERBOSE; }
      else if (!strcmp(a, "-deflate")) { if (opt & FMT_MASK) bad = 1; opt |= FMT_DEFLATE; }
      else if (!strcmp(a, "-gzip")) { if (opt & FMT_MASK) bad = 1; opt |= FMT_GZIP; }
      else if (!strcmp(a, "-zlib")) { if (opt & FMT_MASK) bad = 1; opt |= FMT_ZLIB; }
      else if (!in) in = a;
      else if (!out) out = a;
      else bad = 1;
   }
   if (!bad && (cmd == 't' || cmd == 'T')) return do_self_test(cmd == 'T');
   if (bad || !in || !out) {
      fprintf(stderr, "zultra-b200 (GPU build of zultra; reference tool by Emmanuel Marty)\n");
      fprintf(stderr, "usage: %s [-gzip] [-zlib] [-deflate] [-v] {-c|-cbench|-test} <infile> <outfile>\n", argv[0]);
      fprintf(stderr, "           -gzip: use gzip framing (default)\n");
      fprintf(stderr, "           -zlib: use zlib framing\n");
      fprintf(stderr, "        -deflate: use deflate framing (no framing)\n");
      fprintf(stderr, "              -v: be verbose\n");
      fprintf(stderr, "              -c: check resulting stream after compressing\n");
      fprintf(stderr, "         -cbench: benchmark in-memory compression\n");
      fprintf(stderr, "           -test: run automated self-tests\n");
      return 100;
   }
   if (!(opt & FMT_MASK)) opt |= FMT_GZIP;
   if (cmd == 'z') {
      int r;
      if (dict && (opt & FMT_MASK) != FMT_ZLIB) { fprintf(stderr, "dictionaries are only supported for the zlib framing\n"); return 100; }
      r = do_compress(in, out, dict, opt);
      if (r == 0 && verify) r = do_compare(out, in, dict, opt);
      /* all files are closed: _exit without the CUDA runtime's exit handlers; with ZULTRA_CUDA_TRACE the milestone is printed
         so that the teardown can be timed */
      {
         const char *tr = getenv("ZULTRA_CUDA_TRACE");
         if (tr && atoi(tr)) fprintf(stderr, "[cli %9.2f ms] streams closed\n", (double)(now_us() - g_t0) / 1000.0);
         fflush(NULL);
         _exit(r);
      }
   }
   if (cmd == 'B') return do_cbench(in, out, opt);
   return 100;
}
