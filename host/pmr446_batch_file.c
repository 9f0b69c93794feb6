/*
 * host/pmr446_batch_file.c -- the recommended integration: the reference's loop bodies
 * (/root/reference/src/sdr_pmr446.c:795-823, :881-902, :910-913) replaced by ONE coarse call per
 * chunk, pmr446_batch_execute(), for any number of capture files processed side by side.
 *
 * usage: pmr446_batch_file [-r fs_in] [-8 | -16 | -s8] [-g gain] [-l] [-n chunk] [-d rate] -o out_prefix capture0 [capture1 ...]
 *   -8 / -16 / -s8  captures are cu8 / cs16 / cs8 (default cf32);  writes <out_prefix>.<stream>.<channel>.s16 for all 16 channels
 *   -d rate         also writes <out_prefix>_sNNN_chNN.dsd.s16: every channel's discriminator at `rate` Hz s16 (48000: what
 *                   `dsd -i` reads on stdin from src/dsd_in.c), i.e. one dsd_in per channel from one capture of the band
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../include/pmr446_b200.h"

int main(int argc, char **argv) {
  pmr446_config cfg;
  pmr446_default_config(&cfg);
  cfg.audio_gain = 1.0f;
  const char *prefix = NULL;
  const char *files[256];
  int nfiles = 0;
  for (int i = 1; i < argc; i++) {
    if (!strcmp(argv[i], "-r") && i + 1 < argc) cfg.fs_in = (unsigned)atol(argv[++i]);
    else if (!strcmp(argv[i], "-8")) cfg.in_fmt = PMR446_FMT_CU8;
    else if (!strcmp(argv[i], "-16")) cfg.in_fmt = PMR446_FMT_CS16;
    else if (!strcmp(argv[i], "-s8")) cfg.in_fmt = PMR446_FMT_CS8;
    else if (!strcmp(argv[i], "-g") && i + 1 < argc) cfg.audio_gain = (float)atof(argv[++i]);
    else if (!strcmp(argv[i], "-l")) cfg.lowpass = 1;
    else if (!strcmp(argv[i], "-n") && i + 1 < argc) cfg.max_chunk = (unsigned)atol(argv[++i]);
    else if (!strcmp(argv[i], "-d") && i + 1 < argc) cfg.dsd_rate = (unsigned)atol(argv[++i]);
    else if (!strcmp(argv[i], "-o") && i + 1 < argc) prefix = argv[++i];
    else if (nfiles < 256) files[nfiles++] = argv[i];
  }
  if (!prefix || nfiles == 0) { fprintf(stderr, "usage: %s [-r fs] [-8 | -16 | -s8] [-g gain] [-l] [-n chunk] [-d rate] -o prefix capture...\n", argv[0]); return 1; }
  cfg.n_streams = nfiles;
  pmr446_batch *b = NULL;
  if (pmr446_batch_create(&cfg, &b) != PMR446_OK) { fprintf(stderr, "pmr446_batch_create: %s\n", pmr446_last_error()); return 2; }
  const size_t bps = (size_t)pmr446_bytes_per_sample(cfg.in_fmt);
  const long long ld = pmr446_batch_max_ns(b);
  uint8_t *iq = (uint8_t *)calloc((size_t)nfiles * cfg.max_chunk, bps);
  int16_t *pcm = (int16_t *)calloc((size_t)nfiles * 16 * ld, 2);
  const long long dld = pmr446_batch_max_dsd(b);
  int16_t *dsd = cfg.dsd_rate ? (int16_t *)calloc((size_t)nfiles * 16 * dld, 2) : NULL;
  FILE *fi[256], *fo[256][16], *fd[256][16];
  char name[1024];
  for (int s = 0; s < nfiles; s++) {
    if (!(fi[s] = fopen(files[s], "rb"))) { perror(files[s]); return 2; }
    for (int c = 0; c < 16; c++) {
      snprintf(name, sizeof name, "%s.%d.%02d.s16", prefix, s, c + 1);
      if (!(fo[s][c] = fopen(name, "wb"))) { perror(name); return 2; }
      fd[s][c] = NULL;
      if (!dsd) continue;
      snprintf(name, sizeof name, "%s_s%03d_ch%02d.dsd.s16", prefix, s, c + 1);
      if (!(fd[s][c] = fopen(name, "wb"))) { perror(name); return 2; }
    }
  }
  unsigned long long total = 0;
  for (;;) {
    size_t n = cfg.max_chunk;
    for (int s = 0; s < nfiles; s++) {   /* all streams advance in lock-step: use the shortest read */
      size_t rd = fread(iq + (size_t)s * cfg.max_chunk * bps, bps, cfg.max_chunk, fi[s]);
      if (rd < n) n = rd;
    }
    if (n == 0) break;
    pmr446_outputs out;
    memset(&out, 0, sizeof out);
    out.pcm = pcm;
    out.ld = ld;
    out.dsd_pcm = dsd;
    out.dsd_ld = dld;
    unsigned ny = 0, ns = 0;
    if (pmr446_batch_execute(b, iq, (long long)cfg.max_chunk * bps, (unsigned)n, &out, &ny, &ns) != PMR446_OK) {
      fprintf(stderr, "pmr446_batch_execute: %s\n", pmr446_last_error());
      return 3;
    }
    for (int s = 0; s < nfiles; s++)
      for (int c = 0; c < 16; c++) {
        fwrite(pcm + ((size_t)s * 16 + c) * ld, 2, ns, fo[s][c]);
        if (dsd) fwrite(dsd + ((size_t)s * 16 + c) * dld, 2, (size_t)pmr446_batch_last_dsd(b), fd[s][c]);
      }
    total += n;
    if (n < cfg.max_chunk) break;
  }
  fprintf(stderr, "processed %llu samples per stream, %d stream(s)\n", total, nfiles);
  pmr446_batch_destroy(b);
  return 0;
}
