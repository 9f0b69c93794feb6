/*
 * host/dsd446_pipe.c -- dsd_in on a recorded (or piped) capture: cu8 / cs16 / cs8 / cf32 IQ in, 48 kHz s16 on stdout for
 * `dsd -i -`, exactly the pipe the reference feeds (/root/reference/src/dsd_in.c:159-180).  The loop body
 * :167-175 (DC block, msresamp down to 12.5 kHz, freqdem, msresamp_rrrf up to 48 kHz, s16 cast) is ONE call,
 * dsd446_batch_execute(); SoapySDR's readStream (:161) is an fread into pinned memory.
 *
 * usage: dsd446_pipe [-r fs_in] [-8 | -16 | -s8] [-n chunk] capture|-   > audio.s16
 *   -8 cu8, -16 cs16, -s8 cs8 capture (default cf32)
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../include/pmr446_b200.h"

int main(int argc, char **argv) {
  dsd446_config cfg;
  dsd446_default_config(&cfg);
  const char *in_path = NULL;
  for (int i = 1; i < argc; i++) {
    if (!strcmp(argv[i], "-r") && i + 1 < argc) cfg.fs_in = (unsigned)atol(argv[++i]);
    else if (!strcmp(argv[i], "-8")) cfg.in_fmt = PMR446_FMT_CU8;
    else if (!strcmp(argv[i], "-16")) cfg.in_fmt = PMR446_FMT_CS16;
    else if (!strcmp(argv[i], "-s8")) cfg.in_fmt = PMR446_FMT_CS8;
    else if (!strcmp(argv[i], "-n") && i + 1 < argc) cfg.max_chunk = (unsigned)atol(argv[++i]);
    else in_path = argv[i];
  }
  if (!in_path) { fprintf(stderr, "usage: %s [-r fs] [-8 | -16 | -s8] [-n chunk] capture|-  > audio.s16\n", argv[0]); return 1; }
  dsd446_batch *b = NULL;
  if (dsd446_batch_create(&cfg, &b) != PMR446_OK) { fprintf(stderr, "dsd446_batch_create: %s\n", pmr446_last_error()); return 2; }
  FILE *fi = strcmp(in_path, "-") ? fopen(in_path, "rb") : stdin;
  if (!fi) { perror(in_path); return 2; }
  const size_t bps = (size_t)pmr446_bytes_per_sample(cfg.in_fmt);
  const long long out_ld = dsd446_batch_max_out(b);
  void *iq = NULL;
  if (pmr446_host_alloc(&iq, (unsigned long long)cfg.max_chunk * bps) != PMR446_OK) { fprintf(stderr, "%s\n", pmr446_last_error()); return 2; }
  int16_t *pcm = (int16_t *)calloc((size_t)out_ld, sizeof(int16_t));
  setvbuf(stdout, NULL, _IONBF, 0);   /* :157 */
  unsigned long long total = 0;
  for (;;) {
    const size_t n = fread(iq, bps, cfg.max_chunk, fi);
    if (n == 0) break;
    dsd446_outputs out;
    memset(&out, 0, sizeof out);
    out.pcm = pcm;
    out.out_ld = out_ld;
    unsigned ny = 0, nz = 0;
    if (dsd446_batch_execute(b, iq, 0, (unsigned)n, &out, &ny, &nz) != PMR446_OK) { fprintf(stderr, "dsd446_batch_execute: %s\n", pmr446_last_error()); return 3; }
    if (fwrite(pcm, 2, nz, stdout) != nz) { perror("stdout"); return 3; }
    total += nz;
  }
  fprintf(stderr, "%llu s16 samples written\n", total);
  if (fi != stdin) fclose(fi);
  pmr446_host_free(iq);
  free(pcm);
  dsd446_batch_destroy(b);
  return 0;
}
