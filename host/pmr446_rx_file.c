/*
 * host/pmr446_rx_file.c -- the reference program's behaviour on a recorded capture: scan the 16 PMR446
 * channels, open the squelch on the strongest one, play (here: write a WAV of) its audio, report CTCSS codes,
 * optionally print the ASCII waterfall with the channel footer.  Everything between reading a chunk and
 * queueing audio (/root/reference/src/sdr_pmr446.c:795-913) is ONE call, pmr446_receiver_execute().
 *
 * Replaces around that call:
 *   SoapySDR readStream (src/shared.c, :788-793)      -> fread of a cu8 / cs16 / cs8 / cf32 capture (or stdin) into pinned memory
 *   RtAudio output callback (:520-593)                -> WAV writer (s16 or float32, 12.5 kHz mono)
 *   LOG lines (:613-626, :838, :852, :861)            -> the same messages from pmr446_rx_status.events
 *   waterfall row + footer (:630-666, :914-918)       -> printed from the ascii row and the status
 *
 * usage: pmr446_rx_file [-r fs_in] [-8 | -16 | -s8] [-g audio_gain] [-s squelch_dB] [-m excluded,channels] [-L] [-l]
 *                       [-w W] [-n chunk] [-f] -o out.wav capture|-
 *   -8 cu8, -16 cs16, -s8 cs8 capture (default cf32)
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../include/pmr446_b200.h"

#define FOOTER_TAIL 64

static void put_le(FILE *f, uint32_t v, int bytes) {
  for (int i = 0; i < bytes; i++) fputc((int)((v >> (8 * i)) & 0xff), f);
}

/* 44-byte canonical WAV header; sizes are patched by wav_finish() when the output is seekable */
static void wav_begin(FILE *f, unsigned rate, int is_float) {
  const unsigned bytes = is_float ? 4 : 2;
  fwrite("RIFF", 1, 4, f); put_le(f, 0xffffffffu, 4); fwrite("WAVE", 1, 4, f);
  fwrite("fmt ", 1, 4, f); put_le(f, 16, 4); put_le(f, is_float ? 3 : 1, 2); put_le(f, 1, 2);
  put_le(f, rate, 4); put_le(f, rate * bytes, 4); put_le(f, bytes, 2); put_le(f, 8 * bytes, 2);
  fwrite("data", 1, 4, f); put_le(f, 0xffffffffu, 4);
}

static void wav_finish(FILE *f, unsigned long long data_bytes) {
  if (fseek(f, 4, SEEK_SET) != 0) return;
  put_le(f, (uint32_t)(36 + data_bytes), 4);
  fseek(f, 40, SEEK_SET);
  put_le(f, (uint32_t)data_bytes, 4);
}

/* the footer line under the waterfall: channel numbers, "^^" under the active one, "--" for masked ones (:630-666) */
static void draw_footer(char *footer, size_t w_len, unsigned num_channels, unsigned long long mask, const pmr446_rx_status *st,
                        float centre_mhz) {
  const float ch_width = (float)w_len / (float)num_channels;
  for (unsigned i = 0; i < num_channels; i++) {
    const size_t at = (size_t)roundf(((float)i * ch_width) + (ch_width / 2) + 2);
    int len;
    if (st->active_chan == (int)i) len = snprintf(&footer[at], w_len, "%s", "^^");
    else if (mask & (1ull << i)) len = snprintf(&footer[at], w_len, "%02u", i + 1);
    else len = snprintf(&footer[at], w_len, "%s", "--");
    footer[at + (size_t)len] = ' ';
  }
  char *tail = &footer[w_len + 6];
  if (st->active_chan >= 0 && st->tone_detected)
    snprintf(tail, FOOTER_TAIL - 6, "%8.3f MHz [%d]  [CTCSS:  %02d (%3.2fHz)]", centre_mhz, st->active_chan + 1, st->ctcss_index + 1, st->ctcss_freq);
  else if (st->active_chan >= 0)
    snprintf(tail, FOOTER_TAIL - 6, "%8.3f MHz [%d]", centre_mhz, st->active_chan + 1);
  else
    snprintf(tail, FOOTER_TAIL - 6, "%8.3f MHz", centre_mhz);
}

int main(int argc, char **argv) {
  pmr446_rx_config cfg;
  pmr446_rx_default_config(&cfg);
  const char *out_path = NULL, *in_path = NULL;
  int want_float = 0;
  for (int i = 1; i < argc; i++) {
    if (!strcmp(argv[i], "-r") && i + 1 < argc) cfg.chain.fs_in = (unsigned)atol(argv[++i]);
    else if (!strcmp(argv[i], "-8")) cfg.chain.in_fmt = PMR446_FMT_CU8;
    else if (!strcmp(argv[i], "-16")) cfg.chain.in_fmt = PMR446_FMT_CS16;
    else if (!strcmp(argv[i], "-s8")) cfg.chain.in_fmt = PMR446_FMT_CS8;
    else if (!strcmp(argv[i], "-g") && i + 1 < argc) cfg.chain.audio_gain = (float)atof(argv[++i]);
    else if (!strcmp(argv[i], "-s") && i + 1 < argc) cfg.squelch_level = (float)atof(argv[++i]);
    else if (!strcmp(argv[i], "-m") && i + 1 < argc) {   /* comma-separated 1-based channels to exclude (:283-297) */
      for (char *tok = strtok(argv[++i], ","); tok; tok = strtok(NULL, ",")) {
        long ch = atol(tok);
        if (ch >= 1 && ch <= 64) cfg.channel_mask &= ~(1ull << (ch - 1));
      }
    } else if (!strcmp(argv[i], "-L")) cfg.lock_mode = PMR446_LOCK_MAX;
    else if (!strcmp(argv[i], "-l")) cfg.chain.lowpass = 1;
    else if (!strcmp(argv[i], "-w") && i + 1 < argc) cfg.chain.waterfall = (unsigned)atol(argv[++i]);
    else if (!strcmp(argv[i], "-n") && i + 1 < argc) cfg.chain.max_chunk = (unsigned)atol(argv[++i]);
    else if (!strcmp(argv[i], "-f")) want_float = 1;
    else if (!strcmp(argv[i], "-o") && i + 1 < argc) out_path = argv[++i];
    else in_path = argv[i];
  }
  if (!out_path || !in_path) {
    fprintf(stderr, "usage: %s [-r fs] [-8 | -16 | -s8] [-g gain] [-s squelch] [-m ch,ch] [-L] [-l] [-w W] [-n chunk] [-f] -o out.wav capture|-\n", argv[0]);
    return 1;
  }
  pmr446_receiver *rx = NULL;
  if (pmr446_receiver_create(&cfg, &rx) != PMR446_OK) { fprintf(stderr, "pmr446_receiver_create: %s\n", pmr446_last_error()); return 2; }
  FILE *fi = strcmp(in_path, "-") ? fopen(in_path, "rb") : stdin;
  FILE *fo = fopen(out_path, "wb");
  if (!fi || !fo) { perror(fi ? out_path : in_path); return 2; }
  const size_t bps = (size_t)pmr446_bytes_per_sample(cfg.chain.in_fmt);
  const unsigned W = cfg.chain.waterfall, M = cfg.chain.num_channels;
  const long long ld = pmr446_receiver_max_ns(rx);
  void *iq = NULL;
  if (pmr446_host_alloc(&iq, (unsigned long long)cfg.chain.max_chunk * bps) != PMR446_OK) { fprintf(stderr, "%s\n", pmr446_last_error()); return 2; }
  float *audio = (float *)calloc((size_t)ld, sizeof(float));
  int16_t *pcm = (int16_t *)calloc((size_t)ld, sizeof(int16_t));
  char *ascii = (char *)calloc((size_t)W + 1, 1), *footer = (char *)malloc((size_t)W + FOOTER_TAIL + 1);
  float peak[2] = {0, 0};
  const float centre_mhz = (446.0e6f + (float)(M / 2) * (float)cfg.chain.channel_width) * 1e-6f;   /* SDR_FREQUENCY, :28 */
  if (W) {
    memset(footer, ' ', (size_t)W + FOOTER_TAIL);
    footer[(size_t)W + FOOTER_TAIL] = '\0';
    footer[1] = '[';
    footer[W + 4] = ']';
  }
  wav_begin(fo, cfg.chain.channel_width, want_float);
  unsigned long long data_bytes = 0, samples_in = 0;
  int prev_active = -1;
  for (;;) {
    const size_t n = fread(iq, bps, cfg.chain.max_chunk, fi);
    if (n == 0) break;
    pmr446_rx_status st;
    pmr446_rx_outputs out;
    memset(&out, 0, sizeof out);
    out.status = &st;
    out.audio = want_float ? audio : NULL;
    out.pcm = want_float ? NULL : pcm;
    out.ld = ld;
    out.ascii = W ? ascii : NULL;
    out.peak = W ? peak : NULL;
    unsigned ns = 0;
    if (pmr446_receiver_execute(rx, iq, 0, (unsigned)n, &out, &ns) != PMR446_OK) { fprintf(stderr, "pmr446_receiver_execute: %s\n", pmr446_last_error()); return 3; }
    samples_in += n;
    if (W == 0) {   /* the reference logs only when the waterfall is off */
      if (st.events & PMR446_EV_TUNED) fprintf(stderr, "Tuned to channel %d (RSSI: %4.2fdB)\n", st.active_chan + 1, st.rssi);
      if (st.events & PMR446_EV_CHANGED) fprintf(stderr, "Changed active channel from %d to %d\n", prev_active + 1, st.active_chan + 1);
      if (st.events & PMR446_EV_DETUNED) fprintf(stderr, "Detuned from channel %d\n", prev_active + 1);
      if (st.events & PMR446_EV_CTCSS_ACQUIRED) fprintf(stderr, "Acquired CTCSS code: %d (frequency: %3.2fHz)\n", st.ctcss_index + 1, st.ctcss_freq);
      if (st.events & PMR446_EV_CTCSS_CHANGED) fprintf(stderr, "CTCSS code change: %d (frequency: %3.2fHz)\n", st.ctcss_index + 1, st.ctcss_freq);
      if (st.events & PMR446_EV_CTCSS_LOST) fprintf(stderr, "Lost CTCSS code\n");
    } else {
      draw_footer(footer, W, M, cfg.channel_mask, &st, centre_mhz);
      printf(" > %s < pk%5.1fdB [%5.2f] [max SNR: %5.1fdB]        \n%s\r", ascii, peak[0], peak[1], st.rssi, footer);
      fflush(stdout);
    }
    prev_active = st.active_chan;
    if (st.n_audio) {
      if (want_float) fwrite(audio, sizeof(float), st.n_audio, fo);
      else fwrite(pcm, sizeof(int16_t), st.n_audio, fo);
      data_bytes += (unsigned long long)st.n_audio * (want_float ? 4 : 2);
    }
  }
  wav_finish(fo, data_bytes);
  if (W) printf("\n");
  fprintf(stderr, "%llu samples in, %llu audio bytes out\n", samples_in, data_bytes);
  fclose(fo);
  if (fi != stdin) fclose(fi);
  pmr446_host_free(iq);
  free(audio); free(pcm); free(ascii); free(footer);
  pmr446_receiver_destroy(rx);
  return 0;
}
