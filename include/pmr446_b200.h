/*
 * pmr446_b200.h -- C ABI of the B200-native PMR446 receive DSP library (libpmr446_b200.so).
 *
 * This is the coarse, batched tier of the drop-in boundary (SURVEY.md 8b): each call replaces
 * one loop body of the reference's main() for n_streams independent IQ streams at once.
 * Buffer conventions are the reference's: interleaved I/Q input, channel-major
 * [num_channels][ld] outputs (ch_buff_mat_t, /root/reference/src/sdr_pmr446.c:51), counts
 * returned through pointers, all state carried inside the handle between calls, every
 * function returns 0 (== LIQUID_OK) on success.
 *
 *   pmr446_batch_execute*()  replaces  src/sdr_pmr446.c:795-823  (DC block, msresamp, ring
 *                                      buffer carry, NCO mix, firpfbch analyzer, transpose),
 *                                      :881-902 for every channel (freqdem, 377-tap HP FIR,
 *                                      wdelay complement, gain, de-emphasis, optional LP FIR),
 *                                      :910-913 (asgram waterfall row).
 *   dsd446_batch_execute*()  replaces  src/dsd_in.c:167-175 (DC block, msresamp down, freqdem,
 *                                      msresamp_rrrf up, s16 conversion).
 *   pmr446_receiver_execute*() replaces src/sdr_pmr446.c:795-913 as the reference runs it: the same
 *                                      front half, then RSSI (:330-336, :668-700), the squelch /
 *                                      selector state machine (:828-874), the selected channel's
 *                                      audio chain (:876-908) and the CTCSS detector (:338-418, :605-628).
 *
 * The liquid-dsp-signature shim (second tier) is declared in pmr446_liquid_shim.h.
 * All arithmetic runs on the GPU; there is no CPU fallback: without a CUDA device every
 * create() fails with PMR446_ENODEV.
 */
#ifndef PMR446_B200_H
#define PMR446_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMR446_OK 0
#define PMR446_EINVAL (-1)     /* bad argument / unsupported configuration */
#define PMR446_ENODEV (-2)     /* no usable CUDA device */
#define PMR446_ECUDA (-3)      /* CUDA runtime error, see pmr446_last_error() */
#define PMR446_ERANGE (-4)     /* chunk larger than max_chunk / output ld too small */
#define PMR446_ENOMEM (-5)

#define PMR446_FMT_CF32 0      /* interleaved float32 I,Q  (SOAPY_SDR_CF32, src/shared.c:62) */
#define PMR446_FMT_CU8 1       /* interleaved uint8 I,Q, converted as (u8 - 127.4)/128 */

typedef struct {
  int n_streams;           /* independent IQ streams processed per call */
  int device;              /* CUDA device ordinal; -1 = current device */
  unsigned fs_in;          /* input sample rate, Hz (SDR_SAMPLERATE, include/sdr_pmr446.h:13) */
  int in_fmt;              /* PMR446_FMT_* */
  unsigned num_channels;   /* NUM_CHANNELS, src/sdr_pmr446.c:23 (16); any M in [2, 4096] whose generic channelizer
                              (56 M bytes of shared memory) fits the device's opt-in per-block limit (all of them on a B200) */
  unsigned channel_width;  /* CHANNEL_WIDTH_HZ, :22 (12500) */
  unsigned pfb_m;          /* firpfbch_crcf_create_kaiser semi-length, :437 (13) */
  float pfb_as;            /* ... stop-band attenuation, :437 (80 dB) */
  float resamp_as;         /* msresamp_crcf_create attenuation, :426 (60 dB) */
  float dc_alpha;          /* iirfilt_crcf_create_dc_blocker, :422 (0.0005) */
  float kf;                /* freqdem_create, :440 (0.5) */
  float audio_gain;        /* SDR_DEFAULT_AUDIO_GAIN, :33 (4.0) */
  int lowpass;             /* -l: apply the 103-tap audio low-pass, :900-902 */
  unsigned waterfall;      /* -w W: asgram width, 0 = off, :473-477; any W in [2, 2048] (nfft = 4 W, any factorisation) */
  unsigned max_chunk;      /* largest n per execute call (SDR_INPUT_CHUNK, :30) */
  const float *hp_taps;    /* CTCSS-removal FIR, NULL = the reference's 377 taps (:56-104) */
  unsigned hp_len;
  const float *lp_taps;    /* audio low-pass FIR, NULL = the reference's 103 taps (:106-119) */
  unsigned lp_len;
  float deemph_b0, deemph_b1, deemph_a1; /* :461-463; y = b0 x + b1 x[-1] - a1 y[-1].  Any |a1| < 1 whose warm-up
                              k = ceil(log(2^-30) / log|a1|) fits an audio tile: |a1| <= 0.977 with the low-pass, 0.979
                              without; create() refuses other poles with PMR446_EINVAL */
  int deemph_fir;          /* APP_FIR_DEEMPH build of the reference: the 101-tap FIR de-emphasis (:122-135, :458, :896)
                              instead of the one-pole filter; served by the fast-convolution audio kernel only
                              (batch API; composite responses up to 1000 taps) */
} pmr446_config;

/* Per-call outputs.  Any pointer may be NULL.  For *_execute() these are HOST pointers, for
 * *_execute_device() DEVICE pointers.  Stream s, channel c, sample k of a channel-major array
 * lives at base[(s * num_channels + c) * ld + k]. */
typedef struct {
  float *res;              /* [n_streams][res_ld] complex (re,im) un-mixed resampler output, ny valid */
  long long res_ld;        /* complex samples per stream row */
  float *chan;             /* [n_streams][M][ld] complex channelizer output (chan_bufs, :743) */
  float *demod;            /* [n_streams][M][ld] discriminator output (tmp_buf1 after :881) */
  float *lpcomp;           /* [n_streams][M][ld] delayed - high-passed (tmp_buf1 after :889) */
  float *audio;            /* [n_streams][M][ld] float audio (tmp_buf2 after :898/:901) */
  int16_t *pcm;            /* [n_streams][M][ld] (int16_t)(audio * 32767), saturated at full scale */
  long long ld;            /* samples per channel row (SDR_CHANNEL_BUF_SIZE, :37) */
  char *ascii;             /* [n_streams][W] waterfall row (asgramcf_execute, :912) */
  float *peak;             /* [n_streams][2] peak value (dB) and frequency */
  float *psd;              /* [n_streams][4W] dB values behind the row */
  /* Selector taps, 16-channel kernel only, one call = one RSSI window (average_power, :330-336; find_max_rssi_channel
   * reads them, :668-700).  With the host-buffer call they switch the time slicing off. */
  float *rssi;             /* [n_streams][M] 20 log10(mean |chan|) over this call's ns frames, dB */
  float *chan_edge;        /* [n_streams][M][2] complex: channel sample of this call's first and last frame
                              (what freqdem's r_prime needs when the active channel changes, :866, :881) */
} pmr446_outputs;

typedef struct pmr446_batch pmr446_batch;

/* Fills cfg with the reference's parameters (src/sdr_pmr446.c:18-46, :420-480), n_streams = 1. */
void pmr446_default_config(pmr446_config *cfg);
int pmr446_batch_create(const pmr446_config *cfg, pmr446_batch **out);
int pmr446_batch_destroy(pmr446_batch *b);
/* Largest ny / ns one call can return (SDR_RESAMP_BUF_SIZE / SDR_CHANNEL_BUF_SIZE, :36-37, :730-732). */
long long pmr446_batch_max_res(const pmr446_batch *b);
long long pmr446_batch_max_ns(const pmr446_batch *b);
/* Host-buffer call: copies n samples per stream to the GPU, runs the chain, copies the
 * requested outputs back, and returns when they are in place.  iq_stride = bytes between
 * streams in `iq`.  *ny = resampler outputs, *ns = channel samples produced by this call. */
int pmr446_batch_execute(pmr446_batch *b, const void *iq, long long iq_stride, unsigned n, const pmr446_outputs *out,
                         unsigned *ny, unsigned *ns);
/* Device-buffer call: `iq` and the outputs are device pointers; work is enqueued on
 * `cuda_stream` (a cudaStream_t, NULL = default stream) and the call returns without waiting. */
int pmr446_batch_execute_device(pmr446_batch *b, const void *iq, long long iq_stride, unsigned n, const pmr446_outputs *out,
                                unsigned *ny, unsigned *ns, void *cuda_stream);
/* Device call: demod_out[s][k] = discriminator output of channel `channel[s]` (device array, -1 = skip the stream) for the
 * ns frames of the LAST execute call, read from the library's discriminator ring -- the squelch selector's tap
 * (src/sdr_pmr446.c:876-881) without materialising all M rows. */
int pmr446_batch_gather_channel(pmr446_batch *b, const int *channel, float *demod_out, long long ld, void *cuda_stream);
/* Kernels launched by the last execute call (for the benchmark's gpu_launches field). */
int pmr446_batch_last_launches(const pmr446_batch *b);
/* Resets all filter state to stream start (t = 0). */
int pmr446_batch_reset(pmr446_batch *b);
/* Per-kernel device timing (CUDA events on the launch stream).  After pmr446_batch_timing(b, 1)
 * every execute call records events around its kernels; pmr446_batch_get_timings() waits for the
 * device and returns, per tag, the accumulated milliseconds and the number of intervals since
 * timing was enabled.  Tags: 1 DC-blocker carry, 2-4 half-band/resampler cascade launches,
 * 5 history save, 6 channelizer+discriminator, 7 audio FIR chain, 8 waterfall, 9 output gathers. */
#define PMR446_TIMING_TAGS 10
int pmr446_batch_timing(pmr446_batch *b, int enable);
int pmr446_batch_get_timings(pmr446_batch *b, double *total_ms, long long *count, int n);

/* ---- receiver: RSSI, squelch / channel selector, selected-channel audio, CTCSS detector ---------
 * What the reference actually plays: per chunk it measures every enabled channel
 * (average_power, src/sdr_pmr446.c:330-336; find_max_rssi_channel, :668-700), runs the
 * scanning/tuned state machine (:828-874) and demodulates ONLY the active channel through one
 * freqdem / FIR / delay / de-emphasis chain whose state carries over channel changes (:876-908);
 * the complementary low-pass branch feeds a DC blocker and a 38-tone Goertzel bank over blocks of
 * 2441 samples (ctcss_execute :605-628, ctcss_detector_analyze :365-407).  One call = one chunk
 * of every stream; the state machine runs on the GPU, one thread per stream, no host round trip. */
#define PMR446_LOCK_START 0    /* lock_mode_start: stay on the first channel that opened the squelch */
#define PMR446_LOCK_MAX 1      /* lock_mode_max: follow the strongest channel (:848-857) */
#define PMR446_CTCSS_TONES 38  /* CTCSS_NUM_FREQS, include/sdr_pmr446.h:14 */
#define PMR446_EV_TUNED 1      /* "Tuned to channel" :838 */
#define PMR446_EV_CHANGED 2    /* "Changed active channel" :852 */
#define PMR446_EV_DETUNED 4    /* "Detuned from channel" :861 */
#define PMR446_EV_CTCSS_ACQUIRED 8   /* :616 */
#define PMR446_EV_CTCSS_CHANGED 16   /* :619 */
#define PMR446_EV_CTCSS_LOST 32      /* :624 */

typedef struct {
  pmr446_config chain;             /* DSP parameters; num_channels <= 64 (MAX_CHANNELS, :18) */
  float squelch_level;             /* -s, SDR_DEFAULT_SQUELCH_LEVEL :34 (18 dB); closes 5 dB lower (:859) */
  unsigned long long channel_mask; /* -m, bit i enables channel i (:155, :678) */
  int lock_mode;                   /* PMR446_LOCK_* (:156) */
  unsigned ctcss_block;            /* CTCSS_BLOCK_SIZE :46 (2441) */
  float ctcss_dc_alpha;            /* :450 (0.0005) */
} pmr446_rx_config;

typedef struct {
  int state;            /* proc_scanning 0 / proc_tuned 1 after this chunk (include/sdr_pmr446.h:17-21) */
  int active_chan;      /* chain->active_chan: -1 or 0-based channel */
  float rssi;           /* chain->rssi: strongest - mean of the enabled channels, dB */
  unsigned n_audio;     /* audio samples this call appended for the stream (0 or ns) */
  int tone_detected;    /* ctcss_detector->tone_detected */
  int ctcss_index;      /* ctcss_detector->max_power_index (code - 1) */
  float ctcss_freq;     /* chain->ctcss_freq: -1 at start, tone table entry, 0 after a detune */
  float max_power;      /* ctcss_detector->max_power */
  int events;           /* PMR446_EV_* raised by this chunk (the reference's LOG lines) */
} pmr446_rx_status;

/* Host pointers for pmr446_receiver_execute(), device pointers for _execute_device(); any may be NULL. */
typedef struct {
  float *rssi;               /* [n_streams][M] average_power per channel, dB */
  pmr446_rx_status *status;  /* [n_streams] */
  float *audio;              /* [n_streams][ld] selected-channel audio (what :903-905 queues for the DAC) */
  int16_t *pcm;              /* [n_streams][ld] */
  float *ctcss_in;           /* [n_streams][ld] CTCSS branch after its DC blocker (:606) */
  float *ctcss_power;        /* [n_streams][38] Goertzel powers of the last finished block */
  long long ld;
  char *ascii;               /* [n_streams][W] waterfall row, as pmr446_outputs */
  float *peak;               /* [n_streams][2] */
} pmr446_rx_outputs;

typedef struct pmr446_receiver pmr446_receiver;
void pmr446_rx_default_config(pmr446_rx_config *cfg);
int pmr446_receiver_create(const pmr446_rx_config *cfg, pmr446_receiver **out);
int pmr446_receiver_destroy(pmr446_receiver *r);
long long pmr446_receiver_max_ns(const pmr446_receiver *r);
int pmr446_receiver_execute(pmr446_receiver *r, const void *iq, long long iq_stride, unsigned n, const pmr446_rx_outputs *out,
                            unsigned *ns);
int pmr446_receiver_execute_device(pmr446_receiver *r, const void *iq, long long iq_stride, unsigned n, const pmr446_rx_outputs *out,
                                   unsigned *ns, void *cuda_stream);
int pmr446_receiver_last_launches(const pmr446_receiver *r);
/* Back to stream start: scanning, no active channel, all filter state zero. */
int pmr446_receiver_reset(pmr446_receiver *r);

/* ---- dsd_in chain: single-channel FM demodulator feeding DSD (src/dsd_in.c) ------------------- */
typedef struct {
  int n_streams;
  int device;
  unsigned fs_in;          /* SDR_SAMPLERATE, include/dsd_in.h:11 */
  int in_fmt;
  unsigned fs_sig;         /* SIG_SAMPLERATE, src/dsd_in.c:23 (12500) */
  unsigned fs_audio;       /* AUDIO_SAMPLERATE, :22 (48000) */
  unsigned max_chunk;      /* SDR_INPUT_CHUNK, :25 (200000) */
  float dc_alpha;          /* :97 */
  float resamp_as;         /* :100, :104 */
  float kf;                /* :108 */
} dsd446_config;

typedef struct {
  float *res;              /* [n_streams][res_ld] complex 12.5 kHz stream (resamp_buf, :168), ny valid */
  float *fm;               /* [n_streams][res_ld] discriminator output (fm_out_buf, :169) */
  long long res_ld;
  float *audio;            /* [n_streams][out_ld] 48 kHz float (out_buf, :170), nz valid */
  int16_t *pcm;            /* [n_streams][out_ld] s16 (buf_out_s, :172-175; sized out_size, not the
                              reference's overflowing res_size, SURVEY.md 3.2) */
  long long out_ld;
} dsd446_outputs;

typedef struct dsd446_batch dsd446_batch;
void dsd446_default_config(dsd446_config *cfg);
int dsd446_batch_create(const dsd446_config *cfg, dsd446_batch **out);
int dsd446_batch_destroy(dsd446_batch *b);
long long dsd446_batch_max_res(const dsd446_batch *b);   /* res_size, src/dsd_in.c:137 */
long long dsd446_batch_max_out(const dsd446_batch *b);   /* out_size, :138 */
int dsd446_batch_last_launches(const dsd446_batch *b);  /* kernels launched by the last execute call (like pmr446_batch_last_launches) */
int dsd446_batch_execute(dsd446_batch *b, const void *iq, long long iq_stride, unsigned n, const dsd446_outputs *out, unsigned *ny,
                         unsigned *nz);
int dsd446_batch_execute_device(dsd446_batch *b, const void *iq, long long iq_stride, unsigned n, const dsd446_outputs *out,
                                unsigned *ny, unsigned *nz, void *cuda_stream);
int dsd446_batch_reset(dsd446_batch *b);

/* ---- host-only introspection (no GPU needed): the filter design the kernels run with --------- */
/* msresamp_crcf_create(rate, as) plan: stage count, semi-lengths m[g] (g = 0 lowest rate), 24-bit
 * phase step, filter-bank size; optionally the half-band taps [16][20] and the bank [npfb][14]. */
int pmr446_design_msresamp(float rate, float as, unsigned *stages, unsigned *m, unsigned *step, unsigned *npfb, float *hb_taps,
                           float *pfb);
/* firpfbch_crcf_create_kaiser(ANALYZER, M, m, as) branch taps, taps[i*2m + n] = h[i + n*M]. */
int pmr446_design_pfbch(unsigned M, unsigned m, float as, float *taps);
/* spgram window of asgramcf_create(W). */
int pmr446_design_asgram_window(unsigned W, float *w);
/* nco_crcf_set_frequency(dtheta) as a 32-bit phase increment. */
unsigned pmr446_design_nco_dtheta(float dtheta);
/* How msresamp_crcf_create(rate, as) (src/sdr_pmr446.c:425-426, src/dsd_in.c:100) is cut into kernel launches for the
 * given input format, e.g. "fused[3,5,10]+arb" or "cascade[3,3,3,3] | cascade[3,5] | tile[10]+arb"; every decimating
 * rate liquid accepts (0 < rate <= 1) has a plan.  buf receives the NUL-terminated description. */
int pmr446_describe_frontend(float rate, float as, int in_fmt, int with_dc, char *buf, int len);
/* Total msresamp outputs after n_in inputs since stream start (decimating rates). */
long long pmr446_count_resampled(float rate, float as, long long n_in);

const char *pmr446_last_error(void);
/* Page-locked host buffers for the host-buffer calls: captures read into them (file, SDR driver, socket) reach the
 * GPU at full PCIe rate and let the time-sliced copy in pmr446_batch_execute() overlap the kernels.  Replaces the
 * reference's stack arrays (src/sdr_pmr446.c:738-745). */
int pmr446_host_alloc(void **ptr, unsigned long long bytes);
int pmr446_host_free(void *ptr);
/* Measures the FP32 FFMA issue peak of the current device (TFLOP/s) with a register-only
 * kernel; used as the roofline denominator by bench.py. */
int pmr446_measure_fp32_peak(double *tflops, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif
