// C-ABI implementation of the batched PMR446 chain (include/pmr446_b200.h).
//
// Host logic only: per-chunk bookkeeping in absolute sample indices (how many half-band,
// resampler, frame and audio samples exist after N input samples is closed-form, SURVEY.md
// Appendix A.5 / B), ring-buffer management and kernel launches.  All DSP arithmetic is in
// frontend.cuh / backend.cuh / spectrum.cuh.  Mirrors the reference's init_liquid()
// (/root/reference/src/sdr_pmr446.c:420-480) and main-loop body (:795-913).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/pmr446_b200.h"
#include "../../include/pmr446_taps.h"
#include "audio_fft.cuh"
#include "audio_fft4.cuh"
#include "backend.cuh"
#include "channelizer.cuh"
#include "channelizer_generic.cuh"
#include "common_host.hpp"
#include "frontend_host.hpp"
#include "design.hpp"
#include "dsd.cuh"
#include "frontend.cuh"
#include "spectrum.cuh"

using namespace pmr;

// ================================================================================================
// PMR446 batch
// ================================================================================================
struct pmr446_batch {
  pmr446_config cfg;
  int S = 0;                 // streams
  int device = 0;
  Frontend fe;               // DC + msresamp -> resampled ring
  // channelizer
  int M = 16;                // channels
  bool generic = false;      // generic-M kernel instead of the 16-channel register kernel
  bool generic_tile = false; // ... its register-tiled variant (26 taps per branch, 10 frames of M samples in shared memory)
  DevBuf d_pfb_taps, d_mixed, d_tw;
  std::vector<int> radix;
  unsigned dtheta = 0;
  bool nco_lut = false;
  // demod ring [S*16][cap]
  DevBuf d_demod;
  long long demod_cap = 0;
  // audio
  DirectAudio au;            // direct-form chain: lpcomp, and audio / pcm when the response does not fit the FFT tile
  DevBuf d_mag;              // [S][max_tiles][16] per-tile sums of |chan| (RSSI)
  int max_tiles = 0;
  long long last_f0 = 0, last_ns = 0;   // frame range of the last execute call (pmr446_batch_gather_channel)
  DevBuf d_out_rssi, d_out_edge;
  int fft_halo = AF_HALO;    // overlap of the FFT audio tile (AF_HALO or AF_HALO_LONG)
  bool fft_audio = false;    // audio / pcm by fast convolution (audio_fft4_kernel); the direct-form kernel serves lpcomp
  DevBuf d_resp, d_aftw;
  // waterfall
  Waterfall wf;
  // per-channel DSD feed (cfg.dsd_rate != 0): msresamp_rrrf over every discriminator row, no state of its own
  design::MsresampPlan dsd;
  DevBuf d_dsd_pfb;          // [npfb][16] bank rows of the arbitrary stage
  int dsd_period = 32;       // (near-)period of its phase sequence (dsd_backend_kernel)
  long long max_dsd = 0, last_dsd = 0;
  // staging for the host-buffer call
  DevBuf d_in2[2], d_out_res, d_out_chan, d_out_demod, d_out_lpcomp, d_out_audio, d_out_pcm, d_out_ascii, d_out_peak, d_out_psd, d_out_dsd_audio,
      d_out_dsd_pcm;
  long long max_res = 0, max_ns = 0;
  cudaStream_t own_stream = nullptr, copy_stream = nullptr, out_stream = nullptr;
  cudaEvent_t ev_out = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
  int launches = 0;
  Timer timer;
};

extern "C" void pmr446_default_config(pmr446_config* c) {
  memset(c, 0, sizeof(*c));
  c->n_streams = 1;
  c->device = -1;
  c->fs_in = 1024000;
  c->in_fmt = PMR446_FMT_CF32;
  c->num_channels = 16;
  c->channel_width = 12500;
  c->pfb_m = 13;
  c->pfb_as = 80.0f;
  c->resamp_as = 60.0f;
  c->dc_alpha = 0.0005f;
  c->kf = 0.5f;
  c->audio_gain = 4.0f;
  c->lowpass = 0;
  c->waterfall = 0;
  c->max_chunk = 100000;
  c->hp_taps = nullptr;
  c->hp_len = 0;
  c->lp_taps = nullptr;
  c->lp_len = 0;
  c->deemph_b0 = (float)(PMR446_DEEMPH_B0 / PMR446_DEEMPH_A0);
  c->deemph_b1 = (float)(PMR446_DEEMPH_B1 / PMR446_DEEMPH_A0);
  c->deemph_a1 = (float)(PMR446_DEEMPH_A1 / PMR446_DEEMPH_A0);
}

extern "C" int pmr446_batch_create(const pmr446_config* cfg, pmr446_batch** out) {
  if (!cfg || !out) return fail(PMR446_EINVAL, "null argument");
  *out = nullptr;
  if (cfg->n_streams < 1 || cfg->max_chunk < 1 || cfg->fs_in == 0) return fail(PMR446_EINVAL, "bad n_streams/max_chunk/fs_in");
  if (cfg->num_channels < 2 || cfg->num_channels > 4096 || cfg->pfb_m < 1 || cfg->pfb_m > 32)
    return fail(PMR446_EINVAL, "num_channels must be in [2, 4096] and pfb_m in [1, 32]");
  if (int rc = select_device(cfg->device)) return rc;
  cudaGetLastError();   // start from a clean slate: the check at the end only sees errors raised in here
  std::unique_ptr<pmr446_batch, int (*)(pmr446_batch*)> b(new pmr446_batch(), pmr446_batch_destroy);   // freed on every early return
  b->cfg = *cfg;
  b->S = cfg->n_streams;
  cudaGetDevice(&b->device);
  const int S = b->S;
  const int M = b->M = (int)cfg->num_channels;
  b->generic = !(M == 16 && cfg->pfb_m == 13);   // the register-window kernel is specialised for 16 x 26 taps
  int smem_cap = 0;                               // per-block shared memory with opt-in (232 448 B on a B200)
  cudaDeviceGetAttribute(&smem_cap, cudaDevAttrMaxSharedMemoryPerBlockOptin, b->device);

  float fs_res = (float)(cfg->num_channels * cfg->channel_width);
  int rc = b->fe.init(S, cfg->in_fmt, fs_res / (float)cfg->fs_in, cfg->resamp_as, true, cfg->dc_alpha, cfg->max_chunk,
                      /*extra_hist=*/std::max<long long>(std::max<long long>((long long)M * (2 * cfg->pfb_m + CG_FT + 4), (long long)cfg->waterfall),
                                                         16LL * (CH_FR + CH_HIST + 2)) + 64);   // a call recomputes at most one channelizer tile
  if (rc) return rc;
  b->max_res = b->fe.max_out_per_chunk();
  b->max_ns = b->max_res / M + 1;

  // channelizer (A.7, A.8)
  std::vector<float> taps = design::pfbch_taps((unsigned)M, cfg->pfb_m, cfg->pfb_as);
  if ((rc = b->d_pfb_taps.alloc(taps.size() * sizeof(float)))) return rc;
  if (b->generic) {
    // the generic kernel walks the branches across lanes: store tap n of all branches contiguously ([n][M])
    const unsigned pp = 2 * cfg->pfb_m;
    std::vector<float> tt(taps.size());
    for (unsigned i = 0; i < (unsigned)M; i++)
      for (unsigned n = 0; n < pp; n++) tt[(size_t)n * M + i] = taps[(size_t)i * pp + n];
    taps.swap(tt);
  }
  cudaMemcpy(b->d_pfb_taps.p, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice);
  float offset = -0.5f * (float)(cfg->num_channels - 1) / (float)cfg->num_channels * 2 * M_PI;  // :432-433
  b->dtheta = design::nco_dtheta(offset);
  b->nco_lut = (b->dtheta & ((1u << 27) - 1)) == 0;
  if (b->generic) {
    unsigned nn = (unsigned)M;
    while (nn % 4 == 0) { b->radix.push_back(4); nn /= 4; }
    for (unsigned pr = 2; nn > 1;) {
      if (nn % pr == 0) { b->radix.push_back((int)pr); nn /= pr; }
      else pr++;
    }
    if (b->radix.size() > 16) return fail(PMR446_EINVAL, "num_channels has more than 16 prime factors");
    std::vector<float2> tw(M);
    for (int k = 0; k < M; k++) {
      double a = -2.0 * M_PI * (double)k / (double)M;
      tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    if ((rc = b->d_tw.alloc((size_t)M * sizeof(float2))) || (rc = b->d_mixed.alloc_zero((size_t)S * b->fe.out_cap * sizeof(float2)))) return rc;
    cudaMemcpy(b->d_tw.p, tw.data(), (size_t)M * sizeof(float2), cudaMemcpyHostToDevice);
    const size_t smem = (size_t)M * (3 * sizeof(float2) + CG_FT * sizeof(float));
    if (smem > (size_t)smem_cap) return fail(PMR446_EINVAL, "num_channels too large for the shared-memory FFT");
    cudaFuncSetAttribute(channelize_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    b->generic_tile = cfg->pfb_m == 13 && channelize_generic_tile_smem(M) <= (size_t)smem_cap;
    if (b->generic_tile)
      cudaFuncSetAttribute(channelize_generic_tile_kernel<26>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)channelize_generic_tile_smem(M));
  }

  b->max_tiles = (int)(b->max_ns / CH_TL + 3);
  if (!b->generic && (rc = b->d_mag.alloc_zero((size_t)S * b->max_tiles * 16 * sizeof(float)))) return rc;
  // demod ring: history for the audio FIR halo + one chunk
  b->demod_cap = next_pow2(b->max_ns + std::max(AU_MAXHALO + AU_MAXLEAD, AF_N) + 64);
  if ((rc = b->d_demod.alloc_zero((size_t)S * M * b->demod_cap * sizeof(float)))) return rc;
  if (cfg->dsd_rate) {
    // the plan and its checks of dsd446_batch_create (src/dsd_in.c:104)
    b->dsd = design::msresamp_plan((float)cfg->dsd_rate / cfg->channel_width, cfg->resamp_as);
    if (!b->dsd.interp || b->dsd.stages != 1 || b->dsd.sub_len != 14 || b->dsd.m[0] > 10)
      return fail(PMR446_EINVAL, "dsd_rate: need one half-band stage after the arbitrary resampler (2 < dsd_rate / channel_width <= 4)");
    if (b->dsd.step < (1u << 23) || b->dsd.step > (1u << 24)) return fail(PMR446_EINVAL, "dsd_rate: arbitrary stage outside [1, 2]");
    // a call's first output reaches back 2 m - 1 outputs and 13 taps: at most 13 + 2 m frames behind its first frame
    if (b->demod_cap < b->max_ns + 13 + 2 * (long long)b->dsd.m[0] + 1) return fail(PMR446_EINVAL, "internal: discriminator ring too short for dsd_rate");
    b->max_dsd = 2 * ((long long)design::arb_outputs_after((uint64_t)b->max_ns, b->dsd.step) + 1);
    b->dsd_period = dsd_arb_period(b->dsd.step, b->dsd.bits);
    if ((b->max_dsd / 2 + DSB_KB - 1) / DSB_KB * (long long)S * M > 0x7fffffffLL) return fail(PMR446_EINVAL, "dsd_rate: too many rows for one launch");
    std::vector<float> rows((size_t)b->dsd.npfb * 16, 0.0f);
    for (unsigned i = 0; i < b->dsd.npfb; i++)
      for (unsigned k = 0; k < 14; k++) rows[(size_t)i * 16 + k] = b->dsd.pfb[(size_t)i * 14 + k];
    if ((rc = b->d_dsd_pfb.alloc(rows.size() * 4))) return rc;
    cudaMemcpy(b->d_dsd_pfb.p, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice);
  }

  // audio filters; the de-emphasis pole's warm-up also sets the length of its impulse response below
  if ((rc = b->au.init(*cfg))) return rc;
  // fast-convolution response: hp (x gain) * de-emphasis * optional low-pass, as one impulse response < AF_HALO
  {
    const std::vector<float>& hpt = b->au.hp;
    const std::vector<float>& lpt = b->au.lp;
    const unsigned fir_len = (unsigned)hpt.size() + (cfg->lowpass ? (unsigned)lpt.size() - 1 : 0) + (cfg->deemph_fir ? PMR446_FIR_DEEMPH_TAPS_LEN - 1 : 0);
    const double a1 = cfg->deemph_a1;
    const unsigned de_len = (unsigned)std::max(24, b->au.de_warm);   // the pole's response is cut where it is below 2^-30
    if (fir_len + de_len <= (unsigned)AF_HALO_LONG) {
      b->fft_halo = fir_len + de_len <= (unsigned)AF_HALO ? AF_HALO : AF_HALO_LONG;
      std::vector<double> h(hpt.begin(), hpt.end());
      for (auto& x : h) x *= (double)cfg->audio_gain;
      // de-emphasis (A.1): y[n] = b0 x[n] + b1 x[n-1] - a1 y[n-1]
      std::vector<double> de(de_len);
      de[0] = cfg->deemph_b0;
      de[1] = (double)cfg->deemph_b1 - a1 * de[0];
      for (size_t n = 2; n < de.size(); n++) de[n] = -a1 * de[n - 1];
      if (cfg->deemph_fir) {   // APP_FIR_DEEMPH: the reference's 101-tap table instead of the pole
        std::vector<float> df(PMR446_FIR_DEEMPH_TAPS_LEN);
        pmr446_fir_deemph_taps_fill(df.data());
        de.assign(df.begin(), df.end());
      }
      auto conv = [](const std::vector<double>& x, const std::vector<double>& y) {
        std::vector<double> z(x.size() + y.size() - 1, 0.0);
        for (size_t i = 0; i < x.size(); i++)
          for (size_t j = 0; j < y.size(); j++) z[i + j] += x[i] * y[j];
        return z;
      };
      h = conv(h, de);
      if (cfg->lowpass) h = conv(h, std::vector<double>(lpt.begin(), lpt.end()));
      std::vector<float2> resp(AF_N), tw(AF_N);
      for (int k = 0; k < AF_N; k++) {
        const double a = -2.0 * M_PI * (double)k / (double)AF_N;
        tw[k] = make_float2((float)cos(a), (float)sin(a));
      }
      for (int k0 = 0; k0 < 16; k0++)
        for (int t = 0; t < 256; t++) {
          const int k = (t >> 4) + 16 * (t & 15) + 256 * k0;
          double re = 0.0, im = 0.0;
          for (size_t n = 0; n < h.size(); n++) {
            const double a = -2.0 * M_PI * (double)(((long long)k * (long long)n) % AF_N) / (double)AF_N;
            re += h[n] * cos(a);
            im += h[n] * sin(a);
          }
          resp[k0 * 256 + t] = make_float2((float)(re / AF_N), (float)(im / AF_N));
        }
      if ((rc = b->d_resp.alloc(AF_N * sizeof(float2))) || (rc = b->d_aftw.alloc(AF_N * sizeof(float2)))) return rc;
      cudaMemcpy(b->d_resp.p, resp.data(), AF_N * sizeof(float2), cudaMemcpyHostToDevice);
      cudaMemcpy(b->d_aftw.p, tw.data(), AF_N * sizeof(float2), cudaMemcpyHostToDevice);
      b->fft_audio = true;
    }
  }
  if (cfg->deemph_fir && !b->fft_audio) return fail(PMR446_EINVAL, "deemph_fir needs the fast-convolution audio path (filters too long for its tile)");
  if (cfg->waterfall > 0 && (rc = b->wf.init(S, cfg->waterfall))) return rc;
  cudaFuncSetAttribute(audio_fft4_kernel<AF_HALO>, cudaFuncAttributeMaxDynamicSharedMemorySize, AF4_SMEM_BYTES);
  cudaFuncSetAttribute(audio_fft4_kernel<AF_HALO_LONG>, cudaFuncAttributeMaxDynamicSharedMemorySize, AF4_SMEM_BYTES);
  CUDA_TRY(cudaStreamCreateWithFlags(&b->own_stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&b->out_stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaEventCreateWithFlags(&b->ev_out, cudaEventDisableTiming));
  for (int i = 0; i < 2; i++) {
    CUDA_TRY(cudaEventCreateWithFlags(&b->ev_copied[i], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&b->ev_free[i], cudaEventDisableTiming));
  }
  // every table upload and attribute call above is synchronous: one check for all of them
  if (cudaDeviceSynchronize() != cudaSuccess || cudaGetLastError() != cudaSuccess) return fail(PMR446_ECUDA, "CUDA error while setting up the batch");
  *out = b.release();
  return PMR446_OK;
}

extern "C" int pmr446_batch_destroy(pmr446_batch* b) {
  if (!b) return PMR446_OK;
  cudaSetDevice(b->device);
  cudaDeviceSynchronize();
  if (b->own_stream) cudaStreamDestroy(b->own_stream);
  if (b->copy_stream) cudaStreamDestroy(b->copy_stream);
  if (b->out_stream) cudaStreamDestroy(b->out_stream);
  if (b->ev_out) cudaEventDestroy(b->ev_out);
  for (int i = 0; i < 2; i++) {
    if (b->ev_copied[i]) cudaEventDestroy(b->ev_copied[i]);
    if (b->ev_free[i]) cudaEventDestroy(b->ev_free[i]);
  }
  delete b;
  return PMR446_OK;
}

extern "C" long long pmr446_batch_max_res(const pmr446_batch* b) { return b ? b->max_res : 0; }
extern "C" long long pmr446_batch_max_ns(const pmr446_batch* b) { return b ? b->max_ns : 0; }
extern "C" int pmr446_batch_last_launches(const pmr446_batch* b) { return b ? b->launches : 0; }
extern "C" long long pmr446_batch_max_dsd(const pmr446_batch* b) { return b ? b->max_dsd : 0; }
extern "C" long long pmr446_batch_last_dsd(const pmr446_batch* b) { return b ? b->last_dsd : 0; }

static __global__ void gather_channel_kernel(const float* ring, long long stride, long long mask, int M, long long f0, long long ns, const int* channel,
                                             float* out, long long ld) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int s = blockIdx.y, c = channel[s];
  if (k >= ns || c < 0 || c >= M) return;
  out[(long long)s * ld + k] = ring[((long long)s * M + c) * stride + ((f0 + k) & mask)];
}

extern "C" int pmr446_batch_gather_channel(pmr446_batch* b, const int* channel, float* demod_out, long long ld, void* cuda_stream) {
  if (!b || !channel || !demod_out) return fail(PMR446_EINVAL, "null argument");
  if (b->last_ns > ld) return fail(PMR446_ERANGE, "ld too small");
  if (b->last_ns == 0) return PMR446_OK;
  cudaSetDevice(b->device);
  gather_channel_kernel<<<dim3((unsigned)((b->last_ns + 255) / 256), b->S), 256, 0, (cudaStream_t)cuda_stream>>>(
      (const float*)b->d_demod.p, b->demod_cap, b->demod_cap - 1, b->M, b->last_f0, b->last_ns, channel, demod_out, ld);
  CUDA_TRY(cudaGetLastError());
  return PMR446_OK;
}

extern "C" int pmr446_batch_timing(pmr446_batch* b, int enable) {
  if (!b) return fail(PMR446_EINVAL, "null handle");
  cudaSetDevice(b->device);
  cudaDeviceSynchronize();
  b->timer.clear();
  b->timer.enabled = enable != 0;
  return PMR446_OK;
}

extern "C" int pmr446_batch_get_timings(pmr446_batch* b, double* total_ms, long long* count, int n) {
  if (!b || !total_ms || !count) return fail(PMR446_EINVAL, "null argument");
  cudaSetDevice(b->device);
  CUDA_TRY(cudaDeviceSynchronize());
  b->timer.collect();
  for (int i = 0; i < n && i < TM_NTAGS; i++) { total_ms[i] = b->timer.total_ms[i]; count[i] = b->timer.count[i]; }
  return PMR446_OK;
}

extern "C" int pmr446_batch_reset(pmr446_batch* b) {
  if (!b) return fail(PMR446_EINVAL, "null handle");
  cudaSetDevice(b->device);
  cudaDeviceSynchronize();
  if (int rc = b->fe.reset()) return rc;
  CUDA_TRY(cudaMemset(b->d_demod.p, 0, b->d_demod.bytes));
  // cudaMemset on device memory is asynchronous to the host and the execute paths run on non-blocking streams, which
  // do not order against the legacy stream: finish the memsets before any execute call can start
  CUDA_TRY(cudaDeviceSynchronize());
  return PMR446_OK;
}

long long pmr::batch_frames_after(const pmr446_batch* b, unsigned n) {
  return b->fe.outputs_after(b->fe.n_in + (long long)n) / b->M - b->fe.n_out / b->M;
}

// Resampler outputs of the DSD feed once frames [0, F) exist; a call completing [F0, F1) owns [k(F0), k(F1)).
static long long dsd_outputs_after(const pmr446_batch* b, long long F) { return (long long)design::arb_outputs_after((uint64_t)F, b->dsd.step); }

// The caller's leading dimensions against the counts of a call of n samples (closed form), before any state advances: a
// rejected call leaves the handle untouched.
static int check_ld(const pmr446_batch* b, unsigned n, const pmr446_outputs* out) {
  if (out->res && b->fe.outputs_after(b->fe.n_in + (long long)n) - b->fe.n_out > out->res_ld) return fail(PMR446_ERANGE, "res_ld too small");
  if ((out->chan || out->demod || out->lpcomp || out->audio || out->pcm) && batch_frames_after(b, n) > out->ld) return fail(PMR446_ERANGE, "ld too small");
  if (out->dsd_audio || out->dsd_pcm) {
    if (!b->cfg.dsd_rate) return fail(PMR446_EINVAL, "dsd_audio / dsd_pcm need dsd_rate != 0");
    const long long f0 = b->fe.n_out / b->M, f1 = f0 + batch_frames_after(b, n);
    if (2 * (dsd_outputs_after(b, f1) - dsd_outputs_after(b, f0)) > out->dsd_ld) return fail(PMR446_ERANGE, "dsd_ld too small");
  }
  return PMR446_OK;
}

extern "C" int pmr446_batch_execute_device(pmr446_batch* b, const void* iq, long long iq_stride, unsigned n, const pmr446_outputs* out,
                                           unsigned* ny_out, unsigned* ns_out, void* cuda_stream) {
  if (!b || !out) return fail(PMR446_EINVAL, "null argument");
  if (n > b->cfg.max_chunk) return fail(PMR446_ERANGE, "chunk larger than max_chunk");
  cudaSetDevice(b->device);
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int S = b->S;
  b->launches = 0;
  b->last_dsd = 0;

  // ---- validate BEFORE any state advances: a failed call leaves the handle untouched ----------
  const int M = b->M;
  if (int rc = check_ld(b, n, out)) return rc;
  if ((out->rssi || out->chan_edge) && b->generic) return fail(PMR446_EINVAL, "rssi / chan_edge outputs need the 16-channel kernel");
  const long long tf0 = b->fe.n_out / M, tf1 = tf0 + batch_frames_after(b, n);
  if (!b->generic && (tf1 + CH_TL - 1) / CH_TL - tf0 / CH_TL > b->max_tiles) return fail(PMR446_ERANGE, "internal: tile count exceeds allocation");
  // ---- front end: [r0, r1) new resampler outputs in fe.out ring ------------------------------
  long long r0 = b->fe.n_out, r1 = 0;
  b->timer.mark(st, TM_START);
  // The fused front end leaves the zero-input part of its DC blocker to the consumer of the ring.  channelize16_kernel
  // adds it while staging its tiles; if anything else reads the new samples (res output, generic channelizer, waterfall)
  // the ring is finished in place first (one read-modify-write pass over the chunk).
  const bool want_wf_now = b->cfg.waterfall > 0 && (out->ascii || out->peak || out->psd);
  const bool defer_zir = !b->generic && !out->res && !want_wf_now;
  int rc = b->fe.execute(iq, iq_stride, n, st, &b->launches, &b->timer, defer_zir);
  if (rc) return rc;
  r1 = b->fe.n_out;
  const long long ny = r1 - r0;
  const long long f0 = r0 / M, f1 = r1 / M, ns = f1 - f0;  // frames: cbuffer carry of r % M samples (:804)
  b->last_f0 = f0;
  b->last_ns = ns;

  if (out->res && ny > 0) {
    gather_ring_kernel<float2><<<dim3((unsigned)((ny + 255) / 256), S), 256, 0, st>>>((const float2*)b->fe.out.p, b->fe.out_cap, b->fe.out_cap - 1,
                                                                                      r0, ny, (float2*)out->res, out->res_ld);
    b->launches++;
    b->timer.mark(st, TM_GATHER);
  }

  if (ny > 0 && b->generic) {
    // generic-M channelizer: mix once per sample -- every new sample, also in a call that completes no frame: the frames
    // of later calls read it from the mixed ring
    nco_mix_kernel<<<dim3((unsigned)((ny + 255) / 256), S), 256, 0, st>>>((const float2*)b->fe.out.p, (float2*)b->d_mixed.p, b->fe.out_cap,
                                                                          b->fe.out_cap - 1, r0, ny, b->dtheta);
    b->launches++;
  }
  if (ns > 0 && b->generic) {
    // ---- generic-M channelizer: FFT-based analysis bank over the mixed ring ---------------------------------------------
    ChanGenParams gp;
    memset(&gp, 0, sizeof gp);
    gp.mixed = (const float2*)b->d_mixed.p;
    gp.stride = b->fe.out_cap;
    gp.mask = b->fe.out_cap - 1;
    gp.r1 = r1;
    gp.n_streams = S;
    gp.M = M;
    gp.p = 2 * (int)b->cfg.pfb_m;
    gp.tile0 = f0 / CG_FT;
    gp.tiles = (int)((f1 + CG_FT - 1) / CG_FT - gp.tile0);
    gp.f0 = f0;
    gp.f1 = f1;
    gp.ref = 1.0f / (2 * M_PI * b->cfg.kf);
    gp.taps = (const float*)b->d_pfb_taps.p;
    gp.twiddle = (const float2*)b->d_tw.p;
    gp.n_stages = (int)b->radix.size();
    for (size_t i = 0; i < b->radix.size(); i++) gp.radix[i] = b->radix[i];
    gp.demod = (float*)b->d_demod.p;
    gp.demod_stride = b->demod_cap;
    gp.demod_mask = b->demod_cap - 1;
    gp.chan = (float2*)out->chan;
    gp.chan_ld = out->ld;
    const size_t smem = (size_t)M * (3 * sizeof(float2) + CG_FT * sizeof(float));
    if (b->generic_tile) channelize_generic_tile_kernel<26><<<(unsigned)((long long)S * gp.tiles), 512, channelize_generic_tile_smem(M), st>>>(gp);
    else channelize_generic_kernel<<<(unsigned)((long long)S * gp.tiles), 256, smem, st>>>(gp);
    b->launches++;
    b->timer.mark(st, TM_CHANNELIZE);
  } else if (ns > 0) {
    // ---- channelizer + discriminator --------------------------------------------------------
    ChanParams cp;
    cp.res = (const float2*)b->fe.out.p;
    cp.res_stride = b->fe.out_cap;
    cp.res_mask = b->fe.out_cap - 1;
    cp.r1 = r1;
    cp.n_streams = S;
    cp.tile0 = f0 / CH_TL;
    cp.tiles = (int)((f1 + CH_TL - 1) / CH_TL - cp.tile0);
    cp.f0 = f0;
    cp.f1 = f1;
    cp.dtheta = b->dtheta;
    cp.ref = 1.0f / (2 * M_PI * b->cfg.kf);
    cp.taps = (const float*)b->d_pfb_taps.p;
    cp.demod = (float*)b->d_demod.p;
    cp.demod_stride = b->demod_cap;
    cp.demod_mask = b->demod_cap - 1;
    cp.chan = (float2*)out->chan;
    cp.chan_ld = out->ld;
    memset(&cp.corr, 0, sizeof cp.corr);
    if (const Correction* pc = b->fe.pending_corr()) cp.corr = *pc;
    ChanTaps tp;
    tp.mag_part = out->rssi ? (float*)b->d_mag.p : nullptr;
    tp.edge = (float2*)out->chan_edge;
    if (cp.tiles > b->max_tiles) return fail(PMR446_ERANGE, "internal: tile count exceeds allocation");
    long long warps = (long long)S * cp.tiles;   // one warp per (stream, frame tile)
    unsigned blocks = (unsigned)((warps * 32 + 127) / 128);
    const bool taps = tp.mag_part || tp.edge;
    if (b->nco_lut && !taps) channelize16_kernel<true, false><<<blocks, 128, 0, st>>>(cp, tp);
    else if (b->nco_lut) channelize16_kernel<true, true><<<blocks, 128, 0, st>>>(cp, tp);
    else if (!taps) channelize16_kernel<false, false><<<blocks, 128, 0, st>>>(cp, tp);
    else channelize16_kernel<false, true><<<blocks, 128, 0, st>>>(cp, tp);
    b->launches++;
    if (out->rssi) {
      rssi_finalize_kernel<<<(S * 16 + 127) / 128, 128, 0, st>>>((const float*)b->d_mag.p, cp.tiles, S * 16, ns, out->rssi);
      b->launches++;
    }
    b->timer.mark(st, TM_CHANNELIZE);
    b->fe.fix_pending(st, &b->launches, false, &b->timer);   // the ring's tail is the next call's history: finish it in place
  } else if (out->rssi) {   // empty window: 0 / 0 like the reference's average_power()
    rssi_finalize_kernel<<<(S * 16 + 127) / 128, 128, 0, st>>>((const float*)b->d_mag.p, 0, S * 16, 0, out->rssi);
    b->launches++;
  }
  b->fe.fix_pending(st, &b->launches, true, &b->timer);      // no channelizer launch in this call (ns == 0): nothing was deferred to
  if (ns > 0) {
    if (out->demod) {
      gather_ring_kernel<float><<<dim3((unsigned)((ns + 255) / 256), S * M), 256, 0, st>>>((const float*)b->d_demod.p, b->demod_cap,
                                                                                           b->demod_cap - 1, f0, ns, out->demod, out->ld);
      b->launches++;
      b->timer.mark(st, TM_GATHER);
    }
    // ---- audio chain ------------------------------------------------------------------------
    const bool fft_now = b->fft_audio && (out->audio || out->pcm);
    if (fft_now) {
      AudioFftParams fp;
      fp.demod = (const float*)b->d_demod.p;
      fp.demod_stride = b->demod_cap;
      fp.demod_mask = b->demod_cap - 1;
      fp.rows = S * M;
      // tiles anchored at the call's first sample: ceil(ns / own) transforms per row instead of one more whenever the call
      // straddles the absolute grid (3.49 tiles' worth of a 1 s step: 4 instead of 4.49 on average)
      const long long af_own = AF_N - b->fft_halo;
      fp.tiles = (int)((f1 - f0 + af_own - 1) / af_own);
      fp.tile0 = 0;
      fp.f0 = f0;
      fp.f1 = f1;
      fp.resp = (const float2*)b->d_resp.p;
      fp.tw = (const float2*)b->d_aftw.p;
      fp.audio = out->audio;
      fp.pcm = out->pcm;
      fp.out_ld = out->ld;
      const unsigned fgrid = (unsigned)((long long)((fp.rows + 3) / 4) * fp.tiles);   // four rows per block (audio_fft4.cuh)
      if (b->fft_halo == AF_HALO) audio_fft4_kernel<AF_HALO><<<fgrid, AF_T, AF4_SMEM_BYTES, st>>>(fp);
      else audio_fft4_kernel<AF_HALO_LONG><<<fgrid, AF_T, AF4_SMEM_BYTES, st>>>(fp);
      b->launches++;
      b->timer.mark(st, TM_AUDIO);
    }
    if (fft_now ? out->lpcomp != nullptr : (out->audio || out->pcm || out->lpcomp)) {
      AudioParams ap;
      memset(&ap, 0, sizeof ap);
      ap.demod = (const float*)b->d_demod.p;
      ap.demod_stride = b->demod_cap;
      ap.demod_mask = b->demod_cap - 1;
      ap.rows = S * M;
      const long long own = AU_SPAN - b->au.lead;
      ap.tile0 = f0 / own;
      ap.tiles = (int)((f1 + own - 1) / own - ap.tile0);
      ap.f0 = f0;
      ap.f1 = f1;
      ap.audio = fft_now ? nullptr : out->audio;
      ap.pcm = fft_now ? nullptr : out->pcm;
      ap.lpcomp = out->lpcomp;
      ap.out_ld = out->ld;
      b->au.launch(ap, st);
      b->launches++;
      b->timer.mark(st, TM_AUDIO);
    }
  }
  // ---- per-channel DSD feed: msresamp_rrrf (src/dsd_in.c:170-175) over every discriminator row -------------------------------
  if (ns > 0 && (out->dsd_audio || out->dsd_pcm)) {
    const long long k0 = dsd_outputs_after(b, f0), k1 = dsd_outputs_after(b, f1);
    if (k1 > k0) {
      // dsd_in's back end over every (stream, channel) row of the discriminator ring, s16 saturated
      DsdBackendParams bp;
      memset(&bp, 0, sizeof bp);
      bp.fm = (const float*)b->d_demod.p;
      bp.fm_stride = b->demod_cap;
      bp.fm_mask = b->demod_cap - 1;
      bp.k0 = k0;
      bp.k1 = k1;
      bp.step = b->dsd.step;
      bp.bits = (int)b->dsd.bits;
      bp.period = b->dsd_period;
      bp.groups = DSB_T / b->dsd_period;
      bp.pfb = (const float*)b->d_dsd_pfb.p;
      bp.m = (int)b->dsd.m[0];
      for (size_t j = 0; j < b->dsd.hb[0].size() && j < 20; j++) bp.hb[j] = b->dsd.hb[0][j];
      bp.audio = out->dsd_audio;
      bp.pcm = out->dsd_pcm;
      bp.out_ld = out->dsd_ld;
      bp.tiles = (int)((k1 - k0 + DSB_KB - 1) / DSB_KB);
      const unsigned g = (unsigned)((long long)bp.tiles * S * M);
      if (bp.m == 10) dsd_backend_kernel<10, true><<<g, DSB_T, 0, st>>>(bp);   // the 60 dB plan
      else dsd_backend_kernel<0, true><<<g, DSB_T, 0, st>>>(bp);
      b->launches++;
      b->timer.mark(st, TM_DSD);
    }
    b->last_dsd = 2 * (k1 - k0);
  }
  // ---- waterfall on the un-mixed resampler output of this chunk (:910-913) -------------------
  if (b->cfg.waterfall > 0 && (out->ascii || out->peak || out->psd)) {
    rc = b->wf.execute((const float2*)b->fe.out.p, b->fe.out_cap, r0, ny, out->ascii, out->peak, out->psd, st, &b->launches);
    if (rc) return rc;
    b->timer.mark(st, TM_WATERFALL);
  }
  CUDA_TRY(cudaGetLastError());
  if (ny_out) *ny_out = (unsigned)ny;
  if (ns_out) *ns_out = (unsigned)ns;
  return PMR446_OK;
}

extern "C" int pmr446_batch_execute(pmr446_batch* b, const void* iq, long long iq_stride, unsigned n, const pmr446_outputs* out, unsigned* ny_out,
                                    unsigned* ns_out) {
  if (!b || !out || (!iq && n)) return fail(PMR446_EINVAL, "null argument");
  if (n > b->cfg.max_chunk) return fail(PMR446_ERANGE, "chunk larger than max_chunk");
  cudaSetDevice(b->device);
  cudaStream_t st = b->own_stream, cs = b->copy_stream;
  const int S = b->S, M = b->M;
  const size_t bps = (size_t)fmt_bytes_per_sample(b->cfg.in_fmt);
  const unsigned W = b->cfg.waterfall;
  if ((iq_stride = host_iq_stride(iq_stride, n, bps, S)) < 0) return (int)iq_stride;
  int rc;
  if ((rc = check_ld(b, n, out))) return rc;   // the caller's dimensions, before the first slice advances the state
  // Large chunks are cut in time into sub-chunks so that the host->device copy of sub-chunk k+1 overlaps
  // the kernels of sub-chunk k (all filter state carries across execute_device calls, so the result is the
  // same).  Not done when a waterfall row is requested: asgram produces one row per call (:911-912).
  const bool want_wf = W && (out->ascii || out->peak || out->psd);
  const bool want_sel = out->rssi || out->chan_edge;   // one call = one RSSI window: no time slices
  const unsigned K = (!want_wf && !want_sel && n >= 8u * 65536u) ? 8u : 1u;
  const unsigned sub = K == 1 ? n : ((n + K - 1) / K + 255u) / 256u * 256u;
  const long long pitch = ((long long)(sub ? sub : 1) * (long long)bps + 255) / 256 * 256;
  for (int i = 0; i < (K > 1 ? 2 : 1); i++)
    if ((rc = b->d_in2[i].ensure((size_t)S * pitch))) return rc;
  pmr446_outputs d = *out;
  const long long ld = b->max_ns, rld = b->max_res;
  d.ld = ld;
  d.res_ld = rld;
  Staging stage;
  d.res = stage(out->res, b->d_out_res, (size_t)S * rld * 8);
  d.chan = stage(out->chan, b->d_out_chan, (size_t)S * M * ld * 8);
  d.demod = stage(out->demod, b->d_out_demod, (size_t)S * M * ld * 4);
  d.lpcomp = stage(out->lpcomp, b->d_out_lpcomp, (size_t)S * M * ld * 4);
  d.audio = stage(out->audio, b->d_out_audio, (size_t)S * M * ld * 4);
  d.pcm = stage(out->pcm, b->d_out_pcm, (size_t)S * M * ld * 2);
  d.ascii = stage(W ? out->ascii : nullptr, b->d_out_ascii, (size_t)S * W);
  d.peak = stage(W ? out->peak : nullptr, b->d_out_peak, (size_t)S * 2 * 4);
  d.psd = stage(W ? out->psd : nullptr, b->d_out_psd, (size_t)S * 4 * W * 4);
  d.rssi = stage(out->rssi, b->d_out_rssi, (size_t)S * M * 4);
  d.chan_edge = stage(out->chan_edge, b->d_out_edge, (size_t)S * M * 2 * 8);
  const long long dld = b->max_dsd;
  d.dsd_ld = dld;
  d.dsd_audio = stage(out->dsd_audio, b->d_out_dsd_audio, (size_t)S * M * dld * 4);
  d.dsd_pcm = stage(out->dsd_pcm, b->d_out_dsd_pcm, (size_t)S * M * dld * 2);
  if (stage.rc) return stage.rc;
  unsigned ny_tot = 0, ns_tot = 0;
  long long dsd_tot = 0;
  int launches = 0;
  unsigned off = 0;
  // device -> host copies of a column range of every requested output; with time slices they run on their own stream
  // right behind each slice's kernels, i.e. concurrently with the next slices' host -> device copies (PCIe is duplex)
  auto back_range = [&](cudaStream_t s2, unsigned y0, unsigned ny_k, unsigned s0, unsigned ns_k, long long d0, long long nd_k) {
    copy_back(s2, out->res, d.res, out->res_ld, rld, 8, S, y0, ny_k);
    copy_back(s2, out->chan, d.chan, out->ld, ld, 8, (long long)S * M, s0, ns_k);
    copy_back(s2, out->demod, d.demod, out->ld, ld, 4, (long long)S * M, s0, ns_k);
    copy_back(s2, out->lpcomp, d.lpcomp, out->ld, ld, 4, (long long)S * M, s0, ns_k);
    copy_back(s2, out->audio, d.audio, out->ld, ld, 4, (long long)S * M, s0, ns_k);
    copy_back(s2, out->pcm, d.pcm, out->ld, ld, 2, (long long)S * M, s0, ns_k);
    copy_back(s2, out->dsd_audio, d.dsd_audio, out->dsd_ld, dld, 4, (long long)S * M, d0, nd_k);
    copy_back(s2, out->dsd_pcm, d.dsd_pcm, out->dsd_ld, dld, 2, (long long)S * M, d0, nd_k);
  };
  for (unsigned k = 0; k == 0 || off < n; k++) {
    const unsigned len = std::min(sub, n - off);
    const int buf = (int)(k & 1u);
    if (k >= 2) CUDA_TRY(cudaStreamWaitEvent(cs, b->ev_free[buf], 0));   // kernels of sub-chunk k-2 have read this buffer
    if (len) CUDA_TRY(cudaMemcpy2DAsync(b->d_in2[buf].p, pitch, (const char*)iq + (size_t)off * bps, iq_stride, (size_t)len * bps, S,
                                        cudaMemcpyHostToDevice, cs));
    CUDA_TRY(cudaEventRecord(b->ev_copied[buf], cs));
    CUDA_TRY(cudaStreamWaitEvent(st, b->ev_copied[buf], 0));
    pmr446_outputs dk = d;
    if (dk.res) dk.res += 2 * (size_t)ny_tot;
    if (dk.chan) dk.chan += 2 * (size_t)ns_tot;
    if (dk.demod) dk.demod += ns_tot;
    if (dk.lpcomp) dk.lpcomp += ns_tot;
    if (dk.audio) dk.audio += ns_tot;
    if (dk.pcm) dk.pcm += ns_tot;
    if (dk.dsd_audio) dk.dsd_audio += dsd_tot;   // a slice's columns start where the previous slices' k(F) left off
    if (dk.dsd_pcm) dk.dsd_pcm += dsd_tot;
    unsigned ny = 0, ns = 0;
    rc = pmr446_batch_execute_device(b, b->d_in2[buf].p, pitch, len, &dk, &ny, &ns, st);
    if (rc) return rc;
    launches += b->launches;
    CUDA_TRY(cudaEventRecord(b->ev_free[buf], st));
    if (K > 1) {
      CUDA_TRY(cudaEventRecord(b->ev_out, st));
      CUDA_TRY(cudaStreamWaitEvent(b->out_stream, b->ev_out, 0));
      back_range(b->out_stream, ny_tot, ny, ns_tot, ns, dsd_tot, b->last_dsd);
    }
    ny_tot += ny;
    ns_tot += ns;
    dsd_tot += b->last_dsd;
    off += len;
  }
  b->launches = launches;
  b->last_dsd = dsd_tot;
  const unsigned ny = ny_tot, ns = ns_tot;
  if (K == 1) back_range(st, 0, ny, 0, ns, 0, dsd_tot);
  copy_back(st, out->rssi, d.rssi, M, M, 4, S, 0, M);
  copy_back(st, out->chan_edge, d.chan_edge, 2 * M, 2 * M, 8, S, 0, 2 * M);
  if (W) {
    copy_back(st, out->ascii, d.ascii, W, W, 1, S, 0, W);
    copy_back(st, out->peak, d.peak, 2, 2, 4, S, 0, 2);
    copy_back(st, out->psd, d.psd, 4 * W, 4 * W, 4, S, 0, 4 * W);
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  CUDA_TRY(cudaStreamSynchronize(b->out_stream));
  if (ny_out) *ny_out = ny;
  if (ns_out) *ns_out = ns;
  return PMR446_OK;
}

// ================================================================================================
// FP32 peak probe: 8 independent FFMA chains per thread, register operands only.
// ================================================================================================
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters, float a, float bb) {
  float x[8];
#pragma unroll
  for (int i = 0; i < 8; i++) x[i] = (float)(threadIdx.x + i);
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < 16; u++) {
#pragma unroll
      for (int i = 0; i < 8; i++) x[i] = fmaf(x[i], a, bb);
    }
  }
  float s = 0.0f;
#pragma unroll
  for (int i = 0; i < 8; i++) s += x[i];
  if (s == 12345.678f) out[0] = s;
}

extern "C" int pmr446_measure_fp32_peak(double* tflops, void* cuda_stream) {
  if (!tflops) return fail(PMR446_EINVAL, "null argument");
  cudaStream_t st = (cudaStream_t)cuda_stream;
  int dev = 0, sms = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  float* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, 4));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  const int iters = 4096, blocks = sms * 8;
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    cudaEventRecord(e0, st);
    fp32_peak_kernel<<<blocks, 256, 0, st>>>(d, iters, 0.999f, 0.001f);
    cudaEventRecord(e1, st);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    double flops = 2.0 * 8 * 16 * (double)iters * 256.0 * blocks;
    double tf = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  CUDA_TRY(cudaGetLastError());
  *tflops = best;
  return PMR446_OK;
}

extern "C" const char* pmr446_last_error(void) { return pmr::last_error_string().c_str(); }

extern "C" int pmr446_host_alloc(void** ptr, unsigned long long bytes) {
  if (!ptr) return fail(PMR446_EINVAL, "null argument");
  *ptr = nullptr;
  if (int rc = select_device(-1)) return rc;
  if (cudaHostAlloc(ptr, bytes ? (size_t)bytes : 16, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    *ptr = nullptr;
    return fail(PMR446_ENOMEM, "cudaHostAlloc failed");
  }
  return PMR446_OK;
}

extern "C" int pmr446_host_free(void* ptr) {
  if (ptr) CUDA_TRY(cudaFreeHost(ptr));
  return PMR446_OK;
}

// ================================================================================================
// Host-only introspection of the filter design and the sample-count bookkeeping (no GPU needed).
// ================================================================================================
extern "C" int pmr446_design_msresamp(float rate, float as, unsigned* stages, unsigned* m /*[16]*/, unsigned* step, unsigned* npfb,
                                      float* hb_taps /*[16][20] or NULL*/, float* pfb /*[npfb][14] or NULL*/) {
  if (!(rate > 0.0f) || !stages || !m || !step || !npfb) return fail(PMR446_EINVAL, "bad argument");
  design::MsresampPlan p = design::msresamp_plan(rate, as);
  if (p.stages > 16) return fail(PMR446_EINVAL, "too many stages");
  *stages = p.stages;
  *step = p.step;
  *npfb = p.npfb;
  for (unsigned i = 0; i < p.stages; i++) {
    m[i] = p.m[i];
    if (hb_taps)
      for (size_t j = 0; j < 20; j++) hb_taps[i * 20 + j] = j < p.hb[i].size() ? p.hb[i][j] : 0.0f;
  }
  if (pfb) memcpy(pfb, p.pfb.data(), p.pfb.size() * sizeof(float));
  return PMR446_OK;
}

// How the front end would run msresamp_crcf_create(rate, as) for the given input format: "fused[3,5,10]+arb",
// "cascade[3,3,3,3] | cascade[3,5] | tile[10]+arb", ... or an error.  Host logic only (no GPU needed).
extern "C" int pmr446_describe_frontend(float rate, float as, int in_fmt, int with_dc, char* buf, int len) {
  if (!(rate > 0.0f) || !buf || len < 8) return fail(PMR446_EINVAL, "bad argument");
  if (rate > 1.0f) return fail(PMR446_EINVAL, "front end only decimates (rate <= 1)");
  design::MsresampPlan p = design::msresamp_plan(rate, as);
  std::vector<std::vector<int>> groups;
  bool fused = false, front6 = false;
  if (int rc = Frontend::plan_groups(p, in_fmt, &groups, &fused, &front6)) return rc;
  std::string out;
  for (size_t l = 0; l < groups.size(); l++) {
    const bool arb = l + 1 == groups.size();
    const int src = l == 0 ? fmt_source(in_fmt) : SRC_RING;
    const int dc = (l == 0 && with_dc) ? ((groups.size() >= 2 || fused) ? DC_ZSR : DC_SCAN) : DC_NONE;
    int ms[4] = {0, 0, 0, 0}, G = 0;
    for (size_t k = 0; k < groups[l].size() && k < 4; k++) ms[k] = groups[l][k];
    const bool tile = arb && src == SRC_RING && groups[l].size() == 1 && ms[0] == 10 && p.step == (3u << 23);
    const bool f6 = front6 && l == 0;
    if (!fused && !tile && !f6 && !pick_cascade(src, dc, arb, ms, &G)) return fail(PMR446_EINVAL, "resampler plan not built: kernel not instantiated");
    if (l) out += " | ";
    out += fused ? "fused[" : (f6 ? "front6[" : (tile ? "tile[" : "cascade["));
    for (size_t k = 0; k < groups[l].size(); k++) out += (k ? "," : "") + std::to_string(groups[l][k]);
    out += arb ? "]+arb" : "]";
  }
  snprintf(buf, (size_t)len, "%s", out.c_str());
  return PMR446_OK;
}

extern "C" int pmr446_design_pfbch(unsigned M, unsigned m, float as, float* taps /*[M][2m]*/) {
  if (!M || !m || !taps) return fail(PMR446_EINVAL, "bad argument");
  std::vector<float> t = design::pfbch_taps(M, m, as);
  memcpy(taps, t.data(), t.size() * sizeof(float));
  return PMR446_OK;
}

extern "C" int pmr446_design_asgram_window(unsigned W, float* w) {
  if (W < 2 || !w) return fail(PMR446_EINVAL, "bad argument");
  std::vector<float> t = design::asgram_window(W);
  memcpy(w, t.data(), t.size() * sizeof(float));
  return PMR446_OK;
}

extern "C" unsigned pmr446_design_nco_dtheta(float dtheta) { return design::nco_dtheta(dtheta); }

extern "C" int pmr446_bytes_per_sample(int in_fmt) { return fmt_bytes_per_sample(in_fmt); }

// Outputs of the decimating msresamp after n_in input samples in total (closed form, SURVEY.md A.2/A.5).
extern "C" long long pmr446_count_resampled(float rate, float as, long long n_in) {
  design::MsresampPlan p = design::msresamp_plan(rate, as);
  if (p.interp || n_in < 0) return -1;
  return (long long)design::arb_outputs_after((uint64_t)(n_in >> p.stages), p.step);
}
