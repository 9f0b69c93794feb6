// pmr446_receiver_*: the reference's receiver behaviour for n_streams receivers per call -- RSSI per
// channel, squelch / selector state machine, the selected channel's audio chain and the CTCSS
// detector (/root/reference/src/sdr_pmr446.c:828-908, :605-628, :330-418), layered on the batched
// front half (pmr446_batch_execute_device with the channelizer output kept on the device).
#include <math.h>

#include <memory>
#include <vector>

#include "../../include/pmr446_taps.h"
#include "backend.cuh"
#include "common_host.hpp"
#include "receiver.cuh"

using namespace pmr;

struct pmr446_receiver {
  pmr446_rx_config cfg;
  pmr446_batch* batch = nullptr;
  int S = 0, M = 0, device = 0;
  long long max_ns = 0, sel_cap = 0;
  DevBuf d_chan, d_rssi, d_state, d_u, d_range, d_sel, d_lpcomp, d_coef, d_freqs, d_edge, d_selchan, d_selrow;
  bool fused = false;        // 16-channel kernel: RSSI and edge samples come out of the channelizer, no [S][M][ns] buffer
  DirectAudio au;            // the selected channel's audio chain
  // staging for the host-buffer call
  DevBuf d_in, d_o_rssi, d_o_status, d_o_audio, d_o_pcm, d_o_ctcss_in, d_o_power, d_o_ascii, d_o_peak;
  cudaStream_t own_stream = nullptr;
  int launches = 0;
};

extern "C" void pmr446_rx_default_config(pmr446_rx_config* c) {
  memset(c, 0, sizeof(*c));
  pmr446_default_config(&c->chain);
  c->squelch_level = 18.0f;
  c->channel_mask = ~0ull;
  c->lock_mode = PMR446_LOCK_START;
  c->ctcss_block = 2441;
  c->ctcss_dc_alpha = 0.0005f;
}

static int rx_init_state(pmr446_receiver* r) {
  std::vector<RxState> st((size_t)r->S);
  for (auto& s : st) {
    memset(&s, 0, sizeof s);
    s.active = -1;          // src/sdr_pmr446.c:148
    s.ctcss_freq = -1.0f;   // :149
  }
  CUDA_TRY(cudaMemcpy(r->d_state.p, st.data(), st.size() * sizeof(RxState), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemset(r->d_u.p, 0, r->d_u.bytes));
  CUDA_TRY(cudaMemset(r->d_sel.p, 0, r->d_sel.bytes));
  return 0;
}

extern "C" int pmr446_receiver_create(const pmr446_rx_config* cfg, pmr446_receiver** out) {
  if (!cfg || !out) return fail(PMR446_EINVAL, "null argument");
  *out = nullptr;
  const unsigned M = cfg->chain.num_channels;
  if (M > 64) return fail(PMR446_EINVAL, "the receiver's channel mask covers at most 64 channels");
  const unsigned long long all = M == 64 ? ~0ull : ((1ull << M) - 1);
  if ((cfg->channel_mask & all) == 0) return fail(PMR446_EINVAL, "channel_mask enables no channel");   // :725
  if (cfg->ctcss_block < 1) return fail(PMR446_EINVAL, "ctcss_block must be positive");
  if (cfg->chain.deemph_fir) return fail(PMR446_EINVAL, "the receiver runs the direct-form audio chain: deemph_fir is not available");
  if (cfg->chain.dsd_rate) return fail(PMR446_EINVAL, "the receiver has no per-channel DSD feed: dsd_rate must be 0");
  pmr446_batch* batch = nullptr;
  int rc = pmr446_batch_create(&cfg->chain, &batch);
  if (rc) return rc;
  std::unique_ptr<pmr446_receiver, int (*)(pmr446_receiver*)> r(new pmr446_receiver(), pmr446_receiver_destroy);   // freed on every early return
  r->batch = batch;
  r->cfg = *cfg;
  cudaGetLastError();
  cudaGetDevice(&r->device);
  const int S = r->S = cfg->chain.n_streams;
  r->M = (int)M;
  r->max_ns = pmr446_batch_max_ns(r->batch);
  r->sel_cap = next_pow2(r->max_ns + AU_MAXHALO + AU_MAXLEAD + 64);
  // tone coefficients 2 cos(2 pi f / fs_audio), fs_audio = channel width (:24, :360-361)
  float coef[RX_TONES];
  const double fs_audio = (double)cfg->chain.channel_width;
  for (int j = 0; j < RX_TONES; j++) coef[j] = 2.0f * cosf((float)((2.0 * M_PI * pmr446_ctcss_freqs[j]) / fs_audio));
  r->fused = (M == 16 && cfg->chain.pfb_m == 13);
  if (r->fused) {
    if ((rc = r->d_edge.alloc_zero((size_t)S * M * 2 * sizeof(float2)))) return rc;
    if ((rc = r->d_selrow.alloc((size_t)S * r->max_ns * sizeof(float)))) return rc;
  } else if ((rc = r->d_chan.alloc((size_t)S * M * r->max_ns * sizeof(float2)))) {
    return rc;
  }
  if ((rc = r->d_selchan.alloc_zero((size_t)S * sizeof(int)))) return rc;
  if ((rc = r->d_rssi.alloc_zero((size_t)S * M * sizeof(float)))) return rc;
  if ((rc = r->d_state.alloc((size_t)S * sizeof(RxState)))) return rc;
  if ((rc = r->d_u.alloc((size_t)S * 3 * RX_TONES * sizeof(float)))) return rc;
  if ((rc = r->d_range.alloc_zero((size_t)S * 2 * sizeof(long long)))) return rc;
  if ((rc = r->d_sel.alloc((size_t)S * r->sel_cap * sizeof(float)))) return rc;
  if ((rc = r->d_lpcomp.alloc((size_t)S * r->max_ns * sizeof(float)))) return rc;
  if ((rc = r->au.init(cfg->chain))) return rc;
  if ((rc = r->d_coef.alloc(sizeof coef))) return rc;
  if ((rc = r->d_freqs.alloc(sizeof pmr446_ctcss_freqs))) return rc;
  if ((rc = rx_init_state(r.get()))) return rc;
  cudaMemcpy(r->d_coef.p, coef, sizeof coef, cudaMemcpyHostToDevice);
  cudaMemcpy(r->d_freqs.p, pmr446_ctcss_freqs, sizeof pmr446_ctcss_freqs, cudaMemcpyHostToDevice);
  CUDA_TRY(cudaStreamCreateWithFlags(&r->own_stream, cudaStreamNonBlocking));
  if (cudaDeviceSynchronize() != cudaSuccess || cudaGetLastError() != cudaSuccess) return fail(PMR446_ECUDA, "CUDA error while setting up the receiver");
  *out = r.release();
  return PMR446_OK;
}

extern "C" int pmr446_receiver_destroy(pmr446_receiver* r) {
  if (!r) return PMR446_OK;
  cudaSetDevice(r->device);
  cudaDeviceSynchronize();
  if (r->own_stream) cudaStreamDestroy(r->own_stream);
  pmr446_batch_destroy(r->batch);
  delete r;
  return PMR446_OK;
}

extern "C" long long pmr446_receiver_max_ns(const pmr446_receiver* r) { return r ? r->max_ns : 0; }
extern "C" int pmr446_receiver_last_launches(const pmr446_receiver* r) { return r ? r->launches : 0; }

extern "C" int pmr446_receiver_reset(pmr446_receiver* r) {
  if (!r) return fail(PMR446_EINVAL, "null handle");
  cudaSetDevice(r->device);
  cudaDeviceSynchronize();
  if (int rc = pmr446_batch_reset(r->batch)) return rc;
  if (int rc = rx_init_state(r)) return rc;
  CUDA_TRY(cudaDeviceSynchronize());   // see pmr446_batch_reset
  return PMR446_OK;
}

// The caller's leading dimension against the frames of a call of n samples (closed form), before the batch advances
// any state: a rejected call leaves the handle untouched.
static int check_ld(const pmr446_receiver* r, unsigned n, const pmr446_rx_outputs* out) {
  if ((out->audio || out->pcm || out->ctcss_in) && batch_frames_after(r->batch, n) > out->ld) return fail(PMR446_ERANGE, "ld too small");
  return PMR446_OK;
}

extern "C" int pmr446_receiver_execute_device(pmr446_receiver* r, const void* iq, long long iq_stride, unsigned n, const pmr446_rx_outputs* out,
                                              unsigned* ns_out, void* cuda_stream) {
  if (!r || !out) return fail(PMR446_EINVAL, "null argument");
  if (int rc = check_ld(r, n, out)) return rc;
  cudaSetDevice(r->device);
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int S = r->S, M = r->M;
  // front half: DC block .. channelizer, channel samples kept in d_chan [S][M][max_ns]
  pmr446_outputs bo;
  memset(&bo, 0, sizeof bo);
  bo.chan = r->fused ? nullptr : (float*)r->d_chan.p;
  bo.rssi = r->fused ? (float*)r->d_rssi.p : nullptr;
  bo.chan_edge = r->fused ? (float*)r->d_edge.p : nullptr;
  bo.ld = r->max_ns;
  bo.ascii = out->ascii;
  bo.peak = out->peak;
  unsigned ny = 0, ns = 0;
  int rc = pmr446_batch_execute_device(r->batch, iq, iq_stride, n, &bo, &ny, &ns, st);
  if (rc) return rc;
  r->launches = pmr446_batch_last_launches(r->batch);

  float* rssi = (float*)r->d_rssi.p;
  RxState* state = (RxState*)r->d_state.p;
  if (!r->fused) rssi_kernel<<<S * M, 128, 0, st>>>((const float2*)r->d_chan.p, r->max_ns, (int)ns, rssi);
  if (out->rssi) CUDA_TRY(cudaMemcpyAsync(out->rssi, rssi, (size_t)S * M * sizeof(float), cudaMemcpyDeviceToDevice, st));
  SquelchParams sp;
  sp.rssi = rssi;
  sp.st = state;
  sp.u = (float*)r->d_u.p;
  sp.sel_range = (long long*)r->d_range.p;
  sp.sel_chan = (int*)r->d_selchan.p;
  sp.S = S;
  sp.M = M;
  sp.ns = (int)ns;
  sp.squelch = r->cfg.squelch_level;
  sp.mask = r->cfg.channel_mask;
  sp.lock_max = r->cfg.lock_mode == PMR446_LOCK_MAX;
  squelch_kernel<<<(S + 127) / 128, 128, 0, st>>>(sp);
  r->launches += 2;
  if (ns > 0) {
    const float ref = 1.0f / (2 * (float)M_PI * r->cfg.chain.kf);
    if (r->fused) {
      if ((rc = pmr446_batch_gather_channel(r->batch, (const int*)r->d_selchan.p, (float*)r->d_selrow.p, r->max_ns, st))) return rc;
      rx_append_kernel<<<dim3((ns + 255) / 256, S), 256, 0, st>>>((const float*)r->d_selrow.p, r->max_ns, (const float2*)r->d_edge.p, M, (int)ns, state,
                                                                    ref, (float*)r->d_sel.p, r->sel_cap, r->sel_cap - 1);
      r->launches++;
    } else {
      rx_demod_kernel<<<dim3((ns + 255) / 256, S), 256, 0, st>>>((const float2*)r->d_chan.p, r->max_ns, M, (int)ns, state, ref, (float*)r->d_sel.p,
                                                                   r->sel_cap, r->sel_cap - 1);
    }
    AudioParams ap;
    memset(&ap, 0, sizeof ap);
    ap.demod = (const float*)r->d_sel.p;
    ap.demod_stride = r->sel_cap;
    ap.demod_mask = r->sel_cap - 1;
    ap.rows = S;
    const long long own = AU_SPAN - r->au.lead;
    ap.tiles = (int)((ns + own - 1) / own + 1);   // a row's range may straddle one more tile boundary than its length suggests
    ap.row_range = (const long long*)r->d_range.p;
    ap.audio = out->audio;
    ap.pcm = out->pcm;
    ap.lpcomp = (float*)r->d_lpcomp.p;
    ap.out_ld = out->ld;
    ap.lpcomp_ld = r->max_ns;
    r->au.launch(ap, st);
    r->launches += 2;
  }
  CtcssParams cp;
  cp.lpcomp = (const float*)r->d_lpcomp.p;
  cp.ld = r->max_ns;
  cp.st = state;
  cp.u = (float*)r->d_u.p;
  cp.coef = (const float*)r->d_coef.p;
  cp.freqs = (const float*)r->d_freqs.p;
  cp.dc_a1 = -1.0f + r->cfg.ctcss_dc_alpha;
  cp.block = r->cfg.ctcss_block;
  cp.ctcss_in = out->ctcss_in;
  cp.power_out = out->ctcss_power;
  cp.status = out->status;
  cp.out_ld = out->ld;
  ctcss_kernel<<<S, CT_THREADS, 0, st>>>(cp);
  r->launches++;
  CUDA_TRY(cudaGetLastError());
  if (ns_out) *ns_out = ns;
  return PMR446_OK;
}

extern "C" int pmr446_receiver_execute(pmr446_receiver* r, const void* iq, long long iq_stride, unsigned n, const pmr446_rx_outputs* out,
                                       unsigned* ns_out) {
  if (!r || !out || (!iq && n)) return fail(PMR446_EINVAL, "null argument");
  if (n > r->cfg.chain.max_chunk) return fail(PMR446_ERANGE, "chunk larger than max_chunk");
  cudaSetDevice(r->device);
  cudaStream_t st = r->own_stream;
  const int S = r->S, M = r->M;
  const size_t bps = (size_t)fmt_bytes_per_sample(r->cfg.chain.in_fmt);
  const unsigned W = r->cfg.chain.waterfall;
  if ((iq_stride = host_iq_stride(iq_stride, n, bps, S)) < 0) return (int)iq_stride;
  int rc;
  if ((rc = check_ld(r, n, out))) return rc;
  const long long pitch = ((long long)(n ? n : 1) * (long long)bps + 255) / 256 * 256;
  if ((rc = r->d_in.ensure((size_t)S * pitch))) return rc;
  if (n) CUDA_TRY(cudaMemcpy2DAsync(r->d_in.p, pitch, iq, iq_stride, (size_t)n * bps, S, cudaMemcpyHostToDevice, st));
  const long long ld = r->max_ns;
  pmr446_rx_outputs d;
  memset(&d, 0, sizeof d);
  d.ld = ld;
  Staging stage;
  d.rssi = stage(out->rssi, r->d_o_rssi, (size_t)S * M * 4);
  d.status = stage(out->status, r->d_o_status, (size_t)S * sizeof(pmr446_rx_status));
  d.audio = stage(out->audio, r->d_o_audio, (size_t)S * ld * 4);
  d.pcm = stage(out->pcm, r->d_o_pcm, (size_t)S * ld * 2);
  d.ctcss_in = stage(out->ctcss_in, r->d_o_ctcss_in, (size_t)S * ld * 4);
  d.ctcss_power = stage(out->ctcss_power, r->d_o_power, (size_t)S * RX_TONES * 4);
  d.ascii = stage(W ? out->ascii : nullptr, r->d_o_ascii, (size_t)S * W);
  d.peak = stage(W ? out->peak : nullptr, r->d_o_peak, (size_t)S * 2 * 4);
  if (stage.rc) return stage.rc;
  unsigned ns = 0;
  if ((rc = pmr446_receiver_execute_device(r, r->d_in.p, pitch, n, &d, &ns, st))) return rc;
  copy_back(st, out->rssi, d.rssi, M, M, 4, S, 0, M);
  copy_back(st, out->status, d.status, 1, 1, sizeof(pmr446_rx_status), S, 0, 1);
  copy_back(st, out->audio, d.audio, out->ld, ld, 4, S, 0, ns);
  copy_back(st, out->pcm, d.pcm, out->ld, ld, 2, S, 0, ns);
  copy_back(st, out->ctcss_in, d.ctcss_in, out->ld, ld, 4, S, 0, ns);
  copy_back(st, out->ctcss_power, d.ctcss_power, RX_TONES, RX_TONES, 4, S, 0, RX_TONES);
  if (W) {
    copy_back(st, out->ascii, d.ascii, W, W, 1, S, 0, W);
    copy_back(st, out->peak, d.peak, 2, 2, 4, S, 0, 2);
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  if (ns_out) *ns_out = ns;
  return PMR446_OK;
}
