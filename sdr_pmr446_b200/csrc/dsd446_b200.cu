// C-ABI implementation of the batched dsd_in chain (include/pmr446_b200.h, dsd446_*).
// Mirrors init_liquid() and the main-loop body of /root/reference/src/dsd_in.c:95-112, :159-180:
//   DC block -> msresamp_crcf down to 12.5 kHz -> freqdem -> msresamp_rrrf up to 48 kHz -> s16.
// Host logic only; arithmetic is in frontend.cuh (shared with the PMR chain) and dsd.cuh.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <memory>
#include <vector>

#include "../../include/pmr446_b200.h"
#include "common_host.hpp"
#include "frontend_host.hpp"
#include "design.hpp"
#include "dsd.cuh"

using namespace pmr;

struct dsd446_batch {
  dsd446_config cfg;
  int S = 0, device = 0;
  Frontend fe;                    // DC + decimating msresamp -> 12.5 kHz ring
  design::MsresampPlan up;        // interpolating msresamp_rrrf plan
  DevBuf d_fm, d_pfb_up;
  long long fm_cap = 0;
  int launches = 0;          // kernels launched by the last execute call
  int arb_period = 32;       // (near-)period of the up-sampler's phase sequence in outputs (dsd_backend_kernel)
  long long n_z = 0;              // arbitrary-resampler outputs produced so far
  long long max_res = 0, max_out = 0;
  DevBuf d_in, d_res, d_fmout, d_audio, d_pcm;
  cudaStream_t own_stream = nullptr;
};

extern "C" void dsd446_default_config(dsd446_config* c) {
  memset(c, 0, sizeof(*c));
  c->n_streams = 1;
  c->device = -1;
  c->fs_in = 1024000;
  c->in_fmt = PMR446_FMT_CF32;
  c->fs_sig = 12500;
  c->fs_audio = 48000;
  c->max_chunk = 200000;
  c->dc_alpha = 0.0005f;
  c->resamp_as = 60.0f;
  c->kf = 0.5f;
}

extern "C" int dsd446_batch_destroy(dsd446_batch* b) {
  if (!b) return PMR446_OK;
  cudaSetDevice(b->device);
  cudaDeviceSynchronize();
  if (b->own_stream) cudaStreamDestroy(b->own_stream);
  delete b;
  return PMR446_OK;
}

extern "C" int dsd446_batch_create(const dsd446_config* cfg, dsd446_batch** out) {
  if (!cfg || !out) return fail(PMR446_EINVAL, "null argument");
  *out = nullptr;
  if (cfg->n_streams < 1 || cfg->max_chunk < 1 || cfg->fs_in == 0 || cfg->fs_sig == 0) return fail(PMR446_EINVAL, "bad configuration");
  if (int rc = select_device(cfg->device)) return rc;
  cudaGetLastError();   // clean slate for the check at the end
  std::unique_ptr<dsd446_batch, int (*)(dsd446_batch*)> b(new dsd446_batch(), dsd446_batch_destroy);   // freed on every early return
  b->cfg = *cfg;
  b->S = cfg->n_streams;
  cudaGetDevice(&b->device);
  int rc = b->fe.init(b->S, cfg->in_fmt, ((float)cfg->fs_sig) / cfg->fs_in, cfg->resamp_as, true, cfg->dc_alpha, cfg->max_chunk, 64);
  if (rc) return rc;
  b->up = design::msresamp_plan(((float)cfg->fs_audio) / cfg->fs_sig, cfg->resamp_as);
  if (!b->up.interp || b->up.stages != 1 || b->up.sub_len != 14 || b->up.m[0] > 10)
    return fail(PMR446_EINVAL, "up-sampler plan not built: need one half-band stage after the arbitrary resampler (2 < rate <= 4)");
  if (b->up.step < (1u << 23) || b->up.step > (1u << 24)) return fail(PMR446_EINVAL, "up-sampler plan not built: arbitrary stage outside (1, 2]");
  b->arb_period = dsd_arb_period(b->up.step, b->up.bits);
  b->max_res = b->fe.max_out_per_chunk();
  const long long max_z = (long long)design::arb_outputs_after((uint64_t)b->max_res, b->up.step) + 2;
  b->max_out = 2 * max_z;
  b->fm_cap = next_pow2(b->max_res + 64);
  std::vector<float> rows((size_t)b->up.npfb * 16, 0.0f);
  for (unsigned i = 0; i < b->up.npfb; i++)
    for (unsigned k = 0; k < 14; k++) rows[(size_t)i * 16 + k] = b->up.pfb[(size_t)i * 14 + k];
  if ((rc = b->d_fm.alloc_zero((size_t)b->S * b->fm_cap * 4)) || (rc = b->d_pfb_up.alloc(rows.size() * 4))) return rc;
  cudaMemcpy(b->d_pfb_up.p, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice);
  CUDA_TRY(cudaStreamCreateWithFlags(&b->own_stream, cudaStreamNonBlocking));
  if (cudaDeviceSynchronize() != cudaSuccess || cudaGetLastError() != cudaSuccess) return fail(PMR446_ECUDA, "CUDA error while setting up the dsd batch");
  *out = b.release();
  return PMR446_OK;
}

extern "C" long long dsd446_batch_max_res(const dsd446_batch* b) { return b ? b->max_res : 0; }
extern "C" long long dsd446_batch_max_out(const dsd446_batch* b) { return b ? b->max_out : 0; }
extern "C" int dsd446_batch_last_launches(const dsd446_batch* b) { return b ? b->launches : 0; }

extern "C" int dsd446_batch_reset(dsd446_batch* b) {
  if (!b) return fail(PMR446_EINVAL, "null handle");
  cudaSetDevice(b->device);
  cudaDeviceSynchronize();
  if (int rc = b->fe.reset()) return rc;
  b->n_z = 0;
  CUDA_TRY(cudaMemset(b->d_fm.p, 0, b->d_fm.bytes));
  CUDA_TRY(cudaDeviceSynchronize());   // see pmr446_batch_reset
  return PMR446_OK;
}

// The caller's leading dimensions against the counts of a call of n samples (closed form), before any state advances: a
// rejected call leaves the handle untouched.
static int check_ld(const dsd446_batch* b, unsigned n, const dsd446_outputs* out) {
  const long long r1 = b->fe.outputs_after(b->fe.n_in + (long long)n);
  const long long nz = 2 * ((long long)design::arb_outputs_after((uint64_t)r1, b->up.step) - b->n_z);
  if ((out->res || out->fm) && r1 - b->fe.n_out > out->res_ld) return fail(PMR446_ERANGE, "res_ld too small");
  if ((out->audio || out->pcm) && nz > out->out_ld) return fail(PMR446_ERANGE, "out_ld too small");
  return PMR446_OK;
}

extern "C" int dsd446_batch_execute_device(dsd446_batch* b, const void* iq, long long iq_stride, unsigned n, const dsd446_outputs* out,
                                           unsigned* ny_out, unsigned* nz_out, void* cuda_stream) {
  if (!b || !out) return fail(PMR446_EINVAL, "null argument");
  if (n > b->cfg.max_chunk) return fail(PMR446_ERANGE, "chunk larger than max_chunk");
  cudaSetDevice(b->device);
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int S = b->S;
  int launches = 0;
  const long long r0 = b->fe.n_out;
  int rc = check_ld(b, n, out);
  if (rc) return rc;
  rc = b->fe.execute(iq, iq_stride, n, st, &launches);   // src/dsd_in.c:167-168
  if (rc) return rc;
  const long long r1 = b->fe.n_out, ny = r1 - r0;
  const long long k0 = b->n_z, k1 = (long long)design::arb_outputs_after((uint64_t)r1, b->up.step);
  const long long nz = 2 * (k1 - k0);
  if (ny > 0) {
    dim3 g((unsigned)((ny + 255) / 256), S);
    dsd_freqdem_kernel<<<g, 256, 0, st>>>((const float2*)b->fe.out.p, b->fe.out_cap, b->fe.out_cap - 1, (float*)b->d_fm.p, b->fm_cap,
                                          b->fm_cap - 1, r0, r1, (float)(1.0f / (2 * M_PI * b->cfg.kf)));   // :169
    launches += 1 + (out->res ? 1 : 0) + (out->fm ? 1 : 0);
    if (out->res) gather_ring_kernel<float2><<<g, 256, 0, st>>>((const float2*)b->fe.out.p, b->fe.out_cap, b->fe.out_cap - 1, r0, ny,
                                                                 (float2*)out->res, out->res_ld);
    if (out->fm) gather_ring_kernel<float><<<g, 256, 0, st>>>((const float*)b->d_fm.p, b->fm_cap, b->fm_cap - 1, r0, ny, out->fm, out->res_ld);
  }
  if (k1 > k0 && (out->audio || out->pcm)) {                  // :170-175
    DsdBackendParams bp;
    memset(&bp, 0, sizeof bp);
    bp.fm = (const float*)b->d_fm.p;
    bp.fm_stride = b->fm_cap;
    bp.fm_mask = b->fm_cap - 1;
    bp.k0 = k0;
    bp.k1 = k1;
    bp.step = b->up.step;
    bp.bits = (int)b->up.bits;
    bp.period = b->arb_period;
    bp.groups = DSB_T / b->arb_period;
    bp.pfb = (const float*)b->d_pfb_up.p;
    bp.m = (int)b->up.m[0];
    for (size_t j = 0; j < b->up.hb[0].size() && j < 20; j++) bp.hb[j] = b->up.hb[0][j];
    bp.audio = out->audio;
    bp.pcm = out->pcm;
    bp.out_ld = out->out_ld;
    bp.tiles = (int)((k1 - k0 + DSB_KB - 1) / DSB_KB);
    const unsigned g = (unsigned)((long long)bp.tiles * S);
    if (bp.m == 10) dsd_backend_kernel<10, false><<<g, DSB_T, 0, st>>>(bp);   // the reference's 60 dB plan
    else dsd_backend_kernel<0, false><<<g, DSB_T, 0, st>>>(bp);
    launches++;
  }
  b->launches = launches;
  b->n_z = k1;
  CUDA_TRY(cudaGetLastError());
  if (ny_out) *ny_out = (unsigned)ny;
  if (nz_out) *nz_out = (unsigned)nz;
  return PMR446_OK;
}

extern "C" int dsd446_batch_execute(dsd446_batch* b, const void* iq, long long iq_stride, unsigned n, const dsd446_outputs* out, unsigned* ny_out,
                                    unsigned* nz_out) {
  if (!b || !out || (!iq && n)) return fail(PMR446_EINVAL, "null argument");
  if (n > b->cfg.max_chunk) return fail(PMR446_ERANGE, "chunk larger than max_chunk");
  cudaSetDevice(b->device);
  cudaStream_t st = b->own_stream;
  const int S = b->S;
  const size_t bps = (size_t)fmt_bytes_per_sample(b->cfg.in_fmt);
  if ((iq_stride = host_iq_stride(iq_stride, n, bps, S)) < 0) return (int)iq_stride;
  int rc;
  if ((rc = check_ld(b, n, out))) return rc;
  const long long in_row = (long long)((b->cfg.max_chunk * bps + 63) / 64 * 64);
  if ((rc = b->d_in.ensure((size_t)S * in_row))) return rc;
  if (n) CUDA_TRY(cudaMemcpy2DAsync(b->d_in.p, in_row, iq, iq_stride, (size_t)n * bps, S, cudaMemcpyHostToDevice, st));
  dsd446_outputs d = *out;
  d.res_ld = b->max_res;
  d.out_ld = b->max_out;
  Staging stage;
  d.res = stage(out->res, b->d_res, (size_t)S * d.res_ld * 8);
  d.fm = stage(out->fm, b->d_fmout, (size_t)S * d.res_ld * 4);
  d.audio = stage(out->audio, b->d_audio, (size_t)S * d.out_ld * 4);
  d.pcm = stage(out->pcm, b->d_pcm, (size_t)S * d.out_ld * 2);
  if (stage.rc) return stage.rc;
  unsigned ny = 0, nz = 0;
  if ((rc = dsd446_batch_execute_device(b, b->d_in.p, in_row, n, &d, &ny, &nz, st))) return rc;
  copy_back(st, out->res, d.res, out->res_ld, d.res_ld, 8, S, 0, ny);
  copy_back(st, out->fm, d.fm, out->res_ld, d.res_ld, 4, S, 0, ny);
  copy_back(st, out->audio, d.audio, out->out_ld, d.out_ld, 4, S, 0, nz);
  copy_back(st, out->pcm, d.pcm, out->out_ld, d.out_ld, 2, S, 0, nz);
  CUDA_TRY(cudaStreamSynchronize(st));
  if (ny_out) *ny_out = ny;
  if (nz_out) *nz_out = nz;
  return PMR446_OK;
}
