// audio_kernel: 377-tap CTCSS-removal high-pass FIR, complementary low-pass branch, audio gain,
// 1-pole de-emphasis, optional 103-tap low-pass, s16 conversion.  Replaces
// /root/reference/src/sdr_pmr446.c:882-902 (firfilt_rrrf_execute_block, wdelayf, iirfilt_rrrf;
// SURVEY.md Appendix A.1, A.10, A.11) for every channel, and the s16 cast of src/dsd_in.c:172-175.
//
// Direct form.  Since audio_fft_kernel (fast convolution) took over the audio / s16 outputs of the batched chain, this
// kernel serves the complementary CTCSS branch (lpcomp), the receiver's squelch-selected rows (per-row sample ranges) and
// configurations whose composite impulse response does not fit the FFT tile.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "audio_fft.cuh"   // pcm_sat

namespace pmr {

// One block = one (stream, channel) row x one time tile.  Thread t owns 16 consecutive output
// samples; the tile's input (with a halo of taps-1 samples) sits in shared memory with one pad
// word every 16 so that the per-thread sliding windows (lane stride 17 words) are bank-conflict
// free.  The FIR runs 16 taps x 16 outputs per step from registers: 256 FFMA per 16 LDS (samples)
// + 4 LDS.128 (broadcast taps).  The first `lead` outputs of a tile are lead-in (de-emphasis
// warm-up, low-pass halo) and are not stored; threads whose outputs are not needed skip the FIR.
struct AudioParams {
  const float* demod;      // ring [rows][demod_stride]
  long long demod_stride, demod_mask;
  int rows;                // n_streams * 16
  int tiles;               // tiles per row
  long long tile0;         // tile k covers outputs [k*own, (k+1)*own), own = AU_SPAN - lead
  long long f0, f1;        // owned samples
  const long long* row_range;   // optional [rows][2]: per-row {f0, f1} (device memory) replacing f0/f1/tile0 -- the
                           // squelch-selected stream of the receiver advances at a different pace per stream
  int lead;                // lead-in outputs per tile (multiple of 16; 16 without, 128 with the low-pass)
  const float* hp_taps;    // [HP_PAD] zero-padded to a multiple of 16
  int hp_chunks;           // HP_PAD / 16
  int hp_delay;            // (hp_len - 1) / 2
  const float* lp_taps;    // optional second FIR (103 taps padded); nullptr = off
  int lp_chunks;
  float gain;
  float de_b0, de_b1, de_a1;
  float* audio;            // optional [rows][out_ld] float audio, column = f - f0
  short* pcm;              // optional [rows][out_ld]
  float* lpcomp;           // optional [rows][out_ld]
  long long out_ld;
  long long lpcomp_ld;     // row stride of lpcomp; 0 = out_ld
  int de_warm;             // audio_kernel<true>: de-emphasis warm-up per thread (deemph_warmup(de_a1)); lead >= de_warm
};

constexpr int AU_THREADS = 128;
constexpr int AU_SPAN = AU_THREADS * 16;   // outputs computed per tile (incl. lead-in)
constexpr int AU_LEAD_LP = 128;            // lead-in with the 103-tap low-pass (>= 112 + 8)
constexpr int AU_LEAD_MIN = 16;            // lead-in without it (de-emphasis warm-up of 8)
constexpr int AU_MAXHALO = 384;            // >= padded HP length
constexpr int AU_MAXLEAD = AU_SPAN / 2;    // longest lead-in a tile may spend on de-emphasis warm-up

// Samples after which the one-pole de-emphasis has forgotten a state dropped at the start of a span to 2^-30 of its value:
// the least k with |a1|^k <= 2^-30.  -1 if the pole does not decay (|a1| >= 1).
inline int deemph_warmup(double a1) {
  const double m = fabs(a1);
  if (!(m < 1.0)) return -1;
  if (m < 0x1p-30) return 1;
  return (int)ceil(log(0x1p-30) / log(m));
}

// Lead-in of an audio_kernel tile: every stored output sees the low-pass span (16 lp_chunks - 1 with the low-pass) of
// de-emphasis outputs, each warmed up over `warm` samples inside the tile.  The reference's pole (warm-up 5) keeps
// AU_LEAD_MIN / AU_LEAD_LP.  -1 if the warm-up does not fit (lead > AU_MAXLEAD).
inline int audio_lead(bool lowpass, int lp_chunks, int warm) {
  const int base = lowpass ? AU_LEAD_LP : AU_LEAD_MIN;
  const int need = ((lowpass ? 16 * lp_chunks - 1 : 0) + warm + 15) / 16 * 16;
  const int lead = need > base ? need : base;
  return lead > AU_MAXLEAD ? -1 : lead;
}

__device__ __forceinline__ int padidx(int i) { return i + (i >> 4); }

// acc[r] += sum_k taps[k] * x[base + r - k], r < 16, k < 16*chunks, for this thread.
// xs is the padded tile; `top` = padded-layout-free index of x[base] (multiple of 16).
__device__ __forceinline__ void fir16(const float* __restrict__ xs, const float* __restrict__ ts, int top, int chunks, float* acc) {
  // window registers: lo = x[top - 16kb - 15 .. top - 16kb], hi = previous lo
  float wa[16], wb[16];
  // first chunk needs x[top .. top + 15] as the "hi" part (r - kk > 0)
  {
    const float* q = xs + padidx(top);
#pragma unroll
    for (int i = 0; i < 16; i++) wb[i] = q[i];   // top is a multiple of 16: no pad inside
  }
  auto step = [&](float* lo, const float* hi, int kb) {
    // lo[i] = x[top - 16(kb+1) + i], i < 16 ; hi[i] = x[top - 16 kb + i]
    const float* q = xs + padidx(top - 16 * (kb + 1));
#pragma unroll
    for (int i = 0; i < 16; i++) lo[i] = q[i];
    const float4* t4 = (const float4*)(ts + 16 * kb);
    float4 t0 = t4[0], t1 = t4[1], t2 = t4[2], t3 = t4[3];
    const float tk[16] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w, t2.x, t2.y, t2.z, t2.w, t3.x, t3.y, t3.z, t3.w};
#pragma unroll
    for (int kk = 0; kk < 16; kk++) {
#pragma unroll
      for (int r = 0; r < 16; r++) {
        const int d = r - kk;  // x index relative to top - 16 kb
        const float xv = d >= 0 ? hi[d] : lo[16 + d];
        acc[r] = fmaf(tk[kk], xv, acc[r]);
      }
    }
  };
  int kb = 0;
#pragma unroll 1
  for (; kb + 1 < chunks; kb += 2) {
    step(wa, wb, kb);
    step(wb, wa, kb + 1);
  }
  if (kb < chunks) step(wa, wb, kb);
}

// LONG_POLE = false: the de-emphasis state of each thread's 16 outputs is rebuilt from 8 samples of warm-up (pole
// magnitude up to 0.074 for 2^-30); true: from p.de_warm samples, for poles that decay more slowly.
template <bool LONG_POLE>
static __global__ void __launch_bounds__(AU_THREADS) audio_kernel(AudioParams p) {
  extern __shared__ float smem[];
  // layout: xs[padidx(AU_MAXHALO + AU_SPAN + 16)] input tile; ys[...] second buffer (gain*hp, then de-emph)
  constexpr int XN = AU_MAXHALO + AU_SPAN + 16;
  float* xs = smem;
  float* ys = smem + padidx(XN) + 1;
  float* ts = ys + padidx(AU_LEAD_LP + AU_SPAN + 16) + 1;   // taps (16-byte aligned below)
  ts = (float*)(((uintptr_t)ts + 15) & ~(uintptr_t)15);

  const int row = blockIdx.x / p.tiles;
  const int lead = p.lead, own = AU_SPAN - lead;
  long long pf0 = p.f0, pf1 = p.f1, tile = p.tile0 + blockIdx.x % p.tiles;
  if (p.row_range) {
    pf0 = p.row_range[2 * row];
    pf1 = p.row_range[2 * row + 1];
    tile = pf0 / own + blockIdx.x % p.tiles;
    if (tile * own >= pf1) return;   // block-uniform
  }
  const long long o0 = tile * own - lead;   // absolute index of computed output 0 (multiple of 16)
  const float* drow = p.demod + (long long)row * p.demod_stride;
  const int t = threadIdx.x;
  // everything below is 32-bit and relative to o0
  const long long lo64 = pf0 - o0, hi64 = pf1 - o0;
  const int f0r = (int)(lo64 < -(1 << 28) ? -(1 << 28) : lo64);                 // first owned output, relative
  const int f1r = (int)(hi64 > (1 << 28) ? (1 << 28) : hi64);                   // one past the last available input/output
  const int z0r = (int)(-o0 > (1 << 28) ? (1 << 28) : (-o0 < -(1 << 28) ? -(1 << 28) : -o0));   // stream start, relative

  // load x[o0 - AU_MAXHALO .. o0 + AU_SPAN): four samples per thread and step; negative absolute
  // indices (before the stream start) and samples not yet produced read as zero
  {
    const unsigned base32 = (unsigned)(o0 - AU_MAXHALO), dmask = (unsigned)p.demod_mask;
    for (int i = 4 * t; i < AU_MAXHALO + AU_SPAN; i += 4 * AU_THREADS) {
      const int rel = i - AU_MAXHALO;   // relative to o0
      float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      if (rel >= z0r && rel + 4 <= f1r) {
        v = *(const float4*)(drow + ((base32 + (unsigned)i) & dmask));
      } else if (rel + 4 > z0r && rel < f1r) {
        const float* q = drow;
        if (rel + 0 >= z0r && rel + 0 < f1r) v.x = q[(base32 + (unsigned)i + 0u) & dmask];
        if (rel + 1 >= z0r && rel + 1 < f1r) v.y = q[(base32 + (unsigned)i + 1u) & dmask];
        if (rel + 2 >= z0r && rel + 2 < f1r) v.z = q[(base32 + (unsigned)i + 2u) & dmask];
        if (rel + 3 >= z0r && rel + 3 < f1r) v.w = q[(base32 + (unsigned)i + 3u) & dmask];
      }
      float* d = xs + padidx(i);
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
  }
  const int hp_n = p.hp_chunks * 16, lp_n = p.lp_taps ? p.lp_chunks * 16 : 0;
  for (int i = t; i < hp_n; i += AU_THREADS) ts[i] = p.hp_taps[i];
  for (int i = t; i < lp_n; i += AU_THREADS) ts[hp_n + i] = p.lp_taps[i];
  __syncthreads();

  // is any of this thread's 16 outputs stored, or needed as lead-in by a stored one?
  const int ob = 16 * t;                                     // relative index of this thread's first output
  const bool need = (ob < f1r) && (ob + 16 + lead > f0r);

  // high-pass FIR: outputs o0 + 16 t + r
  float acc[16];
#pragma unroll
  for (int r = 0; r < 16; r++) acc[r] = 0.0f;
  const int top = AU_MAXHALO + 16 * t;
  if (need) fir16(xs, ts, top, p.hp_chunks, acc);

  const bool own_thread = (ob >= lead);
  // complementary low-pass branch (A.11): delayed input minus high-pass output
  if (p.lpcomp && own_thread && need) {
    float* lrow = p.lpcomp + (long long)row * (p.lpcomp_ld ? p.lpcomp_ld : p.out_ld);
#pragma unroll
    for (int r = 0; r < 16; r++) {
      const int f = ob + r;
      if (f >= f0r && f < f1r) lrow[f - f0r] = xs[padidx(top + r - p.hp_delay)] - acc[r];
    }
  }
  // gain, then de-emphasis (A.1, Direct Form II): v = x - a1 v1 ; y = b0 v + b1 v1
#pragma unroll
  for (int r = 0; r < 16; r++) {
    acc[r] *= p.gain;
    ys[padidx(AU_LEAD_LP + 16 * t + r)] = acc[r];
  }
  __syncthreads();
  {
    float v1 = 0.0f;
    if (LONG_POLE) {
      // outputs before the tile's first one read as zero: start at the later of the warm-up span and the tile start
      for (int k = min(p.de_warm, 16 * t); k >= 1; k--) v1 = fmaf(-p.de_a1, v1, ys[padidx(AU_LEAD_LP + 16 * t - k)]);
    } else {
      // the reference's pole magnitude is 0.0146: eight samples of warm-up reproduce the running state to < 1e-14
#pragma unroll
      for (int k = 8; k >= 1; k--) {
        const int idx = AU_LEAD_LP + 16 * t - k;
        const float xv = (idx >= AU_LEAD_LP) ? ys[padidx(idx)] : 0.0f;
        v1 = fmaf(-p.de_a1, v1, xv);
      }
    }
#pragma unroll
    for (int r = 0; r < 16; r++) {
      const float v0 = fmaf(-p.de_a1, v1, acc[r]);
      acc[r] = fmaf(p.de_b0, v0, p.de_b1 * v1);
      v1 = v0;
    }
  }
  if (p.lp_taps) {
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 16; r++) ys[padidx(AU_LEAD_LP + 16 * t + r)] = acc[r];
    if (t < AU_LEAD_LP / 16) {
#pragma unroll
      for (int r = 0; r < 16; r++) ys[padidx(16 * t + r)] = 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 16; r++) acc[r] = 0.0f;
    if (need && own_thread) fir16(ys, ts + hp_n, AU_LEAD_LP + 16 * t, p.lp_chunks, acc);
  }
  // stage through shared memory for coalesced, arbitrarily aligned stores
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 16; r++) xs[padidx(16 * t + r)] = acc[r];
  __syncthreads();
  float* arow = p.audio ? p.audio + (long long)row * p.out_ld : nullptr;
  short* prow = p.pcm ? p.pcm + (long long)row * p.out_ld : nullptr;
  const int s_lo = lead > f0r ? lead : f0r, s_hi = AU_SPAN < f1r ? AU_SPAN : f1r;   // stored outputs, relative
  for (int i = s_lo + t; i < s_hi; i += AU_THREADS) {
    const float v = xs[padidx(i)];
    if (arow) arow[i - f0r] = v;
    if (prow) prow[i - f0r] = pcm_sat(v);
  }
}

}  // namespace pmr
