// channelize16_kernel: NCO mix-down + 16-channel polyphase analysis filter bank + 16-point DFT +
// NBFM discriminator.  Replaces the inner loop /root/reference/src/sdr_pmr446.c:804-823
// (nco_crcf_mix_down/step, firpfbch_crcf_analyzer_execute, transpose) and
// freqdem_demodulate_block (:881) for every channel (SURVEY.md Appendix A.7-A.9).
//
// Round-2 mapping (round 1: one sample per lane and frame, 1.47 ms per 1024-stream step, 98 warp instructions per frame):
// one warp walks a tile of 160 frames of one stream in five batches of 32 frames, all in its own shared-memory slice.
//  Staging: the batch's 32 new frames (16 samples each) go from the 200 kHz ring to shared memory with 128-bit loads;
//   on the way in each sample gets (a) the zero-input part of the front end's DC blocker when the fused front end left
//   it to its consumer (Correction, frontend.cuh) and (b) the NCO phasor -- theta_j = j dtheta only depends on j mod 32
//   when 32 dtheta = 0 mod 2^32 (the reference's 17/32-cycle step), so a lane multiplies by four constants.  The 25
//   frames of filter history are kept from the previous batch.
//  Phase A (branch filters): lane = (branch i, half g): 8 consecutive frames of its branch per pass from a 33-sample
//   register window, all 26 taps in registers, one packed FFMA2 per complex tap (scalar-broadcast operand); two passes
//   cover the lane's 16 frames.  The commutator sends resampled sample 16 f + 15 - i to branch i; the dot product of
//   frame f goes to shared memory row f, column n = 15 - i (the DFT input index).
//  Phase B + C: lane = frame: 16-point forward DFT in registers, the channel values go back to the lane's shared-memory row
//   and the previous frame's are read from the row before it (row -1 = the last frame of the previous batch), discriminator arg(conj(y[f-1]) y[f]) with a polynomial
//   atan2 (|err| < 3e-7 rad), and for every channel ONE coalesced 128-byte store of 32 consecutive frames into the
//   channel's ring row -- no transpose pass.
// Frame 0 of a tile only provides the "previous frame" of frame 1, so a tile owns 159 frames.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "audio_fft.cuh"   // dft16 / af_dig
#include "frontend.cuh"    // Correction
#include "packed_f32.cuh"

namespace pmr {

struct ChanParams {
  const float2* res;       // resampler output ring [n_streams][res_stride]
  long long res_stride, res_mask;
  long long r1;            // resampler outputs available: [.., r1)
  int n_streams;
  int tiles;               // tiles per stream
  long long tile0;         // index of the first tile (tile k covers frames [k*TL, (k+1)*TL))
  long long f0, f1;        // owned frames [f0, f1)
  unsigned dtheta;         // NCO phase increment per sample (A.7)
  float ref;               // 1 / (2 pi kf)
  const float* taps;       // [16][26] branch taps, newest first
  float* demod;            // ring [n_streams*16][demod_stride]
  long long demod_stride, demod_mask;
  float2* chan;            // optional: [n_streams][16][chan_ld], column = f - f0
  long long chan_ld;
  Correction corr;         // zero-input response of the front end's DC blocker still to be added to ring samples >= corr.from
};
struct ChanTaps {          // selector taps, only read by the TAPS instantiation
  float* mag_part;         // optional: [n_streams][tiles][16] sum of |y| over the owned frames of each tile (RSSI, :330-336)
  float2* edge;            // optional: [n_streams][16][2] channel sample of the first (f0) and last (f1 - 1) owned frame
};

constexpr int CH_NB = 5;                      // batches per tile
constexpr int CH_FR = 32 * CH_NB;             // computed frames per tile
constexpr int CH_TL = CH_FR - 1;              // owned frames per tile
constexpr int CH_HIST = 25;                   // frames of branch-filter history in front of a batch (26 taps)
constexpr int CH_XN = (CH_HIST + 32) * 16;    // float2 per sample buffer: 57 frames
constexpr int CH_V_STRIDE = 17;               // float2 per frame row of the branch-output buffer (16 + 1 pad)
constexpr int CH_SMEM_WARP = CH_XN + 33 * CH_V_STRIDE + 1;    // 33 rows (row 0 = the previous batch's last frame); even: the
                                                              // sample buffers of all four warps stay 16-byte aligned
static_assert(CH_SMEM_WARP % 2 == 0 && CH_XN % 2 == 0, "128-bit shared-memory accesses need 16-byte aligned warp slices");

// atan2 by a degree-17 odd minimax polynomial on [0, 1] (Abramowitz & Stegun 4.4.49, |err| <= 2e-8 in
// exact arithmetic, < 3e-7 rad in float32); (0, 0) falls back to libm for the signed-zero cases.
__device__ __forceinline__ float fast_atan2f(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  // (+-0, +-0): the quotient is taken as 0, and the quadrant comes from the SIGN BITS below, which gives libm's
  // atan2(+-0, +0) = +-0 and atan2(+-0, -0) = +-pi without a branch
  const float a = __fdividef(mn, mx == 0.0f ? 1.0f : mx);
  const float s = a * a;
  float r = 0.0028662257f;
  r = fmaf(r, s, -0.0161657367f);
  r = fmaf(r, s, 0.0429096138f);
  r = fmaf(r, s, -0.0752896400f);
  r = fmaf(r, s, 0.1065626393f);
  r = fmaf(r, s, -0.1420889944f);
  r = fmaf(r, s, 0.1999355085f);
  r = fmaf(r, s, -0.3333314528f);
  r = fmaf(r, s, 1.0f);
  r *= a;
  if (ay > ax) r = 1.57079632679489662f - r;
  if (__float_as_int(x) < 0) r = 3.14159265358979324f - r;
  return copysignf(r, y);
}
// two at once: the quotient and the quadrant logic stay scalar, the polynomial runs packed (9 FFMA2 for two arguments)
__device__ __forceinline__ float2 fast_atan2f_x2(float y0, float x0, float y1, float x1) {
  const float ax0 = fabsf(x0), ay0 = fabsf(y0), ax1 = fabsf(x1), ay1 = fabsf(y1);
  const float mx0 = fmaxf(ax0, ay0), mn0 = fminf(ax0, ay0), mx1 = fmaxf(ax1, ay1), mn1 = fminf(ax1, ay1);
  const float2 a = make_float2(__fdividef(mn0, mx0 == 0.0f ? 1.0f : mx0), __fdividef(mn1, mx1 == 0.0f ? 1.0f : mx1));
  const float2 s = fmul2(a, a);
  auto k2 = [](float c) { return make_float2(c, c); };
  float2 r = k2(0.0028662257f);
  r = ffma2(r, s, k2(-0.0161657367f));
  r = ffma2(r, s, k2(0.0429096138f));
  r = ffma2(r, s, k2(-0.0752896400f));
  r = ffma2(r, s, k2(0.1065626393f));
  r = ffma2(r, s, k2(-0.1420889944f));
  r = ffma2(r, s, k2(0.1999355085f));
  r = ffma2(r, s, k2(-0.3333314528f));
  r = ffma2(r, s, k2(1.0f));
  r = fmul2(r, a);
  if (ay0 > ax0) r.x = 1.57079632679489662f - r.x;
  if (ay1 > ax1) r.y = 1.57079632679489662f - r.y;
  if (__float_as_int(x0) < 0) r.x = 3.14159265358979324f - r.x;
  if (__float_as_int(x1) < 0) r.y = 3.14159265358979324f - r.y;
  return make_float2(copysignf(r.x, y0), copysignf(r.y, y1));
}

// forward 16-point DFT like dft16<false> (audio_fft.cuh; output q ends in v[af_dig(q)]) with the plain complex
// additions as packed FADD2: 6 packed + 4 scalar instructions per radix-4 butterfly instead of 16 scalar ones
__device__ __forceinline__ void dft4p(float2& a, float2& b, float2& c, float2& d) {
  const float2 s0 = fadd2(a, c), s2 = fadd2(b, d);
  const float2 s1 = fsub2(a, c), s3 = fsub2(b, d);
  a = fadd2(s0, s2);
  c = fsub2(s0, s2);
  b = make_float2(s1.x + s3.y, s1.y - s3.x);
  d = make_float2(s1.x - s3.y, s1.y + s3.x);
}
__device__ __forceinline__ void dft16p(float2* v) {
#pragma unroll
  for (int m0 = 0; m0 < 4; m0++) dft4p(v[m0], v[m0 + 4], v[m0 + 8], v[m0 + 12]);
  rot16<1, false>(v[5]);  rot16<2, false>(v[9]);   rot16<3, false>(v[13]);
  rot16<2, false>(v[6]);  rot16<4, false>(v[10]);  rot16<6, false>(v[14]);
  rot16<3, false>(v[7]);  rot16<6, false>(v[11]);  rot16<9, false>(v[15]);
#pragma unroll
  for (int q1 = 0; q1 < 4; q1++) dft4p(v[4 * q1], v[4 * q1 + 1], v[4 * q1 + 2], v[4 * q1 + 3]);
}

__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

template <bool TAPS> struct TapState { float macc[16]; };
template <> struct TapState<false> {};

// TAPS = the selector taps (mag_part / edge) are wanted: a separate instantiation, so that the throughput path carries
// none of their registers.
template <bool NCO_CONST, bool TAPS>
__global__ void __launch_bounds__(128, TAPS ? 3 : 4) channelize16_kernel(ChanParams p, ChanTaps tp) {
  __shared__ __align__(16) float2 ch_smem[4 * CH_SMEM_WARP];
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (warp >= (long long)p.n_streams * p.tiles) return;   // warp-uniform
  float2* const X = ch_smem + (threadIdx.x >> 5) * CH_SMEM_WARP;   // [57 frames][16 samples], mixed
  float2* const V = X + CH_XN + CH_V_STRIDE;                       // [-1 .. 31 frames][17]: branch outputs (column = DFT input index), then
                                                                   // channel values; row -1 = the previous batch's last frame
  const int s = (int)(warp / p.tiles);
  const int tile_idx = (int)(warp % p.tiles);
  const long long fa = (p.tile0 + tile_idx) * CH_TL, fs = fa - 1;  // computed frames are fs + k, k in [0, 160)
  const float2* res = p.res + (long long)s * p.res_stride;

  // ---- staging bounds, 32-bit and relative to J0 = index of the sample X[0] of batch 0 ------------------------------------
  const long long J0 = 16 * (fs - CH_HIST);
  auto clampi = [](long long v) { return (int)(v < -(1 << 29) ? -(1 << 29) : (v > (1 << 29) ? (1 << 29) : v)); };
  const int lo_rel = clampi(-J0);               // samples with jrel < lo_rel lie before the stream start: zero
  const int hi_rel = clampi(p.r1 - J0);         // samples with jrel >= hi_rel do not exist yet: zero
  const unsigned j0_32 = (unsigned)J0, rmask = (unsigned)p.res_mask;
  const Correction& cr = p.corr;
  const float2* vrow = cr.v_seg ? cr.v_seg + (long long)s * cr.nseg : nullptr;
  const int from_rel = clampi(cr.from - J0), seg_rel0 = clampi(J0 - cr.seg0_out);
  const unsigned smask = (1u << cr.seg_shift) - 1u;
  const float nalpha = -cr.alpha;
  // NCO phasors (A.7): theta_j = j dtheta mod 2^32.  A lane always stages samples with the same j mod 32 per region
  // (history region: X index 2 lane + 64 i; new-frame region: 400 + 2 lane + 64 i), so four constants when 32 dtheta = 0.
  float pcs[2][2], psn[2][2];
  if (NCO_CONST) {
#pragma unroll
    for (int reg = 0; reg < 2; reg++)
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const unsigned th = (j0_32 + (unsigned)(reg * CH_HIST * 16 + 2 * lane + e)) * p.dtheta;
        sincospif((float)(int)th * (1.0f / 2147483648.0f), &psn[reg][e], &pcs[reg][e]);
      }
  }
  // stages X[pp], X[pp + 1] (pp even) of the batch whose X[0] is sample J0 + boff
  auto stage_pair = [&](int pp, int boff, int reg) {
    const int jrel = boff + pp;
    float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (jrel + 1 >= lo_rel && jrel < hi_rel) {
      v = *(const float4*)(res + ((j0_32 + (unsigned)jrel) & rmask));   // jrel even: aligned, never straddles the ring's end
      if (jrel < lo_rel) { v.x = 0.0f; v.y = 0.0f; }
      if (jrel + 1 >= hi_rel) { v.z = 0.0f; v.w = 0.0f; }
      if (vrow && jrel + 1 >= from_rel) {
        // x -= alpha V0[segment] E[k]: the producer's segments hold an even number of ring samples, both share one
        const int rel = seg_rel0 + jrel;
        const int sg = rel >> cr.seg_shift;
        if (rel >= 0 && sg < cr.nseg) {
          const float2 v0 = vrow[sg];
          const float2 e = *(const float2*)(cr.e + cr.halo_out + ((unsigned)rel & smask));
          const float ax = nalpha * v0.x, ay = nalpha * v0.y;
          if (jrel >= from_rel && jrel >= lo_rel) { v.x = fmaf(ax, e.x, v.x); v.y = fmaf(ay, e.x, v.y); }
          if (jrel + 1 < hi_rel) { v.z = fmaf(ax, e.y, v.z); v.w = fmaf(ay, e.y, v.w); }
        }
      }
      float c0, s0, c1, s1;
      if (NCO_CONST) {
        c0 = pcs[reg][0]; s0 = psn[reg][0]; c1 = pcs[reg][1]; s1 = psn[reg][1];
      } else {
        const unsigned th = (j0_32 + (unsigned)jrel) * p.dtheta;
        sincospif((float)(int)th * (1.0f / 2147483648.0f), &s0, &c0);
        sincospif((float)(int)(th + p.dtheta) * (1.0f / 2147483648.0f), &s1, &c1);
      }
      v = make_float4(fmaf(v.x, c0, v.y * s0), fmaf(v.y, c0, -v.x * s0),    // x conj(e^{j theta})
                      fmaf(v.z, c1, v.w * s1), fmaf(v.w, c1, -v.z * s1));
    }
    *(float4*)(X + pp) = v;
  };

  // branch taps of this lane (phase A): branch i, newest sample first
  const int br = lane & 15, half = lane >> 4;
  float h[26];
#pragma unroll
  for (int n = 0; n < 26; n++) h[n] = __ldg(p.taps + br * 26 + n);

  // ownership of computed frame k (relative to fs): [own_lo, own_hi), and never k = 0
  long long lo64 = (fa > p.f0 ? fa : p.f0) - fs, hi64 = ((fa + CH_TL) < p.f1 ? (fa + CH_TL) : p.f1) - fs;
  const int own_lo = (int)(lo64 < 1 ? 1 : (lo64 > 4096 ? 4096 : lo64)), own_hi = (int)(hi64 < 0 ? 0 : (hi64 > 4096 ? 4096 : hi64));
  const unsigned fs32 = (unsigned)fs, dmask = (unsigned)p.demod_mask;
  const int crel = clampi(fs - p.f0);
  const int k_zero = (fs <= 0 && fs > -4096) ? (int)(-fs) : -1;   // computed frame k is absolute frame 0: r_prime = 0
  float* const drow0 = p.demod + (long long)s * 16 * p.demod_stride;
  float2* const crow0 = p.chan ? p.chan + (long long)s * 16 * p.chan_ld : nullptr;
  TapState<TAPS> ta;
  int k_first = -1, k_last = -1;
  if constexpr (TAPS) {
#pragma unroll
    for (int c = 0; c < 16; c++) ta.macc[c] = 0.0f;
    k_first = (int)(p.f0 - fs > 4096 ? -1 : (p.f0 - fs < 0 ? -1 : p.f0 - fs));
    k_last = (int)(p.f1 - 1 - fs > 4096 ? -1 : (p.f1 - 1 - fs < 0 ? -1 : p.f1 - 1 - fs));
  }

  // batches that hold no owned frame (a chunk boundary inside the tile) are skipped: the first one needed is the one
  // with the frame before the first owned frame, the last one the one with the last owned frame
  const bool any = own_hi > own_lo;             // (every launched tile owns a frame; kept warp-uniform and safe anyway)
  const int b_first = any ? (own_lo - 1) / 32 : 0, b_last = any ? (own_hi - 1) / 32 : -1;

  if (lane < 16) V[-CH_V_STRIDE + lane] = make_float2(0.0f, 0.0f);

  // steady-state staging (warp-uniform per batch): every new sample of the batch exists and they all take the same
  // correction path.  Then the batch's eight 128-bit loads per lane are issued back to back when it is staged, from L2:
  // its samples were prefetched there one batch ahead (128 registers, 4 blocks per SM; holding the loads in registers
  // across the previous batch's phase B + C instead takes 168 registers, 3 blocks per SM).
  auto steady = [&](int b, bool& corr_all) {
    const int jb = 512 * b + CH_HIST * 16, rel_b = seg_rel0 + jb;
    corr_all = vrow && jb >= from_rel && rel_b >= 0 && ((rel_b + 511) >> cr.seg_shift) < cr.nseg;
    const bool corr_none = !vrow || jb + 512 <= from_rel;
    return NCO_CONST && jb >= lo_rel && jb + 512 <= hi_rel && (corr_all || corr_none);
  };
  // history of the first batch, steady state: all seven 128-bit loads per lane in flight at once (the guarded
  // stage_pair loop below takes one DRAM round trip per pair)
  auto stage_history_fast = [&](int b) {
    const int jb = 512 * b, rel_b = seg_rel0 + jb;
    constexpr int NP = (CH_HIST * 16 / 2 + 31) / 32;   // 7, the last one partial
    const bool corr_all = vrow && jb >= from_rel && rel_b >= 0 && ((rel_b + CH_HIST * 16 - 1) >> cr.seg_shift) < cr.nseg;
    const bool corr_none = !vrow || jb + CH_HIST * 16 <= from_rel;
    if (!(NCO_CONST && jb >= lo_rel && jb + CH_HIST * 16 <= hi_rel && (corr_all || corr_none))) return false;
    float4 hv[NP];
#pragma unroll
    for (int i = 0; i < NP; i++) {
      const int pp = 2 * lane + 64 * i;
      hv[i] = pp < CH_HIST * 16 ? *(const float4*)(res + ((j0_32 + (unsigned)(jb + pp)) & rmask)) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
    if (corr_all) {
#pragma unroll
      for (int i = 0; i < NP; i++) {
        const int pp = 2 * lane + 64 * i;
        if (pp < CH_HIST * 16) {
          const unsigned rel = (unsigned)(rel_b + pp);
          const float2 v0 = vrow[rel >> cr.seg_shift];
          const float2 e = *(const float2*)(cr.e + cr.halo_out + (rel & smask));
          const float ax = nalpha * v0.x, ay = nalpha * v0.y;
          hv[i] = make_float4(fmaf(ax, e.x, hv[i].x), fmaf(ay, e.x, hv[i].y), fmaf(ax, e.y, hv[i].z), fmaf(ay, e.y, hv[i].w));
        }
      }
    }
    const float c0 = pcs[0][0], s0 = psn[0][0], c1 = pcs[0][1], s1 = psn[0][1];
#pragma unroll
    for (int i = 0; i < NP; i++) {
      const int pp = 2 * lane + 64 * i;
      if (pp < CH_HIST * 16)
        *(float4*)(X + pp) = make_float4(fmaf(hv[i].x, c0, hv[i].y * s0), fmaf(hv[i].y, c0, -hv[i].x * s0),
                                         fmaf(hv[i].z, c1, hv[i].w * s1), fmaf(hv[i].w, c1, -hv[i].z * s1));
    }
    return true;
  };
  auto prefetch_l2 = [&](int b) {
    const int jb = 512 * b + CH_HIST * 16;
#pragma unroll
    for (int i = 0; i < 8; i++) asm volatile("prefetch.global.L2 [%0];" ::"l"(res + ((j0_32 + (unsigned)(jb + 2 * lane + 64 * i)) & rmask)));
  };
  // steady() is monotone in the batch index, so a tile whose first and last batch are steady with the same correction
  // mode (almost every tile) needs no per-batch evaluation
  bool ca_next = false, ca_last = false;
  bool fast_next = any && steady(b_first, ca_next);
  const bool tile_steady = fast_next && steady(b_last, ca_last) && ca_last == ca_next;
  if (any && !stage_history_fast(b_first))
    for (int pp = 2 * lane; pp < CH_HIST * 16; pp += 64) stage_pair(pp, 512 * b_first, 0);   // history of the first batch

#pragma unroll 1
  for (int batch = b_first; batch <= b_last; batch++) {
    const int boff = 512 * batch;
    const bool fast = fast_next, corr_all = ca_next;
    if (batch > b_first) {   // the last 25 frames of the previous batch become this batch's history
      __syncwarp();
      constexpr int NC = (CH_HIST * 16 / 2 + 31) / 32;   // float4 copies per lane: 200 in all
      float4 t[NC];
#pragma unroll
      for (int i = 0; i < NC; i++) {
        const int q = 2 * (lane + 32 * i);
        if (q < CH_HIST * 16) t[i] = *(const float4*)(X + 512 + q);
      }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < NC; i++) {
        const int q = 2 * (lane + 32 * i);
        if (q < CH_HIST * 16) *(float4*)(X + q) = t[i];
      }
    }
    // ---- staging: 32 new frames = 512 samples, 8 pairs per lane --------------------------------------------------------------
    if (fast) {
      float4 t[8];
#pragma unroll
      for (int i = 0; i < 8; i++) t[i] = *(const float4*)(res + ((j0_32 + (unsigned)(boff + CH_HIST * 16 + 2 * lane + 64 * i)) & rmask));
      if (corr_all) {
        const int rel_b = seg_rel0 + boff + CH_HIST * 16;
        float2 v0[8], e[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const unsigned rel = (unsigned)(rel_b + 2 * lane + 64 * i);
          v0[i] = vrow[rel >> cr.seg_shift];
          e[i] = *(const float2*)(cr.e + cr.halo_out + (rel & smask));
        }
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const float ax = nalpha * v0[i].x, ay = nalpha * v0[i].y;
          t[i] = make_float4(fmaf(ax, e[i].x, t[i].x), fmaf(ay, e[i].x, t[i].y), fmaf(ax, e[i].y, t[i].z), fmaf(ay, e[i].y, t[i].w));
        }
      }
      const float c0 = pcs[1][0], s0 = psn[1][0], c1 = pcs[1][1], s1 = psn[1][1];
#pragma unroll
      for (int i = 0; i < 8; i++)
        *(float4*)(X + CH_HIST * 16 + 2 * lane + 64 * i) = make_float4(fmaf(t[i].x, c0, t[i].y * s0), fmaf(t[i].y, c0, -t[i].x * s0),
                                                                        fmaf(t[i].z, c1, t[i].w * s1), fmaf(t[i].w, c1, -t[i].z * s1));
    } else {
#pragma unroll 1
      for (int i = 0; i < 8; i++) stage_pair(CH_HIST * 16 + 2 * lane + 64 * i, boff, 1);
    }
    __syncwarp();
    if (batch < b_last) prefetch_l2(batch + 1);
    // ---- phase A: branch filters.  Frame kk of the batch sits in X frames kk .. kk + 25 (newest last) --------------------------
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
      const int kk0 = 16 * half + 8 * pass;
      const float2* xb = X + kk0 * 16 + (15 - br);
      float2 w[33];
#pragma unroll
      for (int q = 0; q < 33; q++) w[q] = xb[16 * q];
#pragma unroll
      for (int r = 0; r < 8; r++) {
        float2 acc = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int n = 0; n < 26; n++) acc = fma_tap(h[n], w[25 + r - n], acc);
        V[(kk0 + r) * CH_V_STRIDE + 15 - br] = acc;
      }
    }
    __syncwarp();
    fast_next = batch < b_last && (tile_steady || steady(batch + 1, ca_next));
    // ---- phase B + C: lane = frame kk = 32 batch + lane ------------------------------------------------------------------------
    {
      float2* const row = V + lane * CH_V_STRIDE;
      float2 v[16];
#pragma unroll
      for (int n = 0; n < 16; n++) v[n] = row[n];
      dft16p(v);
      // channel values back into the lane's own row (natural channel order): the next lane's "previous frame"
#pragma unroll
      for (int c = 0; c < 16; c++) row[c] = v[af_dig(c)];
      __syncwarp();
      const int kk = 32 * batch + lane;
      const bool own = kk >= own_lo && kk < own_hi;
      const float2* prow = row - CH_V_STRIDE;                    // lane 0: row -1, the previous batch's last frame
      float dm[16];
#pragma unroll
      for (int c = 0; c < 16; c += 2) {
        const float2 y0 = v[af_dig(c)], y1 = v[af_dig(c + 1)];
        const float2 p0 = prow[c], p1 = prow[c + 1];
        // arg(conj(prev) y) with separate mul / add like the C reference (A.9)
        const float re0 = __fadd_rn(__fmul_rn(p0.x, y0.x), __fmul_rn(p0.y, y0.y));
        const float im0 = __fsub_rn(__fmul_rn(p0.x, y0.y), __fmul_rn(p0.y, y0.x));
        const float re1 = __fadd_rn(__fmul_rn(p1.x, y1.x), __fmul_rn(p1.y, y1.y));
        const float im1 = __fsub_rn(__fmul_rn(p1.x, y1.y), __fmul_rn(p1.y, y1.x));
        const float2 a = fast_atan2f_x2(im0, re0, im1, re1);
        dm[c] = a.x * p.ref;
        dm[c + 1] = a.y * p.ref;
      }
      if (kk == k_zero) {   // absolute frame 0 (one lane, once per stream): r_prime = +0 + 0i exactly as the reference starts
#pragma unroll
        for (int c = 0; c < 16; c++) {
          const float2 y = v[af_dig(c)];
          const float re = __fadd_rn(__fmul_rn(0.0f, y.x), __fmul_rn(0.0f, y.y));
          const float im = __fsub_rn(__fmul_rn(0.0f, y.y), __fmul_rn(0.0f, y.x));
          dm[c] = fast_atan2f(im, re) * p.ref;
        }
      }
      if (own) {
        float* dptr = drow0 + ((fs32 + (unsigned)kk) & dmask);          // channel c lives demod_stride further per channel
#pragma unroll
        for (int c = 0; c < 16; c++) { *dptr = dm[c]; dptr += p.demod_stride; }
        if (crow0) {
          float2* cptr = crow0 + (crel + kk);
#pragma unroll
          for (int c = 0; c < 16; c++) { *cptr = v[af_dig(c)]; cptr += p.chan_ld; }
        }
        if constexpr (TAPS) {
#pragma unroll
          for (int c = 0; c < 16; c++) {
            const float2 y = v[af_dig(c)];
            ta.macc[c] += sqrt_approx(fmaf(y.x, y.x, y.y * y.y));   // MUFU.SQRT, 1 ulp: the RSSI is a mean of 12 500 of these, compared to 1e-3 dB
          }
          if ((kk == k_first || kk == k_last) && tp.edge) {   // one lane of one batch per call
            float2* e = tp.edge + (long long)s * 32;
#pragma unroll
            for (int c = 0; c < 16; c++) {
              if (kk == k_first) e[2 * c] = v[af_dig(c)];
              if (kk == k_last) e[2 * c + 1] = v[af_dig(c)];
            }
          }
        }
      }
      __syncwarp();   // every lane has read its previous frame
      if (lane < 16) V[-CH_V_STRIDE + lane] = V[31 * CH_V_STRIDE + lane];
    }
  }
  if constexpr (TAPS) {
    if (tp.mag_part) {
#pragma unroll
      for (int c = 0; c < 16; c++) {
        float m = ta.macc[c];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m += __shfl_xor_sync(0xffffffffu, m, o);
        if (lane == 0) tp.mag_part[((long long)s * p.tiles + tile_idx) * 16 + c] = m;
      }
    }
  }
}

// rssi[s][c] = 20 log10(sum over the tiles of mag_part / ns): average_power() of the reference for every channel
static __global__ void rssi_finalize_kernel(const float* mag_part, int tiles, int rows, long long ns, float* rssi) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;   // r = s * 16 + c
  if (r >= rows) return;
  const float* m = mag_part + (long long)(r >> 4) * tiles * 16 + (r & 15);
  float acc = 0.0f;
  for (int t = 0; t < tiles; t++) acc += m[(long long)t * 16];
  rssi[r] = 20.0f * log10f(acc / (float)ns);
}

}  // namespace pmr
