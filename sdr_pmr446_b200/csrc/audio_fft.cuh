// Shared pieces of the fast-convolution audio chain (audio_fft4_kernel, audio_fft4.cuh): its constants, its parameter
// block, the saturating s16 cast, and the radix-4 / radix-16 DFT helpers on (re, im) register pairs that the
// channelizer, the register DFTs (reg_dft.cuh) and the waterfall (spectrum_fast.cuh) reuse.
//
// The audio chain replaces the same reference lines as audio_kernel (/root/reference/src/sdr_pmr446.c:882-902:
// 377-tap CTCSS-removal FIR, gain, de-emphasis, optional 103-tap low-pass; SURVEY.md Appendix A.1, A.10, A.11) and the
// s16 cast of src/dsd_in.c:172-175.  The three filters in series are one LTI system whose impulse response is shorter
// than 512 samples (377 + 103 - 1 FIR taps followed by the de-emphasis pole 0.0146, below 1e-60 after 32 more
// samples).  Overlap-save with 4096-point transforms: forward FFT, multiply by the precomputed response H (which
// carries gain and 1/N), inverse FFT, keep the last 3584 samples.  ~70 flop per audio sample instead of the 759 of the
// direct form.
//
// FFT layout: 256 threads x 16 points in registers, three radix-16 passes (4096 = 16^3), data exchanged through
// shared memory between passes (conflict-free: 16-lane groups read consecutive or stride-17 elements); the inter-pass
// twiddles are powers of one table entry per thread and pass, built by a depth-4 product tree in registers.  The
// forward transform leaves X[k2 + 16 k1 + 256 k0] in register k0 of thread 16 k2 + k1; H is stored in that order and
// the inverse transform walks the same exchanges backwards, so no reordering pass exists.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "packed_f32.cuh"

namespace pmr {

// PMR audio float -> s16: (int16_t)(v * 32767) like src/dsd_in.c:172-175, but SATURATING.  The reference's PMR path hands
// float audio to RtAudio, where the device clips; with the default audio_gain = 4 a full-deviation signal reaches +-1.6,
// and a wrapping cast would flip its sign.  (dsd_in's own cast, dsd.cuh, stays the plain C cast for bit parity.)
#ifndef PMR_PCM_SAT_DEFINED
#define PMR_PCM_SAT_DEFINED
__device__ __forceinline__ short pcm_sat(float v) { return (short)__float2int_rz(fminf(fmaxf(v * 32767.0f, -32768.0f), 32767.0f)); }
#endif

constexpr int AF_N = 4096;
constexpr int AF_T = 256;
constexpr int AF_HALO = 512;              // overlap of the standard tile: >= length of the composite impulse response - 1
constexpr int AF_HALO_LONG = 1024;        // second instantiation for longer responses (FIR de-emphasis + low-pass: 579 taps)
constexpr int AF_SMEM = 16 * 272;         // float2 elements of the exchange buffer

struct AudioFftParams {
  const float* demod;        // ring [rows][demod_stride]
  long long demod_stride, demod_mask;
  int rows;                  // n_streams * num_channels
  int tiles;                 // tiles per group of four rows; tile k covers outputs [f0 + k own, f0 + (k + 1) own), own = AF_N - HALO
  long long tile0;           // unread, 0: keeps f0 / f1 at the parameter offsets audio_fft4_kernel was scheduled and timed with
  long long f0, f1;          // owned samples; samples >= f1 do not exist yet
  const float2* resp;        // [AF_N] response, element k0 * 256 + t = H[(t >> 4) + 16 (t & 15) + 256 k0] / N
  const float2* tw;          // [AF_N] exp(-2 pi i k / N)
  float* audio;              // optional [rows][out_ld], column = f - f0
  short* pcm;                // optional [rows][out_ld]
  long long out_ld;
};

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return fadd2(a, b); }   // one packed FADD2 (same rounding as two FADDs)
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return fsub2(a, b); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x)); }

// 4-point DFT in place: (a, b, c, d) -> (y0, y1, y2, y3); INV conjugates the kernel
template <bool INV>
__device__ __forceinline__ void dft4(float2& a, float2& b, float2& c, float2& d) {
  const float2 s0 = cadd(a, c), s1 = csub(a, c), s2 = cadd(b, d), s3 = csub(b, d);
  a = cadd(s0, s2);
  c = csub(s0, s2);
  if (!INV) {
    b = make_float2(s1.x + s3.y, s1.y - s3.x);
    d = make_float2(s1.x - s3.y, s1.y + s3.x);
  } else {
    b = make_float2(s1.x - s3.y, s1.y + s3.x);
    d = make_float2(s1.x + s3.y, s1.y - s3.x);
  }
}

// v *= W16^K (forward) or its conjugate (INV), K a compile-time constant
template <int K, bool INV>
__device__ __forceinline__ void rot16(float2& v) {
  constexpr float C1 = 0.92387953251128674f, S1 = 0.38268343236508977f, R = 0.70710678118654752f;
  constexpr int k = K & 15;
  // W16^k = (cos(pi k / 8), -sin(pi k / 8))
  constexpr float cs[16] = {1.0f, C1, R, S1, 0.0f, -S1, -R, -C1, -1.0f, -C1, -R, -S1, 0.0f, S1, R, C1};
  constexpr float sn[16] = {0.0f, S1, R, C1, 1.0f, C1, R, S1, 0.0f, -S1, -R, -C1, -1.0f, -C1, -R, -S1};
  if (k == 0) return;
  if (k == 4) { v = INV ? make_float2(-v.y, v.x) : make_float2(v.y, -v.x); return; }
  const float wr = cs[k], wi = INV ? sn[k] : -sn[k];
  v = make_float2(fmaf(v.x, wr, -v.y * wi), fmaf(v.x, wi, v.y * wr));
}

// register that holds output q of dft16
__host__ __device__ constexpr int af_dig(int q) { return 4 * (q & 3) + (q >> 2); }

// 16-point DFT of v[0..16) (natural order); output q ends in v[af_dig(q)]
template <bool INV>
__device__ __forceinline__ void dft16(float2* v) {
#pragma unroll
  for (int m0 = 0; m0 < 4; m0++) dft4<INV>(v[m0], v[m0 + 4], v[m0 + 8], v[m0 + 12]);
  rot16<1, INV>(v[5]);  rot16<2, INV>(v[9]);   rot16<3, INV>(v[13]);
  rot16<2, INV>(v[6]);  rot16<4, INV>(v[10]);  rot16<6, INV>(v[14]);
  rot16<3, INV>(v[7]);  rot16<6, INV>(v[11]);  rot16<9, INV>(v[15]);
#pragma unroll
  for (int q1 = 0; q1 < 4; q1++) dft4<INV>(v[4 * q1], v[4 * q1 + 1], v[4 * q1 + 2], v[4 * q1 + 3]);
}

// v[af_dig(k)] *= w^k (or conj(w)^k), k = 1..15, with the powers built by a depth-4 product tree: one table load per
// thread and pass instead of fifteen scattered ones (the table gathers saturated the L1 pipe)
template <bool CONJ>
__device__ __forceinline__ void twiddle_powers(float2* v, float2 w) {
  if (CONJ) w.y = -w.y;
  float2 pw[16];
  pw[1] = w;
  pw[2] = cmul(w, w);
  pw[3] = cmul(pw[2], w);
  pw[4] = cmul(pw[2], pw[2]);
  pw[5] = cmul(pw[4], w);
  pw[6] = cmul(pw[4], pw[2]);
  pw[7] = cmul(pw[4], pw[3]);
  pw[8] = cmul(pw[4], pw[4]);
#pragma unroll
  for (int k = 9; k < 16; k++) pw[k] = cmul(pw[8], pw[k - 8]);
#pragma unroll
  for (int k = 1; k < 16; k++) v[af_dig(k)] = cmul(v[af_dig(k)], pw[k]);
}

}  // namespace pmr
