// audio_fft4_kernel: the audio chain of every channel by fast convolution (method, transform layout and response table:
// audio_fft.cuh), FOUR channel rows per block, so that every floating-point instruction is a packed one.
//
// Two rows per block (one complex number row1 + i row2 per register pair, round 1's kernel) make complex additions one
// FADD2, but a multiplication by a twiddle needs the swapped pair and falls back to four scalar FMUL / FFMA, and the +-i
// rotations of the radix-4 butterflies to two scalar FADDs -- 47 % of its instructions were scalar FP32 and it was bound
// by issue slots (77 % busy at 60 % FMA pipe, profiles/ncu_r02v_audio_fft.md).  Here a register pair holds the SAME
// component of TWO sequences (A = row0 + i row1, B = row2 + i row3): C2 = {(re A, re B), (im A, im B)}.  Both sequences
// go through identical operations with identical twiddles, so a complex multiplication is four packed instructions for
// two products (twiddle components as scalar-broadcast operands), a rotation by +-i is a pair swap that costs nothing,
// and the index / predicate / barrier overhead of a tile is shared by four rows.
//
// Two more differences from round 1's kernel.  (1) The exchange buffer gives every k2 row 272 elements in BOTH layouts, so the rows a 16-thread group
// (k2 = t >> 4) reads and writes in the middle passes are its own: five of the seven block barriers are __syncwarp() and the
// eight warps of a block drift apart through the FP-heavy and the shared-memory-heavy phases instead of marching in step
// (the FMA pipe was 56 % busy with 1.3 warps waiting on it per issue: phases, not capacity).  (2) Tiles are counted from the
// call's first sample f0, not from the stream start: tile k yields outputs [f0 + k own, f0 + (k + 1) own), so a call of ns
// samples costs ceil(ns / own) transforms.  Chunking therefore changes the summation order of the fast convolution (1e-7 of
// the signal, DESIGN.md section 4), like it changes the DC blocker's segment grid.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "audio_fft.cuh"
#include "packed_f32.cuh"

namespace pmr {

struct C2 {
  float2 r, i;   // real parts (sequence A, sequence B), imaginary parts (A, B)
};

__device__ __forceinline__ float2 fmul2s(float2 a, float s) { return fmul2(a, make_float2(s, s)); }
__device__ __forceinline__ C2 c2add(const C2& a, const C2& b) { return C2{fadd2(a.r, b.r), fadd2(a.i, b.i)}; }
__device__ __forceinline__ C2 c2sub(const C2& a, const C2& b) { return C2{fsub2(a.r, b.r), fsub2(a.i, b.i)}; }
// a (wx + i wy) for both sequences
__device__ __forceinline__ C2 c2mul(const C2& a, float wx, float wy) {
  C2 d;
  d.r = fma_tap(-wy, a.i, fmul2s(a.r, wx));
  d.i = fma_tap(wx, a.i, fmul2s(a.r, wy));
  return d;
}

template <bool INV>
__device__ __forceinline__ void dft4_c2(C2& a, C2& b, C2& c, C2& d) {
  const C2 s0 = c2add(a, c), s1 = c2sub(a, c), s2 = c2add(b, d), s3 = c2sub(b, d);
  a = c2add(s0, s2);
  c = c2sub(s0, s2);
  if (!INV) {   // b = s1 - i s3, d = s1 + i s3
    b = C2{fadd2(s1.r, s3.i), fsub2(s1.i, s3.r)};
    d = C2{fsub2(s1.r, s3.i), fadd2(s1.i, s3.r)};
  } else {
    b = C2{fsub2(s1.r, s3.i), fadd2(s1.i, s3.r)};
    d = C2{fadd2(s1.r, s3.i), fsub2(s1.i, s3.r)};
  }
}

// v *= W16^K (forward) or its conjugate (INV)
template <int K, bool INV>
__device__ __forceinline__ void rot16_c2(C2& v) {
  constexpr float C1 = 0.92387953251128674f, S1 = 0.38268343236508977f, R = 0.70710678118654752f;
  constexpr int k = K & 15;
  constexpr float cs[16] = {1.0f, C1, R, S1, 0.0f, -S1, -R, -C1, -1.0f, -C1, -R, -S1, 0.0f, S1, R, C1};
  constexpr float sn[16] = {0.0f, S1, R, C1, 1.0f, C1, R, S1, 0.0f, -S1, -R, -C1, -1.0f, -C1, -R, -S1};
  if (k == 0) return;
  if (k == 4) {   // times -i (forward) / +i (inverse)
    const float2 r = v.r, i = v.i;
    if (!INV) { v.r = i; v.i = make_float2(-r.x, -r.y); }
    else { v.r = make_float2(-i.x, -i.y); v.i = r; }
    return;
  }
  v = c2mul(v, cs[k], INV ? sn[k] : -sn[k]);
}

template <bool INV>
__device__ __forceinline__ void dft16_c2(C2* v) {
#pragma unroll
  for (int m0 = 0; m0 < 4; m0++) dft4_c2<INV>(v[m0], v[m0 + 4], v[m0 + 8], v[m0 + 12]);
  rot16_c2<1, INV>(v[5]);  rot16_c2<2, INV>(v[9]);   rot16_c2<3, INV>(v[13]);
  rot16_c2<2, INV>(v[6]);  rot16_c2<4, INV>(v[10]);  rot16_c2<6, INV>(v[14]);
  rot16_c2<3, INV>(v[7]);  rot16_c2<6, INV>(v[11]);  rot16_c2<9, INV>(v[15]);
#pragma unroll
  for (int q1 = 0; q1 < 4; q1++) dft4_c2<INV>(v[4 * q1], v[4 * q1 + 1], v[4 * q1 + 2], v[4 * q1 + 3]);
}

// v[af_dig(k)] *= w^k (or conj(w)^k): the powers are one scalar product tree per thread, shared by both sequences
template <bool CONJ>
__device__ __forceinline__ void twiddle_powers_c2(C2* v, float2 w) {
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
  for (int k = 1; k < 16; k++) v[af_dig(k)] = c2mul(v[af_dig(k)], pw[k].x, pw[k].y);
}

constexpr int AF4_SMEM_BYTES = 2 * AF_SMEM * (int)sizeof(float2);

template <int HALO>
static __global__ void __launch_bounds__(AF_T, 2) audio_fft4_kernel(AudioFftParams p) {
  constexpr int AF_OWN = AF_N - HALO;
  extern __shared__ float2 af4_sm[];
  float2* const smr = af4_sm;
  float2* const smi = af4_sm + AF_SMEM;
  const int t = threadIdx.x;
  const int quad = blockIdx.x / p.tiles;
  const long long tile = blockIdx.x % p.tiles;                // counted from the call's first sample (anchored tiles)
  const int row0 = 4 * quad;
  const int nrow = p.rows - row0 < 4 ? p.rows - row0 : 4;   // rows that exist; the others compute on row0's samples, unused
  const long long o0 = p.f0 + tile * AF_OWN - HALO;         // absolute index of tile sample 0
  const float* d0 = p.demod + (long long)row0 * p.demod_stride;
  const float* d1 = p.demod + (long long)(nrow > 1 ? row0 + 1 : row0) * p.demod_stride;
  const float* d2 = p.demod + (long long)(nrow > 2 ? row0 + 2 : row0) * p.demod_stride;
  const float* d3 = p.demod + (long long)(nrow > 3 ? row0 + 3 : row0) * p.demod_stride;
  const long long lo64 = -o0, hi64 = p.f1 - o0;
  const int z0 = (int)(lo64 > (1 << 28) ? (1 << 28) : (lo64 < 0 ? 0 : lo64));           // first sample with n >= 0
  const int z1 = (int)(hi64 > (1 << 28) ? (1 << 28) : (hi64 < 0 ? 0 : hi64));           // one past the last existing one
  const unsigned base32 = (unsigned)o0, dmask = (unsigned)p.demod_mask;

  C2 x[16];
  // thread t holds tile samples t + 256 m
  if (z0 == 0 && z1 >= AF_N) {   // block-uniform: the whole tile exists
#pragma unroll
    for (int m = 0; m < 16; m++) {
      const unsigned idx = (base32 + (unsigned)(t + 256 * m)) & dmask;
      x[m].r = make_float2(d0[idx], d2[idx]);
      x[m].i = make_float2(d1[idx], d3[idx]);
    }
  } else {
#pragma unroll
    for (int m = 0; m < 16; m++) {
      const int i = t + 256 * m;
      x[m].r = x[m].i = make_float2(0.0f, 0.0f);
      if (i >= z0 && i < z1) {
        const unsigned idx = (base32 + (unsigned)i) & dmask;
        x[m].r = make_float2(d0[idx], d2[idx]);
        x[m].i = make_float2(d1[idx], d3[idx]);
      }
    }
  }
  const int hi4 = t >> 4, lo4 = t & 15;

  // ---- forward: over m (-> k2), twiddle W^(t k2) ----
  dft16_c2<false>(x);
  twiddle_powers_c2<false>(x, __ldg(p.tw + t));
#pragma unroll
  for (int k2 = 0; k2 < 16; k2++) { smr[k2 * 272 + t] = x[af_dig(k2)].r; smi[k2 * 272 + t] = x[af_dig(k2)].i; }
  __syncthreads();
  // thread (k2 = hi4, a = lo4): over b (-> k1), twiddle W^(16 a k1)
#pragma unroll
  for (int m = 0; m < 16; m++) { x[m].r = smr[hi4 * 272 + lo4 + 16 * m]; x[m].i = smi[hi4 * 272 + lo4 + 16 * m]; }
  dft16_c2<false>(x);
  twiddle_powers_c2<false>(x, __ldg(p.tw + 16 * lo4));
  __syncwarp();   // the exchange stays inside the 16-thread group (k2 = hi4), whose buffer rows no other warp touches here
#pragma unroll
  for (int k1 = 0; k1 < 16; k1++) { smr[hi4 * 272 + k1 * 17 + lo4] = x[af_dig(k1)].r; smi[hi4 * 272 + k1 * 17 + lo4] = x[af_dig(k1)].i; }
  __syncwarp();   // the exchange stays inside the 16-thread group (k2 = hi4), whose buffer rows no other warp touches here
  // thread (k2 = hi4, k1 = lo4): over a (-> k0)
#pragma unroll
  for (int a = 0; a < 16; a++) { x[a].r = smr[hi4 * 272 + lo4 * 17 + a]; x[a].i = smi[hi4 * 272 + lo4 * 17 + a]; }
  dft16_c2<false>(x);

  // ---- multiply by the response (includes 1/N and the audio gain); the result of bin k0 moves to register k0 ----
  {
    C2 y[16];
#pragma unroll
    for (int k0 = 0; k0 < 16; k0++) {
      const float2 h = __ldg(p.resp + k0 * 256 + t);
      y[k0] = c2mul(x[af_dig(k0)], h.x, h.y);
    }
#pragma unroll
    for (int k0 = 0; k0 < 16; k0++) x[k0] = y[k0];
  }

  // ---- inverse: over k0 (-> a), twiddle conj W^(a (16 k1 + k2)) ----
  dft16_c2<true>(x);
  twiddle_powers_c2<true>(x, __ldg(p.tw + 16 * lo4 + hi4));
  __syncwarp();   // the exchange stays inside the 16-thread group (k2 = hi4), whose buffer rows no other warp touches here
#pragma unroll
  for (int a = 0; a < 16; a++) { smr[hi4 * 272 + lo4 * 17 + a] = x[af_dig(a)].r; smi[hi4 * 272 + lo4 * 17 + a] = x[af_dig(a)].i; }
  __syncwarp();   // the exchange stays inside the 16-thread group (k2 = hi4), whose buffer rows no other warp touches here
  // thread (k2 = hi4, a = lo4): over k1 (-> b), twiddle conj W^(16 b k2)
#pragma unroll
  for (int k1 = 0; k1 < 16; k1++) { x[k1].r = smr[hi4 * 272 + k1 * 17 + lo4]; x[k1].i = smi[hi4 * 272 + k1 * 17 + lo4]; }
  dft16_c2<true>(x);
  twiddle_powers_c2<true>(x, __ldg(p.tw + 16 * hi4));
  __syncwarp();   // the exchange stays inside the 16-thread group (k2 = hi4), whose buffer rows no other warp touches here
#pragma unroll
  for (int b = 0; b < 16; b++) { smr[hi4 * 272 + lo4 + 16 * b] = x[af_dig(b)].r; smi[hi4 * 272 + lo4 + 16 * b] = x[af_dig(b)].i; }
  __syncthreads();
  // thread t: over k2 (-> m): tile samples t + 256 m
#pragma unroll
  for (int k2 = 0; k2 < 16; k2++) { x[k2].r = smr[k2 * 272 + t]; x[k2].i = smi[k2 * 272 + t]; }
  dft16_c2<true>(x);

  // ---- keep samples HALO.. of the tile that this call owns ----
  const long long own_hi = (p.f0 + (tile + 1) * AF_OWN < p.f1 ? p.f0 + (tile + 1) * AF_OWN : p.f1) - o0;
  const int s_lo = HALO, s_hi = (int)(own_hi > AF_N ? AF_N : (own_hi < 0 ? 0 : own_hi));
  const long long col0 = o0 - p.f0;   // column of tile sample 0
  const long long r0o = (long long)row0 * p.out_ld;
#pragma unroll
  for (int m = HALO / 256; m < 16; m++) {
    const int i = t + 256 * m;
    if (i >= s_lo && i < s_hi) {
      const C2 y = x[af_dig(m)];
      const long long at = r0o + col0 + i;
      const float yv[4] = {y.r.x, y.i.x, y.r.y, y.i.y};   // rows row0 .. row0 + 3
      if (p.audio) {
#pragma unroll
        for (int j = 0; j < 4; j++)
          if (j < nrow) p.audio[at + j * p.out_ld] = yv[j];
      }
      if (p.pcm) {
#pragma unroll
        for (int j = 0; j < 4; j++)
          if (j < nrow) p.pcm[at + j * p.out_ld] = pcm_sat(yv[j]);
      }
    }
  }
}

}  // namespace pmr
