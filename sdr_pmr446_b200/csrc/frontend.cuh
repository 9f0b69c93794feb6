// Front-end kernels: cu8/cf32/cs16/cs8 load -> DC blocker -> half-band decimator cascade -> arbitrary
// resampler.  Replaces iirfilt_crcf_execute_block + msresamp_crcf_execute of the reference
// (/root/reference/src/sdr_pmr446.c:795-796, /root/reference/src/dsd_in.c:167-168; algorithm:
// SURVEY.md Appendix A.1-A.5).
//
// B200 design ("segment-sequential"): every thread owns one time segment of one stream and
// runs the cascade over it sample-group by sample-group with all filter windows in registers,
// exactly like the CPU does for a whole stream -- but ~10^5-10^6 segments run concurrently.
// A segment starts H samples early (zero state) so that its owned outputs only depend on real
// samples (the cascade is FIR).  Taps are compile-time-indexed constant-bank operands of the
// FFMAs; no shared memory is used.  Lanes of a warp read 32-byte (cu8) / 64-128-byte (cf32)
// pieces of different segments, i.e. whole DRAM sectors, and the next group's raw data is
// fetched into registers one iteration ahead so the load latency hides behind ~400 FFMAs.
// All per-iteration index arithmetic is 32-bit and relative to the segment start.
//
// The one IIR element, the DC blocker v[n] = x[n] + c v[n-1], y = v[n] - v[n-1], is linear, so
// a segment's output is (zero-state response to its own samples) + (zero-input response to the
// state V0 at its warm-up start).  DC_ZSR mode computes the zero-state part with no dependence
// on other segments and records the segment's local sum; dc_scan_kernel chains the sums into
// V0 per segment; the zero-input part, -alpha V0 E[k] with E = (cascade applied to c^i) a fixed
// table that is exactly geometric past the warm-up, is added by the NEXT launch while it loads
// the ring (Correction).  DC_SCAN mode (used when there is no next launch) gets V0 up front from
// dc_local_kernel + dc_scan_kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "packed_f32.cuh"

namespace pmr {

enum { SRC_CU8 = 0, SRC_CF32 = 1, SRC_RING = 2, SRC_CS16 = 3, SRC_CS8 = 4 };
enum { DC_NONE = 0, DC_SCAN = 1, DC_ZSR = 2 };

// Zero-input-response correction applied while loading a ring written by a DC_ZSR launch.
struct Correction {
  const float2* v_seg;   // [n_streams][nseg] V0 of the producer's segments; nullptr = off
  const float* e;        // [(halo + seg_len) / D] response of the producer's cascade to c^i
  long long from;        // ring samples with index >= from still need the correction
  long long seg0_out;    // producer's seg0 / D (ring index of segment 0's first owned output)
  int seg_shift;         // log2(producer seg_len / D)
  int halo_out;          // producer halo / D
  int nseg;
  float alpha;
  float rho_pow[16];     // (c^D)^i: E[k + i] = E[k] rho^i for k >= halo_out
};

// Per-launch view of the input signal of all streams.
//  two-source (SRC_CU8 / SRC_CF32 / SRC_CS16 / SRC_CS8): samples [hist_base, n0) live in `hist`, [n0, n1) in `cur`.
//  ring (SRC_RING): sample n lives at cur[n & ring_mask]; samples with n < 0 read as zero.
struct SrcView {
  const void* hist;
  const void* cur;
  long long hist_stride;  // bytes between streams
  long long cur_stride;   // bytes between streams
  long long hist_base;    // absolute index of hist[0]; multiple of 16
  long long n0, n1;       // new samples are [n0, n1)
  long long ring_mask;
  int cur_aligned;        // n0 % 16 == 0 and cur/cur_stride 16-byte aligned (two-source only)
  Correction corr;
};

struct CascadeParams {
  SrcView src;
  int n_streams;
  int nseg;               // segments per stream
  long long seg0;         // absolute start of segment 0 (multiple of the group size)
  int seg_len;            // input samples per segment (multiple of group size and of D)
  int halo;               // warm-up samples before a segment (multiple of the group size)
  long long out0, out1;   // owned half-band outputs [out0, out1)
  float scale;            // 2^-NST, folded into the last stage's outputs
  // DC blocker
  float alpha;
  const float2* v_seg;    // DC_SCAN: [n_streams][nseg] V at (segment start - halo)
  float2* sums;           // DC_ZSR: [n_streams][nseg] local sums out
  long long dc_end;       // DC_ZSR: sums stop at this absolute index (next chunk's P_0)
  // arbitrary resampler
  unsigned step;
  int bits;
  const float* pfb;       // [npfb][16] rows padded to 16 floats
  // destination ring (cf32)
  float2* dst;
  long long dst_stride;   // float2 elements between streams
  long long dst_mask;
  // half-band taps of the (up to 4) stages of this launch: [stage][j], j < 2m, newest first.
  // Kernel parameters live in constant bank 0, so these become c[0x0][imm] FFMA operands.
  float hb[4][20];
};

// A group of G raw samples held in registers between fetch (issue the loads) and convert.
template <int SRC, int G>
struct Raw;
template <int G>
struct Raw<SRC_CU8, G> { unsigned w[G / 2]; };   // 2 bytes per sample
template <int G>
struct Raw<SRC_CF32, G> { unsigned w[2 * G]; };  // 8 bytes per sample
template <int G>
struct Raw<SRC_RING, G> { unsigned w[2 * G]; };
template <int G>
struct Raw<SRC_CS16, G> { unsigned w[G]; };      // 4 bytes per sample
template <int G>
struct Raw<SRC_CS8, G> { unsigned w[G / 2]; };   // 2 bytes per sample

// 256-bit global accesses (LDG/STG.E.ENL2.256 on sm_100): a lane's 32-byte piece is one DRAM sector and,
// with every lane on a different cache line, costs one L1 wavefront instead of two 128-bit ones.
__device__ __forceinline__ void ldg256_stream(const void* p, unsigned* w) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "l"(p));
}
__device__ __forceinline__ void ldg256(const void* p, unsigned* w) {
  asm volatile("ld.global.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "l"(p) : "memory");
}
__device__ __forceinline__ void stg256(void* p, const float* f) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" :: "l"(p), "f"(f[0]), "f"(f[1]), "f"(f[2]), "f"(f[3]), "f"(f[4]), "f"(f[5]),
               "f"(f[6]), "f"(f[7]) : "memory");
}

// Per-thread loader state: `fast` means every group of the thread's range can be read with aligned
// vector loads from one place, so fetch() is a pointer bump; otherwise each sample is guarded.
template <int SRC>
struct Loader;

// byte k of w as a float, exactly: one PRMT drops the byte into the mantissa of 2^23 (0x4B000000), one FADD removes
// the 2^23 -- both on the ALU/FMA pipes instead of the quarter-rate I2F conversion unit
__device__ __forceinline__ float u8f(unsigned w, int k) {
  return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540u + (unsigned)k)) - 8388608.0f;
}

// Iterations [lo, hi) of a thread whose groups of G samples start at qb that lie wholly inside the current chunk
// [n0, n1) and can therefore be read with aligned vector loads (none unless the chunk is aligned, see SrcView).
template <int G>
__device__ __forceinline__ void fast_iters(const SrcView& v, long long qb, int* lo_out, int* hi_out) {
  *lo_out = *hi_out = 0;
  if (v.cur_aligned) {
    const long long lo = (v.n0 - qb + G - 1) / G, hi = (v.n1 - qb) / G;
    *lo_out = (int)(lo < 0 ? 0 : (lo > (1 << 30) ? (1 << 30) : lo));
    *hi_out = (int)(hi < 0 ? 0 : (hi > (1 << 30) ? (1 << 30) : hi));
  }
}

// ---- cu8 two-source --------------------------------------------------------------------
template <>
struct Loader<SRC_CU8> {
  const uint8_t* hist;
  const uint8_t* cur;
  const uint8_t* fp;
  int fast_lo, fast_hi;   // iterations [fast_lo, fast_hi) read whole aligned groups of the current chunk
  template <int G>
  __device__ __forceinline__ void init(const SrcView& v, int s, long long qb) {
    hist = (const uint8_t*)v.hist + (long long)s * v.hist_stride;
    cur = (const uint8_t*)v.cur + (long long)s * v.cur_stride;
    fast_iters<G>(v, qb, &fast_lo, &fast_hi);
    fp = cur + 2 * (qb - v.n0);
  }
  template <int G>
  __device__ __forceinline__ void fetch(int it, Raw<SRC_CU8, G>& r) const {
    static_assert(G % 16 == 0, "cu8 groups are loaded 32 bytes at a time");
    if (it >= fast_lo && it < fast_hi) {
#pragma unroll
      for (int i = 0; i < G / 16; i++) ldg256_stream(fp + (size_t)it * (2 * G) + 32 * i, r.w + 8 * i);
    }
  }
  // converts with the SoapyRTLSDR rule (u8 - 127.4)/128 (SURVEY.md 8a row a0)
  template <int G>
  __device__ __forceinline__ void convert(const SrcView& v, long long q, int it, const Raw<SRC_CU8, G>& r, float* xr, float* xi) const {
    const float k = 1.0f / 128.0f, c0 = -127.4f / 128.0f;
    if (it >= fast_lo && it < fast_hi) {
#pragma unroll
      for (int j = 0; j < G / 2; j++) {   // one 32-bit word = two samples
        xr[2 * j] = fmaf(u8f(r.w[j], 0), k, c0);
        xi[2 * j] = fmaf(u8f(r.w[j], 1), k, c0);
        xr[2 * j + 1] = fmaf(u8f(r.w[j], 2), k, c0);
        xi[2 * j + 1] = fmaf(u8f(r.w[j], 3), k, c0);
      }
    } else {
#pragma unroll
      for (int i = 0; i < G; i++) {  // static indices keep xr/xi in registers
        const long long n = q + i;
        float re = 0.0f, im = 0.0f;
        if (n >= 0 && n < v.n1 && (n >= v.n0 || n >= v.hist_base)) {
          const uint8_t* b = (n >= v.n0) ? cur + 2 * (n - v.n0) : hist + 2 * (n - v.hist_base);
          re = fmaf((float)b[0], k, c0);
          im = fmaf((float)b[1], k, c0);
        }
        xr[i] = re;
        xi[i] = im;
      }
    }
  }
};

// ---- cf32 two-source -------------------------------------------------------------------
template <>
struct Loader<SRC_CF32> {
  const float2* hist;
  const float2* cur;
  const float2* fp;
  int fast_lo, fast_hi;
  template <int G>
  __device__ __forceinline__ void init(const SrcView& v, int s, long long qb) {
    hist = (const float2*)((const char*)v.hist + (long long)s * v.hist_stride);
    cur = (const float2*)((const char*)v.cur + (long long)s * v.cur_stride);
    fast_iters<G>(v, qb, &fast_lo, &fast_hi);
    fp = cur + (qb - v.n0);
  }
  template <int G>
  __device__ __forceinline__ void fetch(int it, Raw<SRC_CF32, G>& r) const {
    if (it >= fast_lo && it < fast_hi) {
#pragma unroll
      for (int i = 0; i < G / 4; i++) ldg256_stream(fp + (size_t)it * G + 4 * i, r.w + 8 * i);
    }
  }
  template <int G>
  __device__ __forceinline__ void convert(const SrcView& v, long long q, int it, const Raw<SRC_CF32, G>& r, float* xr, float* xi) const {
    if (it >= fast_lo && it < fast_hi) {
#pragma unroll
      for (int i = 0; i < G; i++) { xr[i] = __uint_as_float(r.w[2 * i]); xi[i] = __uint_as_float(r.w[2 * i + 1]); }
    } else {
#pragma unroll
      for (int i = 0; i < G; i++) {
        const long long n = q + i;
        float2 w = make_float2(0.0f, 0.0f);
        if (n >= 0 && n < v.n1) {
          if (n >= v.n0) w = cur[n - v.n0];
          else if (n >= v.hist_base) w = hist[n - v.hist_base];
        }
        xr[i] = w.x;
        xi[i] = w.y;
      }
    }
  }
};

// ---- cs16 / cs8 two-source ---------------------------------------------------------------
// x 2^-15 (cs16) and x 2^-7 (cs8) exactly, without the I2F unit: x with its sign bit flipped is the unsigned x + 2^15
// (x + 2^7); dropped into the mantissa of 2^23 it reads as 2^23 + 2^15 + x, and one FFMA by the power of two with the
// scaled bias as addend leaves x 2^-15 (the product is exact, and so is the sum: it is representable).
// s16f: half h (0 = I, the low half; 1 = Q) of a cs16 word.  s8f: byte k of a cs8 word already XORed with 0x80808080.
__device__ __forceinline__ float s16f(unsigned w, int h) {
  return fmaf(__uint_as_float((h ? (w >> 16) : (w & 0xFFFFu)) ^ 0x4B008000u), 0x1p-15f, -257.0f);
}
__device__ __forceinline__ float s8f(unsigned wb, int k) {
  return fmaf(__uint_as_float(__byte_perm(wb, 0x4B000000u, 0x7540u + (unsigned)k)), 0x1p-7f, -65537.0f);
}

template <>
struct Loader<SRC_CS16> {
  const unsigned* hist;   // one 32-bit word per sample: I in the low half, Q in the high half
  const unsigned* cur;
  const unsigned* fp;
  int fast_lo, fast_hi;
  template <int G>
  __device__ __forceinline__ void init(const SrcView& v, int s, long long qb) {
    hist = (const unsigned*)((const char*)v.hist + (long long)s * v.hist_stride);
    cur = (const unsigned*)((const char*)v.cur + (long long)s * v.cur_stride);
    fast_iters<G>(v, qb, &fast_lo, &fast_hi);
    fp = cur + (qb - v.n0);
  }
  template <int G>
  __device__ __forceinline__ void fetch(int it, Raw<SRC_CS16, G>& r) const {
    static_assert(G % 8 == 0, "cs16 groups are loaded 32 bytes at a time");
    if (it >= fast_lo && it < fast_hi) {
#pragma unroll
      for (int i = 0; i < G / 8; i++) ldg256_stream(fp + (size_t)it * G + 8 * i, r.w + 8 * i);
    }
  }
  template <int G>
  __device__ __forceinline__ void convert(const SrcView& v, long long q, int it, const Raw<SRC_CS16, G>& r, float* xr, float* xi) const {
    if (it >= fast_lo && it < fast_hi) {
#pragma unroll
      for (int i = 0; i < G; i++) { xr[i] = s16f(r.w[i], 0); xi[i] = s16f(r.w[i], 1); }
    } else {
#pragma unroll
      for (int i = 0; i < G; i++) {
        const long long n = q + i;
        float re = 0.0f, im = 0.0f;
        if (n >= 0 && n < v.n1 && (n >= v.n0 || n >= v.hist_base)) {
          const unsigned w = (n >= v.n0) ? cur[n - v.n0] : hist[n - v.hist_base];
          re = s16f(w, 0);
          im = s16f(w, 1);
        }
        xr[i] = re;
        xi[i] = im;
      }
    }
  }
};

template <>
struct Loader<SRC_CS8> {
  const uint8_t* hist;
  const uint8_t* cur;
  const uint8_t* fp;
  int fast_lo, fast_hi;
  template <int G>
  __device__ __forceinline__ void init(const SrcView& v, int s, long long qb) {
    hist = (const uint8_t*)v.hist + (long long)s * v.hist_stride;
    cur = (const uint8_t*)v.cur + (long long)s * v.cur_stride;
    fast_iters<G>(v, qb, &fast_lo, &fast_hi);
    fp = cur + 2 * (qb - v.n0);
  }
  template <int G>
  __device__ __forceinline__ void fetch(int it, Raw<SRC_CS8, G>& r) const {
    static_assert(G % 16 == 0, "cs8 groups are loaded 32 bytes at a time");
    if (it >= fast_lo && it < fast_hi) {
#pragma unroll
      for (int i = 0; i < G / 16; i++) ldg256_stream(fp + (size_t)it * (2 * G) + 32 * i, r.w + 8 * i);
    }
  }
  template <int G>
  __device__ __forceinline__ void convert(const SrcView& v, long long q, int it, const Raw<SRC_CS8, G>& r, float* xr, float* xi) const {
    if (it >= fast_lo && it < fast_hi) {
#pragma unroll
      for (int j = 0; j < G / 2; j++) {   // one 32-bit word = two samples
        const unsigned wb = r.w[j] ^ 0x80808080u;
        xr[2 * j] = s8f(wb, 0);
        xi[2 * j] = s8f(wb, 1);
        xr[2 * j + 1] = s8f(wb, 2);
        xi[2 * j + 1] = s8f(wb, 3);
      }
    } else {
#pragma unroll
      for (int i = 0; i < G; i++) {
        const long long n = q + i;
        float re = 0.0f, im = 0.0f;
        if (n >= 0 && n < v.n1 && (n >= v.n0 || n >= v.hist_base)) {
          const uint8_t* b = (n >= v.n0) ? cur + 2 * (n - v.n0) : hist + 2 * (n - v.hist_base);
          const unsigned wb = ((unsigned)b[0] | ((unsigned)b[1] << 8)) ^ 0x8080u;
          re = s8f(wb, 0);
          im = s8f(wb, 1);
        }
        xr[i] = re;
        xi[i] = im;
      }
    }
  }
};

// ---- cf32 ring (library-owned intermediate), with the optional zero-input-response correction ----
template <>
struct Loader<SRC_RING> {
  const float2* ring;
  unsigned q32, mask32;
  int fast_hi;            // iterations [0, fast_hi) read whole groups below n1
  // correction state
  const float2* vrow;     // producer V0 row of this stream, nullptr = off
  int relc, from_rel;     // (q_begin - seg0_out), (from - seg0_out)
  template <int G>
  __device__ __forceinline__ void init(const SrcView& v, int s, long long qb) {
    ring = (const float2*)((const char*)v.cur + (long long)s * v.cur_stride);
    q32 = (unsigned)qb;
    mask32 = (unsigned)v.ring_mask;
    const long long hi = qb >= 0 ? (v.n1 - qb) / G : 0;
    fast_hi = (int)(hi < 0 ? 0 : (hi > (1 << 30) ? (1 << 30) : hi));
    vrow = v.corr.v_seg ? v.corr.v_seg + (long long)s * v.corr.nseg : nullptr;
    const long long r = qb - v.corr.seg0_out, f = v.corr.from - v.corr.seg0_out;
    relc = (int)(r < -(1 << 30) ? -(1 << 30) : r);
    from_rel = (int)(f > (1 << 30) ? (1 << 30) : f);
  }
  template <int G>
  __device__ __forceinline__ void fetch(int it, Raw<SRC_RING, G>& r) const {
    if (it < fast_hi) {
      const float2* p = ring + ((q32 + (unsigned)(it * G)) & mask32);
#pragma unroll
      for (int i = 0; i < G / 4; i++) ldg256(p + 4 * i, r.w + 8 * i);
    }
  }
  template <int G>
  __device__ __forceinline__ void convert(const SrcView& v, long long q, int it, const Raw<SRC_RING, G>& r, float* xr, float* xi) const {
    if (it < fast_hi) {
#pragma unroll
      for (int i = 0; i < G; i++) { xr[i] = __uint_as_float(r.w[2 * i]); xi[i] = __uint_as_float(r.w[2 * i + 1]); }
    } else {
#pragma unroll
      for (int i = 0; i < G; i++) {
        const long long n = q + i;
        float2 w = make_float2(0.0f, 0.0f);
        if (n >= 0 && n < v.n1) w = ring[(unsigned)n & mask32];
        xr[i] = w.x;
        xi[i] = w.y;
      }
    }
    // zero-input response of the producer's DC blocker: x -= alpha V0[seg] E[k].  The producer's
    // segment grid is aligned to 16 ring samples, so a group never straddles two segments, and
    // E[k0 + i] = E[k0] rho^i because every corrected sample lies past the producer's warm-up.
    if (vrow) {
      const int rel = relc + it * G;
      if (rel + G > from_rel && rel >= 0) {
        const Correction& c = v.corr;
        const int t = rel >> c.seg_shift;
        if (t < c.nseg) {
          const float2 v0 = vrow[t];
          const float e0 = __ldg(c.e + (rel - (t << c.seg_shift)) + c.halo_out);
          const float ar = -c.alpha * v0.x * e0, ai = -c.alpha * v0.y * e0;
#pragma unroll
          for (int i = 0; i < G; i++) {
            if (rel + i >= from_rel) {
              xr[i] = fmaf(ar, c.rho_pow[i], xr[i]);
              xi[i] = fmaf(ai, c.rho_pow[i], xi[i]);
            }
          }
        }
      }
    }
  }
};

// ---- one half-band decimator stage held in registers (A.4) ------------------------------
//   out[o] = x_odd[o - M] + sum_{j<2M} h[j] * x_even[o - j]
// processes B input pairs per call; STAGE selects the row of CascadeParams::hb.  Samples are (re, im) register pairs and
// every tap is one packed FFMA2 with the tap as a scalar constant-bank / uniform-register operand (packed_f32.cuh).
template <int M, int B, int STAGE>
struct HbStage {
  float2 he[2 * M - 1];  // previous even samples, oldest first
  float2 ho[M];          // previous odd samples, oldest first
  __device__ __forceinline__ void reset() {
#pragma unroll
    for (int i = 0; i < 2 * M - 1; i++) he[i] = make_float2(0.0f, 0.0f);
#pragma unroll
    for (int i = 0; i < M; i++) ho[i] = make_float2(0.0f, 0.0f);
  }
  template <bool SCALE>
  __device__ __forceinline__ void run(const CascadeParams& p, const float2* x, float2* y, float scale) {
    float2 e[2 * M - 1 + B], o[M + B];
#pragma unroll
    for (int i = 0; i < 2 * M - 1; i++) e[i] = he[i];
#pragma unroll
    for (int i = 0; i < M; i++) o[i] = ho[i];
#pragma unroll
    for (int b = 0; b < B; b++) { e[2 * M - 1 + b] = x[2 * b]; o[M + b] = x[2 * b + 1]; }
#pragma unroll
    for (int b = 0; b < B; b++) {
      float2 acc = o[b];
#pragma unroll
      for (int j = 0; j < 2 * M; j++) acc = fma_tap(p.hb[STAGE][j], e[2 * M - 1 + b - j], acc);
      y[b] = SCALE ? fmul2(acc, make_float2(scale, scale)) : acc;
    }
#pragma unroll
    for (int i = 0; i < 2 * M - 1; i++) he[i] = e[B + i];
#pragma unroll
    for (int i = 0; i < M; i++) ho[i] = o[B + i];
  }
};
template <int B, int STAGE>
struct HbStage<0, B, STAGE> {  // absent stage
  __device__ __forceinline__ void reset() {}
};

// ---- DC blocker local sums: S_t = sum_j c^(len-1-j) x[P_t + j] over segment t (A.1) -------
// (only used in DC_SCAN mode, i.e. single-launch plans)
struct DcLocalParams {
  SrcView src;
  int n_streams, nseg;
  long long p0;       // P_0 = seg0 - halo
  int seg_len;
  long long end;      // sums stop at `end` (next chunk's P_0)
  float c;            // 1 - alpha
  float2* sums;       // [n_streams][nseg]
};

template <int SRC>
__global__ void __launch_bounds__(128) dc_local_kernel(DcLocalParams p) {
  long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)p.n_streams * p.nseg) return;
  int s = (int)(gid / p.nseg), t = (int)(gid % p.nseg);
  long long a = p.p0 + (long long)t * p.seg_len;
  long long b = a + p.seg_len;
  if (b > p.end) b = p.end;
  float sr = 0.0f, si = 0.0f;
  if (a < 0) a = 0;  // P_0 and seg_len are multiples of 16, so a stays group-aligned
  Loader<SRC> ld;
  ld.template init<16>(p.src, s, a);
  int it = 0;
  for (long long q = a; q < b; q += 16, it++) {
    float xr[16], xi[16];
    Raw<SRC, 16> raw;
    ld.template fetch<16>(it, raw);
    ld.template convert<16>(p.src, q, it, raw, xr, xi);
#pragma unroll
    for (int i = 0; i < 16; i++)
      if (q + i < b) { sr = fmaf(p.c, sr, xr[i]); si = fmaf(p.c, si, xi[i]); }
  }
  p.sums[gid] = make_float2(sr, si);
}

struct DcScanParams {
  // The fused cu8 front end runs its recurrence on X = u8 - 127 (exact integers) instead of x = X / 128 + c0' (see
  // cu8_pair_x): sums / v_lag are then in X units and the consumers' V0 is unit_scale * V_X.  Every other plan: 1.
  float unit_scale;
  int n_streams, nseg;
  const float2* sums;
  float2* v_seg;      // out: V at each segment's warm-up start
  float2* v_lag;      // in/out: V at P_0 of this chunk -> V at `end`
  long long p0, end;
  int seg_len;
  float c, decay_full;  // 1 - alpha and c^seg_len
};
// one warp per stream: lanes take 32 consecutive segments, a shuffle scan composes the affine maps
// V -> d V + s (d = c^len), the carry moves to the next 32 segments.
static __global__ void __launch_bounds__(128) dc_scan_kernel(DcScanParams p) {
  const int s = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (s >= p.n_streams) return;
  float2 carry = p.v_lag[s];
  for (int base = 0; base < p.nseg; base += 32) {
    const int t = base + lane;
    float d = 1.0f;
    float2 sm = make_float2(0.0f, 0.0f);
    if (t < p.nseg) {
      long long a = p.p0 + (long long)t * p.seg_len, b = a + p.seg_len;
      if (b > p.end) b = p.end;
      if (a < 0) a = 0;
      const long long len = b - a;
      if (len > 0) {
        d = (len == p.seg_len) ? p.decay_full : powf(p.c, (float)len);
        sm = p.sums[(long long)s * p.nseg + t];
      }
    }
    // inclusive scan of (d, sm): (d2, s2) o (d1, s1) = (d1 d2, d2 s1 + s2)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float dp = __shfl_up_sync(0xffffffffu, d, o);
      const float sx = __shfl_up_sync(0xffffffffu, sm.x, o), sy = __shfl_up_sync(0xffffffffu, sm.y, o);
      if (lane >= o) {
        sm.x = fmaf(d, sx, sm.x);
        sm.y = fmaf(d, sy, sm.y);
        d *= dp;
      }
    }
    // V after segment t = d * carry + sm ; V before segment t = that of lane - 1 (or the carry)
    float2 after = make_float2(fmaf(d, carry.x, sm.x), fmaf(d, carry.y, sm.y));
    float bx = __shfl_up_sync(0xffffffffu, after.x, 1), by = __shfl_up_sync(0xffffffffu, after.y, 1);
    if (lane == 0) { bx = carry.x; by = carry.y; }
    if (t < p.nseg) p.v_seg[(long long)s * p.nseg + t] = make_float2(p.unit_scale * bx, p.unit_scale * by);
    carry.x = __shfl_sync(0xffffffffu, after.x, 31);
    carry.y = __shfl_sync(0xffffffffu, after.y, 31);
  }
  if (lane == 0) p.v_lag[s] = carry;
}

// The same scan with one BLOCK of 256 threads per stream (256 segments per pass): for a few streams with thousands of
// segments each (the wideband configuration: 4 streams x 7800 segments) the warp version above is a long serial loop.
static __global__ void __launch_bounds__(256) dc_scan_block_kernel(DcScanParams p) {
  __shared__ float wd[8], wsx[8], wsy[8];
  __shared__ float2 s_carry;
  const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = p.v_lag[s];
  __syncthreads();
  for (int base = 0; base < p.nseg; base += 256) {
    const float2 carry = s_carry;
    const int t = base + threadIdx.x;
    float d = 1.0f;
    float2 sm = make_float2(0.0f, 0.0f);
    if (t < p.nseg) {
      long long a = p.p0 + (long long)t * p.seg_len, b = a + p.seg_len;
      if (b > p.end) b = p.end;
      if (a < 0) a = 0;
      const long long len = b - a;
      if (len > 0) {
        d = (len == p.seg_len) ? p.decay_full : powf(p.c, (float)len);
        sm = p.sums[(long long)s * p.nseg + t];
      }
    }
    // inclusive scan of the affine maps V -> d V + s inside the warp: (d2, s2) o (d1, s1) = (d1 d2, d2 s1 + s2)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float dp = __shfl_up_sync(0xffffffffu, d, o);
      const float sx = __shfl_up_sync(0xffffffffu, sm.x, o), sy = __shfl_up_sync(0xffffffffu, sm.y, o);
      if (lane >= o) {
        sm.x = fmaf(d, sx, sm.x);
        sm.y = fmaf(d, sy, sm.y);
        d *= dp;
      }
    }
    if (lane == 31) { wd[warp] = d; wsx[warp] = sm.x; wsy[warp] = sm.y; }
    __syncthreads();
    // the maps of the preceding warps, composed in order, applied to the carry: V before this warp's first segment
    float2 vin = carry;
    for (int w = 0; w < warp; w++) vin = make_float2(fmaf(wd[w], vin.x, wsx[w]), fmaf(wd[w], vin.y, wsy[w]));
    const float2 after = make_float2(fmaf(d, vin.x, sm.x), fmaf(d, vin.y, sm.y));
    float bx = __shfl_up_sync(0xffffffffu, after.x, 1), by = __shfl_up_sync(0xffffffffu, after.y, 1);
    if (lane == 0) { bx = vin.x; by = vin.y; }
    if (t < p.nseg) p.v_seg[(long long)s * p.nseg + t] = make_float2(p.unit_scale * bx, p.unit_scale * by);
    __syncthreads();
    if (threadIdx.x == 255) s_carry = after;
    __syncthreads();
  }
  if (threadIdx.x == 0) p.v_lag[s] = s_carry;
}

// in-place zero-input-response correction of the last `count` samples of a ring (they are the
// next chunk's history, which the next launch reads as already corrected)
static __global__ void zir_tail_kernel(float2* ring, long long ring_stride, long long ring_mask, Correction c, long long start, int count) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  const int s = blockIdx.y;
  const long long n = start + k;
  if (n < c.from) return;
  const long long rel = n - c.seg0_out;
  if (rel < 0) return;
  const int t = (int)(rel >> c.seg_shift);
  if (t >= c.nseg) return;
  const float2 v0 = c.v_seg[(long long)s * c.nseg + t];
  const float e = c.e[(int)(rel - ((long long)t << c.seg_shift)) + c.halo_out];
  float2* p = ring + (long long)s * ring_stride + (n & ring_mask);
  float2 x = *p;
  x.x = fmaf(-c.alpha * v0.x, e, x.x);
  x.y = fmaf(-c.alpha * v0.y, e, x.y);
  *p = x;
}

// ---- the cascade kernel ----------------------------------------------------------------------
// Stage list MA,MB,MC,MD = semi-lengths in execution order (highest rate first), 0 = absent.
// G = input samples per loop iteration (multiple of 2^NST).
template <int SRC, int DC, int G, int MA, int MB, int MC, int MD, bool ARB>
__global__ void __launch_bounds__(128, 3) cascade_kernel(CascadeParams p) {
  constexpr int NST = (MA > 0) + (MB > 0) + (MC > 0) + (MD > 0);
  constexpr int D = 1 << NST;
  constexpr int NO = G / D;  // outputs per iteration
  // The lanes of a warp sit at different resampler phases unless the plan is periodic, so every output reads a
  // different row of the filter bank: from global memory that is one L1 wavefront per lane and load.  A copy in
  // shared memory with rows 20 floats apart (16-byte aligned, 8 bank groups) serves a quarter-warp per wavefront.
  constexpr int BANK_STRIDE = 20;
  __shared__ __align__(16) float sbank[ARB ? 256 * BANK_STRIDE : 4];
  if (ARB) {
    const int rows = 1 << p.bits;   // <= 256 (checked by the host)
    for (int i = threadIdx.x; i < rows * 16; i += blockDim.x) sbank[(i >> 4) * BANK_STRIDE + (i & 15)] = __ldg(p.pfb + i);
    __syncthreads();
  }
  long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)p.n_streams * p.nseg) return;
  const int s = (int)(gid / p.nseg), t = (int)(gid % p.nseg);
  const long long T0 = p.seg0 + (long long)t * p.seg_len;
  long long i_lo = T0 / D, i_hi = (T0 + p.seg_len) / D;
  if (i_lo < p.out0) i_lo = p.out0;
  if (i_hi > p.out1) i_hi = p.out1;
  long long qb = T0 - p.halo;
  // DC_ZSR: where this segment's local sum is complete (the next segment's warm-up start)
  long long q_cap = qb + p.seg_len;
  if (DC == DC_ZSR && q_cap > p.dc_end) q_cap = p.dc_end;

  float2 v = make_float2(0.0f, 0.0f);
  if (DC == DC_SCAN && qb > 0) v = p.v_seg[gid];
  if (qb < 0) qb = 0;
  long long q_end = i_hi > i_lo ? i_hi * D : qb;
  if (DC == DC_ZSR && q_cap > q_end) q_end = q_cap;
  if (q_end <= qb) {
    if (DC == DC_ZSR) p.sums[gid] = make_float2(0.0f, 0.0f);
    return;
  }
  // everything below is 32-bit and relative to qb (a multiple of G and D)
  const int n_it = (int)((q_end - qb + G - 1) / G);
  const int cap_it = (DC == DC_ZSR) ? (q_cap > qb ? (int)((q_cap - qb) / G) : 0) : -1;   // q_cap is a multiple of G
  const long long ob = qb / D;                                          // absolute index of local output 0
  int own_lo = (int)(i_lo - ob), own_hi = (int)(i_hi - ob);             // owned local outputs [own_lo, own_hi)
  if (i_hi <= i_lo) own_lo = own_hi = 0;

  HbStage<MA, G / 2, 0> sa;
  HbStage<MB, G / 4, 1> sb;
  HbStage<MC, G / 8, 2> sc;
  HbStage<MD, G / 16, 3> sd;
  sa.reset(); sb.reset(); sc.reset(); sd.reset();

  // arbitrary resampler state (A.5): output j goes with input floor(j step / 2^24)
  float2 w[13 + NO];
  float2 obuf[4];                  // four outputs (one 32-byte sector) are gathered per store
  unsigned phase = 0, j32 = 0;
  if (ARB) {
#pragma unroll
    for (int i = 0; i < 4; i++) obuf[i] = make_float2(0.0f, 0.0f);
#pragma unroll
    for (int i = 0; i < 13 + NO; i++) w[i] = make_float2(0.0f, 0.0f);
    if (i_lo > 0) {
      const unsigned long long num = (unsigned long long)i_lo << 24;
      const unsigned long long j = (num + p.step - 1) / p.step;
      phase = (unsigned)(j * p.step - num);
      j32 = (unsigned)j;
    }
  }
  unsigned ob_first = j32 & 3u;   // first slot of the current group of four that belongs to this segment
  float2* dst = p.dst + (long long)s * p.dst_stride;
  const unsigned dmask = (unsigned)p.dst_mask;
  const unsigned ob32 = (unsigned)ob;
  const float scale = p.scale;
  const float2 nalpha = make_float2(-p.alpha, -p.alpha);

  Loader<SRC> ld;
  ld.template init<G>(p.src, s, qb);
  Raw<SRC, G> cur;
  ld.template fetch<G>(0, cur);
  for (int it = 0; it < n_it; it++) {
    Raw<SRC, G> nxt;
    if (it + 1 < n_it) ld.template fetch<G>(it + 1, nxt);   // one group ahead
    float xr[G], xi[G];
    ld.template convert<G>(p.src, qb + (long long)it * G, it, cur, xr, xi);
    cur = nxt;
    float2 x[G];
#pragma unroll
    for (int i = 0; i < G; i++) x[i] = make_float2(xr[i], xi[i]);
    if (DC == DC_ZSR) {
      if (it == cap_it) p.sums[gid] = v;
    }
    if (DC != DC_NONE) {
#pragma unroll
      for (int i = 0; i < G; i++) {
        const float2 y = ffma2(nalpha, v, x[i]);   // y = x - alpha v ; v += y  (A.1)
        v = fadd2(v, y);
        x[i] = y;
      }
    }
    // half-band stages; the launch's scale rides on the last present stage
    float2 a[G / 2 > 0 ? G / 2 : 1], b2[G / 4 > 0 ? G / 4 : 1], c[G / 8 > 0 ? G / 8 : 1], d[G / 16 > 0 ? G / 16 : 1];
    float2* out = x;
    if constexpr (MA > 0) { sa.template run<NST == 1>(p, x, a, scale); out = a; }
    if constexpr (MB > 0) { sb.template run<NST == 2>(p, a, b2, scale); out = b2; }
    if constexpr (MC > 0) { sc.template run<NST == 3>(p, b2, c, scale); out = c; }
    if constexpr (MD > 0) { sd.template run<NST == 4>(p, c, d, scale); out = d; }

    const int o0 = it * NO;                       // local index of this iteration's first output
    const int lo = own_lo - o0, hi = own_hi - o0; // owned b are [lo, hi)
    const bool all = lo <= 0 && hi >= NO;
    if constexpr (!ARB) {
      if (all && (NO % 4 == 0)) {
        float2* d2 = dst + ((ob32 + (unsigned)o0) & dmask);
#pragma unroll
        for (int b = 0; b < NO / 4; b++) {
          const float f[8] = {out[4 * b].x, out[4 * b].y, out[4 * b + 1].x, out[4 * b + 1].y, out[4 * b + 2].x, out[4 * b + 2].y, out[4 * b + 3].x, out[4 * b + 3].y};
          stg256(d2 + 4 * b, f);
        }
      } else if (all && (NO % 2 == 0)) {
        float4* d4 = (float4*)(dst + ((ob32 + (unsigned)o0) & dmask));
#pragma unroll
        for (int b = 0; b < NO / 2; b++) d4[b] = make_float4(out[2 * b].x, out[2 * b].y, out[2 * b + 1].x, out[2 * b + 1].y);
      } else if (hi > 0 && lo < NO) {
#pragma unroll
        for (int b = 0; b < NO; b++)
          if (b >= lo && b < hi) dst[(ob32 + (unsigned)(o0 + b)) & dmask] = out[b];
      }
    } else {
#pragma unroll
      for (int b = 0; b < NO; b++) w[13 + b] = out[b];
      if (hi > 0 && lo < NO) {
#pragma unroll
        for (int b = 0; b < NO; b++) {
          if (all || (b >= lo && b < hi)) {
            // decimating plans have step >= 2^24: at most one output per pushed sample
            if (phase < (1u << 24)) {
              const float4* row = (const float4*)(sbank + (phase >> (24 - p.bits)) * BANK_STRIDE);
              const float4 h0 = row[0], h1 = row[1], h2 = row[2], h3 = row[3];
              const float h[14] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w, h2.x, h2.y, h2.z, h2.w, h3.x, h3.y};
              float2 y = make_float2(0.0f, 0.0f);
#pragma unroll
              for (int k = 0; k < 14; k++) y = fma_tap(h[k], w[13 + b - k], y);
              const unsigned slot = j32 & 3u;
#pragma unroll
              for (int sl = 0; sl < 4; sl++)
                if (slot == (unsigned)sl) obuf[sl] = y;
              if (slot == 3u) {
                float2* d2 = dst + ((j32 - 3u) & dmask);
                if (ob_first == 0u) {
                  const float f[8] = {obuf[0].x, obuf[0].y, obuf[1].x, obuf[1].y, obuf[2].x, obuf[2].y, obuf[3].x, obuf[3].y};
                  stg256(d2, f);
                } else {
#pragma unroll
                  for (int sl = 1; sl < 4; sl++)
                    if ((unsigned)sl >= ob_first) d2[sl] = obuf[sl];
                  ob_first = 0u;
                }
              }
              j32++;
              phase += p.step;
            }
            phase -= (1u << 24);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 13; i++) w[i] = w[NO + i];
    }
  }
  if (ARB) {   // outputs of an unfinished group of four
    const unsigned pend = j32 & 3u;
    float2* d2 = dst + ((j32 - pend) & dmask);
#pragma unroll
    for (int sl = 0; sl < 3; sl++)
      if ((unsigned)sl >= ob_first && (unsigned)sl < pend) d2[sl] = obuf[sl];
  }
  if (DC == DC_ZSR) {
    if (cap_it >= n_it) p.sums[gid] = v;
  }
}

}  // namespace pmr
