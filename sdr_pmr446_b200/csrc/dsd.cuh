// Back-end kernels of the dsd_in chain: discriminator on the 12.5 kHz complex stream, real
// interpolating multi-stage resampler (arbitrary x1.92 then one half-band x2), s16 conversion.
// Replaces freqdem_demodulate_block, msresamp_rrrf_execute and the cast loop of
// /root/reference/src/dsd_in.c:169-175 (SURVEY.md Appendix A.2-A.5, A.9; rows a13, a14).
// The rates here are tiny (12.5 k -> 48 k samples/s per stream) next to the 1-2.4 Msps front end,
// so these are plain one-thread-per-output kernels over the library's rings.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "audio_fft.cuh"   // pcm_sat

namespace pmr {

// fm[n] = arg(conj(x[n-1]) x[n]) * ref, n in [n0, n1); x[-1] = 0
static __global__ void dsd_freqdem_kernel(const float2* res, long long res_stride, long long res_mask, float* fm, long long fm_stride, long long fm_mask,
                                   long long n0, long long n1, float ref) {
  const long long n = n0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n1) return;
  const int s = blockIdx.y;
  const float2* r = res + (long long)s * res_stride;
  const float2 x = r[n & res_mask];
  float2 p = make_float2(0.0f, 0.0f);
  if (n > 0) p = r[(n - 1) & res_mask];
  const float re = __fadd_rn(__fmul_rn(p.x, x.x), __fmul_rn(p.y, x.y));
  const float im = __fsub_rn(__fmul_rn(p.x, x.y), __fmul_rn(p.y, x.x));
  fm[(long long)s * fm_stride + (n & fm_mask)] = atan2f(im, re) * ref;
}

// arbitrary resampler on a real ring (A.5): z[k] = sum_t pfb[idx_k][t] * fm[i_k - t],
// i_k = floor(k*step / 2^24), idx_k = (k*step mod 2^24) >> (24 - bits).
// One block = 256 consecutive outputs of one stream: their inputs are staged in shared memory, the bank rows (16 floats,
// 64-byte aligned) come from global memory with four 128-bit loads.
constexpr int DSD_XS = 1216;  // inputs staged per block: enough for 1024 outputs at any step >= 2^23 (rate <= 2), 4.9 KB
constexpr int DSD_RB = 4;     // outputs per thread: a block of 256 threads covers 1024 consecutive outputs
static __global__ void __launch_bounds__(256) dsd_arb_kernel(const float* fm, long long fm_stride, long long fm_mask, float* z, long long z_stride,
                                                             long long z_mask, long long k0, long long k1, unsigned step, int bits, const float* pfb) {
  __shared__ float xs[DSD_XS];
  const int s = blockIdx.y;
  const long long kb = k0 + (long long)blockIdx.x * (256 * DSD_RB);
  const long long kend = kb + 256 * DSD_RB < k1 ? kb + 256 * DSD_RB : k1;
  if (kb >= k1) return;
  const float* f = fm + (long long)s * fm_stride;
  const long long i_first = (long long)(((unsigned long long)kb * step) >> 24) - 13;
  const long long i_last = (long long)(((unsigned long long)(kend - 1) * step) >> 24);
  const int count = (int)(i_last - i_first + 1);
  const bool staged = count <= DSD_XS;   // block-uniform
  if (staged) {
    for (int c = threadIdx.x; c < count; c += 256) {
      const long long n = i_first + c;
      xs[c] = n >= 0 ? f[n & fm_mask] : 0.0f;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < DSD_RB; r++) {
    const long long k = kb + threadIdx.x + 256 * r;
    if (k >= kend) break;
    const unsigned long long ph = (unsigned long long)k * step;
    const long long i = (long long)(ph >> 24);
    const unsigned idx = (unsigned)(ph & 0xffffffu) >> (24 - bits);
    // the row straight from the (L1 / L2 resident, 16 KB) bank: a x1.92 resampler cycles through 25 of its 256 rows
    const float4* row = (const float4*)(pfb + ((size_t)idx << 4));
    const float4 h0 = __ldg(row), h1 = __ldg(row + 1), h2 = __ldg(row + 2), h3 = __ldg(row + 3);
    const float h[14] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w, h2.x, h2.y, h2.z, h2.w, h3.x, h3.y};
    float acc = 0.0f;
    if (staged) {
      const float* x = xs + (int)(i - i_first);
#pragma unroll
      for (int t = 0; t < 14; t++) acc = fmaf(h[t], x[-t], acc);
    } else {
#pragma unroll
      for (int t = 0; t < 14; t++) {
        const long long n = i - t;
        const float v = n >= 0 ? f[n & fm_mask] : 0.0f;
        acc = fmaf(h[t], v, acc);
      }
    }
    z[(long long)s * z_stride + (k & z_mask)] = acc;
  }
}

// half-band interpolator (A.4) + s16: out[2k] = z[k - m], out[2k+1] = sum_j h[j] z[k - j]
struct DsdInterpParams {
  const float* z;
  long long z_stride, z_mask;
  long long k0, k1;
  int m;
  float hb[20];
  float* audio;      // optional [n_streams][out_ld]
  short* pcm;        // optional [n_streams][out_ld]
  long long out_ld;
};
// one block = 256 consecutive input positions k of one stream, staged with their 2m - 1 predecessors
static __global__ void __launch_bounds__(256) dsd_interp_kernel(DsdInterpParams p) {
  __shared__ float zs[256 + 20];
  const int s = blockIdx.y;
  const long long kb = p.k0 + (long long)blockIdx.x * 256;
  if (kb >= p.k1) return;
  const float* z = p.z + (long long)s * p.z_stride;
  const int hist = 2 * p.m - 1;
  for (int c = threadIdx.x; c < 256 + hist; c += 256) {
    const long long n = kb - hist + c;
    zs[c] = (n >= 0 && n < p.k1) ? z[n & p.z_mask] : 0.0f;
  }
  __syncthreads();
  const long long k = kb + threadIdx.x;
  if (k >= p.k1) return;
  const float* q = zs + threadIdx.x + hist;   // q[-j] = z[k - j]
  const float y0 = q[-p.m];
  float y1 = 0.0f;
  for (int j = 0; j < 2 * p.m; j++) y1 = fmaf(p.hb[j], q[-j], y1);
  const long long o = (long long)s * p.out_ld + 2 * (k - p.k0);
  if (p.audio) {
    p.audio[o] = y0;
    p.audio[o + 1] = y1;
  }
  if (p.pcm) {
    const short a = (short)__float2int_rz(y0 * 32767.0f), b = (short)__float2int_rz(y1 * 32767.0f);
    if (((o | (long long)(uintptr_t)p.pcm >> 1) & 1) == 0) {
      *(short2*)(p.pcm + o) = make_short2(a, b);
    } else {
      p.pcm[o] = a;
      p.pcm[o + 1] = b;
    }
  }
}

// ---- dsd_backend_kernel: the arbitrary resampler, the half-band interpolator and the s16 cast in ONE launch (batched dsd path) ----
// dsd_arb_kernel gathers a 64-byte filter-bank row per OUTPUT (lanes of a warp hit ~25 different rows: 16-25 L1 wavefronts per
// 128-bit load; 0.32 ms per 1024-stream second for 24.6 M outputs) and hands z to dsd_interp_kernel through a ring in HBM (0.17 ms,
// one output pair per thread).  Here a block owns KB consecutive resampler outputs of one row (a dsd_in stream, or one (stream,
// channel) row of the batch chain's discriminator ring for its per-channel DSD feed):
//  phase 1: thread (j, g) computes outputs ks + j + P (g + G n), n = 0, 1, ...  P is the (near-)period of the phase sequence found on
//   the host (x1.92 = 48/25: P = 48, after which the 24-bit phase has moved by -16/2^24), so a thread's bank row changes once in
//   ~4000 outputs and its 14 taps stay in REGISTERS; the input window comes from shared memory (lanes read neighbouring words).  The
//   2m - 1 outputs in front of the block are recomputed from the discriminator ring instead of being read back: no z ring at all.
//  phase 2: out[2k] = z[k - m], out[2k + 1] = sum_j h[j] z[k - j] from shared memory, float / s16 pair stores.
// Same operations in the same order as the two kernels it replaces (bit-identical results).  The s16 cast wraps like dsd_in's
// (SAT = false) or saturates (SAT = true, pcm_sat: the batch chain's DSD feed).
constexpr int DSB_T = 192;                 // threads per block
constexpr int DSB_KB = 1536;               // resampler outputs per block (3072 output samples)
constexpr int DSB_HIST = 19;               // 2 m - 1 for the largest half-band (m = 10)
constexpr int DSB_XS = DSB_KB + DSB_HIST + 32;   // staged inputs: rate >= 1 means at most one input per output, + 13 of filter history
struct DsdBackendParams {
  const float* fm;           // discriminator ring [rows][fm_stride]
  long long fm_stride, fm_mask;
  int tiles;                 // blocks per row: block b serves row b / tiles (rows folded into gridDim.x: no 65535-row limit)
  long long k0, k1;          // resampler outputs of this call
  unsigned step;             // 2^24 / rate of the arbitrary stage, in [2^23, 2^24]
  int bits;                  // log2(number of bank rows)
  int period, groups;        // P and G = DSB_T / P
  const float* pfb;          // [rows][16] bank, newest tap first
  int m;                     // half-band semi-length
  float hb[20];
  float* audio;              // optional [rows][out_ld]
  short* pcm;                // optional [rows][out_ld]
  long long out_ld;
};
// (Near-)period P <= DSB_T of the arbitrary stage's phase sequence: after P outputs the 24-bit phase is back within 1/16 of a bank
// row, so a thread that computes outputs k, k + P, k + 2P, ... keeps its bank row in registers (x1.92: P = 48, drift -16 / 2^24).
inline int dsd_arb_period(unsigned step, unsigned bits) {
  const unsigned tol = (1u << (24 - bits)) / 16;
  for (int P = 1; P <= DSB_T; P++) {
    const unsigned r = (unsigned)(((unsigned long long)P * step) & 0xffffffu);
    if (r <= tol || (1u << 24) - r <= tol) return P;
  }
  return 32;
}
template <int M, bool SAT>   // M: half-band semi-length known at compile time (unrolled taps from the constant bank), 0 = use p.m
static __global__ void __launch_bounds__(DSB_T) dsd_backend_kernel(DsdBackendParams p) {
  __shared__ float xs[DSB_XS];
  __shared__ float zs[DSB_KB + DSB_HIST];
  const long long s = blockIdx.x / p.tiles;
  const long long kb = p.k0 + (long long)(blockIdx.x % p.tiles) * DSB_KB;
  if (kb >= p.k1) return;
  const long long kend = kb + DSB_KB < p.k1 ? kb + DSB_KB : p.k1;
  const int m = M ? M : p.m;
  const int hist = 2 * m - 1;
  const long long ks = kb - hist;                       // first z this block needs (z[k < 0] = 0)
  const long long kf = ks > 0 ? ks : 0;
  const float* f = p.fm + s * p.fm_stride;
  const long long i_first = (long long)(((unsigned long long)kf * p.step) >> 24) - 13;
  const long long i_last = (long long)(((unsigned long long)(kend - 1) * p.step) >> 24);
  const int count = (int)(i_last - i_first + 1);        // <= KB + hist + 14 for step <= 2^24 (checked on the host)
  for (int c = threadIdx.x; c < count; c += DSB_T) {
    const long long n = i_first + c;
    xs[c] = n >= 0 ? f[n & p.fm_mask] : 0.0f;
  }
  __syncthreads();
  // ---- phase 1 ----
  if ((int)threadIdx.x < p.period * p.groups) {
    const int j = threadIdx.x % p.period, g = threadIdx.x / p.period;
    float h[14];
#pragma unroll
    for (int t = 0; t < 14; t++) h[t] = 0.0f;
    unsigned cur = 0xffffffffu;
    for (long long k = ks + j + (long long)p.period * g; k < kend; k += (long long)p.period * p.groups) {
      float acc = 0.0f;
      if (k >= 0) {
        const unsigned long long ph = (unsigned long long)k * p.step;
        const unsigned idx = (unsigned)(ph & 0xffffffu) >> (24 - p.bits);
        if (idx != cur) {
          const float4* row = (const float4*)(p.pfb + ((size_t)idx << 4));
          const float4 h0 = __ldg(row), h1 = __ldg(row + 1), h2 = __ldg(row + 2), h3 = __ldg(row + 3);
          h[0] = h0.x; h[1] = h0.y; h[2] = h0.z; h[3] = h0.w; h[4] = h1.x; h[5] = h1.y; h[6] = h1.z; h[7] = h1.w;
          h[8] = h2.x; h[9] = h2.y; h[10] = h2.z; h[11] = h2.w; h[12] = h3.x; h[13] = h3.y;
          cur = idx;
        }
        const float* x = xs + (int)((long long)(ph >> 24) - i_first);
#pragma unroll
        for (int t = 0; t < 14; t++) acc = fmaf(h[t], x[-t], acc);
      }
      zs[(int)(k - ks)] = acc;
    }
  }
  __syncthreads();
  // ---- phase 2 ----
  for (long long k = kb + threadIdx.x; k < kend; k += DSB_T) {
    const float* q = zs + (int)(k - ks);   // q[-j] = z[k - j]
    const float y0 = q[-m];
    float y1 = 0.0f;
    if (M) {
#pragma unroll
      for (int j = 0; j < 2 * M; j++) y1 = fmaf(p.hb[j], q[-j], y1);
    } else {
      for (int j = 0; j < 2 * m; j++) y1 = fmaf(p.hb[j], q[-j], y1);
    }
    const long long o = s * p.out_ld + 2 * (k - p.k0);
    if (p.audio) {
      p.audio[o] = y0;
      p.audio[o + 1] = y1;
    }
    if (p.pcm) {
      const short a = SAT ? pcm_sat(y0) : (short)__float2int_rz(y0 * 32767.0f), b = SAT ? pcm_sat(y1) : (short)__float2int_rz(y1 * 32767.0f);
      if (((o | (long long)(uintptr_t)p.pcm >> 1) & 1) == 0) {
        *(short2*)(p.pcm + o) = make_short2(a, b);
      } else {
        p.pcm[o] = a;
        p.pcm[o + 1] = b;
      }
    }
  }
}

}  // namespace pmr
