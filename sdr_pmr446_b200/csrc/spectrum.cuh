// Waterfall (asgram / spgram) kernels -- replaces asgramcf_write + asgramcf_execute of the
// reference (/root/reference/src/sdr_pmr446.c:473-477, :910-913; SURVEY.md Appendix A.13).
//
// Per chunk and stream: Welch periodogram of the UN-mixed resampler output with a Hann window
// of length W, hop W/2, zero-padded nfft = 4W transform (W is the terminal width, so nfft is in
// general not a power of two: 480 for W = 120, 6400 for W = 1600), |X|^2 summed over the chunk,
// then dB, fft-shift, peak search, 4-bin column reduction and the 10-level character map.
// The FFT is a shared-memory Stockham autosort with radices 4/2/3/5 (any other prime factor
// falls back to a generic radix-p butterfly); one block walks the transforms of one
// (stream, part) and keeps the |X|^2 accumulator in shared memory.  No tensor cores, no cuFFT.
#pragma once
#include <cuda_runtime.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common_host.hpp"
#include "reg_dft.cuh"

namespace pmr {

template <int R>
__device__ __forceinline__ void wf_stage(const float2* __restrict__ x, float2* __restrict__ y, const float2* __restrict__ tw, int N, int Ns);
struct WfParams {
  const float2* res;       // resampler output ring
  long long res_stride, res_mask;
  long long r0;            // first sample of this chunk
  long long ny;            // samples in this chunk
  int W, nfft, hop;
  int n_transforms;        // floor(ny / hop)
  int parts;               // blocks per stream
  int groups, tg;          // block-per-transform kernel: independent thread groups per block and threads per group
  const float* window;     // [W] scaled Hann
  const float2* twiddle;   // [nfft] exp(-2 pi i k / nfft)
  int n_stages;
  int radix[16];
  float* partial;          // [n_streams][parts][nfft]
};

template <int R>
__device__ __forceinline__ void wf_stage(const float2* __restrict__ x, float2* __restrict__ y, const float2* __restrict__ tw, int N, int Ns,
                                         int first, int stride) {
  const int nb = N / R;
  const int tstep = N / (Ns * R);
  const float inv_ns = 1.0f / (float)Ns;
  for (int j = first; j < nb; j += stride) {
    const int k = j - (int)(((float)j + 0.5f) * inv_ns) * Ns;   // j mod Ns without an integer division (exact for j < 2^20)
    float2 v[R];
    // twiddles W^(r k tstep), r = 1 .. R-1, as powers of ONE table entry: the gathers (a different cache line per lane in
    // the early stages) made these stages load/store-bound
    const float2 w1 = tw[k * tstep];
    float2 wr = w1;
#pragma unroll
    for (int r = 0; r < R; r++) {
      float2 a = x[j + r * nb];
      if (r > 0) {
        a = make_float2(a.x * wr.x - a.y * wr.y, a.x * wr.y + a.y * wr.x);
        if (r + 1 < R) wr = make_float2(wr.x * w1.x - wr.y * w1.y, wr.x * w1.y + wr.y * w1.x);
      }
      v[r] = a;
    }
    const int j0 = (j - k) * R + k;
    if (R == 2) {
      y[j0] = make_float2(v[0].x + v[1].x, v[0].y + v[1].y);
      y[j0 + Ns] = make_float2(v[0].x - v[1].x, v[0].y - v[1].y);
    } else if (R == 4) {
      // forward DFT: W4 = -i
      const float2 s02 = make_float2(v[0].x + v[2].x, v[0].y + v[2].y), d02 = make_float2(v[0].x - v[2].x, v[0].y - v[2].y);
      const float2 s13 = make_float2(v[1].x + v[3].x, v[1].y + v[3].y), d13 = make_float2(v[1].x - v[3].x, v[1].y - v[3].y);
      y[j0] = make_float2(s02.x + s13.x, s02.y + s13.y);
      y[j0 + Ns] = make_float2(d02.x + d13.y, d02.y - d13.x);      // d02 - i d13
      y[j0 + 2 * Ns] = make_float2(s02.x - s13.x, s02.y - s13.y);
      y[j0 + 3 * Ns] = make_float2(d02.x - d13.y, d02.y + d13.x);  // d02 + i d13
    } else {
      if (R == 3) dft3(v);
      else dft5(v);
#pragma unroll
      for (int q = 0; q < R; q++) y[j0 + q * Ns] = v[q];
    }
  }
}

template <int R>
__device__ __forceinline__ void wf_stage(const float2* __restrict__ x, float2* __restrict__ y, const float2* __restrict__ tw, int N, int Ns) {
  wf_stage<R>(x, y, tw, N, Ns, (int)threadIdx.x, (int)blockDim.x);
}

// generic prime radix p (reads straight from shared memory, O(p) per output).  One work item per OUTPUT (j, q), so
// a large prime (nfft = 4 * 67: four butterflies of 67 points) still spreads over the whole block / warp.
__device__ __forceinline__ void wf_stage_generic(int R, const float2* __restrict__ x, float2* __restrict__ y, const float2* __restrict__ tw, int N, int Ns,
                                                 int first, int stride) {
  const int nb = N / R, tstep = N / (Ns * R), rstep = N / R;
  for (int idx = first; idx < N; idx += stride) {
    const int j = idx % nb, q = idx / nb;
    const int k = j % Ns;
    const int j0 = (j - k) * R + k;
    // a sum of up to 4096 terms that cancel to a small output in most bins: accumulated in double, so the only float32
    // rounding left is that of the inputs, the twiddle table and the result (a float32 running sum lost ~p ulp of the
    // largest terms, e.g. 4e-6 of the stage RMS in the weak bins of a 1828 = 4 x 457 channel bank)
    double ax = x[j].x, ay = x[j].y;
    int t = 0;   // (r k tstep + ((q r) mod R) rstep) mod N: the product of the two twiddles is one table entry
    for (int r = 1; r < R; r++) {
      t += k * tstep + q * rstep;
      while (t >= N) t -= N;
      const float2 a = x[j + r * nb];
      const float2 w = tw[t];
      ax = fma((double)a.x, (double)w.x, fma(-(double)a.y, (double)w.y, ax));
      ay = fma((double)a.x, (double)w.y, fma((double)a.y, (double)w.x, ay));
    }
    y[j0 + q * Ns] = make_float2((float)ax, (float)ay);
  }
}

// Large transforms (nfft > 1024, e.g. 6400 for the wideband configuration's W = 1600).  A block holds `groups` independent
// thread groups of `tg` threads; each group walks its own transforms with its own ping-pong buffers and its own named barrier,
// so while one group waits at a stage barrier the other one computes (one 1024-thread group per block -- round 1 -- spent
// most of its time at those barriers).  |X|^2 accumulates in registers (bins lt + k tg).
constexpr int WFB_NM = 16;   // accumulator registers per thread: nfft <= 16 tg
static __global__ void __launch_bounds__(1024) wf_accumulate_kernel(WfParams p) {
  extern __shared__ float2 wf_smem[];
  const int g = threadIdx.x / p.tg, lt = threadIdx.x - g * p.tg;
  float2* a = wf_smem + (size_t)g * 2 * p.nfft;
  float2* b = a + p.nfft;
  auto group_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "r"(p.tg) : "memory"); };
  const int s = blockIdx.x / p.parts, part = blockIdx.x % p.parts;
  const float2* res = p.res + (long long)s * p.res_stride;
  float acc[WFB_NM];
#pragma unroll
  for (int k = 0; k < WFB_NM; k++) acc[k] = 0.0f;
  // transform t (1-based) fires after t*hop samples of the chunk and sees the last W of them
  for (int t = 1 + part * p.groups + g; t <= p.n_transforms; t += p.parts * p.groups) {
    group_sync();
    const long long first = (long long)t * p.hop - p.W;  // chunk-local index of window sample 0
    // nfft = 4 W with a leading radix-4 stage: its inputs 1..3 are the zero padding, so the stage is the load itself
    const bool lead4 = p.radix[0] == 4 && p.nfft == 4 * p.W;
    if (lead4) {
      for (int i = lt; i < p.W; i += p.tg) {
        const long long li = first + i;
        float2 v = make_float2(0.0f, 0.0f);
        if (li >= 0) {
          const float2 x = res[(p.r0 + li) & p.res_mask];
          const float w = p.window[i];
          v = make_float2(x.x * w, x.y * w);
        }
        b[4 * i] = v; b[4 * i + 1] = v; b[4 * i + 2] = v; b[4 * i + 3] = v;
      }
    } else {
      for (int i = lt; i < p.nfft; i += p.tg) {
        float2 v = make_float2(0.0f, 0.0f);
        if (i < p.W) {
          const long long li = first + i;
          if (li >= 0) {
            const float2 x = res[(p.r0 + li) & p.res_mask];
            const float w = p.window[i];
            v = make_float2(x.x * w, x.y * w);
          }
        }
        a[i] = v;
      }
    }
    group_sync();
    float2 *x = lead4 ? b : a, *y = lead4 ? a : b;
    int Ns = lead4 ? 4 : 1;
    for (int st = lead4 ? 1 : 0; st < p.n_stages; st++) {
      const int R = p.radix[st];
      if (R == 4) wf_stage<4>(x, y, p.twiddle, p.nfft, Ns, lt, p.tg);
      else if (R == 2) wf_stage<2>(x, y, p.twiddle, p.nfft, Ns, lt, p.tg);
      else if (R == 3) wf_stage<3>(x, y, p.twiddle, p.nfft, Ns, lt, p.tg);
      else if (R == 5) wf_stage<5>(x, y, p.twiddle, p.nfft, Ns, lt, p.tg);
      else wf_stage_generic(R, x, y, p.twiddle, p.nfft, Ns, lt, p.tg);
      Ns *= R;
      float2* tmp = x; x = y; y = tmp;
      group_sync();
    }
#pragma unroll
    for (int k = 0; k < WFB_NM; k++) {
      const int i = lt + k * p.tg;
      if (i < p.nfft) { const float2 z = x[i]; acc[k] = fmaf(z.x, z.x, fmaf(z.y, z.y, acc[k])); }
    }
  }
  float* out = p.partial + (((long long)s * p.parts + part) * p.groups + g) * p.nfft;
#pragma unroll
  for (int k = 0; k < WFB_NM; k++) {
    const int i = lt + k * p.tg;
    if (i < p.nfft) out[i] = acc[k];
  }
}

// ---- small transforms (nfft <= 1024): one WARP per transform ----------------------------------------------------------
// A 480-point transform has 96..240 butterflies per stage: a whole block on one transform leaves most threads idle and
// pays a block barrier per stage.  Here every warp of the block walks its own transforms (ping-pong buffers private to
// the warp, __syncwarp between stages, |X|^2 accumulated in registers: bin lane + 32 m), the twiddle table sits in
// shared memory, and because nfft = 4 W with a leading radix-4 stage whose inputs 1..3 are the zero padding, that stage
// is the load itself (each windowed sample is written to its four outputs).
constexpr int WFW_WARPS = 8;   // at most; the launch uses as many as fit in 96 KB of shared memory

template <int R>
__device__ __forceinline__ void wf_stage_warp(const float2* __restrict__ x, float2* __restrict__ y, const float2* __restrict__ tw, int N, int Ns,
                                              float inv_ns, int lane) {
  const int nb = N / R, tstep = N / (Ns * R);
  for (int j = lane; j < nb; j += 32) {
    const int k = j - (int)(((float)j + 0.5f) * inv_ns) * Ns;   // j mod Ns (exact for j < 2^20)
    float2 v[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
      float2 a = x[j + r * nb];
      if (r > 0) {
        const float2 w = tw[r * k * tstep];   // r k tstep < N
        a = make_float2(a.x * w.x - a.y * w.y, a.x * w.y + a.y * w.x);
      }
      v[r] = a;
    }
    const int j0 = (j - k) * R + k;
    if (R == 2) {
      y[j0] = make_float2(v[0].x + v[1].x, v[0].y + v[1].y);
      y[j0 + Ns] = make_float2(v[0].x - v[1].x, v[0].y - v[1].y);
    } else if (R == 4) {
      const float2 s02 = make_float2(v[0].x + v[2].x, v[0].y + v[2].y), d02 = make_float2(v[0].x - v[2].x, v[0].y - v[2].y);
      const float2 s13 = make_float2(v[1].x + v[3].x, v[1].y + v[3].y), d13 = make_float2(v[1].x - v[3].x, v[1].y - v[3].y);
      y[j0] = make_float2(s02.x + s13.x, s02.y + s13.y);
      y[j0 + Ns] = make_float2(d02.x + d13.y, d02.y - d13.x);
      y[j0 + 2 * Ns] = make_float2(s02.x - s13.x, s02.y - s13.y);
      y[j0 + 3 * Ns] = make_float2(d02.x - d13.y, d02.y + d13.x);
    } else {
      if (R == 3) dft3(v);
      else dft5(v);
#pragma unroll
      for (int q = 0; q < R; q++) y[j0 + q * Ns] = v[q];
    }
  }
}

template <int NM>   // accumulator registers per lane: nfft <= 32 NM
static __global__ void __launch_bounds__(32 * WFW_WARPS) wf_accumulate_warp_kernel(WfParams p) {
  extern __shared__ float2 wf_smem[];
  const int N = p.nfft, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float2* tw = wf_smem;                              // [N]
  float2* a = wf_smem + N + (size_t)w * 2 * N;       // this warp's ping
  float2* b = a + N;                                 // and pong
  const int s = blockIdx.x / p.parts, part = blockIdx.x % p.parts;
  const float2* res = p.res + (long long)s * p.res_stride;
  for (int i = threadIdx.x; i < N; i += blockDim.x) tw[i] = p.twiddle[i];
  __syncthreads();
  float acc[NM];
#pragma unroll
  for (int m = 0; m < NM; m++) acc[m] = 0.0f;
  const bool lead4 = p.radix[0] == 4 && N == 4 * p.W;    // first stage folded into the load
  const int nw = blockDim.x >> 5;
  for (int t = 1 + part + p.parts * w; t <= p.n_transforms; t += p.parts * nw) {
    const long long first = (long long)t * p.hop - p.W;  // chunk-local index of window sample 0
    if (lead4) {
      for (int i = lane; i < p.W; i += 32) {
        const long long li = first + i;
        float2 v = make_float2(0.0f, 0.0f);
        if (li >= 0) {
          const float2 x = res[(p.r0 + li) & p.res_mask];
          const float wv = p.window[i];
          v = make_float2(x.x * wv, x.y * wv);
        }
        b[4 * i] = v; b[4 * i + 1] = v; b[4 * i + 2] = v; b[4 * i + 3] = v;
      }
    } else {
      for (int i = lane; i < N; i += 32) {
        float2 v = make_float2(0.0f, 0.0f);
        const long long li = first + i;
        if (i < p.W && li >= 0) {
          const float2 x = res[(p.r0 + li) & p.res_mask];
          const float wv = p.window[i];
          v = make_float2(x.x * wv, x.y * wv);
        }
        a[i] = v;
      }
    }
    __syncwarp();
    float2 *x = lead4 ? b : a, *y = lead4 ? a : b;
    int Ns = lead4 ? 4 : 1;
    for (int st = lead4 ? 1 : 0; st < p.n_stages; st++) {
      const int R = p.radix[st];
      const float inv = 1.0f / (float)Ns;
      if (R == 4) wf_stage_warp<4>(x, y, tw, N, Ns, inv, lane);
      else if (R == 2) wf_stage_warp<2>(x, y, tw, N, Ns, inv, lane);
      else if (R == 3) wf_stage_warp<3>(x, y, tw, N, Ns, inv, lane);
      else if (R == 5) wf_stage_warp<5>(x, y, tw, N, Ns, inv, lane);
      else wf_stage_generic(R, x, y, tw, N, Ns, lane, 32);   // other primes
      Ns *= R;
      float2* tmp = x; x = y; y = tmp;
      __syncwarp();
    }
#pragma unroll
    for (int m = 0; m < NM; m++) {
      const int i = lane + 32 * m;
      if (i < N) { const float2 z = x[i]; acc[m] = fmaf(z.x, z.x, fmaf(z.y, z.y, acc[m])); }
    }
    __syncwarp();
  }
  // block reduction of the warps' accumulators through the (now idle) transform buffers
  __syncthreads();
  float* red = (float*)(wf_smem + N);   // [WFW_WARPS][N]
#pragma unroll
  for (int m = 0; m < NM; m++) {
    const int i = lane + 32 * m;
    if (i < N) red[(size_t)w * N + i] = acc[m];
  }
  __syncthreads();
  float* out = p.partial + ((long long)s * p.parts + part) * N;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float sum = 0.0f;
    for (int q = 0; q < nw; q++) sum += red[(size_t)q * N + i];
    out[i] = sum;
  }
}

struct WfFinalParams {
  const float* partial;
  int parts, W, nfft, n_transforms;
  float ref, div;
  char* ascii;   // [n_streams][W]
  float* peak;   // [n_streams][2]
  float* psd;    // [n_streams][nfft]
  float* scratch;  // [n_streams][nfft] dB values when psd == nullptr
  float* blk_v;    // [n_streams][nblk] peak of every 256-bin block (wf_db_kernel -> wf_finalize_kernel)
  int* blk_i;
  int nblk;
};

// Two launches: wf_db_kernel gives every output bin its own thread (sum of the partial spectra in their fixed order, fftshift,
// 10 log10) and reduces the peak per 256-bin block; wf_finalize_kernel reduces the block peaks and draws the row.  (One block per
// stream doing all of it took 0.51 ms for four 6400-bin spectra with 37 partials each -- 42 % of the wideband step: 925 dependent
// global loads per thread.)
static __global__ void __launch_bounds__(256) wf_db_kernel(WfFinalParams p) {
  const int s = blockIdx.y;
  const int i = blockIdx.x * 256 + threadIdx.x;
  __shared__ float best_v[256];
  __shared__ int best_i[256];
  if (p.n_transforms == 0) {
    if (p.psd && i < p.nfft) p.psd[(long long)s * p.nfft + i] = 0.0f;
    return;
  }
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  if (i < p.nfft) {
    float* db = (p.psd ? p.psd : p.scratch) + (long long)s * p.nfft;
    const int k = (i + p.nfft / 2) % p.nfft;
    const float* src = p.partial + (long long)s * p.parts * p.nfft + k;
    float a = 0.0f;
    int q = 0;
    for (; q + 8 <= p.parts; q += 8) {   // eight loads in flight, added in the order q = 0, 1, 2, ...
      float t[8];
#pragma unroll
      for (int j = 0; j < 8; j++) t[j] = src[(long long)(q + j) * p.nfft];
#pragma unroll
      for (int j = 0; j < 8; j++) a += t[j];
    }
    for (; q < p.parts; q++) a += src[(long long)q * p.nfft];
    const float v = a > 1e-12f ? a : 1e-12f;
    const float d = 10.0f * log10f(v * (1.0f / (float)p.n_transforms));
    db[i] = d;
    bv = d;
    bi = i;
  }
  best_v[threadIdx.x] = bv;
  best_i[threadIdx.x] = bi;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const float v2 = best_v[threadIdx.x + o];
      const int i2 = best_i[threadIdx.x + o];
      if (v2 > best_v[threadIdx.x] || (v2 == best_v[threadIdx.x] && i2 < best_i[threadIdx.x])) {
        best_v[threadIdx.x] = v2;
        best_i[threadIdx.x] = i2;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    p.blk_v[(long long)s * gridDim.x + blockIdx.x] = best_v[0];
    p.blk_i[(long long)s * gridDim.x + blockIdx.x] = best_i[0];
  }
}

static __global__ void __launch_bounds__(256) wf_finalize_kernel(WfFinalParams p) {
  const int s = blockIdx.x;
  __shared__ float best_v[256];
  __shared__ int best_i[256];
  char* ascii = p.ascii ? p.ascii + (long long)s * p.W : nullptr;
  if (p.n_transforms == 0) {  // asgramcf_execute with no transforms: blanks, peak 0
    if (ascii) for (int i = threadIdx.x; i < p.W; i += blockDim.x) ascii[i] = ' ';
    if (p.peak && threadIdx.x == 0) { p.peak[2 * s] = 0.0f; p.peak[2 * s + 1] = 0.0f; }
    return;
  }
  const float* db = (p.psd ? p.psd : p.scratch) + (long long)s * p.nfft;
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  for (int b = threadIdx.x; b < p.nblk; b += blockDim.x) {   // block peaks, lowest index first on a tie
    const float v2 = p.blk_v[(long long)s * p.nblk + b];
    const int i2 = p.blk_i[(long long)s * p.nblk + b];
    if (v2 > bv || (v2 == bv && i2 < bi)) { bv = v2; bi = i2; }
  }
  best_v[threadIdx.x] = bv;
  best_i[threadIdx.x] = bi;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const float v2 = best_v[threadIdx.x + o];
      const int i2 = best_i[threadIdx.x + o];
      if (v2 > best_v[threadIdx.x] || (v2 == best_v[threadIdx.x] && i2 < best_i[threadIdx.x])) {
        best_v[threadIdx.x] = v2;
        best_i[threadIdx.x] = i2;
      }
    }
    __syncthreads();
  }
  if (p.peak && threadIdx.x == 0) {
    p.peak[2 * s] = best_v[0];
    p.peak[2 * s + 1] = (float)best_i[0] / (float)p.nfft - 0.5f;
  }
  if (ascii) {
    const char levelchar[11] = " .,-+*&NM#";
    for (int i = threadIdx.x; i < p.W; i += blockDim.x) {
      float val = db[4 * i];
#pragma unroll
      for (int j = 1; j < 4; j++) val = fmaxf(val, db[4 * i + j]);
      char c = levelchar[0];
      for (int j = 0; j < 10; j++)
        if (val > p.ref + (float)j * p.div) c = levelchar[j];
      ascii[i] = c;
    }
  }
}

}  // namespace pmr
#include "spectrum_fast.cuh"
namespace pmr {

// init() and execute() are force-inlined: the kernels above are static (one copy per translation unit), so the code that
// sets their attributes and launches them must not be merged across translation units by the linker either.
struct Waterfall {
  int S = 0;
  unsigned W = 0, nfft = 0;
  int parts = 1;
  float ref = -40.0f, div = 2.0f;   // asgramcf_set_scale(-40, 2), src/sdr_pmr446.c:476
  std::vector<int> radix;
  DevBuf d_window, d_twiddle, d_partial, d_scratch, d_blk;
  size_t smem = 0;
  bool warp_kernel = false;   // nfft <= 1024: one warp per transform
  int wf_warps = 1;
  int groups = 1, tg = 256;   // block-per-transform kernel: thread groups per block, threads per group
  int fast_p = 0;             // W = 8 P with P in {8, 10, 12, 15, 16, 20}: register-resident kernel (spectrum_fast.cuh)
  float2 twp[WFF_MAXP];

  __attribute__((always_inline)) inline int init(int n_streams, unsigned width) {
    S = n_streams;
    W = width;
    nfft = 4 * width;
    if (W < 2 || W > 2048) return fail(PMR446_EINVAL, "waterfall width must be in [2, 2048]");
    unsigned n = nfft;
    while (n % 4 == 0) { radix.push_back(4); n /= 4; }
    for (unsigned pr = 2; n > 1;) {
      if (n % pr == 0) { radix.push_back((int)pr); n /= pr; }
      else pr++;
    }
    if (radix.size() > 16) return fail(PMR446_EINVAL, "waterfall width has too many prime factors");
    std::vector<float> w = design::asgram_window(W);
    std::vector<float2> tw(nfft);
    for (unsigned k = 0; k < nfft; k++) {
      double a = -2.0 * M_PI * (double)k / (double)nfft;
      tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    // enough (stream, part) blocks to fill the GPU: one block needs nfft * 20 bytes of shared memory (block-per-transform
    // kernel) or nfft * 8 * (1 + 2 * 8 warps) bytes (warp-per-transform kernel, nfft <= 1024)
    {
      const char* env = getenv("PMR446_WATERFALL");   // "generic" keeps round 1's shared-memory kernels (A/B runs)
      const unsigned P = W / 8;
      if (W % 8 == 0 && (P == 8 || P == 10 || P == 12 || P == 15 || P == 16 || P == 20) && !(env && strcmp(env, "generic") == 0)) {
        fast_p = (int)P;
        for (unsigned m = 0; m < P; m++) {
          const double a = -2.0 * M_PI * (double)m / (double)P;
          twp[m] = make_float2((float)cos(a), (float)sin(a));
        }
      }
    }
    warp_kernel = nfft <= 1024;
    if (!warp_kernel && !fast_p) {
      tg = nfft > 4096 ? 512 : 256;                                   // nfft <= 8192 = 16 tg
      groups = (int)std::max<size_t>(1, std::min<size_t>(1024 / tg, (200 * 1024) / ((size_t)nfft * 2 * sizeof(float2))));
    }
    wf_warps = std::max(1, std::min(WFW_WARPS, (int)((96 * 1024 / (nfft * sizeof(float2)) - 1) / 2)));
    {
      const size_t per_block = warp_kernel ? (size_t)nfft * sizeof(float2) * (1 + 2 * wf_warps) : (size_t)nfft * 2 * sizeof(float2) * groups;
      const int per_sm = fast_p ? 3 : (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / per_block));
      // the fast kernel's blocks are long (a whole stream's transforms): eight waves of them keep the tail short
      parts = std::max(1, std::min(128, ((fast_p ? 8 : 1) * 148 * per_sm + S - 1) / S));
    }
    int rc;
    if ((rc = d_window.alloc(W * sizeof(float))) || (rc = d_twiddle.alloc(nfft * sizeof(float2))) ||
        (rc = d_partial.alloc((size_t)S * parts * groups * nfft * sizeof(float))) || (rc = d_scratch.alloc((size_t)S * nfft * sizeof(float))) ||
        (rc = d_blk.alloc((size_t)S * ((nfft + 255) / 256) * 2 * sizeof(float))))
      return rc;
    CUDA_TRY(cudaMemcpy(d_window.p, w.data(), W * sizeof(float), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_twiddle.p, tw.data(), nfft * sizeof(float2), cudaMemcpyHostToDevice));
    smem = warp_kernel ? (size_t)nfft * sizeof(float2) * (1 + 2 * wf_warps) : (size_t)nfft * 2 * sizeof(float2) * groups;
    if (warp_kernel && smem > 48 * 1024) {
      CUDA_TRY(cudaFuncSetAttribute(wf_accumulate_warp_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      CUDA_TRY(cudaFuncSetAttribute(wf_accumulate_warp_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      CUDA_TRY(cudaFuncSetAttribute(wf_accumulate_warp_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (!warp_kernel) CUDA_TRY(cudaFuncSetAttribute(wf_accumulate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return 0;
  }

  __attribute__((always_inline)) inline int execute(const float2* res, long long res_cap, long long r0, long long ny, char* ascii, float* peak,
                                                    float* psd, cudaStream_t st,
              int* launches) {
    WfParams p;
    p.res = res;
    p.res_stride = res_cap;
    p.res_mask = res_cap - 1;
    p.r0 = r0;
    p.ny = ny;
    p.W = (int)W;
    p.nfft = (int)nfft;
    p.hop = (int)(W / 2);
    p.n_transforms = (int)(ny / p.hop);
    p.parts = parts;
    p.groups = groups;
    p.tg = tg;
    p.window = (const float*)d_window.p;
    p.twiddle = (const float2*)d_twiddle.p;
    p.n_stages = (int)radix.size();
    for (size_t i = 0; i < radix.size(); i++) p.radix[i] = radix[i];
    p.partial = (float*)d_partial.p;
    if (p.n_transforms > 0 && fast_p) {
      WfFastParams fpar;
      fpar.w = p;
      memcpy(fpar.twp, twp, sizeof twp);
      const unsigned grid = (unsigned)(S * parts), thr = 32 * WFF_WARPS;
      switch (fast_p) {
        case 8: wf_accumulate_fast_kernel<8><<<grid, thr, 0, st>>>(fpar); break;
        case 10: wf_accumulate_fast_kernel<10><<<grid, thr, 0, st>>>(fpar); break;
        case 12: wf_accumulate_fast_kernel<12><<<grid, thr, 0, st>>>(fpar); break;
        case 15: wf_accumulate_fast_kernel<15><<<grid, thr, 0, st>>>(fpar); break;
        case 16: wf_accumulate_fast_kernel<16><<<grid, thr, 0, st>>>(fpar); break;
        default: wf_accumulate_fast_kernel<20><<<grid, thr, 0, st>>>(fpar); break;
      }
      (*launches)++;
    } else if (p.n_transforms > 0) {
      // a large transform leaves room for one block per SM only: give it 32 warps to hide the shared-memory latency
      if (warp_kernel && nfft <= 256) wf_accumulate_warp_kernel<8><<<S * parts, 32 * wf_warps, smem, st>>>(p);
      else if (warp_kernel && nfft <= 512) wf_accumulate_warp_kernel<16><<<S * parts, 32 * wf_warps, smem, st>>>(p);
      else if (warp_kernel) wf_accumulate_warp_kernel<32><<<S * parts, 32 * wf_warps, smem, st>>>(p);
      else wf_accumulate_kernel<<<S * parts, groups * tg, smem, st>>>(p);
      (*launches)++;
    }
    WfFinalParams f;
    f.partial = p.partial;
    f.parts = (warp_kernel || fast_p) ? parts : parts * groups;
    f.W = p.W;
    f.nfft = p.nfft;
    f.n_transforms = p.n_transforms;
    f.ref = ref;
    f.div = div;
    f.ascii = ascii;
    f.peak = peak;
    f.psd = psd;
    f.scratch = (float*)d_scratch.p;
    f.nblk = (int)((nfft + 255) / 256);
    f.blk_v = (float*)d_blk.p;
    f.blk_i = (int*)d_blk.p + (size_t)S * f.nblk;
    wf_db_kernel<<<dim3((unsigned)f.nblk, (unsigned)S), 256, 0, st>>>(f);
    wf_finalize_kernel<<<S, 256, 0, st>>>(f);
    (*launches) += 2;
    CUDA_TRY(cudaGetLastError());
    return 0;
  }
};

}  // namespace pmr
