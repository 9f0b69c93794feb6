// fused_frontend_kernel: the WHOLE front end of a rate-2/3 plan in one pass, nothing stored in between --
//   cu8 load -> (u8 - 127.4)/128 -> DC blocker -> half-band m=3 -> m=5 -> m=10 -> 14-tap arbitrary resampler (x 2/3)
// i.e. iirfilt_crcf_execute_block + msresamp_crcf_execute of the reference for 2.4 Msps input
// (/root/reference/src/sdr_pmr446.c:795-796; SURVEY.md Appendix A.1-A.5), replacing round 1's two launches
// (cascade_kernel -> 600 kHz ring in HBM -> hbarb_tile_kernel) and their 9.8 GB of ring traffic per 1024-stream step.
//
// Same "segment-sequential" mapping as cascade_kernel (frontend.cuh): one thread = one time segment of one stream, run
// like the CPU does with every filter window in registers -- but
//  * all samples are (re, im) PAIRS in 64-bit register pairs and every FIR tap is ONE packed FFMA2 (Blackwell's
//    fma.rn.f32x2) with the tap as a scalar uniform-register operand: half the FMA instructions of the scalar form;
//  * an iteration is 48 input samples = three 16-sample sub-blocks through DC + the first two half-bands, then 12 samples
//    at 600 kHz -> 6 at 300 kHz -> 4 resampler outputs (one 32-byte sector, one 256-bit store).  The resampler phase has
//    period 2 (step = 1.5): outputs 2q, 2q + 1 come from inputs 3q, 3q + 1 with the two filter-bank rows as
//    constant-bank operands -- no bank gathers, no phase arithmetic;
//  * raw bytes travel global -> shared memory by cp.async FF_CPD sub-blocks ahead of their use (no registers in flight).
// The DC blocker runs in its zero-state form (DC_ZSR, see frontend.cuh); the zero-input part is added by the consumer of
// the 200 kHz ring (channelize16_kernel while it stages its tile) or in place by zir_tail_kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "frontend.cuh"
#include "packed_f32.cuh"

namespace pmr {

constexpr int FF_THREADS = 128;

struct FusedParams {
  CascadeParams c;       // source view, segment grid, DC blocker, destination ring, hb[0..2] = taps of m = 3, 5, 10
  float arb[2][14];      // filter-bank rows of the two resampler phases, newest first
  float w0;              // DC blocker state (X units) of a stream that has been silent for ever: CU8_XBIAS / alpha
};

// one half-band decimator stage on pairs: out[o] = x_odd[o - M] + sum_{j < 2M} h[j] x_even[o - j]   (A.4)
template <int M, int B>
struct HbPair {
  float2 he[2 * M - 1], ho[M];   // previous even / odd samples, oldest first
  __device__ __forceinline__ void reset() {
#pragma unroll
    for (int i = 0; i < 2 * M - 1; i++) he[i] = make_float2(0.0f, 0.0f);
#pragma unroll
    for (int i = 0; i < M; i++) ho[i] = make_float2(0.0f, 0.0f);
  }
  template <bool SCALE>
  __device__ __forceinline__ void run(const float* h, const float2* x, float2* y, float scale) {
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
      for (int j = 0; j < 2 * M; j++) acc = fma_tap(h[j], e[2 * M - 1 + b - j], acc);   // h points into the kernel parameters
      y[b] = SCALE ? fmul2(acc, make_float2(scale, scale)) : acc;
    }
#pragma unroll
    for (int i = 0; i < 2 * M - 1; i++) he[i] = e[B + i];
#pragma unroll
    for (int i = 0; i < M; i++) ho[i] = o[B + i];
  }
};

// cu8 -> X = u8 - 127 as an exact small integer (one PRMT per byte + one packed FADD2 per sample).  The sample itself is
// x = X / 128 + c0' with c0' = -(fl(127.4) - 127) / 128, both exactly representable, and everything after it is linear:
// the 1 / 128 rides on the kernel's final power-of-two scale (exact), and the constant c0' is what the DC blocker removes
// -- in X units "x was zero for ever" is the blocker state W = CU8_XBIAS / alpha instead of 0, which is where the segment
// that starts at the head of a stream starts (FusedParams::w0); every other segment starts from zero state as before and
// the affine scan carries the difference.  With V_X(0) = w0 the true state is exactly v = V_X / 128 + c0' / alpha, so the
// zero-input term the consumers add is -alpha (V_X / 128) E[k]: DcScanParams::unit_scale, nothing else changes.
// One FMA-pipe instruction per sample less than converting to x itself (7.5 % of the fused kernel's FMA work).
constexpr float CU8_XBIAS = 127.40000152587890625f - 127.0f;   // X of a zero-valued ("no sample") x
__device__ __forceinline__ float2 cu8_pair_x(unsigned w, int k) {
  const float2 raw = make_float2(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540u + (unsigned)(2 * k))),
                                 __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540u + (unsigned)(2 * k + 1))));
  return fadd2(raw, make_float2(-8388735.0f, -8388735.0f));    // -(2^23 + 127)
}

constexpr int FF_G = 48;        // input samples per iteration
constexpr int FF_SUB = 16;      // ... in three sub-blocks of 16 (32 bytes of cu8)
constexpr int FF_D = 8;         // decimation of the three half-bands
constexpr int FF_NO = 4;        // resampler outputs per iteration

// Every history lives in registers (~250 registers, 2 blocks per SM); keeping the m = 10 and resampler histories in shared
// memory instead (167 registers, 3 blocks per SM) measured 2.75 ms against 2.68 ms (1024 streams): occupancy is not what
// limits this kernel.
// The raw bytes travel global -> shared memory with cp.async, FF_CPD sub-blocks ahead (thread-private 32-byte slots, no
// registers in flight).  Register loads two sub-blocks ahead behind an L1 prefetch arrived late: ptxas sinks them to
// within ~300 instructions of their use (5 % of the kernel's stall samples on the first PRMT of a sub-block; l1tex hit
// rate 10 %: the L1 prefetch does not hold).
constexpr int FF_CPD = 6;
// src_bytes = 0 reads nothing and zero-fills: the guard costs no branch, the iteration stays ONE basic block
__device__ __forceinline__ void cp_async16(unsigned smem, const void* gmem, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ uint4 lds128_v(unsigned smem) {   // volatile: stays behind the wait_group in front of it
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem));
  return v;
}
// The DC blocker always runs, in X units (cu8_pair_x): the host folds 1 / 128 into p.scale.
static __global__ void __launch_bounds__(FF_THREADS, 2) fused_frontend_kernel(FusedParams fp) {
  extern __shared__ __align__(16) char ff_stage[];   // FF_CPD x 32 bytes per thread
  const CascadeParams& p = fp.c;
  long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)p.n_streams * p.nseg) return;
  const int s = (int)(gid / p.nseg), t = (int)(gid % p.nseg);
  const long long T0 = p.seg0 + (long long)t * p.seg_len;
  long long i_lo = T0 / FF_D, i_hi = (T0 + p.seg_len) / FF_D;     // owned 300 kHz samples
  if (i_lo < p.out0) i_lo = p.out0;
  if (i_hi > p.out1) i_hi = p.out1;
  long long qb = T0 - p.halo;
  long long q_cap = qb + p.seg_len;                               // where this segment's local DC sum is complete
  if (q_cap > p.dc_end) q_cap = p.dc_end;
  if (qb < 0) qb = 0;
  long long q_end = i_hi > i_lo ? i_hi * FF_D : qb;
  if (q_cap > q_end) q_end = q_cap;
  if (q_end <= qb) {
    p.sums[gid] = make_float2(0.0f, 0.0f);
    return;
  }
  // everything below is 32-bit and relative to qb (a multiple of 48: every iteration starts at resampler phase 0)
  const int n_it = (int)((q_end - qb + FF_G - 1) / FF_G);
  const int cap_it = q_cap > qb ? (int)((q_cap - qb) / FF_G) : 0;
  const long long ob = qb / FF_D;                                  // absolute 300 kHz index of local sample 0
  int own_lo = (int)(i_lo - ob), own_hi = (int)(i_hi - ob);
  if (i_hi <= i_lo) own_lo = own_hi = 0;

  HbPair<3, FF_SUB / 2> sa;
  HbPair<5, FF_SUB / 4> sb;
  HbPair<10, FF_G / 8> sc;
  sa.reset(); sb.reset(); sc.reset();
  float2 aw[13];                                                   // resampler window: previous 300 kHz samples, oldest first
#pragma unroll
  for (int i = 0; i < 13; i++) aw[i] = make_float2(0.0f, 0.0f);
  float2 v = make_float2(0.0f, 0.0f);                              // DC blocker state (zero-state response)
  if (T0 - p.halo <= 0) v = make_float2(fp.w0, fp.w0);             // head of the stream: see cu8_pair_x

  float2* dst = p.dst + (long long)s * p.dst_stride;
  const unsigned dmask = (unsigned)p.dst_mask;
  const unsigned jb32 = (unsigned)(qb / 12);                       // ring index of local resampler output 0 (multiple of 4)
  const float scale = p.scale;
  const float2 nalpha = make_float2(-p.alpha, -p.alpha);

  Loader<SRC_CU8> ld;
  ld.template init<FF_SUB>(p.src, s, qb);
  Raw<SRC_CU8, FF_SUB> raw[3];
  // slot k of the thread = two 16-byte pieces at stage[(2 k + h) * blockDim.x + threadIdx.x]; sub-block sbi uses slot
  // sbi mod FF_CPD = 3 (it & 1) + sub.  One commit group per sub-block step (empty when the sub-block is not a whole aligned
  // group of the chunk), so "all but the newest FF_CPD - 1 groups" is always the group of the sub-block about to be read.
  const unsigned stage = (unsigned)__cvta_generic_to_shared(ff_stage) + 16u * threadIdx.x, spitch = 16u * blockDim.x;
  const uint8_t* const cp_dummy = (const uint8_t*)((uintptr_t)ld.cur & ~(uintptr_t)31);
  auto cp_issue = [&](int sbi, int slot) {
    const bool ok = sbi >= ld.fast_lo && sbi < ld.fast_hi;
    const uint8_t* g = ok ? ld.fp + (size_t)sbi * (2 * FF_SUB) : cp_dummy;   // zero-size copy: never read, but the address stays 16-byte aligned
    cp_async16(stage + (unsigned)(2 * slot) * spitch, g, ok ? 16 : 0);
    cp_async16(stage + (unsigned)(2 * slot + 1) * spitch, g + 16, ok ? 16 : 0);
    asm volatile("cp.async.commit_group;");
  };
  auto cp_take = [&](int sbi, int slot, Raw<SRC_CU8, FF_SUB>& r) {
    asm volatile("cp.async.wait_group %0;" ::"n"(FF_CPD - 1));
    const uint4 a = lds128_v(stage + (unsigned)(2 * slot) * spitch), b = lds128_v(stage + (unsigned)(2 * slot + 1) * spitch);
    r.w[0] = a.x; r.w[1] = a.y; r.w[2] = a.z; r.w[3] = a.w; r.w[4] = b.x; r.w[5] = b.y; r.w[6] = b.z; r.w[7] = b.w;
  };
#pragma unroll
  for (int i = 0; i < FF_CPD; i++) cp_issue(i, i);
  const float2 cpole = make_float2(1.0f - p.alpha, 1.0f - p.alpha);   // exact: alpha is 1 - fl(1 - alpha_nominal)

  // One iteration = 48 input samples.  FAST: all three sub-blocks are whole aligned 32-byte groups of the current chunk --
  // straight-line code (one basic block, so the scheduler overlaps the DC recurrence of one sub-block with the FIR work
  // of another); otherwise the guarded per-sample loader fills the same registers.
  auto iteration = [&](const int it, auto fast_tag) {
    constexpr bool FAST = decltype(fast_tag)::value;
    float2 cin[12];                                                // 600 kHz samples of this iteration
#pragma unroll
    for (int sub = 0; sub < 3; sub++) {
      const int sbi = 3 * it + sub;
      const int slot = 3 * (it & 1) + sub;
      cp_take(sbi, slot, raw[sub]);
      float2 x[FF_SUB];
      if (FAST) {
#pragma unroll
        for (int j = 0; j < FF_SUB / 2; j++) {
          x[2 * j] = cu8_pair_x(raw[sub].w[j], 0);
          x[2 * j + 1] = cu8_pair_x(raw[sub].w[j], 1);
        }
      } else {
        float xr[FF_SUB], xi[FF_SUB];
        ld.template convert<FF_SUB>(p.src, qb + (long long)sbi * FF_SUB, sbi, raw[sub], xr, xi);
#pragma unroll
        for (int i = 0; i < FF_SUB; i++)   // X = (x - c0') * 128, exact (a sample) or CU8_XBIAS (a zero: before the stream start)
          x[i] = make_float2(fmaf(xr[i], 128.0f, CU8_XBIAS), fmaf(xi[i], 128.0f, CU8_XBIAS));
      }
      cp_issue(sbi + FF_CPD, slot);   // refill the slot just emptied (its words are in x by now)
      // A.1 dc blocker, zero-state part: y = x - alpha v[n-1], v[n] = (1 - alpha) v[n-1] + x.  Only the one-FFMA2
      // recurrence of v is serial; the outputs hang off it.
#pragma unroll
      for (int i = 0; i < FF_SUB; i++) {
        const float2 y = ffma2(nalpha, v, x[i]);
        v = ffma2(cpole, v, x[i]);
        x[i] = y;
      }
      float2 a[FF_SUB / 2], b[FF_SUB / 4];
      sa.template run<false>(p.hb[0], x, a, 1.0f);
      sb.template run<false>(p.hb[1], a, b, 1.0f);
#pragma unroll
      for (int i = 0; i < 4; i++) cin[4 * sub + i] = b[i];
    }
    float2 c[6];                                                   // 300 kHz, scaled by 2^-3 like msresamp2 does
    sc.template run<true>(p.hb[2], cin, c, scale);
    // arbitrary resampler (A.5), phase period 2: outputs 4 it + {0, 1, 2, 3} sit at local inputs 6 it + {0, 1, 3, 4}
    float2 w[13 + 6];
#pragma unroll
    for (int i = 0; i < 13; i++) w[i] = aw[i];
#pragma unroll
    for (int i = 0; i < 6; i++) w[13 + i] = c[i];
    float2 o[4];
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const int io = 3 * (r / 2) + (r % 2);
      float2 acc = make_float2(0.0f, 0.0f);
#pragma unroll
      for (int k = 0; k < 14; k++) acc = fma_tap(fp.arb[r % 2][k], w[13 + io - k], acc);
      o[r] = acc;
    }
#pragma unroll
    for (int i = 0; i < 13; i++) aw[i] = w[6 + i];

    const int lo = own_lo - 6 * it, hi = own_hi - 6 * it;          // owned local inputs of this iteration are [lo, hi)
    float2* d4 = dst + ((jb32 + 4u * (unsigned)it) & dmask);       // 32-byte aligned, never straddles the ring's end
    if (lo <= 0 && hi >= 5) {
      const float f[8] = {o[0].x, o[0].y, o[1].x, o[1].y, o[2].x, o[2].y, o[3].x, o[3].y};
      stg256(d4, f);
    } else if (hi > 0 && lo < 5) {
#pragma unroll
      for (int r = 0; r < 4; r++) {
        const int io = 3 * (r / 2) + (r % 2);
        if (io >= lo && io < hi) d4[r] = o[r];
      }
    }
  };
  for (int it = 0; it < n_it; it++) {
    if (it == cap_it) p.sums[gid] = v;
    if (3 * it >= ld.fast_lo && 3 * it + 2 < ld.fast_hi) iteration(it, std::true_type());
    else iteration(it, std::false_type());
  }
  if (cap_it >= n_it) p.sums[gid] = v;
}

// ---- front6_kernel: the first SIX half-band stages of a deep plan in one pass (dsd_in: 2.4 Msps -> 37.5 kHz, /root/reference/
// src/dsd_in.c:167-168 with msresamp's stage list 3,3,3,3,3,5,10 or 3,3,3,3,5,10) -------------------------------------------------
// Same structure as fused_frontend_kernel: iteration = 64 input samples = four 16-sample sub-blocks through cvt + DC + two m=3
// stages, then 16 -> 8 -> 4 -> 2 -> 1 samples through the other four.  Replaces cascade_kernel<cu8, DC_ZSR, 16, 3,3,3,3> (whose
// 16-sample iterations spend more instructions moving the late stages' windows than filtering) AND the launch after it.
struct Front6Params {
  CascadeParams c;      // c.hb[0..3] = taps of stages 1-4 (all m = 3)
  float hb5[20], hb6[20];
  float w0;             // as FusedParams::w0
};
constexpr int F6_G = 64, F6_D = 64;

constexpr int F6_CPD = 8;   // cp.async depth in sub-blocks (two iterations), see fused_frontend_kernel
template <int ME, int MF>
__global__ void __launch_bounds__(FF_THREADS, 2) front6_kernel(Front6Params fp) {
  extern __shared__ __align__(16) char f6_stage[];   // F6_CPD x 32 bytes per thread
  const CascadeParams& p = fp.c;
  long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)p.n_streams * p.nseg) return;
  const int s = (int)(gid / p.nseg), t = (int)(gid % p.nseg);
  const long long T0 = p.seg0 + (long long)t * p.seg_len;
  long long i_lo = T0 / F6_D, i_hi = (T0 + p.seg_len) / F6_D;
  if (i_lo < p.out0) i_lo = p.out0;
  if (i_hi > p.out1) i_hi = p.out1;
  long long qb = T0 - p.halo;
  long long q_cap = qb + p.seg_len;
  if (q_cap > p.dc_end) q_cap = p.dc_end;
  if (qb < 0) qb = 0;
  long long q_end = i_hi > i_lo ? i_hi * F6_D : qb;
  if (q_cap > q_end) q_end = q_cap;
  if (q_end <= qb) {
    p.sums[gid] = make_float2(0.0f, 0.0f);
    return;
  }
  const int n_it = (int)((q_end - qb + F6_G - 1) / F6_G);
  const int cap_it = q_cap > qb ? (int)((q_cap - qb) / F6_G) : 0;
  const long long ob = qb / F6_D;
  int own_lo = (int)(i_lo - ob), own_hi = (int)(i_hi - ob);
  if (i_hi <= i_lo) own_lo = own_hi = 0;

  HbPair<3, 8> sa;
  HbPair<3, 4> sb;
  HbPair<ME, 2> se;
  HbPair<MF, 1> sf;
  sa.reset(); sb.reset(); se.reset(); sf.reset();
  float2 v = make_float2(0.0f, 0.0f);   // DC blocker state in X units, see cu8_pair_x
  if (T0 - p.halo <= 0) v = make_float2(fp.w0, fp.w0);
  float2* dst = p.dst + (long long)s * p.dst_stride;
  const unsigned dmask = (unsigned)p.dst_mask, ob32 = (unsigned)ob;
  const float scale = p.scale;
  const float2 nalpha = make_float2(-p.alpha, -p.alpha), cpole = make_float2(1.0f - p.alpha, 1.0f - p.alpha);

  Loader<SRC_CU8> ld;
  ld.template init<FF_SUB>(p.src, s, qb);
  Raw<SRC_CU8, FF_SUB> raw[4];
  const unsigned stage = (unsigned)__cvta_generic_to_shared(f6_stage) + 16u * threadIdx.x, spitch = 16u * blockDim.x;
  const uint8_t* const cp_dummy = (const uint8_t*)((uintptr_t)ld.cur & ~(uintptr_t)31);
  auto cp_issue = [&](int sbi, int slot) {
    const bool ok = sbi >= ld.fast_lo && sbi < ld.fast_hi;
    const uint8_t* g = ok ? ld.fp + (size_t)sbi * (2 * FF_SUB) : cp_dummy;   // zero-size copy: never read, but the address stays 16-byte aligned
    cp_async16(stage + (unsigned)(2 * slot) * spitch, g, ok ? 16 : 0);
    cp_async16(stage + (unsigned)(2 * slot + 1) * spitch, g + 16, ok ? 16 : 0);
    asm volatile("cp.async.commit_group;");
  };
  auto cp_take = [&](int slot, Raw<SRC_CU8, FF_SUB>& r) {
    asm volatile("cp.async.wait_group %0;" ::"n"(F6_CPD - 1));
    const uint4 a = lds128_v(stage + (unsigned)(2 * slot) * spitch), b = lds128_v(stage + (unsigned)(2 * slot + 1) * spitch);
    r.w[0] = a.x; r.w[1] = a.y; r.w[2] = a.z; r.w[3] = a.w; r.w[4] = b.x; r.w[5] = b.y; r.w[6] = b.z; r.w[7] = b.w;
  };
#pragma unroll
  for (int i = 0; i < F6_CPD; i++) cp_issue(i, i);

  HbPair<3, 4> sc4;   // stages 3 and 4 run per HALF iteration (32 inputs): shorter live ranges than 16-sample staging arrays
  HbPair<3, 2> sd2;
  sc4.reset(); sd2.reset();
  auto iteration = [&](const int it, auto fast_tag) {
    constexpr bool FAST = decltype(fast_tag)::value;
    float2 d[4];
#pragma unroll
    for (int half = 0; half < 2; half++) {
      float2 cin[8];
#pragma unroll
      for (int s2 = 0; s2 < 2; s2++) {
        const int sub = 2 * half + s2;
        const int sbi = 4 * it + sub;
        const int slot = 4 * (it & 1) + sub;
        cp_take(slot, raw[sub]);
        float2 x[FF_SUB];
        if (FAST) {
#pragma unroll
          for (int j = 0; j < FF_SUB / 2; j++) {
            x[2 * j] = cu8_pair_x(raw[sub].w[j], 0);
            x[2 * j + 1] = cu8_pair_x(raw[sub].w[j], 1);
          }
        } else {
          float xr[FF_SUB], xi[FF_SUB];
          ld.template convert<FF_SUB>(p.src, qb + (long long)sbi * FF_SUB, sbi, raw[sub], xr, xi);
#pragma unroll
          for (int i = 0; i < FF_SUB; i++)
            x[i] = make_float2(fmaf(xr[i], 128.0f, CU8_XBIAS), fmaf(xi[i], 128.0f, CU8_XBIAS));
        }
        cp_issue(sbi + F6_CPD, slot);
#pragma unroll
        for (int i = 0; i < FF_SUB; i++) {
          const float2 y = ffma2(nalpha, v, x[i]);
          v = ffma2(cpole, v, x[i]);
          x[i] = y;
        }
        float2 a[8], b[4];
        sa.template run<false>(p.hb[0], x, a, 1.0f);
        sb.template run<false>(p.hb[1], a, b, 1.0f);
#pragma unroll
        for (int i = 0; i < 4; i++) cin[4 * s2 + i] = b[i];
      }
      float2 c[4], dd[2];
      sc4.template run<false>(p.hb[2], cin, c, 1.0f);
      sd2.template run<false>(p.hb[3], c, dd, 1.0f);
      d[2 * half] = dd[0];
      d[2 * half + 1] = dd[1];
    }
    float2 e[2], f[1];
    se.template run<false>(fp.hb5, d, e, 1.0f);
    sf.template run<true>(fp.hb6, e, f, scale);
    if (it >= own_lo && it < own_hi) dst[(ob32 + (unsigned)it) & dmask] = f[0];
  };
  for (int it = 0; it < n_it; it++) {
    if (it == cap_it) p.sums[gid] = v;
    if (4 * it >= ld.fast_lo && 4 * it + 3 < ld.fast_hi) iteration(it, std::true_type());
    else iteration(it, std::false_type());
  }
  if (cap_it >= n_it) p.sums[gid] = v;
}

}  // namespace pmr
