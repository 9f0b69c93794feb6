// Host-side owner of the front end: plans the multi-stage resampler as a short chain of
// cascade_kernel launches, keeps the rings / raw history / DC-blocker carry, and turns one
// execute() call into launches using closed-form absolute sample counts.  Device counterpart of
// iirfilt_crcf + msresamp_crcf (/root/reference/src/sdr_pmr446.c:422-428,795-796;
// src/dsd_in.c:97-101,167-168; SURVEY.md Appendix A.1-A.5).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "common_host.hpp"
#include "design.hpp"
#include "frontend.cuh"
#include "frontend_fused.cuh"
#include "hbarb_tile.cuh"

namespace pmr {

typedef void (*cascade_fn)(CascadeParams);

// One cascade launch: a run of half-band stages (execution order, highest rate first), optionally
// preceded by the DC blocker and followed by the arbitrary resampler.
struct Level {
  int src = SRC_RING;
  int dc = DC_NONE;
  bool arb = false;
  int ms[6] = {0, 0, 0, 0, 0, 0};
  int nst = 0, D = 1, G = 16, unit = 16, halo = 0, seg_len = 1024;
  float hb[6][20];
  float scale = 1.0f;
  cascade_fn fn = nullptr;
  bool tile = false;      // last level runs hbarb_tile_kernel<10, 2, 3> instead of the segment-sequential cascade
  bool fused = false;     // the only level: fused_frontend_kernel (cu8 -> m = 3, 5, 10 -> resampler x 2/3) in one pass
  bool front6 = false;    // level 0 of a deep plan: front6_kernel (cu8 -> six half-bands) in one pass
  float arb_rows[2][14];
  DevBuf ring;            // output ring [S][cap] float2
  long long cap = 0;
  long long n_in = 0, n_out = 0;   // absolute counts: inputs seen, outputs written
  long long max_in = 0, max_out = 0;  // per chunk
};

template <int SRC, int DC, int G, int A, int B, int C, int D, bool ARB>
static cascade_fn cfn() { return cascade_kernel<SRC, DC, G, A, B, C, D, ARB>; }

// Instantiated stage combinations.  msresamp's half-band design (A.3) always yields semi-lengths 3, ..., 3, 5, 10 in
// execution order, so the groups below ([3,3,3,3], [3,3], [3,5], [3], [5,10], [5], [10] without resampler; [10] / none with it)
// tile ANY decimating plan: Frontend::init() cuts the stage list greedily into them.
inline cascade_fn pick_cascade(int src, int dc, bool arb, const int* ms, int* G) {
  auto is = [&](int a, int b, int c, int d) { return ms[0] == a && ms[1] == b && ms[2] == c && ms[3] == d; };
  *G = 16;
#define PMR_GROUPS(SRC, DC)                                                         \
  if (is(5, 0, 0, 0)) return cfn<SRC, DC, 16, 5, 0, 0, 0, false>();                 \
  if (is(5, 10, 0, 0)) return cfn<SRC, DC, 16, 5, 10, 0, 0, false>();               \
  if (is(3, 5, 0, 0)) return cfn<SRC, DC, 16, 3, 5, 0, 0, false>();                 \
  if (is(3, 0, 0, 0)) return cfn<SRC, DC, 16, 3, 0, 0, 0, false>();                 \
  if (is(3, 3, 0, 0)) return cfn<SRC, DC, 16, 3, 3, 0, 0, false>();                 \
  if (is(3, 3, 3, 3)) return cfn<SRC, DC, 16, 3, 3, 3, 3, false>();   \
  if (is(10, 0, 0, 0)) return cfn<SRC, DC, 16, 10, 0, 0, 0, false>();
  if (!arb) {
    if (dc == DC_ZSR && src == SRC_CU8) { PMR_GROUPS(SRC_CU8, DC_ZSR) }
    if (dc == DC_ZSR && src == SRC_CF32) { PMR_GROUPS(SRC_CF32, DC_ZSR) }
    if (dc == DC_ZSR && src == SRC_CS16) { PMR_GROUPS(SRC_CS16, DC_ZSR) }
    if (dc == DC_ZSR && src == SRC_CS8) { PMR_GROUPS(SRC_CS8, DC_ZSR) }
    if (dc == DC_NONE && src == SRC_CF32) { PMR_GROUPS(SRC_CF32, DC_NONE) }   // stand-alone msresamp_crcf (liquid shim): no DC blocker
    if (dc == DC_NONE && src == SRC_RING) { PMR_GROUPS(SRC_RING, DC_NONE) }
  } else {
    if (dc == DC_NONE && src == SRC_RING && is(10, 0, 0, 0)) { *G = 8; return cfn<SRC_RING, DC_NONE, 8, 10, 0, 0, 0, true>(); }
    if (dc == DC_NONE && src == SRC_RING && is(0, 0, 0, 0)) { *G = 8; return cfn<SRC_RING, DC_NONE, 8, 0, 0, 0, 0, true>(); }
    if (dc == DC_SCAN && src == SRC_CU8 && is(0, 0, 0, 0)) return cfn<SRC_CU8, DC_SCAN, 16, 0, 0, 0, 0, true>();
    if (dc == DC_SCAN && src == SRC_CF32 && is(0, 0, 0, 0)) return cfn<SRC_CF32, DC_SCAN, 16, 0, 0, 0, 0, true>();
    if (dc == DC_SCAN && src == SRC_CS16 && is(0, 0, 0, 0)) return cfn<SRC_CS16, DC_SCAN, 16, 0, 0, 0, 0, true>();
    if (dc == DC_SCAN && src == SRC_CS8 && is(0, 0, 0, 0)) return cfn<SRC_CS8, DC_SCAN, 16, 0, 0, 0, 0, true>();
    if (dc == DC_NONE && src == SRC_CF32 && is(0, 0, 0, 0)) return cfn<SRC_CF32, DC_NONE, 16, 0, 0, 0, 0, true>();
  }
#undef PMR_GROUPS
  return nullptr;
}

// Cuts an execution-order stage list (3, ..., 3, 5 [, 10]) into instantiated groups, longest first.
inline bool cut_groups(std::vector<int> order, std::vector<std::vector<int>>* groups) {
  static const std::vector<std::vector<int>> known = {{3, 3, 3, 3}, {5, 10}, {3, 5}, {3, 3}, {3}, {5}, {10}};
  size_t i = 0;
  while (i < order.size()) {
    bool hit = false;
    for (const auto& k : known) {
      if (i + k.size() > order.size() || !std::equal(k.begin(), k.end(), order.begin() + i)) continue;
      // [3, 5] would strand a following 3-run; it only matches at the end of the 3s by construction (5 follows the 3s)
      groups->push_back(k);
      i += k.size();
      hit = true;
      break;
    }
    if (!hit) return false;
  }
  return true;
}

struct Frontend {
  // How a plan is cut into launches (pure host logic, also exported through pmr446_describe_frontend for the CPU tests):
  // groups[0 .. n-2] are half-band groups, groups[n-1] is the resampler's launch (with the last half-band, or empty).
  static int plan_groups(const design::MsresampPlan& plan, int in_fmt, std::vector<std::vector<int>>* groups, bool* fused, bool* front6 = nullptr) {
    if (front6) *front6 = false;
    // execution-order stage list: plan.m[stages-1] runs first
    std::vector<int> order;
    for (int g = (int)plan.stages - 1; g >= 0; g--) order.push_back((int)plan.m[g]);
    std::vector<int> last;
    // Two-stage plans whose resampler phase is not periodic (1.024 Msps -> 200 kHz: [5, 10], step 21 474 836): both
    // half-bands run in the first launch and the last one is the resampler alone -- the ring between them then sits at
    // the lowest rate (half the traffic) and the per-lane filter-bank gathers no longer share a kernel with the 58-register
    // m = 10 window.  A single half-band also runs on its own (the resampler kernel with a half-band only reads a ring).
    // Otherwise the last half-band goes with the resampler (tiled kernel when the phase has period 2).
    // (The two launches measured 1.35 + 1.14 ms at 1024 x 1.024 Msps against 0.57 + 2.34 ms for ONE launch of [5, 10] +
    // resampler behind a DC pre-pass over the raw input.)
    const bool split_arb = (order.size() == 2 && order[0] == 5 && order[1] == 10 && plan.step != (3u << 23)) || order.size() == 1;
    // cs16 and cs8 take the cf32 plans below: the fused and front6 kernels read cu8 only.
    // 2.4 Msps cu8 -> 200 kHz ([3, 5, 10] + rate 2/3): everything in ONE launch, no intermediate ring (frontend_fused.cuh)
    *fused = in_fmt == PMR446_FMT_CU8 && order.size() == 3 && order[0] == 3 && order[1] == 5 && order[2] == 10 && plan.step == (3u << 23);
    // deep cu8 plans (dsd_in: 3,3,3,3,3,5,10 at 2.4 Msps, 3,3,3,3,5,10 at 1.024 Msps): the first six stages in one launch
    const bool six = front6 && in_fmt == PMR446_FMT_CU8 && (order.size() == 6 || order.size() == 7) && order[0] == 3 && order[1] == 3 &&
                     order[2] == 3 && order[3] == 3 && ((order[4] == 3 && order[5] == 5) || (order[4] == 5 && order[5] == 10));
    if (*fused) {
      groups->push_back(order);
    } else if (six) {
      *front6 = true;
      groups->emplace_back(order.begin(), order.begin() + 6);
      groups->emplace_back(order.begin() + 6, order.end());   // [10] + resampler, or the resampler alone
    } else {
      if (!order.empty() && !split_arb) { last.push_back(order.back()); order.pop_back(); }
      if (!cut_groups(order, groups)) return fail(PMR446_EINVAL, "resampler plan not built: unexpected half-band stage list");
      groups->push_back(last);   // may be empty (rate >= 0.5)
    }
    return 0;
  }

  int S = 0, fmt = 0;
  bool dc = true;
  float alpha = 0.0f, alpha_eff = 0.0f, c_pole = 1.0f;
  design::MsresampPlan plan;
  std::vector<Level> levels;
  // level-0 raw history (two buffers, swapped every call)
  DevBuf hist[2];
  int hist_cur = 0;
  long long hist_base = 0;
  int hist_cap = 0;       // samples
  int bps = 8;            // bytes per input sample
  // DC blocker carry (A.1): V at (segment 0 start - halo) of the next chunk
  DevBuf v_lag, sums, v_seg, e_table;
  int max_seg0 = 0;
  DevBuf pfb;
  long long n_in = 0;     // raw samples consumed so far
  struct OutView { void* p; } out;   // final ring (levels.back())
  long long out_cap = 0, n_out = 0;
  unsigned max_chunk = 0;
  // A fused level leaves the DC blocker's zero-input part of the samples [pending.from, n_out) of the OUT ring to its
  // consumer (see execute(defer_zir)); tail_fix = how much history the ring keeps for the next call
  Correction pending;
  bool has_pending = false;
  long long tail_fix = 0;

  long long max_out_per_chunk() const { return levels.empty() ? 0 : levels.back().max_out; }
  // resampler outputs that exist once n_total raw samples have been consumed (closed form, A.2/A.5): lets the callers
  // validate their output buffers BEFORE execute() advances any state
  long long outputs_after(long long n_total) const {
    return (long long)design::arb_outputs_after((uint64_t)(n_total >> plan.stages), plan.step);
  }

  // E[k]: response of level 0's stage chain (zero state) to the sequence c^i, i >= 0, in float64
  std::vector<float> zir_table(const Level& L) const {
    const int n_in = L.halo + L.seg_len;
    std::vector<double> x(n_in);
    double v = 1.0;
    for (int i = 0; i < n_in; i++) { x[i] = v; v *= (double)c_pole; }
    for (int k = 0; k < L.nst; k++) {
      const int m = L.ms[k];
      std::vector<double> y(x.size() / 2);
      for (size_t o = 0; o < y.size(); o++) {
        const long long d = 2 * (long long)o + 1 - 2 * m;
        double acc = d >= 0 ? x[d] : 0.0;
        for (int j = 0; j < 2 * m; j++) {
          const long long e = 2 * (long long)o - 2 * j;
          if (e >= 0) acc += (double)L.hb[k][j] * x[e];
        }
        y[o] = acc;
      }
      x.swap(y);
    }
    for (auto& xv : x) xv *= (double)L.scale;
    if (L.fused) {   // ... followed by the arbitrary resampler (A.5): output j sits at input (j step) >> 24
      std::vector<double> y;
      for (uint64_t j = 0;; j++) {
        const uint64_t ph = j * (uint64_t)plan.step, pos = ph >> 24;
        if (pos >= x.size()) break;
        const unsigned row = (unsigned)((ph & ((1u << 24) - 1)) >> (24 - plan.bits));
        double acc = 0.0;
        for (unsigned k = 0; k < plan.sub_len && k <= pos; k++) acc += (double)plan.pfb[(size_t)row * plan.sub_len + k] * x[pos - k];
        y.push_back(acc);
      }
      x.swap(y);
    }
    std::vector<float> e(x.size());
    for (size_t i = 0; i < x.size(); i++) e[i] = (float)x[i];
    return e;
  }

  int init(int n_streams, int in_fmt, float rate, float as, bool with_dc, float dc_alpha, unsigned max_chunk_, long long extra_hist) {
    S = n_streams;
    fmt = in_fmt;
    dc = with_dc;
    alpha = dc_alpha;
    // liquid stores a1 = -1 + alpha rounded to float32 and computes y = v[n] - v[n-1] with
    // v[n] = x - a1 v[n-1]; the effective feedback is therefore 1 - fl(1 - alpha), not alpha.
    c_pole = 1.0f - alpha;
    alpha_eff = 1.0f - c_pole;
    max_chunk = max_chunk_;
    bps = fmt_bytes_per_sample(in_fmt);
    if (rate > 1.0f) return fail(PMR446_EINVAL, "front end only decimates (rate <= 1)");
    plan = design::msresamp_plan(rate, as);
    if (plan.sub_len != 14) return fail(PMR446_EINVAL, "arbitrary resampler kernel is specialised for 14 taps");
    if (plan.step < (1u << 24)) return fail(PMR446_EINVAL, "internal: decimating plan with arbitrary rate > 1");
    if (plan.bits > 8) return fail(PMR446_EINVAL, "resampler filter bank larger than 256 rows");
    std::vector<std::vector<int>> groups;   // pre-launch groups, then the arb launch
    bool want_fused = false, want_front6 = false;
    if (int rc = plan_groups(plan, in_fmt, &groups, &want_fused, &want_front6)) return rc;
    // the fused and front6 kernels always run the DC blocker (every caller that passes cu8 asks for it)
    if ((want_fused || want_front6) && !dc) return fail(PMR446_EINVAL, "internal: cu8 front end planned without the DC blocker");
    levels.resize(groups.size());
    long long max_in = max_chunk;
    int stage_cursor = (int)plan.stages - 1;  // index into plan.m / plan.hb of the next stage to place
    for (size_t l = 0; l < groups.size(); l++) {
      Level& L = levels[l];
      L.src = (l == 0) ? fmt_source(in_fmt) : SRC_RING;
      L.fused = want_fused;
      L.front6 = want_front6 && l == 0;
      L.dc = (l == 0 && dc) ? ((groups.size() >= 2 || L.fused) ? DC_ZSR : DC_SCAN) : DC_NONE;
      L.arb = (l + 1 == groups.size());
      L.nst = (int)groups[l].size();
      L.D = 1 << L.nst;
      memset(L.hb, 0, sizeof L.hb);
      int halo = 0;
      for (int k = 0; k < L.nst; k++) {
        L.ms[k] = groups[l][k];
        const std::vector<float>& t = plan.hb[stage_cursor];
        for (size_t j = 0; j < t.size(); j++) L.hb[k][j] = t[j];
        halo += (4 * L.ms[k] - 2 + 1) << k;
        stage_cursor--;
      }
      if (L.arb) halo += 14 * L.D;
      L.scale = 1.0f / (float)L.D;
      if (!L.fused && !L.front6) L.fn = pick_cascade(L.src, L.dc, L.arb, L.ms, &L.G);
      if (!L.fn && !L.fused && !L.front6) {
        char msg[160];
        snprintf(msg, sizeof msg, "resampler plan not built: level %zu src=%d dc=%d arb=%d stages=[%d,%d,%d,%d]", l, L.src, L.dc,
                 (int)L.arb, L.ms[0], L.ms[1], L.ms[2], L.ms[3]);
        return fail(PMR446_EINVAL, msg);
      }
      // segment granularity; a DC_ZSR producer aligns its grid to 16 ring samples so that the
      // consumer's groups never straddle two producer segments (Loader<SRC_RING> correction)
      L.unit = std::max(16, L.D);
      if (L.dc == DC_ZSR) L.unit = std::max(L.unit, 16 * L.D);
      L.halo = (halo + L.D + L.unit - 1) / L.unit * L.unit;
      // segment length: as long as possible while keeping >= ~150k threads in flight
      int seg = 4096;
      int seg_min = 256;
      while (seg_min < 4 * L.halo || seg_min < L.unit) seg_min <<= 1;
      while (seg > seg_min && (long long)S * ((max_in + seg - 1) / seg) < 148LL * 1024) seg >>= 1;
      L.seg_len = std::max(seg, seg_min);
      if (L.fused) {
        // every segment starts at resampler phase 0 on a 48-sample grid and holds 2^k resampler outputs (the consumer
        // finds its producer segment with a shift): seg_len = 12 * 2^k
        L.G = FF_G;
        L.unit = FF_G;
        L.halo = (halo + L.D + FF_G - 1) / FF_G * FF_G;
        int sl = 6144;
        while (sl > 1536 && (long long)S * ((max_in + sl - 1) / sl) < 148LL * 256) sl >>= 1;
        L.seg_len = sl;
        for (int r = 0; r < 2; r++) {
          const unsigned row = (unsigned)((((unsigned long long)r * plan.step) & ((1u << 24) - 1)) >> (24 - plan.bits));
          for (int k = 0; k < 14; k++) L.arb_rows[r][k] = plan.pfb[(size_t)row * plan.sub_len + k];
        }
      }
      if (L.front6) {   // long segments: the warm-up of six stages is 1024 samples
        L.G = F6_G;
        int sl = 16384;
        while (sl > 4096 && (long long)S * ((max_in + sl - 1) / sl) < 148LL * 256) sl >>= 1;
        L.seg_len = std::max(sl, seg_min);
      }
      if (L.arb && !L.fused) {
        // equal resampler phase at every segment start (all lanes of a warp then emit outputs in
        // lock-step) needs (seg_len / D) * 2^24 = 0 mod step
        unsigned long long g = plan.step, b = 1ull << 24;
        while (b) { unsigned long long tt = g % b; g = b; b = tt; }
        const unsigned long long k = plan.step / g;
        if (k > 1 && k <= 64) {
          const long long q = (long long)k * std::max(L.unit, L.D);
          L.seg_len = (int)std::max<long long>(q, L.seg_len / q * q);
        }
      }
      if (L.arb && L.src == SRC_RING && L.nst == 1 && L.ms[0] == 10 && plan.step == 3u << 23) {
        // rate 2/3: the resampler phase has period 2 -> tiled kernel; a call recomputes at most one tile, so the
        // producer ring must keep (and zir_tail_kernel must fix) that much corrected history
        L.tile = true;
        const int th = HT_R / 2 * 3 * HT_THREADS;
        L.halo = (2 * (th + HT_HH + 19) + L.unit - 1) / L.unit * L.unit;
        for (int r = 0; r < 2; r++) {
          const unsigned row = (unsigned)((((unsigned long long)r * plan.step) & ((1u << 24) - 1)) >> (24 - plan.bits));
          for (int k = 0; k < 14; k++) L.arb_rows[r][k] = plan.pfb[(size_t)row * plan.sub_len + k];
        }
        cudaFuncSetAttribute(hbarb_tile_kernel<10, 2, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hbarb_tile_smem<10, 2, 3>());
      }
      L.max_in = max_in;
      long long max_hb = max_in / L.D + 1;
      L.max_out = L.arb ? (long long)design::arb_outputs_after((uint64_t)max_hb, plan.step) + 2 : max_hb;
      long long need = L.max_out + 64 + (l + 1 < groups.size() ? 0 : extra_hist);
      if (l + 1 < groups.size()) need += 4096;  // next level's halo (checked below)
      L.cap = next_pow2(need);
      if (int rc = L.ring.alloc_zero((size_t)S * L.cap * sizeof(float2))) return rc;
      max_in = L.max_out;
    }
    for (size_t l = 1; l < levels.size(); l++)
      if (levels[l].halo + 64 > 4096) return fail(PMR446_EINVAL, "internal: halo exceeds ring slack");
    // arbitrary resampler bank, rows padded to 16 floats
    std::vector<float> rows((size_t)plan.npfb * 16, 0.0f);
    for (unsigned i = 0; i < plan.npfb; i++)
      for (unsigned k = 0; k < plan.sub_len; k++) rows[(size_t)i * 16 + k] = plan.pfb[(size_t)i * plan.sub_len + k];
    if (int rc = pfb.alloc(rows.size() * sizeof(float))) return rc;
    CUDA_TRY(cudaMemcpy(pfb.p, rows.data(), rows.size() * sizeof(float), cudaMemcpyHostToDevice));
    // raw history and DC carry
    Level& L0 = levels[0];
    hist_cap = L0.halo + L0.unit;
    for (int i = 0; i < 2; i++)
      if (int rc = hist[i].alloc_zero((size_t)S * hist_cap * bps)) return rc;
    max_seg0 = (int)((max_chunk + 2 * L0.unit + L0.seg_len - 1) / L0.seg_len) + 2;
    if (int rc = v_lag.alloc_zero((size_t)S * sizeof(float2))) return rc;
    if (int rc = sums.alloc_zero((size_t)S * max_seg0 * sizeof(float2))) return rc;
    if (int rc = v_seg.alloc_zero((size_t)S * max_seg0 * sizeof(float2))) return rc;
    tail_fix = extra_hist;
    if (L0.dc == DC_ZSR) {
      std::vector<float> e = zir_table(L0);
      if (int rc = e_table.alloc((e.size() + 16) * sizeof(float))) return rc;
      CUDA_TRY(cudaMemset(e_table.p, 0, e_table.bytes));
      CUDA_TRY(cudaMemcpy(e_table.p, e.data(), e.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    reset_counters();
    out.p = levels.back().ring.p;
    out_cap = levels.back().cap;
    return 0;
  }

  void reset_counters() {
    n_in = 0;
    n_out = 0;
    hist_cur = 0;
    hist_base = -(long long)levels[0].halo;
    for (auto& L : levels) L.n_in = L.n_out = 0;
  }
  // zeroes all state; asynchronous on the legacy stream: the caller synchronises the device before returning
  int reset() {
    reset_counters();
    for (auto& L : levels) CUDA_TRY(cudaMemset(L.ring.p, 0, L.ring.bytes));
    for (int i = 0; i < 2; i++) CUDA_TRY(cudaMemset(hist[i].p, 0, hist[i].bytes));
    CUDA_TRY(cudaMemset(v_lag.p, 0, v_lag.bytes));
    return 0;
  }

  // Consumes n raw samples per stream ([n_in, n_in + n)); afterwards n_out is the absolute
  // number of output samples in the `out` ring.
  // the cu8 kernels that run the DC recurrence on X = u8 - 127 (cu8_pair_x): sums / v_lag in X units, 1 / 128 in the scale
  static bool integer_units(const Level& L) { return L.dc == DC_ZSR && (L.fused || L.front6); }
  // few streams with many segments: one block per stream; otherwise one warp per stream
  void launch_dc_scan(const DcScanParams& sp, cudaStream_t st) const {
    if (S <= 64 && sp.nseg > 128) dc_scan_block_kernel<<<S, 256, 0, st>>>(sp);
    else dc_scan_kernel<<<(unsigned)(((long long)S * 32 + 127) / 128), 128, 0, st>>>(sp);
  }

  // defer_zir: the caller's consumer applies pending_corr() while it reads the ring and then calls fix_pending(false);
  // otherwise execute() finishes the ring itself (one extra read-modify-write pass over the new samples).
  const Correction* pending_corr() const { return has_pending ? &pending : nullptr; }
  void fix_pending(cudaStream_t st, int* launches, bool all, Timer* tm = nullptr) {
    if (!has_pending) return;
    has_pending = false;
    const Level& L = levels.back();
    const long long start = all ? pending.from : std::max(pending.from, L.n_out - tail_fix), count = L.n_out - start;
    if (count <= 0) return;
    zir_tail_kernel<<<dim3((unsigned)((count + 127) / 128), S), 128, 0, st>>>((float2*)L.ring.p, L.cap, L.cap - 1, pending, start, (int)count);
    *launches += 1;
    if (tm) tm->mark(st, TM_HIST);
  }

  int execute(const void* iq, long long iq_stride, unsigned n, cudaStream_t st, int* launches, Timer* tm = nullptr, bool defer_zir = false) {
    const long long n0 = n_in, n1 = n_in + n;
    has_pending = false;
    Timer dummy;
    if (!tm) tm = &dummy;
    SrcView v0;
    memset(&v0, 0, sizeof v0);
    v0.hist = hist[hist_cur].p;
    v0.hist_stride = (long long)hist_cap * bps;
    v0.hist_base = hist_base;
    v0.cur = iq;
    v0.cur_stride = iq_stride;
    v0.n0 = n0;
    v0.n1 = n1;
    // fast path: 256-bit vector loads straight from the caller's buffer
    v0.cur_aligned = (n0 % 16 == 0) && (((uintptr_t)iq) % 32 == 0) && (iq_stride % 32 == 0);

    Correction corr;               // set by a DC_ZSR level for its consumer
    memset(&corr, 0, sizeof corr);
    long long lvl_n0 = n0, lvl_n1 = n1;
    for (size_t l = 0; l < levels.size(); l++) {
      Level& L = levels[l];
      const long long seg0 = lvl_n0 / L.unit * L.unit, seg0_next = lvl_n1 / L.unit * L.unit;
      const long long out0 = lvl_n0 / L.D, out1 = lvl_n1 / L.D;
      long long span = (out1 > out0) ? out1 * L.D - seg0 : seg0_next - seg0;
      const int nseg = (int)((span + L.seg_len - 1) / L.seg_len);
      SrcView sv;
      if (l == 0) {
        sv = v0;
      } else {
        const Level& P = levels[l - 1];
        memset(&sv, 0, sizeof sv);
        sv.cur = P.ring.p;
        sv.cur_stride = P.cap * (long long)sizeof(float2);
        sv.n0 = lvl_n0;
        sv.n1 = lvl_n1;
        sv.ring_mask = P.cap - 1;
        sv.cur_aligned = 1;
        sv.corr = corr;
      }
      const long long threads = (long long)S * nseg;
      const unsigned blocks = (unsigned)((threads + 127) / 128);
      DcScanParams sp;
      if (L.dc != DC_NONE) {
        if (nseg > max_seg0) return fail(PMR446_ERANGE, "internal: segment count exceeds allocation");
        sp.n_streams = S;
        sp.nseg = nseg;
        sp.sums = (const float2*)sums.p;
        sp.v_seg = (float2*)v_seg.p;
        sp.v_lag = (float2*)v_lag.p;
        sp.p0 = seg0 - L.halo;
        sp.seg_len = L.seg_len;
        sp.end = seg0_next - L.halo;
        sp.c = c_pole;
        sp.decay_full = (float)pow((double)c_pole, (double)L.seg_len);
        sp.unit_scale = integer_units(L) ? 1.0f / 128.0f : 1.0f;
      }
      if (L.dc == DC_SCAN && nseg > 0) {   // V0 per segment up front: local sums, then the scan
        DcLocalParams dp;
        dp.src = sv;
        dp.n_streams = S;
        dp.nseg = nseg;
        dp.p0 = sp.p0;
        dp.seg_len = L.seg_len;
        dp.end = sp.end;
        dp.c = c_pole;
        dp.sums = (float2*)sums.p;
        if (L.src == SRC_CU8) dc_local_kernel<SRC_CU8><<<blocks, 128, 0, st>>>(dp);
        else if (L.src == SRC_CS16) dc_local_kernel<SRC_CS16><<<blocks, 128, 0, st>>>(dp);
        else if (L.src == SRC_CS8) dc_local_kernel<SRC_CS8><<<blocks, 128, 0, st>>>(dp);
        else dc_local_kernel<SRC_CF32><<<blocks, 128, 0, st>>>(dp);
        launch_dc_scan(sp, st);
        *launches += 2;
        tm->mark(st, TM_DC);
      }
      long long new_out = L.n_out;
      if (L.tile) {
        const long long j0 = L.n_out, j1 = out1 > out0 ? (long long)design::arb_outputs_after((uint64_t)out1, plan.step) : L.n_out;
        if (j1 > j0) {
          HbArbParams hp;
          memset(&hp, 0, sizeof hp);
          hp.ring = (const float2*)sv.cur;
          hp.ring_stride = levels[l - 1].cap;
          hp.ring_mask = sv.ring_mask;
          hp.n1 = lvl_n1;
          hp.corr = sv.corr;
          hp.n_streams = S;
          hp.tile0 = j0 / HT_TJ;
          hp.tiles = (int)((j1 + HT_TJ - 1) / HT_TJ - hp.tile0);
          hp.j0 = j0;
          hp.j1 = j1;
          hp.scale = L.scale;
          memcpy(hp.hb, L.hb[0], sizeof hp.hb);
          memcpy(hp.arb, L.arb_rows, sizeof hp.arb);
          hp.dst = (float2*)L.ring.p;
          hp.dst_stride = L.cap;
          hp.dst_mask = L.cap - 1;
          hbarb_tile_kernel<10, 2, 3><<<(unsigned)((long long)S * hp.tiles), HT_THREADS, hbarb_tile_smem<10, 2, 3>(), st>>>(hp);
          *launches += 1;
          tm->mark(st, TM_CASCADE0 + (int)std::min<size_t>(l, 2));
          new_out = j1;
        }
      } else if (L.front6) {
        if (out1 > out0 || (L.dc == DC_ZSR && nseg > 0)) {
          Front6Params fp;
          memset(&fp, 0, sizeof fp);
          CascadeParams& cp = fp.c;
          cp.src = sv;
          cp.n_streams = S;
          cp.nseg = nseg;
          cp.seg0 = seg0;
          cp.seg_len = L.seg_len;
          cp.halo = L.halo;
          cp.out0 = out0;
          cp.out1 = out1;
          cp.scale = integer_units(L) ? L.scale / 128.0f : L.scale;
          fp.w0 = (float)((double)CU8_XBIAS / (double)alpha_eff);
          cp.alpha = alpha_eff;
          cp.sums = (float2*)sums.p;
          cp.dc_end = seg0_next - L.halo;
          cp.dst = (float2*)L.ring.p;
          cp.dst_stride = L.cap;
          cp.dst_mask = L.cap - 1;
          memcpy(cp.hb, L.hb, sizeof cp.hb);
          memcpy(fp.hb5, L.hb[4], sizeof fp.hb5);
          memcpy(fp.hb6, L.hb[5], sizeof fp.hb6);
          // cp.async staging as in the fused kernel (2.87 ms per dsd_in step against 2.90 ms with register loads)
          const size_t f6_smem = (size_t)F6_CPD * 32 * FF_THREADS;
          if (L.ms[4] == 3) front6_kernel<3, 5><<<blocks, FF_THREADS, f6_smem, st>>>(fp);
          else front6_kernel<5, 10><<<blocks, FF_THREADS, f6_smem, st>>>(fp);
          *launches += 1;
          tm->mark(st, TM_CASCADE0);
          if (out1 > out0) new_out = out1;
        }
      } else if (L.fused) {
        if (out1 > out0 || (L.dc == DC_ZSR && nseg > 0)) {
          FusedParams fp;
          memset(&fp, 0, sizeof fp);
          CascadeParams& cp = fp.c;
          cp.src = sv;
          cp.n_streams = S;
          cp.nseg = nseg;
          cp.seg0 = seg0;
          cp.seg_len = L.seg_len;
          cp.halo = L.halo;
          cp.out0 = out0;
          cp.out1 = out1;
          cp.scale = integer_units(L) ? L.scale / 128.0f : L.scale;   // 2^-3 * 2^-7, exact
          cp.alpha = alpha_eff;
          cp.sums = (float2*)sums.p;
          cp.dc_end = seg0_next - L.halo;
          cp.dst = (float2*)L.ring.p;
          cp.dst_stride = L.cap;
          cp.dst_mask = L.cap - 1;
          memcpy(cp.hb, L.hb, sizeof cp.hb);
          memcpy(fp.arb, L.arb_rows, sizeof fp.arb);   // (folding cp.scale into these taps saves 6 FMUL2 of 590 and ran 3 % slower)
          fp.w0 = (float)((double)CU8_XBIAS / (double)alpha_eff);
          // raw bytes staged global -> shared memory by cp.async six sub-blocks ahead (2.456 ms against 2.486 ms with register loads).
          // 32-thread blocks: the same 8 warps per SM, but the 10.6 "waves" of 128-thread blocks end in a shorter tail (2.62 vs 2.68 ms)
          const int thr = 32;
          const unsigned fblocks = (unsigned)((threads + thr - 1) / thr);
          fused_frontend_kernel<<<fblocks, thr, (size_t)FF_CPD * 32 * thr, st>>>(fp);
          *launches += 1;
          tm->mark(st, TM_CASCADE0);
          if (out1 > out0) new_out = (long long)design::arb_outputs_after((uint64_t)out1, plan.step);
        }
      } else if (out1 > out0 || (L.dc == DC_ZSR && nseg > 0)) {
        CascadeParams cp;
        memset(&cp, 0, sizeof cp);
        cp.src = sv;
        cp.n_streams = S;
        cp.nseg = nseg;
        cp.seg0 = seg0;
        cp.seg_len = L.seg_len;
        cp.halo = L.halo;
        cp.out0 = out0;
        cp.out1 = out1;
        cp.scale = L.scale;
        cp.alpha = alpha_eff;
        cp.v_seg = (const float2*)v_seg.p;
        cp.sums = (float2*)sums.p;
        cp.dc_end = seg0_next - L.halo;
        cp.step = plan.step;
        cp.bits = (int)plan.bits;
        cp.pfb = (const float*)pfb.p;
        cp.dst = (float2*)L.ring.p;
        cp.dst_stride = L.cap;
        cp.dst_mask = L.cap - 1;
        memcpy(cp.hb, L.hb, sizeof cp.hb);
        L.fn<<<blocks, 128, 0, st>>>(cp);
        *launches += 1;
        tm->mark(st, TM_CASCADE0 + (int)std::min<size_t>(l, 2));
        if (out1 > out0) new_out = L.arb ? (long long)design::arb_outputs_after((uint64_t)out1, plan.step) : out1;
      }
      if (L.dc == DC_ZSR && nseg > 0) {   // chain the local sums the cascade just wrote into V0 per segment
        launch_dc_scan(sp, st);
        *launches += 1;
        tm->mark(st, TM_DC);
        // ring samples per input sample of this level: 1 / D, or 1 / 12 with the x 2/3 resampler fused in
        const int per_out = L.fused ? 12 : L.D;
        int shift = 0;
        while ((1 << shift) < L.seg_len / per_out) shift++;
        corr.v_seg = (const float2*)v_seg.p;
        corr.e = (const float*)e_table.p;
        corr.from = L.fused ? L.n_out : out0;
        corr.seg0_out = seg0 / per_out;
        corr.seg_shift = shift;
        corr.halo_out = L.halo / per_out;
        corr.nseg = nseg;
        corr.alpha = alpha_eff;
        for (int i = 0; i < 16; i++) corr.rho_pow[i] = (float)pow((double)c_pole, (double)(i * L.D));
      } else {
        memset(&corr, 0, sizeof corr);
      }
      if (l > 0 && sv.corr.v_seg) {
        // the consumer has read its input: fix the tail of the producer's ring in place, it is the
        // next chunk's history
        const Level& P = levels[l - 1];
        const int count = L.halo + L.unit;
        const long long start = lvl_n1 - count;
        zir_tail_kernel<<<dim3((count + 127) / 128, S), 128, 0, st>>>((float2*)P.ring.p, P.cap, P.cap - 1, sv.corr, start, count);
        *launches += 1;
        tm->mark(st, TM_HIST);
      }
      L.n_in = lvl_n1;
      lvl_n0 = L.n_out;
      L.n_out = new_out;
      lvl_n1 = new_out;
    }
    // save the raw tail for the next call
    {
      const Level& L0 = levels[0];
      const long long new_base = n1 / L0.unit * L0.unit - L0.halo;
      const int count = (int)(n1 - new_base);
      if (count > hist_cap) return fail(PMR446_ERANGE, "internal: history overflow");
      DevBuf& dst = hist[hist_cur ^ 1];
      dim3 grid((count + 127) / 128, S);
      if (count > 0) {
        if (bps == 2) hist_update_kernel<uint16_t><<<grid, 128, 0, st>>>(v0, (uint16_t*)dst.p, hist_cap, new_base, count);
        else if (bps == 4) hist_update_kernel<uint32_t><<<grid, 128, 0, st>>>(v0, (uint32_t*)dst.p, hist_cap, new_base, count);
        else hist_update_kernel<float2><<<grid, 128, 0, st>>>(v0, (float2*)dst.p, hist_cap, new_base, count);
        *launches += 1;
        tm->mark(st, TM_HIST);
      }
      hist_cur ^= 1;
      hist_base = new_base;
    }
    n_in = n1;
    n_out = levels.back().n_out;
    if (corr.v_seg) {   // set by the LAST level: only a fused level does that
      pending = corr;
      has_pending = true;
      if (!defer_zir) fix_pending(st, launches, true, tm);
    }
    return 0;
  }
};

}  // namespace pmr
