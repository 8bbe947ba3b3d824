// NP+ forward / backward for sm_100a — replaces MRFPPlus.Normalization_Perturbation_Plus
// (/root/reference/deepv3.py:268-277) and its autograd backward (closed form, SURVEY.md §8 a-1).
//
// Both directions are the same memory-bound shape:  y = a[n,c] * x + b[n,c]  where (a, b) depend on the
// plane sums of x for ALL planes of the local batch (batch std of the plane means + global channel max).
// One cooperative persistent kernel, one CTA per SM, work in "units" (a unit = <= 32 KiB slice of one plane):
//   phase A  a producer thread streams units into a shared-memory ring with 1-D TMA bulk copies
//            (cp.async.bulk + mbarrier complete_tx); 16 consumer warps reduce each unit from shared memory
//            (128-bit LDS, fp32 lane partials, double warp-shuffle tree); the last warp to finish a unit folds the
//            16 warp partials in fixed order.  Units come from a grid-wide atomic queue, framed by two static
//            sets per CTA that STAY ON CHIP: a head of 2 units kept in the consumers' registers plus up to 8 units
//            parked in tensor memory (TMEM is otherwise idle: no MMA here) and a tail of up to 7 units left in the ring
//            (17 x 32 KiB x 148 SMs = 80 MB);
//   barrier  grid-wide (cooperative groups);
//   stats    grid-parallel per-channel statistics, second barrier, then every CTA reduces max_c d / arg-max /
//            the backward's cross-channel sum and derives (a, b) for its resident units;
//   phase B  resident units first (no re-read at all), then the rest from a second atomic queue in DESCENDING
//            order — most recently read first, so the re-read is served from L2 while it lasts; the producer warp
//            derives each unit's (a, b) one batch ahead; 128-bit streaming (evict-first) stores.
// HBM traffic therefore sits between 1R+1W (everything cached on chip) and 2R+1W.
// A register-staged variant of the same algorithm (no TMA; scalar loads) handles planes whose size or base
// address is not a multiple of 16 bytes.
#include "common.cuh"
#include "ptx.cuh"
#include <cooperative_groups.h>
#include <math.h>
#include <stdlib.h>
#include <atomic>

namespace cg = cooperative_groups;

namespace mrfp {
namespace {
using namespace ptx;

constexpr int kConsumers = 512;                 // consumer threads (16 warps)
constexpr int kWarps = kConsumers / 32;
constexpr int kBatch = 4;                       // vectors per consumer thread per unit
constexpr int kUnitVecs = kConsumers * kBatch;  // 2048 float4 = 32 KiB
constexpr int kMaxSlots = 7;
constexpr int kTmemUnits = 8;                    // 512 TMEM columns / 64 columns per parked unit
constexpr int kRegUnits = 2;                     // head units a consumer thread keeps in registers (16 floats each)

struct NpGeom {
  int N, C, HW;
  int P;         // planes = N*C
  int K;         // units per plane
  int Q;         // vectors per unit (last unit of a plane may be shorter)
  int HWV;       // HW / VEC
  long long U;   // total units = P*K
  int slots;     // ring slots / resident units per CTA
  int max_local_planes;   // scalar path: planes a CTA can touch
  int grid;      // CTAs
  int keep_units;  // ring path: units (grid-wide) loaded with an L2 evict_last hint because phase B re-reads them
  long long scratch_off;   // scalar path, doubles: ps[0..scratch_off) partials, then pm[P], then chan[4*C]
  int grab;      // ring path: units taken from the phase-A queue per atomic
  int grab_b;    // ring path: units taken from the phase-B queue per atomic (small: the tail of phase B ends the kernel)
  int u_dyn;     // ring path: units [0, u_dyn) are handed out dynamically; the rest is the static resident tail
  int tmem_units;  // ring path: head units per CTA parked in tensor memory
  int reg_units;   // ring path: head units per CTA parked in the consumers' registers (0 or kRegUnits), before the TMEM ones
  int mid_units;   // ring path: units before the keep_units band loaded with L2 evict_normal
  int heads_last;  // ring path: phase B writes the register / TMEM heads after the re-read queue instead of before it
};

// ------------------------------------------------------------------------------------------------------
// statistics shared by both kernels
// ------------------------------------------------------------------------------------------------------
// unit partials are written by other CTAs earlier in this launch: read through L2 (ld.global.cg)
__device__ __forceinline__ double plane_total(const double* ps, int plane, const NpGeom& g) {
  const double* p = ps + (long long)plane * g.K;
  if (g.K <= 8) {                       // all loads leave together (one L2 round trip), summed in index order
    double v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = k < g.K ? __ldcg(p + k) : 0.0;
    double s = v[0];
#pragma unroll
    for (int k = 1; k < 8; ++k) s += v[k];
    return s;
  }
  double s = 0;
#pragma unroll 4
  for (int k = 0; k < g.K; ++k) s += __ldcg(p + k);
  return s;
}

__device__ __forceinline__ double group_sum(double v, int width) {   // xor-butterfly inside aligned lane groups
  for (int o = width >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct NpShared {
  double w_best[kWarps + 1], w_tsum[kWarps + 1];
  int w_c[kWarps + 1], w_nan[kWarps + 1];
  double dmax, T;
  int cstar;
};

// Stage 1: per-channel statistics of the plane means over the local batch (deepv3.py:272):
//   chan[4c..] = { mbar, d = unbiased std of the plane means, dL/ds (backward only), - }
// and, when `pm` is given, the plane totals pm[p] (sum over HW).  Warp `wfirst` of `wcount` takes every
// wcount-th channel group: (blockIdx*nwarps+warp, gridDim*nwarps) spreads the work over the grid (scalar kernel,
// followed by a second grid barrier); (warp, nwarps) makes every CTA compute the whole table for itself (ring kernel).
template <bool BWD>
__device__ void np_stage1(const double* ps, const float* __restrict__ mean_in, const float* __restrict__ eps,
                          const NpGeom& g, double* pm, double* chan, int wfirst, int wcount) {
  const int lane = threadIdx.x & 31;
  const double inv_hw = 1.0 / (double)g.HW;
  // lanes = (channel sub-group, batch index): group width = pow2 >= N (capped at 32)
  int gw = 1;
  while (gw < g.N && gw < 32) gw <<= 1;
  const int cpw = 32 / gw, sub = lane % gw, cg_i = lane / gw;
  for (int cbase = wfirst * cpw; cbase < g.C; cbase += wcount * cpw) {    // warp-uniform trip count
    const int c = cbase + cg_i;
    const bool valid = c < g.C;
    double s = 0, m0 = 0, G0 = 0;
    if (valid) {
      for (int n = sub; n < g.N; n += gw) {
        const int p = n * g.C + c;
        const double tot = plane_total(ps, p, g);
        if (pm) pm[p] = tot;
        const double m = BWD ? (double)mean_in[p] : tot * inv_hw;
        if (n == sub) { m0 = m; G0 = tot; }
        s += m;
      }
    }
    const double mbar = group_sum(s, gw) / (double)g.N;
    double q = 0, l = 0;
    if (valid) {
      for (int n = sub; n < g.N; n += gw) {
        const int p = n * g.C + c;
        double m, G;
        if (n == sub) { m = m0; G = G0; }
        else { G = plane_total(ps, p, g); m = BWD ? (double)mean_in[p] : G * inv_hw; }
        q += (m - mbar) * (m - mbar);
        if (BWD) l += (double)eps[p] * m * G;                            // dL/ds[c] = sum_n eps*m*G
      }
    }
    const double d = sqrt(group_sum(q, gw) / (double)(g.N - 1));         // N == 1 -> 0/0 -> NaN, as torch.std
    const double dLds = BWD ? group_sum(l, gw) : 0.0;
    if (valid && sub == 0) {
      chan[4 * c + 0] = mbar;
      chan[4 * c + 1] = d;
      chan[4 * c + 2] = dLds;
    }
  }
}

// Stage 2a (every CTA): global max / arg-max of d and the backward's cross-channel sum -> sh.dmax, sh.cstar, sh.T
template <bool BWD>
__device__ void np_global_reduce(const double* chan, const NpGeom& g, NpShared& sh, int nthreads) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;
  double best = -1.0, tsum = 0.0;
  int bestc = 0x7fffffff;
  bool anynan = false;
  for (int c = tid; c < g.C; c += nthreads) {
    const double d = __ldcg(chan + 4 * c + 1);
    if (d != d) anynan = true;
    if (d > best) { best = d; bestc = c; }
    if (BWD) tsum += __ldcg(chan + 4 * c + 2) * d;
  }
  // block arg-max (first index wins on ties), NaN-propagating like Tensor.max (deepv3.py:273)
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oc = __shfl_xor_sync(0xffffffffu, bestc, o);
    const int on = __shfl_xor_sync(0xffffffffu, (int)anynan, o);
    tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
    if (ob > best || (ob == best && oc < bestc)) { best = ob; bestc = oc; }
    anynan = anynan || (on != 0);
  }
  if (lane == 0) { sh.w_best[warp] = best; sh.w_c[warp] = bestc; sh.w_nan[warp] = anynan; sh.w_tsum[warp] = tsum; }
  __syncthreads();
  if (tid == 0) {
    double b = sh.w_best[0], t = sh.w_tsum[0];
    int bc = sh.w_c[0], nn = sh.w_nan[0];
    for (int i = 1; i < nwarps; ++i) {
      if (sh.w_best[i] > b || (sh.w_best[i] == b && sh.w_c[i] < bc)) { b = sh.w_best[i]; bc = sh.w_c[i]; }
      nn |= sh.w_nan[i];
      t += sh.w_tsum[i];
    }
    sh.dmax = nn ? (double)NAN : b;
    sh.cstar = bc;
    sh.T = 1.5 * t / (sh.dmax * sh.dmax);     // sum_c dL/ds[c] * 1.5 * d[c] / dmax^2
  }
  __syncthreads();
}

// Stage 2b: (a, b) of plane p, y = a*x + b, in two steps so that a caller can put other work between the loads and
// their first use.  `publish`: this thread also writes the (N,C) side outputs of the plane.
struct NpCoefIn {
  double tot, mbar, d, dLds;
  float alpha, eps, mean;
};
template <bool BWD>
__device__ __forceinline__ NpCoefIn np_coef_load(int p, const double* pm, const double* chan,
                                                 const float* __restrict__ mean_in, const float* __restrict__ alpha,
                                                 const float* __restrict__ eps, const NpGeom& g) {
  NpCoefIn r;
  const int c = p % g.C;
  r.tot = __ldcg(pm + p);
  r.mbar = __ldcg(chan + 4 * c + 0);
  r.d = __ldcg(chan + 4 * c + 1);
  r.dLds = BWD ? __ldcg(chan + 4 * c + 2) : 0.0;
  r.alpha = alpha[p];
  r.eps = eps[p];
  r.mean = BWD ? mean_in[p] : 0.f;
  return r;
}
template <bool BWD>
__device__ __forceinline__ float2 np_coef_finish(const NpCoefIn& r, int p, bool publish, float* __restrict__ mean_out,
                                                 float* __restrict__ beta_out, const NpGeom& g, const NpShared& sh) {
  const double inv_hw = 1.0 / (double)g.HW, dmax = sh.dmax;
  const double a = (double)r.alpha;
  const double beta = 1.0 + (double)r.eps * (r.d / dmax * 1.5);          // deepv3.py:273,275
  double b;
  if (!BWD) {
    const double m = r.tot * inv_hw;
    b = (beta - a) * m;                                                   // out = a*x + (beta-a)*m  (:276)
    if (publish) {
      mean_out[p] = (float)m;
      if (beta_out) beta_out[p] = (float)beta;
    }
  } else {
    const double m = (double)r.mean;
    double dLdd = 1.5 / dmax * r.dLds;
    if (p % g.C == sh.cstar) dLdd -= sh.T;
    // torch's std_backward zero-fills where std == 0
    const double dd_dm = (r.d == 0.0) ? 0.0 : (m - r.mbar) / ((double)(g.N - 1) * r.d);
    const double dLdm = (beta - a) * r.tot + dLdd * dd_dm;
    b = dLdm * inv_hw;
  }
  return make_float2((float)a, (float)b);
}
template <bool BWD>
__device__ __forceinline__ float2 np_plane_coef(int p, bool publish, const double* pm, const double* chan,
                                                const float* __restrict__ mean_in, const float* __restrict__ alpha,
                                                const float* __restrict__ eps, float* __restrict__ mean_out,
                                                float* __restrict__ beta_out, const NpGeom& g, const NpShared& sh) {
  return np_coef_finish<BWD>(np_coef_load<BWD>(p, pm, chan, mean_in, alpha, eps, g), p, publish, mean_out, beta_out, g, sh);
}

// ------------------------------------------------------------------------------------------------------
// TMA-ring kernel with grid-wide dynamic unit queues (planes and base addresses 16-byte aligned)
// ------------------------------------------------------------------------------------------------------
// SMs do not stream from HBM at the same rate (the slowest took 40 % longer than the fastest on a static
// split), so both passes hand units out from atomic counters in batches of g.grab:
//   phase A   units [0, u_dyn) in ascending order from counterA, then a STATIC tail of `slots` units per CTA
//             (unit u_dyn + blockIdx*slots + j) which stays resident in the ring;
//   phase B   the resident tail first (no re-read), then units [0, u_dyn) in DESCENDING order from counterB —
//             the most recently read data first, so the re-read is served from L2 while it lasts.
// A fill of ring slot s carries its unit index (and, in phase B, the plane's (a, b) pair) in shared memory next to
// the slot.  Both counters are zero when a launch begins: the control block is zero-filled ONCE by the owner of the
// workspace (mrfp_npplus_ws_init, or an allocation that zero-fills), and every launch re-arms it for the next one — CTA 0 clears
// counter_b at kernel entry (it is first read behind the second grid barrier) and counter_a right behind the first grid
// barrier (its last use precedes that barrier).  No per-launch host value enters the kernel, so a launch captured in a
// CUDA graph replays correctly.
struct NpCtrl {
  unsigned long long reserved;
  unsigned int counter_a;
  unsigned int counter_b;
  unsigned int pad[12];
};

// Tensor memory as a scratchpad: this kernel issues no MMA, so the SM's 256 KiB of TMEM (128 lanes x 512 32-bit
// columns) hold 8 more resident units.  A consumer thread parks the 16 floats it owns of a unit in 16 columns of
// its own lane (tcgen05.st 32x32b.x16) and reads them back in phase B (tcgen05.ld); warp w may only touch lanes
// 32*(w%4)..+31, so the unit occupies columns [64*j + 16*(w/4), +16) of every lane.
__device__ __forceinline__ void tmem_park(uint32_t taddr, const float4 (&v)[kBatch]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "f"(v[0].x), "f"(v[0].y), "f"(v[0].z), "f"(v[0].w), "f"(v[1].x), "f"(v[1].y), "f"(v[1].z), "f"(v[1].w),
        "f"(v[2].x), "f"(v[2].y), "f"(v[2].z), "f"(v[2].w), "f"(v[3].x), "f"(v[3].y), "f"(v[3].z), "f"(v[3].w) : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_fetch(uint32_t taddr, float4 (&v)[kBatch]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=f"(v[0].x), "=f"(v[0].y), "=f"(v[0].z), "=f"(v[0].w), "=f"(v[1].x), "=f"(v[1].y), "=f"(v[1].z), "=f"(v[1].w),
        "=f"(v[2].x), "=f"(v[2].y), "=f"(v[2].z), "=f"(v[2].w), "=f"(v[3].x), "=f"(v[3].y), "=f"(v[3].z), "=f"(v[3].w)
      : "r"(taddr));
  tcgen05_wait_ld();
}

template <bool BWD>
__global__ void __launch_bounds__(kConsumers + 32, 1)
npplus_ring_kernel(const float* __restrict__ x, const float* __restrict__ alpha, const float* __restrict__ eps,
                   const float* __restrict__ mean_in, float* __restrict__ out, float* __restrict__ mean_out,
                   float* __restrict__ beta_out, unsigned char* ws, const NpGeom g, unsigned long long* trace) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // resident units of this CTA: a static HEAD of T units parked in TMEM at the very start (their imbalance is absorbed
  // by the dynamic queue that follows) and a static TAIL of S units that stays in the ring
  const int S = g.slots, RG = g.reg_units, T = g.reg_units + g.tmem_units;   // T: all head units (registers first, then TMEM)
  auto stamp = [&](int i) {
    if (trace && threadIdx.x == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      trace[blockIdx.x * 8 + i] = t;
    }
  };
  stamp(0);
  float4* ring = reinterpret_cast<float4*>(smem_raw);                                   // S x 32 KiB
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)S * kUnitVecs * 16);  // [S]
  uint64_t* empty = full + S;                                                           // [S]
  volatile double* wp = reinterpret_cast<volatile double*>(empty + S);                  // [S][kWarps] warp partials of a fill
  float2* slot_coef = reinterpret_cast<float2*>(const_cast<double*>(wp) + S * kWarps);  // [S]
  volatile int* slot_unit = reinterpret_cast<volatile int*>(slot_coef + S);             // [S]
  int* slot_cnt = const_cast<int*>(slot_unit) + S;                                      // [S] warps that delivered their partial
  __shared__ NpShared sh;
  __shared__ float2 head_coef[kTmemUnits + kRegUnits];
  float4 preg0[kBatch] = {}, preg1[kBatch] = {};             // register-parked head units (consumer threads); a third one spills
  __shared__ uint32_t tmem_base_s;

  NpCtrl* ctrl = reinterpret_cast<NpCtrl*>(ws);
  double* ps = reinterpret_cast<double*>(ws + sizeof(NpCtrl));      // [U] unit partials
  double* pm = ps + g.U;                                            // [P] plane totals
  double* chan = pm + g.P;                                          // [4C] channel statistics

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool is_producer = warp == kWarps;
  const int u_dyn = g.u_dyn;
  const int head0 = (int)blockIdx.x * T;                 // unit space: [heads: grid*T][dynamic queue: u_dyn][tails: grid*S]
  const int dyn0 = (int)gridDim.x * T;
  const int tail0 = dyn0 + u_dyn + (int)blockIdx.x * S;
  const int last_len = g.HWV - (g.K - 1) * g.Q;          // the last unit of a plane may be shorter
  const float4* xv = reinterpret_cast<const float4*>(x);
  float4* ov = reinterpret_cast<float4*>(out);

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kWarps); slot_cnt[s] = 0; }
    mbar_fence_init();
    if (blockIdx.x == 0) ctrl->counter_b = 0;            // read behind the second grid barrier only
  }
  if (is_producer && T > RG) {                           // the whole TMEM (one CTA per SM, no MMA in this kernel)
    tmem_alloc<512>(&tmem_base_s);
    tmem_relinquish();
    tcgen05_before_sync();
  }
  __syncthreads();
  tcgen05_after_sync();
  // this thread's window into TMEM: its own lane, 16 columns per parked unit
  const uint32_t tmem_mine = T > RG ? tmem_base_s + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * 16) : 0u;

  // ring position of the next fill; producer and consumers count the same fills, so they agree after phase A
  int s = 0, k = 0;
  auto advance = [&]() { if (++s == S) { s = 0; ++k; } };
  auto unit_src = [&](int u, uint32_t* bytes) {
    const int plane = u / g.K, part = u - plane * g.K;
    *bytes = (uint32_t)(part == g.K - 1 ? last_len : g.Q) * 16u;
    return (long long)plane * g.HWV + part * g.Q;
  };

  // ---------------- phase A ----------------
  if (is_producer) {
    if (lane == 0) {
      const uint64_t pol_keep = policy_evict_last(), pol_mid = policy_evict_normal(), pol_stream = policy_evict_first();
      auto issue = [&](int u, uint64_t pol) {
        if (k > 0) mbar_wait(&empty[s], (k - 1) & 1);    // all 16 warps released the previous fill of this slot
        uint32_t bytes;
        const long long off = unit_src(u, &bytes);
        slot_unit[s] = u;
        mbar_expect_tx(&full[s], bytes);
        bulk_load_hint(ring + (size_t)s * kUnitVecs, xv + off, bytes, &full[s], pol);
        advance();
      };
      for (int j = 0; j < T; ++j) issue(head0 + j, pol_stream);
      // the last g.keep_units of the dynamic range are the first ones re-read in phase B: ask L2 to keep them
      const int keep_lo = u_dyn - g.keep_units, mid_lo = keep_lo - g.mid_units;
      unsigned base = blockIdx.x * g.grab;               // the first batch of every CTA is static, the queue starts behind them
      const unsigned q0 = gridDim.x * (unsigned)g.grab;
      while (base < (unsigned)u_dyn) {
        const unsigned nbase = q0 + atomicAdd(&ctrl->counter_a, (unsigned)g.grab);   // in flight while this batch is issued
        for (int q = 0; q < g.grab && base + q < (unsigned)u_dyn; ++q) {
          const int u = (int)base + q;
          issue(dyn0 + u, u >= keep_lo ? pol_keep : (u >= mid_lo ? pol_mid : pol_stream));
        }
        base = nbase;
      }
      for (int j = 0; j < S; ++j) issue(tail0 + j, pol_stream);
    }
  } else {
    for (;;) {
      mbar_wait(&full[s], k & 1);
      const int u = slot_unit[s];
      const int plane = u / g.K, part = u - plane * g.K;
      const int len = part == g.K - 1 ? last_len : g.Q;
      const float4* src = ring + (size_t)s * kUnitVecs;
      const int hj = u - head0;                          // 0 .. T-1: position in this CTA's head
      float4 v[kBatch];
      float acc = 0.f;
#pragma unroll
      for (int b = 0; b < kBatch; ++b) {
        const int i = tid + b * kConsumers;
        v[b] = i < len ? src[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        acc += (v[b].x + v[b].y) + (v[b].z + v[b].w);
      }
      if (hj >= 0 && hj < RG) {                          // registers first ...
#pragma unroll
        for (int b = 0; b < kBatch; ++b) {
          if (hj == 0) preg0[b] = v[b]; else preg1[b] = v[b];
        }
      } else if (hj >= RG && hj < T) {                   // ... then tensor memory
        tmem_park(tmem_mine + (uint32_t)((hj - RG) * 64), v);
      }
      const double w = warp_sum((double)acc);
      const bool stays = u >= tail0;                     // the S tail fills stay in the ring until phase B
      if (lane == 0) {
        wp[s * kWarps + warp] = w;
        __threadfence_block();
        if (atomicAdd(&slot_cnt[s], 1) == kWarps - 1) {  // last warp of this fill: fold the 16 partials in fixed order
          __threadfence_block();
          double t = 0;
#pragma unroll
          for (int i = 0; i < kWarps; ++i) t += wp[s * kWarps + i];
          ps[u] = t;
          slot_cnt[s] = 0;
        }
        if (!stays) mbar_arrive(&empty[s]);
      }
      advance();
      if (u == tail0 + S - 1) break;
    }
  }
  if (is_producer) {                                     // lanes 1..31 of the producer warp: adopt lane 0's ring position
    s = __shfl_sync(0xffffffffu, s, 0);
    k = __shfl_sync(0xffffffffu, k, 0);
  }
  __syncthreads();
  stamp(1);
  __threadfence();
  cg::this_grid().sync();
  stamp(2);
  if (blockIdx.x == 0 && tid == 0) ctrl->counter_a = 0;  // every phase-A grab precedes the barrier: ready for the next launch

  // ---------------- statistics ----------------
  np_stage1<BWD>(ps, mean_in, eps, g, pm, chan, blockIdx.x * (kWarps + 1) + warp, gridDim.x * (kWarps + 1));
  stamp(5);
  __threadfence();
  cg::this_grid().sync();
  stamp(6);
  np_global_reduce<BWD>(chan, g, sh, kConsumers + 32);
  stamp(7);
  if (tid < S + T) {                                     // the resident units
    const int u = tid < T ? head0 + tid : tail0 + (tid - T), plane = u / g.K;
    const float2 ab = np_plane_coef<BWD>(plane, u - plane * g.K == 0, pm, chan, mean_in, alpha, eps, mean_out, beta_out, g, sh);
    if (tid < T) head_coef[tid] = ab;
    else {
      int sl = s + (tid - T);                            // tail fill j sits in slot (s + j) mod S
      if (sl >= S) sl -= S;
      slot_coef[sl] = ab;
    }
  }
  __syncthreads();
  stamp(3);

  // ---------------- phase B ----------------
  if (is_producer) {
    const uint64_t pol_stream = policy_evict_first();
    // software pipeline, one batch deep: while batch j is being issued (which blocks on free slots), the index of
    // batch j+1 and the inputs of its (a, b) pairs are already in flight
    auto grab = [&]() {
      unsigned v = 0;
      if (lane == 0) v = atomicAdd(&ctrl->counter_b, (unsigned)g.grab_b);
      return v;
    };
    unsigned idx = __shfl_sync(0xffffffffu, grab(), 0);
    unsigned nidx = grab();
    NpCoefIn ci = {};
    int u = 0, cnt = 0;
    auto stage = [&](unsigned id) {                      // lane q < cnt takes queue entry (u_dyn-1-id-q): start its loads
      cnt = id < (unsigned)u_dyn ? min(g.grab_b, u_dyn - (int)id) : 0;
      if (lane < cnt) {
        u = dyn0 + u_dyn - 1 - (int)id - lane;
        ci = np_coef_load<BWD>(u / g.K, pm, chan, mean_in, alpha, eps, g);
      }
    };
    stage(idx);
    while (cnt > 0) {
      float2 ab = make_float2(0.f, 0.f);
      const int cur_u = u, cur_cnt = cnt;
      if (lane < cnt) {
        const int plane = u / g.K;
        ab = np_coef_finish<BWD>(ci, plane, u - plane * g.K == 0, mean_out, beta_out, g, sh);
      }
      idx = __shfl_sync(0xffffffffu, nidx, 0);
      nidx = grab();
      stage(idx);                                        // loads for the next batch leave before this one blocks
      for (int q = 0; q < cur_cnt; ++q) {
        const int uq = __shfl_sync(0xffffffffu, cur_u, q);
        const float ax = __shfl_sync(0xffffffffu, ab.x, q), ay = __shfl_sync(0xffffffffu, ab.y, q);
        if (lane == 0) {
          mbar_wait(&empty[s], (k - 1) & 1);             // k >= 1 here: every slot took a phase-A fill
          uint32_t bytes;
          const long long off = unit_src(uq, &bytes);
          slot_unit[s] = uq;
          slot_coef[s] = make_float2(ax, ay);
          mbar_expect_tx(&full[s], bytes);
          bulk_load_hint(ring + (size_t)s * kUnitVecs, xv + off, bytes, &full[s], pol_stream);
        }
        advance();
      }
    }
    if (lane == 0) {
      mbar_wait(&empty[s], (k - 1) & 1);
      slot_unit[s] = -1;                                 // end marker: completes one phase of full[s] without data
      mbar_arrive(&full[s]);
    }
  } else {
    auto emit = [&](int u, const float2 ab, float4 (&v)[kBatch]) {
      const int plane = u / g.K, part = u - plane * g.K;
      const int len = part == g.K - 1 ? last_len : g.Q;
      float4* dst = ov + (long long)plane * g.HWV + part * g.Q;
#pragma unroll
      for (int b = 0; b < kBatch; ++b) {
        const int idx = tid + b * kConsumers;
        if (idx < len)
          st_stream_f4(dst + idx, make_float4(fmaf(ab.x, v[b].x, ab.y), fmaf(ab.x, v[b].y, ab.y), fmaf(ab.x, v[b].z, ab.y),
                                              fmaf(ab.x, v[b].w, ab.y)));
      }
    };
    // the ring part of the tail first (frees the slots for the producer), then the TMEM part, then the queue
    auto emit_heads = [&]() {
      if (RG > 0) { emit(head0, head_coef[0], preg0); emit(head0 + 1, head_coef[1], preg1); }
      for (int j = RG; j < T; ++j) {
        float4 v[kBatch];
        tmem_fetch(tmem_mine + (uint32_t)((j - RG) * 64), v);
        emit(head0 + j, head_coef[j], v);
      }
    };
    for (int i = 0;; ++i) {
      if (i == S && !g.heads_last) emit_heads();
      if (i >= S) mbar_wait(&full[s], k & 1);            // the first S fills are the resident tail, waited for in phase A
      const int u = slot_unit[s];
      if (u < 0) break;
      const float2 ab = slot_coef[s];
      const float4* src = ring + (size_t)s * kUnitVecs;
      float4 v[kBatch];
#pragma unroll
      for (int b = 0; b < kBatch; ++b) v[b] = src[tid + b * kConsumers];   // (slack beyond a short unit is never stored)
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[s]);
      emit(u, ab, v);
      if (i < S) { if (++s == S) s = 0; }                // replaying the tail does not start a new round
      else advance();
    }
    if (g.heads_last) emit_heads();
  }
  if (T > RG) {
    tcgen05_before_sync();
    __syncthreads();
    if (is_producer) {
      tcgen05_after_sync();
      tmem_dealloc<512>(tmem_base_s);
    }
  }
  if (trace) { __syncthreads(); stamp(4); }
}

// ------------------------------------------------------------------------------------------------------
// register-staged scalar kernel (any HW, any alignment)
// ------------------------------------------------------------------------------------------------------
template <bool BWD>
__global__ void __launch_bounds__(kConsumers, 1)
npplus_scalar_kernel(const float* __restrict__ x, const float* __restrict__ alpha, const float* __restrict__ eps,
                     const float* __restrict__ mean_in, float* __restrict__ out, float* __restrict__ mean_out,
                     float* __restrict__ beta_out, double* ps, const NpGeom g, unsigned long long* /*trace*/) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* cache = reinterpret_cast<float*>(smem_raw);                                        // slots x Q floats
  float2* coef = reinterpret_cast<float2*>(smem_raw + align_up((size_t)g.slots * g.Q * 4, 16));
  __shared__ NpShared sh;
  __shared__ double red2[2][kWarps];

  const int tid = threadIdx.x;
  const long long u0 = g.U * (long long)blockIdx.x / gridDim.x;
  const long long u1 = g.U * (long long)(blockIdx.x + 1) / gridDim.x;
  const long long cache_from = u1 - g.slots;   // units >= cache_from live in shared memory
  auto unit_len = [&](long long u) { return min(g.Q, g.HWV - (int)(u % g.K) * g.Q); };
  auto unit_off = [&](long long u) { return (u / g.K) * (long long)g.HWV + (u % g.K) * (long long)g.Q; };

  for (long long u = u0; u < u1; ++u) {
    const int len = unit_len(u);
    const float* src = x + unit_off(u);
    float* keep = (u >= cache_from) ? cache + (size_t)(u - cache_from) * g.Q : nullptr;
    float acc = 0.f;
    for (int i = tid; i < len; i += kConsumers) {
      const float v = ld_stream_f1(src + i);
      acc += v;
      if (keep) keep[i] = v;
    }
    const double w = warp_sum((double)acc);
    double* rb = red2[u & 1];
    if ((tid & 31) == 0) rb[tid >> 5] = w;
    __syncthreads();
    if (tid == 0) {
      double t = 0;
#pragma unroll
      for (int i = 0; i < kWarps; ++i) t += rb[i];
      ps[u] = t;
    }
  }
  __threadfence();
  cg::this_grid().sync();
  double* pm = ps + g.scratch_off;
  double* chan = pm + g.P;
  np_stage1<BWD>(ps, mean_in, eps, g, pm, chan, blockIdx.x * kWarps + (threadIdx.x >> 5), gridDim.x * kWarps);
  __threadfence();
  cg::this_grid().sync();
  np_global_reduce<BWD>(chan, g, sh, kConsumers);
  const int pl0 = (int)(u0 / g.K);
  {
    const int pl1 = (u1 > u0) ? (int)((u1 - 1) / g.K) : pl0 - 1;
    for (int j = tid; j <= pl1 - pl0; j += kConsumers)   // the CTA owning unit 0 of a plane publishes its side outputs
      coef[j] = np_plane_coef<BWD>(pl0 + j, (long long)(pl0 + j) * g.K >= u0, pm, chan, mean_in, alpha, eps, mean_out,
                                   beta_out, g, sh);
    __syncthreads();
  }
  for (long long u = u1 - 1; u >= u0; --u) {
    const int len = unit_len(u);
    const float2 ab = coef[(int)(u / g.K) - pl0];
    float* dst = out + unit_off(u);
    if (u >= cache_from) {
      const float* keep = cache + (size_t)(u - cache_from) * g.Q;
      for (int i = tid; i < len; i += kConsumers) st_stream_f1(dst + i, fmaf(ab.x, keep[i], ab.y));
    } else {
      const float* src = x + unit_off(u);
      for (int i = tid; i < len; i += kConsumers) st_stream_f1(dst + i, fmaf(ab.x, ld_stream_f1(src + i), ab.y));
    }
  }
}

struct NpLaunch {
  NpGeom g;
  int grid;
  size_t smem;
};

constexpr int kMaxGrid = 1024;

// workspace layout (bytes): [NpCtrl 64][ps: units][pm: P][chan: 4C]
size_t ws_layout_bytes(int N, int C, int HW) {
  const long long P = (long long)N * C;
  const long long u_scalar = P * (((long long)HW + kUnitVecs - 1) / kUnitVecs);                 // 2048 floats per unit
  const long long u_ring = P * (((long long)HW / 4 + kUnitVecs - 1) / kUnitVecs + 1);           // 2048 float4 per unit
  const long long units = u_scalar > u_ring ? u_scalar : u_ring;
  return (size_t)(sizeof(NpCtrl) + 8 * (units + P + 4LL * C));
}

void plan_launch(int N, int C, int HW, bool ring, const DeviceInfo& di, NpLaunch* L) {
  NpGeom& g = L->g;
  const int vec = ring ? 4 : 1;
  g.N = N; g.C = C; g.HW = HW; g.P = N * C;
  g.HWV = HW / vec;
  g.Q = g.HWV < kUnitVecs ? g.HWV : kUnitVecs;
  g.K = (g.HWV + g.Q - 1) / g.Q;                                 // last unit of a plane may be shorter
  g.U = (long long)g.P * g.K;
  const int sms = di.sm_count < kMaxGrid ? di.sm_count : kMaxGrid;
  L->grid = (int)((g.U < sms) ? g.U : sms);
  g.grid = L->grid;
  const long long upc = (g.U + L->grid - 1) / L->grid;           // units per CTA (static split: max)
  const long long min_upc = g.U / L->grid;                       // ... (min, >= 1)
  g.max_local_planes = (int)(upc / g.K + 2);
  g.scratch_off = g.U;
  g.keep_units = 0; g.grab = 1; g.grab_b = 1; g.u_dyn = 0; g.tmem_units = 0; g.reg_units = 0; g.mid_units = 0; g.heads_last = 0;
  const size_t slack = 1024;                                     // static smem + alignment
  if (ring) {
    long long grab = upc / 8;
    constexpr long long grab_a = 2;                              // measured: 2 beats 1 (queue-bound) and 4, 8
    g.grab = (int)(grab < 1 ? 1 : (grab > grab_a ? grab_a : grab));
    constexpr int grab_b = 2;
    g.grab_b = g.grab < grab_b ? g.grab : grab_b;
    // per slot: the unit, two mbarriers, 16 warp partials, (a, b), unit index, fold counter
    const size_t per_slot = (size_t)kUnitVecs * 16 + 16 + kWarps * 8 + 8 + 4 + 4;
    long long s = (long long)(((size_t)di.max_smem_optin - slack) / per_slot);
    if (s > kMaxSlots) s = kMaxSlots;
    if (s > min_upc) s = min_upc;                                // every CTA owns a full static tail
    if (s < 1) s = 1;
    g.slots = (int)s;
    long long t = min_upc - s;
    if (t > kTmemUnits) t = kTmemUnits;
    g.tmem_units = (int)(t < 0 ? 0 : t);
    g.reg_units = (min_upc - s - g.tmem_units >= kRegUnits) ? kRegUnits : 0;
    g.u_dyn = (int)(g.U - (long long)L->grid * (g.slots + g.tmem_units + g.reg_units));
    L->smem = align_up((size_t)g.slots * per_slot, 16);
    // L2 share asked to keep the last-read units for the phase-B re-read (0-100 MiB measured the same DRAM traffic)
    g.keep_units = (int)((64LL << 20) / ((long long)kUnitVecs * 16));
  } else {
    const size_t coef_bytes = align_up((size_t)g.max_local_planes * sizeof(float2), 16);
    const size_t unit_bytes = (size_t)g.Q * 4;
    long long s = (long long)(((size_t)di.max_smem_optin - slack - coef_bytes) / unit_bytes);
    if (s > min_upc) s = min_upc;   // the resident window must not start before u0
    g.slots = (int)s;
    L->smem = align_up((size_t)g.slots * unit_bytes, 16) + coef_bytes;
  }
}

template <bool BWD>
int run(const float* x, const float* alpha, const float* eps, const float* mean_in, float* out, float* mean_out,
        float* beta_out, void* ws, size_t ws_bytes, int N, int C, int HW, void* stream) {
  if (!x || !alpha || !eps || !out || !ws || (BWD && !mean_in) || (!BWD && !mean_out)) return MRFP_ERR_NULL_POINTER;
  if (N <= 0 || C <= 0 || HW <= 0 || (long long)N * C > (1 << 24)) return MRFP_ERR_BAD_SHAPE;
  if (ws_bytes < mrfp_npplus_ws_bytes(N, C, HW) || ((uintptr_t)ws & 15)) return MRFP_ERR_WORKSPACE;
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const bool ring = (HW % 4 == 0) && (((uintptr_t)x | (uintptr_t)out) & 15) == 0;
  NpLaunch L;
  plan_launch(N, C, HW, ring, di, &L);
  if (ring && L.g.U >= (1LL << 31)) return MRFP_ERR_BAD_SHAPE;
  NpGeom g = L.g;
  // debug: MRFP_NPPLUS_TRACE=1 and a workspace with room for grid*8 extra u64 -> per-CTA phase timestamps
  static const bool want_trace = getenv("MRFP_NPPLUS_TRACE") != nullptr;
  const size_t base = align_up(mrfp_npplus_ws_bytes(N, C, HW), 8);
  unsigned long long* trace = nullptr;
  if (want_trace && ws_bytes >= base + (size_t)L.grid * 64) trace = (unsigned long long*)((char*)ws + base);
  if (ring) {
    unsigned char* wsb = (unsigned char*)ws;
    void* args[] = {(void*)&x, (void*)&alpha, (void*)&eps, (void*)&mean_in, (void*)&out, (void*)&mean_out,
                    (void*)&beta_out, (void*)&wsb, (void*)&g, (void*)&trace};
    void* kern = (void*)npplus_ring_kernel<BWD>;
    MRFP_SMEM_OPT_IN(kern, di.max_smem_optin - 1024, di.device);   // once per device: the ring takes what the SM has (minus the static part)
    MRFP_CUDA_TRY(cudaLaunchCooperativeKernel(kern, dim3(L.grid), dim3(kConsumers + 32), args, L.smem, (cudaStream_t)stream));
  } else {
    double* ps = (double*)((char*)ws + sizeof(NpCtrl));
    void* args[] = {(void*)&x, (void*)&alpha, (void*)&eps, (void*)&mean_in, (void*)&out,
                    (void*)&mean_out, (void*)&beta_out, (void*)&ps, (void*)&g, (void*)&trace};
    void* kern = (void*)npplus_scalar_kernel<BWD>;
    MRFP_SMEM_OPT_IN(kern, di.max_smem_optin - 1024, di.device);
    MRFP_CUDA_TRY(cudaLaunchCooperativeKernel(kern, dim3(L.grid), dim3(kConsumers), args, L.smem, (cudaStream_t)stream));
  }
  return MRFP_OK;
}

}  // namespace
}  // namespace mrfp

extern "C" int mrfp_npplus_ws_init(void* ws, size_t ws_bytes, void* stream) {
  if (!ws) return MRFP_ERR_NULL_POINTER;
  if (ws_bytes < sizeof(mrfp::NpCtrl) || ((uintptr_t)ws & 15)) return MRFP_ERR_WORKSPACE;
  MRFP_CUDA_TRY(cudaMemsetAsync(ws, 0, sizeof(mrfp::NpCtrl), (cudaStream_t)stream));
  return MRFP_OK;
}

extern "C" size_t mrfp_npplus_ws_bytes(int N, int C, int HW) {
  if (N <= 0 || C <= 0 || HW <= 0) return 0;
  return mrfp::ws_layout_bytes(N, C, HW);
}

extern "C" int mrfp_npplus_fwd_f32(const float* x, const float* alpha, const float* eps, float* out, float* mean,
                                   float* beta, void* ws, size_t ws_bytes, int N, int C, int HW, void* stream) {
  return mrfp::run<false>(x, alpha, eps, nullptr, out, mean, beta, ws, ws_bytes, N, C, HW, stream);
}

extern "C" int mrfp_npplus_bwd_f32(const float* gout, const float* alpha, const float* eps, const float* mean,
                                   float* gin, void* ws, size_t ws_bytes, int N, int C, int HW, void* stream) {
  return mrfp::run<true>(gout, alpha, eps, mean, gin, nullptr, nullptr, ws, ws_bytes, N, C, HW, stream);
}
