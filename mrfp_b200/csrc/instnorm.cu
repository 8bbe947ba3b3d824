// InstanceNorm2d(affine) [+ ReLU] [+ plane sums for NP+] with the plane RESIDENT ON CHIP, sm_100a (SURVEY.md 8f-3).
//
// The reference's trunk normalises per (n, c) plane at three places next to the MRFP insertion points
// (wt_layer=[0,0,4,4,4,0,0]): the stem (Resnet.py:534-536, 64 x 384^2 at a 768^2 crop), the end of layer1
// (Resnet.py:176-178 + :218-225, 256 x 192^2 — the producer of NP+ call 2) and the end of layer2 (512 x 96^2), each
// followed by a ReLU.  Unlike NP+, a plane's statistics need nothing from other planes, so a plane (or a slice of
// it) can stay in shared memory between the statistics and the write: one thread-block CLUSTER per plane, every CTA
// holds one slice (1-D TMA bulk loads, per-chunk mbarriers so the first reduction overlaps the loads), partial sums
// meet through distributed shared memory, and the plane is read from HBM exactly once:
//   forward   1R + 1W   (ATen: statistics + normalise + ReLU = 3R + 2W)
//   backward  2R + 1W   (gy and x once each; ATen: ReLU backward + batch-norm backward = 5R + 2W)
// Statistics are two-pass over the resident copy (mean first, then centred squares; double across lanes) — the same
// biased variance F.instance_norm uses.  Planes too large for an 8-CTA cluster fall back to re-reading global memory.
#include "hrfp.cuh"
#include "ptx.cuh"
#include <cooperative_groups.h>
#include <math.h>
#include <atomic>

namespace cg = cooperative_groups;

namespace mrfp {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kChunkElems = 4096;                 // 16 KiB per TMA bulk copy / mbarrier
constexpr int kMaxChunks = 16;                    // <= 256 KiB per buffer (more than shared memory holds)
constexpr int kMaxCluster = 8;                    // portable cluster size

struct Red2 { double a, b; };

// block-wide sum of two doubles (fixed order), result in every thread
__device__ __forceinline__ Red2 block_sum2(double a, double b, double (*s_w)[2]) {
  a = warp_sum(a); b = warp_sum(b);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();                                 // s_w may still be read from the previous round
  if (lane == 0) { s_w[warp][0] = a; s_w[warp][1] = b; }
  __syncthreads();
  Red2 r{0.0, 0.0};
#pragma unroll
  for (int i = 0; i < kWarps; ++i) { r.a += s_w[i][0]; r.b += s_w[i][1]; }
  return r;
}

// Cluster exchange, push model: every CTA WRITES its partials into each peer's shared memory, one cluster barrier, then
// everybody reads its own copy in rank order.  Nothing remote is read after the barrier, so a CTA may exit right after
// its last one (no trailing barrier).  cl_arrive() at kernel entry + cl_wait() before the first push guarantee that
// every peer has started (its shared memory exists) without ever blocking in practice.
__device__ __forceinline__ void cl_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cl_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
constexpr int kPubVals = 4;
__device__ __forceinline__ void cluster_push(cg::cluster_group& cluster, double (*s_pub)[kPubVals], unsigned cr, double v0, double v1,
                                             double v2, double v3) {
  if (threadIdx.x < cluster.num_blocks()) {
    double* dst = cluster.map_shared_rank(&s_pub[cr][0], threadIdx.x);
    dst[0] = v0; dst[1] = v1; dst[2] = v2; dst[3] = v3;
  }
  __syncwarp();
  cl_arrive();
  cl_wait();
}

// Brings the CTA's slice of one plane into shared memory.  VEC: chunked 1-D bulk copies (thread 0 issues, everyone
// waits per chunk while reducing); otherwise a plain element copy.
template <bool VEC>
__device__ __forceinline__ void issue_slice_load(float* dst, const float* src, int len, uint64_t* bars) {
  if (VEC) {
    if (threadIdx.x == 0) {
      const int nchunk = (len + kChunkElems - 1) / kChunkElems;
      for (int k = 0; k < nchunk; ++k) {
        const int n = min(kChunkElems, len - k * kChunkElems);
        ptx::mbar_expect_tx(&bars[k], (uint32_t)n * 4u);
        ptx::bulk_load(dst + k * kChunkElems, src + k * kChunkElems, (uint32_t)n * 4u, &bars[k]);
      }
    }
  } else {
    for (int i = threadIdx.x; i < len; i += kThreads) dst[i] = src[i];
  }
}

// ------------------------------------------------------------------------------------------------ forward
template <bool VEC, bool RESIDENT>
__global__ void __launch_bounds__(kThreads)
instnorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                    float* __restrict__ y, float* __restrict__ mean_out, float* __restrict__ invstd_out,
                    double* __restrict__ psum, int C, int HW, float eps, int relu, int slice) {
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned cs = cluster.num_blocks(), cr = cluster.block_rank();
  const long long plane = blockIdx.x / cs;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* buf = reinterpret_cast<float*>(smem_raw);
  __shared__ __align__(8) uint64_t bars[kMaxChunks];
  __shared__ double s_w[kWarps][2];
  __shared__ double s_pub[kMaxCluster][kPubVals];    // written by the peers (cluster_push)
  __shared__ double s_ps[kMaxCluster];
  __shared__ __align__(8) uint64_t ps_bar;           // rank 0: the plane-sum partials land here (st.async + complete_tx)
  if (cs > 1) {
    if (psum && cr == 0 && threadIdx.x == 0) {
      ptx::mbar_init(&ps_bar, 1);
      ptx::mbar_fence_init();
      ptx::mbar_expect_tx(&ps_bar, cs * 8u);
    }
    cl_arrive();                                   // matched by the cl_wait() in front of the first push
  }

  const int tid = threadIdx.x;
  const int begin = (int)cr * slice;
  const int len = max(0, min(slice, HW - begin));
  const float* src = x + plane * (long long)HW + begin;
  float* dst = y + plane * (long long)HW + begin;
  const int nchunk = (len + kChunkElems - 1) / kChunkElems;

  if (RESIDENT) {
    if (VEC) {
      if (tid == 0) {
        for (int k = 0; k < nchunk; ++k) ptx::mbar_init(&bars[k], 1);
        ptx::mbar_fence_init();
      }
      __syncthreads();
    }
    issue_slice_load<VEC>(buf, src, len, bars);
    if (!VEC) __syncthreads();
  }
  const float* in = RESIDENT ? buf : src;

  // pass 1: sum -> mean
  float acc = 0.f;
  if (VEC) {
    for (int k = 0; k < nchunk; ++k) {
      if (RESIDENT) ptx::mbar_wait(&bars[k], 0);
      const int n4 = min(kChunkElems, len - k * kChunkElems) >> 2;
      const float4* p = reinterpret_cast<const float4*>(in + k * kChunkElems);
      float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int i = tid; i < n4; i += kThreads) {
        const float4 v = RESIDENT ? p[i] : ld_stream_f4(p + i);
        a4.x += v.x; a4.y += v.y; a4.z += v.z; a4.w += v.w;
      }
      acc += (a4.x + a4.y) + (a4.z + a4.w);
    }
  } else {
    for (int i = tid; i < len; i += kThreads) acc += in[i];
  }
  // the slice's own mean first: the squares are centred locally, and ONE exchange combines the slices exactly
  const double sum_l = block_sum2((double)acc, 0.0, s_w).a;
  const float mean_l = len > 0 ? (float)(sum_l / (double)len) : 0.f;

  // pass 2: squares centred on the slice mean
  acc = 0.f;
  if (VEC) {
    const float4* p = reinterpret_cast<const float4*>(in);
    float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = tid; i < (len >> 2); i += kThreads) {
      const float4 v = p[i];
      const float dx = v.x - mean_l, dy = v.y - mean_l, dz = v.z - mean_l, dw = v.w - mean_l;
      a4.x = fmaf(dx, dx, a4.x); a4.y = fmaf(dy, dy, a4.y); a4.z = fmaf(dz, dz, a4.z); a4.w = fmaf(dw, dw, a4.w);
    }
    acc = (a4.x + a4.y) + (a4.z + a4.w);
  } else {
    for (int i = tid; i < len; i += kThreads) { const float d = in[i] - mean_l; acc = fmaf(d, d, acc); }
  }
  const double m2_l = block_sum2((double)acc, 0.0, s_w).a;
  // sum_x (x - mu)^2 = sum_k [ M2_k + 2 (m_k - mu)(S_k - n_k m_k) + n_k (m_k - mu)^2 ]   (m_k: the fp32 centre slice k used)
  double mu, m2 = 0.0;
  if (cs > 1) {
    cl_wait();                                     // (arrived at kernel entry) every peer is running
    cluster_push(cluster, s_pub, cr, sum_l, m2_l, (double)len, (double)mean_l);
    double tot = 0.0;
    for (unsigned k = 0; k < cs; ++k) tot += s_pub[k][0];
    mu = tot / (double)HW;
    for (unsigned k = 0; k < cs; ++k) {
      const double dm = s_pub[k][3] - mu;
      m2 += s_pub[k][1] + 2.0 * dm * (s_pub[k][0] - s_pub[k][2] * s_pub[k][3]) + s_pub[k][2] * dm * dm;
    }
  } else {
    mu = sum_l / (double)HW;
    const double dm = (double)mean_l - mu;
    m2 = m2_l + 2.0 * dm * (sum_l - (double)len * (double)mean_l) + (double)len * dm * dm;
  }
  const float mean = (float)mu;
  const float invstd = (float)(1.0 / sqrt(fmax(m2, 0.0) / (double)HW + (double)eps));

  // pass 3: y = (x - mean) * (gamma * invstd) + beta, optional ReLU, optional plane sum of y
  const int c = (int)(plane % C);
  const float a = (gamma ? gamma[c] : 1.f) * invstd, b = beta ? beta[c] : 0.f;
  const float lo = relu ? 0.f : -INFINITY;
  acc = 0.f;
  if (VEC) {
    const float4* p = reinterpret_cast<const float4*>(in);
    float4* q = reinterpret_cast<float4*>(dst);
    float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = tid; i < (len >> 2); i += kThreads) {
      float4 v = p[i];
      v.x = fmaxf(fmaf(v.x - mean, a, b), lo); v.y = fmaxf(fmaf(v.y - mean, a, b), lo);
      v.z = fmaxf(fmaf(v.z - mean, a, b), lo); v.w = fmaxf(fmaf(v.w - mean, a, b), lo);
      a4.x += v.x; a4.y += v.y; a4.z += v.z; a4.w += v.w;
      q[i] = v;
    }
    acc = (a4.x + a4.y) + (a4.z + a4.w);
  } else {
    for (int i = tid; i < len; i += kThreads) {
      const float v = fmaxf(fmaf(in[i] - mean, a, b), lo);
      acc += v;
      dst[i] = v;
    }
  }
  if (psum) {
    const double ys = block_sum2((double)acc, 0.0, s_w).a;
    if (cs > 1) {
      // Only rank 0 needs the partials, and this exchange comes AFTER the output stores: a cluster barrier here would
      // make every thread's release fence wait for its stores to drain (ncu: membar stalls).  An asynchronous remote
      // store that completes bytes on rank 0's mbarrier carries the value without any fence; the other CTAs are done.
      if (tid == 0) {
        uint32_t dst, bar;
        asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(dst) : "r"(ptx::smem_u32(&s_ps[cr])));
        asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(bar) : "r"(ptx::smem_u32(&ps_bar)));
        asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];"
                     ::"r"(dst), "l"(__double_as_longlong(ys)), "r"(bar) : "memory");
        if (cr == 0) {
          ptx::mbar_wait(&ps_bar, 0);
          double t = 0.0;
          for (unsigned k = 0; k < cs; ++k) t += s_ps[k];
          psum[plane] = t;
        }
      }
    } else if (tid == 0) {
      psum[plane] = ys;
    }
  }
  if (cr == 0 && tid == 0) { mean_out[plane] = mean; invstd_out[plane] = invstd; }
}

// ------------------------------------------------------------------------------------------------ backward
// xh = (x - mean) * invstd;  g' = gy * [y > 0] (ReLU variant; y recomputed with the forward's expression);
// S1 = sum g', S2 = sum g' * xh;  gx = gamma * invstd * (g' - S1/HW - xh * S2/HW);  d_gamma += S2, d_beta += S1.
template <bool VEC, bool RESIDENT>
__global__ void __launch_bounds__(kThreads)
instnorm_bwd_kernel(const float* __restrict__ gy, const float* __restrict__ x, const float* __restrict__ gamma,
                    const float* __restrict__ beta, const float* __restrict__ mean_in, const float* __restrict__ invstd_in,
                    float* __restrict__ gx, float* __restrict__ dgamma_part, float* __restrict__ dbeta_part, int C, int HW,
                    int relu, int slice, const float2* __restrict__ np_coef) {
  // np_coef (SURVEY.md 8f-1): the incoming tensor is the gradient of NP+(y), not of y; NP+'s own backward
  // gy = a'[plane] * g + b'[plane] is applied as the elements are consumed, so gy is never written or re-read
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned cs = cluster.num_blocks(), cr = cluster.block_rank();
  const long long plane = blockIdx.x / cs;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* bx = reinterpret_cast<float*>(smem_raw);
  float* bg = bx + slice;                          // slice is a multiple of 4: both buffers 16-byte aligned
  __shared__ __align__(8) uint64_t bars[2 * kMaxChunks];
  __shared__ double s_w[kWarps][2];
  __shared__ double s_pub[kMaxCluster][kPubVals];    // written by the peers (cluster_push)
  if (cs > 1) cl_arrive();                         // matched by the cl_wait() in front of the push

  const int tid = threadIdx.x;
  const int begin = (int)cr * slice;
  const int len = max(0, min(slice, HW - begin));
  const long long off = plane * (long long)HW + begin;
  const int nchunk = (len + kChunkElems - 1) / kChunkElems;

  if (RESIDENT) {
    if (VEC) {
      if (tid == 0) {
        for (int k = 0; k < 2 * nchunk; ++k) ptx::mbar_init(&bars[k], 1);
        ptx::mbar_fence_init();
      }
      __syncthreads();
      if (tid == 0) {                               // interleave the two streams chunk by chunk
        for (int k = 0; k < nchunk; ++k) {
          const uint32_t nb = (uint32_t)min(kChunkElems, len - k * kChunkElems) * 4u;
          ptx::mbar_expect_tx(&bars[2 * k], nb);
          ptx::bulk_load(bx + k * kChunkElems, x + off + k * kChunkElems, nb, &bars[2 * k]);
          ptx::mbar_expect_tx(&bars[2 * k + 1], nb);
          ptx::bulk_load(bg + k * kChunkElems, gy + off + k * kChunkElems, nb, &bars[2 * k + 1]);
        }
      }
    } else {
      for (int i = tid; i < len; i += kThreads) { bx[i] = x[off + i]; bg[i] = gy[off + i]; }
      __syncthreads();
    }
  }
  const int c = (int)(plane % C);
  const float mean = mean_in[plane], invstd = invstd_in[plane];
  const float gm = gamma ? gamma[c] : 1.f;
  const float a = gm * invstd, b = beta ? beta[c] : 0.f;
  const float2 npc = np_coef ? np_coef[plane] : make_float2(1.f, 0.f);
  const float* px = RESIDENT ? bx : x + off;
  const float* pg = RESIDENT ? bg : gy + off;

  // pass 1: xh and g' (kept in place when resident), S1, S2
  float s1 = 0.f, s2 = 0.f;
  auto one = [&](float xv, float gv, float& xh, float& gp) {
    const float d = xv - mean;
    xh = d * invstd;
    gp = (relu && !(fmaf(d, a, b) > 0.f)) ? 0.f : fmaf(npc.x, gv, npc.y);
    s1 += gp;
    s2 = fmaf(gp, xh, s2);
  };
  if (VEC) {
    for (int k = 0; k < nchunk; ++k) {
      if (RESIDENT) { ptx::mbar_wait(&bars[2 * k], 0); ptx::mbar_wait(&bars[2 * k + 1], 0); }
      const int n4 = min(kChunkElems, len - k * kChunkElems) >> 2;
      const float4* p = reinterpret_cast<const float4*>(px + k * kChunkElems);
      const float4* q = reinterpret_cast<const float4*>(pg + k * kChunkElems);
      for (int i = tid; i < n4; i += kThreads) {
        const float4 xv = RESIDENT ? p[i] : ld_stream_f4(p + i);
        const float4 gv = RESIDENT ? q[i] : ld_stream_f4(q + i);
        float4 xh, gp;
        one(xv.x, gv.x, xh.x, gp.x); one(xv.y, gv.y, xh.y, gp.y); one(xv.z, gv.z, xh.z, gp.z); one(xv.w, gv.w, xh.w, gp.w);
        if (RESIDENT) {
          reinterpret_cast<float4*>(bx + k * kChunkElems)[i] = xh;
          reinterpret_cast<float4*>(bg + k * kChunkElems)[i] = gp;
        }
      }
    }
  } else {
    for (int i = tid; i < len; i += kThreads) {
      float xh, gp;
      one(px[i], pg[i], xh, gp);
      if (RESIDENT) { bx[i] = xh; bg[i] = gp; }
    }
  }
  Red2 t = block_sum2((double)s1, (double)s2, s_w);
  if (cs > 1) {
    cl_wait();
    cluster_push(cluster, s_pub, cr, t.a, t.b, 0.0, 0.0);
    t.a = 0.0; t.b = 0.0;
    for (unsigned k = 0; k < cs; ++k) { t.a += s_pub[k][0]; t.b += s_pub[k][1]; }
  }
  const float m1 = (float)(t.a / (double)HW), m2 = (float)(t.b / (double)HW);

  // pass 2: gx (each thread re-reads exactly the elements it wrote in pass 1)
  float* out = gx + off;
  auto fin = [&](float xh, float gp) { return a * (gp - m1 - xh * m2); };
  if (VEC) {
    for (int i = tid; i < (len >> 2); i += kThreads) {
      float4 xh, gp;
      if (RESIDENT) {
        xh = reinterpret_cast<const float4*>(bx)[i];
        gp = reinterpret_cast<const float4*>(bg)[i];
      } else {
        const float4 xv = reinterpret_cast<const float4*>(px)[i], gv = reinterpret_cast<const float4*>(pg)[i];
        const float s1_keep = s1, s2_keep = s2;      // (the sums are final: `one` is reused only for its xh / g')
        one(xv.x, gv.x, xh.x, gp.x); one(xv.y, gv.y, xh.y, gp.y); one(xv.z, gv.z, xh.z, gp.z); one(xv.w, gv.w, xh.w, gp.w);
        s1 = s1_keep; s2 = s2_keep;
      }
      reinterpret_cast<float4*>(out)[i] = make_float4(fin(xh.x, gp.x), fin(xh.y, gp.y), fin(xh.z, gp.z), fin(xh.w, gp.w));
    }
  } else {
    for (int i = tid; i < len; i += kThreads) {
      float xh, gp;
      if (RESIDENT) { xh = bx[i]; gp = bg[i]; }
      else { const float s1_keep = s1, s2_keep = s2; one(px[i], pg[i], xh, gp); s1 = s1_keep; s2 = s2_keep; }
      out[i] = fin(xh, gp);
    }
  }
  if (cr == 0 && tid == 0) { dgamma_part[plane] = (float)t.b; dbeta_part[plane] = (float)t.a; }
}

// slice geometry: the smallest cluster whose slice fits `want` bytes per buffer set, else the largest cluster if it
// fits `cap`, else non-resident (slices are still spread over an 8-CTA cluster so one plane keeps 8 SMs busy)
struct Geo { int cs, slice; bool resident; size_t smem; };
Geo pick_geo(int HW, int nbuf, int max_smem_optin) {
  constexpr int want_kb = 72;      // three CTAs per SM; 48 KB and 144-200 KB slices measured slower (profiles/README.md)
  const size_t want = (size_t)(want_kb > 0 ? want_kb : 72) << 10;
  const size_t cap = (size_t)max_smem_optin - 2048;              // static shared memory of the kernels
  Geo g{};
  for (int pass = 0; pass < 2; ++pass) {
    const size_t lim = pass == 0 ? (want < cap ? want : cap) : cap;
    for (int cs = 1; cs <= kMaxCluster; cs *= 2) {
      const int slice = (int)align_up((size_t)(HW + cs - 1) / cs, 4);
      const size_t bytes = (size_t)slice * 4 * nbuf;
      if (bytes <= lim && slice <= kMaxChunks * kChunkElems) {
        g.cs = cs; g.slice = slice; g.resident = true; g.smem = bytes;
        return g;
      }
    }
  }
  g.cs = HW >= 8 * 16384 ? kMaxCluster : 1;
  g.slice = (int)align_up((size_t)(HW + g.cs - 1) / g.cs, 4);
  g.resident = false; g.smem = 0;
  return g;
}

// ------------------------------------------------------------------------------------------------ persistent ring variant
// The kernels above pay a load -> compute -> store sequence per CTA, so a CTA's HBM loads and stores never overlap
// (131 us for (8,256,192,192) forward with one CTA per SM where the traffic alone takes ~95 us).  Here a CTA (or cluster) is PERSISTENT and
// walks a sequence of planes: a producer lane streams 8 KiB chunks of consecutive planes into a 26-slot shared-memory
// ring with 1-D bulk copies; the consumers run the passes of plane p over its <= 18 resident chunks while the other
// slots already receive the head of the next plane, and every chunk's slot is handed back to the producer as soon
// as the output pass has stored it — loads of plane p+1 run under the compute and the stores of plane p.
// Same arithmetic, in the same order per CTA slice, as the kernels above (results are bit-identical for equal geometry).
constexpr int kRChunk = 2048;                    // floats per ring chunk (8 KiB)
constexpr int kRSlots = 26;                      // 208 KiB ring
constexpr int kRMaxRes = 18;                     // chunks of the plane in work a CTA may hold (x and gy together in backward)
constexpr int kRCons = 256;                      // consumer threads (8 warps) + one producer warp
constexpr int kRWarps = kRCons / 32;

struct RingArgs {
  const float* x; const float* gy; const float* gamma; const float* beta;
  float* out;                                    // forward: y; backward: gx
  float* mean; float* invstd;                    // forward: written; backward: read
  double* psum; float* dgamma_part; float* dbeta_part;
  int C, HW, relu, slice, planes;
  float eps;
};

__device__ __forceinline__ void cons_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kRCons) : "memory"); }

__device__ __forceinline__ Red2 cons_sum2(double a, double b, double (*s_w)[2]) {
  a = warp_sum(a); b = warp_sum(b);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  cons_bar();
  if (lane == 0) { s_w[warp][0] = a; s_w[warp][1] = b; }
  cons_bar();
  Red2 r{0.0, 0.0};
#pragma unroll
  for (int i = 0; i < kRWarps; ++i) { r.a += s_w[i][0]; r.b += s_w[i][1]; }
  return r;
}

// cluster-wide sum among the consumers; the producer warp joins every cluster barrier (ring_producer_sync)
__device__ __forceinline__ Red2 ring_cluster_sum2(cg::cluster_group& cluster, Red2 mine, double (*s_pub)[2], int& rnd) {
  const unsigned cs = cluster.num_blocks();
  if (cs == 1) return mine;
  const int slot = rnd % 3;                      // a slot is rewritten only after two further cluster barriers
  ++rnd;
  if (threadIdx.x == 0) { s_pub[slot][0] = mine.a; s_pub[slot][1] = mine.b; }
  cluster.sync();
  Red2 r{0.0, 0.0};
  for (unsigned k = 0; k < cs; ++k) {
    const double* remote = cluster.map_shared_rank(&s_pub[slot][0], k);
    r.a += remote[0]; r.b += remote[1];
  }
  return r;
}

template <bool BWD>
__global__ void __launch_bounds__(kRCons + 32, 1)
instnorm_ring_kernel(const RingArgs a) {
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned cs = cluster.num_blocks(), cr = cluster.block_rank();
  const int ncl = (int)(gridDim.x / cs), q = (int)(blockIdx.x / cs);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* ring = reinterpret_cast<float*>(smem_raw);                 // [kRSlots][kRChunk]
  __shared__ __align__(8) uint64_t full[kRSlots], empty[kRSlots];
  __shared__ double s_w[kRWarps][2];
  __shared__ double s_pub[3][2];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool is_producer = warp == kRWarps;
  const int begin = (int)cr * a.slice;
  const int len = max(0, min(a.slice, a.HW - begin));
  const int nch = (len + kRChunk - 1) / kRChunk;                    // chunks per stream of this CTA's slice
  constexpr int NB = BWD ? 2 : 1;
  const int F = NB * nch;                                           // ring fills per plane
  const int H = min(F, kRSlots - F);                                // fills of the NEXT plane that fit beside the one in work
  const int nsync = cs == 1 ? 0 : (BWD ? 1 : 2);                    // cluster barriers before the output pass

  if (tid == 0) {
    for (int s = 0; s < kRSlots; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], kRWarps); }
    ptx::mbar_fence_init();
  }
  __syncthreads();

  if (is_producer) {
    int fill = 0;
    auto issue = [&](int plane, int j0, int j1) {                   // fills j0..j1-1 of `plane` (lane 0 only)
      for (int j = j0; j < j1; ++j, ++fill) {
        const int slot = fill % kRSlots, round = fill / kRSlots;
        if (round > 0) ptx::mbar_wait(&empty[slot], (round - 1) & 1);
        const int chunk = BWD ? (j >> 1) : j;
        const float* base = (BWD && (j & 1)) ? a.gy : a.x;
        const uint32_t bytes = (uint32_t)min(kRChunk, len - chunk * kRChunk) * 4u;
        ptx::mbar_expect_tx(&full[slot], bytes);
        ptx::bulk_load(ring + (size_t)slot * kRChunk, base + (long long)plane * a.HW + begin + chunk * kRChunk, bytes, &full[slot]);
      }
    };
    if (lane == 0 && q < a.planes) issue(q, 0, F);
    for (int p = q; p < a.planes; p += ncl) {
      const int pn = p + ncl;
      if (lane == 0 && pn < a.planes) issue(pn, 0, H);              // slots freed by the output pass of the plane before p
      __syncwarp();
      for (int i = 0; i < nsync; ++i) cluster.sync();               // the statistics barriers of plane p
      if (lane == 0 && pn < a.planes) issue(pn, H, F);              // slots freed by the output pass of plane p
      __syncwarp();
      if (!BWD && a.psum && cs > 1) cluster.sync();                 // the plane-sum barrier after the output pass
    }
  } else {
    int cfill = 0, rnd = 0;
    for (int p = q; p < a.planes; p += ncl) {
      const int c = p % a.C;
      const float gm = a.gamma ? a.gamma[c] : 1.f, bt = a.beta ? a.beta[c] : 0.f;
      const long long off = (long long)p * a.HW + begin;
      auto slot_of = [&](int j) { return (cfill + j) % kRSlots; };
      auto wait_fill = [&](int j) { ptx::mbar_wait(&full[slot_of(j)], ((cfill + j) / kRSlots) & 1); };
      auto release = [&](int j) {                                   // this warp is done with fill j of the plane
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&empty[slot_of(j)]);
      };
      if (!BWD) {
        // pass 1: sum -> mean (chunk by chunk as the copies land)
        float acc = 0.f;
        for (int j = 0; j < nch; ++j) {
          wait_fill(j);
          const int n4 = min(kRChunk, len - j * kRChunk) >> 2;
          const float4* s4 = reinterpret_cast<const float4*>(ring + (size_t)slot_of(j) * kRChunk);
          float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
          for (int i = tid; i < n4; i += kRCons) { const float4 v = s4[i]; a4.x += v.x; a4.y += v.y; a4.z += v.z; a4.w += v.w; }
          acc += (a4.x + a4.y) + (a4.z + a4.w);
        }
        Red2 t = ring_cluster_sum2(cluster, cons_sum2((double)acc, 0.0, s_w), s_pub, rnd);
        const float mean = (float)(t.a / (double)a.HW);
        // pass 2: centred squares -> invstd
        float4 q4 = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = 0; j < nch; ++j) {
          const int n4 = min(kRChunk, len - j * kRChunk) >> 2;
          const float4* s4 = reinterpret_cast<const float4*>(ring + (size_t)slot_of(j) * kRChunk);
          for (int i = tid; i < n4; i += kRCons) {
            const float4 v = s4[i];
            const float dx = v.x - mean, dy = v.y - mean, dz = v.z - mean, dw = v.w - mean;
            q4.x = fmaf(dx, dx, q4.x); q4.y = fmaf(dy, dy, q4.y); q4.z = fmaf(dz, dz, q4.z); q4.w = fmaf(dw, dw, q4.w);
          }
        }
        t = ring_cluster_sum2(cluster, cons_sum2((double)((q4.x + q4.y) + (q4.z + q4.w)), 0.0, s_w), s_pub, rnd);
        const float invstd = (float)(1.0 / sqrt(t.a / (double)a.HW + (double)a.eps));
        // pass 3: normalise, ReLU, store; hand every chunk back as soon as this warp has read it
        const float sc = gm * invstd, lo = a.relu ? 0.f : -INFINITY;
        float4 y4 = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = 0; j < nch; ++j) {
          const int n4 = min(kRChunk, len - j * kRChunk) >> 2;
          const float4* s4 = reinterpret_cast<const float4*>(ring + (size_t)slot_of(j) * kRChunk);
          float4* d4 = reinterpret_cast<float4*>(a.out + off + j * kRChunk);
          for (int i = tid; i < n4; i += kRCons) {
            float4 v = s4[i];
            v.x = fmaxf(fmaf(v.x - mean, sc, bt), lo); v.y = fmaxf(fmaf(v.y - mean, sc, bt), lo);
            v.z = fmaxf(fmaf(v.z - mean, sc, bt), lo); v.w = fmaxf(fmaf(v.w - mean, sc, bt), lo);
            y4.x += v.x; y4.y += v.y; y4.z += v.z; y4.w += v.w;
            d4[i] = v;
          }
          release(j);
        }
        if (a.psum) {
          t = ring_cluster_sum2(cluster, cons_sum2((double)((y4.x + y4.y) + (y4.z + y4.w)), 0.0, s_w), s_pub, rnd);
          if (cr == 0 && tid == 0) a.psum[p] = t.a;
        }
        if (cr == 0 && tid == 0) { a.mean[p] = mean; a.invstd[p] = invstd; }
      } else {
        const float mean = a.mean[p], invstd = a.invstd[p];
        const float sc = gm * invstd;
        // pass 1: xhat and g' in place, S1, S2
        float s1 = 0.f, s2 = 0.f;
        auto one = [&](float& xv, float& gv) {
          const float d = xv - mean;
          xv = d * invstd;
          gv = (a.relu && !(fmaf(d, sc, bt) > 0.f)) ? 0.f : gv;
          s1 += gv;
          s2 = fmaf(gv, xv, s2);
        };
        for (int j = 0; j < nch; ++j) {
          wait_fill(2 * j); wait_fill(2 * j + 1);
          const int n4 = min(kRChunk, len - j * kRChunk) >> 2;
          float4* x4 = reinterpret_cast<float4*>(ring + (size_t)slot_of(2 * j) * kRChunk);
          float4* g4 = reinterpret_cast<float4*>(ring + (size_t)slot_of(2 * j + 1) * kRChunk);
          for (int i = tid; i < n4; i += kRCons) {
            float4 xv = x4[i], gv = g4[i];
            one(xv.x, gv.x); one(xv.y, gv.y); one(xv.z, gv.z); one(xv.w, gv.w);
            x4[i] = xv; g4[i] = gv;
          }
        }
        const Red2 t = ring_cluster_sum2(cluster, cons_sum2((double)s1, (double)s2, s_w), s_pub, rnd);
        const float m1 = (float)(t.a / (double)a.HW), m2 = (float)(t.b / (double)a.HW);
        // pass 2: gx (each thread re-reads exactly the elements it wrote in pass 1)
        for (int j = 0; j < nch; ++j) {
          const int n4 = min(kRChunk, len - j * kRChunk) >> 2;
          const float4* x4 = reinterpret_cast<const float4*>(ring + (size_t)slot_of(2 * j) * kRChunk);
          const float4* g4 = reinterpret_cast<const float4*>(ring + (size_t)slot_of(2 * j + 1) * kRChunk);
          float4* d4 = reinterpret_cast<float4*>(a.out + off + j * kRChunk);
          for (int i = tid; i < n4; i += kRCons) {
            const float4 xh = x4[i], gp = g4[i];
            d4[i] = make_float4(sc * (gp.x - m1 - xh.x * m2), sc * (gp.y - m1 - xh.y * m2), sc * (gp.z - m1 - xh.z * m2),
                                sc * (gp.w - m1 - xh.w * m2));
          }
          // the slots were written through the generic proxy: order those writes before the bulk copy that refills them
          ptx::fence_proxy_async_smem();
          release(2 * j); release(2 * j + 1);
        }
        if (cr == 0 && tid == 0) { a.dgamma_part[p] = (float)t.b; a.dbeta_part[p] = (float)t.a; }
      }
      cfill += F;
    }
  }
  if (cs > 1) cluster.sync();                      // peers may still be reading this CTA's published partials
}

// ring geometry: smallest cluster whose slice fits kRMaxRes chunks; 0 = not eligible / not chosen.
// Measured on B200 (tools/bench_instnorm.py, profiles/README.md): one consumer group per SM serialises the three
// passes of a plane, so the ring only wins where the one-shot kernels are down to ONE resident CTA per SM anyway (slices
// above ~100 KB: the backward of the 64 x 384^2 stem, 223 us vs 258 us); everywhere else several one-shot CTAs per SM
// overlap each other's loads and stores better (forward (8,256,192,192): 135 us vs 184 us).  MRFP_IN_RING = 0 never,
// 1 (default) only in that regime, 2 wherever the geometry allows.
int ring_cluster_size(int HW, int nbuf, size_t oneshot_smem) {
  static const int mode = getenv("MRFP_IN_RING") ? atoi(getenv("MRFP_IN_RING")) : 1;
  if (mode <= 0 || (HW & 3) || HW < kRChunk) return 0;
  if (mode == 1 && oneshot_smem <= (100u << 10)) return 0;
  for (int cs = 1; cs <= kMaxCluster; cs *= 2) {
    const int slice = (int)align_up((size_t)(HW + cs - 1) / cs, 4);
    if (nbuf * ((slice + kRChunk - 1) / kRChunk) <= kRMaxRes) return cs;
  }
  return 0;
}

template <bool BWD>
cudaError_t launch_ring(RingArgs a, int cs, int sm_count, cudaStream_t s) {
  constexpr size_t smem = (size_t)kRSlots * kRChunk * 4;
  auto kern = instnorm_ring_kernel<BWD>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  a.slice = (int)align_up((size_t)(a.HW + cs - 1) / cs, 4);
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(kRCons + 32); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int ncl = sm_count / cs;                        // one CTA per SM; clusters that cannot be co-resident simply run later
  if (cs > 1) {
    static std::atomic<int> cached[2][kMaxCluster + 1];          // co-resident clusters per (direction, cluster size); 0 = not asked yet
    int active = cached[BWD ? 1 : 0][cs].load(std::memory_order_relaxed);
    if (active == 0) {
      cfg.gridDim = dim3((unsigned)(ncl * cs));
      if (cudaOccupancyMaxActiveClusters(&active, kern, &cfg) != cudaSuccess || active <= 0) active = ncl;
      cached[BWD ? 1 : 0][cs].store(active, std::memory_order_relaxed);
    }
    if (active < ncl) ncl = active;
  }
  if (ncl > a.planes) ncl = a.planes;
  cfg.gridDim = dim3((unsigned)(ncl * cs));
  return cudaLaunchKernelEx(&cfg, kern, a);
}

template <typename K, typename... Args>
cudaError_t launch_cluster(K kern, long long planes, const Geo& g, cudaStream_t s, Args... args) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(planes * g.cs)); cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = g.smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)g.cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

}  // namespace
}  // namespace mrfp

using namespace mrfp;

extern "C" int mrfp_instnorm_fwd_f32(const float* x, const float* gamma, const float* beta, float* y, float* mean,
                                     float* invstd, double* psum, int N, int C, int HW, float eps, int relu, void* stream) {
  if (!x || !y || !mean || !invstd) return MRFP_ERR_NULL_POINTER;
  if (N <= 0 || C <= 0 || HW <= 0 || (long long)N * C > (1ll << 28)) return MRFP_ERR_BAD_SHAPE;
  if (psum && ((uintptr_t)psum & 7)) return MRFP_ERR_WORKSPACE;
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const bool vec = (HW & 3) == 0 && (((uintptr_t)x | (uintptr_t)y) & 15) == 0;
  cudaStream_t s = (cudaStream_t)stream;
  const long long planes = (long long)N * C;
  cudaError_t e;
  const Geo g = pick_geo(HW, 1, di.max_smem_optin);
  if (const int rcs = vec ? ring_cluster_size(HW, 1, g.resident ? g.smem : 0) : 0) {
    RingArgs a = {x, nullptr, gamma, beta, y, mean, invstd, psum, nullptr, nullptr, C, HW, relu, 0, (int)planes, eps};
    MRFP_CUDA_TRY(launch_ring<false>(a, rcs, di.sm_count, s));
    return MRFP_OK;
  }
  if (g.resident)
    e = vec ? launch_cluster(instnorm_fwd_kernel<true, true>, planes, g, s, x, gamma, beta, y, mean, invstd, psum, C, HW, eps, relu, g.slice)
            : launch_cluster(instnorm_fwd_kernel<false, true>, planes, g, s, x, gamma, beta, y, mean, invstd, psum, C, HW, eps, relu, g.slice);
  else
    e = vec ? launch_cluster(instnorm_fwd_kernel<true, false>, planes, g, s, x, gamma, beta, y, mean, invstd, psum, C, HW, eps, relu, g.slice)
            : launch_cluster(instnorm_fwd_kernel<false, false>, planes, g, s, x, gamma, beta, y, mean, invstd, psum, C, HW, eps, relu, g.slice);
  MRFP_CUDA_TRY(e);
  return MRFP_OK;
}

static int instnorm_bwd_impl(const float* gy, const float* x, const float* gamma, const float* beta, const float* mean,
                             const float* invstd, float* gx, float* dgamma_part, float* dbeta_part, int N, int C, int HW,
                             int relu, void* stream, const float2* np_coef) {
  if (!gy || !x || !mean || !invstd || !gx || !dgamma_part || !dbeta_part) return MRFP_ERR_NULL_POINTER;
  if (N <= 0 || C <= 0 || HW <= 0 || (long long)N * C > (1ll << 28)) return MRFP_ERR_BAD_SHAPE;
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const bool vec = (HW & 3) == 0 && (((uintptr_t)x | (uintptr_t)gy | (uintptr_t)gx) & 15) == 0;
  cudaStream_t s = (cudaStream_t)stream;
  const long long planes = (long long)N * C;
  cudaError_t e;
  const Geo g = pick_geo(HW, 2, di.max_smem_optin);
  if (const int rcs = (vec && !np_coef) ? ring_cluster_size(HW, 2, g.resident ? g.smem : 0) : 0) {
    RingArgs a = {x, gy, gamma, beta, gx, const_cast<float*>(mean), const_cast<float*>(invstd), nullptr, dgamma_part, dbeta_part,
                  C, HW, relu, 0, (int)planes, 0.f};
    MRFP_CUDA_TRY(launch_ring<true>(a, rcs, di.sm_count, s));
    return MRFP_OK;
  }
  if (g.resident)
    e = vec ? launch_cluster(instnorm_bwd_kernel<true, true>, planes, g, s, gy, x, gamma, beta, mean, invstd, gx, dgamma_part, dbeta_part, C, HW, relu, g.slice, np_coef)
            : launch_cluster(instnorm_bwd_kernel<false, true>, planes, g, s, gy, x, gamma, beta, mean, invstd, gx, dgamma_part, dbeta_part, C, HW, relu, g.slice, np_coef);
  else
    e = vec ? launch_cluster(instnorm_bwd_kernel<true, false>, planes, g, s, gy, x, gamma, beta, mean, invstd, gx, dgamma_part, dbeta_part, C, HW, relu, g.slice, np_coef)
            : launch_cluster(instnorm_bwd_kernel<false, false>, planes, g, s, gy, x, gamma, beta, mean, invstd, gx, dgamma_part, dbeta_part, C, HW, relu, g.slice, np_coef);
  MRFP_CUDA_TRY(e);
  return MRFP_OK;
}

extern "C" int mrfp_instnorm_bwd_f32(const float* gy, const float* x, const float* gamma, const float* beta,
                                     const float* mean, const float* invstd, float* gx, float* dgamma_part,
                                     float* dbeta_part, int N, int C, int HW, int relu, void* stream) {
  return instnorm_bwd_impl(gy, x, gamma, beta, mean, invstd, gx, dgamma_part, dbeta_part, N, C, HW, relu, stream, nullptr);
}

// Backward of  NP+(ReLU(InstanceNorm(x)))  in one chain of passes (SURVEY.md 8f-1: NP+ call 2, deepv3.py:334-335, folded
// into its producer's backward, Resnet.py:218-225): plane totals of g (1R) -> NP+ backward coefficients (one block) ->
// the InstanceNorm backward with gy = a'*g + b' applied on load (2R + 1W).  The gradient of the NP+ input is never
// written: 3R + 1W instead of (2R + 1W) + (2R + 1W).  ws: >= N*C*16 bytes, 16-byte aligned.
extern "C" int mrfp_instnorm_bwd_np_f32(const float* g, const float* x, const float* gamma, const float* beta,
                                        const float* mean, const float* invstd, const float* np_alpha, const float* np_eps,
                                        const float* np_mean, void* ws, size_t ws_bytes, float* gx, float* dgamma_part,
                                        float* dbeta_part, int N, int C, int HW, int relu, void* stream) {
  if (!g || !np_alpha || !np_eps || !np_mean || !ws) return MRFP_ERR_NULL_POINTER;
  if (N <= 0 || C <= 0 || HW <= 0) return MRFP_ERR_BAD_SHAPE;
  if (ws_bytes < (size_t)N * C * 16 || ((uintptr_t)ws & 15)) return MRFP_ERR_WORKSPACE;
  double* psum = reinterpret_cast<double*>(ws);
  float2* coef = reinterpret_cast<float2*>(psum + (size_t)N * C);
  cudaStream_t s = (cudaStream_t)stream;
  int rc = plane_sums(g, psum, (long long)N * C, HW, s);
  if (rc) return rc;
  rc = np_coef_launch(true, psum, np_alpha, np_eps, np_mean, coef, nullptr, nullptr, N, C, HW, s);
  if (rc) return rc;
  return instnorm_bwd_impl(g, x, gamma, beta, mean, invstd, gx, dgamma_part, dbeta_part, N, C, HW, relu, stream, coef);
}
