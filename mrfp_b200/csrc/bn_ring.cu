// Bulk-copy (TMA 1-D) forms of the row passes of the HRFP chain (bf16 NHWC), sm_100a.
//
// The LDG-based row kernels in hrfp.cu plateau near 4.3-4.8 TB/s of HBM reads (ncu: warps on the long scoreboard, HBM
// channels 32-63 % busy).  Here every pass runs as several single-buffered CTAs per SM: a CTA copies one work item (a row
// segment of <= 12-20 KiB plus the contiguous span of the other tensor it gathers from) with `cp.async.bulk` + mbarrier
// complete_tx, waits, computes from shared memory, writes results from registers and takes the next item; the copy /
// compute / store phases of the 3-5 CTAs on an SM overlap each other.  This is the form of the forward BN/ReLU/resample
// pass and of the BN-backward reduce and apply passes on the bf16 path (521 / 573 / 675 us vs 550 / 720 / 850 us for the
// LDG kernels; a single persistent ring per SM measured slower than both, profiles/README.md).
#include "hrfp.cuh"
#include "ptx.cuh"

namespace mrfp {
namespace {

using namespace ptx;

// U1[c] = sum mask*dA, U2[c] = sum mask*dA*y over all destination pixels; mask = [scale*y + shift > 0], y gathered.
// Each CTA copies one item (a <= 20 KiB gradient segment + the gathered span of the conv-output row) into its own buffer,
// waits, reduces from shared memory and takes the next item; four such CTAs per SM overlap each other's phases.
constexpr int kBDaBytes = 20480;
constexpr int kBYBytes = 26624;                 // 1.25x the segment (x0.8 down-sampling stages) + one pixel of 256 channels + slack
constexpr int kBThreads = 256;

__global__ void __launch_bounds__(kBThreads, 4)
bn_bwd_reduce_bulk_kernel(const __nv_bfloat16* __restrict__ dA, const __nv_bfloat16* __restrict__ y,
                          const int* __restrict__ idx_h, const int* __restrict__ idx_w, const float* __restrict__ stats,
                          double* __restrict__ acc, int N, int C, int IH, int IW, int OH, int OW, int pseg, int nseg,
                          int items, int rev) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* s_da = smem_raw;
  unsigned char* s_y = smem_raw + kBDaBytes;
  __shared__ __align__(8) uint64_t bar;
  __shared__ float s_acc[2 * kMaxC];
  const int tid = threadIdx.x;
  const int cg = C >> 3, cgs = 31 - __clz(cg);
  const int c = (tid & (cg - 1)) << 3, pl = tid >> cgs, pstep = kBThreads >> cgs;
  if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  for (int i = tid; i < 2 * kMaxC; i += kBThreads) s_acc[i] = 0.f;
  __syncthreads();
  pdl_sync();
  float scale[8], shift[8], u1[8], u2[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    scale[j] = stats[2 * kMaxC + c + j]; shift[j] = stats[3 * kMaxC + c + j];
    u1[j] = 0.f; u2[j] = 0.f;
  }
  uint32_t phase = 0;
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int itr = rev ? items - 1 - it : it;
    const int row = itr / nseg, seg = itr - row * nseg;
    const int n = row / OH, oh = row - n * OH;
    const int ow0 = seg * pseg, npx = min(pseg, OW - ow0);
    const int s0 = idx_w[ow0];
    if (tid == 0) {
      const int s1 = idx_w[ow0 + npx - 1];
      const uint32_t dab = (uint32_t)(npx * C * 2), yb = (uint32_t)((s1 - s0 + 1) * C * 2);
      mbar_expect_tx(&bar, dab + yb);
      bulk_load(s_da, dA + ((long long)row * OW + ow0) * C, dab, &bar);
      bulk_load(s_y, y + (((long long)n * IH + idx_h[oh]) * IW + s0) * C, yb, &bar);
    }
    int j = pl < npx ? idx_w[ow0 + pl] - s0 : 0;         // first look-up travels with the copies
    mbar_wait(&bar, phase);
    phase ^= 1u;
    for (int px = pl; px < npx; px += pstep) {
      const int jn = px + pstep < npx ? idx_w[ow0 + px + pstep] - s0 : 0;
      float g[8], yv[8];
      unpack8(*reinterpret_cast<const uint4*>(s_da + ((size_t)px * C + c) * 2), g);
      unpack8(*reinterpret_cast<const uint4*>(s_y + ((size_t)j * C + c) * 2), yv);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float t = fmaf(scale[i], yv[i], shift[i]) > 0.f ? g[i] : 0.f;
        u1[i] += t;
        u2[i] = fmaf(t, yv[i], u2[i]);
      }
      j = jn;
    }
    __syncthreads();                                     // every read of the buffer precedes the next item's copies
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    atomicAdd(&s_acc[c + j], u1[j]);
    atomicAdd(&s_acc[kMaxC + c + j], u2[j]);
  }
  __syncthreads();
  for (int i = tid; i < C; i += kBThreads) {
    atomicAdd(acc + i, (double)s_acc[i]);
    atomicAdd(acc + kMaxC + i, (double)s_acc[kMaxC + i]);
  }
}


// BN-backward APPLY pass in the same shape: an item is a segment of one SOURCE row (its y values, <= 12 KiB) plus the
// contiguous spans of the <= 2 destination rows that hold its replicas (lo tables: replicas of source s are the
// destinations [lo[s], lo[s+1])); the result segment goes straight from registers to global memory.
//   dY[src] = P * [scale*y + shift > 0] * sum_replicas dA - cnt * (Q + R * y)        (constants as in hrfp.cu)
constexpr int kAYBytes = 12288;
constexpr int kADaBytes = 16384;                // per destination row: 1.25x the segment + one 256-channel pixel + slack

__global__ void __launch_bounds__(kBThreads, 3)
bn_bwd_apply_bulk_kernel(const __nv_bfloat16* __restrict__ dA, const __nv_bfloat16* __restrict__ y, __nv_bfloat16* __restrict__ dY,
                         const int* __restrict__ lo_h, const int* __restrict__ lo_w, const float* __restrict__ stats,
                         const float* __restrict__ gamma, const double* __restrict__ acc, int N, int C, int IH, int IW, int OH,
                         int OW, double count, int pseg, int nseg, int items, int rev, int c_real) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* s_y = smem_raw;
  unsigned char* s_da = smem_raw + kAYBytes;             // [2][kADaBytes]
  __shared__ __align__(8) uint64_t bar;
  __shared__ __align__(16) float s_scale[kMaxC], s_shift[kMaxC], s_P[kMaxC], s_Q[kMaxC], s_R[kMaxC];
  const int tid = threadIdx.x;
  const int cg = C >> 3, cgs = 31 - __clz(cg);
  const int c = (tid & (cg - 1)) << 3, pl = tid >> cgs, pstep = kBThreads >> cgs;
  if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  pdl_sync();
  for (int j = tid; j < C; j += kBThreads) {
    const double mean = stats[j], invstd = stats[kMaxC + j], gm = j < c_real ? gamma[j] : 0.f;   // padded channels: dY = 0
    s_scale[j] = stats[2 * kMaxC + j]; s_shift[j] = stats[3 * kMaxC + j];
    const double S1 = acc[j], S2 = invstd * (acc[kMaxC + j] - mean * S1);
    const double M1 = gm * S1 / count, M2 = gm * S2 / count;
    const double r = invstd * invstd * M2;
    s_P[j] = (float)(invstd * gm); s_R[j] = (float)r; s_Q[j] = (float)(invstd * M1 - mean * r);
  }
  __syncthreads();
  auto ld8 = [&](const float* t, float (&v)[8]) {
    const float4 a = *reinterpret_cast<const float4*>(t + c), b = *reinterpret_cast<const float4*>(t + c + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  };
  // the thread's constants stay in registers (3 CTAs per SM; reading them from shared memory at 4 CTAs per SM: 808 vs 680 us)
  float r_scale[8], r_shift[8], r_P[8], r_Q[8], r_R[8];
  ld8(s_scale, r_scale); ld8(s_shift, r_shift); ld8(s_P, r_P); ld8(s_Q, r_Q); ld8(s_R, r_R);
  uint32_t phase = 0;
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int itr = rev ? items - 1 - it : it;
    const int row = itr / nseg, seg = itr - row * nseg;  // row = n * IH + sy
    const int n = row / IH, sy = row - n * IH;
    const int x0 = seg * pseg, npx = min(pseg, IW - x0);
    const int h0 = lo_h[sy], nh = lo_h[sy + 1] - h0;      // <= 2 (host check)
    const int d0 = lo_w[x0], dspan = lo_w[x0 + npx] - d0;
    if (tid == 0) {
      const uint32_t yb = (uint32_t)(npx * C * 2), dab = (uint32_t)(dspan * C * 2);
      mbar_expect_tx(&bar, yb + (uint32_t)nh * dab);
      bulk_load(s_y, y + ((long long)row * IW + x0) * C, yb, &bar);
      if (dab)
        for (int a = 0; a < nh; ++a)
          bulk_load(s_da + (size_t)a * kADaBytes, dA + (((long long)n * OH + h0 + a) * OW + d0) * C, dab, &bar);
    }
    int w0 = 0, w1 = 0;
    if (pl < npx) { w0 = lo_w[x0 + pl]; w1 = lo_w[x0 + pl + 1]; }          // look-ups travel with the copies
    mbar_wait(&bar, phase);
    phase ^= 1u;
    for (int x = pl; x < npx; x += pstep) {
      int nw0 = 0, nw1 = 0;
      if (x + pstep < npx) { nw0 = lo_w[x0 + x + pstep]; nw1 = lo_w[x0 + x + pstep + 1]; }
      float sd[8], yv[8], o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) sd[j] = 0.f;
      for (int a = 0; a < nh; ++a)
        for (int b = w0; b < w1; ++b) {
          float g[8];
          unpack8(*reinterpret_cast<const uint4*>(s_da + (size_t)a * kADaBytes + ((size_t)(b - d0) * C + c) * 2), g);
#pragma unroll
          for (int j = 0; j < 8; ++j) sd[j] += g[j];
        }
      unpack8(*reinterpret_cast<const uint4*>(s_y + ((size_t)x * C + c) * 2), yv);
      const float cnt = (float)(nh * (w1 - w0));
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float t = fmaf(r_scale[j], yv[j], r_shift[j]) > 0.f ? sd[j] : 0.f;
        o[j] = r_P[j] * t - cnt * fmaf(r_R[j], yv[j], r_Q[j]);
      }
      *reinterpret_cast<uint4*>(dY + ((long long)row * IW + x0 + x) * C + c) = pack8(o);
      w0 = nw0; w1 = nw1;
    }
    __syncthreads();                                     // every read of the buffers precedes the next item's copies
  }
}


// Forward element-wise pass of a stage in the same shape: A_next[n][oh][ow][:] = ReLU(scale * Y[n][ih[oh]][iw[ow]][:] + shift).
// An item is a <= 16 KiB segment of one destination row; the span of the source row it gathers from arrives by one bulk
// copy, the result goes from registers to global memory.
constexpr int kFDstBytes = 16384;
constexpr int kFYBytes = 21504;                 // 1.25x (x0.8 down-sampling stages) + one 256-channel pixel + slack

__global__ void __launch_bounds__(kBThreads, 5)
bn_relu_resample_bulk_kernel(const __nv_bfloat16* __restrict__ y, __nv_bfloat16* __restrict__ a, const int* __restrict__ idx_h,
                             const int* __restrict__ idx_w, const float* __restrict__ scale, const float* __restrict__ shift,
                             int N, int C, int IH, int IW, int OH, int OW, int pseg, int nseg, int items, int rev) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x;
  const int cg = C >> 3, cgs = 31 - __clz(cg);
  const int c = (tid & (cg - 1)) << 3, pl = tid >> cgs, pstep = kBThreads >> cgs;
  if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  __syncthreads();
  pdl_sync();
  float sc[8], sf[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = scale[c + j]; sf[j] = shift[c + j]; }
  uint32_t phase = 0;
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int itr = rev ? items - 1 - it : it;
    const int row = itr / nseg, seg = itr - row * nseg;
    const int n = row / OH, oh = row - n * OH;
    const int ow0 = seg * pseg, npx = min(pseg, OW - ow0);
    const int s0 = idx_w[ow0];
    if (tid == 0) {
      const uint32_t yb = (uint32_t)((idx_w[ow0 + npx - 1] - s0 + 1) * C * 2);
      mbar_expect_tx(&bar, yb);
      bulk_load(smem_raw, y + (((long long)n * IH + idx_h[oh]) * IW + s0) * C, yb, &bar);
    }
    int j = pl < npx ? idx_w[ow0 + pl] - s0 : 0;         // first look-up travels with the copy
    mbar_wait(&bar, phase);
    phase ^= 1u;
    __nv_bfloat16* dst = a + ((long long)row * OW + ow0) * C + c;
    for (int px = pl; px < npx; px += pstep) {
      const int jn = px + pstep < npx ? idx_w[ow0 + px + pstep] - s0 : 0;
      float v[8];
      unpack8(*reinterpret_cast<const uint4*>(smem_raw + ((size_t)j * C + c) * 2), v);
      uint32_t w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        w[i] = pack_bf16x2(fmaxf(fmaf(sc[2 * i], v[2 * i], sf[2 * i]), 0.f), fmaxf(fmaf(sc[2 * i + 1], v[2 * i + 1], sf[2 * i + 1]), 0.f));
      *reinterpret_cast<uint4*>(dst + (size_t)px * C) = make_uint4(w[0], w[1], w[2], w[3]);
      j = jn;
    }
    __syncthreads();                                     // every read of the buffer precedes the next item's copy
  }
}

}  // namespace

int bn_relu_resample_bulk(const __nv_bfloat16* y, __nv_bfloat16* a, const int* idx_h, const int* idx_w, const int* host_idx_w,
                          const float* scale, const float* shift, int N, int C, int IH, int IW, int OH, int OW, bool reverse,
                          cudaStream_t stream) {
  if (C < 64 || C > kMaxC || (C & (C - 1))) return MRFP_ERR_UNSUPPORTED;
  int nseg = (OW * 2 * C + kFDstBytes - 1) / kFDstBytes;
  int pseg = (OW + nseg - 1) / nseg;
  for (;;) {
    bool ok = true;
    nseg = (OW + pseg - 1) / pseg;
    for (int sgi = 0; sgi < nseg && ok; ++sgi) {
      const int ow0 = sgi * pseg, ow1 = (ow0 + pseg < OW ? ow0 + pseg : OW) - 1;
      ok = (host_idx_w[ow1] - host_idx_w[ow0] + 1) * C * 2 <= kFYBytes;
    }
    if (ok) break;
    if (--pseg < 8) return MRFP_ERR_UNSUPPORTED;
  }
  const long long items = (long long)N * OH * nseg;
  if (items <= 0 || items > 0x3fffffff) return MRFP_ERR_UNSUPPORTED;
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const long long cap = (long long)di.sm_count * 5;
  launch_k(bn_relu_resample_bulk_kernel, dim3((unsigned)(items < cap ? items : cap)), dim3(kBThreads), (size_t)kFYBytes, stream, y, a,
           idx_h, idx_w, scale, shift, N, C, IH, IW, OH, OW, pseg, nseg, (int)items, reverse ? 1 : 0);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

int bn_bwd_apply_bulk(const __nv_bfloat16* dA, const __nv_bfloat16* y, __nv_bfloat16* dY, const int* lo_h, const int* lo_w,
                      const int* host_lo_h, const int* host_lo_w, const float* stats, const float* gamma, const double* acc,
                      int N, int C, int IH, int IW, int OH, int OW, double count, bool reverse, cudaStream_t stream, int c_real) {
  if (C < 64 || C > kMaxC || (C & (C - 1))) return MRFP_ERR_UNSUPPORTED;
  for (int i = 0; i < IH; ++i)
    if (host_lo_h[i + 1] - host_lo_h[i] > 2) return MRFP_ERR_UNSUPPORTED;        // two destination-row buffers
  int nseg = (IW * 2 * C + kAYBytes - 1) / kAYBytes;
  int pseg = (IW + nseg - 1) / nseg;
  for (;;) {
    bool ok = true;
    nseg = (IW + pseg - 1) / pseg;
    for (int sgi = 0; sgi < nseg && ok; ++sgi) {
      const int x0 = sgi * pseg, x1 = x0 + pseg < IW ? x0 + pseg : IW;
      ok = (host_lo_w[x1] - host_lo_w[x0]) * C * 2 <= kADaBytes;
    }
    if (ok) break;
    if (--pseg < 8) return MRFP_ERR_UNSUPPORTED;
  }
  const long long items = (long long)N * IH * nseg;
  if (items <= 0 || items > 0x3fffffff) return MRFP_ERR_UNSUPPORTED;
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const size_t smem = (size_t)kAYBytes + 2 * kADaBytes;
  MRFP_SMEM_OPT_IN(bn_bwd_apply_bulk_kernel, smem, di.device);
  const long long cap = (long long)di.sm_count * 3;
  launch_k(bn_bwd_apply_bulk_kernel, dim3((unsigned)(items < cap ? items : cap)), dim3(kBThreads), smem, stream, dA, y, dY, lo_h,
           lo_w, stats, gamma, acc, N, C, IH, IW, OH, OW, count, pseg, nseg, (int)items, reverse ? 1 : 0,
           c_real > 0 ? c_real : C);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

int bn_bwd_reduce_bulk(const __nv_bfloat16* dA, const __nv_bfloat16* y, const int* idx_h, const int* idx_w,
                       const int* host_idx_w, const float* stats, double* acc, int N, int C, int IH, int IW, int OH, int OW,
                       bool reverse, cudaStream_t stream) {
  if (C < 64 || C > kMaxC || (C & (C - 1))) return MRFP_ERR_UNSUPPORTED;
  int nseg = (OW * 2 * C + kBDaBytes - 1) / kBDaBytes;
  int pseg = (OW + nseg - 1) / nseg;                     // balanced segments
  for (;;) {
    bool ok = true;
    nseg = (OW + pseg - 1) / pseg;
    for (int sgi = 0; sgi < nseg && ok; ++sgi) {
      const int ow0 = sgi * pseg, ow1 = (ow0 + pseg < OW ? ow0 + pseg : OW) - 1;
      ok = (host_idx_w[ow1] - host_idx_w[ow0] + 1) * C * 2 <= kBYBytes;
    }
    if (ok) break;
    if (--pseg < 8) return MRFP_ERR_UNSUPPORTED;
  }
  const long long items = (long long)N * OH * nseg;
  if (items <= 0 || items > 0x3fffffff) return MRFP_ERR_UNSUPPORTED;
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const size_t smem = (size_t)kBDaBytes + kBYBytes;
  MRFP_SMEM_OPT_IN(bn_bwd_reduce_bulk_kernel, smem, di.device);
  const long long cap = (long long)di.sm_count * 4;
  launch_k(bn_bwd_reduce_bulk_kernel, dim3((unsigned)(items < cap ? items : cap)), dim3(kBThreads), smem, stream, dA, y, idx_h, idx_w,
           stats, acc, N, C, IH, IW, OH, OW, pseg, nseg, (int)items, reverse ? 1 : 0);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

}  // namespace mrfp
