// HRFP chain for sm_100a — replaces /root/reference/deepv3.py:320-330 (+ :355-357) and its autograd backward:
// 8 x [conv3x3 (frozen random weights, bias 0) -> nearest resample -> BatchNorm2d(train) -> ReLU].
//
// Data layout in HBM: activations and conv outputs are NHWC (channels innermost) in the plan's element type
// (bf16 for the tcgen05 path, fp32 for the CUDA-core parity path); the module boundary stays fp32 NCHW.
// Per stage k the forward runs
//   conv            A_k (NHWC, conv resolution) -> Y_k (saved), and in its epilogue the replication-count
//                   weighted per-channel sum / sum of squares (= BN batch statistics of the RESAMPLED tensor)
//   bn_finalize     (N,C)-free: mean, invstd, scale, shift, running-stat update (a-8)
//   bn_relu_resample   Y_k --gather by LUT, scale/shift, ReLU--> A_{k+1}      (one bandwidth pass)
// so the resampled / normalised / rectified tensors of the reference (4 passes per stage) never exist.
// Backward per stage: bn_bwd_reduce (sums over replicas) -> bn_bwd_apply (dY at conv resolution) -> dgrad conv
// (the same conv kernel with rotated, transposed weights).  No weight gradients (deepv3.py:221-237).
#include "hrfp.cuh"
#include "ptx.cuh"
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <new>

namespace mrfp {
namespace {

// ------------------------------------------------------------------------------------------------------
// element access: 8 consecutive channels
// ------------------------------------------------------------------------------------------------------
template <typename T> struct Elem;
template <> struct Elem<float> {
  static __device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  static __device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
  }
  static __device__ __forceinline__ float to_float(float x) { return x; }
  static __device__ __forceinline__ float from_float(float x) { return x; }
  struct Raw { float4 a, b; };                       // 8 channels as loaded, before unpacking
  static __device__ __forceinline__ Raw load_raw(const float* p) {
    return Raw{*reinterpret_cast<const float4*>(p), *reinterpret_cast<const float4*>(p + 4)};
  }
  static __device__ __forceinline__ void add_raw(const Raw& r, float (&v)[8]) {
    v[0] += r.a.x; v[1] += r.a.y; v[2] += r.a.z; v[3] += r.a.w; v[4] += r.b.x; v[5] += r.b.y; v[6] += r.b.z; v[7] += r.b.w;
  }
};
template <> struct Elem<__nv_bfloat16> {
  static __device__ __forceinline__ void load8(const __nv_bfloat16* p, float (&v)[8]) { unpack8(*reinterpret_cast<const uint4*>(p), v); }
  static __device__ __forceinline__ void store8(__nv_bfloat16* p, const float (&v)[8]) { *reinterpret_cast<uint4*>(p) = pack8(v); }
  static __device__ __forceinline__ float to_float(__nv_bfloat16 x) { return __bfloat162float(x); }
  static __device__ __forceinline__ __nv_bfloat16 from_float(float x) { return __float2bfloat16_rn(x); }
  typedef uint4 Raw;
  static __device__ __forceinline__ Raw load_raw(const __nv_bfloat16* p) { return *reinterpret_cast<const uint4*>(p); }
  static __device__ __forceinline__ void add_raw(const Raw& r, float (&v)[8]) {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] += __uint_as_float(w[i] << 16);
      v[2 * i + 1] += __uint_as_float(w[i] & 0xffff0000u);
    }
  }
};

// ------------------------------------------------------------------------------------------------------
// layout conversion at the module boundary
// ------------------------------------------------------------------------------------------------------
// Both kernels move a 64-channel x 128-pixel tile through shared memory, so the fp32 NCHW side is touched in 512-byte
// runs per channel (16-byte accesses, a full warp per run) and the NHWC side in whole 128-byte channel vectors.
constexpr int kLayPx = 128;
constexpr int kLayRow = 133;                          // odd row pitch; pixel px sits in column (px & 3) * 33 + (px >> 2),
__device__ __forceinline__ int lay_col(int px) { return (px & 3) * 33 + (px >> 2); }   // so both access patterns spread over the banks

// src fp32 [N][C][HW] -> dst T [N][HW][CD]; CD >= C is the stored channel count of a padded stem (channels C..CD-1 are
// written as zeros); accumulate adds into dst (gradient of OCout_dec joining the chain).
template <typename T>
__global__ void __launch_bounds__(256)
nchw_to_nhwc_kernel(const float* __restrict__ src, T* __restrict__ dst, int C, int CD, int HW, int accumulate,
                    double* __restrict__ psum) {
  pdl_sync();
  __shared__ float tile[64][kLayRow];   // [channel][lay_col(pixel)]
  // channel tiles fastest in the grid: the CTAs that write the slices of the same NHWC pixels run together
  const int n = blockIdx.z, c0 = blockIdx.x * 64, p0 = blockIdx.y * kLayPx, t = threadIdx.x;
  const float* s = src + (size_t)n * C * HW;
  T* d = dst + (size_t)n * CD * HW;
  const bool vec = (HW & 3) == 0 && ((uintptr_t)src & 15) == 0;
  {
    const int px = (t & 31) * 4, crow = t >> 5;
#pragma unroll
    for (int pass = 0; pass < 8; ++pass) {
      const int c = crow + pass * 8, p = p0 + px;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c0 + c < C) {
        const float* q = s + (size_t)(c0 + c) * HW + p;
        if (vec && p + 3 < HW) v = *reinterpret_cast<const float4*>(q);
        else {
          if (p < HW) v.x = q[0];
          if (p + 1 < HW) v.y = q[1];
          if (p + 2 < HW) v.z = q[2];
          if (p + 3 < HW) v.w = q[3];
        }
      }
      const int col = px >> 2;                          // lay_col(px + k) = 33 * k + col
      tile[c][col] = v.x; tile[c][33 + col] = v.y; tile[c][66 + col] = v.z; tile[c][99 + col] = v.w;
      if (psum) {                                        // plane totals for the fused NP+ (a warp = one channel row)
        const float ps = warp_sum((v.x + v.y) + (v.z + v.w));
        if ((t & 31) == 0 && c0 + c < C) atomicAdd(psum + (size_t)n * C + c0 + c, (double)ps);
      }
    }
  }
  __syncthreads();
  {
    const int cg = t & 7, pl = t >> 3;
#pragma unroll
    for (int pass = 0; pass < kLayPx / 32; ++pass) {
      const int px = pl + pass * 32, p = p0 + px, c = c0 + cg * 8;
      if (p < HW && c < CD) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = tile[cg * 8 + j][lay_col(px)];
        T* q = d + (size_t)p * CD + c;
        if (accumulate) {
          float o[8];
          Elem<T>::load8(q, o);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] += o[j];
        }
        Elem<T>::store8(q, v);
      }
    }
  }
}

// The same conversion for the bf16 path without the fp32 tile (plain form: no accumulation, no plane sums): a thread
// loads float4 = four consecutive pixels of one channel, packs two bf16 pairs, and `stmatrix.x4.trans` scatters the
// transposed 8x8 blocks into a [pixel][64 channels] bf16 tile (the per-lane row addresses are chosen so that a float4 is
// exactly the thread's share of two matrices: matrix rows {4i, 4i+1} and {4i+2, 4i+3}); the tile leaves as whole 128-byte
// channel vectors.  16-byte chunks are XOR-swizzled so that both the matrix stores and the row reads spread over the banks.
__device__ __forceinline__ int stm_swz(int px) { return (((px >> 2) & 3) << 1) | (px & 1); }

__global__ void __launch_bounds__(256)
nchw_to_nhwc_stm_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int C, int HW, double* __restrict__ psum) {
  pdl_sync();
  __shared__ __align__(128) unsigned char sm[kLayPx * 128];        // [pixel][64 ch bf16]
  const int n = blockIdx.z, c0 = blockIdx.x * 64, p0 = blockIdx.y * kLayPx, t = threadIdx.x;
  const int warp = t >> 5, lane = t & 31, q = lane & 3;
  const float* s = src + ((size_t)n * C + c0 + warp * 8 + (lane >> 2)) * HW + p0;   // this thread's channel row
  // row of matrix m (= lane >> 3) this lane addresses: pixel (within a 32-pixel group) 16 (m >> 1) + 4 (j >> 1) + 2 (m & 1) + (j & 1)
  const int j = lane & 7, m = lane >> 3;
  const int prow = 16 * (m >> 1) + 4 * (j >> 1) + 2 * (m & 1) + (j & 1);
  float csum = 0.f;                                   // this thread's share of its channel's plane total (fused NP+)
#pragma unroll
  for (int it = 0; it < kLayPx / 32; ++it) {
    const int pa = it * 32 + 4 * q, pb = pa + 16;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (p0 + pa < HW) a = *reinterpret_cast<const float4*>(s + pa);            // HW % 4 == 0: a float4 is in or out as a whole
    if (p0 + pb < HW) b = *reinterpret_cast<const float4*>(s + pb);
    csum += ((a.x + a.y) + (a.z + a.w)) + ((b.x + b.y) + (b.z + b.w));
    uint32_t r[4];
    {
      const __nv_bfloat162 h0 = __floats2bfloat162_rn(a.x, a.y), h1 = __floats2bfloat162_rn(a.z, a.w);
      const __nv_bfloat162 h2 = __floats2bfloat162_rn(b.x, b.y), h3 = __floats2bfloat162_rn(b.z, b.w);
      r[0] = *reinterpret_cast<const uint32_t*>(&h0); r[1] = *reinterpret_cast<const uint32_t*>(&h1);
      r[2] = *reinterpret_cast<const uint32_t*>(&h2); r[3] = *reinterpret_cast<const uint32_t*>(&h3);
    }
    const int px = it * 32 + prow;
    const uint32_t addr = ptx::smem_u32(sm + px * 128 + ((warp ^ stm_swz(px)) << 4));
    asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};"
                 ::"r"(addr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
  }
  if (psum) {                                         // the four lanes of a channel, then one double atomic per (CTA, channel)
    csum += __shfl_xor_sync(0xffffffffu, csum, 1);
    csum += __shfl_xor_sync(0xffffffffu, csum, 2);
    if (q == 0) atomicAdd(psum + (size_t)n * C + c0 + warp * 8 + (lane >> 2), (double)csum);
  }
  __syncthreads();
  __nv_bfloat16* d = dst + ((size_t)n * HW + p0) * C + c0;
#pragma unroll
  for (int k = 0; k < kLayPx * 8 / 256; ++k) {
    const int e = t + k * 256, px = e >> 3, chunk = e & 7;
    if (p0 + px < HW)
      *reinterpret_cast<uint4*>(d + (size_t)px * C + chunk * 8) =
          *reinterpret_cast<const uint4*>(sm + px * 128 + ((chunk ^ stm_swz(px)) << 4));
  }
}

// the stmatrix kernel serves the bf16 path when the tile decomposition is exact (no channel padding)
template <typename T>
static bool stm_layout_ok(int C, int CD, int HW, const float* src) {
  return sizeof(T) == 2 && C == CD && (C & 63) == 0 && (HW & 3) == 0 && ((uintptr_t)src & 15) == 0;
}

// out fp32 [N][C][OH][OW] = f(Y[n][ih[oh]][iw[ow]][c]) (+ add), f = identity or ReLU(scale*y + shift)
template <typename T, bool BILIN>
__global__ void __launch_bounds__(256)
nhwc_to_nchw_kernel(const T* __restrict__ y, float* __restrict__ out, const float* __restrict__ add,
                    const int* __restrict__ idx_h, const int* __restrict__ idx_w, const float* __restrict__ scale,
                    const float* __restrict__ shift, int C, int CS, int IH, int IW, int OH, int OW,
                    const float2* __restrict__ coef, const float* __restrict__ add_lo, int LH, int LW) {
  // C: channels of the fp32 NCHW side; CS >= C: channel stride of the NHWC side (padded stem)
  pdl_sync();
  __shared__ float tile[64][kLayRow];   // [channel][lay_col(pixel)]
  // flat grid, output rows fastest, then channel tiles, then w-tiles
  const int ct = (C + 63) >> 6, rows = (int)(gridDim.x / (((OW + kLayPx - 1) / kLayPx) * ct));
  const int orow = blockIdx.x % rows, rem = blockIdx.x / rows;
  const int n = orow / OH, oh = orow - n * OH, t = threadIdx.x;
  const int c0 = (rem % ct) * 64, w0 = (rem / ct) * kLayPx;
  const int sh = idx_h ? idx_h[oh] : oh;
  const T* row = y + ((size_t)n * IH + sh) * IW * CS;
  {
    const int cg = t & 7, pl = t >> 3, c = c0 + cg * 8;
    float sc[8], sf[8];
    if (scale && c < CS) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { sc[j] = scale[c + j]; sf[j] = shift[c + j]; }
    }
#pragma unroll
    for (int pass = 0; pass < kLayPx / 32; ++pass) {
      const int px = pl + pass * 32, ow = w0 + px;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
      if (ow < OW && c < CS) {
        const int sw = idx_w ? idx_w[ow] : ow;
        Elem<T>::load8(row + (size_t)sw * CS + c, v);
        if (scale) {
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = fmaxf(fmaf(sc[j], v[j], sf[j]), 0.f);
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) tile[cg * 8 + j][lay_col(px)] = v[j];
    }
  }
  __syncthreads();
  {
    const int px = (t & 31) * 4, crow = t >> 5;
    const bool vec = (OW & 3) == 0;
    if (BILIN) {
      // HRFP+ tail (deepv3.py:356-357): the add operand is Upsample(dec1) — bilinear, align_corners=True
      // (mynn.py:114-119) — evaluated here from the low-resolution tensor with ATen's own formula
      // (upsample_bilinear2d: src = dst * (in-1)/(out-1), lambda weights, same association), so dec1 at (h/2, w/2)
      // never exists.  Row and column weights are the same for every channel pass of this thread.
      const float rh = OH > 1 ? (float)(LH - 1) / (float)(OH - 1) : 0.f;
      const float rw = OW > 1 ? (float)(LW - 1) / (float)(OW - 1) : 0.f;
      const float h1r = rh * (float)oh;
      const int h1 = (int)h1r, h1p = h1 < LH - 1 ? 1 : 0;
      const float hl1 = h1r - (float)h1, hl0 = 1.f - hl1;
      int w1[4], w1p[4];
      float wl0[4], wl1[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ow = min(w0 + px + i, OW - 1);
        const float w1r = rw * (float)ow;
        w1[i] = (int)w1r;
        w1p[i] = w1[i] < LW - 1 ? 1 : 0;
        wl1[i] = w1r - (float)w1[i]; wl0[i] = 1.f - wl1[i];
      }
#pragma unroll
      for (int pass = 0; pass < 8; ++pass) {
        const int c = crow + pass * 8, ow = w0 + px;
        if (c0 + c < C && ow < OW) {
          const size_t o = (((size_t)n * C + c0 + c) * OH + oh) * OW + ow;
          const int col = px >> 2;
          const float vv[4] = {tile[c][col], tile[c][33 + col], tile[c][66 + col], tile[c][99 + col]};
          const float* r0 = add_lo + (((size_t)n * C + c0 + c) * LH + h1) * LW;
          const float* r1 = r0 + (size_t)h1p * LW;
          float res[4];
#pragma unroll
          for (int i = 0; i < 4; ++i)
            res[i] = vv[i] + (hl0 * (wl0[i] * r0[w1[i]] + wl1[i] * r0[w1[i] + w1p[i]]) +
                              hl1 * (wl0[i] * r1[w1[i]] + wl1[i] * r1[w1[i] + w1p[i]]));
          if (vec && ow + 3 < OW) *reinterpret_cast<float4*>(out + o) = make_float4(res[0], res[1], res[2], res[3]);
          else
            for (int i = 0; i < 4 && ow + i < OW; ++i) out[o + i] = res[i];
        }
      }
      return;
    }
#pragma unroll
    for (int pass = 0; pass < 8; ++pass) {
      const int c = crow + pass * 8, ow = w0 + px;
      if (c0 + c < C && ow < OW) {
        const size_t o = (((size_t)n * C + c0 + c) * OH + oh) * OW + ow;
        const int col = px >> 2;
        float4 v = make_float4(tile[c][col], tile[c][33 + col], tile[c][66 + col], tile[c][99 + col]);
        // out = v + add, or with the fused NP+: out = v + (a * add + b) with the plane's (a, b)
        const float2 ab = coef ? coef[(size_t)n * C + c0 + c] : make_float2(1.f, 0.f);
        if (vec && ow + 3 < OW) {
          if (add) {
            const float4 a4 = *reinterpret_cast<const float4*>(add + o);
            v.x += fmaf(ab.x, a4.x, ab.y); v.y += fmaf(ab.x, a4.y, ab.y); v.z += fmaf(ab.x, a4.z, ab.y); v.w += fmaf(ab.x, a4.w, ab.y);
          }
          *reinterpret_cast<float4*>(out + o) = v;
        } else {
          const float vv[4] = {v.x, v.y, v.z, v.w};
          for (int i = 0; i < 4 && ow + i < OW; ++i) out[o + i] = add ? vv[i] + fmaf(ab.x, add[o + i], ab.y) : vv[i];
        }
      }
    }
  }
}

// HRFP+ tail with the low-resolution operand STAGED by bulk copies (deepv3.py:356-357, the x2 Upsample of the reference
// geometry).  The generic BILIN path above issues 16 scalar global loads per four outputs (about six distinct values):
// it is bound by load latency, 909 us for 1.96 GB.  Here the two source rows a tile needs — for each of its CT channels
// the span [ws, ws + cnt) of rows h1 and h1 + h1p, at most 80 floats when the scale is <= 1/2 — arrive in shared memory
// as 2 CT 1-D bulk copies (one per thread, one mbarrier) while the threads gather and transpose the tile of Y.  The
// kernel is bound by instruction issue, not by memory (a staged variant that kept ATen's association and selected its
// taps from four consecutive floats ran at 978 us), so the interpolation is made separable: one vertical blend of the
// staged rows per tile, then two taps and three flops per output (same formula, different association: ~1 ulp from
// ATen's).
constexpr int kSegFloats = 72;                  // 64 + taps + alignment, rounded up to a multiple of 4
// CT channels per tile: 64 -> 71 KB (3 tiles per SM), 32 -> 35 KB (5-6 tiles per SM; the kernel is latency-bound, so the
// narrower tile wins although it touches the NHWC side in 64-byte pieces)
template <int CT> constexpr size_t staged_smem() { return sizeof(float) * (CT * kLayRow + CT * 2 * kSegFloats); }

template <typename T, int CT>
__global__ void __launch_bounds__(256, CT == 32 ? 5 : 3)
hrfp_plus_bilinear_staged_kernel(const T* __restrict__ y, float* __restrict__ out, const int* __restrict__ idx_h,
                                 const int* __restrict__ idx_w, const float* __restrict__ scale, const float* __restrict__ shift,
                                 int C, int IH, int IW, int OH, int OW, const float* __restrict__ add_lo, int LH, int LW) {
  pdl_sync();
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float (*tile)[kLayRow] = reinterpret_cast<float (*)[kLayRow]>(smem_raw);          // [channel][lay_col(pixel)]
  float* stage = reinterpret_cast<float*>(smem_raw) + CT * kLayRow;                 // [channel][row 0/1][kSegFloats]
  __shared__ __align__(8) uint64_t bar;
  const int ct = (C + CT - 1) / CT, rows = (int)(gridDim.x / (((OW + kLayPx - 1) / kLayPx) * ct));
  // channel tiles fastest: the CTAs that read the same NHWC pixels (each a 64-byte slice of a 512-byte pixel) run at the
  // same time, so a DRAM page is used by all of them while it is open (rows-fastest order: 724 us, see profiles/README.md)
  const int ctile = blockIdx.x % ct, rest = blockIdx.x / ct;
  const int orow = rest % rows, wtile = rest / rows;
  const int n = orow / OH, oh = orow - n * OH, t = threadIdx.x;
  const int c0 = ctile * CT, w0 = wtile * kLayPx;
  const int nch = min(CT, C - c0);
  // ATen's upsample_bilinear2d(align_corners=True) source coordinates
  const float rh = OH > 1 ? (float)(LH - 1) / (float)(OH - 1) : 0.f;
  const float rw = OW > 1 ? (float)(LW - 1) / (float)(OW - 1) : 0.f;
  const float h1r = rh * (float)oh;
  const int h1 = (int)h1r, h1p = h1 < LH - 1 ? 1 : 0;
  const float hl1 = h1r - (float)h1, hl0 = 1.f - hl1;
  const int ws = (int)(rw * (float)w0) & ~3;                                        // 16-byte aligned start of the staged span
  const int w_hi = min(LW - 1, (int)(rw * (float)min(w0 + kLayPx - 1, OW - 1)) + 1);
  const int cnt = min(kSegFloats, (w_hi - ws + 4) & ~3);
  if (t == 0) {
    ptx::mbar_init(&bar, 1);
    ptx::mbar_fence_init();
    ptx::mbar_expect_tx(&bar, (uint32_t)(nch * 2 * cnt) * 4u);
  }
  __syncthreads();
  if (t < 2 * nch) {
    const int c = t >> 1, r = t & 1;
    const float* src = add_lo + (((size_t)n * C + c0 + c) * LH + h1 + (r ? h1p : 0)) * LW + ws;
    ptx::bulk_load(stage + (size_t)t * kSegFloats, src, (uint32_t)cnt * 4u, &bar);
  }
  const int sh = idx_h ? idx_h[oh] : oh;
  const T* row = y + ((size_t)n * IH + sh) * IW * C;
  {
    constexpr int CG = CT / 8, PL = 256 / CG;            // channel groups of 8, pixel lanes
    const int cg = t % CG, pl = t / CG, c = c0 + cg * 8;
    float sc[8], sf[8];
    if (c < C) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { sc[j] = scale[c + j]; sf[j] = shift[c + j]; }
    }
#pragma unroll
    for (int pass = 0; pass < kLayPx / PL; ++pass) {
      const int px = pl + pass * PL, ow = w0 + px;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
      if (ow < OW && c < C) {
        const int sw = idx_w ? idx_w[ow] : ow;
        Elem<T>::load8(row + (size_t)sw * C + c, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaxf(fmaf(sc[j], v[j], sf[j]), 0.f);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) tile[cg * 8 + j][lay_col(px)] = v[j];
    }
  }
  __syncthreads();
  ptx::mbar_wait(&bar, 0);
  // vertical blend of the two staged rows, vb[c][k] = hl0 * r0[k] + hl1 * r1[k], written back over row 0 SPLIT BY PARITY
  // (even columns in floats [0, 36), odd columns in [36, 72)): at the x2 scale consecutive lanes read every second
  // column, which is a 2-way bank conflict on the plain layout and conflict-free on the split one
  {
    constexpr int TPC = 256 / CT, NB = (kSegFloats / 4 + TPC - 1) / TPC;    // threads per channel, float4 per thread
    const int c = t / TPC, k0 = t % TPC;
    float4 bl[NB];
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      const int k4 = k0 + q * TPC;
      if (c < nch && k4 < (cnt >> 2)) {
        const float4 a = reinterpret_cast<const float4*>(stage + (size_t)(2 * c) * kSegFloats)[k4];
        const float4 b = reinterpret_cast<const float4*>(stage + (size_t)(2 * c + 1) * kSegFloats)[k4];
        bl[q] = make_float4(fmaf(hl1, b.x, hl0 * a.x), fmaf(hl1, b.y, hl0 * a.y), fmaf(hl1, b.z, hl0 * a.z), fmaf(hl1, b.w, hl0 * a.w));
      }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      const int k4 = k0 + q * TPC;
      if (c < nch && k4 < (cnt >> 2)) {
        float* vb = stage + (size_t)(2 * c) * kSegFloats;
        *reinterpret_cast<float2*>(vb + 2 * k4) = make_float2(bl[q].x, bl[q].z);
        *reinterpret_cast<float2*>(vb + kSegFloats / 2 + 2 * k4) = make_float2(bl[q].y, bl[q].w);
      }
    }
  }
  __syncthreads();
  {
    const int px = (t & 31) * 4, crow = t >> 5;
    const bool vec = (OW & 3) == 0;
    int o0[4], o1[4];                                      // staged columns of the two horizontal taps of each output
    float wl0[4], wl1[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int ow = min(w0 + px + i, OW - 1);
      const float w1r = rw * (float)ow;
      const int w1 = (int)w1r;
      const int k0 = w1 - ws, k1 = k0 + (w1 < LW - 1 ? 1 : 0);
      o0[i] = (k0 & 1) * (kSegFloats / 2) + (k0 >> 1);     // parity-split position of column k
      o1[i] = (k1 & 1) * (kSegFloats / 2) + (k1 >> 1);
      wl1[i] = w1r - (float)w1; wl0[i] = 1.f - wl1[i];
    }
#pragma unroll
    for (int pass = 0; pass < CT / 8; ++pass) {
      const int c = crow + pass * 8, ow = w0 + px;
      if (c0 + c < C && ow < OW) {
        const size_t o = (((size_t)n * C + c0 + c) * OH + oh) * OW + ow;
        const int col = px >> 2;
        const float vv[4] = {tile[c][col], tile[c][33 + col], tile[c][66 + col], tile[c][99 + col]};
        const float* vb = stage + (size_t)(2 * c) * kSegFloats;
        float res[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) res[i] = vv[i] + fmaf(wl0[i], vb[o0[i]], wl1[i] * vb[o1[i]]);
        if (vec && ow + 3 < OW) *reinterpret_cast<float4*>(out + o) = make_float4(res[0], res[1], res[2], res[3]);
        else
          for (int i = 0; i < 4 && ow + i < OW; ++i) out[o + i] = res[i];
      }
    }
  }
}

// HRFP+ tail without the fp32 transposition tile (bf16 path).  The ablation of the staged kernel put 360 of its 724 us
// on "gather Y, BN/ReLU, scalar stores into a [channel][pixel] fp32 tile, read the tile back".  Here the source-pixel span
// of the tile's row arrives in shared memory AS bf16 NHWC (16-byte cp.async, chunks XOR-swizzled by the pixel index),
// and `ldmatrix.x4.trans` hands every thread, for one fixed channel, PAIRS OF CONSECUTIVE DESTINATION PIXELS: the eight
// row addresses a matrix takes are per-lane, so they also perform the nearest-neighbour gather.  BN/ReLU, the two
// horizontal taps of the (vertically pre-blended) low-resolution row and the add happen in registers; a warp's store
// instruction writes 32 contiguous bytes in each of eight channel planes.
constexpr int kLdmSeg = 76;                     // row pitch in floats: 76 * ch mod 32 = 12 * ch mod 32 is distinct for 8 channels
constexpr int kLdmSpan = 120;                   // source pixels a 128-pixel tile may gather from (128 * 332/384 + 2 = 113)
constexpr size_t kLdmSmem = (size_t)kLdmSpan * 128 + sizeof(float) * 64 * 2 * kLdmSeg + 128 * sizeof(float4) + 128 * sizeof(int);

__global__ void __launch_bounds__(256, 4)
hrfp_plus_tail_ldm_kernel(const __nv_bfloat16* __restrict__ y, float* __restrict__ out, const int* __restrict__ idx_h,
                          const int* __restrict__ idx_w, const float* __restrict__ scale, const float* __restrict__ shift,
                          int C, int IH, int IW, int OH, int OW, const float* __restrict__ add_lo, int LH, int LW) {
  pdl_sync();
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* ysm = smem_raw;                                                    // [span pixel][64 ch bf16], swizzled
  float* stage = reinterpret_cast<float*>(smem_raw + (size_t)kLdmSpan * 128);       // [row 0/1][channel][kLdmSeg]
  float4* pix = reinterpret_cast<float4*>(stage + 64 * 2 * kLdmSeg);               // per destination pixel: o0, o1, wl0, wl1
  int* spx = reinterpret_cast<int*>(pix + 128);                                     // per destination pixel: source pixel - s0
  __shared__ __align__(8) uint64_t bar;
  const int ct = C >> 6, rows = (int)(gridDim.x / (((OW + kLayPx - 1) / kLayPx) * ct));
  const int ctile = blockIdx.x % ct, rest = blockIdx.x / ct;                        // channel tiles fastest
  const int orow = rest % rows, wtile = rest / rows;
  const int n = orow / OH, oh = orow - n * OH, t = threadIdx.x;
  const int c0 = ctile * 64, w0 = wtile * kLayPx;
  const float rh = OH > 1 ? (float)(LH - 1) / (float)(OH - 1) : 0.f;               // ATen upsample_bilinear2d(align_corners=True)
  const float rw = OW > 1 ? (float)(LW - 1) / (float)(OW - 1) : 0.f;
  const float h1r = rh * (float)oh;
  const int h1 = (int)h1r, h1p = h1 < LH - 1 ? 1 : 0;
  const float hl1 = h1r - (float)h1, hl0 = 1.f - hl1;
  const int ws = (int)(rw * (float)w0) & ~3;
  const int w_last = min(w0 + kLayPx - 1, OW - 1);
  const int w_hi = min(LW - 1, (int)(rw * (float)w_last) + 1);
  const int cnt = min(kLdmSeg, (w_hi - ws + 4) & ~3);
  if (t == 0) {
    ptx::mbar_init(&bar, 1);
    ptx::mbar_fence_init();
    ptx::mbar_expect_tx(&bar, (uint32_t)(64 * 2 * cnt) * 4u);
  }
  __syncthreads();
  if (t < 128) {                                                                     // the two low-resolution rows of 64 channels
    const int c = t >> 1, r = t & 1;
    const float* src = add_lo + (((size_t)n * C + c0 + c) * LH + h1 + (r ? h1p : 0)) * LW + ws;
    ptx::bulk_load(stage + (size_t)(r * 64 + c) * kLdmSeg, src, (uint32_t)cnt * 4u, &bar);
  }
  // the span of the source row this tile gathers from, 64 channels of every pixel
  const int s0 = idx_w[w0], nsp = idx_w[w_last] - s0 + 1;
  const __nv_bfloat16* yrow = y + (((size_t)n * IH + idx_h[oh]) * IW + s0) * C + c0;
  for (int e = t; e < nsp * 8; e += 256) {
    const int p = e >> 3, ch = e & 7;
    const uint32_t dst = ptx::smem_u32(ysm + p * 128 + ((ch ^ (p & 7)) << 4));
    ptx::cp_async_cg16(dst, yrow + (size_t)p * C + ch * 8);
  }
  ptx::cp_async_commit();
  if (t < 128) {
    const int ow = min(w0 + t, OW - 1);
    const float w1r = rw * (float)ow;
    const int w1 = (int)w1r;
    const float wl1 = w1r - (float)w1;
    pix[t] = make_float4(__int_as_float(w1 - ws), __int_as_float(w1 - ws + (w1 < LW - 1 ? 1 : 0)), 1.f - wl1, wl1);
    spx[t] = idx_w[ow] - s0;
  }
  ptx::cp_async_wait<0>();
  ptx::mbar_wait(&bar, 0);
  __syncthreads();
  {                                                                                  // vertical blend in place over row 0
    const int c = t >> 2;
    float4* p0 = reinterpret_cast<float4*>(stage + (size_t)c * kLdmSeg);
    const float4* p1 = reinterpret_cast<const float4*>(stage + (size_t)(64 + c) * kLdmSeg);
    for (int k4 = t & 3; k4 < (cnt >> 2); k4 += 4) {
      const float4 a = p0[k4], b = p1[k4];
      p0[k4] = make_float4(fmaf(hl1, b.x, hl0 * a.x), fmaf(hl1, b.y, hl0 * a.y), fmaf(hl1, b.z, hl0 * a.z), fmaf(hl1, b.w, hl0 * a.w));
    }
  }
  __syncthreads();
  const int warp = t >> 5, lane = t & 31;
  const int ch = warp * 8 + (lane >> 2);                                             // this thread's channel, whole kernel
  const float sc = scale[c0 + ch], sf = shift[c0 + ch];
  const float* vb = stage + (size_t)ch * kLdmSeg;
  float* orow_p = out + (((size_t)n * C + c0 + ch) * OH + oh) * OW + w0;
  const bool pair_ok = (OW & 1) == 0;
#pragma unroll
  for (int iter = 0; iter < 4; ++iter) {
    // lane L supplies row (L & 7) of matrix (L >> 3): the source pixel of destination pixel (4 iter + L/8) * 8 + L%8
    const int sidx = spx[(4 * iter + (lane >> 3)) * 8 + (lane & 7)];
    const uint32_t addr = ptx::smem_u32(ysm + sidx * 128 + ((warp ^ (sidx & 7)) << 4));
    uint32_t r[4];
    ptx::ldsm_x4_trans(addr, r);
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const int px = (4 * iter + m) * 8 + 2 * (lane & 3);                            // this thread's pixel pair of matrix m
      const float y0 = fmaxf(fmaf(sc, __uint_as_float(r[m] << 16), sf), 0.f);
      const float y1 = fmaxf(fmaf(sc, __uint_as_float(r[m] & 0xffff0000u), sf), 0.f);
      const float4 t0 = pix[px], t1 = pix[px + 1];
      const float o0 = y0 + fmaf(t0.z, vb[__float_as_int(t0.x)], t0.w * vb[__float_as_int(t0.y)]);
      const float o1 = y1 + fmaf(t1.z, vb[__float_as_int(t1.x)], t1.w * vb[__float_as_int(t1.y)]);
      const int ow = w0 + px;
      if (pair_ok && ow + 1 < OW) *reinterpret_cast<float2*>(orow_p + px) = make_float2(o0, o1);
      else {
        if (ow < OW) orow_p[px] = o0;
        if (ow + 1 < OW) orow_p[px + 1] = o1;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// forward element-wise pass: A_next[n][oh][ow][c] = ReLU(scale[c] * Y[n][ih[oh]][iw[ow]][c] + shift[c])
// ------------------------------------------------------------------------------------------------------
// A block walks whole output rows (the source row is block-uniform); a thread keeps a fixed 8-channel group, so the
// BN scale/shift live in registers and no per-element index arithmetic is left.
template <typename T>
__global__ void __launch_bounds__(256)
bn_relu_resample_kernel(const T* __restrict__ y, T* __restrict__ a, const int* __restrict__ idx_h,
                        const int* __restrict__ idx_w, const float* __restrict__ scale,
                        const float* __restrict__ shift, int N, int C, int IH, int IW, int OH, int OW, int rev) {
  pdl_sync();
  const int cg = C >> 3, pstep = 256 / cg;
  const int c = (threadIdx.x % cg) << 3, pl = threadIdx.x / cg;
  float sc[8], sf[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = scale[c + j]; sf[j] = shift[c + j]; }
  for (int r = blockIdx.x; r < N * OH; r += gridDim.x) {
    const int row = rev ? N * OH - 1 - r : r;          // rev: start where the previous kernel of the chain ended (L2)
    const int n = row / OH, oh = row - n * OH;
    const T* yrow = y + ((size_t)n * IH + idx_h[oh]) * IW * C + c;
    T* arow = a + (size_t)row * OW * C + c;
    int ow = pl;
    for (; ow + 3 * pstep < OW; ow += 4 * pstep) {       // four independent 16-byte loads in flight per thread
      float v[4][8];
#pragma unroll
      for (int u = 0; u < 4; ++u) Elem<T>::load8(yrow + (size_t)idx_w[ow + u * pstep] * C, v[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[u][j] = fmaxf(fmaf(sc[j], v[u][j], sf[j]), 0.f);
        Elem<T>::store8(arow + (size_t)(ow + u * pstep) * C, v[u]);
      }
    }
    for (; ow < OW; ow += pstep) {
      float v[8];
      Elem<T>::load8(yrow + (size_t)idx_w[ow] * C, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaxf(fmaf(sc[j], v[j], sf[j]), 0.f);
      Elem<T>::store8(arow + (size_t)ow * C, v);
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// BN statistics finalisation (one block).  acc[0..C) = sum w*y, acc[kMaxC..) = sum w*y^2 over the conv
// output, w = replication count  ==  plain sums over the resampled tensor (SURVEY.md §4).
// ------------------------------------------------------------------------------------------------------
__global__ void bn_finalize_kernel(const double* __restrict__ acc, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float* __restrict__ stats, int C, int c_real,
                                   double count, float momentum, float eps) {
  pdl_sync();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const double mean = acc[c] / count;
    double var = acc[kMaxC + c] / count - mean * mean;
    if (var < 0) var = 0;
    const double invstd = 1.0 / sqrt(var + (double)eps);
    const bool live = c < c_real;                      // padded output channels (zero weights) are pinned to zero
    const float sc = live ? (float)((double)gamma[c] * invstd) : 0.f;
    const float b = (live && beta) ? beta[c] : 0.f;
    stats[0 * kMaxC + c] = (float)mean;
    stats[1 * kMaxC + c] = (float)invstd;
    stats[2 * kMaxC + c] = sc;
    stats[3 * kMaxC + c] = (float)((double)b - mean * (double)sc);
    if (live && running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    if (live && running_var) running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)(var * (count / (count - 1.0)));
  }
}

// ------------------------------------------------------------------------------------------------------
// CUDA-core direct 3x3 convolution, fp32 NHWC (tight-parity math mode).  w: [9][CIN][COUT].
// block = 128 threads: lanes = 32 consecutive pixels, warps = 4 groups of 16 output channels (64 per block).
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
conv3x3_direct_f32_kernel(const float* __restrict__ in, const float* __restrict__ w, float* __restrict__ out,
                          int N, int H, int W, int CIN, int COUT, int dil, const int* __restrict__ cnt_h,
                          const int* __restrict__ cnt_w, double* __restrict__ stat_acc) {
  pdl_sync();
  extern __shared__ float s_w[];   // [CIN][64]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long pix = (long long)blockIdx.x * 32 + lane;
  const bool valid = pix < (long long)N * H * W;
  const int x = (int)(pix % W), y = (int)((pix / W) % H), n = (int)(pix / ((long long)W * H));
  const int cb = blockIdx.y * 64;
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  for (int tap = 0; tap < 9; ++tap) {
    __syncthreads();
    for (int i = threadIdx.x; i < CIN * 64; i += 128) {
      const int ci = i >> 6, co = i & 63;
      s_w[i] = (cb + co < COUT) ? w[((size_t)tap * CIN + ci) * COUT + cb + co] : 0.f;
    }
    __syncthreads();
    const int yy = y + (tap / 3 - 1) * dil, xx = x + (tap % 3 - 1) * dil;
    if (valid && yy >= 0 && yy < H && xx >= 0 && xx < W) {
      const float4* ip = reinterpret_cast<const float4*>(in + (((size_t)n * H + yy) * W + xx) * CIN);
      for (int c4 = 0; c4 < CIN / 4; ++c4) {
        const float4 v = ip[c4];
        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4* wr = reinterpret_cast<const float4*>(s_w + (c4 * 4 + j) * 64 + warp * 16);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 ww = wr[q];
            acc[4 * q + 0] = fmaf(vv[j], ww.x, acc[4 * q + 0]);
            acc[4 * q + 1] = fmaf(vv[j], ww.y, acc[4 * q + 1]);
            acc[4 * q + 2] = fmaf(vv[j], ww.z, acc[4 * q + 2]);
            acc[4 * q + 3] = fmaf(vv[j], ww.w, acc[4 * q + 3]);
          }
        }
      }
    }
  }
  const int co0 = cb + warp * 16;
  if (valid && co0 < COUT) {
    float4* op = reinterpret_cast<float4*>(out + (size_t)pix * COUT + co0);
#pragma unroll
    for (int q = 0; q < 4; ++q) op[q] = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
  }
  if (stat_acc) {
    const float wgt = valid ? (float)(cnt_h[y] * cnt_w[x]) : 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float s1 = warp_sum(wgt * acc[i]);
      const float s2 = warp_sum(wgt * acc[i] * acc[i]);
      if (lane == 0 && co0 + i < COUT) {
        atomicAdd(stat_acc + co0 + i, (double)s1);
        atomicAdd(stat_acc + kMaxC + co0 + i, (double)s2);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// weight packing.  W: (cout_r, cin_r, 3, 3) fp32 OIHW; the packed tensor has cin x cout channels (>= the real counts for a
// padded stem: the extra rows / columns are zeros).
//   layout 0: out[tap][ci][co]     layout 1: out[tap][co][ci]  (K = ci contiguous)
//   flip: tap -> 8 - tap (dgrad: the kernel rotated by 180 degrees)
//   direct fwd   layout 0, no flip, fp32: out[tap][ci][co] = W[co][ci][tap]
//   direct dgrad layout 1, flip,    fp32: out[tap][co][ci] = W[co][ci][8-tap]   (conv input = co, output = ci)
//   tc fwd       layout 1, no flip, bf16 / fp32(tf32): rows = N = co, K = ci contiguous
//   tc dgrad     layout 0, flip,    bf16 / fp32(tf32): rows = N = ci, K = co contiguous
// ------------------------------------------------------------------------------------------------------
struct PackJobs {             // one launch packs every layer for both directions: blockIdx.y = job
  const float* W[2 * kHrfpStages];
  void* out[2 * kHrfpStages];
  int cin[2 * kHrfpStages], cout[2 * kHrfpStages], cin_r[2 * kHrfpStages], cout_r[2 * kHrfpStages];
  unsigned char layout[2 * kHrfpStages], flip[2 * kHrfpStages], bf16[2 * kHrfpStages];
};
__global__ void pack_weights_kernel(const PackJobs jobs) {
  pdl_sync();
  const int job = blockIdx.y;
  const float* __restrict__ W = jobs.W[job];
  void* __restrict__ out = jobs.out[job];
  const int cin = jobs.cin[job], cout = jobs.cout[job], cin_r = jobs.cin_r[job], cout_r = jobs.cout_r[job];
  const int layout = jobs.layout[job], flip = jobs.flip[job], bf16 = jobs.bf16[job];
  const int total = 9 * cin * cout;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int tap = i / (cin * cout), r = i % (cin * cout);
    int ci, co;
    if (layout == 0) { ci = r / cout; co = r % cout; } else { co = r / cin; ci = r % cin; }
    const int st = flip ? 8 - tap : tap;
    const float v = (ci < cin_r && co < cout_r) ? W[((size_t)co * cin_r + ci) * 9 + st] : 0.f;
    if (!bf16) reinterpret_cast<float*>(out)[i] = v;
    else reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
  }
}

// ------------------------------------------------------------------------------------------------------
// backward of [resample -> BN(train) -> ReLU] at one stage.  mask and xhat depend only on Y[src]:
//   reduce (over DESTINATION rows, both streams contiguous):  U1 = sum mask*dA,  U2 = sum mask*dA*y
//          -> S1 = U1, S2 = sum mask*dA*xhat = invstd*(U2 - mean*U1);  M1 = gamma*S1/count, M2 = gamma*S2/count
//   apply  (over SOURCE rows; the replicas of a source pixel are a contiguous <=2x2 rectangle of dA):
//          dY[src] = invstd*(mask*gamma*SdA - cnt*(M1 + xhat*M2)) = P*mask*SdA - cnt*(Q + R*y)
// Threads keep a fixed 8-channel group; a block walks whole rows so the row LUT entry is block-uniform.
// ------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256, 4)
bn_bwd_reduce_kernel(const T* __restrict__ dA, const T* __restrict__ y, const int* __restrict__ idx_h,
                     const int* __restrict__ idx_w, const float* __restrict__ stats, double* __restrict__ acc,
                     int N, int C, int IH, int IW, int OH, int OW, int rev) {
  pdl_sync();
  __shared__ float s_acc[2 * kMaxC];
  const int cg = C >> 3, pstep = 256 / cg;
  const int c = (threadIdx.x % cg) << 3, pl = threadIdx.x / cg;
  for (int i = threadIdx.x; i < 2 * kMaxC; i += 256) s_acc[i] = 0.f;
  float scale[8], shift[8], u1[8], u2[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    scale[j] = stats[2 * kMaxC + c + j]; shift[j] = stats[3 * kMaxC + c + j];
    u1[j] = 0.f; u2[j] = 0.f;
  }
  __syncthreads();
  for (int r = blockIdx.x; r < N * OH; r += gridDim.x) {
    const int row = rev ? N * OH - 1 - r : r;
    const int n = row / OH, oh = row % OH;
    const T* drow = dA + (size_t)row * OW * C + c;
    const T* yrow = y + ((size_t)n * IH + idx_h[oh]) * IW * C + c;
#pragma unroll 2
    for (int ow = pl; ow < OW; ow += pstep) {
      float g[8], yv[8];
      Elem<T>::load8(drow + (size_t)ow * C, g);
      Elem<T>::load8(yrow + (size_t)idx_w[ow] * C, yv);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float t = fmaf(scale[j], yv[j], shift[j]) > 0.f ? g[j] : 0.f;
        u1[j] += t;
        u2[j] = fmaf(t, yv[j], u2[j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    atomicAdd(&s_acc[c + j], u1[j]);
    atomicAdd(&s_acc[kMaxC + c + j], u2[j]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += 256) {
    atomicAdd(acc + i, (double)s_acc[i]);
    atomicAdd(acc + kMaxC + i, (double)s_acc[kMaxC + i]);
  }
}

template <typename T>
__global__ void __launch_bounds__(256, 3)
bn_bwd_apply_kernel(const T* __restrict__ dA, const T* __restrict__ y, T* __restrict__ dY,
                    const int* __restrict__ start_h, const int* __restrict__ cnt_h, const int* __restrict__ start_w,
                    const int* __restrict__ cnt_w, const float* __restrict__ stats, const float* __restrict__ gamma,
                    const double* __restrict__ acc, int N, int C, int IH, int IW, int OH, int OW, double count, int rev,
                    int c_real) {
  pdl_sync();
  // per-channel constants live in shared memory (read as two float4 per use): registers are kept for loads in flight
  __shared__ __align__(16) float s_scale[kMaxC], s_shift[kMaxC], s_P[kMaxC], s_Q[kMaxC], s_R[kMaxC];
  const int cg = C >> 3, pstep = 256 / cg;
  const int c = (threadIdx.x % cg) << 3, pl = threadIdx.x / cg;
  for (int j = threadIdx.x; j < C; j += 256) {
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
  // one source pixel: sum of its <= 2x2 replicas of dA (the reference geometry: x1.2 up, x0.8 down), general loop otherwise
  typedef typename Elem<T>::Raw Raw;
  // raw (still packed) loads of one source pixel: y and its <= 2x2 replicas of dA (the reference geometry: x1.2 up,
  // x0.8 down); zero bit patterns add nothing
  struct Px { Raw y, g00, g01, g10, g11; };
  auto fetch = [&](const T* yrow, const T* d0, int x, int nh, int w0, int nw) {
    Px p = {};
    p.y = Elem<T>::load_raw(yrow + (size_t)x * C);
    const bool a0 = nh > 0, a1 = nh > 1, b0 = nw > 0, b1 = nw > 1;
    const T* q = d0 + (size_t)w0 * C;
    if (a0 && b0) p.g00 = Elem<T>::load_raw(q);
    if (a0 && b1) p.g01 = Elem<T>::load_raw(q + C);
    if (a1 && b0) p.g10 = Elem<T>::load_raw(q + (size_t)OW * C);
    if (a1 && b1) p.g11 = Elem<T>::load_raw(q + (size_t)OW * C + C);
    return p;
  };
  auto finish = [&](const float (&sd)[8], const Raw& yraw, float cnt, T* dst) {
    float o[8], yv[8], k0[8], k1[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) yv[j] = 0.f;
    Elem<T>::add_raw(yraw, yv);
    ld8(s_scale, k0); ld8(s_shift, k1);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaf(k0[j], yv[j], k1[j]) > 0.f ? sd[j] : 0.f;
    ld8(s_P, k0);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] *= k0[j];
    ld8(s_R, k0); ld8(s_Q, k1);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] -= cnt * fmaf(k0[j], yv[j], k1[j]);
    Elem<T>::store8(dst, o);
  };
  auto finish_px = [&](const Px& p, float cnt, T* dst) {
    float sd[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) sd[j] = 0.f;
    Elem<T>::add_raw(p.g00, sd); Elem<T>::add_raw(p.g01, sd); Elem<T>::add_raw(p.g10, sd); Elem<T>::add_raw(p.g11, sd);
    finish(sd, p.y, cnt, dst);
  };
  for (int r = blockIdx.x; r < N * IH; r += gridDim.x) {
    const int row = rev ? N * IH - 1 - r : r;
    const int n = row / IH, sy = row % IH;
    const int h0 = start_h[sy], nh = cnt_h[sy];
    const T* yrow = y + (size_t)row * IW * C + c;
    T* orow = dY + (size_t)row * IW * C + c;
    const T* d0 = dA + ((size_t)n * OH + h0) * OW * C + c;
    int x = pl;
    if (nh <= 2) {
      for (; x + pstep < IW; x += 2 * pstep) {           // two source pixels per iteration: up to 10 loads in flight
        const int x1 = x + pstep;
        const int wa = start_w[x], na = cnt_w[x], wb = start_w[x1], nb = cnt_w[x1];
        if (na > 2 || nb > 2) break;
        const Px pa = fetch(yrow, d0, x, nh, wa, na), pb = fetch(yrow, d0, x1, nh, wb, nb);
        finish_px(pa, (float)(nh * na), orow + (size_t)x * C);
        finish_px(pb, (float)(nh * nb), orow + (size_t)x1 * C);
      }
    }
    for (; x < IW; x += pstep) {                         // row remainder and any other geometry
      const int w0 = start_w[x], nw = cnt_w[x];
      float sd[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) sd[j] = 0.f;
      const Raw yraw = Elem<T>::load_raw(yrow + (size_t)x * C);
      for (int a = 0; a < nh; ++a)
        for (int b = 0; b < nw; ++b) Elem<T>::add_raw(Elem<T>::load_raw(d0 + ((size_t)a * OW + w0 + b) * C), sd);
      finish(sd, yraw, (float)(nh * nw), orow + (size_t)x * C);
    }
  }
}

// Same pass for a stage whose resample is the identity (OCdeclayer1: conv and output resolution are both h/2 x w/2):
// a flat stream, four pixels per thread in flight.
template <typename T>
__global__ void __launch_bounds__(256, 2)
bn_bwd_apply_identity_kernel(const T* __restrict__ dA, const T* __restrict__ y, T* __restrict__ dY,
                             const float* __restrict__ stats, const float* __restrict__ gamma,
                             const double* __restrict__ acc, long long npix, int C, double count, int rev, int c_real) {
  pdl_sync();
  const int cg = C >> 3, pstep = 256 / cg;
  const int c = (threadIdx.x % cg) << 3, pl = threadIdx.x / cg;
  float scale[8], shift[8], P[8], Q[8], R[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const double mean = stats[c + j], invstd = stats[kMaxC + c + j], gm = c + j < c_real ? gamma[c + j] : 0.f;
    scale[j] = stats[2 * kMaxC + c + j]; shift[j] = stats[3 * kMaxC + c + j];
    const double S1 = acc[c + j], S2 = invstd * (acc[kMaxC + c + j] - mean * S1);
    const double M1 = gm * S1 / count, M2 = gm * S2 / count;
    const double r = invstd * invstd * M2;
    P[j] = (float)(invstd * gm); R[j] = (float)r; Q[j] = (float)(invstd * M1 - mean * r);
  }
  typedef typename Elem<T>::Raw Raw;
  constexpr int U = 4;
  const long long chunk = (long long)U * pstep, nchunks = (npix + chunk - 1) / chunk;
  for (long long it = blockIdx.x; it < nchunks; it += gridDim.x) {
    const long long p0 = (rev ? nchunks - 1 - it : it) * chunk + pl;
    Raw g[U] = {}, yv[U] = {};
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long p = p0 + (long long)u * pstep;
      if (p < npix) {
        g[u] = Elem<T>::load_raw(dA + (size_t)p * C + c);
        yv[u] = Elem<T>::load_raw(y + (size_t)p * C + c);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long p = p0 + (long long)u * pstep;
      if (p < npix) {
        float gf[8], yf[8], o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { gf[j] = 0.f; yf[j] = 0.f; }
        Elem<T>::add_raw(g[u], gf); Elem<T>::add_raw(yv[u], yf);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float t = fmaf(scale[j], yf[j], shift[j]) > 0.f ? gf[j] : 0.f;
          o[j] = P[j] * t - fmaf(R[j], yf[j], Q[j]);
        }
        Elem<T>::store8(dY + (size_t)p * C + c, o);
      }
    }
  }
}

__global__ void add_f32_kernel(const float4* __restrict__ a, const float4* __restrict__ b, float4* __restrict__ o,
                               size_t n4, const float* a1, const float* b1, float* o1, size_t n) {
  pdl_sync();
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 x = ld_stream_f4(a + i), y = ld_stream_f4(b + i);
    st_stream_f4(o + i, make_float4(x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w));
  }
  for (size_t i = n4 * 4 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += stride) o1[i] = a1[i] + b1[i];
}

// ------------------------------------------------------------------------------------------------------
// NP+ call 1 folded into the chain (SURVEY.md 8f-1).  x = OCout + NP+(xp) with NP+(xp) = a[n,c]*xp + b[n,c]
// (deepv3.py:268-277, :316-318, :329-330): the plane totals of xp ride on the NCHW->NHWC pass that feeds the chain,
// one block turns them into the per-plane (a, b), and the chain's output pass applies them to its add operand —
// NP+(xp) is never written or re-read.  Backward mirrors it with the totals of g_ocout (gin = alpha*g + dL/dm/HW,
// SURVEY.md 8 a-1).  Same formulas, in double, as npplus.cu.
// ------------------------------------------------------------------------------------------------------
struct NpStem {
  const float* alpha;   // (N,C) draw #1
  const float* eps;     // (N,C) draw #2
  float* mean;          // (N,C) plane means: written by the forward, read by the backward
  float* beta;          // (N,C) forward diagnostic, may be null
  double* psum;         // (N,C) scratch: plane totals
  float2* coef;         // (N,C) scratch: (a, b)
};

template <bool BWD>
__global__ void __launch_bounds__(256)
np_stem_coef_kernel(const double* __restrict__ psum, const float* __restrict__ alpha, const float* __restrict__ eps,
                    const float* __restrict__ mean_in, float2* __restrict__ coef, float* __restrict__ mean_out,
                    float* __restrict__ beta_out, int N, int C, int HW) {
  pdl_sync();
  __shared__ double s_mbar[kMaxC], s_d[kMaxC], s_l[kMaxC];
  __shared__ double w_best[8], w_tsum[8];
  __shared__ int w_c[8], w_nan[8];
  __shared__ double s_dmax, s_T;
  __shared__ int s_cstar;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double inv_hw = 1.0 / (double)HW;
  double best = -1.0, tsum = 0.0;
  int bestc = 0x7fffffff;
  bool anynan = false;
  for (int c = tid; c < C; c += 256) {
    double sm = 0;
    for (int n = 0; n < N; ++n) sm += BWD ? (double)mean_in[n * C + c] : psum[n * C + c] * inv_hw;
    const double mbar = sm / (double)N;
    double q = 0, l = 0;
    for (int n = 0; n < N; ++n) {
      const double G = psum[n * C + c];
      const double m = BWD ? (double)mean_in[n * C + c] : G * inv_hw;
      q += (m - mbar) * (m - mbar);
      if (BWD) l += (double)eps[n * C + c] * m * G;                      // dL/ds[c] = sum_n eps*m*G
    }
    const double d = sqrt(q / (double)(N - 1));                           // N == 1 -> NaN, as torch.std (deepv3.py:272)
    s_mbar[c] = mbar; s_d[c] = d; s_l[c] = l;
    if (d != d) anynan = true;
    if (d > best) { best = d; bestc = c; }
    if (BWD) tsum += l * d;
  }
  for (int o = 16; o > 0; o >>= 1) {                                      // arg-max, first index wins, NaN-propagating
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oc = __shfl_xor_sync(0xffffffffu, bestc, o);
    const int on = __shfl_xor_sync(0xffffffffu, (int)anynan, o);
    tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
    if (ob > best || (ob == best && oc < bestc)) { best = ob; bestc = oc; }
    anynan = anynan || (on != 0);
  }
  if (lane == 0) { w_best[warp] = best; w_c[warp] = bestc; w_nan[warp] = anynan; w_tsum[warp] = tsum; }
  __syncthreads();
  if (tid == 0) {
    double b = w_best[0], t = w_tsum[0];
    int bc = w_c[0], nn = w_nan[0];
    for (int i = 1; i < 8; ++i) {
      if (w_best[i] > b || (w_best[i] == b && w_c[i] < bc)) { b = w_best[i]; bc = w_c[i]; }
      nn |= w_nan[i];
      t += w_tsum[i];
    }
    s_dmax = nn ? (double)NAN : b;
    s_cstar = bc;
    s_T = 1.5 * t / (s_dmax * s_dmax);
  }
  __syncthreads();
  const double dmax = s_dmax;
  for (int p = tid; p < N * C; p += 256) {
    const int c = p % C;
    const double a = (double)alpha[p], d = s_d[c];
    const double beta = 1.0 + (double)eps[p] * (d / dmax * 1.5);         // deepv3.py:273,275
    double b;
    if (!BWD) {
      const double m = psum[p] * inv_hw;
      b = (beta - a) * m;                                                 // out = a*x + (beta-a)*m  (:276)
      mean_out[p] = (float)m;
      if (beta_out) beta_out[p] = (float)beta;
    } else {
      const double m = (double)mean_in[p];
      double dLdd = 1.5 / dmax * s_l[c];
      if (c == s_cstar) dLdd -= s_T;
      const double dd_dm = (d == 0.0) ? 0.0 : (m - s_mbar[c]) / ((double)(N - 1) * d);   // std_backward zero-fills
      b = ((beta - a) * psum[p] + dLdd * dd_dm) * inv_hw;
    }
    coef[p] = make_float2((float)a, (float)b);
  }
}

// ------------------------------------------------------------------------------------------------------
// host: geometry (must be bit-identical to ATen's upsample_nearest2d index rule)
// ------------------------------------------------------------------------------------------------------
float index_scale(int in, int out, bool has_sf, double sf) { return has_sf ? (float)(1.0 / sf) : ((float)in / (float)out); }
void make_index(int in, int out, bool has_sf, double sf, int* idx) {
  const float scale = index_scale(in, out, has_sf, sf);
  for (int d = 0; d < out; ++d) {
    int s = (int)floorf((float)d * scale);
    idx[d] = s < in - 1 ? s : in - 1;
  }
}

int grid_for(long long work_items, int block, int sm_count, int waves = 8) {
  long long g = (work_items + block - 1) / block;
  const long long cap = (long long)sm_count * waves;
  if (g > cap) g = cap;
  return g < 1 ? 1 : (int)g;
}

// blocks for a row-walking kernel (several waves of blocks: a plain cap measured better than an even split)
int even_grid(int rows, int cap) { return rows < cap ? rows : cap; }

bool pow2_ge8(int c) { return c >= 8 && c <= kMaxC && (c & (c - 1)) == 0; }

// Stored channel count of the stem inside the chain: the row kernels keep fixed 8-channel groups with a power-of-two
// number of groups, the tensor-core convolutions need K and N in multiples of 64 — a narrower or odd stem
// (MobileNetV2: 16, ShuffleNetV2: 24 / 116 channels, SURVEY.md 8f-2) is zero-padded to the next such width.  The
// padded input channels meet zero weights, the padded output channels have zero weights, BN scale and shift.
int stem_pad(int cin, int mode) {
  int p = 8;
  while (p < cin) p <<= 1;
  const int lo = mode == MRFP_MATH_FP32 ? 16 : 64;
  return p < lo ? lo : p;
}

constexpr size_t kDirectConvSmemMax = (size_t)kMaxC * 64 * sizeof(float);

template <typename T>
int launch_direct_conv(const T* in, const void* w, T* out, int N, int H, int W, int cin, int cout, int dil, const int* cnt_h,
                       const int* cnt_w, double* acc, const DeviceInfo& di, cudaStream_t s) {
  if constexpr (sizeof(T) == 4) {
    dim3 g((unsigned)(((long long)N * H * W + 31) / 32), (cout + 63) / 64);
    const size_t smem = (size_t)cin * 64 * sizeof(float);
    MRFP_SMEM_OPT_IN(conv3x3_direct_f32_kernel, kDirectConvSmemMax, di.device);
    launch_k(conv3x3_direct_f32_kernel, dim3(g), dim3(128), smem, s, in, reinterpret_cast<const float*>(w), out, N, H, W, cin, cout,
             dil, cnt_h, cnt_w, acc);
    return MRFP_OK;
  } else {
    return MRFP_ERR_UNSUPPORTED;
  }
}

// --- single passes of a stage, shared by the chain and by the debug hooks (variant 0: LDG row kernel, 1: product path) ---
template <typename T>
int run_resample(const mrfp_hrfp_plan* P, int k, const int* lut, const T* Y, T* A, const float* stats, bool rev, bool bulk,
                 const DeviceInfo& di, cudaStream_t s) {
  const HrfpStage& st = P->st[k];
  int rf = MRFP_ERR_UNSUPPORTED;
  if constexpr (sizeof(T) == 2) {
    if (bulk)
      rf = bn_relu_resample_bulk(Y, A, lut + st.idx_h, lut + st.idx_w, P->lut.data() + st.idx_w, stats + 2 * kMaxC,
                                 stats + 3 * kMaxC, P->N, st.cout, st.ch, st.cw, st.oh, st.ow, rev, s);
  }
  if (rf == MRFP_ERR_UNSUPPORTED) {
    launch_k(bn_relu_resample_kernel<T>, dim3(even_grid(P->N * st.oh, di.sm_count * 8)), dim3(256), 0, s, Y, A, lut + st.idx_h,
             lut + st.idx_w, stats + 2 * kMaxC, stats + 3 * kMaxC, P->N, st.cout, st.ch, st.cw, st.oh, st.ow, rev ? 1 : 0);
    rf = MRFP_OK;
  }
  return rf;
}

template <typename T>
int run_bwd_reduce(const mrfp_hrfp_plan* P, int k, const int* lut, const T* dA, const T* Y, const float* stats, double* acc,
                   bool rev, bool bulk, const DeviceInfo& di, cudaStream_t s) {
  const HrfpStage& st = P->st[k];
  int rr = MRFP_ERR_UNSUPPORTED;
  if constexpr (sizeof(T) == 2) {
    if (bulk)
      rr = bn_bwd_reduce_bulk(dA, Y, lut + st.idx_h, lut + st.idx_w, P->lut.data() + st.idx_w, stats, acc, P->N, st.cout, st.ch,
                              st.cw, st.oh, st.ow, rev, s);
  }
  if (rr == MRFP_ERR_UNSUPPORTED) {
    launch_k(bn_bwd_reduce_kernel<T>, dim3(even_grid(P->N * st.oh, di.sm_count * 8)), dim3(256), 0, s, dA, Y, lut + st.idx_h,
             lut + st.idx_w, stats, acc, P->N, st.cout, st.ch, st.cw, st.oh, st.ow, rev ? 1 : 0);
    rr = MRFP_OK;
  }
  return rr;
}

template <typename T>
int run_bwd_apply(const mrfp_hrfp_plan* P, int k, const int* lut, const T* dA, const T* Y, T* dY, const float* stats,
                  const float* gamma, const double* acc, bool rev, bool product, const DeviceInfo& di, cudaStream_t s) {
  const HrfpStage& st = P->st[k];
  const double count = (double)P->N * st.oh * st.ow;
  if (product && st.oh == st.ch && st.ow == st.cw) {   // identity resample (OCdeclayer1): flat stream
    const long long npix = (long long)P->N * st.ch * st.cw;
    launch_k(bn_bwd_apply_identity_kernel<T>, dim3(di.sm_count * 8), dim3(256), 0, s, dA, Y, dY, stats, gamma, acc, npix, st.cout,
             count, rev ? 1 : 0, st.cout_real);
    return MRFP_OK;
  }
  int ra = MRFP_ERR_UNSUPPORTED;
  if constexpr (sizeof(T) == 2) {
    if (product)
      ra = bn_bwd_apply_bulk(dA, Y, dY, lut + st.lo_h, lut + st.lo_w, P->lut.data() + st.lo_h, P->lut.data() + st.lo_w, stats,
                             gamma, acc, P->N, st.cout, st.ch, st.cw, st.oh, st.ow, count, rev, s, st.cout_real);
  }
  if (ra == MRFP_ERR_UNSUPPORTED) {
    launch_k(bn_bwd_apply_kernel<T>, dim3(even_grid(P->N * st.ch, di.sm_count * 9)), dim3(256), 0, s, dA, Y, dY,
             lut + st.start_h, lut + st.cnt_h, lut + st.start_w, lut + st.cnt_w, stats, gamma, acc, P->N, st.cout, st.ch, st.cw,
             st.oh, st.ow, count, rev ? 1 : 0, st.cout_real);
    ra = MRFP_OK;
  }
  return ra;
}

// fp32 NCHW (C planes) -> T NHWC with CD stored channels
template <typename T>
void run_nchw_to_nhwc(const float* src, T* dst, int N, int C, int CD, int HW, bool accumulate, double* psum, bool allow_stm,
                      cudaStream_t s) {
  dim3 g((CD + 63) / 64, (HW + kLayPx - 1) / kLayPx, N);
  if constexpr (sizeof(T) == 2) {
    if (allow_stm && !accumulate && stm_layout_ok<T>(C, CD, HW, src)) {
      launch_k(nchw_to_nhwc_stm_kernel, dim3(g), dim3(256), 0, s, src, dst, C, HW, psum);
      return;
    }
  }
  launch_k(nchw_to_nhwc_kernel<T>, dim3(g), dim3(256), 0, s, src, dst, C, CD, HW, accumulate ? 1 : 0, psum);
}

template <typename T>
int hrfp_forward(const mrfp_hrfp_plan* P, const float* xp, const float* const* W, const float* const* gamma,
                 const float* const* beta, float* const* rmean, float* const* rvar, float momentum, float eps,
                 const float* x_add, float* ocout, float* ocout_dec, const int* lut, char* saved, char* ws,
                 cudaStream_t s, const DeviceInfo& di, const NpStem* np) {
  double* acc = reinterpret_cast<double*>(ws + P->acc_fwd_off);
  unsigned int* fin_counters = reinterpret_cast<unsigned int*>(acc + (size_t)kHrfpStages * 2 * kMaxC);   // [8], zeroed with acc
  if (np) MRFP_CUDA_TRY(cudaMemsetAsync(np->psum, 0, (size_t)P->N * P->cin * sizeof(double), s));
  MRFP_CUDA_TRY(cudaMemsetAsync(acc, 0, (size_t)kHrfpStages * 2 * kMaxC * sizeof(double) + kHrfpStages * sizeof(unsigned int), s));
  const int last = ocout ? kHrfpStages : 4;
  const bool tc = P->mode != MRFP_MATH_FP32;
  // L2-friendly ordering: a kernel starts walking its tensor where its producer finished.  Forward: every conv walks
  // front to back, every BN/ReLU/resample pass back to front (-0.8 % on the step).
  {
    PackJobs jobs = {};
    for (int k = 0; k < last; ++k) {
      const HrfpStage& st = P->st[k];
      for (int d = 0; d < 2; ++d) {
        const int j = 2 * k + d;
        jobs.W[j] = W[k];
        jobs.out[j] = d == 0 ? (void*)(ws + st.wf_off) : (void*)(saved + st.wb_off);
        jobs.cin[j] = st.cin; jobs.cout[j] = st.cout; jobs.cin_r[j] = st.cin_real; jobs.cout_r[j] = st.cout_real;
        jobs.layout[j] = (unsigned char)(tc ? (d == 0 ? 1 : 0) : (d == 0 ? 0 : 1));
        jobs.flip[j] = (unsigned char)d;
        jobs.bf16[j] = (unsigned char)(P->mode == MRFP_MATH_BF16);
      }
    }
    launch_k(pack_weights_kernel, dim3(64, 2 * last), dim3(256), 0, s, jobs);
  }
  T* bufA = reinterpret_cast<T*>(ws + P->bufs_off);
  T* bufB = reinterpret_cast<T*>(ws + P->bufs_off + P->buf_a_bytes);
  {
    const int HW = P->xh * P->xw;
    run_nchw_to_nhwc<T>(xp, bufA, P->N, P->cin, P->st[0].cin, HW, false, np ? np->psum : (double*)nullptr, true, s);
    if (np)      // NP+ call 1 folded into the chain: plane totals came with the layout pass, (a, b) per plane from one block
      launch_k(np_stem_coef_kernel<false>, dim3(1), dim3(256), 0, s, (const double*)np->psum, np->alpha, np->eps,
               (const float*)nullptr, np->coef, np->mean, np->beta, P->N, P->cin, HW);
  }
  T* cur = bufA;
  T* nxt = bufB;
  for (int k = 0; k < last; ++k) {
    const HrfpStage& st = P->st[k];
    T* Y = reinterpret_cast<T*>(saved + st.y_off);
    double* a = acc + (size_t)k * 2 * kMaxC;
    float* stats = reinterpret_cast<float*>(saved + P->stats_off) + (size_t)k * 4 * kMaxC;
    const double count = (double)P->N * st.oh * st.ow;
    // operand of this conv built on chip from Y_{k-1} (conv_gather.cu) instead of read from a materialised A_k
    const bool gathered = tc && k > 0 && (P->fuse & 1) && sizeof(T) == 2 &&
                          conv3x3_gather_supported(0, P->N, st.ch, st.cw, P->st[k - 1].ch, P->st[k - 1].cw, st.cin, st.cout, st.dil);
    if (k > 0 && !gathered) {     // A_k = ReLU(BN(nearest(Y_{k-1}))) as a tensor in HBM
      const HrfpStage& pv = P->st[k - 1];
      int rf = run_resample<T>(P, k - 1, lut, reinterpret_cast<const T*>(saved + pv.y_off), nxt, stats - 4 * kMaxC, true, true, di, s);
      if (rf) return rf;
      T* t = cur; cur = nxt; nxt = t;
    }
    if (tc) {
      ConvBnFinalize fin = {};
      fin.gamma = gamma[k]; fin.beta = beta ? beta[k] : nullptr;
      fin.running_mean = rmean ? rmean[k] : nullptr; fin.running_var = rvar ? rvar[k] : nullptr;
      fin.stats = stats;
      fin.counter = fin_counters + k;
      fin.count = count; fin.momentum = momentum; fin.eps = eps; fin.cout_real = st.cout_real;
      int rc;
      if (gathered) {
        const HrfpStage& pv = P->st[k - 1];
        rc = conv3x3_gather_fwd(saved + pv.y_off, pv.ch, pv.cw, lut + pv.idx_h, lut + pv.idx_w, stats - 4 * kMaxC, ws + st.wf_off, Y,
                                P->N, st.ch, st.cw, st.cin, st.cout, st.dil, lut + st.cnt_h, lut + st.cnt_w, a, s, false, &fin,
                                &P->maps_g[0][k]);
      } else {
        rc = conv3x3_tc(cur, ws + st.wf_off, Y, P->esize, P->N, st.ch, st.cw, st.cin, st.cout, st.dil, lut + st.cnt_h,
                        lut + st.cnt_w, a, s, false, &fin, nullptr, &P->maps[0][k]);
      }
      if (rc) return rc;
    } else {
      int rc = launch_direct_conv<T>(cur, ws + st.wf_off, Y, P->N, st.ch, st.cw, st.cin, st.cout, st.dil, lut + st.cnt_h,
                                     lut + st.cnt_w, a, di, s);
      if (rc) return rc;
      launch_k(bn_finalize_kernel, dim3(1), dim3(256), 0, s, (const double*)a, gamma[k], beta ? beta[k] : (const float*)nullptr,
               rmean ? rmean[k] : (float*)nullptr, rvar ? rvar[k] : (float*)nullptr, stats, st.cout, st.cout_real, count,
               momentum, eps);
    }
    if (k == 3 && ocout_dec) {
      const unsigned g = (unsigned)(((st.ow + kLayPx - 1) / kLayPx) * ((st.cout + 63) / 64)) * (unsigned)(P->N * st.oh);
      launch_k(nhwc_to_nchw_kernel<T, false>, dim3(g), dim3(256), 0, s, (const T*)Y, ocout_dec, (const float*)nullptr,
               lut + st.idx_h, lut + st.idx_w, (const float*)(stats + 2 * kMaxC), (const float*)(stats + 3 * kMaxC), st.cout,
               st.cout, st.ch, st.cw, st.oh, st.ow, (const float2*)nullptr, (const float*)nullptr, 0, 0);
    }
    if (k == kHrfpStages - 1) {
      const unsigned g = (unsigned)(((st.ow + kLayPx - 1) / kLayPx) * ((st.cout_real + 63) / 64)) * (unsigned)(P->N * st.oh);
      // with the fused NP+ the add operand is xp itself under the plane's affine map: OCout + (a*xp + b)
      launch_k(nhwc_to_nchw_kernel<T, false>, dim3(g), dim3(256), 0, s, (const T*)Y, ocout, np ? xp : x_add, lut + st.idx_h,
               lut + st.idx_w, (const float*)(stats + 2 * kMaxC), (const float*)(stats + 3 * kMaxC), st.cout_real, st.cout,
               st.ch, st.cw, st.oh, st.ow, np ? (const float2*)np->coef : (const float2*)nullptr, (const float*)nullptr, 0, 0);
    }
  }
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

// Fallback of the rank-K form of the classifier tail's gradient (G (pixels, 64) bf16, W2T (C, 64) bf16, classes beyond K
// zero): dA[px][c] = sum_k G[px][k] W2T[c][k], for the launches that cannot take it as a k-block of the stage-4 dgrad
// (encoder-only backward, fusion switched off).  Plain CUDA cores: 8 channels of one pixel per thread.
__global__ void __launch_bounds__(256)
rankk_expand_kernel(const __nv_bfloat16* __restrict__ G, const __nv_bfloat16* __restrict__ W2T, __nv_bfloat16* __restrict__ dA,
                    long long npix, int C) {
  extern __shared__ float s_w[];                         // [C][32] fp32 (<= 24 classes are non-zero)
  pdl_sync();
  for (int e = threadIdx.x; e < C * 32; e += 256) s_w[e] = __bfloat162float(W2T[(size_t)(e >> 5) * 64 + (e & 31)]);
  __syncthreads();
  const int cg = C >> 3;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < npix * cg; i += (long long)gridDim.x * 256) {
    const long long px = i / cg;
    const int c0 = (int)(i - px * cg) * 8;
    float g[32];
    const uint4* gp = reinterpret_cast<const uint4*>(G + px * 64);
#pragma unroll
    for (int q = 0; q < 4; ++q) unpack8(__ldg(gp + q), reinterpret_cast<float (&)[8]>(g[8 * q]));
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float a = 0.f;
#pragma unroll
      for (int k = 0; k < 32; ++k) a = fmaf(g[k], s_w[(c0 + j) * 32 + k], a);
      o[j] = a;
    }
    *reinterpret_cast<uint4*>(dA + px * C + c0) = pack8(o);
  }
}

template <typename T>
int rankk_expand(const void* g64, const void* w2t, T* dA, long long npix, int C, const DeviceInfo& di, cudaStream_t s) {
  if constexpr (sizeof(T) != 2) {
    return MRFP_ERR_UNSUPPORTED;
  } else {
    launch_k(rankk_expand_kernel, dim3((unsigned)(di.sm_count * 8)), dim3(256), (size_t)C * 32 * sizeof(float), s,
             static_cast<const __nv_bfloat16*>(g64), static_cast<const __nv_bfloat16*>(w2t), reinterpret_cast<__nv_bfloat16*>(dA), npix, C);
    MRFP_CUDA_TRY(cudaGetLastError());
    return MRFP_OK;
  }
}

// The gradient of OCout_dec in one of the forms of include/mrfp_b200.h (MRFP_DEC_GRAD_*): g is the fp32 NCHW tensor, the
// NHWC tensor in the chain's element type, or the rank-K factor G with w2t = W2T.
struct DecGrad {
  int form;
  const void* g;
  const void* w2t;
};

// That gradient as the NHWC tensor dst (N, h/2, w/2, C) in the chain's element type.  Only the fp32 form is ever added to
// what dst holds (FP32 mode); the other forms only overwrite it.
template <typename T>
int materialise_dec(const mrfp_hrfp_plan* P, const DecGrad& dec, T* dst, bool accumulate, const DeviceInfo& di, cudaStream_t s) {
  const HrfpStage& st = P->st[3];
  const long long npix = (long long)P->N * st.oh * st.ow;
  switch (dec.form) {
    case MRFP_DEC_GRAD_F32:
      run_nchw_to_nhwc<T>(static_cast<const float*>(dec.g), dst, P->N, st.cout, st.cout, st.oh * st.ow, accumulate,
                          (double*)nullptr, true, s);
      return MRFP_OK;
    case MRFP_DEC_GRAD_NHWC:
      MRFP_CUDA_TRY(cudaMemcpyAsync(dst, dec.g, (size_t)npix * st.cout * sizeof(T), cudaMemcpyDeviceToDevice, s));
      return MRFP_OK;
    default:
      return rankk_expand<T>(dec.g, dec.w2t, dst, npix, st.cout, di, s);
  }
}

template <typename T>
int hrfp_backward(const mrfp_hrfp_plan* P, const float* g_ocout, const DecGrad& dec, const float* const* gamma,
                  const int* lut, const char* saved, float* g_xp, char* ws, cudaStream_t s, const DeviceInfo& di,
                  const NpStem* np) {
  double* acc = reinterpret_cast<double*>(ws + P->acc_bwd_off);
  if (np && !g_ocout) np = nullptr;                      // no gradient through `x`: NP+ contributes nothing
  if (np) MRFP_CUDA_TRY(cudaMemsetAsync(np->psum, 0, (size_t)P->N * P->cin * sizeof(double), s));
  MRFP_CUDA_TRY(cudaMemsetAsync(acc, 0, (size_t)kHrfpStages * 2 * kMaxC * sizeof(double), s));
  T* g0 = reinterpret_cast<T*>(ws + P->bufs_off);
  T* g1 = reinterpret_cast<T*>(ws + P->bufs_off + P->buf_g_bytes);
  T* dY = reinterpret_cast<T*>(ws + P->bufs_off + 2 * P->buf_g_bytes);
  const bool tc = P->mode != MRFP_MATH_FP32;
  T* dA = nullptr;    // gradient wrt the stage output A_{k+1}, NHWC at (oh, ow)
  T* other = g1;
  bool at_end = true;     // where the last kernel that touched dA finished (the layout kernels walk front to back)
  for (int k = kHrfpStages - 1; k >= 0; --k) {
    const HrfpStage& st = P->st[k];
    if (k == kHrfpStages - 1 && g_ocout) {      // with the fused NP+ backward this pass also takes the plane totals of g_ocout
      run_nchw_to_nhwc<T>(g_ocout, g0, P->N, st.cout_real, st.cout, st.oh * st.ow, false, np ? np->psum : (double*)nullptr, true, s);
      if (np)
        launch_k(np_stem_coef_kernel<true>, dim3(1), dim3(256), 0, s, (const double*)np->psum, np->alpha, np->eps,
                 (const float*)np->mean, np->coef, (float*)nullptr, (float*)nullptr, P->N, P->cin, P->xh * P->xw);
      dA = g0;
    }
    // The gradient of OCout_dec joins dA_3.  The tensor-core modes add it in the epilogue of stage 4's dgrad (below) when
    // stages 7-4 ran; here it starts the encoder-only backward, or the FP32 mode adds it to dA_3.
    if (k == 3 && dec.form != MRFP_DEC_GRAD_NONE && !(tc && dA)) {
      int rd = materialise_dec<T>(P, dec, dA ? dA : g0, dA != nullptr, di, s);
      if (rd) return rd;
      if (!dA) { dA = g0; other = g1; }
      at_end = true;
    }
    if (!dA) continue;
    const T* Y = reinterpret_cast<const T*>(saved + st.y_off);
    const float* stats = reinterpret_cast<const float*>(saved + P->stats_off) + (size_t)k * 4 * kMaxC;
    double* a = acc + (size_t)k * 2 * kMaxC;
    int rr = run_bwd_reduce<T>(P, k, lut, dA, Y, stats, a, at_end, true, di, s);
    if (rr) return rr;
    at_end = !at_end;
    // dY_k is built inside the dgrad's operand producers from dA_{k+1}, Y_k and the sums (conv_gather.cu) instead of a pass
    // over HBM: identity / down-sampling stages directly, up-sampling stages (up to 2 x 2 replicas per pixel) through an
    // extras stage.  (The fp32 OCout_dec gradient of the unfused tail is staged in the dA buffer, which the gathered dgrad
    // still reads: that case keeps the pass.)
    const bool gathered = tc && (P->fuse & 2) && sizeof(T) == 2 && st.max_rep <= 2 && !(k == 4 && dec.form == MRFP_DEC_GRAD_F32) &&
                          !(st.max_rep > 1 && k == 4) &&
                          conv3x3_gather_supported(st.max_rep <= 1 ? 1 : 2, P->N, st.ch, st.cw, st.oh, st.ow, st.cout, st.cin, st.dil,
                                                   P->lut.data() + st.lo_h, P->lut.data() + st.lo_w);
    if (!gathered) {
      int ra = run_bwd_apply<T>(P, k, lut, dA, Y, dY, stats, gamma[k], a, at_end, true, di, s);
      if (ra) return ra;
      at_end = !at_end;
    }
    // dgrad: conv of dY (cout channels) with the rotated / transposed kernel -> dA_prev (cin channels)
    if (tc) {
      // stage 4's dgrad produces dA_3, which the gradient of OCout_dec joins in the conv epilogue in fp32 (one rounding, and
      // the read-modify-write pass over dA_3 disappears): the NHWC form as the add tile itself, the rank-K form as one more
      // k-block of the gathered dgrad (G and W2T travel through its weight ring), any other case materialised into the
      // buffer apply(4) has just finished reading
      const void* add_src = nullptr;
      const void* rk = nullptr;
      if (k == 4 && dec.form != MRFP_DEC_GRAD_NONE) {
        if (dec.form == MRFP_DEC_GRAD_NHWC) {
          add_src = dec.g;
        } else if (dec.form == MRFP_DEC_GRAD_RANK_K && gathered) {
          add_src = dec.g;
          rk = dec.w2t;
        } else {
          int rd = materialise_dec<T>(P, dec, dA, false, di, s);
          if (rd) return rd;
          add_src = dA;
          at_end = true;
        }
      }
      int rc;
      if (gathered)
        rc = conv3x3_gather_bwd(Y, dA, st.oh, st.ow, lut + st.lo_h, lut + st.lo_w, P->lut.data() + st.lo_h, P->lut.data() + st.lo_w,
                                st.max_rep, stats, gamma[k], a, (double)P->N * st.oh * st.ow, st.cout_real, saved + st.wb_off, other,
                                P->N, st.ch, st.cw, st.cout, st.cin, st.dil, s, at_end, add_src, &P->maps_g[1][k], rk);
      else
        rc = conv3x3_tc(dY, saved + st.wb_off, other, P->esize, P->N, st.ch, st.cw, st.cout, st.cin, st.dil, nullptr, nullptr,
                        nullptr, s, at_end, nullptr, add_src, &P->maps[1][k]);
      if (rc) return rc;
      at_end = !at_end;
    } else {
      int rc = launch_direct_conv<T>(dY, saved + st.wb_off, other, P->N, st.ch, st.cw, st.cout, st.cin, st.dil, nullptr, nullptr,
                                     nullptr, di, s);
      if (rc) return rc;
    }
    T* t = dA; dA = other; other = t;
  }
  if (!dA) {   // no gradient reached the chain
    MRFP_CUDA_TRY(cudaMemsetAsync(g_xp, 0, (size_t)P->N * P->cin * P->xh * P->xw * sizeof(float), s));
    return MRFP_OK;
  }
  const unsigned g = (unsigned)(((P->xw + kLayPx - 1) / kLayPx) * ((P->cin + 63) / 64)) * (unsigned)(P->N * P->xh);
  // fused NP+ backward: g_xp = dA_0 + (a' * g_ocout + b') with the plane's backward coefficients
  const bool np_add = np && g_ocout;
  launch_k(nhwc_to_nchw_kernel<T, false>, dim3(g), dim3(256), 0, s, (const T*)dA, g_xp, np_add ? g_ocout : (const float*)nullptr,
           (const int*)nullptr, (const int*)nullptr, (const float*)nullptr, (const float*)nullptr, P->cin, P->st[0].cin, P->xh,
           P->xw, P->xh, P->xw, np_add ? (const float2*)np->coef : (const float2*)nullptr, (const float*)nullptr, 0, 0);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

}  // namespace

int np_coef_launch(bool backward, const double* psum, const float* alpha, const float* eps, const float* mean_in, float2* coef,
                   float* mean_out, float* beta_out, int N, int C, int HW, cudaStream_t stream) {
  if (C > kMaxC) return MRFP_ERR_UNSUPPORTED;
  if (backward)
    launch_k(np_stem_coef_kernel<true>, dim3(1), dim3(256), 0, stream, psum, alpha, eps, mean_in, coef, (float*)nullptr,
             (float*)nullptr, N, C, HW);
  else
    launch_k(np_stem_coef_kernel<false>, dim3(1), dim3(256), 0, stream, psum, alpha, eps, (const float*)nullptr, coef, mean_out,
             beta_out, N, C, HW);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}
}  // namespace mrfp

using namespace mrfp;

extern "C" int mrfp_hrfp_plan_create(mrfp_hrfp_plan_t** out, int N, int cin, int xh, int xw, int h, int w,
                                     const int* widths, int math_mode) {
  if (!out) return MRFP_ERR_NULL_POINTER;
  *out = nullptr;
  static const int kDefaultWidths[4] = {64, 64, 128, 256};
  const int* wd = widths ? widths : kDefaultWidths;
  if (N <= 0 || xh <= 0 || xw <= 0 || h < 4 || w < 4 || cin <= 0) return MRFP_ERR_BAD_SHAPE;
  if (math_mode != MRFP_MATH_FP32 && math_mode != MRFP_MATH_TF32 && math_mode != MRFP_MATH_BF16) return MRFP_ERR_UNSUPPORTED;
  if (cin > kMaxC) return MRFP_ERR_UNSUPPORTED;
  for (int i = 0; i < 4; ++i)
    if (!pow2_ge8(wd[i])) return MRFP_ERR_UNSUPPORTED;
  // the chain ends at (ceil(h/4), ceil(w/4)) (deepv3.py:327) and its output is added to xp (deepv3.py:330): the two
  // sizes must agree, as torch.add would demand in the reference
  if ((h + 3) / 4 != xh || (w + 3) / 4 != xw) return MRFP_ERR_BAD_SHAPE;
  mrfp_hrfp_plan* P = new (std::nothrow) mrfp_hrfp_plan();
  if (!P) return MRFP_ERR_WORKSPACE;
  P->magic = kPlanMagic;
  P->N = N; P->cin = cin; P->xh = xh; P->xw = xw; P->h = h; P->w = w; P->mode = math_mode;
  P->esize = math_mode == MRFP_MATH_BF16 ? 2 : 4;
  P->cin_pad = stem_pad(cin, math_mode);
  for (int d = 0; d < 2; ++d) {
    for (int k = 0; k < kHrfpStages; ++k) P->maps[d][k].valid = P->maps_g[d][k].valid = 0;
    P->maps_tail[d].valid = 0;
  }
  P->fuse = math_mode == MRFP_MATH_BF16 ? 3 : 0;    // mrfp_hrfp_plan_set_fusion
  // layer table of deepv3.py:221-237, parametrised by the encoder widths and the (padded) stem width
  const int chans[9] = {P->cin_pad, wd[0], wd[1], wd[2], wd[3], wd[2], wd[1], wd[0], P->cin_pad};
  const int dils[8] = {1, 1, 2, 2, 1, 1, 2, 2};
  // resample spec of deepv3.py:320-327
  const double sfs[8] = {1.205, 1.2, 1.2, 0, 0, 0.838, 0.798, 0};
  const int sz_h[8] = {0, 0, 0, h / 2, h / 2, 0, 0, (h + 3) / 4};
  const int sz_w[8] = {0, 0, 0, w / 2, w / 2, 0, 0, (w + 3) / 4};
  int ch = xh, cw = xw;
  size_t y_bytes = 0, wf_bytes = 0, wb_bytes = 0, max_act = 0, max_g = 0, max_dy = 0;
  max_act = (size_t)N * xh * xw * P->cin_pad * P->esize;
  for (int k = 0; k < kHrfpStages; ++k) {
    HrfpStage& st = P->st[k];
    st.cin = chans[k]; st.cout = chans[k + 1]; st.dil = dils[k];
    st.cin_real = k == 0 ? cin : st.cin;
    st.cout_real = k == kHrfpStages - 1 ? cin : st.cout;
    st.ch = ch; st.cw = cw;
    const bool sf = sfs[k] > 0;
    st.oh = sf ? (int)floor((double)ch * sfs[k]) : sz_h[k];
    st.ow = sf ? (int)floor((double)cw * sfs[k]) : sz_w[k];
    if (st.oh <= 0 || st.ow <= 0) { delete P; return MRFP_ERR_BAD_SHAPE; }
    if (math_mode != MRFP_MATH_FP32 && (!conv3x3_tc_supported(st.cin, st.cout, P->esize) ||
                                        !conv3x3_tc_supported(st.cout, st.cin, P->esize))) { delete P; return MRFP_ERR_UNSUPPORTED; }
    std::vector<int>& L = P->lut;
    st.scale_h = index_scale(ch, st.oh, sf, sfs[k]); st.scale_w = index_scale(cw, st.ow, sf, sfs[k]);
    st.idx_h = (int)L.size(); L.resize(L.size() + st.oh); make_index(ch, st.oh, sf, sfs[k], &L[st.idx_h]);
    st.idx_w = (int)L.size(); L.resize(L.size() + st.ow); make_index(cw, st.ow, sf, sfs[k], &L[st.idx_w]);
    const int ph = (ch + 2 * kTileH - 1) / (2 * kTileH) * (2 * kTileH) + 2 * kTileH;   // conv tiles are up to 16 rows tall
    const int pw = (cw + kTileW - 1) / kTileW * kTileW + kTileW;
    st.cnt_h = (int)L.size(); L.resize(L.size() + ph, 0);
    st.cnt_w = (int)L.size(); L.resize(L.size() + pw, 0);
    st.start_h = (int)L.size(); L.resize(L.size() + ch, 0);
    st.start_w = (int)L.size(); L.resize(L.size() + cw, 0);
    for (int d = st.oh - 1; d >= 0; --d) { const int sidx = L[st.idx_h + d]; L[st.cnt_h + sidx]++; L[st.start_h + sidx] = d; }
    for (int d = st.ow - 1; d >= 0; --d) { const int sidx = L[st.idx_w + d]; L[st.cnt_w + sidx]++; L[st.start_w + sidx] = d; }
    st.lo_h = (int)L.size(); L.resize(L.size() + ch + 1, 0);
    st.lo_w = (int)L.size(); L.resize(L.size() + cw + 1, 0);
    for (int sidx = 0, d = 0; sidx <= ch; ++sidx) { while (d < st.oh && L[st.idx_h + d] < sidx) ++d; L[st.lo_h + sidx] = d; }
    for (int sidx = 0, d = 0; sidx <= cw; ++sidx) { while (d < st.ow && L[st.idx_w + d] < sidx) ++d; L[st.lo_w + sidx] = d; }
    st.max_rep = 0;
    for (int i = 0; i < ch; ++i) st.max_rep = L[st.cnt_h + i] > st.max_rep ? L[st.cnt_h + i] : st.max_rep;
    for (int i = 0; i < cw; ++i) st.max_rep = L[st.cnt_w + i] > st.max_rep ? L[st.cnt_w + i] : st.max_rep;
    st.y_off = y_bytes;
    y_bytes += align_up((size_t)N * ch * cw * st.cout * P->esize, 256);
    st.wf_off = wf_bytes; wf_bytes += align_up((size_t)9 * st.cin * st.cout * P->esize, 256);
    st.wb_off = wb_bytes; wb_bytes += align_up((size_t)9 * st.cin * st.cout * P->esize, 256);
    const size_t a_next = (size_t)N * st.oh * st.ow * st.cout * P->esize;   // A_{k+1} and dA_{k+1}
    const size_t dy = (size_t)N * ch * cw * st.cout * P->esize;             // dY_k
    const size_t da_prev = (size_t)N * ch * cw * st.cin * P->esize;         // dA_k
    if (a_next > max_act) max_act = a_next;
    if (a_next > max_g) max_g = a_next;
    if (da_prev > max_g) max_g = da_prev;
    if (dy > max_dy) max_dy = dy;
    ch = st.oh; cw = st.ow;
  }
  // saved: [Y_0..Y_7][stats][dgrad weights]
  P->stats_off = y_bytes;
  const size_t stats_bytes = align_up((size_t)kHrfpStages * 4 * kMaxC * sizeof(float), 256);
  for (int k = 0; k < kHrfpStages; ++k) P->st[k].wb_off += y_bytes + stats_bytes;
  P->saved_bytes = y_bytes + stats_bytes + wb_bytes;
  // ws: [acc fwd][acc bwd][fwd weights][buffers: fwd A/B ping-pong | bwd g0, g1, dY]
  const size_t acc_bytes = (size_t)kHrfpStages * 2 * kMaxC * sizeof(double) + 256;   // + finalisation counters
  P->acc_fwd_off = 0;
  P->acc_bwd_off = acc_bytes;
  for (int k = 0; k < kHrfpStages; ++k) P->st[k].wf_off += 2 * acc_bytes;
  P->bufs_off = align_up(2 * acc_bytes + wf_bytes, 1024);
  P->buf_a_bytes = align_up(max_act, 1024);
  P->buf_g_bytes = align_up(max_g, 1024);
  P->buf_dy_bytes = align_up(max_dy, 1024);
  const size_t fwd = 2 * P->buf_a_bytes, bwd = 2 * P->buf_g_bytes + P->buf_dy_bytes;
  P->ws_bytes = P->bufs_off + (fwd > bwd ? fwd : bwd);
  *out = P;
  return MRFP_OK;
}

extern "C" void mrfp_hrfp_plan_destroy(mrfp_hrfp_plan_t* P) {
  if (P && P->magic == kPlanMagic) { P->magic = 0; delete P; }
}
extern "C" size_t mrfp_hrfp_plan_ws_bytes(const mrfp_hrfp_plan_t* P) { return (P && P->magic == kPlanMagic) ? P->ws_bytes : 0; }
extern "C" size_t mrfp_hrfp_plan_saved_bytes(const mrfp_hrfp_plan_t* P) { return (P && P->magic == kPlanMagic) ? P->saved_bytes : 0; }
extern "C" size_t mrfp_hrfp_plan_lut_bytes(const mrfp_hrfp_plan_t* P) {
  return (P && P->magic == kPlanMagic) ? P->lut.size() * sizeof(int) : 0;
}
extern "C" int mrfp_hrfp_plan_write_luts(const mrfp_hrfp_plan_t* P, void* host_dst, size_t bytes) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  if (!host_dst) return MRFP_ERR_NULL_POINTER;
  if (bytes < P->lut.size() * sizeof(int)) return MRFP_ERR_WORKSPACE;
  memcpy(host_dst, P->lut.data(), P->lut.size() * sizeof(int));
  return MRFP_OK;
}
extern "C" int mrfp_hrfp_plan_set_fusion(mrfp_hrfp_plan_t* P, int bits) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  std::lock_guard<std::mutex> g(P->mu);
  P->fuse = P->mode == MRFP_MATH_BF16 ? (bits & 3) : 0;
  return P->fuse;
}
extern "C" int mrfp_hrfp_plan_stage(const mrfp_hrfp_plan_t* P, int k, int* out7) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  if (!out7) return MRFP_ERR_NULL_POINTER;
  if (k < 0 || k >= kHrfpStages) return MRFP_ERR_BAD_SHAPE;
  const HrfpStage& st = P->st[k];
  out7[0] = st.cin_real; out7[1] = st.cout_real; out7[2] = st.dil; out7[3] = st.ch; out7[4] = st.cw; out7[5] = st.oh; out7[6] = st.ow;
  return MRFP_OK;
}

extern "C" size_t mrfp_hrfp_np_ws_bytes(int N, int C) {
  if (N <= 0 || C <= 0) return 0;
  return (size_t)N * C * (sizeof(double) + sizeof(float2));
}

// NP+ call 1 folded into the chain when alpha, eps, mean and np_ws are all given, not folded (*np = nullptr) when none is
static int np_stem_setup(const mrfp_hrfp_plan_t* P, const float* alpha, const float* eps, const float* mean, float* beta,
                         void* np_ws, NpStem* stem, const NpStem** np) {
  *np = nullptr;
  if (!alpha && !eps && !mean && !np_ws) return MRFP_OK;
  if (!alpha || !eps || !mean || !np_ws || ((uintptr_t)np_ws & 15)) return MRFP_ERR_NULL_POINTER;
  stem->alpha = alpha; stem->eps = eps; stem->mean = const_cast<float*>(mean); stem->beta = beta;
  stem->psum = reinterpret_cast<double*>(np_ws);
  stem->coef = reinterpret_cast<float2*>(stem->psum + (size_t)P->N * P->cin);
  *np = stem;
  return MRFP_OK;
}

extern "C" int mrfp_hrfp_fwd(const mrfp_hrfp_plan_t* P, const float* xp, const float* const* W, const float* const* gamma,
                             const float* const* beta, float* const* running_mean, float* const* running_var, float momentum,
                             float eps, const float* x_add, const float* np_alpha, const float* np_eps, float* np_mean,
                             float* np_beta, void* np_ws, float* ocout, float* ocout_dec, const void* lut, void* saved,
                             void* ws, void* stream) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  if (!xp || !W || !gamma || !lut || !saved || !ws) return MRFP_ERR_NULL_POINTER;
  NpStem stem;
  const NpStem* np;
  int rc = np_stem_setup(P, np_alpha, np_eps, np_mean, np_beta, np_ws, &stem, &np);
  if (rc) return rc;
  if (np && !ocout) return MRFP_ERR_NULL_POINTER;        // the fused form only exists for x = OCout + NP+(xp) ...
  if (np && x_add) return MRFP_ERR_UNSUPPORTED;          // ... where NP+(xp) takes the place of x_add
  if (((uintptr_t)saved | (uintptr_t)ws | (uintptr_t)lut) & 255) return MRFP_ERR_WORKSPACE;
  const int last = ocout ? kHrfpStages : 4;
  for (int k = 0; k < last; ++k)
    if (!W[k] || !gamma[k]) return MRFP_ERR_NULL_POINTER;
  DeviceInfo di;
  rc = get_device_info(&di);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  std::lock_guard<std::mutex> lock(P->mu);               // the plan's tensor-map cache
  if (P->mode == MRFP_MATH_BF16)
    return hrfp_forward<__nv_bfloat16>(P, xp, W, gamma, beta, running_mean, running_var, momentum, eps, x_add, ocout,
                                       ocout_dec, (const int*)lut, (char*)saved, (char*)ws, s, di, np);
  return hrfp_forward<float>(P, xp, W, gamma, beta, running_mean, running_var, momentum, eps, x_add, ocout, ocout_dec,
                             (const int*)lut, (char*)saved, (char*)ws, s, di, np);
}

extern "C" int mrfp_hrfp_bwd(const mrfp_hrfp_plan_t* P, const float* g_ocout, int dec_form, const void* g_dec,
                             const void* w2t64, const float* const* gamma, const float* np_alpha, const float* np_eps,
                             const float* np_mean, void* np_ws, const void* lut, const void* saved, float* g_xp, void* ws,
                             void* stream) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  if (!gamma || !lut || !saved || !g_xp || !ws) return MRFP_ERR_NULL_POINTER;
  NpStem stem;
  const NpStem* np;
  int rc = np_stem_setup(P, np_alpha, np_eps, np_mean, nullptr, np_ws, &stem, &np);
  if (rc) return rc;
  switch (dec_form) {
    case MRFP_DEC_GRAD_NONE:
      break;
    case MRFP_DEC_GRAD_F32:
      if (!g_dec) return MRFP_ERR_NULL_POINTER;
      break;
    case MRFP_DEC_GRAD_NHWC:
      if (!g_dec) return MRFP_ERR_NULL_POINTER;
      if (P->mode == MRFP_MATH_FP32 || ((uintptr_t)g_dec & 15)) return MRFP_ERR_UNSUPPORTED;
      break;
    case MRFP_DEC_GRAD_RANK_K:      // w2t64 is (256, 64): the classifier tail, its producer, exists for 256 channels only
      if (!g_dec || !w2t64) return MRFP_ERR_NULL_POINTER;
      if (P->mode != MRFP_MATH_BF16 || P->st[3].cout != 256 || (((uintptr_t)g_dec | (uintptr_t)w2t64) & 15))
        return MRFP_ERR_UNSUPPORTED;
      break;
    default:
      return MRFP_ERR_UNSUPPORTED;
  }
  if (((uintptr_t)saved | (uintptr_t)ws | (uintptr_t)lut) & 255) return MRFP_ERR_WORKSPACE;
  DeviceInfo di;
  rc = get_device_info(&di);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  std::lock_guard<std::mutex> lock(P->mu);
  const DecGrad dec = {dec_form, g_dec, w2t64};
  if (P->mode == MRFP_MATH_BF16)
    return hrfp_backward<__nv_bfloat16>(P, g_ocout, dec, gamma, (const int*)lut, (const char*)saved, g_xp, (char*)ws, s, di,
                                        np);
  return hrfp_backward<float>(P, g_ocout, dec, gamma, (const int*)lut, (const char*)saved, g_xp, (char*)ws, s, di, np);
}

template <typename T>
static int hrfp_plus_add_impl(const mrfp_hrfp_plan* P, const char* saved, const int* lut, const float* dec1_up,
                              const float* dec1_lo, int lh, int lw, float* out, cudaStream_t s) {
  const HrfpStage& st = P->st[3];
  const T* Y = reinterpret_cast<const T*>(saved + st.y_off);
  const float* stats = reinterpret_cast<const float*>(saved + P->stats_off) + (size_t)3 * 4 * kMaxC;
  const unsigned g = (unsigned)(((st.ow + kLayPx - 1) / kLayPx) * ((st.cout + 63) / 64)) * (unsigned)(P->N * st.oh);
  if (dec1_lo && (lw > st.ow || lh > st.oh)) return MRFP_ERR_BAD_SHAPE;      // an Upsample: the source is not larger
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  // the reference's x2 Upsample: scale <= 1/2 bounds the staged span; 16-byte alignment for the bulk copies
  if (dec1_lo && st.ow > 1 && 2 * (lw - 1) <= st.ow - 1 && (lw & 3) == 0 && ((uintptr_t)dec1_lo & 15) == 0) {
    // bf16 path: the ldmatrix kernel when every tile's source span fits its buffer (host copy of the index table)
    if constexpr (sizeof(T) == 2) {
      if ((st.cout & 63) == 0 && (st.ow & 3) == 0) {
        const int* hidx = P->lut.data() + st.idx_w;
        bool fits = true;
        for (int w0 = 0; w0 < st.ow && fits; w0 += kLayPx) {
          const int w1 = (w0 + kLayPx < st.ow ? w0 + kLayPx : st.ow) - 1;
          fits = hidx[w1] - hidx[w0] + 1 <= kLdmSpan;
        }
        if (fits) {
          const unsigned gl = (unsigned)(((st.ow + kLayPx - 1) / kLayPx) * (st.cout / 64)) * (unsigned)(P->N * st.oh);
          MRFP_SMEM_OPT_IN(hrfp_plus_tail_ldm_kernel, kLdmSmem, di.device);
          launch_k(hrfp_plus_tail_ldm_kernel, dim3(gl), dim3(256), kLdmSmem, s, Y, out, lut + st.idx_h, lut + st.idx_w,
                   stats + 2 * kMaxC, stats + 3 * kMaxC, st.cout, st.ch, st.cw, st.oh, st.ow, dec1_lo, lh, lw);
          MRFP_CUDA_TRY(cudaGetLastError());
          return MRFP_OK;
        }
      }
    }
    // 32-channel tiles: 35 KB, 5-6 tiles per SM (720 vs 742 us for 64-channel tiles)
    const unsigned gs = (unsigned)(((st.ow + kLayPx - 1) / kLayPx) * ((st.cout + 31) / 32)) * (unsigned)(P->N * st.oh);
    MRFP_SMEM_OPT_IN((hrfp_plus_bilinear_staged_kernel<T, 32>), staged_smem<32>(), di.device);
    launch_k(hrfp_plus_bilinear_staged_kernel<T, 32>, dim3(gs), dim3(256), staged_smem<32>(), s, Y, out, lut + st.idx_h,
             lut + st.idx_w, stats + 2 * kMaxC, stats + 3 * kMaxC, st.cout, st.ch, st.cw, st.oh, st.ow, dec1_lo, lh, lw);
    MRFP_CUDA_TRY(cudaGetLastError());
    return MRFP_OK;
  }
  if (dec1_lo)
    launch_k(nhwc_to_nchw_kernel<T, true>, dim3(g), dim3(256), 0, s, Y, out, dec1_up, lut + st.idx_h, lut + st.idx_w,
             stats + 2 * kMaxC, stats + 3 * kMaxC, st.cout, st.cout, st.ch, st.cw, st.oh, st.ow, (const float2*)nullptr, dec1_lo,
             lh, lw);
  else
    launch_k(nhwc_to_nchw_kernel<T, false>, dim3(g), dim3(256), 0, s, Y, out, dec1_up, lut + st.idx_h, lut + st.idx_w,
             stats + 2 * kMaxC, stats + 3 * kMaxC, st.cout, st.cout, st.ch, st.cw, st.oh, st.ow, (const float2*)nullptr, dec1_lo,
             lh, lw);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

extern "C" int mrfp_hrfp_plus_add(const mrfp_hrfp_plan_t* P, const void* saved, const void* lut, const float* dec1_up,
                                  float* out, void* stream) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  if (!saved || !lut || !dec1_up || !out) return MRFP_ERR_NULL_POINTER;
  cudaStream_t s = (cudaStream_t)stream;
  if (P->mode == MRFP_MATH_BF16)
    return hrfp_plus_add_impl<__nv_bfloat16>(P, (const char*)saved, (const int*)lut, dec1_up, nullptr, 0, 0, out, s);
  return hrfp_plus_add_impl<float>(P, (const char*)saved, (const int*)lut, dec1_up, nullptr, 0, 0, out, s);
}

extern "C" int mrfp_hrfp_plus_add_bilinear(const mrfp_hrfp_plan_t* P, const void* saved, const void* lut,
                                           const float* dec1, int lh, int lw, float* out, void* stream) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  if (!saved || !lut || !dec1 || !out) return MRFP_ERR_NULL_POINTER;
  if (lh <= 0 || lw <= 0) return MRFP_ERR_BAD_SHAPE;
  cudaStream_t s = (cudaStream_t)stream;
  if (P->mode == MRFP_MATH_BF16)
    return hrfp_plus_add_impl<__nv_bfloat16>(P, (const char*)saved, (const int*)lut, nullptr, dec1, lh, lw, out, s);
  return hrfp_plus_add_impl<float>(P, (const char*)saved, (const int*)lut, nullptr, dec1, lh, lw, out, s);
}

extern "C" int mrfp_add_f32(const float* a, const float* b, float* out, size_t n, void* stream) {
  if (!a || !b || !out) return MRFP_ERR_NULL_POINTER;
  if (n == 0) return MRFP_OK;
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const bool al = ((((uintptr_t)a | (uintptr_t)b | (uintptr_t)out) & 15) == 0);
  const size_t n4 = al ? n / 4 : 0;
  const int grid = grid_for((long long)(n4 ? n4 : n), 256, di.sm_count, 16);
  launch_k(add_f32_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, (const float4*)a, (const float4*)b, (float4*)out, n4, a, b, out, n);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

// ------------------------------------------------------------------------------------------------------
// test hooks (not part of the public header): ONE element-wise pass of one stage on caller-provided NHWC buffers in the
// plan's element type, so that each product kernel can be pinned on its own against an fp64 evaluation of the same inputs.
//   op 0  forward BN/ReLU/resample   y (N,ch,cw,C) -> out (N,oh,ow,C)          stats = [4][256] mean, invstd, scale, shift
//   op 1  BN-backward reduce         in2 = dA (N,oh,ow,C), y -> acc[0..C) = sum mask*dA, acc[256..) = sum mask*dA*y
//   op 2  BN-backward apply          in2 = dA, y, acc, gamma -> out = dY (N,ch,cw,C)
//   variant 0: the LDG row kernel;  1: the kernel the chain launches (bulk-copy / identity-stream forms on the bf16 path)
// ------------------------------------------------------------------------------------------------------
template <typename T>
static int debug_stage_op(const mrfp_hrfp_plan* P, const int* lut, int k, int op, int variant, const void* y, const void* in2,
                          void* out, const float* stats, const float* gamma, double* acc, cudaStream_t s) {
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const bool product = variant != 0;
  switch (op) {
    case 0: return run_resample<T>(P, k, lut, (const T*)y, (T*)out, stats, false, product, di, s);
    case 1: return run_bwd_reduce<T>(P, k, lut, (const T*)in2, (const T*)y, stats, acc, false, product, di, s);
    case 2: return run_bwd_apply<T>(P, k, lut, (const T*)in2, (const T*)y, (T*)out, stats, gamma, acc, false, product, di, s);
  }
  return MRFP_ERR_BAD_SHAPE;
}

extern "C" int mrfp_debug_stage_op(const mrfp_hrfp_plan_t* P, const void* lut, int k, int op, int variant, const void* y,
                                   const void* in2, void* out, const float* stats, const float* gamma, double* acc,
                                   void* stream) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  if (k < 0 || k >= kHrfpStages) return MRFP_ERR_BAD_SHAPE;
  if (!lut || !y || !stats) return MRFP_ERR_NULL_POINTER;
  if (P->mode == MRFP_MATH_BF16)
    return debug_stage_op<__nv_bfloat16>(P, (const int*)lut, k, op, variant, y, in2, out, stats, gamma, acc, (cudaStream_t)stream);
  return debug_stage_op<float>(P, (const int*)lut, k, op, variant, y, in2, out, stats, gamma, acc, (cudaStream_t)stream);
}

// fp32 NCHW (C planes) -> NHWC with CD stored channels in bf16 (esize 2) or fp32 (esize 4); variant 1 allows the stmatrix
// kernel (bf16, C == CD, C % 64 == 0, HW % 4 == 0); psum (N*C doubles, zeroed by the caller) receives the plane totals
extern "C" int mrfp_debug_nchw_to_nhwc(const float* src, void* dst, int N, int C, int CD, int HW, int esize, int variant,
                                       double* psum, void* stream) {
  if (!src || !dst) return MRFP_ERR_NULL_POINTER;
  if (N <= 0 || C <= 0 || CD < C || (CD & 7) || HW <= 0) return MRFP_ERR_BAD_SHAPE;
  if (esize == 2) run_nchw_to_nhwc<__nv_bfloat16>(src, (__nv_bfloat16*)dst, N, C, CD, HW, false, psum, variant != 0, (cudaStream_t)stream);
  else if (esize == 4) run_nchw_to_nhwc<float>(src, (float*)dst, N, C, CD, HW, false, psum, false, (cudaStream_t)stream);
  else return MRFP_ERR_UNSUPPORTED;
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}
