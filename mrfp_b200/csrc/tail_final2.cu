// HRFP+ tail fused through the classifier (SURVEY.md 8f-4) — replaces, on the bf16 path, the op sequence of
// /root/reference/deepv3.py:356-361:  dec1 = Upsample(dec1, (h/2, w/2));  dec1 = OCout_dec + dec1;  dec2 = final2(dec1)
// with final2 = Conv2d(256, num_classes, 1, bias=True) (deepv3.py:219-220), and its autograd backward.
//
// A 1x1 convolution commutes with the (linear) bilinear interpolation, so
//     dec2 = b2 + Upsample(W2 . dec1) + W2 . OCout_dec
// The first product is a (N, K, h/4, w/4) tensor the host computes with a plain GEMM at LOW resolution; this file
// evaluates the rest per 64-pixel tile of an output row, in persistent CTAs (two per SM) whose inputs arrive by TMA one
// tile ahead (double-buffered, issued by one thread, completion on an mbarrier):
//   * the span of the stored conv output Y_3 the tile gathers from — ONE 3-D box of a tensor map that views Y_3 as
//     [4 groups of 64 channels][pixel][64 channels], landing as four SWIZZLE_128B tiles [64 px][128 bytes];
//   * forward: the two low-resolution rows of every class ([K][2][44] fp32 box; columns beyond the row end and the row
//     below the last one arrive as zeros); backward: the tile's g ([K][64] fp32 box, zeros beyond the row end).
// `ldmatrix` hands the span to the warps as m16n8k16 fragments whose per-lane row addresses perform the nearest-neighbour
// gather (relative source indices of every tile staged once per CTA), BatchNorm + ReLU are applied to the fragments in
// registers (one packed fp32x2 FMA, one rounding to bf16x2, max on the pair), and `mma.sync` contracts against W2 (bf16,
// K <= 24 classes).  Everything that does not change from tile to tile lives in REGISTERS of the persistent CTA: the
// classifier fragments and the BN constants of the warp's channels (forward: warp = one quarter of the channels x 32
// pixels, the four quarter sums meet in the epilogue; backward: warp = 32 channels x all pixels in both products).
// Neither OCout_dec nor the up-sampled dec1 nor their sum (1.2 GB fp32 at batch 8) ever exists; the forward writes 90 MB.
//   Tensor-core choice: the A operand needs a register-side transform (BN/ReLU of gathered rows) and the contraction is
//   11.5 GFLOP per launch against ~0.6 GB of HBM traffic — 5 % of the tensor peak keeps up with the memory system, so
//   warp-level mma.sync on register fragments (no shared-memory round trip for the transformed operand) is the better
//   fit than a tcgen05 pipeline here.
// Backward (one pass over g = dL/d dec2, (N, K, h/2, w/2) fp32):
//     dA3[p][c]   = sum_k g[k][p] W2[k][c]        -> bf16 NHWC, joins the chain as the gradient of OCout_dec (rank K);
//                                                   A fragments by ldmatrix.trans from the bf16 [class][pixel] copy of g,
//                                                   results transposed inside each lane quad and stored from registers
//     gW2[k][c]  += sum_p g[k][p] OCout_dec[c][p]  (OCout_dec regenerated from Y_3 in registers; accumulators stay in
//                                                   registers across the tiles of a persistent CTA)
//     gb2[k]     += sum_p g[k][p]
// The low-resolution half (gradient of W2 . dec1 through the Upsample) is the gather kernel of bilinear.cu plus the
// host's GEMM autograd.
// What was measured on the way (tools/trace_tail.py, profiles/README.md "R2c"): the first form (128-pixel tiles, per-thread
// cp.async of the span, one bulk copy per low-resolution row, W2 fragments and the BN table re-read from shared memory
// per k-block) ran 215 / 363 us at batch 8; per-thread cp.async and per-row bulk copies cost the issuing warps 2400-4300
// cycles per 64-pixel tile, a lane-indexed register pick compiles to divergent branches, a proxy fence per issue and
// global index look-ups sit on the critical path of every barrier.  This form: 133 / 210 us.
#include "hrfp.cuh"
#include "ptx.cuh"
#include <mutex>

namespace mrfp {
namespace {

using namespace ptx;

constexpr int kC = 256;              // channels of OCout_dec (widths[3])
constexpr int kCls = 24;             // classes, padded to three n-blocks of 8 (forward) / 32 (backward k-blocks)
constexpr int kThreads = 256;

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t addr, uint32_t (&r)[2]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
// D += A (16x16, row) * B (16x8, col), bf16 operands, fp32 accumulators
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// launch-constant arguments of both kernels
struct TailArgs {
  const __nv_bfloat16* y;          // Y_3 (N, IH, IW, 256) bf16 NHWC
  const int* idx_h; const int* idx_w;
  const float* scale; const float* shift;
  int N, IH, IW, OH, OW, K;
  const float* w2;                 // (K, 256) fp32
};

// Phase timeline for tools/trace_tail.py (build with MRFP_EXTRA_NVCC_FLAGS=-DMRFP_TAIL_TRACE): clock64 sums of thread 0 of
// every CTA per phase of the tile loop; compiled out otherwise.
#ifdef MRFP_TAIL_TRACE
__device__ unsigned long long g_tail_dbg[16];
#define TR_DECL unsigned long long tr_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long tr_t = clock64();
#define TR(k) do { if (threadIdx.x == 0) { const long long _n = clock64(); tr_acc[k] += (unsigned long long)(_n - tr_t); tr_t = _n; } } while (0)
#define TR_END(off) do { if (threadIdx.x == 0) { for (int _k = 0; _k < 8; ++_k) atomicAdd(&g_tail_dbg[(off) + _k], tr_acc[_k]); } } while (0)
#else
#define TR_DECL
#define TR(k) do { } while (0)
#define TR_END(off) do { } while (0)
#endif

constexpr int kPx = 64;             // output pixels per tile
constexpr int kSpan = 64;           // source pixels a tile's box holds (64 * 332/384 + 2 = 58 needed in the reference geometry)
constexpr int kSeg = 44;            // staged low-resolution row pitch (floats): an Upsample by >= 2 needs <= 40
constexpr int kOutPitch = 68;       // floats; 68 mod 32 = 4: the accumulator scatter is bank-conflict free
constexpr uint32_t kSpanBytes = kSpan * 512;

__device__ __forceinline__ void tma_3d(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// a span buffer is four boxes [64 px][64 ch] (128-byte rows, 16-byte chunks XOR-swizzled by pixel & 7): address of the
// 16-byte chunk `chunk` (8 channels, 0..31) of source pixel `p`
__device__ __forceinline__ uint32_t span_addr(uint32_t base, int p, int chunk) {
  return base + (uint32_t)(chunk >> 3) * (uint32_t)(kSpan * 128) + (uint32_t)p * 128u + (uint32_t)(((chunk & 7) ^ (p & 7)) << 4);
}

struct TileXY { int n, oh, w0, w_last; };
// tile -> (image, output row, segment) for the tiles blockIdx.x, + gridDim.x, ...: divisions once, then carries
struct TileWalk {
  int wt, oh, n, dwt, drow, wtiles, OH, OW;
  __device__ __forceinline__ TileWalk(const TailArgs& a, int tile, int step, int wtiles_) {
    wtiles = wtiles_; OH = a.OH; OW = a.OW;
    const int orow = tile / wtiles;
    wt = tile - orow * wtiles; n = orow / OH; oh = orow - n * OH;
    drow = step / wtiles; dwt = step - drow * wtiles;
  }
  __device__ __forceinline__ void advance() {
    wt += dwt;
    const int carry = wt >= wtiles ? 1 : 0;
    wt -= carry * wtiles;
    oh += drow + carry;
    while (oh >= OH) { oh -= OH; ++n; }
  }
  __device__ __forceinline__ TileXY xy() const {
    TileXY c;
    c.n = n; c.oh = oh; c.w0 = wt * kPx; c.w_last = min(c.w0 + kPx - 1, OW - 1);
    return c;
  }
};

// dynamic shared memory, rounded up to the 1024 bytes the swizzled boxes need (by pointer arithmetic, so that the
// compiler keeps the shared address space)
__device__ __forceinline__ unsigned char* smem_1k(unsigned char* raw) {
  const uint32_t a = smem_u32(raw);
  return raw + (((a + 1023u) & ~1023u) - a);
}

constexpr size_t kFwdSmem = 1024 + (size_t)2 * kSpanBytes + (size_t)4 * kCls * kOutPitch * 4 + (size_t)2 * 2 * kCls * kSeg * 4 +
                             16;       // + the index tables: (wtiles * 65 + OH) ints

// forward: warp = (channel quarter q, pixel-group pair u): 2 x 16 pixels x 64 channels x 24 classes; the four quarter
// sums of a pixel meet in the epilogue
__global__ void __launch_bounds__(kThreads, 2)
tail_final2_fwd_kernel(const __grid_constant__ CUtensorMap tm_y, const __grid_constant__ CUtensorMap tm_lo, const TailArgs a,
                        int LH, int LW, const float* __restrict__ b2, float* __restrict__ out, int wtiles, int num_tiles) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* ysm = smem_1k(smem_raw);                                               // [2][4 boxes][64 px][64 ch bf16]
  float* outst = reinterpret_cast<float*>(ysm + (size_t)2 * kSpanBytes);               // [quarter][class][kOutPitch]
  float* trow = outst + 4 * kCls * kOutPitch;                                          // [buffer][class][row 0/1][kSeg]
  uint64_t* bar = reinterpret_cast<uint64_t*>(trow + 2 * 2 * kCls * kSeg);             // [2] full barriers
  int* rel = reinterpret_cast<int*>(bar + 2);                                           // [wtiles * 64]: source pixel - the tile's first
  int* wstart = rel + wtiles * kPx;                                                    // [wtiles]: first source pixel of a tile
  int* hsrc = wstart + wtiles;                                                          // [OH]: source row of an output row
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int K = a.K;
  const int g = lane >> 2, tq = lane & 3;
  const int amat = lane >> 3, arow = (amat & 1) * 8 + (lane & 7), akc = amat >> 1;
  const int q = warp & 3, u = warp >> 2;
  if (t == 0) {
    mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); mbar_fence_init();
    prefetch_tensormap(&tm_y);
    prefetch_tensormap(&tm_lo);
  }
  pdl_sync();
  // classifier weights -> bf16 [class][channel] (swizzled rows) in the span buffer, from there into B fragments
  for (int e = t; e < kCls * kC; e += kThreads) {
    const int k = e >> 8, c = e & 255;
    const float v = k < K ? a.w2[k * kC + c] : 0.f;
    *reinterpret_cast<__nv_bfloat16*>(ysm + k * 512 + (((c >> 3) ^ (k & 7)) << 4) + (c & 7) * 2) = __float2bfloat16_rn(v);
  }
  for (int e = t; e < wtiles * kPx; e += kThreads) rel[e] = a.idx_w[min(e, a.OW - 1)] - a.idx_w[e & ~(kPx - 1)];
  for (int e = t; e < wtiles; e += kThreads) wstart[e] = a.idx_w[e * kPx];
  for (int e = t; e < a.OH; e += kThreads) hsrc[e] = a.idx_h[e];
  __syncthreads();
  uint32_t bq[4][6];
  uint64_t sq[4][4];                                    // per k-block: (scale, scale), (shift, shift) of channels 2tq, +1 | 8 + 2tq, +1
  {
    const int bn01 = (amat >> 1) * 8 + (lane & 7), bkc = amat & 1;
    const int bn2 = 16 + (lane & 7), bkc2 = (lane >> 3) & 1;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const int kb = 4 * q + kk;
      uint32_t r4[4], r2[2];
      ldsm_x4(smem_u32(ysm) + (uint32_t)bn01 * 512u + (uint32_t)(((kb * 2 + bkc) ^ (bn01 & 7)) << 4), r4);
      ldsm_x2(smem_u32(ysm) + (uint32_t)bn2 * 512u + (uint32_t)(((kb * 2 + bkc2) ^ (bn2 & 7)) << 4), r2);
      bq[kk][0] = r4[0]; bq[kk][1] = r4[1]; bq[kk][2] = r4[2]; bq[kk][3] = r4[3]; bq[kk][4] = r2[0]; bq[kk][5] = r2[1];
      const int c0 = kb * 16 + 2 * tq;
      sq[kk][0] = pack_f32x2(a.scale[c0], a.scale[c0 + 1]); sq[kk][1] = pack_f32x2(a.shift[c0], a.shift[c0 + 1]);
      sq[kk][2] = pack_f32x2(a.scale[c0 + 8], a.scale[c0 + 9]); sq[kk][3] = pack_f32x2(a.shift[c0 + 8], a.shift[c0 + 9]);
    }
  }
  fence_proxy_async_smem();   // the staging writes precede the TMA writes of buffer 0
  __syncthreads();                                     // the staging region becomes span buffer 0
  const float rh = a.OH > 1 ? (float)(LH - 1) / (float)(a.OH - 1) : 0.f;               // ATen upsample_bilinear2d(align_corners=True)
  const float rw = a.OW > 1 ? (float)(LW - 1) / (float)(a.OW - 1) : 0.f;
  // one thread: the tile's span of Y_3 (one box: 64 px x 4 groups of 64 channels) and the two low-resolution rows of
  // every class (one box [K][2][kSeg]; columns beyond the row end and the row below the last arrive as zeros)
  // (no thread ever writes a TMA-target buffer after the prologue, so the issue needs no proxy fence)
  auto issue = [&](const TileXY& c, int b) {
    const int h1 = (int)(rh * (float)c.oh);
    const int ws = (int)(rw * (float)c.w0) & ~3;
    const int pix0 = (c.n * a.IH + hsrc[c.oh]) * a.IW + wstart[c.w0 / kPx];
    mbar_expect_tx(&bar[b], kSpanBytes + 2u * (uint32_t)K * (uint32_t)(kSeg * 4));
    tma_3d(smem_u32(ysm) + (uint32_t)b * kSpanBytes, &tm_y, &bar[b], 0, pix0, 0);
    tma_3d(smem_u32(trow + (size_t)b * 2 * kCls * kSeg), &tm_lo, &bar[b], ws, h1, c.n * K);
  };
  TileWalk walk(a, blockIdx.x, gridDim.x, wtiles);
  if (t == 0) issue(walk.xy(), 0);
  TR_DECL
  int it = 0;
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
    const int b = it & 1;
    const TileXY c = walk.xy();
    __syncthreads();                                   // (A) the previous tile is consumed: the other buffers are free
    TR(0);
    walk.advance();
    if (t == 0 && tile + (int)gridDim.x < num_tiles) issue(walk.xy(), b ^ 1);
    const float h1r = rh * (float)c.oh;
    const float hl1 = h1r - (float)(int)h1r, hl0 = 1.f - hl1;
    const int ws = (int)(rw * (float)c.w0) & ~3;
    TR(1);
    mbar_wait(&bar[b], (uint32_t)(it >> 1) & 1u);      // the copies are visible through the barrier
    TR(2);
    const float* tr = trow + (size_t)b * 2 * kCls * kSeg;
    {
      const int sidx0 = rel[c.w0 + 32 * u + arow], sidx1 = rel[c.w0 + 32 * u + 16 + arow];
      const uint32_t ybase = smem_u32(ysm) + (uint32_t)b * kSpanBytes;
      float acc[2][3][4];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
          for (int r = 0; r < 4; ++r) acc[i][j][r] = 0.f;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const int kb = 4 * q + kk;
        uint32_t a0[4], a1[4];
        ldsm_x4(span_addr(ybase, sidx0, kb * 2 + akc), a0);
        ldsm_x4(span_addr(ybase, sidx1, kb * 2 + akc), a1);
        a0[0] = bn_relu_x2(a0[0], sq[kk][0], sq[kk][1]); a0[1] = bn_relu_x2(a0[1], sq[kk][0], sq[kk][1]);
        a0[2] = bn_relu_x2(a0[2], sq[kk][2], sq[kk][3]); a0[3] = bn_relu_x2(a0[3], sq[kk][2], sq[kk][3]);
        a1[0] = bn_relu_x2(a1[0], sq[kk][0], sq[kk][1]); a1[1] = bn_relu_x2(a1[1], sq[kk][0], sq[kk][1]);
        a1[2] = bn_relu_x2(a1[2], sq[kk][2], sq[kk][3]); a1[3] = bn_relu_x2(a1[3], sq[kk][2], sq[kk][3]);
        mma_bf16(acc[0][0], a0, bq[kk][0], bq[kk][1]);
        mma_bf16(acc[0][1], a0, bq[kk][2], bq[kk][3]);
        mma_bf16(acc[0][2], a0, bq[kk][4], bq[kk][5]);
        mma_bf16(acc[1][0], a1, bq[kk][0], bq[kk][1]);
        mma_bf16(acc[1][1], a1, bq[kk][2], bq[kk][3]);
        mma_bf16(acc[1][2], a1, bq[kk][4], bq[kk][5]);
      }
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int nb = 0; nb < 3; ++nb) {               // c0,c1: (pixel g, class 2tq, 2tq+1); c2,c3: pixel g + 8
          float* o = outst + (size_t)q * kCls * kOutPitch + (nb * 8 + 2 * tq) * kOutPitch + 32 * u + 16 * i + g;
          o[0] = acc[i][nb][0]; o[kOutPitch] = acc[i][nb][1]; o[8] = acc[i][nb][2]; o[kOutPitch + 8] = acc[i][nb][3];
        }
    }
    TR(5);
    __syncthreads();                                   // (C)
    TR(6);
    // ---- quarter sums + bias + the four bilinear taps (ATen's order: rows outside, columns inside): thread = one pixel,
    //      classes cg, cg + 4, ...; a warp writes 128 contiguous bytes of one fp32 NCHW row per class ----
    {
      const int px = t & (kPx - 1), cg = t >> 6, ow = c.w0 + px;
      if (ow < a.OW) {
        const float w1r = rw * (float)ow;
        const int w1 = (int)w1r;
        const float wl1 = w1r - (float)w1, wl0 = 1.f - wl1;
        const int x0 = w1 - ws, x1 = x0 + (w1 < LW - 1 ? 1 : 0);
        float* op = out + (((size_t)c.n * K + cg) * a.OH + c.oh) * a.OW + ow;
        const size_t plane4 = (size_t)4 * a.OH * a.OW;
#pragma unroll 2
        for (int k = cg; k < K; k += 4, op += plane4) {
          const float* v0 = tr + (size_t)k * 2 * kSeg;
          const float* v1 = v0 + kSeg;
          const float* o = outst + k * kOutPitch + px;
          const float acc = (o[0] + o[kCls * kOutPitch]) + (o[2 * kCls * kOutPitch] + o[3 * kCls * kOutPitch]);
          const float up = hl0 * fmaf(wl0, v0[x0], wl1 * v0[x1]) + hl1 * fmaf(wl0, v1[x0], wl1 * v1[x1]);
          *op = acc + ((b2 ? b2[k] : 0.f) + up);
        }
      }
    }
    TR(7);
  }
  TR_END(0);
}

// 4 x 4 transpose among the four lanes of a quad (two butterfly stages, selects only): lane tq holds r[j], j = 0..3;
// afterwards lane tq holds the r[tq] of lanes 0..3 of its quad, in lane order
__device__ __forceinline__ uint4 quad_transpose(const uint32_t (&r)[4], int tq) {
  const bool up = (tq & 2) != 0, odd = (tq & 1) != 0;
  const uint32_t t0 = __shfl_xor_sync(0xffffffffu, up ? r[0] : r[2], 2);
  const uint32_t t1 = __shfl_xor_sync(0xffffffffu, up ? r[1] : r[3], 2);
  const uint32_t a0 = up ? t0 : r[0], a1 = up ? t1 : r[1], a2 = up ? r[2] : t0, a3 = up ? r[3] : t1;
  const uint32_t u0 = __shfl_xor_sync(0xffffffffu, odd ? a0 : a1, 1);
  const uint32_t u1 = __shfl_xor_sync(0xffffffffu, odd ? a2 : a3, 1);
  uint4 o;
  o.x = odd ? u0 : a0; o.y = odd ? a1 : u0; o.z = odd ? u1 : a2; o.w = odd ? a3 : u1;
  return o;
}

constexpr size_t kBwdSmem = 1024 + (size_t)2 * kSpanBytes + (size_t)32 * kPx * 2 + (size_t)2 * 32 * kPx * 4 + 16;
                             // + the index tables: (wtiles * 65 + OH) ints

// backward: warp = channels [32 warp, +32) in both products.  g_tma: g arrives as one [K][64] box per tile; otherwise
// (rows of g not 16-byte aligned) through plain loads.  g64 != nullptr: the RANK-K form — instead of dA = W2^T g the kernel
// leaves g itself as bf16 (N, OH, OW, 64) (classes beyond K zero) and W2T (256, 64) bf16 in w2t64; the stage-4 dgrad takes
// the product as one more k-block of its accumulation (conv_gather.cu, ADD == 2) and dA never exists
__global__ void __launch_bounds__(kThreads, 2)
tail_final2_bwd_kernel(const __grid_constant__ CUtensorMap tm_y, const __grid_constant__ CUtensorMap tm_g, const TailArgs a,
                        const float* __restrict__ gsrc, int g_tma, __nv_bfloat16* __restrict__ dA, float* __restrict__ gW2,
                        float* __restrict__ gb2, int wtiles, int num_tiles, __nv_bfloat16* __restrict__ g64,
                        __nv_bfloat16* __restrict__ w2t64) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* ysm = smem_1k(smem_raw);                          // [2][4 boxes][64 px][64 ch bf16]
  unsigned char* gC = ysm + (size_t)2 * kSpanBytes;               // [32 classes][64 px bf16]   (128-byte rows, swizzled)
  float* gF = reinterpret_cast<float*>(gC + (size_t)32 * kPx * 2);   // [2][32 classes][64 px fp32]: g as it arrives
  uint64_t* bar = reinterpret_cast<uint64_t*>(gF + 2 * 32 * kPx);   // [2] full barriers
  int* rel = reinterpret_cast<int*>(bar + 2);                      // [wtiles * 64]: source pixel - the tile's first
  int* wstart = rel + wtiles * kPx;                               // [wtiles]: first source pixel of a tile
  int* hsrc = wstart + wtiles;                                     // [OH]: source row of an output row
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int K = a.K;
  const int g8 = lane >> 2, tq = lane & 3;
  const int amat = lane >> 3, arow = (amat & 1) * 8 + (lane & 7), akc = amat >> 1;
  if (t == 0) {
    mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); mbar_fence_init();
    prefetch_tensormap(&tm_y);
    if (g_tma) prefetch_tensormap(&tm_g);
  }
  pdl_sync();
  // W2^T -> bf16 [channel][class] (16-byte chunks swizzled by (channel >> 1) & 3) in the span buffer, then into B fragments
  for (int e = t; e < kC * 32; e += kThreads) {
    const int c = e >> 5, k = e & 31;
    const float v = k < K ? a.w2[k * kC + c] : 0.f;
    *reinterpret_cast<__nv_bfloat16*>(ysm + c * 64 + (((k >> 3) ^ ((c >> 1) & 3)) << 4) + (k & 7) * 2) = __float2bfloat16_rn(v);
  }
  for (int e = t; e < 2 * 32 * kPx; e += kThreads) gF[e] = 0.f;    // rows of classes >= K stay zero from here on
  if (g64 != nullptr && blockIdx.x == 0)                            // rank-K form: the classifier transposed, (256, 64) bf16
    for (int e = t; e < kC * 64; e += kThreads) {
      const int c = e >> 6, k = e & 63;
      w2t64[e] = __float2bfloat16_rn(k < K ? a.w2[k * kC + c] : 0.f);
    }
  for (int e = t; e < wtiles * kPx; e += kThreads) rel[e] = a.idx_w[min(e, a.OW - 1)] - a.idx_w[e & ~(kPx - 1)];
  for (int e = t; e < wtiles; e += kThreads) wstart[e] = a.idx_w[e * kPx];
  for (int e = t; e < a.OH; e += kThreads) hsrc[e] = a.idx_h[e];
  __syncthreads();
  uint32_t w1b[2][2][4];                                // [16-channel pair np][class k-block][n-block 2np: b0 b1 | 2np + 1: b0 b1]
  {
    const int bn = (amat >> 1) * 8 + (lane & 7), bkc = amat & 1;
#pragma unroll
    for (int np = 0; np < 2; ++np)
#pragma unroll
      for (int kb = 0; kb < 2; ++kb) {
        const int ch = 32 * warp + np * 16 + bn;
        ldsm_x4(smem_u32(ysm + ch * 64 + (((kb * 2 + bkc) ^ ((ch >> 1) & 3)) << 4)), w1b[np][kb]);
      }
  }
  uint64_t sc[4][2];                                    // (scale, scale), (shift, shift) of channel 32 warp + 8 j + g8
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float s_ = a.scale[32 * warp + j * 8 + g8], b_ = a.shift[32 * warp + j * 8 + g8];
    sc[j][0] = pack_f32x2(s_, s_); sc[j][1] = pack_f32x2(b_, b_);
  }
  float wacc[2][4][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int r = 0; r < 4; ++r) wacc[i][j][r] = 0.f;
  float sg[4] = {0.f, 0.f, 0.f, 0.f};                   // bias-gradient partials of classes warp + 8 i (this lane's two pixels)
  fence_proxy_async_smem();   // staging writes and the zero fill precede the TMA writes
  __syncthreads();                                      // the staging region becomes span buffer 0

  // one thread: the tile's span of Y_3 (one box: 64 px x 4 groups of 64 channels) and its [K][64] box of g (pixels beyond the row end arrive as zeros)
  // (no thread ever writes a TMA-target buffer after the prologue, so the issue needs no proxy fence)
  auto issue = [&](const TileXY& c, int b) {
    const int pix0 = (c.n * a.IH + hsrc[c.oh]) * a.IW + wstart[c.w0 / kPx];
    mbar_expect_tx(&bar[b], kSpanBytes + (g_tma ? (uint32_t)K * (uint32_t)(kPx * 4) : 0u));
    tma_3d(smem_u32(ysm) + (uint32_t)b * kSpanBytes, &tm_y, &bar[b], 0, pix0, 0);
    if (g_tma) tma_3d(smem_u32(gF + (size_t)b * 32 * kPx), &tm_g, &bar[b], c.w0, c.oh, c.n * K);
  };
  auto load_g_slow = [&](const TileXY& c, int b) {       // every thread: generic loads into the staging tile
    float* dstb = gF + (size_t)b * 32 * kPx;
    for (int e = t; e < K * kPx; e += kThreads) {
      const int k = e >> 6, px = e & 63, ow = c.w0 + px;
      dstb[k * kPx + px] = ow < a.OW ? __ldg(gsrc + (((size_t)c.n * K + k) * a.OH + c.oh) * a.OW + ow) : 0.f;
    }
  };
  TileWalk walk(a, blockIdx.x, gridDim.x, wtiles);
  if (t == 0) issue(walk.xy(), 0);
  if (!g_tma) load_g_slow(walk.xy(), 0);
  TR_DECL
  int it = 0;
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
    const int b = it & 1;
    const TileXY c = walk.xy();
    const bool more = tile + (int)gridDim.x < num_tiles;
    __syncthreads();                                   // (A) the previous tile is consumed
    TR(0);
    walk.advance();
    if (more) {
      if (t == 0) issue(walk.xy(), b ^ 1);
      if (!g_tma) load_g_slow(walk.xy(), b ^ 1);
    }
    TR(1);
    TR(2);
    mbar_wait(&bar[b], (uint32_t)(it >> 1) & 1u);
    TR(3);
    {
      const float* gb = gF + (size_t)b * 32 * kPx;
#pragma unroll
      for (int i = 0; i < 4; ++i) {                    // g tile -> bf16 [class][pixel]: a warp writes one whole 128-byte row
        const int k = warp + 8 * i;
        const float2 v = *reinterpret_cast<const float2*>(gb + k * kPx + 2 * lane);
        *reinterpret_cast<uint32_t*>(gC + k * 128 + (((lane >> 2) ^ (k & 7)) << 4) + (lane & 3) * 4) = pack_bf16x2(v.x, v.y);
        sg[i] += v.x + v.y;
      }
    }
    __syncthreads();                                   // (B) gC is visible
    TR(4);
    const uint32_t ybase = smem_u32(ysm) + (uint32_t)b * kSpanBytes;

    if (g64 != nullptr) {
      // ---- (1') rank-K form: the tile of g as bf16 [pixel][64 classes]; 8 pixels x 128 contiguous bytes per warp store ----
      const float* gb = gF + (size_t)b * 32 * kPx;
      const int px = t >> 2, quarter = t & 3;          // 16 classes = 32 bytes per thread
      if (c.w0 + px < a.OW) {
        uint32_t pk[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        if (quarter < 2) {
#pragma unroll
          for (int j = 0; j < 8; ++j) pk[j] = pack_bf16x2(gb[(16 * quarter + 2 * j) * kPx + px], gb[(16 * quarter + 2 * j + 1) * kPx + px]);
        }
        uint4* dst = reinterpret_cast<uint4*>(g64 + (((size_t)c.n * a.OH + c.oh) * a.OW + c.w0 + px) * 64 + 16 * quarter);
        dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
      }
    } else {
      // ---- (1) dA3[px][ch] = sum_k g[k][px] W2[k][ch]: A fragments by ldmatrix.trans from gC, results leave from registers ----
#pragma unroll 2
      for (int mt = 0; mt < kPx / 16; ++mt) {
        uint32_t af[2][4];
#pragma unroll
        for (int kb = 0; kb < 2; ++kb) {                 // matrices: (px 0-7 | px 8-15) x (classes 16 kb + 0-7 | + 8-15)
          const int cls = 16 * kb + (amat >> 1) * 8 + (lane & 7), chunk = 2 * mt + (amat & 1);
          ldsm_x4_trans(smem_u32(gC + cls * 128 + ((chunk ^ (cls & 7)) << 4)), af[kb]);
        }
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll
        for (int np = 0; np < 2; ++np)
#pragma unroll
          for (int kb = 0; kb < 2; ++kb) {
            mma_bf16(acc[2 * np], af[kb], w1b[np][kb][0], w1b[np][kb][1]);
            mma_bf16(acc[2 * np + 1], af[kb], w1b[np][kb][2], w1b[np][kb][3]);
          }
        uint32_t r0[4], r1[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { r0[j] = pack_bf16x2(acc[j][0], acc[j][1]); r1[j] = pack_bf16x2(acc[j][2], acc[j][3]); }
        const uint4 o0 = quad_transpose(r0, tq), o1 = quad_transpose(r1, tq);     // channels 32 warp + 8 tq + 0..7
        const int p0 = 16 * mt + g8, p1 = p0 + 8;
        __nv_bfloat16* drow = dA + (((size_t)c.n * a.OH + c.oh) * a.OW + c.w0) * kC + 32 * warp + 8 * tq;
        if (c.w0 + p0 < a.OW) *reinterpret_cast<uint4*>(drow + (size_t)p0 * kC) = o0;
        if (c.w0 + p1 < a.OW) *reinterpret_cast<uint4*>(drow + (size_t)p1 * kC) = o1;
      }
    }

    TR(5);
    // ---- (2) gW2[k][ch] += sum_px g[k][px] ReLU(BN(Y_3[src(px)][ch])) ----
    {
      const int tm = lane >> 3;                        // B (.trans): matrices (k 0-7 | k 8-15) x (n-block j | j + 1)
      const int brow = (tm & 1) * 8 + (lane & 7);      // pixel within the k-block
      const int bnb = tm >> 1;                         // n-block within the pair
#pragma unroll 2
      for (int kb = 0; kb < kPx / 16; ++kb) {
        uint32_t a0[4], a1[4];
        ldsm_x4(smem_u32(gC + arow * 128 + (((kb * 2 + akc) ^ (arow & 7)) << 4)), a0);
        ldsm_x4(smem_u32(gC + (16 + arow) * 128 + (((kb * 2 + akc) ^ ((16 + arow) & 7)) << 4)), a1);
        const int sidx = rel[c.w0 + kb * 16 + brow];
#pragma unroll
        for (int jp = 0; jp < 2; ++jp) {               // n-block pairs: channels 32 warp + 16 jp + {0..7, 8..15}
          const int chunk = 4 * warp + 2 * jp + bnb;   // 16-byte chunk (8 channels) of the pixel's 256 channels
          uint32_t bf[4];
          ldsm_x4_trans(span_addr(ybase, sidx, chunk), bf);
          bf[0] = bn_relu_x2(bf[0], sc[2 * jp][0], sc[2 * jp][1]); bf[1] = bn_relu_x2(bf[1], sc[2 * jp][0], sc[2 * jp][1]);
          bf[2] = bn_relu_x2(bf[2], sc[2 * jp + 1][0], sc[2 * jp + 1][1]); bf[3] = bn_relu_x2(bf[3], sc[2 * jp + 1][0], sc[2 * jp + 1][1]);
          mma_bf16(wacc[0][2 * jp], a0, bf[0], bf[1]);
          mma_bf16(wacc[0][2 * jp + 1], a0, bf[2], bf[3]);
          mma_bf16(wacc[1][2 * jp], a1, bf[0], bf[1]);
          mma_bf16(wacc[1][2 * jp + 1], a1, bf[2], bf[3]);
        }
      }
    }
    TR(6);
  }
  TR_END(8);
  // ---- publish the CTA's weight- and bias-gradient partials ----
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ch = 32 * warp + j * 8 + 2 * tq;
      const int k0 = mt * 16 + g8, k1 = k0 + 8;
      if (k0 < K) { atomicAdd(gW2 + k0 * kC + ch, wacc[mt][j][0]); atomicAdd(gW2 + k0 * kC + ch + 1, wacc[mt][j][1]); }
      if (k1 < K) { atomicAdd(gW2 + k1 * kC + ch, wacc[mt][j][2]); atomicAdd(gW2 + k1 * kC + ch + 1, wacc[mt][j][3]); }
    }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float s = warp_sum(sg[i]);
    if (lane == 0 && warp + 8 * i < K) atomicAdd(gb2 + warp + 8 * i, s);
  }
}

int tail_args(const mrfp_hrfp_plan* P, const void* saved, const void* lut, const float* w2, int K, TailArgs* a) {
  if (P->mode != MRFP_MATH_BF16) return MRFP_ERR_UNSUPPORTED;
  const HrfpStage& st = P->st[3];
  if (st.cout != kC || K <= 0 || K > kCls) return MRFP_ERR_UNSUPPORTED;
  const int* hidx = P->lut.data() + st.idx_w;           // every tile's source span must fit the buffer
  for (int w0 = 0; w0 < st.ow; w0 += kPx) {
    const int w1 = (w0 + kPx < st.ow ? w0 + kPx : st.ow) - 1;
    if (hidx[w1] - hidx[w0] + 1 > kSpan) return MRFP_ERR_UNSUPPORTED;
  }
  if ((long long)P->N * st.ch * st.cw > 0x7fffffffLL) return MRFP_ERR_BAD_SHAPE;   // pixel coordinate of the tensor map
  const float* stats = reinterpret_cast<const float*>((const char*)saved + P->stats_off) + (size_t)3 * 4 * kMaxC;
  a->y = reinterpret_cast<const __nv_bfloat16*>((const char*)saved + st.y_off);
  a->idx_h = (const int*)lut + st.idx_h; a->idx_w = (const int*)lut + st.idx_w;
  a->scale = stats + 2 * kMaxC; a->shift = stats + 3 * kMaxC;
  a->N = P->N; a->IH = st.ch; a->IW = st.cw; a->OH = st.oh; a->OW = st.ow; a->K = K;
  a->w2 = w2;
  return MRFP_OK;
}

// the launch's two descriptors, cached in the plan per direction and re-encoded when an address or a shape changes
int tail_maps(const mrfp_hrfp_plan* P, int dir, const TailArgs& a, const float* aux, int d0, int d1, int box_w, int box_h,
              bool want_aux, TailMaps* out) {
  std::lock_guard<std::mutex> lock(P->mu);
  TailMaps* m = &P->maps_tail[dir];
  if (!m->valid || m->key[0] != a.y || m->key[1] != aux || m->k != a.K || m->d0 != d0 || m->d1 != d1) {
    m->valid = 0;
    {
      // Y_3 as [4 groups of 64 channels][pixel][64 channels]: one box = 64 pixels x 4 groups, which lands as four
      // SWIZZLE_128B tiles of [64 px][128 bytes]
      const cuuint64_t dims[3] = {64, (cuuint64_t)a.N * a.IH * a.IW, 4};
      const cuuint64_t strides[2] = {(cuuint64_t)kC * 2, 128};
      const cuuint32_t box[3] = {64, kSpan, 4};
      int rc = conv_make_map(&m->y, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, a.y, 3, dims, strides, box, true);
      if (rc) return rc;
    }
    if (want_aux) {                                      // fp32 (N * K, d0, d1): one box = box_w columns of one row of K planes
      const cuuint64_t dims[3] = {(cuuint64_t)d1, (cuuint64_t)d0, (cuuint64_t)a.N * a.K};
      const cuuint64_t strides[2] = {(cuuint64_t)d1 * 4, (cuuint64_t)d0 * d1 * 4};
      const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)a.K};
      int rc = conv_make_map(&m->aux, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, aux, 3, dims, strides, box, false);
      if (rc) return rc;
    } else {
      m->aux = m->y;
    }
    m->key[0] = a.y; m->key[1] = aux; m->k = a.K; m->d0 = d0; m->d1 = d1;
    m->valid = 1;
  }
  *out = *m;
  return MRFP_OK;
}

}  // namespace
}  // namespace mrfp

using namespace mrfp;

extern "C" int mrfp_hrfp_tail_final2_fwd(const mrfp_hrfp_plan_t* P, const void* saved, const void* lut, const float* t_lo,
                                         int lh, int lw, const float* w2, const float* b2, int K, float* out, void* stream) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  if (!saved || !lut || !t_lo || !w2 || !out) return MRFP_ERR_NULL_POINTER;
  if (lh <= 0 || lw <= 0) return MRFP_ERR_BAD_SHAPE;
  TailArgs a;
  int rc = tail_args(P, saved, lut, w2, K, &a);
  if (rc) return rc;
  // the staged low-resolution span: an Upsample by >= 2 (as the reference's), rows 16-byte aligned for the tensor map
  if (lw > a.OW || lh > a.OH || !(a.OW > 1 && 2 * (lw - 1) <= a.OW - 1) || (lw & 3) || ((uintptr_t)t_lo & 15)) return MRFP_ERR_UNSUPPORTED;
  DeviceInfo di;
  rc = get_device_info(&di);
  if (rc) return rc;
  const int wtiles = (a.OW + kPx - 1) / kPx;
  const long long tiles = (long long)a.N * a.OH * wtiles;
  if (tiles > 0x7fffffffLL) return MRFP_ERR_BAD_SHAPE;
  const int grid = (int)(tiles < 2LL * di.sm_count ? tiles : 2LL * di.sm_count);
  TailMaps tm;
  rc = tail_maps(P, 0, a, t_lo, lh, lw, kSeg, 2, true, &tm);
  if (rc) return rc;
  const size_t smem = kFwdSmem + ((size_t)wtiles * (kPx + 1) + a.OH) * sizeof(int);
  if (smem > (size_t)di.max_smem_optin) return MRFP_ERR_UNSUPPORTED;
  MRFP_SMEM_OPT_IN(tail_final2_fwd_kernel, di.max_smem_optin, di.device);
  launch_k(tail_final2_fwd_kernel, dim3(grid), dim3(kThreads), smem, (cudaStream_t)stream, tm.y, tm.aux, a, lh, lw, b2, out, wtiles,
           (int)tiles);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

static int tail_bwd_launch(const mrfp_hrfp_plan_t* P, const void* saved, const void* lut, const float* g, const float* w2, int K,
                           void* g_dec_nhwc, void* g64, void* w2t64, float* g_w2, float* g_b2, void* stream) {
  if (!P || P->magic != kPlanMagic) return MRFP_ERR_BAD_PLAN;
  if (!saved || !lut || !g || !w2 || !g_w2 || !g_b2 || (!g_dec_nhwc && !(g64 && w2t64))) return MRFP_ERR_NULL_POINTER;
  if (((uintptr_t)g_dec_nhwc | (uintptr_t)g64 | (uintptr_t)w2t64) & 15) return MRFP_ERR_WORKSPACE;
  TailArgs a;
  int rc = tail_args(P, saved, lut, w2, K, &a);
  if (rc) return rc;
  DeviceInfo di;
  rc = get_device_info(&di);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  MRFP_CUDA_TRY(cudaMemsetAsync(g_w2, 0, (size_t)K * kC * sizeof(float), s));
  MRFP_CUDA_TRY(cudaMemsetAsync(g_b2, 0, (size_t)K * sizeof(float), s));
  const int wtiles = (a.OW + kPx - 1) / kPx;
  const long long tiles = (long long)a.N * a.OH * wtiles;
  if (tiles > 0x7fffffffLL) return MRFP_ERR_BAD_SHAPE;
  const int grid = (int)(tiles < 2LL * di.sm_count ? tiles : 2LL * di.sm_count);
  const int g_tma = (a.OW & 3) == 0 && ((uintptr_t)g & 15) == 0;     // rows of g 16-byte aligned: one box per tile
  TailMaps tm;
  rc = tail_maps(P, 1, a, g, a.OH, a.OW, kPx, 1, g_tma != 0, &tm);
  if (rc) return rc;
  const size_t smem = kBwdSmem + ((size_t)wtiles * (kPx + 1) + a.OH) * sizeof(int);
  if (smem > (size_t)di.max_smem_optin) return MRFP_ERR_UNSUPPORTED;
  MRFP_SMEM_OPT_IN(tail_final2_bwd_kernel, di.max_smem_optin, di.device);
  launch_k(tail_final2_bwd_kernel, dim3(grid), dim3(kThreads), smem, s, tm.y, tm.aux, a, g, g_tma,
           reinterpret_cast<__nv_bfloat16*>(g_dec_nhwc), g_w2, g_b2, wtiles, (int)tiles, reinterpret_cast<__nv_bfloat16*>(g64),
           reinterpret_cast<__nv_bfloat16*>(w2t64));
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

extern "C" int mrfp_hrfp_tail_final2_bwd(const mrfp_hrfp_plan_t* P, const void* saved, const void* lut, const float* g,
                                         const float* w2, int K, void* g_dec_nhwc, float* g_w2, float* g_b2, void* stream) {
  if (!g_dec_nhwc) return MRFP_ERR_NULL_POINTER;
  return tail_bwd_launch(P, saved, lut, g, w2, K, g_dec_nhwc, nullptr, nullptr, g_w2, g_b2, stream);
}

extern "C" int mrfp_hrfp_tail_final2_bwd_rk(const mrfp_hrfp_plan_t* P, const void* saved, const void* lut, const float* g,
                                            const float* w2, int K, void* g64, void* w2t64, float* g_w2, float* g_b2,
                                            void* stream) {
  if (!g64 || !w2t64) return MRFP_ERR_NULL_POINTER;
  return tail_bwd_launch(P, saved, lut, g, w2, K, nullptr, g64, w2t64, g_w2, g_b2, stream);
}

#ifdef MRFP_TAIL_TRACE
extern "C" int mrfp_debug_tail_trace(unsigned long long* host16, int reset) {
  if (host16) MRFP_CUDA_TRY(cudaMemcpyFromSymbol(host16, mrfp::g_tail_dbg, sizeof(unsigned long long) * 16));
  if (reset) { unsigned long long z[16] = {0}; MRFP_CUDA_TRY(cudaMemcpyToSymbol(mrfp::g_tail_dbg, z, sizeof(z))); }
  return 0;
}
#endif
