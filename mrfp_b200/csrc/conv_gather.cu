// tcgen05 implicit-GEMM 3x3 convolution whose A operand is BUILT ON CHIP from the neighbouring tensors of the chain
// (sm_100a, bf16 operands, fp32 accumulation in TMEM).  Per stage of /root/reference/deepv3.py:320-327 it replaces
//   kGatherFwd    F.interpolate(nearest) -> BatchNorm2d (batch statistics) -> ReLU -> Conv2d         (stage k >= 1)
//                 the activation A_k is produced straight into the operand tile from Y_{k-1} and that BatchNorm's table
//   kGatherBwd    ReLU' -> BatchNorm2d backward -> adjoint of the nearest resample -> Conv2d dgrad   (stages whose resample
//                 never replicates a pixel: the identity and the down-sampling stages) — dY_k is produced from dA_{k+1},
//                 Y_k and the BN-backward sums
//   kGatherBwdRep the same for an up-sampling stage (a source pixel has up to 2 x 2 replicas in dA_{k+1}): the first replica
//                 goes to the gradient side stage, the others to a compacted "extras" stage
// so that A_k (forward) and dY_k (backward) never exist in HBM.
//
// Tile: 16 rows x (8 * MT) columns of output pixels; each 16 x 8 sub-tile is one UMMA M = 128 accumulator.  Per
// 64-channel chunk ONE halo tile is built: the (16 + 2d) x (8 MT + 2d) input neighbourhood, a pixel per 128-byte row,
// rows of the box contiguous, 16-byte pieces XOR-swizzled with bits 7..9 of their own shared-memory address (the
// 128-byte swizzle is a function of the absolute address, so ANY 128-byte-aligned start is a valid view).  The 9 taps
// are 9 start addresses into that tile: an eight-row group of the M tile is 8 consecutive pixels of one image row,
// consecutive groups are one box row (boxw * 128 B) apart = the descriptor's stride-byte-offset.  The element-wise work
// therefore runs ONCE per input element (not once per tap), and the L2->SM operand stream drops to the weights (one
// {64, COUT} TMA box per (chunk, tap), own ring) plus ~1.3-1.9x the input (halo overlap).
//
// Warp roles (448 threads, persistent over tiles): warp 0 = weight TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2-5 = epilogue (conv_common.cuh: TMEM -> staging tile -> TMA store, BN statistics, BN finalisation),
// warps 6-13 = operand producers: cp.async.cg copies (L2 -> shared memory, no registers, no L1 allocation) put the raw
// bf16 values at their final swizzled place nA - 1 stages ahead; the thread that copied a piece rewrites it in place
// (forward: ReLU(scale * y + shift); backward: the BN-backward apply of y and the gradient piece that the same thread
// copied into a side stage) once it has landed.
#include "conv_common.cuh"
#include <algorithm>
#include <atomic>
#include <vector>

namespace mrfp {
namespace {
using namespace convk;
using namespace ptx;

constexpr int kGThreads = 448;
constexpr int kGTileH = 16, kGSubW = 8;        // M sub-tile: 16 rows x 8 columns
constexpr int kProducers = 256;                // warps 6..13
constexpr int kPxLanes = kProducers / 8;       // box pixels handled per pass (8 threads = the 8 16-byte pieces of a pixel)
constexpr int kMaxAStages = 4;
constexpr int kSmemLimit = 232448;             // 227 KB opt-in maximum per CTA

constexpr int kMaxBStages = 6;
constexpr int kGatherFwd = 0, kGatherBwd = 1, kGatherBwdRep = 2;
// staging tiles, row weights, barriers at compile-time offsets; rounded so that everything behind stays 1024-aligned
constexpr int kFixedBytes = (2 * kStageOutBytes + 512 + 8 * (2 * kMaxAStages + 2 * kMaxBStages + 6) + 16 + 1023) / 1024 * 1024;

template <int COUT> struct GCfg {
  static constexpr int kBTileBytes = COUT * 128;
  static constexpr int kBStages = COUT == 256 ? 4 : (COUT == 128 ? 4 : 6);     // preferred depth of the weight ring
};

// what the producers gather from
struct GatherArgs {
  const __nv_bfloat16* y;      // fwd: Y_{k-1} [N][SH][SW][CIN];  bwd: Y_k [N][H][W][CIN]
  const __nv_bfloat16* g;      // bwd: dA_{k+1} [N][SH][SW][CIN]
  const int* tab_h;            // fwd: idx_h [H] (dst -> src row);  bwd: lo_h [H + 1] (first replica of each source row)
  const int* tab_w;
  const float* stats;          // [4][kMaxC] mean, invstd, scale, shift of the BatchNorm in question
  const float* gamma;          // bwd
  const double* acc;           // bwd: [2][kMaxC] sum mask*dA, sum mask*dA*y (bn_bwd_reduce)
  double count;                // bwd: elements per channel of the resampled tensor
  int SH, SW;                  // fwd: resolution of Y_{k-1};  bwd: of dA_{k+1}
  int c_real;                  // bwd: channels of the module's BatchNorm (stored channels beyond it: dY = 0)
};

__device__ __forceinline__ void prod_bar_sync() { asm volatile("bar.sync 2, 256;" ::: "memory"); }
__device__ __forceinline__ void ld8s(uint32_t a, float (&v)[8]) {
  const uint4 x = lds_v4(a), y = lds_v4(a + 16);
  v[0] = __uint_as_float(x.x); v[1] = __uint_as_float(x.y); v[2] = __uint_as_float(x.z); v[3] = __uint_as_float(x.w);
  v[4] = __uint_as_float(y.x); v[5] = __uint_as_float(y.y); v[6] = __uint_as_float(y.z); v[7] = __uint_as_float(y.w);
}

// kGatherFwd:   in[h][w][c] = ReLU(scale[c] * y[idx_h[h]][idx_w[w]][c] + shift[c])
// kGatherBwd:   in[h][w][c] = P[c] * [scale[c]*y+shift[c] > 0] * g[replica of (h,w)][c] - (R[c]*y[h][w][c] + Q[c])  where (h,w) has a
//               replica, 0 where it has none (a pixel the down-sampling skipped receives no gradient)
// each inside the image, 0 in the convolution's zero padding
// ADD: 0 nothing joins the output; 1 a tensor of the output's shape is added in the epilogue (add tile by TMA); 2 a RANK-K
// term joins as one more k-block of the accumulation: out += G[pixel][0:32] . W2T[cout][0:32]^T (the classifier tail's gradient,
// tail_final2.cu) — its two operands travel through the weight ring: tmap_add describes G (N, H, W, 64), tmap_rkw W2T (cout, 64).
// Two UMMA k-steps of 16 read columns 0..31 only: the tail takes <= 24 classes and leaves the columns beyond them zero
// (include/mrfp_b200.h), so columns 32..63 are padding of the 128-byte rows and never enter the product
template <int COUT, int MODE, int ADD, int MT>
__global__ void __launch_bounds__(kGThreads, 1)
conv3x3_gather_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_out,
                      const __grid_constant__ CUtensorMap tmap_add, const __grid_constant__ CUtensorMap tmap_rkw, const GatherArgs ga, int CIN, int dil, int boxw, int tiles_h, int tiles_w, int num_tiles,
                      const int* __restrict__ cnt_h, const int* __restrict__ cnt_w, double* __restrict__ stat_acc, int rev,
                      const ConvBnFinalize fin, const __nv_bfloat16* __restrict__ add_src, int H, int W, int nA, int nB,
                      int a_stage_bytes, int tab_bytes, int e_bytes) {
  using C = GCfg<COUT>;
  using T = __nv_bfloat16;
  constexpr int kBlockK = 64;
  constexpr bool kBwd = MODE != kGatherFwd;
  constexpr int kTmemCols = 2 * MT * COUT;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  // what the epilogue touches sits at compile-time offsets; the weight ring, the halo stages, the gradient side stage
  // (kGatherBwd), the gather tables and the per-channel constants follow at run-time offsets and are addressed explicitly
  unsigned char* sOut = smem;
  float* s_wgt = reinterpret_cast<float*>(sOut + 2 * kStageOutBytes);          // [128]
  uint64_t* full_a = reinterpret_cast<uint64_t*>(s_wgt + 128);
  uint64_t* empty_a = full_a + kMaxAStages;
  uint64_t* full_b = empty_a + kMaxAStages;
  uint64_t* empty_b = full_b + kMaxBStages;
  uint64_t* tmem_full = empty_b + kMaxBStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* add_full = tmem_empty + 2;                                         // ADD: the epilogue's add tile has landed
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(add_full + 2);
  unsigned char* sB = smem + kFixedBytes;                                      // nB weight tiles
  unsigned char* sA = sB + nB * C::kBTileBytes;                                // nA stages of a_stage_bytes (1024-aligned)
  unsigned char* sG = sA + nA * a_stage_bytes;                                 // backward: one stage of gradient pieces
  unsigned char* sE = sG + (kBwd ? a_stage_bytes : 0);                         // kGatherBwdRep: replicas 2..4, one 128-byte row each
  unsigned char* s_tab = sE + e_bytes;                                         // gather tables
  float* s_const = reinterpret_cast<float*>(s_tab + tab_bytes);                // fwd: scale, shift [CIN]; bwd: + P, Q, R

  const int warp = threadIdx.x >> 5;
  const int nchunks = CIN / kBlockK;
  const int boxh = kGTileH + 2 * dil;
  const int npix = boxh * boxw;

  if (threadIdx.x == 0) {
    prefetch_tensormap(&tmap_w);
    prefetch_tensormap(&tmap_out);
    if (ADD) prefetch_tensormap(&tmap_add);
    if (ADD == 2) prefetch_tensormap(&tmap_rkw);
    for (int i = 0; i < nA; ++i) { mbar_init(&full_a[i], kProducers); mbar_init(&empty_a[i], 1); }
    for (int i = 0; i < nB; ++i) { mbar_init(&full_b[i], 1); mbar_init(&empty_b[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4); mbar_init(&add_full[i], 1); }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc<kTmemCols>(tmem_ptr);
    tmem_relinquish();
  }
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_sync();                                 // set-up above overlaps the previous kernel's tail

  if (warp == 0) {
    // ===================== weight TMA producer (whole warp walks, one elected lane issues) =====================
    int bs = 0; uint32_t bph = 0;
    for (int t0 = blockIdx.x; t0 < num_tiles; t0 += gridDim.x) {
      for (int kc = 0; kc < nchunks; ++kc) {
        for (int tap = 0; tap < 9; ++tap) {
          mbar_wait(&empty_b[bs], bph ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&full_b[bs], C::kBTileBytes);
            tma_load_2d(sB + bs * C::kBTileBytes, &tmap_w, &full_b[bs], kc * kBlockK, tap * COUT);
          }
          __syncwarp();
          if (++bs == nB) { bs = 0; bph ^= 1; }
        }
      }
      if constexpr (ADD == 2) {                  // the rank-K block's operands: the tile of G, then W2T
        const int t = rev ? num_tiles - 1 - t0 : t0;
        const int tw = t % tiles_w, th = (t / tiles_w) % tiles_h, n = t / (tiles_w * tiles_h);
        mbar_wait(&empty_b[bs], bph ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&full_b[bs], (uint32_t)(kGTileH * kGSubW * MT * 128));
          tma_load_4d(sB + bs * C::kBTileBytes, &tmap_add, &full_b[bs], 0, tw * kGSubW * MT, th * kGTileH, n);
        }
        __syncwarp();
        if (++bs == nB) { bs = 0; bph ^= 1; }
        mbar_wait(&empty_b[bs], bph ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&full_b[bs], C::kBTileBytes);
          tma_load_2d(sB + bs * C::kBTileBytes, &tmap_rkw, &full_b[bs], 0, 0);
        }
        __syncwarp();
        if (++bs == nB) { bs = 0; bph ^= 1; }
      }
    }
    pdl_trigger();
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp walks with warp-uniform values, one elected lane issues) ==========
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(COUT >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB);
    // K-major, 128-byte swizzle, eight-row groups one box row apart (descriptor fields: LBO = 1, SBO, version 1, SW128)
    const uint64_t desc_hi = (1ull << 16) | ((uint64_t)((uint32_t)boxw * 8u) << 32) | (1ull << 46) | (2ull << 61);
    int as = 0, bs = 0; uint32_t aph = 0, bph = 0;
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int acc = it & 1;
      mbar_wait(&tmem_empty[acc], ((it >> 1) & 1) ^ 1);
      tcgen05_after_sync();
      const uint32_t d_tmem = tmem_u + (uint32_t)(acc * MT * COUT);
      for (int kc = 0; kc < nchunks; ++kc) {
        mbar_wait(&full_a[as], aph);
        const uint64_t da_stage = desc_hi | (uint64_t)(((sA_u + (uint32_t)(as * a_stage_bytes)) >> 4) & 0x3FFFu);
#pragma unroll 3
        for (int tap = 0; tap < 9; ++tap) {
          mbar_wait(&full_b[bs], bph);
          tcgen05_after_sync();
          if (elect_one()) {
            // the tap's view starts (ty * d * boxw + tx * d) box pixels into the halo tile; descriptors advance in 16-byte units
            const uint64_t da = da_stage + (uint64_t)(((tap / 3) * dil * boxw + (tap % 3) * dil) * 8);
            const uint64_t db = make_desc_sw128(sB_u + bs * C::kBTileBytes);
#pragma unroll
            for (int k = 0; k < 4; ++k)
#pragma unroll
              for (int mt = 0; mt < MT; ++mt)
                umma<T>(d_tmem + (uint32_t)(mt * COUT), da + (uint64_t)(mt * kGSubW * 8 + k * 2), db + (uint64_t)(k * 2), idesc,
                        (kc | tap | k) != 0);
            umma_commit(&empty_b[bs]);
            if (tap == 8) umma_commit(&empty_a[as]);     // the halo tile is free once all 9 taps have read it
          }
          __syncwarp();
          if (++bs == nB) { bs = 0; bph ^= 1; }
        }
        if (++as == nA) { as = 0; aph ^= 1; }
      }
      if constexpr (ADD == 2) {                  // + G[pixel][class] . W2T[cout][class]^T: two k-steps cover the <= 24 classes
        static_assert(MT == 1, "the rank-K block is laid out for one M sub-tile");
        const int gs = bs;
        mbar_wait(&full_b[bs], bph);
        if (++bs == nB) { bs = 0; bph ^= 1; }
        const int ws_ = bs;
        mbar_wait(&full_b[bs], bph);
        if (++bs == nB) { bs = 0; bph ^= 1; }
        tcgen05_after_sync();
        if (elect_one()) {
          // G tile as TMA wrote it: [16 rows][8 px][128 B], i.e. eight-pixel groups 1024 bytes apart (SBO = 64 x 16 bytes)
          const uint64_t dg = (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61) |
                              (uint64_t)(((sB_u + (uint32_t)(gs * C::kBTileBytes)) >> 4) & 0x3FFFu);
          const uint64_t dw = make_desc_sw128(sB_u + ws_ * C::kBTileBytes);
#pragma unroll
          for (int k = 0; k < 2; ++k) umma<T>(d_tmem, dg + (uint64_t)(k * 2), dw + (uint64_t)(k * 2), idesc, true);
          umma_commit(&empty_b[gs]);
          umma_commit(&empty_b[ws_]);
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(&tmem_full[acc]);     // accumulator complete
      __syncwarp();
    }
  } else if (warp < 6) {
    // ===================== epilogue (warps 2..5): conv_common.cuh =====================
    EpiSmem es;
    es.sOut = sOut; es.s_wgt = s_wgt; es.scratch = reinterpret_cast<float*>(sA); es.tmem_full = tmem_full; es.tmem_empty = tmem_empty;
    es.add_full = add_full;
    conv_epilogue<COUT, T, kGTileH, kGSubW, MT, true, ADD == 1 ? 3 : 0>(es, tmem_base, tmap_out, tiles_h, tiles_w, num_tiles, cnt_h, cnt_w,
                                                                   stat_acc, rev, fin, add_src, H, W, &tmap_add);
  } else {
    // ===================== operand producers (warps 6..13) =====================
    const int pt = threadIdx.x - 192;            // 0..255
    const int piece = pt & 7;                    // 16-byte piece (8 channels) of a pixel's 128-byte chunk
    const int pl = pt >> 3;                      // pixel lane: box pixels pl, pl + 32, ...
    const uint32_t tab_u = smem_u32(s_tab), sA_u = smem_u32(sA), sG_u = smem_u32(sG), sE_u = smem_u32(sE), const_u = smem_u32(s_const);
    {
      for (int j = pt; j < CIN; j += kProducers) {
        s_const[j] = ga.stats[2 * kMaxC + j]; s_const[CIN + j] = ga.stats[3 * kMaxC + j];
        if constexpr (kBwd) {                    // BN-backward constants from the reduced sums (as bn_bwd_apply, hrfp.cu)
          const double mean = ga.stats[j], invstd = ga.stats[kMaxC + j], gm = j < ga.c_real ? ga.gamma[j] : 0.f;
          const double S1 = ga.acc[j], S2 = invstd * (ga.acc[kMaxC + j] - mean * S1);
          const double M1 = gm * S1 / ga.count, M2 = gm * S2 / ga.count;
          const double r = invstd * invstd * M2;
          s_const[2 * CIN + j] = (float)(invstd * gm); s_const[3 * CIN + j] = (float)(invstd * M1 - mean * r);
          s_const[4 * CIN + j] = (float)r;
        }
      }
    }
    // gather table of a tile (shared by its channel chunks): source pixel of each box pixel, -1 where the operand is zero
    // (the convolution's padding; backward: also a pixel without replica); nT buffers, because the copies run up to
    // nA - 1 chunks — possibly tiles — ahead of the transform
    constexpr int kEnt = MODE == kGatherFwd ? 4 : (MODE == kGatherBwd ? 8 : 16);       // bytes per table entry
    const int nT = kBwd ? 1 : nA;
    const int tab_stride = tab_bytes / nT;
    auto build_table = [&](int seq) {
      const int t0 = blockIdx.x + seq * gridDim.x;
      const int t = rev ? num_tiles - 1 - t0 : t0;
      const int tw = t % tiles_w, th = (t / tiles_w) % tiles_h, n = t / (tiles_w * tiles_h);
      const int h0 = th * kGTileH - dil, w0 = tw * kGSubW * MT - dil;      // image coordinates of box pixel (0, 0)
      const uint32_t tab = tab_u + (uint32_t)((seq % nT) * tab_stride);
      prod_bar_sync();                           // every producer is done with the tile that owned this buffer (first: the constants)
      if constexpr (MODE == kGatherBwdRep) {
        // entry = (y pixel | -1, first replica's pixel in g, slot of the other replicas in the extras stage, nh | nw << 8);
        // the slots are an exclusive prefix sum of (nh * nw - 1) over the box pixels: warp scans + warp totals in shared memory
        const uint32_t scan_u = tab + 16u * (uint32_t)npix;                 // [8] warp totals
        const int lane_ = pt & 31, wid = pt >> 5;
        int carry = 0;
        for (int base = 0; base < npix; base += kProducers) {
          const int p = base + pt;
          int oy = -1, og = 0, nh = 0, nw = 0;
          if (p < npix) {
            const int row = p / boxw, col = p - row * boxw;
            const int h = h0 + row, w = w0 + col;
            if ((unsigned)h < (unsigned)H && (unsigned)w < (unsigned)W) {
              const int dh = ga.tab_h[h], dw = ga.tab_w[w];
              nh = ga.tab_h[h + 1] - dh; nw = ga.tab_w[w + 1] - dw;
              if (nh > 0 && nw > 0) { oy = (n * H + h) * W + w; og = (n * ga.SH + dh) * ga.SW + dw; }
            }
          }
          const int e = oy >= 0 ? nh * nw - 1 : 0;
          int x = e;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, x, o);
            if (lane_ >= o) x += v;
          }
          if (lane_ == 31) sts_u32(scan_u + 4u * (uint32_t)wid, (uint32_t)x);
          prod_bar_sync();
          int before = carry, total = carry;
#pragma unroll
          for (int i = 0; i < kProducers / 32; ++i) {
            const int v = (int)lds_u32(scan_u + 4u * (uint32_t)i);
            if (i < wid) before += v;
            total += v;
          }
          if (p < npix) sts_v4(tab + 16u * (uint32_t)p, (uint32_t)oy, (uint32_t)og, (uint32_t)(before + x - e), (uint32_t)(nh | (nw << 8)));
          carry = total;
          prod_bar_sync();                       // the warp totals are reused by the next pass
        }
      } else {
      for (int p = pt; p < npix; p += kProducers) {
        const int row = p / boxw, col = p - row * boxw;
        const int h = h0 + row, w = w0 + col;
        const bool in = (unsigned)h < (unsigned)H && (unsigned)w < (unsigned)W;
        if constexpr (MODE == kGatherFwd) {
          const int off = in ? (n * ga.SH + ga.tab_h[h]) * ga.SW + ga.tab_w[w] : -1;
          sts_u32(tab + 4u * (uint32_t)p, (uint32_t)off);
        } else {
          int oy = -1, og = 0;
          if (in) {
            const int dh = ga.tab_h[h], dw = ga.tab_w[w];
            if (ga.tab_h[h + 1] > dh && ga.tab_w[w + 1] > dw) { oy = (n * H + h) * W + w; og = (n * ga.SH + dh) * ga.SW + dw; }
          }
          sts_v2(tab + 8u * (uint32_t)p, (uint32_t)oy, (uint32_t)og);
        }
      }
      prod_bar_sync();
      }
    };
    const int my_tiles = (num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int nitems = my_tiles * nchunks;       // an item = one 64-channel chunk of one tile = one halo stage
    constexpr int U = MT == 2 ? 13 : 8;          // box pixels per thread: ceil(20 * 20 / 32), ceil(20 * 12 / 32)
    // a stage is 1024-byte aligned and a thread's pixels are 32 apart: the swizzle phase of its rows is the constant pl & 7
    const uint32_t my_off = (uint32_t)pl * 128u + (uint32_t)((piece ^ (pl & 7)) << 4);
    // backward: the gradient side stage is single, so the copies run one item ahead of the MMAs but never ahead of the transform
    const int LA = kBwd ? 0 : nA - 1;
    int i_item = 0, i_seq = -1, i_kc = 0, i_as = 0; uint32_t i_ph = 0;
    // issues the copies of the next item; returns the mask of this thread's live pixels (bit u: operand not identically zero)
    auto issue_next = [&]() -> uint32_t {
      uint32_t valid = 0;
      if (i_item < nitems) {
        if (i_kc == 0) build_table(++i_seq);
        const uint32_t tab = tab_u + (uint32_t)((i_seq % nT) * tab_stride) + (uint32_t)(kEnt * pl);
        mbar_wait(&empty_a[i_as], i_ph ^ 1);
        const uint32_t dst0 = sA_u + (uint32_t)(i_as * a_stage_bytes) + my_off;
        const int c0 = i_kc * kBlockK + piece * 8;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (pl + kPxLanes * u < npix) {
            const int off = (int)lds_u32(tab + (uint32_t)(kEnt * kPxLanes * u));
            const __nv_bfloat16* src = off >= 0 ? ga.y + (size_t)off * CIN + c0 : ga.y;
            // an identically-zero pixel: source size 0 zero-fills the 16 bytes
            cp_async_cg16_zfill(dst0 + (uint32_t)(kPxLanes * 128 * u), src, off >= 0 ? 16u : 0u);
            if constexpr (kBwd) {
              if (off >= 0) {
                const int og = (int)lds_u32(tab + (uint32_t)(kEnt * kPxLanes * u) + 4u);
                const __nv_bfloat16* gp = ga.g + (size_t)og * CIN + c0;
                cp_async_cg16(sG_u + my_off + (uint32_t)(kPxLanes * 128 * u), gp);
                if constexpr (MODE == kGatherBwdRep) {     // replicas (0,1), (1,0), (1,1) -> consecutive rows of the extras stage
                  const int rep = (int)lds_u32(tab + (uint32_t)(kEnt * kPxLanes * u) + 12u);
                  if (rep != (1 | (1 << 8))) {
                    const int nh = rep & 0xff, nw = rep >> 8;
                    uint32_t ed = sE_u + lds_u32(tab + (uint32_t)(kEnt * kPxLanes * u) + 8u) * 128u + (uint32_t)(piece << 4);
                    if (nw > 1) {
                      cp_async_cg16(ed, gp + CIN);
                      ed += 128u;
                    }
                    if (nh > 1) {
                      cp_async_cg16(ed, gp + (size_t)ga.SW * CIN);
                      if (nw > 1) cp_async_cg16(ed + 128u, gp + (size_t)ga.SW * CIN + CIN);
                    }
                  }
                }
              }
            }
            valid |= (off >= 0 ? 1u : 0u) << u;
          }
        }
        if (++i_kc == nchunks) i_kc = 0;
        if (++i_as == nA) { i_as = 0; i_ph ^= 1; }
        ++i_item;
      }
      cp_async_commit();                         // one group per call, empty or not: uniform accounting
      return valid;
    };
    uint32_t vq0 = 0, vq1 = 0, vq2 = 0;          // live-pixel masks of the items in flight, oldest first
    if (LA >= 1) vq0 = issue_next();
    if (LA >= 2) vq1 = issue_next();
    if (LA >= 3) vq2 = issue_next();
    int j_kc = 0, j_as = 0;
    for (int j = 0; j < nitems; ++j) {
      if (LA == 0) vq0 = issue_next();           // backward: copy, wait, transform — the MMAs of item j - 1 run meanwhile
      // item j is the oldest of the groups in flight
      if (LA <= 1) cp_async_wait<0>();
      else if (LA == 2) cp_async_wait<1>();
      else cp_async_wait<2>();
      const uint32_t dst0 = sA_u + (uint32_t)(j_as * a_stage_bytes) + my_off;
      const uint32_t valid = vq0;
      if constexpr (MODE == kGatherFwd) {
        float sc[8], sh[8];
        ld8s(const_u + 4u * (uint32_t)(j_kc * kBlockK + piece * 8), sc);
        ld8s(const_u + 4u * (uint32_t)(CIN + j_kc * kBlockK + piece * 8), sh);
        uint64_t sc2[4], sh2[4];                   // channel pairs for the packed fp32x2 FMA (common.cuh: bn_relu_x2)
#pragma unroll
        for (int q = 0; q < 4; ++q) { sc2[q] = pack_f32x2(sc[2 * q], sc[2 * q + 1]); sh2[q] = pack_f32x2(sh[2 * q], sh[2 * q + 1]); }
#pragma unroll
        for (int u0 = 0; u0 < U; u0 += 5) {        // up to five pixels per batch: their shared-memory reads overlap
          uint4 v[5];
#pragma unroll
          for (int i = 0; i < 5; ++i) {
            v[i] = make_uint4(0u, 0u, 0u, 0u);
            if (u0 + i < U && pl + kPxLanes * (u0 + i) < npix) v[i] = lds_v4(dst0 + (uint32_t)(kPxLanes * 128 * (u0 + i)));
          }
#pragma unroll
          for (int i = 0; i < 5; ++i) {
            if (u0 + i < U) {
              uint4 o = make_uint4(bn_relu_x2(v[i].x, sc2[0], sh2[0]), bn_relu_x2(v[i].y, sc2[1], sh2[1]),
                                   bn_relu_x2(v[i].z, sc2[2], sh2[2]), bn_relu_x2(v[i].w, sc2[3], sh2[3]));
              if (!((valid >> (u0 + i)) & 1u)) o = make_uint4(0u, 0u, 0u, 0u);   // the convolution's zero padding stays zero
              if (pl + kPxLanes * (u0 + i) < npix) sts_v4(dst0 + (uint32_t)(kPxLanes * 128 * (u0 + i)), o.x, o.y, o.z, o.w);
            }
          }
        }
      } else {
        const uint32_t cb = const_u + 4u * (uint32_t)(j_kc * kBlockK + piece * 8);
        float sc[8], sh[8], cP[8], cQ[8], cR[8];
        ld8s(cb, sc); ld8s(cb + 4u * (uint32_t)CIN, sh); ld8s(cb + 8u * (uint32_t)CIN, cP); ld8s(cb + 12u * (uint32_t)CIN, cQ);
        ld8s(cb + 16u * (uint32_t)CIN, cR);
        const uint32_t g0 = sG_u + my_off;
#pragma unroll
        for (int u0 = 0; u0 < U; u0 += 3) {        // three pixels per batch (six shared-memory reads in flight)
          uint4 vy[3], vg[3];
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            vy[i] = vg[i] = make_uint4(0u, 0u, 0u, 0u);
            if (u0 + i < U && ((valid >> (u0 + i)) & 1u)) {
              vy[i] = lds_v4(dst0 + (uint32_t)(kPxLanes * 128 * (u0 + i)));
              vg[i] = lds_v4(g0 + (uint32_t)(kPxLanes * 128 * (u0 + i)));
            }
          }
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            if (u0 + i < U && ((valid >> (u0 + i)) & 1u)) {      // a dead pixel keeps the zeros its copy filled in
              float y[8], g[8];
              unpack8(vy[i], y); unpack8(vg[i], g);
              float cnt = 1.f;
              if constexpr (MODE == kGatherBwdRep) {             // the other replicas, in the order (0,1), (1,0), (1,1)
                const uint32_t te = tab_u + (uint32_t)(16 * (pl + kPxLanes * (u0 + i)));
                const int rep = (int)lds_u32(te + 12u);
                const int nx = (rep & 0xff) * (rep >> 8) - 1;
                if (nx > 0) {
                  const uint32_t ea = sE_u + lds_u32(te + 8u) * 128u + (uint32_t)(piece << 4);
                  for (int x = 0; x < nx; ++x) {
                    float e8[8];
                    unpack8(lds_v4(ea + 128u * (uint32_t)x), e8);
#pragma unroll
                    for (int q = 0; q < 8; ++q) g[q] += e8[q];
                  }
                  cnt = (float)(nx + 1);
                }
              }
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float t = fmaf(sc[q], y[q], sh[q]) > 0.f ? g[q] : 0.f;
                if constexpr (MODE == kGatherBwdRep) y[q] = cP[q] * t - cnt * fmaf(cR[q], y[q], cQ[q]);
                else y[q] = cP[q] * t - fmaf(cR[q], y[q], cQ[q]);
              }
              const uint4 o = pack8(y);
              sts_v4(dst0 + (uint32_t)(kPxLanes * 128 * (u0 + i)), o.x, o.y, o.z, o.w);
            }
          }
        }
      }
      // generic-proxy writes -> visible to the tensor core's (async-proxy) reads, then one arrival per producer thread
      fence_proxy_async_smem();
      mbar_arrive(&full_a[j_as]);
      if (++j_kc == nchunks) j_kc = 0;
      if (++j_as == nA) j_as = 0;
      if (LA >= 1) {
        vq0 = vq1; vq1 = vq2;
        const uint32_t vn = issue_next();        // item j + LA: its stage is free once the MMAs of item j - 1 have retired
        if (LA == 1) vq0 = vn; else if (LA == 2) vq1 = vn; else vq2 = vn;
      }
    }
  }
  tcgen05_before_sync();
  __syncthreads();
  if (warp == 1) {
    tcgen05_after_sync();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// shared-memory carve-up of one launch: weight ring, halo stages (+ the gradient side stage, + the extras stage), gather
// tables, per-channel constants behind the fixed part.  Forward: as many halo stages as fit (the copies run nA - 1 stages
// ahead), a shallower weight ring if that buys the third stage.  Backward: two halo stages + the side stage(s).
struct SmemPlan { int mt, boxw, a_stage, tab_bytes, e_bytes, nA, nB, smem; };
SmemPlan smem_plan_mt(int mode, int cout, int cin, int dil, int mt, int e_rows) {
  const int b_pref = cout == 256 ? GCfg<256>::kBStages : (cout == 128 ? GCfg<128>::kBStages : GCfg<64>::kBStages);
  const int b_tile = cout * 128;
  SmemPlan p = {};
  p.mt = mt;
  p.boxw = kGSubW * mt + 2 * dil;
  const int npix = p.boxw * (kGTileH + 2 * dil);
  p.a_stage = (int)align_up((size_t)npix * 128, 1024);
  p.e_bytes = mode == kGatherBwdRep ? (int)align_up((size_t)e_rows * 128, 1024) : 0;
  const int ent = mode == kGatherFwd ? 4 : (mode == kGatherBwd ? 8 : 16);
  const int tab1 = (int)align_up((size_t)npix * ent + (mode == kGatherBwdRep ? 64 : 0), 16);
  const int consts = (mode == kGatherFwd ? 2 : 5) * cin * 4;
  const int base = kFixedBytes + consts + 1024 /* alignment slack */;
  auto stages_for = [&](int nb) {                    // halo stages that fit next to nb weight tiles
    const int left = kSmemLimit - base - nb * b_tile - p.e_bytes;
    if (mode != kGatherFwd) return left >= 3 * p.a_stage + tab1 ? 2 : 0;
    int n = left / (p.a_stage + tab1);
    return n > kMaxAStages ? kMaxAStages : n;
  };
  const int want = mode == kGatherFwd ? 3 : 2;
  const int nb_min = mode == kGatherFwd ? 4 : 3;      // forward: a third halo stage is not worth a weight ring below 4 (measured
                                                        // on the 256-wide stage: 2 stages + 4 tiles 345 us, 3 + 3 373 us)
  p.nB = b_pref;
  p.nA = stages_for(p.nB);
  for (int nb = b_pref - 1; nb >= nb_min && p.nA < want; --nb) // the deepest weight ring that still leaves the wanted stages
    if (stages_for(nb) > p.nA) { p.nB = nb; p.nA = stages_for(nb); }
  if (p.nA < 2) { p.nA = 0; return p; }
  p.tab_bytes = (mode == kGatherFwd ? p.nA : 1) * tab1;
  p.smem = base + p.nB * b_tile + (p.nA + (mode == kGatherFwd ? 0 : 1)) * p.a_stage + p.e_bytes + p.tab_bytes;
  return p;
}

// rows of the extras stage a tile can need: max over tiles of sum over live box pixels of (nh * nw - 1) — separable in the
// row / column replica counts (lo tables on the host: first replica of each source row / column)
int extras_rows(const int* lo_h, const int* lo_w, int H, int W, int dil, int mt) {
  const int boxh = kGTileH + 2 * dil, boxw = kGSubW * mt + 2 * dil, tile_w = kGSubW * mt;
  auto axis = [&](const int* lo, int size, int tile, int box, std::vector<std::pair<int, int>>& out) {
    for (int t0 = 0; t0 < size; t0 += tile) {
      int reps = 0, live = 0;
      for (int i = t0 - dil; i < t0 - dil + box; ++i)
        if (i >= 0 && i < size) { const int c = lo[i + 1] - lo[i]; reps += c; live += c > 0; }
      out.emplace_back(reps, live);
    }
  };
  std::vector<std::pair<int, int>> rh, rw;
  axis(lo_h, H, kGTileH, boxh, rh);
  axis(lo_w, W, tile_w, boxw, rw);
  int best = 0;
  for (const auto& a : rh)
    for (const auto& b : rw) best = std::max(best, a.first * b.first - a.second * b.second);
  return best;
}

// the plan of a launch.  The replica form needs 3 + ~0.7 halo-stage equivalents of staging: it fits for the 64-wide
// dilation-1 stages; on the smaller 16 x 8 tile it would fit everywhere, but there the copies — which cannot run ahead of the
// transform for lack of a second side stage — leave the 128-wide dgrad 4x producer-bound (measured 918 us against 371 + 291 us
// for the separate pass + tap kernel), so that fallback is not taken.
SmemPlan smem_plan(int mode, int cout, int cin, int dil, const int* host_lo_h = nullptr, const int* host_lo_w = nullptr, int H = 0,
                   int W = 0) {
  const int mt0 = cout == 256 ? 1 : 2;
  if (mode != kGatherBwdRep) return smem_plan_mt(mode, cout, cin, dil, mt0, 0);
  if (!host_lo_h || !host_lo_w || cout == 256) return SmemPlan{};
  return smem_plan_mt(mode, cout, cin, dil, mt0, extras_rows(host_lo_h, host_lo_w, H, W, dil, mt0));
}

template <int COUT, int MODE, int ADD, int MT>
int launch(const SmemPlan& sp, const GatherArgs& ga, const void* wpack, void* out, int N, int H, int W, int cin, int dil,
           const int* cnt_h, const int* cnt_w, double* stat_acc, int rev, const ConvBnFinalize& fin, const void* add_src,
           const void* rk_w2t, ConvMaps* cache, cudaStream_t stream) {
  ConvMaps local;
  local.valid = 0;
  ConvMaps* m = cache ? cache : &local;
  if (!m->valid || m->key[0] != add_src || m->key[1] != wpack || m->key[2] != out || m->key_aux != rk_w2t) {
    m->valid = 0;
    {
      const cuuint64_t dims[2] = {(cuuint64_t)cin, (cuuint64_t)9 * COUT};
      const cuuint64_t strides[1] = {(cuuint64_t)cin * 2};
      const cuuint32_t box[2] = {64, COUT};
      int rc = conv_make_map(&m->w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, wpack, 2, dims, strides, box);
      if (rc) return rc;
    }
    {
      const cuuint64_t dims[4] = {(cuuint64_t)COUT, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
      const cuuint64_t strides[3] = {(cuuint64_t)COUT * 2, (cuuint64_t)W * COUT * 2, (cuuint64_t)H * W * COUT * 2};
      const cuuint32_t box[4] = {64, kGSubW, kGTileH, 1};
      int rc = conv_make_map(&m->out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, out, 4, dims, strides, box);
      if (rc) return rc;
    }
    if (ADD == 2) {      // rank-K term: add_src is G (N, H, W, 64) bf16, rk_w2t is W2T (COUT, 64) bf16
      const cuuint64_t dims[4] = {64, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
      const cuuint64_t strides[3] = {128, (cuuint64_t)W * 128, (cuuint64_t)H * W * 128};
      const cuuint32_t box[4] = {64, (cuuint32_t)(kGSubW * MT), kGTileH, 1};
      int rc = conv_make_map(&m->in, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, add_src, 4, dims, strides, box);
      if (rc) return rc;
      const cuuint64_t dims2[2] = {64, (cuuint64_t)COUT};
      const cuuint64_t strides2[1] = {128};
      const cuuint32_t box2[2] = {64, COUT};
      rc = conv_make_map(&m->aux, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rk_w2t, 2, dims2, strides2, box2);
      if (rc) return rc;
    } else if (add_src) {       // the tile of add_src that an output chunk is summed with: same geometry as the output (kept in m->in)
      const cuuint64_t dims[4] = {(cuuint64_t)COUT, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
      const cuuint64_t strides[3] = {(cuuint64_t)COUT * 2, (cuuint64_t)W * COUT * 2, (cuuint64_t)H * W * COUT * 2};
      const cuuint32_t box[4] = {64, kGSubW, kGTileH, 1};
      int rc = conv_make_map(&m->in, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, add_src, 4, dims, strides, box);
      if (rc) return rc;
    } else {
      m->in = m->out;
    }
    if (ADD != 2) m->aux = m->w;
    m->key[0] = add_src; m->key[1] = wpack; m->key[2] = out; m->key_aux = rk_w2t;
    m->valid = 1;
  }
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const int tile_w = kGSubW * MT;
  const int tiles_h = (H + kGTileH - 1) / kGTileH, tiles_w = (W + tile_w - 1) / tile_w;
  const int num_tiles = N * tiles_h * tiles_w;
  const int grid = num_tiles < di.sm_count ? num_tiles : di.sm_count;
  auto kern = conv3x3_gather_kernel<COUT, MODE, ADD, MT>;
  MRFP_SMEM_OPT_IN(kern, kSmemLimit, di.device);
  launch_k(kern, dim3(grid), dim3(kGThreads), (size_t)sp.smem, stream, m->w, m->out, m->in, m->aux, ga, cin, dil, sp.boxw, tiles_h, tiles_w,
           num_tiles, cnt_h, cnt_w, stat_acc, rev, fin, static_cast<const __nv_bfloat16*>(ADD == 1 ? add_src : nullptr), H, W, sp.nA, sp.nB, sp.a_stage,
           sp.tab_bytes, sp.e_bytes);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

template <int MODE, int ADD>
int dispatch(const SmemPlan& sp, const GatherArgs& ga, const void* wpack, void* out, int N, int H, int W, int cin, int cout, int dil,
             const int* cnt_h, const int* cnt_w, double* stat_acc, int rev, const ConvBnFinalize& fin, const void* add_src,
             const void* rk_w2t, ConvMaps* cache, cudaStream_t stream) {
  if (sp.nA < 2) return MRFP_ERR_UNSUPPORTED;
#define MRFP_GATHER_CASE(CO, MTV) \
  return launch<CO, MODE, ADD, MTV>(sp, ga, wpack, out, N, H, W, cin, dil, cnt_h, cnt_w, stat_acc, rev, fin, add_src, rk_w2t, cache, stream)
  if (cout == 256 && sp.mt == 1) { if constexpr (MODE != kGatherBwdRep) MRFP_GATHER_CASE(256, 1); }
  if constexpr (ADD != 2) {
  if (cout == 128 && sp.mt == 2) MRFP_GATHER_CASE(128, 2);
  if (cout == 64 && sp.mt == 2) MRFP_GATHER_CASE(64, 2);
  }
#undef MRFP_GATHER_CASE
  return MRFP_ERR_UNSUPPORTED;
}

bool supported(int mode, int N, int H, int W, int SH, int SW, int cin, int cout, int dil, const int* host_lo_h = nullptr,
               const int* host_lo_w = nullptr) {
  if (cin % 64 != 0 || cin > kMaxC || (cout != 64 && cout != 128 && cout != 256)) return false;
  if (dil != 1 && dil != 2) return false;
  if (smem_plan(mode, cout, cin, dil, host_lo_h, host_lo_w, H, W).nA < 2) return false;
  // pixel indices are kept as 32-bit ints in the gather table
  return (long long)N * H * W < (1ll << 31) && (long long)N * SH * SW < (1ll << 31);
}

}  // namespace

bool conv3x3_gather_supported(int mode, int N, int H, int W, int SH, int SW, int cin, int cout, int dil, const int* host_lo_h,
                              const int* host_lo_w) {
  return supported(mode, N, H, W, SH, SW, cin, cout, dil, host_lo_h, host_lo_w);
}

int conv3x3_gather_fwd(const void* y_prev, int SH, int SW, const int* idx_h, const int* idx_w, const float* stats_prev,
                       const void* wpack, void* out, int N, int H, int W, int cin, int cout, int dil, const int* cnt_h,
                       const int* cnt_w, double* stat_acc, cudaStream_t stream, bool reverse_tiles,
                       const ConvBnFinalize* finalize, ConvMaps* cache) {
  if (!supported(kGatherFwd, N, H, W, SH, SW, cin, cout, dil)) return MRFP_ERR_UNSUPPORTED;
  if (((uintptr_t)y_prev | (uintptr_t)wpack | (uintptr_t)out) & 15) return MRFP_ERR_WORKSPACE;
  ConvBnFinalize fin = {};
  if (finalize) {
    if (!stat_acc || !finalize->gamma || !finalize->stats || !finalize->counter) return MRFP_ERR_NULL_POINTER;
    fin = *finalize;
    if (fin.cout_real <= 0 || fin.cout_real > cout) fin.cout_real = cout;
  }
  GatherArgs ga = {};
  ga.y = static_cast<const __nv_bfloat16*>(y_prev);
  ga.tab_h = idx_h; ga.tab_w = idx_w; ga.stats = stats_prev; ga.SH = SH; ga.SW = SW;
  return dispatch<kGatherFwd, 0>(smem_plan(kGatherFwd, cout, cin, dil), ga, wpack, out, N, H, W, cin, cout, dil, cnt_h, cnt_w,
                                 stat_acc, reverse_tiles ? 1 : 0, fin, nullptr, nullptr, cache, stream);
}

int conv3x3_gather_bwd(const void* y, const void* dA, int OH, int OW, const int* lo_h, const int* lo_w, const int* host_lo_h,
                       const int* host_lo_w, int max_rep, const float* stats, const float* gamma, const double* acc, double count,
                       int c_real, const void* wpack, void* out, int N, int H, int W, int cin, int cout, int dil,
                       cudaStream_t stream, bool reverse_tiles, const void* add_src, ConvMaps* cache, const void* rk_w2t) {
  // rk_w2t != nullptr: add_src is the rank-K operand G (N, H, W, 64) and rk_w2t the matrix W2T (cout, 64), see the kernel
  const int mode = max_rep <= 1 ? kGatherBwd : kGatherBwdRep;
  if (max_rep > 2 || (mode == kGatherBwdRep && add_src)) return MRFP_ERR_UNSUPPORTED;
  if (rk_w2t && (!add_src || cout != 256 || ((uintptr_t)rk_w2t & 15))) return MRFP_ERR_UNSUPPORTED;
  if (!supported(mode, N, H, W, OH, OW, cin, cout, dil, host_lo_h, host_lo_w)) return MRFP_ERR_UNSUPPORTED;
  if (((uintptr_t)y | (uintptr_t)dA | (uintptr_t)wpack | (uintptr_t)out | (uintptr_t)add_src) & 15) return MRFP_ERR_WORKSPACE;
  GatherArgs ga = {};
  ga.y = static_cast<const __nv_bfloat16*>(y); ga.g = static_cast<const __nv_bfloat16*>(dA);
  ga.tab_h = lo_h; ga.tab_w = lo_w; ga.stats = stats; ga.gamma = gamma; ga.acc = acc; ga.count = count;
  ga.SH = OH; ga.SW = OW; ga.c_real = c_real;
  const ConvBnFinalize fin = {};
  const int rev = reverse_tiles ? 1 : 0;
  const SmemPlan sp = smem_plan(mode, cout, cin, dil, host_lo_h, host_lo_w, H, W);
  if (mode == kGatherBwdRep)
    return dispatch<kGatherBwdRep, 0>(sp, ga, wpack, out, N, H, W, cin, cout, dil, nullptr, nullptr, nullptr, rev, fin, nullptr, nullptr, cache, stream);
  if (rk_w2t)
    return dispatch<kGatherBwd, 2>(sp, ga, wpack, out, N, H, W, cin, cout, dil, nullptr, nullptr, nullptr, rev, fin, add_src, rk_w2t, cache, stream);
  if (add_src)
    return dispatch<kGatherBwd, 1>(sp, ga, wpack, out, N, H, W, cin, cout, dil, nullptr, nullptr, nullptr, rev, fin, add_src, nullptr, cache, stream);
  return dispatch<kGatherBwd, 0>(sp, ga, wpack, out, N, H, W, cin, cout, dil, nullptr, nullptr, nullptr, rev, fin, nullptr, nullptr, cache, stream);
}

}  // namespace mrfp

// test hook (host only, no device call): the shared-memory plan of a launch — out[0..5] = M sub-tiles, halo stages (0: the
// kernel refuses this geometry), weight-ring slots, dynamic shared memory bytes, bytes of the extras stage, box width
extern "C" int mrfp_debug_gather_plan(int mode, int cout, int cin, int dil, const int* host_lo_h, const int* host_lo_w, int H, int W,
                                      int* out6) {
  if (!out6 || mode < 0 || mode > 2) return MRFP_ERR_NULL_POINTER;
  const mrfp::SmemPlan p = mrfp::smem_plan(mode, cout, cin, dil, host_lo_h, host_lo_w, H, W);
  out6[0] = p.mt; out6[1] = p.nA; out6[2] = p.nB; out6[3] = p.smem; out6[4] = p.e_bytes; out6[5] = p.boxw;
  return MRFP_OK;
}

// test / bench hooks (not part of the public header): single convolutions on caller-provided buffers — the same kernels
// the chain launches
extern "C" int mrfp_debug_conv3x3_gather_fwd(const void* y_prev, int SH, int SW, const int* idx_h, const int* idx_w,
                                             const float* stats_prev, const void* wpack, void* out, int N, int H, int W, int cin,
                                             int cout, int dil, const int* cnt_h, const int* cnt_w, double* stat_acc, void* stream) {
  return mrfp::conv3x3_gather_fwd(y_prev, SH, SW, idx_h, idx_w, stats_prev, wpack, out, N, H, W, cin, cout, dil, cnt_h, cnt_w,
                                  stat_acc, (cudaStream_t)stream, false, nullptr, nullptr);
}
extern "C" int mrfp_debug_conv3x3_gather_bwd(const void* y, const void* dA, int OH, int OW, const int* lo_h, const int* lo_w,
                                             const int* host_lo_h, const int* host_lo_w, int max_rep, const float* stats,
                                             const float* gamma, const double* acc, double count, const void* wpack, void* out, int N,
                                             int H, int W, int cin, int cout, int dil, const void* add_src, void* stream) {
  return mrfp::conv3x3_gather_bwd(y, dA, OH, OW, lo_h, lo_w, host_lo_h, host_lo_w, max_rep, stats, gamma, acc, count, cin, wpack, out, N,
                                  H, W, cin, cout, dil, (cudaStream_t)stream, false, add_src, nullptr, nullptr);
}
// ... the stage-4 form with the rank-K term: g64 (N, H, W, 64) bf16 and w2t (cout, 64) bf16, of which columns 0..31 enter the
// product (see conv3x3_gather_kernel, ADD == 2)
extern "C" int mrfp_debug_conv3x3_gather_bwd_rk(const void* y, const void* dA, int OH, int OW, const int* lo_h, const int* lo_w,
                                                const int* host_lo_h, const int* host_lo_w, const float* stats, const float* gamma,
                                                const double* acc, double count, const void* wpack, void* out, int N, int H, int W,
                                                int cin, int cout, int dil, const void* g64, const void* w2t, void* stream) {
  return mrfp::conv3x3_gather_bwd(y, dA, OH, OW, lo_h, lo_w, host_lo_h, host_lo_w, 1, stats, gamma, acc, count, cin, wpack, out, N, H, W,
                                  cin, cout, dil, (cudaStream_t)stream, false, g64, nullptr, w2t);
}
