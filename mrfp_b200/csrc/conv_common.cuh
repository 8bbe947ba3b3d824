// Pieces shared by the two tcgen05 convolution kernels of the HRFP chain (conv_tc.cu: one TMA box per tap;
// conv_gather.cu: operand halo tile built by producer warps from the previous stage's conv output): element traits, PTX
// wrappers, and the epilogue (TMEM -> swizzled staging tile -> TMA store, BN batch statistics of the stored tile, BN
// finalisation by the last CTA).
#pragma once
#include "hrfp.cuh"
#include "ptx.cuh"

namespace mrfp {
namespace convk {

constexpr int kATileBytes = 128 * 128;          // 128 pixels x 128 B (64 bf16 / 32 fp32 channels)
constexpr int kStageOutBytes = 128 * 128;       // 128 pixels x 128 B

template <typename T> struct Elem;
template <> struct Elem<__nv_bfloat16> {
  static constexpr int kBlockK = 64;            // channels per k-step = 128 bytes = one swizzle row
  static constexpr uint32_t kFmt = 1;           // UMMA instruction-descriptor operand format: BF16
  static constexpr CUtensorMapDataType kLoadType = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  static constexpr CUtensorMapDataType kStoreType = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
};
template <> struct Elem<float> {
  static constexpr int kBlockK = 32;
  static constexpr uint32_t kFmt = 2;           // TF32
  static constexpr CUtensorMapDataType kLoadType = CU_TENSOR_MAP_DATA_TYPE_TFLOAT32;   // fp32 in HBM, tf32 on the way in
  static constexpr CUtensorMapDataType kStoreType = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
};

__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
               ::"r"(ptx::smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(ptx::smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(ptx::smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(ptx::smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(ptx::smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(ptx::smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T with fp32 accumulation, issued by one thread for the CTA
template <typename T>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  if constexpr (sizeof(T) == 2) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
  }
}
// K-major, 128-byte swizzle, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor, version 1)
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  ptx::tcgen05_wait_ld();
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

// Geometry of a CTA tile: MT sub-tiles of TH x TW = 128 output pixels (one TMEM lane per pixel), stacked vertically
// (HMT = false, the tap kernel) or side by side (HMT = true, the gather kernel).
template <int TH, int TW, int MT, bool HMT> struct TileGeom {
  __device__ static __forceinline__ int h0(int th) { return th * TH * (HMT ? 1 : MT); }
  __device__ static __forceinline__ int w0(int tw) { return tw * TW * (HMT ? MT : 1); }
  __device__ static __forceinline__ int dh(int mt) { return HMT ? 0 : mt * TH; }
  __device__ static __forceinline__ int dw(int mt) { return HMT ? mt * TW : 0; }
};

struct EpiSmem {
  uint64_t* add_full;         // [2] (ADD == 3 only, initialised with count 1): the add tile has landed in staging buffer b
  unsigned char* sOut;        // 2 staging tiles of kStageOutBytes, 1024-byte aligned
  float* s_wgt;               // [128]
  float* scratch;             // >= 8 * COUT floats, idle once every MMA of the CTA has retired (the operand ring)
  uint64_t* tmem_full;        // [2]
  uint64_t* tmem_empty;       // [2]
};

// Runs on warps 2..5 of the CTA (128 threads).  The tile walk (blockIdx.x, += gridDim.x, optional reversal) must match the
// producer and MMA warps of the calling kernel.  ADD: 0 compiles the add_src path out; 1 fetches a chunk's 128 bytes of add_src
// one chunk ahead into a second register set (64 registers); 2 keeps one set and fetches behind the chunk's packing (32);
// 3 brings the chunk's add tile by TMA into the very staging buffer the result will be packed into, one chunk ahead (no
// registers, no exposed latency): each thread reads the 128 bytes of its own row and overwrites them with the sum.  (Mode 3
// is for launches without BN statistics — the dgrads: the statistics loop of chunk i would still be reading the buffer that
// the leader refills for chunk i + 1.)
template <int COUT, typename T, int TH, int TW, int MT, bool HMT, int ADD>
__device__ __forceinline__ void conv_epilogue(const EpiSmem& sm, uint32_t tmem_base, const CUtensorMap& tmap_out, int tiles_h,
                                              int tiles_w, int num_tiles, const int* __restrict__ cnt_h,
                                              const int* __restrict__ cnt_w, double* __restrict__ stat_acc, int rev,
                                              const ConvBnFinalize& fin, const T* __restrict__ add_src, int H, int W,
                                              const CUtensorMap* tmap_add = nullptr) {
  using E = Elem<T>;
  using G = TileGeom<TH, TW, MT, HMT>;
  constexpr int kChunkC = 128 / (int)sizeof(T);                // channels of one 128-byte output chunk
  constexpr int kChunks = COUT / kChunkC;                      // chunks per M sub-tile
  constexpr bool kBf16 = sizeof(T) == 2;
  unsigned char* const sOut = sm.sOut;
  float* const s_wgt = sm.s_wgt;
  const uint32_t s_wgt_u = ptx::smem_u32(sm.s_wgt);
  uint64_t* const tmem_full = sm.tmem_full;
  uint64_t* const tmem_empty = sm.tmem_empty;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  (void)E::kFmt;
  // ===================== epilogue (warps 2..5) =====================
  const int q = warp & 3;                     // TMEM lane quarter this warp may access
  const int r = q * 32 + lane;                // accumulator row = pixel inside the tile
  const int hl = r / TW, wl = r % TW;
  const int et = threadIdx.x - 64;            // 0..127 (the epilogue warps are warps 2..5 of the CTA)
  const bool leader = et == 0;                // first epilogue thread issues the TMA stores
  // statistics: thread (word cp of a 128-byte row, row group pg) sums 32 rows of the staging tile (the values that are
  // stored and later normalised), weighted by the replication count of each row's pixel; a word is a channel pair
  // (bf16) or one channel (fp32)
  const int cp = et & 31, pg = et >> 5;
  float a1x[kChunks], a1y[kChunks], a2x[kChunks], a2y[kChunks];      // per 128-byte chunk of the output row (static indices)
#pragma unroll
  for (int j = 0; j < kChunks; ++j) a1x[j] = a1y[j] = a2x[j] = a2y[j] = 0.f;
  // add_src: this thread's 128 bytes of its pixel, fetched ONE CHUNK AHEAD so the loads overlap the previous chunk
  uint4 ad_nxt[8], ad_cur[8];
  uint4 (&ad_use)[8] = *(ADD == 2 ? &ad_nxt : &ad_cur);
  bool ad_nxt_ok = false, ad_ok = false;
  auto add_fetch = [&](int t0_, int jj_) {
    ad_nxt_ok = false;
    if (!ADD || ADD == 3 || add_src == nullptr || t0_ >= num_tiles) return;
    const int t_ = rev ? num_tiles - 1 - t0_ : t0_;
    const int tw_ = t_ % tiles_w, th_ = (t_ / tiles_w) % tiles_h, n_ = t_ / (tiles_w * tiles_h);
    const int mt_ = jj_ / kChunks, j_ = jj_ % kChunks;
    const int hh = G::h0(th_) + G::dh(mt_) + hl, ww = G::w0(tw_) + G::dw(mt_) + wl;
    if (hh < H && ww < W) {
      const uint4* ap = reinterpret_cast<const uint4*>(add_src + (((size_t)n_ * H + hh) * W + ww) * COUT + j_ * kChunkC);
#pragma unroll
      for (int c = 0; c < 8; ++c) ad_nxt[c] = __ldg(ap + c);
      ad_nxt_ok = true;
    }
  };
  add_fetch(blockIdx.x, 0);
  // ADD == 3: the leader loads chunk (t0_, jj_)'s tile of add_src into staging buffer `buf` (TMA zero-fills beyond the image)
  auto add_issue = [&](int t0_, int jj_, int buf) {
    if (t0_ >= num_tiles) return;
    const int t_ = rev ? num_tiles - 1 - t0_ : t0_;
    const int tw_ = t_ % tiles_w, th_ = (t_ / tiles_w) % tiles_h, n_ = t_ / (tiles_w * tiles_h);
    const int mt_ = jj_ / kChunks, j_ = jj_ % kChunks;
    ptx::mbar_expect_tx(&sm.add_full[buf], kStageOutBytes);
    tma_load_4d(sOut + buf * kStageOutBytes, tmap_add, &sm.add_full[buf], j_ * kChunkC, G::w0(tw_) + G::dw(mt_), G::h0(th_) + G::dh(mt_), n_);
  };
  if (ADD == 3 && leader) add_issue(blockIdx.x, 0, 0);
  int it = 0;
  for (int t0 = blockIdx.x; t0 < num_tiles; t0 += gridDim.x, ++it) {
    const int t = rev ? num_tiles - 1 - t0 : t0;
    const int tw = t % tiles_w, th = (t / tiles_w) % tiles_h, n = t / (tiles_w * tiles_h);
    const int h0 = G::h0(th), w0 = G::w0(tw);
    const int acc = it & 1;
    ptx::mbar_wait(&tmem_full[acc], (it >> 1) & 1);
    ptx::tcgen05_after_sync();
#pragma unroll
    for (int jj = 0; jj < MT * kChunks; ++jj) {
      const int mt = jj / kChunks, j = jj % kChunks;
      if (ADD == 1 && add_src != nullptr) {    // rotate the prefetch: this chunk's data, then start the next chunk's loads
#pragma unroll
        for (int c = 0; c < 8; ++c) ad_cur[c] = ad_nxt[c];
        ad_ok = ad_nxt_ok;
        if (jj + 1 < MT * kChunks) add_fetch(t0, jj + 1); else add_fetch(t0 + gridDim.x, 0);
      }
      if (ADD == 2) ad_ok = ad_nxt_ok;
      const int bsel = (MT * kChunks) % 2 == 0 ? (jj & 1) : ((it * MT * kChunks + jj) & 1);
      unsigned char* ob = sOut + bsel * kStageOutBytes;
      const uint32_t ob_u = ptx::smem_u32(ob);
      if (ADD == 3) {
        // the store of the previous chunk must have read the OTHER buffer before the next chunk's add tile lands in it
        if (leader) {
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          if (jj + 1 < MT * kChunks) add_issue(t0, jj + 1, bsel ^ 1); else add_issue(t0 + gridDim.x, 0, bsel ^ 1);
        }
      } else {
        // the TMA store that last read this staging buffer (two chunks ago) must have drained
        if (leader) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      }
      epi_bar_sync();
      if (stat_acc) ptx::sts_f32(s_wgt_u + 4u * (uint32_t)r, (float)(cnt_h[h0 + G::dh(mt) + hl] * cnt_w[w0 + G::dw(mt) + wl]));   // 0 outside the image (zero-padded tables)
      const uint32_t tcol = (uint32_t)((acc * MT + mt) * COUT + j * kChunkC);
      if constexpr (kBf16) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + tcol + (uint32_t)(half * 32), v);
          if (ADD == 3) {                        // this row's half of the add tile, from the buffer the sum goes back into
            if (half == 0) ptx::mbar_wait(&sm.add_full[bsel], (uint32_t)(((it * MT * kChunks + jj) >> 1) & 1));
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const int chunk = half * 4 + c;
              const uint4 a4 = ptx::lds_v4(ob_u + (uint32_t)(r * 128 + ((chunk ^ (r & 7)) << 4)));
              const uint32_t w4[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                v[c * 8 + 2 * i] = __float_as_uint(__uint_as_float(v[c * 8 + 2 * i]) + __uint_as_float(w4[i] << 16));
                v[c * 8 + 2 * i + 1] = __float_as_uint(__uint_as_float(v[c * 8 + 2 * i + 1]) + __uint_as_float(w4[i] & 0xffff0000u));
              }
            }
          }
          if (ADD != 3 && ad_ok) {               // summed in fp32, rounded once
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint4 a4 = ad_use[half * 4 + c];
              const uint32_t w4[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                v[c * 8 + 2 * i] = __float_as_uint(__uint_as_float(v[c * 8 + 2 * i]) + __uint_as_float(w4[i] << 16));
                v[c * 8 + 2 * i + 1] = __float_as_uint(__uint_as_float(v[c * 8 + 2 * i + 1]) + __uint_as_float(w4[i] & 0xffff0000u));
              }
            }
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) {          // four 16-byte chunks (8 channels each) per half
            uint32_t p[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) p[i] = pack_bf16x2(__uint_as_float(v[c * 8 + 2 * i]), __uint_as_float(v[c * 8 + 2 * i + 1]));
            const int chunk = half * 4 + c;
            ptx::sts_v4(ob_u + (uint32_t)(r * 128 + ((chunk ^ (r & 7)) << 4)), p[0], p[1], p[2], p[3]);
          }
        }
      } else {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + tcol, v);
#pragma unroll
        for (int c = 0; c < 8; ++c) {            // eight 16-byte chunks (4 channels each)
          uint4 o = make_uint4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
          if (ad_ok) {
            const uint4 a4 = ad_use[c];
            o.x = __float_as_uint(__uint_as_float(o.x) + __uint_as_float(a4.x));
            o.y = __float_as_uint(__uint_as_float(o.y) + __uint_as_float(a4.y));
            o.z = __float_as_uint(__uint_as_float(o.z) + __uint_as_float(a4.z));
            o.w = __float_as_uint(__uint_as_float(o.w) + __uint_as_float(a4.w));
          }
          ptx::sts_v4(ob_u + (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)), o.x, o.y, o.z, o.w);
        }
      }
      if (ADD == 2 && add_src != nullptr) {    // the single register set is free again: the next chunk's loads
        if (jj + 1 < MT * kChunks) add_fetch(t0, jj + 1); else add_fetch(t0 + gridDim.x, 0);
      }
      if (jj == MT * kChunks - 1) {       // all TMEM reads of this accumulator are done
        ptx::tcgen05_before_sync();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&tmem_empty[acc]);
      }
      ptx::fence_proxy_async_smem();
      epi_bar_sync();
      if (leader) {
        tma_store_4d(&tmap_out, ob, j * kChunkC, w0 + G::dw(mt), h0 + G::dh(mt), n);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      if (stat_acc) {
        // word cp lives in 16-byte chunk cp/4 of a row, position cp%4; 32 lanes read one whole (swizzled) row
        const uint32_t col = ob_u + (uint32_t)((cp & 3) * 4);
        const int ch = cp >> 2;
        float s1x = 0.f, s1y = 0.f, s2x = 0.f, s2y = 0.f;
#pragma unroll 8
        for (int i = 0; i < 32; ++i) {
          const int row = pg * 32 + i;
          const uint32_t w2 = ptx::lds_u32(col + (uint32_t)(row * 128 + ((ch ^ (row & 7)) << 4)));
          const float wg = ptx::lds_f32(s_wgt_u + 4u * (uint32_t)row);
          if constexpr (kBf16) {
            const float y0 = __uint_as_float(w2 << 16), y1 = __uint_as_float(w2 & 0xffff0000u);
            const float t0 = wg * y0, t1 = wg * y1;
            s1x += t0; s1y += t1;
            s2x = fmaf(t0, y0, s2x); s2y = fmaf(t1, y1, s2y);
          } else {
            const float y0 = __uint_as_float(w2);
            const float t0 = wg * y0;
            s1x += t0;
            s2x = fmaf(t0, y0, s2x);
          }
        }
        a1x[j] += s1x; a2x[j] += s2x;
        if constexpr (kBf16) { a1y[j] += s1y; a2y[j] += s2y; }
      }
    }
  }
  if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  if (stat_acc) {
    // the four row groups meet once per kernel, in the first pipeline slot: every load of this CTA has been consumed and
    // every MMA has retired (the last tmem_full), so the operand ring is idle
    float* part = sm.scratch + pg * 2 * COUT;
#pragma unroll
    for (int j = 0; j < kChunks; ++j) {
      if constexpr (kBf16) {
        part[j * 64 + 2 * cp] = a1x[j]; part[j * 64 + 2 * cp + 1] = a1y[j];
        part[COUT + j * 64 + 2 * cp] = a2x[j]; part[COUT + j * 64 + 2 * cp + 1] = a2y[j];
      } else {
        part[j * 32 + cp] = a1x[j];
        part[COUT + j * 32 + cp] = a2x[j];
      }
    }
    epi_bar_sync();
    const float* all = sm.scratch;
    for (int c = et; c < 2 * COUT; c += 128) {
      const float sum = (all[c] + all[2 * COUT + c]) + (all[4 * COUT + c] + all[6 * COUT + c]);
      atomicAdd(stat_acc + (c < COUT ? c : kMaxC + c - COUT), (double)sum);
    }
  }
  if (stat_acc && fin.stats) {
    // BN finalisation by the last CTA to arrive (its adds and everybody else's are visible behind the fences)
    __threadfence();
    epi_bar_sync();
    if (leader) s_wgt[0] = (atomicAdd(fin.counter, 1u) == gridDim.x - 1) ? 1.f : 0.f;
    epi_bar_sync();
    if (s_wgt[0] != 0.f) {
      __threadfence();
      for (int c = et; c < COUT; c += 128) {
        const double mean = __ldcg(stat_acc + c) / fin.count;
        double var = __ldcg(stat_acc + kMaxC + c) / fin.count - mean * mean;
        if (var < 0) var = 0;
        const double invstd = 1.0 / sqrt(var + (double)fin.eps);
        const bool live = c < fin.cout_real;     // padded output channels (zero weights) are pinned to zero
        const float sc = live ? (float)((double)fin.gamma[c] * invstd) : 0.f;
        const float b = (live && fin.beta) ? fin.beta[c] : 0.f;
        fin.stats[0 * kMaxC + c] = (float)mean;
        fin.stats[1 * kMaxC + c] = (float)invstd;
        fin.stats[2 * kMaxC + c] = sc;
        fin.stats[3 * kMaxC + c] = (float)((double)b - mean * (double)sc);
        if (live && fin.running_mean) fin.running_mean[c] = (1.f - fin.momentum) * fin.running_mean[c] + fin.momentum * (float)mean;
        if (live && fin.running_var)
          fin.running_var[c] = (1.f - fin.momentum) * fin.running_var[c] +
                               fin.momentum * (float)(var * (fin.count / (fin.count - 1.0)));
      }
    }
  }
}

}  // namespace convk
}  // namespace mrfp
