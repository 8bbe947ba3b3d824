// tcgen05 implicit-GEMM 3x3 convolution for the HRFP chain (sm_100a), NHWC operands, fp32 accumulation in TMEM.
// Replaces the cuDNN fprop / dgrad calls behind nn.Conv2d at /root/reference/deepv3.py:320-327.
//
// Two element types share one kernel template:
//   __nv_bfloat16  tcgen05.mma kind::f16  (bf16 x bf16 -> fp32), 64 channels per k-step          (MRFP_MATH_BF16)
//   float          tcgen05.mma kind::tf32 (tf32 x tf32 -> fp32), 32 channels per k-step, fp32 in HBM  (MRFP_MATH_TF32:
//                  the arithmetic of the reference's own cuDNN convolutions under torch's TF32 default)
// In both a k-step is 128 bytes per pixel = one row of the 128-byte swizzle, so the tile geometry is identical.
//
// GEMM view per output tile:  D[128 pixels][COUT] = sum over (tap, channel chunk) A_tap[128][KB] * B_tap[COUT][KB]^T
//   * M tile = 8 rows x 16 cols of output pixels (UMMA M = 128, one TMEM lane per pixel)
//   * A operand: one 4-D TMA box {KB ch, 16, 8, 1} of the NHWC input at the tap's (dy,dx)*dilation offset —
//     TMA zero-fills the halo / out-of-image part, so padding costs nothing and no im2col buffer exists;
//     the box lands in shared memory as 128 rows x 128 B with the 128-byte swizzle = canonical K-major UMMA tile
//   * B operand: 2-D TMA box {KB, COUT} of the tap-major packed weights [9*COUT][CIN]
//   * accumulators: 2 TMEM stages x COUT fp32 columns (epilogue of tile i overlaps the MMAs of tile i+1)
// Warp roles (192 threads, persistent over tiles): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer
// (whole warp walks the loops, one elected lane issues), warps 2-5 = epilogue: tcgen05.ld -> pack into a swizzled
// staging tile -> TMA store (clips the ragged image edge) -> replication-count-weighted per-channel column sums of the
// stored tile (BN batch statistics of the resampled tensor); the last CTA finalises the statistics.
#include "conv_common.cuh"
#include <mutex>

namespace mrfp {
namespace {
using namespace convk;
using namespace ptx;

constexpr int kThreads = 192;

// MT = M sub-tiles (of 128 pixels, stacked vertically) per CTA tile.  With MT = 2 one B (weight) tile feeds two
// MMAs, halving the weight traffic per FLOP: the 64/128-wide layers are bound by the L2->SM operand stream
// (~100 B/clk/SM), not by the tensor pipe.  COUT = 256 already fills TMEM (2 x 256 columns) with MT = 1.
template <int COUT> struct Cfg {
  static constexpr int kMT = COUT == 256 ? 1 : 2;
  static constexpr int kAStageBytes = kMT * kATileBytes;
  static constexpr int kBTileBytes = COUT * 128;
  static constexpr int kStages = 4;
  static constexpr int kOutBufs = 2;                                // staging tiles: chunk i+1 is packed while chunk i drains
  static constexpr int kTmemCols = 2 * kMT * COUT;                  // 256 / 512 / 512: powers of two
  static constexpr int kSmemBytes = kStages * (kAStageBytes + kBTileBytes) + kOutBufs * kStageOutBytes +
                                    512 /* row weights */ + 256 /* barriers */ + 1024 /* alignment slack */;
};

template <int COUT, typename T>
__global__ void __launch_bounds__(kThreads, 1)
conv3x3_tc_kernel(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_w,
                  const __grid_constant__ CUtensorMap tmap_out, int CIN, int dil, int tiles_h, int tiles_w,
                  int num_tiles, const int* __restrict__ cnt_h, const int* __restrict__ cnt_w,
                  double* __restrict__ stat_acc, int rev, const ConvBnFinalize fin, const T* __restrict__ add_src, int H, int W) {
  using C = Cfg<COUT>;
  using E = Elem<T>;
  constexpr int kBlockK = E::kBlockK;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* sA = smem;
  unsigned char* sB = sA + C::kStages * C::kAStageBytes;
  unsigned char* sOut = sB + C::kStages * C::kBTileBytes;
  float* s_wgt = reinterpret_cast<float*>(sOut + C::kOutBufs * kStageOutBytes);   // [128] replication count of each tile row's pixel
  uint64_t* full = reinterpret_cast<uint64_t*>(s_wgt + 128);
  uint64_t* empty = full + C::kStages;
  uint64_t* tmem_full = empty + C::kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int nk = 9 * (CIN / kBlockK);       // k-steps per tile

  if (threadIdx.x == 0) {
    prefetch_tensormap(&tmap_in);
    prefetch_tensormap(&tmap_w);
    prefetch_tensormap(&tmap_out);
    for (int i = 0; i < C::kStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4); }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc<C::kTmemCols>(tmem_ptr);
    tmem_relinquish();
  }
  tcgen05_before_sync();
  __syncthreads();
  tcgen05_after_sync();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_sync();                                 // set-up above overlaps the previous kernel's tail

  if (warp == 0) {
    // ===================== TMA producer (whole warp walks, one elected lane issues) =====================
    int stage = 0; uint32_t phase = 0;
    for (int t0 = blockIdx.x; t0 < num_tiles; t0 += gridDim.x) {
      const int t = rev ? num_tiles - 1 - t0 : t0;     // rev: walk the image from its end (where the producer of `in` finished)
      const int tw = t % tiles_w, th = (t / tiles_w) % tiles_h, n = t / (tiles_w * tiles_h);
      const int h0 = th * kTileH * C::kMT, w0 = tw * kTileW;
      for (int tap = 0; tap < 9; ++tap) {
        const int dy = (tap / 3 - 1) * dil, dx = (tap % 3 - 1) * dil;
        for (int kc = 0; kc < CIN / kBlockK; ++kc) {
          mbar_wait(&empty[stage], phase ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&full[stage], C::kAStageBytes + C::kBTileBytes);
            tma_load_4d(sA + stage * C::kAStageBytes, &tmap_in, &full[stage], kc * kBlockK, w0 + dx, h0 + dy, n);
            tma_load_2d(sB + stage * C::kBTileBytes, &tmap_w, &full[stage], kc * kBlockK, tap * COUT);
          }
          __syncwarp();
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    // all loads of this CTA are in flight: let the next kernel of the stream start its set-up (PDL)
    pdl_trigger();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp walks the loops with warp-uniform values (descriptors stay in uniform registers); one elected
    // lane issues the tcgen05 instructions.
    // instruction descriptor: D=f32, A=B=bf16 / tf32, both K-major, N=COUT, M=128
    constexpr uint32_t idesc = (1u << 4) | (E::kFmt << 7) | (E::kFmt << 10) | ((uint32_t)(COUT >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB);
    int stage = 0; uint32_t phase = 0;
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int acc = it & 1;
      mbar_wait(&tmem_empty[acc], ((it >> 1) & 1) ^ 1);
      tcgen05_after_sync();
      const uint32_t d_tmem = tmem_u + (uint32_t)(acc * C::kMT * COUT);
      for (int ks = 0; ks < nk; ++ks) {
        mbar_wait(&full[stage], phase);
        tcgen05_after_sync();
        if (elect_one()) {
          const uint64_t da = make_desc_sw128(sA_u + stage * C::kAStageBytes);
          const uint64_t db = make_desc_sw128(sB_u + stage * C::kBTileBytes);
#pragma unroll
          for (int k = 0; k < 4; ++k)                  // one UMMA_K = 32 bytes of the swizzle row (16 bf16 / 8 tf32)
#pragma unroll
            for (int mt = 0; mt < C::kMT; ++mt)        // the second M sub-tile is the next 128 rows (16 KiB) of the A box
              umma<T>(d_tmem + (uint32_t)(mt * COUT), da + (uint64_t)(mt * (kATileBytes >> 4) + k * 2),
                      db + (uint64_t)(k * 2), idesc, (ks | k) != 0);
          umma_commit(&empty[stage]);                  // frees the smem slot when the MMAs have read it
        }
        __syncwarp();
        if (++stage == C::kStages) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) umma_commit(&tmem_full[acc]);   // accumulator complete
      __syncwarp();
    }
  } else {
    // ===================== epilogue (warps 2..5): conv_common.cuh =====================
    EpiSmem es;
    es.sOut = sOut; es.s_wgt = s_wgt; es.scratch = reinterpret_cast<float*>(sA); es.tmem_full = tmem_full; es.tmem_empty = tmem_empty;
    conv_epilogue<COUT, T, kTileH, kTileW, C::kMT, false, 1>(es, tmem_base, tmap_out, tiles_h, tiles_w, num_tiles, cnt_h, cnt_w,
                                                                stat_acc, rev, fin, add_src, H, W);
  }
  tcgen05_before_sync();
  __syncthreads();
  if (warp == 1) {
    tcgen05_after_sync();
    tmem_dealloc<C::kTmemCols>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------------
// host side: tensor maps (driver entry point fetched through the runtime; no link against libcuda)
// ------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

int make_map(CUtensorMap* m, CUtensorMapDataType dt, const void* base, int rank, const cuuint64_t* dims,
             const cuuint64_t* strides, const cuuint32_t* box, bool swizzle128 = true) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return MRFP_ERR_DRIVER;
  const cuuint32_t ones[4] = {1, 1, 1, 1};
  CUresult r = fn(m, dt, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, ones, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MRFP_OK : MRFP_ERR_DRIVER;
}

template <int COUT, typename T>
int launch(const T* in, const T* wpack, T* out, int N, int H, int W, int cin, int dil, const int* cnt_h, const int* cnt_w,
           double* stat_acc, int rev, const ConvBnFinalize& fin, const T* add_src, ConvMaps* cache, cudaStream_t stream) {
  using E = Elem<T>;
  constexpr int es = (int)sizeof(T);
  constexpr int kChunkC = 128 / es;
  // the three tensor maps depend on the buffer addresses and the (plan-constant) geometry only: a plan keeps them per
  // (stage, direction) and re-encodes when an address changes (the caching allocator hands the same blocks back)
  ConvMaps local;
  local.valid = 0;
  ConvMaps* m = cache ? cache : &local;
  if (!m->valid || m->key[0] != in || m->key[1] != wpack || m->key[2] != out) {
    m->valid = 0;
    {
      const cuuint64_t dims[4] = {(cuuint64_t)cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
      const cuuint64_t strides[3] = {(cuuint64_t)cin * es, (cuuint64_t)W * cin * es, (cuuint64_t)H * W * cin * es};
      const cuuint32_t box[4] = {(cuuint32_t)E::kBlockK, kTileW, (cuuint32_t)(kTileH * Cfg<COUT>::kMT), 1};
      int rc = make_map(&m->in, E::kLoadType, in, 4, dims, strides, box);
      if (rc) return rc;
    }
    {
      const cuuint64_t dims[2] = {(cuuint64_t)cin, (cuuint64_t)9 * COUT};
      const cuuint64_t strides[1] = {(cuuint64_t)cin * es};
      const cuuint32_t box[2] = {(cuuint32_t)E::kBlockK, COUT};
      int rc = make_map(&m->w, E::kLoadType, wpack, 2, dims, strides, box);
      if (rc) return rc;
    }
    {
      const cuuint64_t dims[4] = {(cuuint64_t)COUT, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
      const cuuint64_t strides[3] = {(cuuint64_t)COUT * es, (cuuint64_t)W * COUT * es, (cuuint64_t)H * W * COUT * es};
      const cuuint32_t box[4] = {(cuuint32_t)kChunkC, kTileW, kTileH, 1};
      int rc = make_map(&m->out, E::kStoreType, out, 4, dims, strides, box);
      if (rc) return rc;
    }
    m->key[0] = in; m->key[1] = wpack; m->key[2] = out;
    m->valid = 1;
  }
  DeviceInfo di;
  int rc = get_device_info(&di);
  if (rc) return rc;
  const int th_px = kTileH * Cfg<COUT>::kMT;
  const int tiles_h = (H + th_px - 1) / th_px, tiles_w = (W + kTileW - 1) / kTileW;
  const int num_tiles = N * tiles_h * tiles_w;
  const int grid = num_tiles < di.sm_count ? num_tiles : di.sm_count;
  auto kern = conv3x3_tc_kernel<COUT, T>;
  MRFP_SMEM_OPT_IN(kern, Cfg<COUT>::kSmemBytes, di.device);
  launch_k(kern, dim3(grid), dim3(kThreads), Cfg<COUT>::kSmemBytes, stream, m->in, m->w, m->out, cin, dil, tiles_h, tiles_w,
           num_tiles, cnt_h, cnt_w, stat_acc, rev, fin, add_src, H, W);
  MRFP_CUDA_TRY(cudaGetLastError());
  return MRFP_OK;
}

template <typename T>
int dispatch(const void* in, const void* wpack, void* out, int N, int H, int W, int cin, int cout, int dil, const int* cnt_h,
             const int* cnt_w, double* stat_acc, int rev, const ConvBnFinalize& fin, const void* add_src, ConvMaps* cache,
             cudaStream_t stream) {
  const T* i = static_cast<const T*>(in); const T* w = static_cast<const T*>(wpack); const T* a = static_cast<const T*>(add_src);
  T* o = static_cast<T*>(out);
  switch (cout) {
    case 64: return launch<64, T>(i, w, o, N, H, W, cin, dil, cnt_h, cnt_w, stat_acc, rev, fin, a, cache, stream);
    case 128: return launch<128, T>(i, w, o, N, H, W, cin, dil, cnt_h, cnt_w, stat_acc, rev, fin, a, cache, stream);
    case 256: return launch<256, T>(i, w, o, N, H, W, cin, dil, cnt_h, cnt_w, stat_acc, rev, fin, a, cache, stream);
  }
  return MRFP_ERR_UNSUPPORTED;
}

}  // namespace

int conv_make_map(CUtensorMap* m, CUtensorMapDataType dt, const void* base, int rank, const cuuint64_t* dims,
                  const cuuint64_t* strides, const cuuint32_t* box, bool swizzle128) {
  return make_map(m, dt, base, rank, dims, strides, box, swizzle128);
}

bool conv3x3_tc_supported(int cin, int cout, int esize) {
  if (esize != 2 && esize != 4) return false;
  const int kb = 128 / esize;
  return cin % kb == 0 && cin <= kMaxC && (cout == 64 || cout == 128 || cout == 256);
}

int conv3x3_tc(const void* in, const void* wpack, void* out, int esize, int N, int H, int W, int cin, int cout, int dil,
               const int* cnt_h, const int* cnt_w, double* stat_acc, cudaStream_t stream, bool reverse_tiles,
               const ConvBnFinalize* finalize, const void* add_src, ConvMaps* cache) {
  ConvBnFinalize fin = {};
  if (finalize) {
    if (!stat_acc || !finalize->gamma || !finalize->stats || !finalize->counter) return MRFP_ERR_NULL_POINTER;
    fin = *finalize;
    if (fin.cout_real <= 0 || fin.cout_real > cout) fin.cout_real = cout;
  }
  const int rev = reverse_tiles ? 1 : 0;
  if (!conv3x3_tc_supported(cin, cout, esize)) return MRFP_ERR_UNSUPPORTED;
  if (((uintptr_t)in | (uintptr_t)wpack | (uintptr_t)out | (uintptr_t)add_src) & 15) return MRFP_ERR_WORKSPACE;
  if (esize == 2)
    return dispatch<__nv_bfloat16>(in, wpack, out, N, H, W, cin, cout, dil, cnt_h, cnt_w, stat_acc, rev, fin, add_src, cache, stream);
  return dispatch<float>(in, wpack, out, N, H, W, cin, cout, dil, cnt_h, cnt_w, stat_acc, rev, fin, add_src, cache, stream);
}

}  // namespace mrfp

// test / bench hooks (not part of the public header): one tcgen05 convolution on caller-provided NHWC buffers —
// the same kernel the chain launches.  bf16: in / wpack / out are bf16; tf32: fp32.
extern "C" int mrfp_debug_conv3x3_bf16(const void* in, const void* wpack, void* out, int N, int H, int W, int cin,
                                       int cout, int dil, const int* cnt_h, const int* cnt_w, double* stat_acc,
                                       void* stream) {
  return mrfp::conv3x3_tc(in, wpack, out, 2, N, H, W, cin, cout, dil, cnt_h, cnt_w, stat_acc, (cudaStream_t)stream, false,
                          nullptr, nullptr, nullptr);
}
extern "C" int mrfp_debug_conv3x3_tf32(const void* in, const void* wpack, void* out, int N, int H, int W, int cin,
                                       int cout, int dil, const int* cnt_h, const int* cnt_w, double* stat_acc,
                                       void* stream) {
  return mrfp::conv3x3_tc(in, wpack, out, 4, N, H, W, cin, cout, dil, cnt_h, cnt_w, stat_acc, (cudaStream_t)stream, false,
                          nullptr, nullptr, nullptr);
}
