/*
 * mrfp_b200.h — C ABI of libmrfp_b200.so: the MRFP training-time hot path (NP+ and HRFP/HRFP+)
 * as hand-written sm_100a CUDA kernels.
 *
 * The reference (airl-iisc/MRFP) has no FFI layer: its boundary for this path is the
 * torch.nn.Module surface of `MRFPPlus` (/root/reference/deepv3.py:152-367).  Each entry point below
 * replaces the ATen/cuDNN op sequence of one reference code span (cited per function); the Python
 * host (`mrfp_b200/`) binds them with ctypes and wraps them in torch.autograd.Function objects that
 * are called from a drop-in `MRFPPlus` module.  INTEGRATION.md shows the binding a maintainer of the
 * reference would add.
 *
 * Conventions
 *   - every data pointer is a DEVICE pointer owned by the caller (PyTorch tensors); the library
 *     never allocates, frees or retains device memory and performs no host<->device copy;
 *   - tensors are contiguous fp32 NCHW at the boundary, exactly what the reference passes around;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no host synchronisation;
 *   - return value: 0 success; < 0 invalid argument (nothing was launched, see mrfp_strerror);
 *     > 0 a cudaError_t raised by a launch / attribute call;
 *   - re-entrant: no global mutable state except once-per-device function attributes and a mutex-guarded cache of TMA
 *     descriptors inside each plan; safe under nn.DataParallel's per-device host threads and under DDP;
 *   - every entry point may be called while `stream` is being captured into a CUDA graph (no synchronisation, no
 *     allocation, no per-launch host state in kernel arguments).
 */
#ifndef MRFP_B200_H_
#define MRFP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRFP_OK                 0
#define MRFP_ERR_NULL_POINTER  (-1)
#define MRFP_ERR_BAD_SHAPE     (-2)
#define MRFP_ERR_WORKSPACE     (-3)   /* workspace / saved buffer too small or misaligned */
#define MRFP_ERR_UNSUPPORTED   (-4)   /* math mode / channel count not built */
#define MRFP_ERR_BAD_PLAN      (-5)
#define MRFP_ERR_DRIVER        (-6)   /* cuTensorMapEncodeTiled entry point unavailable / failed */

#define MRFP_MATH_FP32  0   /* CUDA-core direct convolution, fp32 activations (tight parity mode)   */
#define MRFP_MATH_TF32  1   /* tcgen05 implicit-GEMM convolution, tf32 operands, fp32 activations and accumulation:
                               the arithmetic of the reference's cuDNN convolutions under torch's TF32 default */
#define MRFP_MATH_BF16  2   /* tcgen05 implicit-GEMM convolution, bf16 operands, fp32 accumulation  */

int         mrfp_version(void);
const char* mrfp_strerror(int rc);

/* ------------------------------------------------------------------------------------------------
 * NP+  — replaces MRFPPlus.Normalization_Perturbation_Plus, deepv3.py:268-277 (call sites :317-318,
 * :334-335) and its autograd backward.
 *
 *   m[n,c]   = mean_hw x[n,c,:]                                   (:269)
 *   d[c]     = std_n(m[:,c]) (unbiased);  s[c] = 1.5 d[c]/max_c d  (:272-273)
 *   beta     = 1 + eps * s                                         (:275)   eps   = torch.normal(0,.75) draw
 *   out      = alpha*x - alpha*m + beta*m                          (:276)   alpha = torch.normal(1,.75) draw
 *
 * The two Gaussian draws are made by the host with torch's RNG (parity with the reference's RNG
 * stream) and passed in as (N,C) arrays.  One cooperative persistent kernel: phase A plane sums ->
 * grid barrier -> every CTA derives the (N,C) statistics -> phase B rewrite, re-reading the tail of
 * phase A from shared memory / L2.  N == 1 gives NaN exactly like torch.std (deepv3.py:272).
 * ---------------------------------------------------------------------------------------------- */
size_t mrfp_npplus_ws_bytes(int N, int C, int HW);
/* The first 64 bytes of `ws` are the kernel's queue counters: they must be ZERO when a buffer is used for the first time
 * (mrfp_npplus_ws_init enqueues that memset; an allocation that zero-fills serves as well); from then on the kernels
 * maintain them (the phase-A counter is cleared behind the first grid barrier of every launch, the phase-B counter at
 * kernel entry), so one workspace serves any sequence of stream-ordered calls — including replays of a captured CUDA
 * graph, since no per-launch host value enters the kernel. */
int    mrfp_npplus_ws_init(void* ws, size_t ws_bytes, void* stream);

int mrfp_npplus_fwd_f32(const float* x,       /* (N,C,HW) */
                        const float* alpha,   /* (N,C) draw #1 */
                        const float* eps,     /* (N,C) draw #2 */
                        float* out,           /* (N,C,HW) */
                        float* mean,          /* (N,C) out: plane means, saved for backward */
                        float* beta,          /* (N,C) out (diagnostic; may be NULL) */
                        void* ws, size_t ws_bytes, int N, int C, int HW, void* stream);

/* gin = alpha*g + dL/dm/HW with the closed-form dL/dm through std and max (SURVEY.md §8 a-1). */
int mrfp_npplus_bwd_f32(const float* gout, const float* alpha, const float* eps, const float* mean,
                        float* gin, void* ws, size_t ws_bytes, int N, int C, int HW, void* stream);

/* NP+ with its statistics taken by the producer of the feature (SURVEY.md 8f-1).  deepv3.py:332-335 applies NP+ to the
 * output of layer1, which ends in a ReLU (Resnet.py:218-225): mrfp_relu_psum_f32 is that ReLU (y may alias x) and also
 * leaves psum[n*C+c] = sum_hw y (NC doubles, zeroed by the call); mrfp_npplus_fwd_presummed_f32 is then a single
 * streaming pass (1R+1W) producing the same out / mean / beta as mrfp_npplus_fwd_f32.  ws: >=
 * mrfp_npplus_presummed_ws_bytes(N,C) bytes, 16-byte aligned.  Backward: mrfp_npplus_bwd_f32. */
int mrfp_relu_psum_f32(const float* x, float* y, double* psum, int NC, int HW, void* stream);
size_t mrfp_npplus_presummed_ws_bytes(int N, int C);
int mrfp_npplus_fwd_presummed_f32(const float* x, const double* psum, const float* alpha, const float* eps,
                                  float* out, float* mean, float* beta, void* ws, size_t ws_bytes,
                                  int N, int C, int HW, void* stream);

/* ------------------------------------------------------------------------------------------------
 * HRFP — replaces the chain deepv3.py:320-327 (8 x conv3x3 -> F.interpolate(nearest) -> BatchNorm2d
 * (train) -> ReLU on the layer types of deepv3.py:221-237), the adds deepv3.py:329-330 and
 * :356-357, the BN running-stat side effect, and the autograd input-gradient of all of it.
 * No weight / gamma / beta gradients exist (requires_grad_(False), deepv3.py:221-237).
 * ---------------------------------------------------------------------------------------------- */
typedef struct mrfp_hrfp_plan mrfp_hrfp_plan_t;   /* opaque host-side geometry + launch plan */

/* N: local batch; cin: channels of xp (64 for ResNet-50); (xh,xw): xp size; (h,w): image size —
 * sizes follow deepv3.py:320-327: x1.205, x1.2, x1.2, (h/2,w/2), (h/2,w/2), x0.838, x0.798,
 * (ceil(h/4),ceil(w/4)).  widths[4] = encoder channel counts (64,64,128,256 in the reference). */
int  mrfp_hrfp_plan_create(mrfp_hrfp_plan_t** plan, int N, int cin, int xh, int xw, int h, int w,
                           const int* widths, int math_mode);
void mrfp_hrfp_plan_destroy(mrfp_hrfp_plan_t* plan);

size_t mrfp_hrfp_plan_ws_bytes(const mrfp_hrfp_plan_t* plan);     /* scratch, fwd and bwd */
size_t mrfp_hrfp_plan_saved_bytes(const mrfp_hrfp_plan_t* plan);  /* fwd -> bwd state       */
size_t mrfp_hrfp_plan_lut_bytes(const mrfp_hrfp_plan_t* plan);    /* nearest-index tables   */
/* writes the table blob into HOST memory; the caller uploads it once per plan */
int    mrfp_hrfp_plan_write_luts(const mrfp_hrfp_plan_t* plan, void* host_dst, size_t bytes);
/* per stage k (0..7): out[0..5] = cin, cout, dilation, conv_h, conv_w, out_h; out[6] = out_w */
int    mrfp_hrfp_plan_stage(const mrfp_hrfp_plan_t* plan, int k, int* out7);
/* Operand fusion of the bf16 chain (default: all bits; ignored by the other math modes).
 *   bit 0: the forward F.interpolate -> BatchNorm2d -> ReLU between two convs of deepv3.py:320-327 is computed inside the next
 *          conv's operand producer: the intermediate activation never reaches HBM;
 *   bit 1: ReLU' -> BatchNorm2d backward -> nearest adjoint in front of a dgrad is computed inside that dgrad's operand
 *          producer, for the stages whose resample never replicates a pixel (the identity and the down-sampling stages).
 * 0 keeps every element-wise step as a separate pass (A/B measurements, tests).  Returns the bits in effect, or a negative
 * MRFP_ERR_* code.  Not to be changed between a forward and its backward. */
int    mrfp_hrfp_plan_set_fusion(mrfp_hrfp_plan_t* plan, int bits);

/* Forward.  W[k]: (cout,cin,3,3); gamma/beta[k]: (cout); running_mean/var[k]: (cout) updated in
 * place with `momentum` (unbiased variance) or skipped when the array pointer is NULL.
 *   ocout      (N,cin,xh,xw)      = OCout (+ x_add when x_add != NULL: deepv3.py:330)
 *   ocout_dec  (N,widths[3],h/2,w/2) = OCout_dec, or NULL when HRFP+ is off
 * ocout == NULL runs the encoder half only (decoder output unused when p >= 0.5); with ocout_dec == NULL as
 * well the call only leaves the state for a later mrfp_hrfp_plus_add / mrfp_hrfp_bwd in `saved`.
 * NP+ call 1 folded into the chain (SURVEY.md 8f-1):  ocout = OCout + NP+(xp)  — deepv3.py:316-318 followed by
 * :320-330 when both gates are on — without materialising NP+(xp): the plane totals of xp are taken by the layout pass
 * that feeds the chain, the per-plane (a, b) by one block, and the chain's output pass adds a*xp + b.
 *   np_alpha, np_eps (N,cin): the two Gaussian draws of deepv3.py:274-275;  np_mean (N,cin) out: plane means, needed
 *   by the backward;  np_beta (N,cin) out, may be NULL;  np_ws: >= mrfp_hrfp_np_ws_bytes(N,cin) bytes, 16-byte aligned.
 * np_alpha, np_eps, np_mean and np_ws are all NULL (NP+ not folded in) or all set; folding needs ocout and no x_add. */
size_t mrfp_hrfp_np_ws_bytes(int N, int C);
int mrfp_hrfp_fwd(const mrfp_hrfp_plan_t* plan, const float* xp,
                  const float* const* W, const float* const* gamma, const float* const* beta,
                  float* const* running_mean, float* const* running_var, float momentum, float eps,
                  const float* x_add, const float* np_alpha, const float* np_eps, float* np_mean, float* np_beta,
                  void* np_ws, float* ocout, float* ocout_dec, const void* lut, void* saved, void* ws, void* stream);

/* The form in which the gradient of OCout_dec reaches mrfp_hrfp_bwd (`dec_form`, `g_dec`, `w2t64`). */
#define MRFP_DEC_GRAD_NONE    0  /* OCout_dec unused: g_dec and w2t64 NULL                                   */
#define MRFP_DEC_GRAD_F32     1  /* g_dec (N, widths[3], h/2, w/2) fp32 NCHW                                  */
#define MRFP_DEC_GRAD_NHWC    2  /* g_dec (N, h/2, w/2, widths[3]) in the chain's element type (TF32/BF16)    */
#define MRFP_DEC_GRAD_RANK_K  3  /* g_dec = g64 (N, h/2, w/2, 64) bf16, w2t64 (256, 64) bf16 (BF16, widths[3]==256) */

/* Input gradient wrt xp.  g_ocout may be NULL (that output unused).  The NHWC and rank-K forms must be 16-byte aligned.
 * The rank-K form is W2^T g of the classifier tail left as its two factors (mrfp_hrfp_tail_final2_bwd_rk): the stage-4
 * dgrad accumulates g64 . w2t64^T as one more k-block on the tensor cores (fp32, one rounding together with the
 * convolution's own sum), so the (N, h/2, w/2, 256) tensor — 604 MB at batch 8, 768^2 — is neither written nor read; when
 * the stage-4 dgrad does not run as the operand-fused kernel, or the backward is encoder-only, the library expands the
 * product itself.  np_*: the forward's NP+ draws, plane means and workspace when NP+ was folded in, else all NULL;
 * g_xp then receives the sum of both gradient paths into xp (NP+ is ignored when g_ocout is NULL). */
int mrfp_hrfp_bwd(const mrfp_hrfp_plan_t* plan, const float* g_ocout, int dec_form, const void* g_dec, const void* w2t64,
                  const float* const* gamma, const float* np_alpha, const float* np_eps, const float* np_mean,
                  void* np_ws, const void* lut, const void* saved, float* g_xp, void* ws, void* stream);

/* HRFP+ skip add, deepv3.py:357, fused with the production of OCout_dec: out = dec1_up + OCout_dec where
 * OCout_dec = ReLU(BN(resample(conv4))) is recomputed from the state `saved` by the preceding mrfp_hrfp_fwd
 * (which may then be called with ocout_dec == NULL): the (N,256,h/2,w/2) fp32 tensor is never materialised.
 * dec1_up / out: (N, widths[3], h/2, w/2) fp32 NCHW. */
int mrfp_hrfp_plus_add(const mrfp_hrfp_plan_t* plan, const void* saved, const void* lut, const float* dec1_up,
                       float* out, void* stream);

/* The same with the reference's Upsample in front (deepv3.py:356-357, mynn.py:114-119): out = bilinear(dec1, size =
 * (h/2, w/2), align_corners=True) + OCout_dec, evaluated from the LOW-resolution dec1 (N, widths[3], lh, lw) with ATen's
 * interpolation formula — the upsampled (N,256,h/2,w/2) tensor is never materialised either. */
int mrfp_hrfp_plus_add_bilinear(const mrfp_hrfp_plan_t* plan, const void* saved, const void* lut, const float* dec1,
                                int lh, int lw, float* out, void* stream);

/* HRFP+ tail fused THROUGH the classifier (SURVEY.md 8f-4; bf16 plans, widths[3] == 256, K <= 24 classes) — replaces
 * deepv3.py:356-361: dec1 = Upsample(dec1); dec1 = OCout_dec + dec1; dec2 = final2(dec1), final2 = Conv2d(256, K, 1, bias).
 * A 1x1 convolution commutes with the bilinear interpolation:  dec2 = b2 + Upsample(W2 . dec1) + W2 . OCout_dec.
 *   t_lo (N, K, lh, lw) fp32 = W2 . dec1 at LOW resolution (a plain GEMM, computed by the caller; autograd of that GEMM
 *        yields the gradient to dec1 and the low-resolution half of the gradient to W2);
 *   w2 (K, 256), b2 (K) fp32;  out (N, K, h/2, w/2) fp32 NCHW.
 * Neither OCout_dec, the up-sampled dec1 nor their sum (N, 256, h/2, w/2) is materialised.
 * Backward, given g = dL/d out: g_dec_nhwc (N, h/2, w/2, 256) bf16 = W2^T g (mrfp_hrfp_bwd's MRFP_DEC_GRAD_NHWC),
 * g_w2 (K, 256) = sum_pixels g . OCout_dec^T (the high-resolution half of the weight gradient), g_b2 (K) = sum g; the
 * gradient to t_lo is mrfp_bilinear_up_bwd_f32(g).  MRFP_ERR_UNSUPPORTED: use mrfp_hrfp_plus_add_bilinear + a conv.
 * Inputs arrive through TMA tensor maps the plan caches per direction (re-encoded when an address or shape changes): t_lo
 * must be 16-byte aligned with lw % 4 == 0 and describe an Upsample by >= 2 (else MRFP_ERR_UNSUPPORTED); g may have any
 * alignment (rows that are not 16-byte aligned are read with plain loads). */
int mrfp_hrfp_tail_final2_fwd(const mrfp_hrfp_plan_t* plan, const void* saved, const void* lut, const float* t_lo,
                              int lh, int lw, const float* w2, const float* b2, int K, float* out, void* stream);
int mrfp_hrfp_tail_final2_bwd(const mrfp_hrfp_plan_t* plan, const void* saved, const void* lut, const float* g,
                              const float* w2, int K, void* g_dec_nhwc, float* g_w2, float* g_b2, void* stream);
/* The rank-K form of the same gradient (the default of the Python host; mrfp_hrfp_bwd's MRFP_DEC_GRAD_RANK_K): W2^T g
 * with K <= 24 classes left as its two factors instead of an (N, h/2, w/2, 256) tensor —
 *   g64 (N, h/2, w/2, 64) bf16: g per pixel, classes beyond K zero;   w2t64 (256, 64) bf16: W2 transposed, zero-padded.
 * Everything else as mrfp_hrfp_tail_final2_bwd. */
int mrfp_hrfp_tail_final2_bwd_rk(const mrfp_hrfp_plan_t* plan, const void* saved, const void* lut, const float* g,
                                 const float* w2, int K, void* g64, void* w2t64, float* g_w2, float* g_b2, void* stream);

/* Backward of the reference's Upsample (network/mynn.py:114-119, bilinear, align_corners=True) at the up-sampling sites of
 * the tail (deepv3.py:356, :362), as a gather instead of ATen's atomicAdd scatter:
 *   gl (planes, LH, LW) = adjoint of the up-sampling applied to g (planes, OH, OW), OH >= LH, OW >= LW.
 * The per-axis gather tables are built on the host with ATen's float arithmetic (mrfp_bilinear_bwd_write_table fills
 * mrfp_bilinear_bwd_table_bytes(L, O) bytes; word [1] of a table is the `span_w` argument); the caller uploads them once. */
size_t mrfp_bilinear_bwd_table_bytes(int L, int O);
int    mrfp_bilinear_bwd_write_table(int L, int O, void* host_dst, size_t bytes);
int    mrfp_bilinear_up_bwd_f32(const float* g, float* gl, long long planes, int LH, int LW, int OH, int OW,
                                const void* tab_h, const void* tab_w, int span_w, void* stream);

/* Plain variant of the same add for a materialised OCout_dec: out = a + b (n elements). */
int mrfp_add_f32(const float* a, const float* b, float* out, size_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * InstanceNorm2d(affine=True) [+ ReLU] of the trunk next to the insertion points (SURVEY.md 8f-3) — replaces
 * nn.InstanceNorm2d + nn.ReLU at network/Resnet.py:534-536 / :591-598 (stem, wt_layer[2] == 4) and
 * network/Resnet.py:176-178 + :218-225 (last Bottleneck of layer1 / layer2, iw == 4), and their autograd backward.
 *
 *   y = (x - mean_hw x) / sqrt(var_hw x + eps) * gamma[c] + beta[c]      (biased variance, no running statistics)
 *   y = max(y, 0) when relu != 0;   psum[n*C+c] = sum_hw y when psum != NULL (the plane sums NP+ call 2 needs,
 *   deepv3.py:334-335: layer1's IN + ReLU is its producer)
 *
 * One thread-block cluster per plane keeps the plane in shared memory between the statistics and the write: forward
 * 1R + 1W, backward 2R + 1W of HBM traffic.  x, y, gy, gx: (N,C,HW) fp32; gamma, beta: (C) or NULL (= 1, 0);
 * mean, invstd: (N,C) out (forward) / in (backward).  The backward recomputes the ReLU mask from x with the forward's
 * expression and leaves per-plane partials dgamma_part, dbeta_part (N,C): d_gamma[c] = sum_n dgamma_part[n,c].
 * ---------------------------------------------------------------------------------------------- */
int mrfp_instnorm_fwd_f32(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* invstd,
                          double* psum, int N, int C, int HW, float eps, int relu, void* stream);
int mrfp_instnorm_bwd_f32(const float* gy, const float* x, const float* gamma, const float* beta, const float* mean,
                          const float* invstd, float* gx, float* dgamma_part, float* dbeta_part, int N, int C, int HW,
                          int relu, void* stream);

/* Backward of NP+(ReLU(InstanceNorm(x))) — NP+ call 2 (deepv3.py:334-335) folded into the backward of its producer
 * (Resnet.py:218-225), SURVEY.md 8f-1: g is the gradient of the NP+ OUTPUT; its plane totals (1R), the NP+ backward
 * coefficients (np_alpha, np_eps: the forward's draws; np_mean: the plane means of the NP+ input saved by
 * mrfp_npplus_fwd_presummed_f32) and the InstanceNorm backward with gy = a'*g + b' applied on load (2R + 1W) replace
 * mrfp_npplus_bwd_f32 followed by mrfp_instnorm_bwd_f32 ((2R+1W) + (2R+1W)).  ws: >= N*C*16 bytes, 16-byte aligned; C <= 256. */
int mrfp_instnorm_bwd_np_f32(const float* g, const float* x, const float* gamma, const float* beta, const float* mean,
                             const float* invstd, const float* np_alpha, const float* np_eps, const float* np_mean,
                             void* ws, size_t ws_bytes, float* gx, float* dgamma_part, float* dbeta_part, int N, int C, int HW,
                             int relu, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MRFP_B200_H_ */
