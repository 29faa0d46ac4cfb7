// tcgen05 (5th-gen tensor core) implicit-GEMM convolution for SSNB_FAST_FP16 — interface.
//
// One kernel family computes   out[p, n] = epi( sum_taps sum_c  A[p + shift(tap), c] * B[tap][n][c] )
// over NHWC fp16 tensors: A tiles are 4-D TMA boxes of the activation view (zero-filled outside
// the image = free padding), B tiles are 3-D TMA boxes of the packed weights, accumulators live
// in TMEM, the epilogue fuses folded-BN bias + ReLU (forward) or accumulation (data gradient).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "common.cuh"

namespace ssnb {

constexpr int UMMA_MAX_TAPS = 16;
constexpr int UMMA_V2_PIPE_BYTES = 216 * 1024;   // operand staging of the second-generation kernel

struct UmmaContext {
  bool active = false;
  void* encode_tiled = nullptr;   // cuTensorMapEncodeTiled, resolved through cudaGetDriverEntryPoint
  int num_sms = 148;
  bool attr_set = false;
};

struct UmmaConvParams {
  int W, H, F;                    // output dims; tiles enumerate output pixels (stride 1: the input has the same dims)
  int bw, bh, bf;                 // TMA box in pixels; bw*bh*bf <= 128 rows of the M tile
  int tiles_w, tiles_h, tiles_f;
  int n_tiles, block_n;           // N split of Cout
  int stages, stage_bytes;        // first-generation kernel: smem pipeline depth / stride chosen from block_n
  int kchunks, ntaps, K;          // ceil(K/64), filter taps, reduction channels per tap
  int tap_dy[UMMA_MAX_TAPS], tap_dx[UMMA_MAX_TAPS];
  __half* out; int out_pitch, out_coff, Cout;
  const float* bias;              // [Cout] or nullptr
  int relu, accumulate;
  // horizontal fusion of sibling 1x1 convolutions (same input):
  int kchunks_a1, K1;             // K chunks [0, kchunks_a1) come from tmap_a (K1 real channels), the rest from tmap_a2
  int n_split;                    // output columns >= n_split go to out2 (second destination), else to out
  __half* out2; int out2_pitch, out2_coff;
  // second-generation kernel (umma_conv_v2.cu, every stride-1 plan): ONE halo A box per K chunk covers the tile plus its
  // filter halo, stored [y][frame][x][64 ch]; every tap is a shifted UMMA descriptor view into it.  CTA pairs
  // (cta_group::2): tiles are (N tile, pair of M tiles)
  int v2;                         // 1: launch umma_conv_v2_kernel; 0: the stride-2 forward kernel of umma_conv.cu
  int b_taps;                     // v2: taps per weight stage
  int tiles_q;                    // v2: PAIRS of frame groups = last digit of the tile walk
  int epi_stages, epi_stage_bytes;// v2 TMA-fed epilogue: ring depth (0 = off) and stride (old + activation chunk)
  int a_stages, b_stages, a_stage_bytes, b_stage_bytes;
  int a_load_bytes;               // bytes the halo A box delivers
  int halo_x0, halo_y0;           // box origin relative to the tile origin (min dx, min dy)
  int a_sbo;                      // bytes between consecutive 8-pixel row groups of a tap view
  int tap_aoff[UMMA_MAX_TAPS];    // byte offset of each tap's view inside the A stage
  // data gradient that is the LAST writer of its output: fuse dz = dy * (y > 0), y = activation of the same value
  const __half* mask_y; int mask_pitch, mask_coff;
  // SSNB_EXACT_TC (error-compensated split operands): nseg = 3 runs every K chunk three times,
  //   (A_lo, B_hi), (A_hi, B_lo), (A_hi, B_hi), into the same TMEM accumulator; nseg = 1 is the plain fp16 product.
  // out_f32: the epilogue works in fp32 -- out32 = alpha * acc (+ bias, ReLU | + old out32) -- and, when out_hi is set,
  // also writes the result's fp16 hi / lo operand planes (same pitch / channel offset, lo plane out_lo_off bytes later).
  int nseg, out_f32;
  float alpha;
  const float* alpha_dev;         // optional device scalar multiplied into alpha (1 / the power-of-two scale of the weight planes)
  float* out32; __half* out_hi; long long out_lo_off;
  float* out32_2; __half* out_hi2; long long out_lo_off2;   // fused sibling forward: columns >= n_split go here (pitch / offset: out2_pitch / out2_coff)
  // out_f32 data gradient that is the LAST writer of its output value v: dz = (alpha * acc + old) * (y > 0) with y = the fp32
  // activation of v; the planes written through out_hi then hold dz * plane_scale (the loss scale) for v's producers'
  // weight / data gradients, and *flag is raised when that leaves the fp16 range
  const float* mask32; int mask32_pitch, mask32_coff;
  float plane_scale; int* flag;
};

struct UmmaConvPlan {
  bool enabled = false;
  const __half* mask_y = nullptr; int mask_pitch = 0, mask_coff = 0;   // applied only when launched with mask=true
  CUtensorMap tmap_a, tmap_a2, tmap_b;
  CUtensorMap tmap_a_lo, tmap_a2_lo, tmap_b_lo;   // SSNB_EXACT_TC: LO planes of the three operands (copies of the HI maps otherwise)
  long long b_lo_off = 0;                        // byte offset of the LO weight plane (0: single plane)
  // SSNB_EXACT_TC mask fusion, applied only when launched with mask=true (see UmmaConvParams::mask32)
  const float* mask32 = nullptr; int mask32_pitch = 0, mask32_coff = 0;
  __half* mask_planes = nullptr; long long mask_planes_lo = 0; float mask_plane_scale = 1.0f; int* mask_flag = nullptr;
  CUtensorMap tmap_old, tmap_y;   // TMA-fed epilogue: output (old gradient) and mask-activation tiles, [128 rows][64 ch] boxes
  bool epi_maps_ready = false, epi_mask_ready = false;
  int epi_box[3] = {0, 0, 0}, epi_F = 0;     // box {W, F, H} extents and frame count for encoding tmap_y when the mask is attached
  // geometry of the weight map (each kernel encodes it with its own box)
  const __half* b_ptr = nullptr; unsigned long long b_dims[3] = {0, 0, 0}, b_strides[2] = {0, 0};
  UmmaConvParams p;
};

// SSNB_EXACT_TC binding options: split weights (LO plane `w_lo_off` bytes after the HI plane), fp32 output view `out32`
// (the bind call's own out/dx view then names the fp16 HI plane of the result, lo_off its LO plane; base == nullptr: no
// planes are written), accumulator scale alpha
struct UmmaTcOpts { long long w_lo_off = 0; float* out32 = nullptr; float alpha = 1.0f; const float* alpha_dev = nullptr; float* out32_2 = nullptr; };
void umma_context_init(UmmaContext& ctx, bool fp16);
void umma_context_destroy(UmmaContext& ctx);
// forward convolution plan (stride 1, or stride 2 on the first-generation kernel): in/out views, weights wd = [tap][cout][cin] fp16
int umma_conv_bind_fwd(UmmaContext& ctx, UmmaConvPlan& plan, View in, View out, int F, int cin, int cout, int k, int pad,
                       int stride, const __half* w_tap_n_k, const float* bias, const UmmaTcOpts* tc = nullptr);
// generic tap table variant (conv1 in space-to-depth form: 16 taps of a 4x4 stride-1 convolution)
int umma_conv_bind_taps(UmmaContext& ctx, UmmaConvPlan& plan, View in, View out, int F, int cin, int cout, int ntaps,
                        const int* dy, const int* dx, const __half* w_tap_n_k, const float* bias, int relu, const UmmaTcOpts* tc = nullptr);
// data-gradient plan (stride 1): dz/dx gradient views, weights wf = [tap][cin][cout] fp16
int umma_conv_bind_dgrad(UmmaContext& ctx, UmmaConvPlan& plan, View dz, View dx, int F, int cin, int cout, int k, int pad,
                         const __half* w_tap_k_n, int accumulate, const UmmaTcOpts* tc = nullptr);
// fused forward of sibling 1x1 convs: one input view, weights [n1+n2][cin] (rows stacked), columns [0,n1) -> out1, rest -> out2
int umma_conv_bind_fused_fwd(UmmaContext& ctx, UmmaConvPlan& plan, View in, View out1, View out2, int F, int cin, int n1, int n2,
                             const __half* w_n_k, const float* bias, const UmmaTcOpts* tc = nullptr);
// fused data gradient of sibling 1x1 convs: dx (+)= [dz1 | dz2] * W, weights [cin][pad64(k1) + k2]; dz1 may be empty (k1 = 0)
int umma_conv_bind_fused_dgrad(UmmaContext& ctx, UmmaConvPlan& plan, View dz1, View dz2, View dx, int F, int cin, int k1, int k2,
                               const __half* w_n_k, int accumulate, const UmmaTcOpts* tc = nullptr);
int umma_conv_launch(UmmaContext& ctx, const UmmaConvPlan& plan, cudaStream_t s, bool mask = false);
// second-generation kernel (umma_conv_v2.cu); `p` = plan.p with the per-launch fields (mask) already applied
bool umma_conv_v2_supported(int ntaps);
int umma_conv_v2_launch(UmmaContext& ctx, const UmmaConvPlan& plan, const UmmaConvParams& p, cudaStream_t s);
int umma_conv_set_mask(UmmaContext& ctx, UmmaConvPlan& plan, View y);
// EXACT_TC: y32 = fp32 activation of the output value, dplanes = that value's gradient operand planes (hi base + lo_off)
void umma_conv_set_mask_tc(UmmaConvPlan& plan, View y32, View dplanes, float plane_scale, int* flag);

// host helpers shared by the tensor-core kernels
int umma_resolve_encode(UmmaContext& ctx);
int umma_encode_f16(UmmaContext& ctx, CUtensorMap* m, int rank, void* addr, const cuuint64_t* dims,
                    const cuuint64_t* strides, const cuuint32_t* box, int spatial_stride = 1);

// ---- weight gradient on tcgen05 (umma_wgrad.cu) -------------------------------------------------------
// partial[split][tap][co][ci] = sum over the split's pixels of dz[p, co] * x[p + (r-pad, s-pad), ci]
// (both operands MN-major: the reduction dimension is the pixel index).
struct UmmaWgradParams {
  int W, H, F;
  int bw, bh, bf;                 // 64-pixel TMA box
  int tiles_w, tiles_h, tiles_f;
  int ptiles_per_split, splits;
  int ntaps, tap_dy[UMMA_MAX_TAPS], tap_dx[UMMA_MAX_TAPS];
  int Cout, Cin, m_tiles, n_tiles, block_n;
  int x_stride;                   // 2: stride-2 layers, the x box steps over the input with TMA element stride 2
  float* bias_partial;            // [split][Cout] column sums of dz (bias gradient) from an extra ones-operand MMA, or nullptr
  int taps_per_cta, tap_groups, mma_n;   // taps sharing one dz tile per CTA; N of each tap's MMA
  int stages, stage_bytes;        // pipeline depth / stride
  int run_len, run_stride;        // run_len > 1: x staged as one halo box per 64 channels, the CTA's taps are one run of
                                  // equally spaced descriptor views (tap_xoff, run_stride bytes apart) taken by a single MMA
  int x_box_bytes, x_box_tx, x_sbo, halo_x0, halo_y0, tap_xoff[UMMA_MAX_TAPS];   // box stride in smem / bytes one box delivers
  float* partial;
  int nseg;                       // 3: SSNB_EXACT_TC, every pixel tile runs (dz_lo, x_hi), (dz_hi, x_lo), (dz_hi, x_hi)
};
struct UmmaWgradPlan {
  bool enabled = false;
  CUtensorMap tmap_dz, tmap_x;
  CUtensorMap tmap_dz_lo, tmap_x_lo;              // SSNB_EXACT_TC: LO planes (View::lo_off of the bound views)
  UmmaWgradParams p;
};
// returns the number of splits chosen through *splits (the caller sizes `partial` from it)
int umma_wgrad_bind(UmmaContext& ctx, UmmaWgradPlan& plan, View dz, View x, int F, int cin, int cout, int k, int pad,
                    float* partial, int max_splits, int x_stride = 1);
int umma_wgrad_bind_taps(UmmaContext& ctx, UmmaWgradPlan& plan, View dz, View x, int F, int cin, int cout, int ntaps,
                         const int* dy, const int* dx, float* partial, int max_splits, int x_stride = 1);
int umma_wgrad_launch(UmmaContext& ctx, const UmmaWgradPlan& plan, cudaStream_t s, float* bias_partial = nullptr);

}  // namespace ssnb
