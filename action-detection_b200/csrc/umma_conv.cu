// tcgen05 implicit-GEMM convolution (sm_100a): host-side planning for both kernel generations, and the first-generation
// kernel (per-tap A boxes), which runs the stride-2 forward layers.  Every stride-1 plan runs on umma_conv_v2.cu (halo
// boxes, CTA pairs, warp-uniform role loops).
//
//   warp 0      : TMA producer   (A: 4-D activation box with TMA element stride 2, B: 3-D weight box, SWIZZLE_128B)
//   warp 1      : TMEM allocator + MMA issuer (tcgen05.mma.cta_group::1.kind::f16, M=128, N=block_n)
//   warps 2..9  : epilogue       (tcgen05.ld 32x32b -> bias/ReLU -> fp16 NHWC store, or the SSNB_EXACT_TC fp32 epilogue);
//                 two warps per TMEM lane quadrant take alternating 32-column groups (memory-level parallelism of the stores)
//
// Rows of the M tile are the output pixels of one TMA box (bw x bh x bf); the box steps over the input with stride 2,
// taps shift its origin and rely on TMA's out-of-bounds zero fill for the convolution padding.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>

#include "umma_conv.cuh"
#include "umma_dev.cuh"
#include "umma_epi32.cuh"

namespace ssnb {

namespace {

using namespace umma;
constexpr int MAX_STAGES = 8;
constexpr int PIPE_BYTES = 4 * (BLOCK_M * BLOCK_K * 2 + 256 * BLOCK_K * 2);   // 192 KiB of operand staging
constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;     // 16 KiB
constexpr int NUM_THREADS = 320;
constexpr int EPI_WARPS = 8;
constexpr int TMEM_COLS = 512;
constexpr int BAR_BYTES = 1024;                    // barriers
constexpr int SMEM_BYTES = PIPE_BYTES + 1024 /*align slack*/ + BAR_BYTES;

struct TileCoord { int w0, h0, f0, n0; };
__device__ __forceinline__ TileCoord decode_tile(const UmmaConvParams& p, int tile) {
  TileCoord t;
  const int nt = tile % p.n_tiles;
  int m = tile / p.n_tiles;
  t.n0 = nt * p.block_n;
  t.w0 = (m % p.tiles_w) * p.bw; m /= p.tiles_w;
  t.h0 = (m % p.tiles_h) * p.bh; m /= p.tiles_h;
  t.f0 = m * p.bf;
  return t;
}

// bias / ReLU on one 16-column chunk of an accumulator row, then fp16 store
__device__ __forceinline__ void epilogue_chunk(const UmmaConvParams& p, const uint32_t* r, int col, uint4* dst) {
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
  if (p.bias) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] += __ldg(p.bias + col + j);
  }
  if (p.relu) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
  }
  uint4 q0, q1;
  __half2* g0 = reinterpret_cast<__half2*>(&q0);
  __half2* g1 = reinterpret_cast<__half2*>(&q1);
#pragma unroll
  for (int j = 0; j < 4; ++j) { g0[j] = __floats2half2_rn(v[2 * j], v[2 * j + 1]); g1[j] = __floats2half2_rn(v[8 + 2 * j], v[8 + 2 * j + 1]); }
  dst[0] = q0; dst[1] = q1;
}

// Epilogue role: for every tile of this CTA wait for the accumulator, then TMEM -> registers -> bias/ReLU -> fp16 NHWC
// stores (every thread stores its own accumulator row, 32 bytes per 16 columns).  Row r of the tile is output pixel
// (x, y, f) = (r % bw, (r / bw) % bh, r / (bw*bh)).
__device__ __forceinline__ void epilogue_loop(const UmmaConvParams& p, uint32_t tmem_base, uint64_t* tfull_bar, uint64_t* tempty_bar,
                                              int warp, int lane, int total_tiles, int tile0, int tstep) {
  const int quad = warp & 3;
  const int cpar = (warp - 2) >> 2;
  const int row = quad * 32 + lane;
  const int rw = row % p.bw, rh = (row / p.bw) % p.bh, rf = row / (p.bw * p.bh);
  uint32_t acc = 0, acc_phase = 0;
  for (int tile = tile0; tile < total_tiles; tile += tstep) {
    const TileCoord t = decode_tile(p, tile);
    const int w = t.w0 + rw, h = t.h0 + rh, f = t.f0 + rf;
    const bool valid = (rf < p.bf) && (w < p.W) && (h < p.H) && (f < p.F);
    const long long opix = (long long)(f * p.H + h) * p.W + w;
    __half* orow = p.out + opix * p.out_pitch + p.out_coff;
    mbar_wait(&tfull_bar[acc], acc_phase);
    tc_fence_after();
    const uint32_t taddr = tmem_base + acc * 256 + ((uint32_t)(quad * 32) << 16);
    if (p.out_f32) {
      // SSNB_EXACT_TC: fp32 epilogue + the result's fp16 hi / lo operand planes (umma_epi32.cuh)
      float* orow32 = p.out32 + opix * p.out_pitch + p.out_coff;
      __half* hrow = p.out_hi ? p.out_hi + opix * p.out_pitch + p.out_coff : nullptr;
      const float alpha = p.alpha * (p.alpha_dev ? __ldg(p.alpha_dev) : 1.0f);
      for (int c0 = cpar * 32; c0 < p.block_n; c0 += 64) {
        const bool two = c0 + 16 < p.block_n;
        const int cola = t.n0 + c0, colb = cola + 16;
        uint32_t ra[16], rb[16];
        tmem_ld16(taddr + c0, ra);
        if (two) tmem_ld16(taddr + c0 + 16, rb);
        tmem_ld_wait();
        if (valid && cola < p.Cout) store_chunk32(p, alpha, ra, p.bias + cola, orow32 + cola, hrow ? hrow + cola : nullptr, nullptr, p.out_lo_off);
        if (two && valid && colb < p.Cout) store_chunk32(p, alpha, rb, p.bias + colb, orow32 + colb, hrow ? hrow + colb : nullptr, nullptr, p.out_lo_off);
      }
    } else {
      // two 16-column chunks per iteration: both TMEM loads are in flight before the first use
      for (int c0 = cpar * 32; c0 < p.block_n; c0 += 64) {
        const bool two = c0 + 16 < p.block_n;                       // warp-uniform
        const int cola = t.n0 + c0, colb = cola + 16;
        uint32_t ra[16], rb[16];
        tmem_ld16(taddr + c0, ra);
        if (two) tmem_ld16(taddr + c0 + 16, rb);
        tmem_ld_wait();
        if (valid && cola < p.Cout) epilogue_chunk(p, ra, cola, reinterpret_cast<uint4*>(orow + cola));
        if (two && valid && colb < p.Cout) epilogue_chunk(p, rb, colb, reinterpret_cast<uint4*>(orow + colb));
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(&tempty_bar[acc]);     // 8 arrivals (one per epilogue warp) release it
    }
    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
  }
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
umma_conv_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const __grid_constant__ CUtensorMap tmap_a_lo, const __grid_constant__ CUtensorMap tmap_b_lo, const UmmaConvParams p) {
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B operand tiles need 1024-byte alignment
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  // pipeline depth adapts to the tile: narrow-N layers get up to 8 stages in the same 192 KiB
  const int STAGES = p.stages, STAGE_BYTES = p.stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PIPE_BYTES);
  uint64_t* full_bar = bars;                     // [MAX_STAGES]
  uint64_t* empty_bar = bars + MAX_STAGES;       // [MAX_STAGES]
  uint64_t* tfull_bar = bars + 2 * MAX_STAGES;   // [2] accumulator ready
  uint64_t* tempty_bar = bars + 2 * MAX_STAGES + 2;  // [2] accumulator drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 4);

  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int total_tiles = p.tiles_w * p.tiles_h * p.tiles_f * p.n_tiles;
  const int nseg = p.nseg > 1 ? p.nseg : 1;          // SSNB_EXACT_TC: (A_lo, B_hi), (A_hi, B_lo), (A_hi, B_hi) per (tap, K chunk)
  const int ksteps = p.ntaps * p.kchunks * nseg;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      // bytes the two TMA boxes deliver (zero-filled out-of-bounds elements count; a 7x1x18 box has 126 rows)
      const uint32_t tx_bytes = (uint32_t)(p.bw * p.bh * p.bf + p.block_n) * BLOCK_K * 2;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const TileCoord t = decode_tile(p, tile);
        for (int seg = 3 - nseg; seg < 3; ++seg)
        for (int tap = 0; tap < p.ntaps; ++tap) {
          for (int kc = 0; kc < p.kchunks; ++kc) {
            const CUtensorMap* ma = seg == 0 ? &tmap_a_lo : &tmap_a;
            const CUtensorMap* mb = seg == 1 ? &tmap_b_lo : &tmap_b;
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * STAGE_BYTES;
            uint8_t* sb = sa + A_BYTES;
            mbar_expect_tx(&full_bar[stage], tx_bytes);
            // output pixel (w0, h0) reads input pixel (2 w0 + dx, 2 h0 + dy); the box steps by 2 (element stride)
            tma_load_4d(sa, ma, &full_bar[stage], kc * BLOCK_K, 2 * t.w0 + p.tap_dx[tap], 2 * t.h0 + p.tap_dy[tap], t.f0);
            tma_load_3d(sb, mb, &full_bar[stage], kc * BLOCK_K, t.n0, tap);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      const uint32_t idesc = make_idesc_f16(p.block_n);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);     // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 256;
        int kc = 0;
        for (int ks = 0; ks < ksteps; ++ks) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint32_t sb = sa + A_BYTES;
          // K chunks whose tail is TMA zero fill (Cin % 64 != 0) skip the all-zero MMAs
          const int kvalid = p.K - kc * BLOCK_K;
          if (kvalid >= BLOCK_K) {
#pragma unroll
            for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
              umma_f16(d_tmem, make_desc_k_sw128(sa + k * UMMA_K * 2), make_desc_k_sw128(sb + k * UMMA_K * 2), idesc, (ks | k) ? 1u : 0u);
          } else {
            const int nk = (kvalid + UMMA_K - 1) / UMMA_K;
            for (int k = 0; k < nk; ++k)
              umma_f16(d_tmem, make_desc_k_sw128(sa + k * UMMA_K * 2), make_desc_k_sw128(sb + k * UMMA_K * 2), idesc, (ks | k) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);               // frees the smem slot when these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
          if (++kc == p.kchunks) kc = 0;
        }
        umma_commit(&tfull_bar[acc]);                   // accumulator complete
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ===== epilogue warps 2..9; TMEM lane quadrant = warp % 4, column-group parity = (warp - 2) / 4 =====
    epilogue_loop(p, tmem_base, tfull_bar, tempty_bar, warp, lane, total_tiles, blockIdx.x, gridDim.x);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int resolve_encode(UmmaContext& ctx) {
  if (ctx.encode_tiled) return 0;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
  if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) {
    cudaGetLastError();
    set_thread_error("cuTensorMapEncodeTiled not available from the driver");
    return 2;
  }
  ctx.encode_tiled = fn;
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  ctx.num_sms = sms;
  return 0;
}

int encode(UmmaContext& ctx, CUtensorMap* m, int rank, void* addr, const cuuint64_t* dims, const cuuint64_t* strides,
           const cuuint32_t* box, int spatial_stride = 1) {
  // spatial_stride 2: the box traverses W and H with step 2 (box extents are given in un-strided elements)
  cuuint32_t es[5] = {1, (cuuint32_t)spatial_stride, (cuuint32_t)spatial_stride, 1, 1};
  CUresult r = reinterpret_cast<EncodeTiledFn>(ctx.encode_tiled)(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, addr, dims, strides,
                                                                box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                                                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[128];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled failed (CUresult %d, rank %d)", (int)r, rank);
    set_thread_error(buf);
    return 2;
  }
  return 0;
}

void pick_box(int W, int& bw, int& bh, int& bf) {
  if (W % 8 == 0 && W >= 56) { bw = 8; bh = 8; bf = 2; }
  else if (W % 4 == 0) { bw = 4; bh = 4; bf = 8; }
  else if (W % 2 == 0) { bw = 2; bh = 2; bf = 32; }
  else if (W <= 8) { bw = W; bh = 1; bf = BLOCK_M / W; }
  else { bw = 1; bh = 1; bf = 128; }
}

// Fields shared by both kernels: the N split, K chunks, output view, weight-map geometry and the SSNB_EXACT_TC epilogue.
// Tiles enumerate the pixels of the output view `o`; bind_strided or bind_halo then chooses the box, encodes the tensor maps
// and enables the plan.
int bind_common(UmmaContext& ctx, UmmaConvPlan& plan, View a, View o, int F, int K, int N, int ntaps, const __half* w,
                const UmmaTcOpts* tc) {
  plan.enabled = false;
  if (int rc = resolve_encode(ctx)) return rc;
  if (K % 8 || N % 16 || a.pitch % 8 || a.coff % 8 || o.pitch % 8 || o.coff % 8 || ntaps > UMMA_MAX_TAPS) {
    set_thread_error("umma conv: unsupported channel alignment"); return 1; }
  UmmaConvParams& p = plan.p;
  memset(&p, 0, sizeof(p));
  p.W = o.W; p.H = o.H; p.F = F;
  // N split: equal tiles of block_n <= 256 (multiple of 16); the last tile may overhang N (TMA zero-fills the
  // missing weight rows, the epilogue masks the columns)
  p.n_tiles = (N + 255) / 256;
  p.block_n = (((N + p.n_tiles - 1) / p.n_tiles) + 15) / 16 * 16;
  p.kchunks = (K + BLOCK_K - 1) / BLOCK_K;
  p.K = K;
  p.ntaps = ntaps;
  p.out = reinterpret_cast<__half*>(o.base); p.out_pitch = o.pitch; p.out_coff = o.coff; p.Cout = N;
  p.kchunks_a1 = p.kchunks; p.K1 = K; p.n_split = 1 << 30; p.out2 = p.out; p.out2_pitch = o.pitch; p.out2_coff = o.coff;
  plan.b_ptr = w;
  plan.b_lo_off = tc ? tc->w_lo_off : 0;
  plan.b_dims[0] = K; plan.b_dims[1] = N; plan.b_dims[2] = ntaps;
  plan.b_strides[0] = (unsigned long long)K * 2; plan.b_strides[1] = (unsigned long long)N * K * 2;
  // SSNB_EXACT_TC: three operand segments per K chunk, fp32 epilogue (+ fp16 operand planes of the result)
  p.nseg = tc ? 3 : 1; p.out_f32 = tc ? 1 : 0; p.alpha = tc ? tc->alpha : 1.0f; p.alpha_dev = tc ? tc->alpha_dev : nullptr;
  p.plane_scale = 1.0f;
  p.out32 = tc ? tc->out32 : nullptr; p.out_hi = tc ? reinterpret_cast<__half*>(o.base) : nullptr; p.out_lo_off = tc ? o.lo_off : 0;
  p.out32_2 = p.out32; p.out_hi2 = p.out_hi; p.out_lo_off2 = p.out_lo_off;       // second destination = the first unless a fused bind redirects it
  if (tc && (!tc->out32 || !a.lo_off || !tc->w_lo_off)) { set_thread_error("umma conv: split-operand bind needs operand planes and an fp32 output"); return 1; }
  return 0;
}

// weight map (and its LO plane) with boxes of BLOCK_K channels x `rows` output channels x `taps` taps
int encode_b(UmmaContext& ctx, UmmaConvPlan& plan, int rows, int taps) {
  cuuint64_t dims[3] = {plan.b_dims[0], plan.b_dims[1], plan.b_dims[2]};
  cuuint64_t str[2] = {plan.b_strides[0], plan.b_strides[1]};
  cuuint32_t box[3] = {(cuuint32_t)BLOCK_K, (cuuint32_t)rows, (cuuint32_t)taps};
  __half* w = const_cast<__half*>(plan.b_ptr);
  if (int rc = encode(ctx, &plan.tmap_b, 3, w, dims, str, box)) return rc;
  plan.tmap_b_lo = plan.tmap_b;
  if (plan.b_lo_off) return encode(ctx, &plan.tmap_b_lo, 3, reinterpret_cast<__half*>(reinterpret_cast<char*>(w) + plan.b_lo_off), dims, str, box);
  return 0;
}

// Stride-2 forward on the first-generation kernel: tiles enumerate OUTPUT pixels, the A box steps over the input `a` with
// TMA element stride 2 (box extents in un-strided elements).
int bind_strided(UmmaContext& ctx, UmmaConvPlan& plan, View a) {
  UmmaConvParams& p = plan.p;
  pick_box(p.W, p.bw, p.bh, p.bf);
  p.tiles_w = (p.W + p.bw - 1) / p.bw; p.tiles_h = (p.H + p.bh - 1) / p.bh; p.tiles_f = (p.F + p.bf - 1) / p.bf;
  p.stage_bytes = (A_BYTES + p.block_n * BLOCK_K * 2 + 1023) / 1024 * 1024;
  p.stages = PIPE_BYTES / p.stage_bytes; if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
  cuuint64_t dims[4] = {(cuuint64_t)p.K, (cuuint64_t)a.W, (cuuint64_t)a.H, (cuuint64_t)p.F};
  cuuint64_t str[3] = {(cuuint64_t)a.pitch * 2, (cuuint64_t)a.W * a.pitch * 2, (cuuint64_t)a.H * a.W * a.pitch * 2};
  cuuint32_t box[4] = {(cuuint32_t)BLOCK_K, (cuuint32_t)(2 * p.bw), (cuuint32_t)(2 * p.bh), (cuuint32_t)p.bf};
  if (int rc = encode(ctx, &plan.tmap_a, 4, reinterpret_cast<__half*>(a.base) + a.coff, dims, str, box, 2)) return rc;
  plan.tmap_a_lo = plan.tmap_a;
  if (a.lo_off)
    if (int rc = encode(ctx, &plan.tmap_a_lo, 4, reinterpret_cast<__half*>(reinterpret_cast<char*>(a.base) + a.lo_off) + a.coff, dims, str, box, 2)) return rc;
  if (int rc = encode_b(ctx, plan, p.block_n, 1)) return rc;
  plan.enabled = true;
  return 0;
}

// Stride-1 plans run on the second-generation kernel (umma_conv_v2.cu): halo layout (one A box per K chunk covers the
// tile plus the filter border, taps = shifted UMMA descriptor views; a 1x1 layer is the halo-free case), several taps per
// weight stage, CTA pairs.  A halo row holds its pixels at their exact pitch (bw + halo pixels).  Measured on B200: the
// UMMA unit applies the 128-byte swizzle to absolute shared-memory address bits, so views that start at any 128-byte row
// of a TMA-written tile read correctly with descriptor base_offset 0 (a non-zero base_offset gives wrong data).
// A plan that this kernel cannot take fails the bind.
// `a2` is the second activation source of a fused sibling data gradient (K chunks >= kchunks_a1), or nullptr.
constexpr int V2_STAGES_MAX = 8;
int bind_halo(UmmaContext& ctx, UmmaConvPlan& plan, View a, int F, const View* a2 = nullptr) {
  UmmaConvParams& p = plan.p;
  auto fail = [](const char* why) { set_thread_error(std::string("umma conv v2: ") + why); return 1; };
  if (a.H != p.H || a.W != p.W) return fail("geometry mismatch");
  if (!umma_conv_v2_supported(p.ntaps)) return fail("no kernel instance for this tap count");
  // the v2 epilogue moves 16 fp16 columns per 256-bit access: rows and channel slices must be 32-byte aligned; its
  // shared-memory bias table holds 1024 columns
  if (p.out_pitch % 16 || p.out_coff % 16 || p.out2_pitch % 16 || p.out2_coff % 16 || p.n_split % 16) return fail("output views are not 32-byte aligned");
  if (p.bias && p.n_tiles * p.block_n > 1024) return fail("more than 1024 bias columns");
  int x0 = 0, x1 = 0, y0 = 0, y1 = 0;
  for (int t = 0; t < p.ntaps; ++t) {
    x0 = std::min(x0, p.tap_dx[t]); x1 = std::max(x1, p.tap_dx[t]);
    y0 = std::min(y0, p.tap_dy[t]); y1 = std::max(y1, p.tap_dy[t]);
  }
  int bh = 8;
  while (bh > 1 && a.H % bh) bh >>= 1;
  const int bw = 8, bf = BLOCK_M / (bw * bh);
  const int pw = bw + (x1 - x0), bhh = bh + (y1 - y0);
  if (bhh > 256 || bf > 256) return fail("box limits");
  // TMA-fed epilogue for data gradients (measured on B200, round 2: 9.82 vs 10.00 ms per training step against the
  // register-prefetch epilogue, 0 mismatching launches in tools/umma_diag.py): a ring of 3 x (old-gradient + activation
  // chunk) at the top of the staging area; the operand rings get what is left
  const bool want_ring = !p.bias && !p.relu && !p.out_f32;
  constexpr int EPI_STAGE = 2 * 128 * 128, EPI_STAGES = 3;
  int pipe = UMMA_V2_PIPE_BYTES - (want_ring ? EPI_STAGES * EPI_STAGE : 0);
  bool ring = want_ring;
retry_without_ring:
  const int b_rows = p.block_n / 2;                         // weight rows each CTA of the pair stages per (tap, K chunk)
  const int a_load_bytes = pw * bf * bhh * BLOCK_K * 2;
  const int a_stage = (a_load_bytes + 1023) / 1024 * 1024;
  const int slab = b_rows * BLOCK_K * 2;                    // one tap of the weight stage (multiple of 1024: rows % 8 == 0)
  int b_taps = 1;
  if (p.ntaps > 1) {                                        // several taps per weight stage: fewer barrier hand-offs per K chunk
    for (int g = p.ntaps; g >= 1; --g)
      if (p.ntaps % g == 0 && g * slab <= 48 * 1024 && 2 * a_stage + 3 * g * slab <= pipe) { b_taps = g; break; }
  }
  const int b_stage = (b_taps * slab + 1023) / 1024 * 1024;
  int a_stages, b_stages;
  if (p.ntaps == 1) {                                       // one box + one slab per step: equal ring depths
    a_stages = b_stages = std::min(V2_STAGES_MAX, pipe / (a_stage + b_stage));
    if (a_stages < 3) { if (ring) { ring = false; pipe = UMMA_V2_PIPE_BYTES; goto retry_without_ring; } return fail("operand stages do not fit"); }
  } else {
    a_stages = 3;
    if ((pipe - 3 * a_stage) / b_stage < 3) a_stages = 2;
    b_stages = (pipe - a_stages * a_stage) / b_stage;
    if (b_stages < 2) { if (ring) { ring = false; pipe = UMMA_V2_PIPE_BYTES; goto retry_without_ring; } return fail("operand stages do not fit"); }
    if (b_stages > V2_STAGES_MAX) b_stages = V2_STAGES_MAX;
  }
  p.v2 = 1; p.b_taps = b_taps;
  p.bw = bw; p.bh = bh; p.bf = bf;
  p.tiles_w = (a.W + bw - 1) / bw; p.tiles_h = (a.H + bh - 1) / bh; p.tiles_f = (F + bf - 1) / bf;
  p.tiles_q = (p.tiles_f + 1) / 2;
  p.a_stages = a_stages; p.b_stages = b_stages; p.a_stage_bytes = a_stage; p.b_stage_bytes = b_stage;
  p.a_load_bytes = a_load_bytes; p.halo_x0 = x0; p.halo_y0 = y0; p.a_sbo = pw * BLOCK_K * 2;
  for (int t = 0; t < p.ntaps; ++t) p.tap_aoff[t] = ((p.tap_dy[t] - y0) * bf * pw + p.tap_dx[t] - x0) * BLOCK_K * 2;
  // halo box: dims {C, W, F, H} so that shared memory holds [y][frame][x][64 ch]
  auto encode_a = [&](CUtensorMap* m, const View& v, int channels) -> int {
    cuuint64_t dims[4] = {(cuuint64_t)channels, (cuuint64_t)v.W, (cuuint64_t)F, (cuuint64_t)v.H};
    cuuint64_t str[3] = {(cuuint64_t)v.pitch * 2, (cuuint64_t)v.H * v.W * v.pitch * 2, (cuuint64_t)v.W * v.pitch * 2};
    cuuint32_t box[4] = {(cuuint32_t)BLOCK_K, (cuuint32_t)pw, (cuuint32_t)bf, (cuuint32_t)bhh};
    return encode(ctx, m, 4, reinterpret_cast<__half*>(v.base) + v.coff, dims, str, box);
  };
  auto lo_of = [](View v) { v.base = reinterpret_cast<char*>(v.base) + v.lo_off; return v; };
  if (int rc = encode_a(&plan.tmap_a, a, p.K1)) return rc;
  plan.tmap_a_lo = plan.tmap_a;
  if (a.lo_off) if (int rc = encode_a(&plan.tmap_a_lo, lo_of(a), p.K1)) return rc;
  if (a2) {
    if (int rc = encode_a(&plan.tmap_a2, *a2, p.K - p.K1)) return rc;
    plan.tmap_a2_lo = plan.tmap_a2;
    if (a2->lo_off) if (int rc = encode_a(&plan.tmap_a2_lo, lo_of(*a2), p.K - p.K1)) return rc;
  } else { plan.tmap_a2 = plan.tmap_a; plan.tmap_a2_lo = plan.tmap_a_lo; }
  p.epi_stages = 0; p.epi_stage_bytes = 0; plan.epi_maps_ready = false; plan.epi_mask_ready = false;
  if (ring) {                                               // TMA-fed epilogue: [128 rows][64 ch] boxes of the output view
    p.epi_stages = EPI_STAGES; p.epi_stage_bytes = EPI_STAGE;
    plan.epi_box[0] = bw; plan.epi_box[1] = bf; plan.epi_box[2] = bh; plan.epi_F = F;
    cuuint64_t od[4] = {(cuuint64_t)p.Cout, (cuuint64_t)p.W, (cuuint64_t)F, (cuuint64_t)p.H};
    cuuint64_t os[3] = {(cuuint64_t)p.out_pitch * 2, (cuuint64_t)p.H * p.W * p.out_pitch * 2, (cuuint64_t)p.W * p.out_pitch * 2};
    cuuint32_t ob[4] = {(cuuint32_t)BLOCK_K, (cuuint32_t)bw, (cuuint32_t)bf, (cuuint32_t)bh};
    if (int rc = encode(ctx, &plan.tmap_old, 4, p.out + p.out_coff, od, os, ob)) return rc;
    plan.tmap_y = plan.tmap_old;
    plan.epi_maps_ready = true;
  } else {
    plan.tmap_old = plan.tmap_a; plan.tmap_y = plan.tmap_a;  // valid descriptors, never dereferenced
  }
  if (int rc = encode_b(ctx, plan, b_rows, b_taps)) return rc;
  plan.enabled = true;
  return 0;
}

}  // namespace

int umma_resolve_encode(UmmaContext& ctx) { return resolve_encode(ctx); }
int umma_encode_f16(UmmaContext& ctx, CUtensorMap* m, int rank, void* addr, const cuuint64_t* dims,
                    const cuuint64_t* strides, const cuuint32_t* box, int spatial_stride) {
  return encode(ctx, m, rank, addr, dims, strides, box, spatial_stride);
}

void umma_context_init(UmmaContext& ctx, bool fp16) { ctx.active = fp16; }
void umma_context_destroy(UmmaContext&) {}

int umma_conv_bind_taps(UmmaContext& ctx, UmmaConvPlan& plan, View in, View out, int F, int cin, int cout, int ntaps,
                        const int* dy, const int* dx, const __half* w_tap_n_k, const float* bias, int relu, const UmmaTcOpts* tc) {
  if (int rc = bind_common(ctx, plan, in, out, F, cin, cout, ntaps, w_tap_n_k, tc)) return rc;
  for (int t = 0; t < ntaps; ++t) { plan.p.tap_dy[t] = dy[t]; plan.p.tap_dx[t] = dx[t]; }
  plan.p.bias = bias; plan.p.relu = relu; plan.p.accumulate = 0;
  return bind_halo(ctx, plan, in, F);
}

int umma_conv_bind_fwd(UmmaContext& ctx, UmmaConvPlan& plan, View in, View out, int F, int cin, int cout, int k, int pad,
                       int stride, const __half* w_tap_n_k, const float* bias, const UmmaTcOpts* tc) {
  if (int rc = bind_common(ctx, plan, in, out, F, cin, cout, k * k, w_tap_n_k, tc)) return rc;
  for (int r = 0; r < k; ++r)
    for (int s = 0; s < k; ++s) { plan.p.tap_dy[r * k + s] = r - pad; plan.p.tap_dx[r * k + s] = s - pad; }
  plan.p.bias = bias; plan.p.relu = 1; plan.p.accumulate = 0;
  return stride == 2 ? bind_strided(ctx, plan, in) : bind_halo(ctx, plan, in, F);
}

int umma_conv_bind_dgrad(UmmaContext& ctx, UmmaConvPlan& plan, View dz, View dx, int F, int cin, int cout, int k, int pad,
                         const __half* w_tap_k_n, int accumulate, const UmmaTcOpts* tc) {
  // dx[p, ci] = sum_{r,s,co} dz[p + (pad-r, pad-s), co] * W[co][ci][r][s] : K = cout, N = cin
  if (int rc = bind_common(ctx, plan, dz, dx, F, cout, cin, k * k, w_tap_k_n, tc)) return rc;
  for (int r = 0; r < k; ++r)
    for (int s = 0; s < k; ++s) { plan.p.tap_dy[r * k + s] = pad - r; plan.p.tap_dx[r * k + s] = pad - s; }
  plan.p.bias = nullptr; plan.p.relu = 0; plan.p.accumulate = accumulate;
  return bind_halo(ctx, plan, dz, F);
}

int umma_conv_bind_fused_fwd(UmmaContext& ctx, UmmaConvPlan& plan, View in, View out1, View out2, int F, int cin, int n1, int n2,
                             const __half* w_n_k, const float* bias, const UmmaTcOpts* tc) {
  // bind as one convolution with N = n1 + n2 writing to out1's geometry, then redirect columns >= n1
  View o = out1; o.C = n1 + n2;
  if (out1.H != out2.H || out1.W != out2.W || n1 % 16 || n2 % 16 || out2.pitch % 8 || out2.coff % 8) { set_thread_error("fused fwd: bad views"); return 1; }
  if (int rc = bind_common(ctx, plan, in, o, F, cin, n1 + n2, 1, w_n_k, tc)) return rc;
  plan.p.tap_dy[0] = 0; plan.p.tap_dx[0] = 0;
  plan.p.bias = bias; plan.p.relu = 1; plan.p.accumulate = 0;
  plan.p.n_split = n1; plan.p.out2 = reinterpret_cast<__half*>(out2.base); plan.p.out2_pitch = out2.pitch; plan.p.out2_coff = out2.coff;
  if (tc) {        // EXACT_TC: out1 / out2 are the operand-plane views of the two destinations, tc->out32 / out32_2 their fp32 buffers
    if (!tc->out32_2) { set_thread_error("fused fwd: the split-operand bind needs both fp32 destinations"); return 1; }
    plan.p.out32_2 = tc->out32_2; plan.p.out_hi2 = reinterpret_cast<__half*>(out2.base); plan.p.out_lo_off2 = out2.lo_off;
  }
  return bind_halo(ctx, plan, in, F);
}

int umma_conv_bind_fused_dgrad(UmmaContext& ctx, UmmaConvPlan& plan, View dz1, View dz2, View dx, int F, int cin, int k1, int k2,
                               const __half* w_n_k, int accumulate, const UmmaTcOpts* tc) {
  const int k1p = (k1 + BLOCK_K - 1) / BLOCK_K * BLOCK_K;
  // bind with the first source as the A view; then attach the second source and the full fused K
  View a = k1 ? dz1 : dz2;
  if (int rc = bind_common(ctx, plan, a, dx, F, k1 ? k1 : k2, cin, 1, w_n_k, tc)) return rc;
  UmmaConvParams& p = plan.p;
  p.tap_dy[0] = 0; p.tap_dx[0] = 0; p.bias = nullptr; p.relu = 0; p.accumulate = accumulate;
  if (k1) {
    if (dz2.H != dz1.H || dz2.W != dz1.W || dz2.pitch % 8 || dz2.coff % 8 || k2 % 8) { set_thread_error("fused dgrad: bad views"); return 1; }
    if (tc && !dz2.lo_off) { set_thread_error("fused dgrad: the split-operand bind needs the second source's operand planes"); return 1; }
    p.kchunks_a1 = k1p / BLOCK_K; p.K1 = k1; p.K = k1 + k2;
    p.kchunks = p.kchunks_a1 + (k2 + BLOCK_K - 1) / BLOCK_K;
    // the weight map covers the padded fused K
    plan.b_dims[0] = k1p + k2; plan.b_dims[1] = cin; plan.b_dims[2] = 1;
    plan.b_strides[0] = (unsigned long long)(k1p + k2) * 2; plan.b_strides[1] = (unsigned long long)cin * (k1p + k2) * 2;
  }
  return bind_halo(ctx, plan, a, F, k1 ? &dz2 : nullptr);
}

int umma_conv_set_mask(UmmaContext& ctx, UmmaConvPlan& plan, View y) {
  // the v2 epilogue reads the activation with 256-bit loads
  if (y.pitch % 16 || y.coff % 16) { set_thread_error("umma conv: the mask activation view is not 32-byte aligned"); return 1; }
  plan.mask_y = reinterpret_cast<const __half*>(y.base); plan.mask_pitch = y.pitch; plan.mask_coff = y.coff;
  plan.epi_mask_ready = false;
  if (plan.epi_maps_ready) {                                 // TMA-fed epilogue: the activation tiles come through TMA too
    cuuint64_t d[4] = {(cuuint64_t)plan.p.Cout, (cuuint64_t)y.W, (cuuint64_t)plan.epi_F, (cuuint64_t)y.H};
    cuuint64_t st[3] = {(cuuint64_t)y.pitch * 2, (cuuint64_t)y.H * y.W * y.pitch * 2, (cuuint64_t)y.W * y.pitch * 2};
    cuuint32_t b[4] = {(cuuint32_t)BLOCK_K, (cuuint32_t)plan.epi_box[0], (cuuint32_t)plan.epi_box[1], (cuuint32_t)plan.epi_box[2]};
    plan.epi_mask_ready = encode(ctx, &plan.tmap_y, 4, reinterpret_cast<__half*>(y.base) + y.coff, d, st, b) == 0;
  }
  return 0;
}

void umma_conv_set_mask_tc(UmmaConvPlan& plan, View y32, View dplanes, float plane_scale, int* flag) {
  plan.mask32 = reinterpret_cast<const float*>(y32.base); plan.mask32_pitch = y32.pitch; plan.mask32_coff = y32.coff;
  plan.mask_planes = reinterpret_cast<__half*>(dplanes.base); plan.mask_planes_lo = dplanes.lo_off;
  plan.mask_plane_scale = plane_scale; plan.mask_flag = flag;
}

int umma_conv_launch(UmmaContext& ctx, const UmmaConvPlan& plan, cudaStream_t s, bool mask) {
  if (!plan.enabled) { set_thread_error("umma conv: plan not bound"); return 3; }
  UmmaConvParams p = plan.p;
  if (mask && plan.mask_y) { p.mask_y = plan.mask_y; p.mask_pitch = plan.mask_pitch; p.mask_coff = plan.mask_coff; }
  if (mask && p.out_f32 && plan.mask32) {
    p.mask32 = plan.mask32; p.mask32_pitch = plan.mask32_pitch; p.mask32_coff = plan.mask32_coff;
    p.out_hi = plan.mask_planes; p.out_lo_off = plan.mask_planes_lo; p.plane_scale = plan.mask_plane_scale; p.flag = plan.mask_flag;
  }
  if (p.v2) return umma_conv_v2_launch(ctx, plan, p, s);
  // stride-2 forward: the first-generation kernel of this file
  if (!ctx.attr_set) {
    if (cudaFuncSetAttribute(umma_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess) {
      set_thread_error("umma conv: cannot raise dynamic shared memory limit"); cudaGetLastError(); return 2; }
    ctx.attr_set = true;
  }
  const int total = p.tiles_w * p.tiles_h * p.tiles_f * p.n_tiles;
  const int grid = total < ctx.num_sms ? total : ctx.num_sms;
  umma_conv_kernel<<<grid, NUM_THREADS, SMEM_BYTES, s>>>(plan.tmap_a, plan.tmap_b, plan.tmap_a_lo, plan.tmap_b_lo, p);
  SSNB_LAUNCH_CHECK("umma_conv_kernel");
  return 0;
}

}  // namespace ssnb
