// tcgen05 implicit-GEMM convolution, second generation (sm_100a): the role loops are written warp-uniformly.
//
// Measured on B200 (round 1, ablation runs): with the MMAs, the epilogue AND every TMA load removed, the first-generation
// kernels (umma_conv.cu) still took 85-90 % of their full time -- the single-thread producer / MMA-issue loops
// (divergent `if (lane == 0)` regions: vector registers, R2UR + vote loops around every UTMALDG / UTCHMMA, runtime
// divisions per tile, dynamically indexed parameter arrays in local memory) bounded the kernel, not memory or the tensor
// pipe.  Here every role loop runs on all 32 lanes with warp-uniform control flow and operands (they live in uniform
// registers), one elected lane issues the asynchronous instructions, tiles advance by mixed-radix carry adds instead of
// divisions, the tap loop is unrolled at compile time (NTAPS is a template parameter) and several taps share one weight
// stage, which divides the number of barrier hand-offs per K chunk.
//
//   layout   halo A boxes (one per K chunk, [y][frame][x][64 ch], taps = shifted UMMA descriptor views; a 1x1 layer
//            is the halo-free case), weight stages of G taps x rows x 64 ch
//   pairs    two CTAs of a cluster split two frame-adjacent M tiles and each stages half of the weight rows; the
//            leader issues M = 256 cta_group::2 MMAs
//   warp 0   TMA producer, warp 1 MMA issuer, warps 2..9 epilogue (TMEM -> bias/ReLU or accumulate/mask -> fp16 NHWC)
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
constexpr int NUM_THREADS = 320;
constexpr int EPI_WARPS = 8;
constexpr int TMEM_COLS = 512;
constexpr int MAX_STAGES = 8;
constexpr int BAR_BYTES = 1024;
constexpr int EPI_RING_MAX = 4;                   // stages of the TMA-fed epilogue ring
constexpr int EPI_TENSOR_BYTES = 128 * 128;        // one [128 rows][64 fp16] chunk of the old gradient or of the activation
constexpr int BIAS_MAX = 1024;                     // floats of folded-BN bias staged in shared memory (n_tiles * block_n)
constexpr int SMEM_BYTES = UMMA_V2_PIPE_BYTES + 1024 /*align slack*/ + BAR_BYTES + BIAS_MAX * 4;

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// Tile walk without divisions: digits (N tile, tile column, tile row, frame group) advance by the digits of the grid
// stride with carries.  The last digit counts PAIRS of frame groups and CTA `rank` of the pair owns group 2*mq + rank.
struct TileIter {
  int nt, mw, mh, mq, sn, sw, sh, sq;
  __device__ __forceinline__ void init(const UmmaConvParams& p, int first, int step) {
    nt = first % p.n_tiles; first /= p.n_tiles; mw = first % p.tiles_w; first /= p.tiles_w; mh = first % p.tiles_h; mq = first / p.tiles_h;
    sn = step % p.n_tiles; step /= p.n_tiles; sw = step % p.tiles_w; step /= p.tiles_w; sh = step % p.tiles_h; sq = step / p.tiles_h;
  }
  __device__ __forceinline__ bool valid(const UmmaConvParams& p) const { return mq < p.tiles_q; }
  __device__ __forceinline__ void next(const UmmaConvParams& p) {
    nt += sn; int c = nt >= p.n_tiles ? 1 : 0; nt -= c ? p.n_tiles : 0;
    mw += sw + c; c = mw >= p.tiles_w ? 1 : 0; mw -= c ? p.tiles_w : 0;
    mh += sh + c; c = mh >= p.tiles_h ? 1 : 0; mh -= c ? p.tiles_h : 0;
    mq += sq + c;
  }
};

// one 16-column chunk of an accumulator row: bias / accumulate / ReLU / ReLU-gradient mask, fp16 store (32 bytes)
template <bool HAS_BIAS>
__device__ __forceinline__ void store_chunk(const UmmaConvParams& p, const uint32_t* r, const float4* bias, __half* dst, const U8& old,
                                            const U8& y) {
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
  if (HAS_BIAS && p.bias) {
#pragma unroll
    for (int j = 0; j < 4; ++j) { v[4 * j] += bias[j].x; v[4 * j + 1] += bias[j].y; v[4 * j + 2] += bias[j].z; v[4 * j + 3] += bias[j].w; }
  }
  if (p.accumulate) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&old.v[j]));
      v[2 * j] += a.x; v[2 * j + 1] += a.y;
    }
  }
  if (HAS_BIAS && p.relu) {                  // (bias and ReLU are the forward epilogue)
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
  }
  U8 q;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const __half2 h = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
    q.v[j] = *reinterpret_cast<const uint32_t*>(&h);
  }
  if (p.mask_y) {
    const __half2 zero = __float2half2_rn(0.f);
#pragma unroll
    for (int j = 0; j < 8; ++j) q.v[j] &= __hgt2_mask(*reinterpret_cast<const __half2*>(&y.v[j]), zero);     // keep where y > 0 (NaN -> 0)
  }
  stg256(dst, q);
}

// register budget: 10 warps on 4 sub-partitions = 3 warps on one of them, 16384 / (3 * 32) = 170 -> ptxas caps at 168
// (a __maxnreg__(200) build compiles but cannot launch); two prefetch buffers fit, three spill
// EPI selects the epilogue: 0 register-prefetch (forward, and data gradients whose operand rings leave no room for the
// epilogue ring); 2 TMA-fed (data gradients that read the old gradient / the mask activation: an eleventh warp streams
// those tiles of every 64-column chunk into a shared-memory ring with TMA, the epilogue warps read them with
// conflict-free LDS instead of scattered global loads; validated and measured on B200 in round 2: -0.18 ms per training step).
// EPI == 3: SSNB_EXACT_TC.  The producer walks every K chunk three times -- (A_lo, B_hi), (A_hi, B_lo), (A_hi, B_hi): the
// error-compensated fp16 product, ~22 significand bits per operand -- and the epilogue works in fp32 (out32 = alpha * acc
// + bias, ReLU | + old) and emits the result's own hi / lo operand planes for the consuming convolutions.
template <int NTAPS, int EPI>
__global__ void __launch_bounds__(EPI == 2 ? NUM_THREADS + 32 : NUM_THREADS, 1)
umma_conv_v2_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_a2,
                    const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_old,
                    const __grid_constant__ CUtensorMap tmap_y, const __grid_constant__ CUtensorMap tmap_a_lo,
                    const __grid_constant__ CUtensorMap tmap_a2_lo, const __grid_constant__ CUtensorMap tmap_b_lo,
                    const __grid_constant__ UmmaConvParams p) {
  constexpr bool TMAE = EPI == 2, TC = EPI == 3;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_b = smem + p.a_stages * p.a_stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + UMMA_V2_PIPE_BYTES);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + MAX_STAGES;
  uint64_t* b_full = a_empty + MAX_STAGES;
  uint64_t* b_empty = b_full + MAX_STAGES;
  uint64_t* tfull_bar = b_empty + MAX_STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* e_full = tempty_bar + 2;               // [EPI_RING_MAX] TMA-fed epilogue ring (EPI == 2)
  uint64_t* e_empty = e_full + EPI_RING_MAX;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(e_empty + EPI_RING_MAX);

  // warp index through a shuffle: provably warp-uniform, so the role branches below are uniform branches and the loop
  // state inside them can live in uniform registers
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x / 32), 0), lane = threadIdx.x % 32;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int first = (int)(blockIdx.x >> 1);
  const int step = (int)(gridDim.x >> 1);
  constexpr bool ONE_RING = NTAPS == 1;        // 1x1 layers: A box and weight slab of a step share one barrier pair

  // folded-BN bias of every output column of this launch, zero past Cout: the epilogue reads it with broadcast LDS
  // (a global __ldg there sat on the critical path right after the TMEM load: half of the epilogue's stall samples)
  float* bias_s = reinterpret_cast<float*>(smem + UMMA_V2_PIPE_BYTES + BAR_BYTES);
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a2)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
    if (TC) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a_lo)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a2_lo)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b_lo)) : "memory");
    }
    for (int i = 0; i < MAX_STAGES; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 2 * EPI_WARPS); }
    if (TMAE) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_old)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_y)) : "memory");
      for (int i = 0; i < EPI_RING_MAX; ++i) { mbar_init(&e_full[i], 1); mbar_init(&e_empty[i], EPI_WARPS); }
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  // Programmatic dependent launch: everything above (barrier init, tensor-map prefetch, TMEM allocation) touches nothing the
  // previous kernel of the stream produced, so it overlaps that kernel's tail; from here on its results are needed.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (p.bias)
    for (int i = threadIdx.x; i < p.n_tiles * p.block_n; i += (TMAE ? NUM_THREADS + 32 : NUM_THREADS)) bias_s[i] = i < p.Cout ? __ldg(p.bias + i) : 0.f;
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer (whole warp, one elected lane issues) =====
    const bool el = elect_one();
    TileIter it; it.init(p, first, step);
    uint32_t as = 0, aph = 0, bs = 0, bph = 0;
    const int rows_b = p.block_n / 2;
    const uint32_t a_tx = 2u * (uint32_t)p.a_load_bytes;           // both CTAs' boxes complete on the leader's barrier
    const uint32_t b_tx = 2u * (uint32_t)(rows_b * p.b_taps) * BLOCK_K * 2;
    const int groups = NTAPS / p.b_taps;
    for (; it.valid(p); it.next(p)) {
      const int w0 = it.mw * p.bw + p.halo_x0, h0 = it.mh * p.bh + p.halo_y0;
      const int f0 = (2 * it.mq + (int)rank) * p.bf;
      const int n0 = it.nt * p.block_n + (int)rank * rows_b;
      const int nseg = TC ? p.nseg : 1;
      for (int seg = 3 - nseg; seg < 3; ++seg)
      for (int kc = 0; kc < p.kchunks; ++kc) {
        const CUtensorMap* bmap = (TC && seg == 1) ? &tmap_b_lo : &tmap_b;
        mbar_wait(&a_empty[as], aph ^ 1);
        if (el) {
          uint8_t* sa = smem + as * p.a_stage_bytes;
          const bool src1 = kc < p.kchunks_a1;
          const CUtensorMap* map = (TC && seg == 0) ? (src1 ? &tmap_a_lo : &tmap_a2_lo) : (src1 ? &tmap_a : &tmap_a2);
          const int c0 = (src1 ? kc : kc - p.kchunks_a1) * BLOCK_K;
          if (leader) mbar_expect_tx(&a_full[as], ONE_RING ? a_tx + b_tx : a_tx);
          const uint32_t bar = mapa_shared(smem_u32(&a_full[as]), 0);
          tma_load_4d_pair(sa, map, bar, c0, w0, f0, h0);
          if (ONE_RING) tma_load_3d_pair(smem_b + as * p.b_stage_bytes, bmap, bar, kc * BLOCK_K, n0, 0);
        }
        if (++as == (uint32_t)p.a_stages) { as = 0; aph ^= 1; }
        if (!ONE_RING) {
          for (int g = 0; g < groups; ++g) {
            mbar_wait(&b_empty[bs], bph ^ 1);
            if (el) {
              uint8_t* sb = smem_b + bs * p.b_stage_bytes;
              if (leader) mbar_expect_tx(&b_full[bs], b_tx);
              tma_load_3d_pair(sb, bmap, mapa_shared(smem_u32(&b_full[bs]), 0), kc * BLOCK_K, n0, g * p.b_taps);
            }
            if (++bs == (uint32_t)p.b_stages) { bs = 0; bph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (whole warp walks the pipeline; one elected lane issues; leader CTA of the pair only) =====
    if (leader) {
      const bool el = elect_one();
      const uint32_t idesc = make_idesc_f16_m(256, p.block_n);
      const uint32_t a_hi = desc_hi_sw128(p.a_sbo), b_hi = desc_hi_sw128(1024);
      const uint32_t a_stage_lo = (uint32_t)p.a_stage_bytes >> 4, b_stage_lo = (uint32_t)p.b_stage_bytes >> 4;
      const uint32_t slab_lo = (uint32_t)(p.block_n / 2 * BLOCK_K * 2) >> 4;     // one tap inside a weight stage
      const uint32_t a_base = desc_lo(smem_u32(smem)), b_base = desc_lo(smem_u32(smem_b));
      const int btaps = p.b_taps;
      uint32_t as = 0, aph = 0, bs = 0, bph = 0, acc = 0, acc_phase = 0;
      TileIter it; it.init(p, first, step);
      for (; it.valid(p); it.next(p)) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 256;
        const int nseg = TC ? p.nseg : 1;
        for (int seg = 0; seg < nseg; ++seg)
        for (int kc = 0; kc < p.kchunks; ++kc) {
          mbar_wait(&a_full[as], aph);
          tc_fence_after();
          const uint32_t a_lo0 = a_base + as * a_stage_lo;
          const int kvalid = kc < p.kchunks_a1 ? p.K1 - kc * BLOCK_K : p.K - p.K1 - (kc - p.kchunks_a1) * BLOCK_K;
          const int nk = kvalid >= BLOCK_K ? BLOCK_K / UMMA_K : (kvalid + UMMA_K - 1) / UMMA_K;
          uint32_t b_lo = ONE_RING ? b_base + as * b_stage_lo : 0u;
          int gi = 0;                                             // tap index inside the current weight stage
#pragma unroll
          for (int tap = 0; tap < NTAPS; ++tap) {
            if (!ONE_RING && gi == 0) {
              mbar_wait(&b_full[bs], bph);
              tc_fence_after();
              b_lo = b_base + bs * b_stage_lo;
            }
            if (el) {
              const uint32_t a_lo = a_lo0 + ((uint32_t)p.tap_aoff[tap] >> 4);
#pragma unroll
              for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                if (k < nk) umma_f16_lohi_pair(d_tmem, a_lo + 2 * k, a_hi, b_lo + 2 * k, b_hi, idesc, (seg | kc | tap | k) ? 1u : 0u);
            }
            b_lo += slab_lo;
            if (!ONE_RING && ++gi == btaps) {
              gi = 0;
              if (el) umma_commit_pair(&b_empty[bs]);
              if (++bs == (uint32_t)p.b_stages) { bs = 0; bph ^= 1; }
            }
          }
          if (el) umma_commit_pair(&a_empty[as]);
          if (++as == (uint32_t)p.a_stages) { as = 0; aph ^= 1; }
        }
        if (el) umma_commit_pair(&tfull_bar[acc]);
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (!TMAE || warp < 2 + EPI_WARPS) {
    // ===== epilogue warps 2..9: TMEM lane quadrant = warp % 4 =====
    const int quad = warp & 3;
    const int cpar = (warp - 2) >> 2;
    const int row = quad * 32 + lane;
    const int rw = row % p.bw, rf = (row / p.bw) % p.bf, rh = row / (p.bw * p.bf);      // halo row order: x, frame, y
    uint32_t acc = 0, acc_phase = 0;
    uint32_t es = 0, eph = 0;                                       // TMA-fed epilogue ring position (EPI == 2)
    const uint8_t* epi_ring = smem + UMMA_V2_PIPE_BYTES - p.epi_stages * p.epi_stage_bytes;
    TileIter it; it.init(p, first, step);
    // every thread stores its own accumulator row, 32 bytes per 16 columns; the two warps of a quadrant alternate
    // 32-column groups.  (A shared-memory transposed, fully coalesced variant was measured slower -- 13.6 vs 12.3 ms per
    // training step -- and removed; see profiles/README.md.)
    for (; it.valid(p); it.next(p)) {
      const int w = it.mw * p.bw + rw, h = it.mh * p.bh + rh;
      const int f = (2 * it.mq + (int)rank) * p.bf + rf;
      const int n0 = it.nt * p.block_n;
      const bool valid = (rh < p.bh) && (w < p.W) && (h < p.H) && (f < p.F);
      const long long opix = (long long)(f * p.H + h) * p.W + w;
      __half* orow = p.out + opix * p.out_pitch + p.out_coff;
      __half* orow2 = p.out2 + opix * p.out2_pitch + p.out2_coff - p.n_split;
      const __half* mrow = p.mask_y ? p.mask_y + opix * p.mask_pitch + p.mask_coff : nullptr;
      // Global operands of the epilogue (old gradient to accumulate into, activation for the ReLU-gradient mask) are
      // software-pipelined: the loads of column group i+1 go out before group i is processed, and those of a tile's
      // first group before the wait for its accumulator, so their DRAM/L2 latency overlaps the MMAs and the TMEM reads.
      struct Pre { U8 oa, ob, ya, yb; };
      auto prefetch = [&](int c0, Pre& q) {
        const bool two = c0 + 16 < p.block_n;
        const int cola = n0 + c0, colb = cola + 16;
        const bool va = valid && cola < p.Cout, vb = two && valid && colb < p.Cout;
        if (p.accumulate) {
          if (va) q.oa = ldg256((cola < p.n_split ? orow : orow2) + cola);
          if (vb) q.ob = ldg256((colb < p.n_split ? orow : orow2) + colb);
        }
        if (mrow) {
          if (va) q.ya = ldg256_nc(mrow + cola);
          if (vb) q.yb = ldg256_nc(mrow + colb);
        }
      };
      if (TC) {
        // ---- SSNB_EXACT_TC: fp32 epilogue (no software pipelining of the old-gradient reads yet) ----
        float* orow32 = p.out32 + opix * p.out_pitch + p.out_coff;
        __half* hrow = p.out_hi ? p.out_hi + opix * p.out_pitch + p.out_coff : nullptr;
        // fused sibling forward: columns >= n_split belong to the second destination (its own pitch / channel offset)
        float* orow32_2 = p.out32_2 + opix * p.out2_pitch + p.out2_coff - p.n_split;
        __half* hrow2 = p.out_hi2 ? p.out_hi2 + opix * p.out2_pitch + p.out2_coff - p.n_split : nullptr;
        const float alpha = p.alpha * (p.alpha_dev ? __ldg(p.alpha_dev) : 1.0f);
        const float* mrow32 = p.mask32 ? p.mask32 + opix * p.mask32_pitch + p.mask32_coff : nullptr;
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + acc * 256 + ((uint32_t)(quad * 32) << 16);
        if (cpar * 32 >= p.block_n) {                                    // narrow tile: this warp has no columns, release at once
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(&tempty_bar[acc], 0);
        }
        for (int c0 = cpar * 32; c0 < p.block_n; c0 += 64) {
          const bool two = c0 + 16 < p.block_n;                     // warp-uniform
          const int cola = n0 + c0, colb = cola + 16;
          uint32_t ra[16], rb[16];
          tmem_ld16(taddr + c0, ra);
          if (two) tmem_ld16(taddr + c0 + 16, rb);
          tmem_ld_wait();
          if (c0 + 64 >= p.block_n) {                               // last TMEM read of this tile: hand the accumulator back early
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&tempty_bar[acc], 0);
          }
          if (valid && cola < p.Cout) {
            const bool d1 = cola < p.n_split;
            store_chunk32(p, alpha, ra, bias_s + cola, (d1 ? orow32 : orow32_2) + cola, d1 ? (hrow ? hrow + cola : nullptr) : (hrow2 ? hrow2 + cola : nullptr),
                          mrow32 ? mrow32 + cola : nullptr, d1 ? p.out_lo_off : p.out_lo_off2);
          }
          if (two && valid && colb < p.Cout) {
            const bool d1 = colb < p.n_split;
            store_chunk32(p, alpha, rb, bias_s + colb, (d1 ? orow32 : orow32_2) + colb, d1 ? (hrow ? hrow + colb : nullptr) : (hrow2 ? hrow2 + colb : nullptr),
                          mrow32 ? mrow32 + colb : nullptr, d1 ? p.out_lo_off : p.out_lo_off2);
          }
        }
      } else if (TMAE) {
        // ---- TMA-fed: the operands of 64-column chunk i of this tile are in ring stage `es` (old gradient at +0, activation
        //      at +16 KiB, rows in TMEM lane order, 128-byte rows with the TMA 128-byte swizzle) ----
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + acc * 256 + ((uint32_t)(quad * 32) << 16);
        if (cpar * 32 >= p.block_n) {                                    // narrow tile: this warp has no columns, release at once
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(&tempty_bar[acc], 0);
        }
        const int nchunks = (p.block_n + 63) / 64;
        for (int i = 0; i < nchunks; ++i) {
          const int c0 = i * 64 + cpar * 32;
          mbar_wait(&e_full[es], eph);
          const uint8_t* st = epi_ring + es * p.epi_stage_bytes + row * 128;
          const int sw = row & 7, j0 = cpar * 4;                    // 16-byte chunk index of this warp's first column inside the 64
          U8 oa = {}, ob = {}, ya = {}, yb = {};
          auto lds32 = [&](const uint8_t* base, int j, U8& q) {     // 16 columns = two swizzled 16-byte chunks
            const uint4 lo = *reinterpret_cast<const uint4*>(base + ((j ^ sw) << 4));
            const uint4 hi = *reinterpret_cast<const uint4*>(base + (((j + 1) ^ sw) << 4));
            q.v[0] = lo.x; q.v[1] = lo.y; q.v[2] = lo.z; q.v[3] = lo.w; q.v[4] = hi.x; q.v[5] = hi.y; q.v[6] = hi.z; q.v[7] = hi.w;
          };
          if (p.accumulate) { lds32(st, j0, oa); lds32(st, j0 + 2, ob); }
          if (mrow) { lds32(st + EPI_TENSOR_BYTES, j0, ya); lds32(st + EPI_TENSOR_BYTES, j0 + 2, yb); }
          __syncwarp();
          if (lane == 0) mbar_arrive(&e_empty[es]);                 // release semantics order the shared loads above before it
          if (++es == (uint32_t)p.epi_stages) { es = 0; eph ^= 1; }
          if (c0 < p.block_n) {
            const bool two = c0 + 16 < p.block_n;                   // warp-uniform
            const int cola = n0 + c0, colb = cola + 16;
            const bool va = valid && cola < p.Cout, vb = two && valid && colb < p.Cout;
            float4 ba[4] = {}, bb[4] = {};
            uint32_t ra[16], rb[16];
            tmem_ld16(taddr + c0, ra);
            if (two) tmem_ld16(taddr + c0 + 16, rb);
            tmem_ld_wait();
            if (c0 + 64 >= p.block_n) {                             // last TMEM read of this tile: hand the accumulator back early
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(&tempty_bar[acc], 0);
            }
            if (va) store_chunk<false>(p, ra, ba, orow + cola, oa, ya);
            if (vb) store_chunk<false>(p, rb, bb, orow + colb, ob, yb);
          }
        }
      } else {
        // two rotating prefetch buffers (a third spills under the 168-register cap: measured no faster)
        constexpr int NB = 2;
        Pre pp[NB] = {};                                               // indices are compile-time after unrolling: no register copies
        if (cpar * 32 < p.block_n) prefetch(cpar * 32, pp[0]);
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + acc * 256 + ((uint32_t)(quad * 32) << 16);
        if (cpar * 32 >= p.block_n) {                                      // narrow tile: this warp has no columns, release at once
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(&tempty_bar[acc], 0);
        }
        for (int cbase = cpar * 32; cbase < p.block_n; cbase += 64 * NB) {
  #pragma unroll
          for (int u = 0; u < NB; ++u) {
            const int c0 = cbase + 64 * u;
            if (c0 < p.block_n) {
              // one 32-column group: prefetch the operands of a later group, then TMEM -> registers -> epilogue math
              const bool two = c0 + 16 < p.block_n;                   // warp-uniform
              const int cola = n0 + c0, colb = cola + 16;
              const bool va = valid && cola < p.Cout, vb = two && valid && colb < p.Cout;
              __half* da = (cola < p.n_split ? orow : orow2) + cola;
              __half* db2 = (colb < p.n_split ? orow : orow2) + colb;
              if (c0 + 64 * (NB - 1) < p.block_n) prefetch(c0 + 64 * (NB - 1), pp[(u + NB - 1) % NB]);
              float4 ba[4], bb[4];
              if (p.bias) {
  #pragma unroll
                for (int j = 0; j < 4; ++j) {
                  ba[j] = *reinterpret_cast<const float4*>(bias_s + cola + 4 * j);
                  bb[j] = *reinterpret_cast<const float4*>(bias_s + (two ? colb : cola) + 4 * j);
                }
              }
              uint32_t ra[16], rb[16];
              tmem_ld16(taddr + c0, ra);
              if (two) tmem_ld16(taddr + c0 + 16, rb);
              tmem_ld_wait();
              if (c0 + 64 >= p.block_n) {                             // last TMEM read of this tile: hand the accumulator back early
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(&tempty_bar[acc], 0);
              }
              if (va) store_chunk<true>(p, ra, ba, da, pp[u].oa, pp[u].ya);
              if (vb) store_chunk<true>(p, rb, bb, db2, pp[u].ob, pp[u].yb);
            }
          }
        }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else {
    // ===== epilogue loader (EPI == 2, warp 10): old-gradient / activation chunks of every tile, ring of p.epi_stages =====
    const bool el = elect_one();
    uint8_t* epi_ring = smem + UMMA_V2_PIPE_BYTES - p.epi_stages * p.epi_stage_bytes;
    const uint32_t tx = (p.accumulate ? (uint32_t)EPI_TENSOR_BYTES : 0u) + (p.mask_y ? (uint32_t)EPI_TENSOR_BYTES : 0u);
    const int nchunks = (p.block_n + 63) / 64;
    uint32_t es = 0, eph = 0;
    TileIter it; it.init(p, first, step);
    for (; it.valid(p); it.next(p)) {
      const int w0 = it.mw * p.bw, h0 = it.mh * p.bh;
      const int f0 = (2 * it.mq + (int)rank) * p.bf;
      const int n0 = it.nt * p.block_n;
      for (int i = 0; i < nchunks; ++i) {
        mbar_wait(&e_empty[es], eph ^ 1);
        if (el) {
          uint8_t* st = epi_ring + es * p.epi_stage_bytes;
          if (tx) {
            mbar_expect_tx(&e_full[es], tx);
            if (p.accumulate) tma_load_4d(st, &tmap_old, &e_full[es], n0 + i * 64, w0, f0, h0);
            if (p.mask_y) tma_load_4d(st + EPI_TENSOR_BYTES, &tmap_y, &e_full[es], n0 + i * 64, w0, f0, h0);
          } else {
            mbar_arrive(&e_full[es]);
          }
        }
        if (++es == (uint32_t)p.epi_stages) { es = 0; eph ^= 1; }
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

template <int NTAPS, int EPI>
int launch_one(const UmmaConvPlan& plan, const UmmaConvParams& p, int num_sms, cudaStream_t s) {
  static bool attr_set[64] = {};          // function attributes are per device
  auto kern = umma_conv_v2_kernel<NTAPS, EPI>;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess) {
      set_thread_error("umma conv v2: cannot raise dynamic shared memory limit"); cudaGetLastError(); return 2; }
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  const int total = p.n_tiles * p.tiles_w * p.tiles_h * p.tiles_q;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[2];
  cfg.blockDim = dim3(EPI == 2 ? NUM_THREADS + 32 : NUM_THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = s;
  const int pairs = std::min(total, num_sms / 2);
  cfg.gridDim = dim3(2 * pairs);
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  // programmatic dependent launch: this kernel's prologue may overlap the previous kernel's tail
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization; attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 2;
  if (cudaLaunchKernelEx(&cfg, kern, plan.tmap_a, plan.tmap_a2, plan.tmap_b, plan.tmap_old, plan.tmap_y, plan.tmap_a_lo, plan.tmap_a2_lo,
                         plan.tmap_b_lo, p) != cudaSuccess) {
    set_thread_error(std::string("umma_conv_v2_kernel launch: ") + cudaGetErrorString(cudaGetLastError())); return 2; }
  return 0;
}

template <int EPI>
int launch_taps(const UmmaConvPlan& plan, const UmmaConvParams& p, int num_sms, cudaStream_t s) {
  if (p.ntaps == 1) return launch_one<1, EPI>(plan, p, num_sms, s);
  if (p.ntaps == 4) return launch_one<4, EPI>(plan, p, num_sms, s);
  return launch_one<9, EPI>(plan, p, num_sms, s);
}

}  // namespace

bool umma_conv_v2_supported(int ntaps) { return ntaps == 1 || ntaps == 4 || ntaps == 9; }

int umma_conv_v2_launch(UmmaContext& ctx, const UmmaConvPlan& plan, const UmmaConvParams& p, cudaStream_t s) {
  // data gradients whose epilogue reads global operands (old gradient / activation) and whose plan was bound with the
  // shared-memory ring (p.epi_stages > 0) take the TMA-fed epilogue
  const bool reads = !p.bias && !p.relu && (p.accumulate || p.mask_y);
  const int epi = p.out_f32 ? 3 : ((reads && p.epi_stages > 0 && plan.epi_maps_ready && (!p.mask_y || plan.epi_mask_ready)) ? 2 : 0);
  if (p.out_f32 && p.mask_y) { set_thread_error("umma conv v2: the fp32 epilogue takes its mask through mask32"); return 3; }
  const int rc = epi == 3 ? launch_taps<3>(plan, p, ctx.num_sms, s)
               : epi == 2 ? launch_taps<2>(plan, p, ctx.num_sms, s) : launch_taps<0>(plan, p, ctx.num_sms, s);
  if (rc) return rc;
  SSNB_LAUNCH_CHECK("umma_conv_v2_kernel");
  return 0;
}

}  // namespace ssnb
