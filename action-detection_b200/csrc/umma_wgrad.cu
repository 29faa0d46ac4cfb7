// tcgen05 weight-gradient kernel (sm_100a).  dW[tap][co][ci] = sum_p dz[p, co] * x[p + shift(tap), ci]
// is a GEMM whose reduction runs over pixels, so both operands are MN-major in shared memory:
// a TMA box is [64 pixels][64 channels] (128-byte rows, SWIZZLE_128B) and the UMMA descriptors walk
// it with 8-pixel groups every 1024 B (SBO) and 64-channel atoms every 8 KiB (LBO).
//
//   CTA = (co tile of 128, ci tile of block_n <= 256, tap, pixel split); K loop over 64-pixel boxes.
//   warp 0: TMA producer, warp 1: MMA issuer (M=128, N=block_n, fp32 TMEM accumulator),
//   warps 2..5: epilogue -> split-K partials (reduced in fixed order by wgrad_finalize_kernel).
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <algorithm>

#include "umma_conv.cuh"
#include "umma_dev.cuh"

namespace ssnb {
namespace {

using namespace umma;
constexpr int MAX_STAGES = 8;
constexpr int BOX_BYTES = 64 * 128;                 // [64 px][64 ch] fp16
constexpr int A_BYTES = 2 * BOX_BYTES;              // 128 output channels
constexpr int PIPE_BYTES = 4 * (A_BYTES + 4 * BOX_BYTES);   // 192 KiB of operand staging
constexpr int NUM_THREADS = 192;
constexpr int ONES_OFF = PIPE_BYTES + 1024;                // [64 px][64 ch] tile of fp16 ones (bias-gradient operand), 1 KiB aligned
constexpr int SMEM_BYTES = PIPE_BYTES + 1024 /*align slack*/ + 1024 /*barriers*/ + BOX_BYTES;

__global__ void __launch_bounds__(NUM_THREADS, 1)
umma_wgrad_kernel(const __grid_constant__ CUtensorMap tmap_dz, const __grid_constant__ CUtensorMap tmap_x,
                  const __grid_constant__ CUtensorMap tmap_dz_lo, const __grid_constant__ CUtensorMap tmap_x_lo,
                  const UmmaWgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int STAGES = p.stages, STAGE_BYTES = p.stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + PIPE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + MAX_STAGES;
  uint64_t* tfull_bar = bars + 2 * MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 1);

  // warp index through a shuffle (provably warp-uniform): the role loops below run on all 32 lanes with uniform control
  // flow, one elected lane issues the TMA / MMA instructions (see umma_conv_v2.cu for the measurements behind this)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x / 32), 0), lane = threadIdx.x % 32;
  int id = blockIdx.x;
  const int tgrp = id % p.tap_groups; id /= p.tap_groups;
  const int nt = id % p.n_tiles; id /= p.n_tiles;
  const int mt = id;
  const int tap0 = tgrp * p.taps_per_cta;
  const int ntap = min(p.taps_per_cta, p.ntaps - tap0);        // taps handled by this CTA (share the dz tile)
  const int split = blockIdx.y;
  const int m0 = mt * BLOCK_M, n0 = nt * p.block_n;
  const int ptiles = p.tiles_w * p.tiles_h * p.tiles_f;
  const int pt0 = split * p.ptiles_per_split;
  const int pt1 = min(pt0 + p.ptiles_per_split, ptiles);
  const int nboxes_b = p.block_n / 64;
  const bool run = p.run_len > 1;                  // halo x box, the CTA's taps taken by one MMA (see umma_wgrad_bind_taps)
  // CTAs of the first input tile / tap group also reduce dz over pixels: db[co] = sum_p dz[p, co] = dz^T * 1
  const bool do_bias = p.bias_partial != nullptr && nt == 0 && tgrp == 0;
  const int bias_col = p.taps_per_cta * p.mma_n;
  const int acc_cols = p.taps_per_cta * p.mma_n + (p.bias_partial ? 16 : 0);
  const uint32_t tmem_cols = acc_cols <= 32 ? 32 : (acc_cols <= 64 ? 64 : (acc_cols <= 128 ? 128 : (acc_cols <= 256 ? 256 : 512)));

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_dz)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_x)) : "memory");
    for (int i = 0; i < MAX_STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(tfull_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (do_bias) {
    uint32_t* ones = reinterpret_cast<uint32_t*>(smem + ONES_OFF);
    for (int i = threadIdx.x; i < BOX_BYTES / 4; i += NUM_THREADS) ones[i] = 0x3C003C00u;     // half2(1, 1)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy writes -> visible to the tensor core
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");       // programmatic dependent launch: the prologue above overlapped the previous kernel's tail
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    const bool el = elect_one_lane();
    uint32_t stage = 0, phase = 0;
    const uint32_t tx_bytes = run ? (uint32_t)(2 * BOX_BYTES + nboxes_b * p.x_box_tx) : (uint32_t)(2 + nboxes_b * ntap) * BOX_BYTES;
    // pixel-tile coordinates advance by carries (no divisions in the loop)
    int tw = pt0 % p.tiles_w, th = (pt0 / p.tiles_w) % p.tiles_h, tf = pt0 / (p.tiles_w * p.tiles_h);
    for (int pt = pt0; pt < pt1; ++pt) {
      const int w0 = tw * p.bw, h0 = th * p.bh, f0 = tf * p.bf;
      // SSNB_EXACT_TC (nseg = 3): the tile is staged three times, (dz_lo, x_hi), (dz_hi, x_lo), (dz_hi, x_hi)
      for (int seg = 3 - p.nseg; seg < 3; ++seg) {
      const CUtensorMap* mdz = seg == 0 ? &tmap_dz_lo : &tmap_dz;
      const CUtensorMap* mx = seg == 1 ? &tmap_x_lo : &tmap_x;
      mbar_wait(&empty_bar[stage], phase ^ 1);
      if (el) {
        uint8_t* sa = smem + stage * STAGE_BYTES;
        uint8_t* sb = sa + A_BYTES;
        mbar_expect_tx(&full_bar[stage], tx_bytes);
        if (run) {
          // halo layout: tensor-map dims {C, W, F, H}; ONE x box per 64 input channels covers the tile plus the filter
          // border, every tap of this CTA is a shifted descriptor view into it
          tma_load_4d(sa, mdz, &full_bar[stage], m0, w0, f0, h0);
          tma_load_4d(sa + BOX_BYTES, mdz, &full_bar[stage], m0 + 64, w0, f0, h0);
          for (int b = 0; b < nboxes_b; ++b)
            tma_load_4d(sb + b * p.x_box_bytes, mx, &full_bar[stage], n0 + b * 64, w0 + p.halo_x0, f0, h0 + p.halo_y0);
        } else {
          tma_load_4d(sa, mdz, &full_bar[stage], m0, w0, h0, f0);
          tma_load_4d(sa + BOX_BYTES, mdz, &full_bar[stage], m0 + 64, w0, h0, f0);
          for (int t = 0; t < ntap; ++t)
            for (int b = 0; b < nboxes_b; ++b)
              tma_load_4d(sb + (t * nboxes_b + b) * BOX_BYTES, mx, &full_bar[stage], n0 + b * 64,
                          w0 * p.x_stride + p.tap_dx[tap0 + t], h0 * p.x_stride + p.tap_dy[tap0 + t], f0);
        }
      }
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (++tw == p.tiles_w) { tw = 0; if (++th == p.tiles_h) { th = 0; ++tf; } }
    }
  } else if (warp == 1) {
    const bool el = elect_one_lane();
    const uint32_t idesc = make_idesc_f16_mn(p.mma_n), idesc_bias = make_idesc_f16_mn(16), idesc_run = make_idesc_f16_mn(ntap * p.mma_n);
    // descriptors as (lo, hi) words: hi constant (SBO 1024, version, SWIZZLE_128B), lo = address >> 4 | LBO field
    const uint32_t hi = desc_hi_sw128(1024);
    const uint32_t lbo = (uint32_t)((BOX_BYTES >> 4) & 0x3FFF) << 16;
    const uint32_t base_lo = ((smem_u32(smem) >> 4) & 0x3FFF) | lbo;
    const uint32_t ones_lo = ((smem_u32(smem + ONES_OFF) >> 4) & 0x3FFF) | lbo;
    const uint32_t kstep_lo = (UMMA_K * 128) >> 4;                    // 16 pixel rows
    // x operand of a tap run: views into the halo box, 8-pixel row groups x_sbo bytes apart
    const uint32_t hi_x = desc_hi_sw128(p.x_sbo);
    const uint32_t kstep_x = (uint32_t)(2 * p.x_sbo) >> 4;
    uint32_t stage = 0, phase = 0;
    for (int pt = pt0; pt < pt1; ++pt)
    for (int seg = 3 - p.nseg; seg < 3; ++seg) {
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      const uint32_t sa_lo = base_lo + stage * ((uint32_t)STAGE_BYTES >> 4);
      const uint32_t sb_lo = ((sa_lo + (A_BYTES >> 4)) & 0xFFFFu) | lbo;
      if (el) {
        const uint32_t first = (pt > pt0 || seg > 3 - p.nseg) ? 1u : 0u;
        if (run) {
          // the taps of this CTA form ONE run whose views are `run_stride` bytes apart: a single MMA takes them as
          // consecutive 64-channel N atoms (LBO = run_stride), so the dz tile is read once per K step instead of once
          // per tap (the kernel is bound by those shared-memory reads)
          const uint32_t xb_lo = (sb_lo & 0xFFFFu) + ((uint32_t)p.tap_xoff[tap0] >> 4) + (((uint32_t)p.run_stride >> 4) << 16);
#pragma unroll
          for (int k = 0; k < 64 / UMMA_K; ++k)
            umma_f16_lohi(tmem_base, sa_lo + k * kstep_lo, hi, xb_lo + k * kstep_x, hi_x, idesc_run, first | (uint32_t)k);
        } else {
          // classic layout: one [64 px][64 ch] box per (tap, 64 channels)
          for (int t = 0; t < ntap; ++t) {
            const uint32_t xb_lo = sb_lo + (uint32_t)(t * nboxes_b) * (BOX_BYTES >> 4);
#pragma unroll
            for (int k = 0; k < 64 / UMMA_K; ++k)      // 16 pixel rows (2 groups of 8) per instruction
              umma_f16_lohi(tmem_base + t * p.mma_n, sa_lo + k * kstep_lo, hi, xb_lo + k * kstep_lo, hi, idesc, first | (uint32_t)k);
          }
        }
        if (do_bias && seg != 1) {          // column sums of dz: hi and lo planes once each (seg 1 re-stages dz_hi against x_lo)
#pragma unroll
          for (int k = 0; k < 64 / UMMA_K; ++k)
            umma_f16_lohi(tmem_base + bias_col, sa_lo + k * kstep_lo, hi, ones_lo + k * kstep_lo, hi, idesc_bias, first | (uint32_t)k);
        }
        umma_commit(&empty_bar[stage]);
      }
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
    if (el) umma_commit(tfull_bar);
    __syncwarp();
  } else {
    const int quad = warp & 3;
    const int m = m0 + quad * 32 + lane;            // output channel of this thread's accumulator row
    mbar_wait(tfull_bar, 0);
    tc_fence_after();
    const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16);
    for (int t = 0; t < ntap; ++t) {
      float* orow = p.partial + (((long long)split * p.ntaps + tap0 + t) * p.Cout + m) * p.Cin + n0;
      for (int c0 = 0; c0 < p.mma_n; c0 += 16) {
        uint32_t r[16];
        tmem_ld16(taddr + t * p.mma_n + c0, r);
        tmem_ld_wait();
        if (m < p.Cout) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            if (n0 + c0 + j < p.Cin)      // Cin is a multiple of 4
              *reinterpret_cast<float4*>(orow + c0 + j) = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                                                      __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
          }
        }
      }
    }
    if (do_bias) {
      uint32_t r[16];
      tmem_ld16(taddr + bias_col, r);
      tmem_ld_wait();
      if (m < p.Cout) p.bias_partial[(long long)split * p.Cout + m] = __uint_as_float(r[0]);
    }
    tc_fence_before();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

}  // namespace

int umma_wgrad_bind(UmmaContext& ctx, UmmaWgradPlan& plan, View dz, View x, int F, int cin, int cout, int k, int pad,
                    float* partial, int max_splits, int x_stride) {
  int dy[UMMA_MAX_TAPS], dx[UMMA_MAX_TAPS];
  if (k * k > UMMA_MAX_TAPS) { set_thread_error("umma wgrad: too many taps"); return 1; }
  for (int r = 0; r < k; ++r)
    for (int s = 0; s < k; ++s) { dy[r * k + s] = r - pad; dx[r * k + s] = s - pad; }
  return umma_wgrad_bind_taps(ctx, plan, dz, x, F, cin, cout, k * k, dy, dx, partial, max_splits, x_stride);
}

int umma_wgrad_bind_taps(UmmaContext& ctx, UmmaWgradPlan& plan, View dz, View x, int F, int cin, int cout, int ntaps,
                         const int* tdy, const int* tdx, float* partial, int max_splits, int x_stride) {
  plan.enabled = false;
  if (int rc = umma_resolve_encode(ctx)) return rc;
  if (dz.H != (x.H + x_stride - 1) / x_stride || dz.W != (x.W + x_stride - 1) / x_stride) { set_thread_error("umma wgrad: geometry mismatch"); return 1; }
  if (cin % 8 || cout % 8 || dz.pitch % 8 || dz.coff % 8 || x.pitch % 8 || x.coff % 8 || ntaps > UMMA_MAX_TAPS) {
    set_thread_error("umma wgrad: unsupported channel alignment"); return 1; }
  UmmaWgradParams& p = plan.p;
  memset(&p, 0, sizeof(p));
  p.W = dz.W; p.H = dz.H; p.F = F; p.x_stride = x_stride;     // tiles enumerate dz (output) pixels
  // 64-pixel boxes whose rows are all real-or-zero-filled pixels (the pixel index is the reduction dim)
  if (dz.W % 8 == 0) { p.bw = 8; p.bh = 8; p.bf = 1; }
  else if (dz.W % 4 == 0) { p.bw = 4; p.bh = 4; p.bf = 4; }
  else if (dz.W % 2 == 0) { p.bw = 2; p.bh = 2; p.bf = 16; }
  else { p.bw = 1; p.bh = 1; p.bf = 64; }
  p.tiles_w = (dz.W + p.bw - 1) / p.bw; p.tiles_h = (dz.H + p.bh - 1) / p.bh; p.tiles_f = (F + p.bf - 1) / p.bf;
  p.ntaps = ntaps;
  for (int t = 0; t < ntaps; ++t) { p.tap_dy[t] = tdy[t]; p.tap_dx[t] = tdx[t]; }
  p.Cout = cout; p.Cin = cin;
  p.m_tiles = (cout + BLOCK_M - 1) / BLOCK_M;
  const int chunks = (cin + 63) / 64;
  p.n_tiles = (chunks + 3) / 4;
  p.block_n = ((chunks + p.n_tiles - 1) / p.n_tiles) * 64;
  // several taps per CTA share one dz tile: stage = 2 dz boxes + taps * (block_n/64) x boxes <= 6 boxes, and
  // the accumulators (taps * mma_n fp32 columns) must fit the 512 TMEM columns
  p.mma_n = p.block_n;
  if (p.n_tiles == 1 && cin < p.block_n) p.mma_n = (cin + 15) / 16 * 16;     // narrow inputs (conv1 space-to-depth: 16)
  // Tap runs (stride-1 multi-tap 64-channel layers): ONE x box per 64 input channels covers the 64-pixel tile plus the
  // filter border ([y][frame][x] pixel order, as in umma_conv_v2.cu) and every tap is a shifted descriptor view into it.
  // Where the views of a whole ROW of taps are equally spaced they are consecutive 64-channel N atoms with LBO = the tap
  // spacing (128 B for a 3x3 row, 1 KiB for conv1's four vertical taps), so a single MMA takes the run.  That reads the
  // 4 KiB dz tile once per K step instead of once per tap, which is what bounds this kernel (shared-memory bandwidth):
  // conv2_3x3 283 -> 163 us, conv1 254 -> 148 us.  Without the run the halo layout is SLOWER than per-tap boxes (more
  // taps per CTA, same dz re-reads: 3.7 vs 2.9 ms over the 69 layers), so every other layer keeps the classic layout.
  int x0 = 0, x1 = 0, y0 = 0, y1 = 0;
  for (int t = 0; t < ntaps; ++t) { x0 = std::min(x0, tdx[t]); x1 = std::max(x1, tdx[t]); y0 = std::min(y0, tdy[t]); y1 = std::max(y1, tdy[t]); }
  int hbh = 8;
  while (hbh > 1 && dz.H % hbh) hbh >>= 1;
  const int hbw = 8, hbf = 64 / (hbw * hbh), pw = hbw + (x1 - x0);
  auto off = [&](int t) { return ((tdy[t] - y0) * hbf * pw + (tdx[t] - x0)) * 128; };
  int run_len = 1, run_stride = 0;
  if (x_stride == 1 && ntaps > 1 && dz.W >= 7 && p.block_n == 64 && p.mma_n == 64) {
    for (int r = 4; r >= 2; --r) {                      // longest run length (N = r*64 <= 256) that tiles the tap list evenly
      if (ntaps % r) continue;
      bool ok = true;
      const int st = off(1) - off(0);
      for (int g = 0; g < ntaps / r && ok; ++g)
        for (int i = 1; i < r && ok; ++i) ok = off(g * r + i) - off(g * r + i - 1) == st;
      if (ok && st > 0 && st % 16 == 0) { run_len = r; run_stride = st; break; }
    }
  }
  const int x_box = (pw * hbf * (hbh + (y1 - y0)) * 128 + 1023) / 1024 * 1024;
  const int h_stages = std::min(MAX_STAGES, PIPE_BYTES / (A_BYTES + (p.block_n / 64) * x_box));
  if (h_stages < 3) run_len = 1;                        // the halo boxes leave too few stages: per-tap boxes
  const bool halo = run_len > 1;
  p.run_len = run_len; p.run_stride = run_stride;
  if (halo) {
    p.bw = hbw; p.bh = hbh; p.bf = hbf;
    p.tiles_w = (dz.W + hbw - 1) / hbw; p.tiles_h = dz.H / hbh; p.tiles_f = (F + hbf - 1) / hbf;
    p.taps_per_cta = run_len;
    p.x_box_bytes = x_box; p.x_box_tx = pw * hbf * (hbh + (y1 - y0)) * 128; p.x_sbo = pw * 128; p.halo_x0 = x0; p.halo_y0 = y0;
    p.stage_bytes = A_BYTES + (p.block_n / 64) * x_box; p.stages = h_stages;
    for (int t = 0; t < ntaps; ++t) p.tap_xoff[t] = ((tdy[t] - y0) * hbf * pw + (tdx[t] - x0)) * 128;
  } else {
    p.stage_bytes = A_BYTES + 4 * BOX_BYTES; p.stages = 4;
    // several taps per CTA share one dz tile: stage = 2 dz boxes + taps * (block_n/64) x boxes <= 6 boxes, and
    // the accumulators (taps * mma_n fp32 columns) must fit the 512 TMEM columns
    p.taps_per_cta = 4 / (p.block_n / 64);
    if (p.taps_per_cta < 1) p.taps_per_cta = 1;
    while (p.taps_per_cta > 1 && p.taps_per_cta * p.mma_n > 512) --p.taps_per_cta;
    if (p.taps_per_cta > ntaps) p.taps_per_cta = ntaps;
  }
  p.tap_groups = (ntaps + p.taps_per_cta - 1) / p.taps_per_cta;
  p.taps_per_cta = (ntaps + p.tap_groups - 1) / p.tap_groups;        // balance the groups (9 taps: 3+3+3 rather than 4+4+1)
  const int ptiles = p.tiles_w * p.tiles_h * p.tiles_f;
  const int ctas = p.m_tiles * p.n_tiles * p.tap_groups;
  // one CTA per SM is resident (192 KiB pipeline), so a second wave only runs after the first: ONE wave of CTAs with
  // twice the pixels each does the same work with half the split-K partial traffic (every CTA writes its whole
  // 128 x taps*N fp32 accumulator: 100-250 KB) and no wave tail (conv2_3x3 used to run 300 CTAs = three waves)
  int splits = ctx.num_sms / ctas;
  if (splits < 1) splits = 1;
  if (splits > max_splits) splits = max_splits;
  if (splits > ptiles) splits = ptiles;
  if (splits < 1) splits = 1;
  p.ptiles_per_split = (ptiles + splits - 1) / splits;
  p.splits = (ptiles + p.ptiles_per_split - 1) / p.ptiles_per_split;
  p.partial = partial; p.bias_partial = nullptr;
  p.nseg = (dz.lo_off && x.lo_off) ? 3 : 1;
  if ((dz.lo_off != 0) != (x.lo_off != 0)) { set_thread_error("umma wgrad: both operands or neither must carry LO planes"); return 1; }
  auto lo_ptr = [](const View& v) { return reinterpret_cast<__half*>(reinterpret_cast<char*>(v.base) + v.lo_off) + v.coff; };
  if (halo) {
    cuuint64_t dims[4] = {(cuuint64_t)cout, (cuuint64_t)dz.W, (cuuint64_t)F, (cuuint64_t)dz.H};
    cuuint64_t str[3] = {(cuuint64_t)dz.pitch * 2, (cuuint64_t)dz.H * dz.W * dz.pitch * 2, (cuuint64_t)dz.W * dz.pitch * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)p.bw, (cuuint32_t)p.bf, (cuuint32_t)p.bh};
    if (int rc = umma_encode_f16(ctx, &plan.tmap_dz, 4, reinterpret_cast<__half*>(dz.base) + dz.coff, dims, str, box)) return rc;
    cuuint64_t xd[4] = {(cuuint64_t)cin, (cuuint64_t)x.W, (cuuint64_t)F, (cuuint64_t)x.H};
    cuuint64_t xs[3] = {(cuuint64_t)x.pitch * 2, (cuuint64_t)x.H * x.W * x.pitch * 2, (cuuint64_t)x.W * x.pitch * 2};
    cuuint32_t xb[4] = {64, (cuuint32_t)pw, (cuuint32_t)p.bf, (cuuint32_t)(p.bh + (y1 - y0))};
    if (int rc = umma_encode_f16(ctx, &plan.tmap_x, 4, reinterpret_cast<__half*>(x.base) + x.coff, xd, xs, xb)) return rc;
    plan.tmap_dz_lo = plan.tmap_dz; plan.tmap_x_lo = plan.tmap_x;
    if (p.nseg == 3) {
      if (int rc = umma_encode_f16(ctx, &plan.tmap_dz_lo, 4, lo_ptr(dz), dims, str, box)) return rc;
      if (int rc = umma_encode_f16(ctx, &plan.tmap_x_lo, 4, lo_ptr(x), xd, xs, xb)) return rc;
    }
    plan.enabled = true;
    return 0;
  }
  {
    cuuint64_t dims[4] = {(cuuint64_t)cout, (cuuint64_t)dz.W, (cuuint64_t)dz.H, (cuuint64_t)F};
    cuuint64_t str[3] = {(cuuint64_t)dz.pitch * 2, (cuuint64_t)dz.W * dz.pitch * 2, (cuuint64_t)dz.H * dz.W * dz.pitch * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)p.bw, (cuuint32_t)p.bh, (cuuint32_t)p.bf};
    if (int rc = umma_encode_f16(ctx, &plan.tmap_dz, 4, reinterpret_cast<__half*>(dz.base) + dz.coff, dims, str, box)) return rc;
    plan.tmap_dz_lo = plan.tmap_dz;
    if (p.nseg == 3) if (int rc = umma_encode_f16(ctx, &plan.tmap_dz_lo, 4, lo_ptr(dz), dims, str, box)) return rc;
  }
  {
    cuuint64_t dims[4] = {(cuuint64_t)cin, (cuuint64_t)x.W, (cuuint64_t)x.H, (cuuint64_t)F};
    cuuint64_t str[3] = {(cuuint64_t)x.pitch * 2, (cuuint64_t)x.W * x.pitch * 2, (cuuint64_t)x.H * x.W * x.pitch * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)(p.bw * x_stride), (cuuint32_t)(p.bh * x_stride), (cuuint32_t)p.bf};
    if (int rc = umma_encode_f16(ctx, &plan.tmap_x, 4, reinterpret_cast<__half*>(x.base) + x.coff, dims, str, box, x_stride)) return rc;
    plan.tmap_x_lo = plan.tmap_x;
    if (p.nseg == 3) if (int rc = umma_encode_f16(ctx, &plan.tmap_x_lo, 4, lo_ptr(x), dims, str, box, x_stride)) return rc;
  }
  plan.enabled = true;
  return 0;
}

int umma_wgrad_launch(UmmaContext& ctx, const UmmaWgradPlan& plan, cudaStream_t s, float* bias_partial) {
  if (!plan.enabled) { set_thread_error("umma wgrad: plan not bound"); return 3; }
  static bool attr_set[64] = {};          // function attributes are per device
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    if (cudaFuncSetAttribute(umma_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess) {
      set_thread_error("umma wgrad: cannot raise dynamic shared memory limit"); cudaGetLastError(); return 2; }
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  UmmaWgradParams p = plan.p;
  p.bias_partial = bias_partial;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  cfg.gridDim = dim3((unsigned)(p.m_tiles * p.n_tiles * p.tap_groups), (unsigned)p.splits);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = s;
  // programmatic dependent launch: the kernel's prologue may overlap the previous kernel's tail
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, umma_wgrad_kernel, plan.tmap_dz, plan.tmap_x, plan.tmap_dz_lo, plan.tmap_x_lo, p) != cudaSuccess) {
    set_thread_error(std::string("umma_wgrad_kernel launch: ") + cudaGetErrorString(cudaGetLastError())); return 2; }
  SSNB_LAUNCH_CHECK("umma_wgrad_kernel");
  return 0;
}

}  // namespace ssnb
