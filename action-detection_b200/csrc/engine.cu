// BNInception execution engine: graph table, workspace planner, forward/backward schedules and the
// backbone part of the C ABI (include/ssnb.h).  Replaces the reference's YAML-driven op
// interpreter (model_zoo/bninception/pytorch_load.py:8-61, layer_factory.py:25-83,
// bn_inception.yaml) and the autograd graph PyTorch builds from it.
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include <cuda_profiler_api.h>

#include "../../include/ssnb.h"
#include "common.cuh"
#include "umma_conv.cuh"

namespace ssnb {

std::atomic<long long> g_launches{0};
static thread_local std::string t_error;
void set_thread_error(const std::string& s) { t_error = s; }
const std::string& thread_error() { return t_error; }

// ---- per-launch timing session (see common.cuh) ---------------------------------------------------
thread_local bool t_timing = false;
thread_local LaunchTag t_tag;
struct TimingMark { const char* what; LaunchTag tag; cudaEvent_t ev; };
static thread_local std::vector<TimingMark> t_marks;
static thread_local std::vector<cudaEvent_t> t_event_pool;
static thread_local std::string t_report;
static cudaEvent_t timing_event() {
  if (!t_event_pool.empty()) { cudaEvent_t e = t_event_pool.back(); t_event_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
void timing_mark(const char* what, cudaStream_t s) {
  TimingMark m{what, t_tag, timing_event()};
  if (m.ev && cudaEventRecord(m.ev, s) == cudaSuccess) t_marks.push_back(m);
  else cudaGetLastError();
  t_tag.flop = 0.0;                 // FLOPs belong to the one launch they were set for
}

// ---- graph table ---------------------------------------------------------------------------------
struct BlockSpec { const char* name; int c1, c3r, c3, cdr, cd1, cd2; int pool_max; int cproj; int stride; };
// bn_inception.yaml:30-551
static const BlockSpec kBlocks[10] = {
    {"3a", 64, 64, 64, 64, 96, 96, 0, 32, 1},      {"3b", 64, 64, 96, 64, 96, 96, 0, 64, 1},
    {"3c", 0, 128, 160, 64, 96, 96, 1, 0, 2},      {"4a", 224, 64, 96, 96, 128, 128, 0, 128, 1},
    {"4b", 192, 96, 128, 96, 128, 128, 0, 128, 1}, {"4c", 160, 128, 160, 128, 160, 160, 0, 128, 1},
    {"4d", 96, 128, 192, 160, 192, 192, 0, 128, 1}, {"4e", 0, 128, 192, 192, 256, 256, 1, 0, 2},
    {"5a", 352, 192, 320, 160, 224, 224, 0, 128, 1}, {"5b", 352, 192, 320, 192, 224, 224, 1, 128, 1}};

struct ConvSpec { std::string id; int cin, cout, k, stride, pad; };

static std::vector<ConvSpec> conv_table(int in_ch) {
  std::vector<ConvSpec> v;
  v.push_back({"conv1_7x7_s2", in_ch, 64, 7, 2, 3});
  v.push_back({"conv2_3x3_reduce", 64, 64, 1, 1, 0});
  v.push_back({"conv2_3x3", 64, 192, 3, 1, 1});
  int cx = 192;
  for (const BlockSpec& b : kBlocks) {
    std::string p = std::string("inception_") + b.name + "_";
    if (b.c1) v.push_back({p + "1x1", cx, b.c1, 1, 1, 0});
    v.push_back({p + "3x3_reduce", cx, b.c3r, 1, 1, 0});
    v.push_back({p + "3x3", b.c3r, b.c3, 3, b.stride, 1});
    v.push_back({p + "double_3x3_reduce", cx, b.cdr, 1, 1, 0});
    v.push_back({p + "double_3x3_1", b.cdr, b.cd1, 3, 1, 1});
    v.push_back({p + "double_3x3_2", b.cd1, b.cd2, 3, b.stride, 1});
    if (b.cproj) v.push_back({p + "pool_proj", cx, b.cproj, 1, 1, 0});
    cx = b.c1 + b.c3 + b.cd2 + (b.cproj ? b.cproj : cx);
  }
  return v;
}

// ---- planned objects -----------------------------------------------------------------------------
struct Buffer { std::string name; int H, W, C; size_t off = 0, goff = 0; size_t hoff = 0, ghoff = 0, plane = 0; };   // EXACT_TC: fp16 hi/lo operand planes (lo = hi + plane)
struct Value { std::string name; int buf, coff, C; };
enum OpKind { OP_CONV = 0, OP_MAXPOOL = 1, OP_AVGPOOL = 2, OP_GPOOL = 3, OP_BN1 = 4 };   // OP_BN1: training-mode BatchNorm + ReLU behind conv1 (bn_mode='partial')
struct Op {
  OpKind kind; std::string id; int in_val, out_val;
  int conv = -1, k = 0, stride = 1, pad = 0;
  size_t argmax_off = 0;
  int grad_accumulate = 0;  // backward: dIn += (another consumer wrote first)
  int wsplits = 1, wrows = 0;
  int tsplits = 1;                // upper bound of the split count the tcgen05 weight-gradient planner may pick (sizes `partial`)
  size_t partial_off = 0, bias_partial_off = 0;   // this layer's split-K partials (own region: finalised in one batch)
  UmmaConvPlan umma;        // tcgen05 forward plan (FAST mode, stride-1 layers)
  UmmaConvPlan umma_dgrad;  // tcgen05 data-gradient plan
  UmmaWgradPlan umma_wgrad; // tcgen05 weight-gradient plan
  int pool_consumer = -1;   // conv whose only consumer is a k3/s2 max pool: that pool's op index (backward gather is folded in)
  bool folded_into_conv = false;   // max pool whose backward runs inside its producer conv's mask+bias pass
  bool dgrad_masks = false; // this op's data gradient is the LAST writer of d(in_val): it applies the ReLU mask of in_val
  bool bias_in_wgrad = false;// conv: bias gradient comes out of the tcgen05 weight-gradient kernel (ones operand)
  bool dy_premasked = false;// conv: d(out) arrives already masked, the backward pass only needs the bias column sums
  bool raw = false;         // conv whose BatchNorm runs unfused in training mode: no fold, no ReLU in the epilogue, no ReLU mask in backward
  int fuse_role = 0;        // sibling 1x1 fusion: 1 = leader (launches the fused kernels), 2 = follower
  int fuse_block = -1;
};
struct PackedConv { size_t wf, wd, bias, scale; size_t wf16 = 0, wd16 = 0, wplane = 0, wmax = 0; };   // EXACT_TC: fp16 hi planes of wf / wd, lo = hi + wplane
// the 1x1 convolutions of one inception block that read the block input (1x1, 3x3_reduce, double_3x3_reduce)
struct FusedBlock {
  int op1 = -1, op_r3 = -1, op_rd = -1;   // op indices (op1 = -1 for 3c/4e)
  int c1 = 0, c3r = 0, cdr = 0, cx = 0;
  size_t w_fwd = 0, bias = 0, w_dg = 0;   // stacked forward weights/bias, K-concatenated data-gradient weights
  size_t w_fwd_plane = 0, w_dg_plane = 0, wmax = 0;   // EXACT_TC: LO plane distance of both; shared (absmax, 1/scale) slot of the three layers
  UmmaConvPlan fwd, dgrad;
  bool enabled = false;
};

}  // namespace ssnb

using namespace ssnb;

struct ssnb_engine {
  ssnb_config cfg;
  int F = 0;
  bool fp16 = false;
  bool tc = false;                  // SSNB_EXACT_TC: fp32 storage + glue, convolutions as split-operand (hi/lo fp16) tcgen05 MMAs
  size_t esz = 4;
  size_t up_plane = 0, s2d_plane = 0, s2d_w_plane = 0;
  int* tc_flag = nullptr;           // device int: set when a split pass saw |x * grad_scale| beyond the fp16 range
  size_t tc_flag_off = 0, wmax_off = 0;
  bool bn1_train = false;           // bn_mode='partial': the first BatchNorm2d in training mode (bn_train.cu)
  const float *bn1_gamma = nullptr, *bn1_beta = nullptr; float *bn1_rmean = nullptr, *bn1_rvar = nullptr, *bn1_dgamma = nullptr, *bn1_dbeta = nullptr;
  float bn1_momentum = 0.1f, bn1_eps = 1e-5f;
  size_t bn_stat_off = 0, bn_partial_off = 0;
  std::vector<ConvSpec> convs;
  std::vector<Buffer> bufs;
  std::vector<Value> vals;
  std::map<std::string, int> val_by_name;
  std::vector<Op> ops;
  std::vector<PackedConv> packed;
  std::vector<FusedBlock> fused;
  size_t ws_bytes = 0, partial_off = 0, partial_bytes = 0, bpartial_off = 0;
  size_t s2d_off = 0, s2d_w_off = 0, up_off = 0;   // FAST mode: space-to-depth input + weights, zero-upsampled dz
  bool fold_pools = true;                            // SSNB_DISABLE_FUSION=1 also keeps the max-pool backward separate
  bool s2d_ready = false;                            // backbone_fwd converted the input directly
  int Cs = 0;                                        // channels of the space-to-depth input (4*Cin rounded up to 8)
  char* ws = nullptr;
  bool weights_ready = false;
  std::vector<float*> dw, db;
  std::vector<int> pending_finalize;  // conv ops whose partials wait for the batched finalize of this backward
  int grad_accumulate = 0;          // 1: dw/db += (autograd-style accumulation into existing .grad), 0: overwrite
  std::string error;
  long long launches0 = 0;
  UmmaContext umma_ctx;

  int fail(int code, const std::string& msg) { error = msg; return code; }
  View view(int val, bool grad) const {
    const Value& v = vals[val];
    const Buffer& b = bufs[v.buf];
    View w;
    w.base = ws + (grad ? b.goff : b.off);
    w.H = b.H; w.W = b.W; w.C = v.C; w.pitch = b.C; w.coff = v.coff;
    return w;
  }
  // EXACT_TC: the fp16 hi/lo operand planes of a value (activation or gradient)
  View planes(int val, bool grad) const {
    const Value& v = vals[val];
    const Buffer& b = bufs[v.buf];
    View w;
    w.base = ws + (grad ? b.ghoff : b.hoff);
    w.H = b.H; w.W = b.W; w.C = v.C; w.pitch = b.C; w.coff = v.coff; w.lo_off = (long long)b.plane;
    return w;
  }
};

namespace ssnb {

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
// profiling aid: SSNB_PROFILE_FWD_OPS / SSNB_PROFILE_BWD_OPS = comma-separated op ids; the engine brackets those ops of a whole
// forward / backward pass with cudaProfilerStart/Stop (use with `ncu --profile-from-start off`)
static bool profiled_op(const char* env, const std::string& id) {
  const char* e = getenv(env);
  if (!e || !*e) return false;
  const std::string list = std::string(",") + e + ",";
  return list.find("," + id + ",") != std::string::npos;
}
static int pool_out(int h, int k, int s, int p) {   // ceil_mode (layer_factory.py:46-50)
  int o = (h + 2 * p - k + s - 1) / s + 1;
  if ((o - 1) * s >= h + p) --o;
  return o;
}

static int add_buffer(ssnb_engine* e, const std::string& name, int H, int W, int C) {
  e->bufs.push_back({name, H, W, C});
  return (int)e->bufs.size() - 1;
}
static int add_value(ssnb_engine* e, const std::string& name, int buf, int coff, int C) {
  e->vals.push_back({name, buf, coff, C});
  e->val_by_name[name] = (int)e->vals.size() - 1;
  return (int)e->vals.size() - 1;
}

static void build_graph(ssnb_engine* e) {
  const int cin = e->cfg.in_channels;
  e->convs = conv_table(cin);
  int ci = 0;
  auto conv_op = [&](int in_val, int out_val) {
    const ConvSpec& c = e->convs[ci];
    Op o; o.kind = OP_CONV; o.id = c.id; o.in_val = in_val; o.out_val = out_val; o.conv = ci;
    o.k = c.k; o.stride = c.stride; o.pad = c.pad;
    e->ops.push_back(o);
    ++ci;
  };
  auto pool_op = [&](OpKind kind, const std::string& id, int in_val, int out_val, int k, int s, int p) {
    Op o; o.kind = kind; o.id = id; o.in_val = in_val; o.out_val = out_val; o.k = k; o.stride = s; o.pad = p;
    e->ops.push_back(o);
  };
  auto whole = [&](const std::string& name, int H, int W, int C) {
    return add_value(e, name, add_buffer(e, name, H, W, C), 0, C);
  };
  int x = whole("data", 224, 224, cin);
  int v;
  if (e->bn1_train) {
    const int raw = whole("conv1_7x7_s2_raw", 112, 112, 64); conv_op(x, raw); e->ops.back().raw = true;
    v = whole("conv1_7x7_s2_bn", 112, 112, 64);
    pool_op(OP_BN1, "conv1_7x7_s2_bn", raw, v, 0, 1, 0); x = v;
  } else {
    v = whole("conv1_7x7_s2_bn", 112, 112, 64); conv_op(x, v); x = v;
  }
  v = whole("pool1_3x3_s2", 56, 56, 64); pool_op(OP_MAXPOOL, "pool1_3x3_s2", x, v, 3, 2, 0); x = v;
  v = whole("conv2_3x3_reduce_bn", 56, 56, 64); conv_op(x, v); x = v;
  v = whole("conv2_3x3_bn", 56, 56, 192); conv_op(x, v); x = v;
  v = whole("pool2_3x3_s2", 28, 28, 192); pool_op(OP_MAXPOOL, "pool2_3x3_s2", x, v, 3, 2, 0); x = v;
  int H = 28, cx = 192;
  for (const BlockSpec& b : kBlocks) {
    const std::string p = std::string("inception_") + b.name + "_";
    const int OHW = (b.stride == 2) ? pool_out(H, 3, 2, 0) : H;
    const int ctot = b.c1 + b.c3 + b.cd2 + (b.cproj ? b.cproj : cx);
    const int cat = add_buffer(e, p + "output", OHW, OHW, ctot);
    const int red = add_buffer(e, p + "reduce", H, H, b.c3r + b.cdr);
    int off = 0;
    if (b.c1) { v = add_value(e, p + "1x1_bn", cat, off, b.c1); conv_op(x, v); off += b.c1; }
    int r3 = add_value(e, p + "3x3_reduce_bn", red, 0, b.c3r); conv_op(x, r3);
    v = add_value(e, p + "3x3_bn", cat, off, b.c3); conv_op(r3, v); off += b.c3;
    int rd = add_value(e, p + "double_3x3_reduce_bn", red, b.c3r, b.cdr); conv_op(x, rd);
    int d1 = whole(p + "double_3x3_1_bn", H, H, b.cd1); conv_op(rd, d1);
    v = add_value(e, p + "double_3x3_2_bn", cat, off, b.cd2); conv_op(d1, v); off += b.cd2;
    if (b.stride == 2) {
      v = add_value(e, p + "pool", cat, off, cx);
      pool_op(OP_MAXPOOL, p + "pool", x, v, 3, 2, 0);
    } else {
      int pl = whole(p + "pool", H, H, cx);
      pool_op(b.pool_max ? OP_MAXPOOL : OP_AVGPOOL, p + "pool", x, pl, 3, 1, 1);
      v = add_value(e, p + "pool_proj_bn", cat, off, b.cproj); conv_op(pl, v);
    }
    x = add_value(e, p + "output", cat, 0, ctot);
    H = OHW; cx = ctot;
  }
  // global_pool writes the caller's feat tensor; it has no workspace buffer
  Op g; g.kind = OP_GPOOL; g.id = "global_pool"; g.in_val = x; g.out_val = -1; g.k = 7;
  e->ops.push_back(g);
}

static void plan(ssnb_engine* e) {
  const size_t F = (size_t)e->F;
  size_t off = 0;
  for (Buffer& b : e->bufs) { b.off = off; off = align_up(off + F * b.H * b.W * b.C * e->esz, 1024); }
  if (e->cfg.training)
    for (Buffer& b : e->bufs) { b.goff = off; off = align_up(off + F * b.H * b.W * b.C * e->esz, 1024); }
  if (e->tc) {
    for (Buffer& b : e->bufs) {
      if (b.C % 8) continue;                              // the network input (3 / 10 channels) has no planes: conv1 reads its own packed copy
      b.plane = align_up(F * b.H * b.W * b.C * 2, 1024);
      b.hoff = off; off += 2 * b.plane;
      if (e->cfg.training) { b.ghoff = off; off += 2 * b.plane; }
    }
  }
  e->tc_flag_off = off; off = align_up(off + 256, 1024);      // gradient overflow flag (every mode)
  if (e->bn1_train) { e->bn_stat_off = off; off = align_up(off + 4 * 64 * 4, 1024); e->bn_partial_off = off; off = align_up(off + (size_t)1200 * 2 * 64 * 4, 1024); }
  for (Op& o : e->ops)
    if (o.kind == OP_MAXPOOL) {
      const Buffer& ob = e->bufs[e->vals[o.out_val].buf];
      o.argmax_off = off;
      off = align_up(off + F * ob.H * ob.W * e->vals[o.out_val].C, 1024);
    }
  e->packed.resize(e->convs.size());
  for (size_t i = 0; i < e->convs.size(); ++i) {
    const ConvSpec& c = e->convs[i];
    const size_t n = (size_t)c.cout * c.cin * c.k * c.k;
    e->packed[i].wf = off; off = align_up(off + n * e->esz, 1024);
    e->packed[i].wd = off; off = align_up(off + n * e->esz, 1024);
    e->packed[i].bias = off; off = align_up(off + c.cout * 4, 256);
    e->packed[i].scale = off; off = align_up(off + c.cout * 4, 256);
    if (e->tc) {
      e->packed[i].wplane = align_up(n * 2, 1024);
      e->packed[i].wf16 = off; off += 2 * e->packed[i].wplane;
      e->packed[i].wd16 = off; off += 2 * e->packed[i].wplane;
    }
  }
  if (e->tc) {      // per layer: [0] max |folded weight| (atomicMax target, zeroed before every pack), [1] 1 / plane scale (the kernels' alpha_dev)
    e->wmax_off = off;
    for (size_t i = 0; i < e->convs.size(); ++i) e->packed[i].wmax = off + i * 8;
    off = align_up(off + (e->convs.size() + 16) * 8, 1024);     // + one shared slot per fused sibling block
  }
  // backward bookkeeping: accumulate flags + split-K sizing
  size_t pmax = 0;
  if (e->cfg.training) {
    std::vector<char> written(e->vals.size(), 0);
    for (int i = (int)e->ops.size() - 1; i >= 0; --i) {
      Op& o = e->ops[i];
      o.grad_accumulate = written[o.in_val];
      written[o.in_val] = 1;
      if (o.kind == OP_CONV) {
        const ConvSpec& c = e->convs[o.conv];
        const Buffer& ob = e->bufs[e->vals[o.out_val].buf];
        const long long M = (long long)F * ob.H * ob.W;
        const int taps = c.k * c.k;
        const bool flat = c.cin < 16;
        const long long tiles = (long long)((c.cout + 63) / 64) * (flat ? (taps * c.cin + 63) / 64 : ((c.cin + 63) / 64) * taps);
        long long splits = (592 + tiles - 1) / tiles;
        if (splits > 128) splits = 128;
        while (splits > 1 && M / splits < 256) --splits;
        long long rows = (M + splits - 1) / splits;
        rows = (rows + 15) / 16 * 16;
        splits = (M + rows - 1) / rows;
        o.wsplits = (int)splits; o.wrows = (int)rows;
        // tcgen05 path: one CTA per SM is resident, so the planner wants num_sms / (M tiles x N tiles x tap groups) pixel
        // splits; the SIMT heuristic above used to cap it and left 57-75 % of the SMs busy on most 3x3 layers
        {
          const int chunks = (c.cin + 63) / 64, n_tiles = (chunks + 3) / 4, block_n = ((chunks + n_tiles - 1) / n_tiles) * 64;
          const int tpc = std::max(1, 4 / (block_n / 64));
          const int ctas = ((c.cout + 127) / 128) * n_tiles * ((taps + tpc - 1) / tpc);
          o.tsplits = std::max(o.wsplits, std::min(128, std::max(1, 148 / ctas)));
        }
        if (e->fp16 || e->tc) splits = std::max<long long>(splits, o.tsplits);
        const size_t need = (size_t)splits * taps * c.cout * c.cin * 4;
        if (need > pmax) pmax = need;
      }
    }
  }
  if (e->fp16 || e->tc) {
    for (int i = 0; i < (int)e->ops.size(); ++i) {
      const Op& o = e->ops[i];
      if (o.kind != OP_CONV || o.k != 1) continue;
      const std::string& id = o.id;
      const std::string suf = "_3x3_reduce";
      if (id.size() < suf.size() || id.compare(id.size() - suf.size(), suf.size(), suf) != 0 || id.find("double") != std::string::npos) continue;
      const std::string pre = id.substr(0, id.size() - suf.size() + 1);      // "inception_3a_"
      FusedBlock fb; fb.op_r3 = i;
      for (int j = 0; j < (int)e->ops.size(); ++j) {
        if (e->ops[j].id == pre + "1x1") fb.op1 = j;
        if (e->ops[j].id == pre + "double_3x3_reduce") fb.op_rd = j;
      }
      if (fb.op_rd < 0) continue;
      fb.cx = e->convs[o.conv].cin; fb.c3r = e->convs[o.conv].cout; fb.cdr = e->convs[e->ops[fb.op_rd].conv].cout;
      fb.c1 = fb.op1 >= 0 ? e->convs[e->ops[fb.op1].conv].cout : 0;
      const int n = fb.c1 + fb.c3r + fb.cdr, kf = (fb.c1 + 63) / 64 * 64 + fb.c3r + fb.cdr;
      fb.w_fwd_plane = align_up((size_t)n * fb.cx * 2, 1024); fb.w_dg_plane = align_up((size_t)fb.cx * kf * 2, 1024);
      if (e->tc) fb.w_fwd_plane = fb.w_dg_plane = std::max(fb.w_fwd_plane, fb.w_dg_plane);     // one LO-plane distance for both (split_all_kernel)
      fb.w_fwd = off; off += (e->tc ? 2 : 1) * fb.w_fwd_plane;
      fb.bias = off; off = align_up(off + (size_t)n * 4, 256);
      fb.w_dg = off; off += (e->tc ? 2 : 1) * fb.w_dg_plane;
      if (e->tc) {       // the three layers share ONE power-of-two plane scale (their operands are stacked / K-concatenated in one launch)
        if (e->fused.size() >= 16) continue;
        fb.wmax = e->wmax_off + (e->convs.size() + e->fused.size()) * 8;
        for (int j : {fb.op1, fb.op_r3, fb.op_rd}) if (j >= 0) e->packed[e->ops[j].conv].wmax = fb.wmax;
      }
      e->fused.push_back(fb);
    }
  }
  if (e->fp16) {
    for (int i = 0; i < (int)e->ops.size(); ++i) {
      Op& po = e->ops[i];
      if (po.kind != OP_MAXPOOL || po.k != 3 || po.stride != 2) continue;
      int producer = -1, consumers = 0;
      for (int j = 0; j < (int)e->ops.size(); ++j) {
        if (e->ops[j].out_val == po.in_val && e->ops[j].kind == OP_CONV) producer = j;
        if (e->ops[j].in_val == po.in_val) ++consumers;
      }
      if (producer >= 0 && consumers == 1 && e->vals[po.in_val].C % 8 == 0) { e->ops[producer].pool_consumer = i; po.folded_into_conv = true; }
    }
    e->Cs = (4 * e->cfg.in_channels + 7) / 8 * 8;
    e->s2d_off = off; off = align_up(off + F * 112 * 112 * 4 * e->Cs * 2, 1024);   // packed: 4 horizontal neighbours per pixel
    e->s2d_w_off = off; off = align_up(off + (size_t)16 * 64 * e->Cs * 2, 1024);
    if (e->cfg.training) {
      size_t up = 0;
      for (const Op& o : e->ops)
        if (o.kind == OP_CONV && o.stride == 2 && o.conv != 0) {
          const Buffer& ib = e->bufs[e->vals[o.in_val].buf];
          up = std::max(up, F * ib.H * ib.W * (size_t)e->convs[o.conv].cout * 2);
        }
      e->up_off = off; off = align_up(off + up, 1024);
      pmax = std::max(pmax, (size_t)128 * 16 * 64 * e->Cs * 4);
    }
  }
  if (e->tc) {
    for (int i = 0; i < (int)e->ops.size(); ++i) {      // convolutions whose only consumer is a k3/s2/pad0 max pool: backward gather folded in
      Op& po = e->ops[i];
      if (po.kind != OP_MAXPOOL || po.k != 3 || po.stride != 2 || po.pad != 0) continue;
      int producer = -1, consumers = 0;
      for (int j = 0; j < (int)e->ops.size(); ++j) {
        if (e->ops[j].out_val == po.in_val && e->ops[j].kind == OP_CONV) producer = j;
        if (e->ops[j].in_val == po.in_val) ++consumers;
      }
      if (producer >= 0 && consumers == 1 && e->vals[po.in_val].C % 4 == 0) { e->ops[producer].pool_consumer = i; po.folded_into_conv = true; }
    }
    e->Cs = (4 * e->cfg.in_channels + 7) / 8 * 8;
    e->s2d_plane = align_up(F * 112 * 112 * 4 * e->Cs * 2, 1024);
    e->s2d_off = off; off += 2 * e->s2d_plane;
    e->s2d_w_plane = align_up((size_t)16 * 64 * e->Cs * 2, 1024);
    e->s2d_w_off = off; off += 2 * e->s2d_w_plane;
    if (e->cfg.training) {
      size_t up = 0;
      for (const Op& o : e->ops)
        if (o.kind == OP_CONV && o.stride == 2 && o.conv != 0) {
          const Buffer& ib = e->bufs[e->vals[o.in_val].buf];
          up = std::max(up, F * ib.H * ib.W * (size_t)e->convs[o.conv].cout * 2);
        }
      e->up_plane = align_up(up, 1024);
      e->up_off = off; off += 2 * e->up_plane;
      pmax = std::max(pmax, (size_t)128 * 16 * 64 * e->Cs * 4);
    }
  }
  e->partial_off = off; e->partial_bytes = pmax; off = align_up(off + pmax, 1024);
  if (e->cfg.training)
    for (Op& o : e->ops)
      if (o.kind == OP_CONV) {
        const ConvSpec& c = e->convs[o.conv];
        const int nsplit = (e->fp16 || e->tc) ? std::max(o.wsplits, o.tsplits) : o.wsplits;
        size_t need = (size_t)nsplit * c.k * c.k * c.cout * c.cin * 4;
        if (o.conv == 0 && (e->fp16 || e->tc)) need = std::max(need, (size_t)128 * 16 * 64 * e->Cs * 4);
        o.partial_off = off; off = align_up(off + need, 1024);
        o.bias_partial_off = off; off = align_up(off + (size_t)std::max(nsplit, 128) * c.cout * 4, 256);
      }
  e->bpartial_off = off; off = align_up(off + (size_t)1024 * 512 * 4, 1024);   // column-sum partials: <= 1024 CTAs x 512 channels
  e->ws_bytes = off;
}

// ---- op execution --------------------------------------------------------------------------------
#define DISPATCH(e, call_f, call_h) ((e)->fp16 ? (call_h) : (call_f))

// timing tags (common.cuh): the next launch is the convolution `o` in pass `phase`
static double conv_flops(const ssnb_engine* e, const Op& o) {
  const ConvSpec& c = e->convs[o.conv];
  const Buffer& ob = e->bufs[e->vals[o.out_val].buf];
  return 2.0 * e->F * ob.H * ob.W * (double)c.cout * c.cin * c.k * c.k;
}
static inline void tag_next(int phase, double flop) { t_tag.phase = phase; t_tag.flop = flop; }

// EXACT_TC: operand planes of a value produced by a kernel that only wrote fp32 (pools, SIMT convolutions, value_write)
static int tc_split_value(ssnb_engine* e, int val, bool grad, float scale, cudaStream_t s) {
  if (!e->tc || !e->bufs[e->vals[val].buf].plane) return 0;
  return launch_split_view(e->view(val, grad), e->F, scale, e->planes(val, grad), grad ? e->tc_flag : nullptr, s);
}

static int run_fwd_impl(ssnb_engine* e, const Op& o, const float* input_nchw, float* feat, cudaStream_t s);
static int run_fwd(ssnb_engine* e, const Op& o, const float* input_nchw, float* feat, cudaStream_t s) {
  if (e->tc && o.kind == OP_CONV && o.umma.enabled) {
    // split-operand tcgen05 convolution: reads the input's hi/lo planes, writes fp32 + the output's planes
    if (o.conv == 0 && !e->s2d_ready)
      if (int rc = launch_nhwc_to_s2d_split(e->view(o.in_val, false), e->F, (__half*)(e->ws + e->s2d_off), (long long)e->s2d_plane, e->Cs, s)) return rc;
    tag_next(0, conv_flops(e, o));
    return umma_conv_launch(e->umma_ctx, o.umma, s);
  }
  tag_next(0, 0.0);
  if (o.kind == OP_BN1) {
    if (!e->bn1_gamma || !e->bn1_beta) { set_thread_error("bn1_train engine: call ssnb_set_bn1 first"); return SSNB_ESTATE; }
    return launch_bn_train_fwd(e->view(o.in_val, false), e->view(o.out_val, false), e->tc ? e->planes(o.out_val, false) : View(), e->F, e->bn1_gamma,
                               e->bn1_beta, e->bn1_eps, e->bn1_momentum, e->bn1_rmean, e->bn1_rvar, (float*)(e->ws + e->bn_stat_off),
                               (float*)(e->ws + e->bn_partial_off), 1200, s);
  }
  if (e->tc && (o.kind == OP_MAXPOOL || o.kind == OP_AVGPOOL) && e->bufs[e->vals[o.out_val].buf].plane) {
    // vectorised fp32 pooling that also emits the output's operand planes (glue_fp32.cu)
    const View in = e->view(o.in_val, false), out = e->view(o.out_val, false), pl = e->planes(o.out_val, false);
    if (o.kind == OP_MAXPOOL) return launch_maxpool_fwd_f4(in, out, pl, e->F, o.k, o.stride, o.pad, (uint8_t*)(e->ws + o.argmax_off), s);
    return launch_avgpool3_f4(in, out, pl, e->F, 0, s);
  }
  if (int rc = run_fwd_impl(e, o, input_nchw, feat, s)) return rc;
  return (e->tc && o.out_val >= 0) ? tc_split_value(e, o.out_val, false, 1.0f, s) : 0;
}

static int run_fwd_impl(ssnb_engine* e, const Op& o, const float* input_nchw, float* feat, cudaStream_t s) {
  const int F = e->F;
  if (o.kind == OP_CONV) {
    const ConvSpec& c = e->convs[o.conv];
    const View in = e->view(o.in_val, false), out = e->view(o.out_val, false);
    if (e->fp16 && o.umma.enabled) {
      if (o.conv == 0 && !e->s2d_ready)   // conv1 runs as a 4x4 stride-1 convolution over the space-to-depth input
        if (int rc = launch_nhwc_to_s2d(in, F, (__half*)(e->ws + e->s2d_off), e->Cs, s)) return rc;
      tag_next(0, conv_flops(e, o));
      return umma_conv_launch(e->umma_ctx, o.umma, s);
    }
    ConvArgs a;
    a.src = in.base; a.SH = in.H; a.SW = in.W; a.Csrc = in.C; a.src_pitch = in.pitch; a.src_coff = in.coff;
    a.dst = out.base; a.DH = out.H; a.DW = out.W; a.Cdst = out.C; a.dst_pitch = out.pitch; a.dst_coff = out.coff;
    a.wgt = e->ws + e->packed[o.conv].wf; a.bias = (const float*)(e->ws + e->packed[o.conv].bias);
    a.F = F; a.k = c.k; a.stride = c.stride; a.pad = c.pad; a.relu = o.raw ? 0 : 1; a.accumulate = 0; a.dgrad = 0;
    tag_next(0, conv_flops(e, o));
    return DISPATCH(e, launch_conv<float>(a, s), launch_conv<__half>(a, s));
  }
  if (o.kind == OP_MAXPOOL) {
    const View in = e->view(o.in_val, false), out = e->view(o.out_val, false);
    uint8_t* am = (uint8_t*)(e->ws + o.argmax_off);
    if (e->fp16 && in.C % 8 == 0) return launch_maxpool_fwd_h8(in, out, F, o.k, o.stride, o.pad, am, s);
    return DISPATCH(e, launch_maxpool_fwd<float>(in, out, F, o.k, o.stride, o.pad, am, s),
                    launch_maxpool_fwd<__half>(in, out, F, o.k, o.stride, o.pad, am, s));
  }
  if (o.kind == OP_AVGPOOL) {
    const View in = e->view(o.in_val, false), out = e->view(o.out_val, false);
    if (e->fp16 && in.C % 8 == 0) return launch_avgpool3_h8(in, out, F, 0, s);
    return DISPATCH(e, launch_avgpool3_fwd<float>(in, out, F, 0, s), launch_avgpool3_fwd<__half>(in, out, F, 0, s));
  }
  if (o.kind == OP_GPOOL) {
    if (!feat) return e->fail(SSNB_EINVAL, "global_pool needs the feat output pointer");
    const View in = e->view(o.in_val, false);
    return DISPATCH(e, launch_gpool_fwd<float>(in, F, feat, s), launch_gpool_fwd<__half>(in, F, feat, s));
  }
  return SSNB_EINVAL;
}

static int run_bwd(ssnb_engine* e, const Op& o, const float* dfeat, cudaStream_t s, bool skip_dgrad = false, bool full = false) {
  const int F = e->F;
  const float gs = e->fp16 ? e->cfg.grad_scale : 1.0f;
  int rc = 0;
  tag_next(3, 0.0);
  if (o.kind == OP_GPOOL) {
    if (!dfeat) return e->fail(SSNB_EINVAL, "global_pool backward needs dfeat");
    const View din = e->view(o.in_val, true);
    const void* ym = (full && e->fold_pools && o.dgrad_masks) ? e->view(o.in_val, false).base : nullptr;
    return DISPATCH(e, launch_gpool_bwd<float>(dfeat, gs, din, F, ym, s), launch_gpool_bwd<__half>(dfeat, gs, din, F, ym, s));
  }
  if (o.kind == OP_BN1) {
    return launch_bn_train_bwd(e->view(o.in_val, false), e->view(o.out_val, true), e->view(o.out_val, false), e->view(o.in_val, true),
                               e->tc ? e->planes(o.in_val, true) : View(), e->cfg.grad_scale, e->tc_flag, F, e->bn1_gamma, (float*)(e->ws + e->bn_stat_off),
                               (float*)(e->ws + e->bn_partial_off), 1200, e->bn1_dgamma, e->bn1_dbeta, e->grad_accumulate, s);
  }
  if (o.kind == OP_MAXPOOL) {
    if (full && (e->fp16 || e->tc) && e->fold_pools && o.folded_into_conv) return 0;      // gathered by the producer conv's mask+bias pass
    const View din = e->view(o.in_val, true), dout = e->view(o.out_val, true);
    const uint8_t* am = (const uint8_t*)(e->ws + o.argmax_off);
    if (e->tc && din.C % 4 == 0) return launch_maxpool_bwd_f4(din, dout, F, o.k, o.stride, o.pad, am, o.grad_accumulate, s);
    if (e->fp16 && din.C % 8 == 0) return launch_maxpool_bwd_h8(din, dout, F, o.k, o.stride, o.pad, am, o.grad_accumulate, s);
    return DISPATCH(e, launch_maxpool_bwd<float>(din, dout, F, o.k, o.stride, o.pad, am, o.grad_accumulate, s),
                    launch_maxpool_bwd<__half>(din, dout, F, o.k, o.stride, o.pad, am, o.grad_accumulate, s));
  }
  if (o.kind == OP_AVGPOOL) {
    const View din = e->view(o.in_val, true), dout = e->view(o.out_val, true);
    if (e->tc && din.C % 4 == 0) return launch_avgpool3_f4(dout, din, View(), F, o.grad_accumulate, s);
    if (e->fp16 && din.C % 8 == 0) return launch_avgpool3_h8(dout, din, F, o.grad_accumulate, s);
    return DISPATCH(e, launch_avgpool3_fwd<float>(dout, din, F, o.grad_accumulate, s),
                    launch_avgpool3_fwd<__half>(dout, din, F, o.grad_accumulate, s));
  }
  // convolution: dz = dy * (y > 0); db, dW from dz; dx = dgrad(dz)
  const ConvSpec& c = e->convs[o.conv];
  const View x = e->view(o.in_val, false), y = e->view(o.out_val, false);
  const View dx = e->view(o.in_val, true), dy = e->view(o.out_val, true);
  const float* scale = (const float*)(e->ws + e->packed[o.conv].scale);
  float* partial = (float*)(e->ws + o.partial_off);
  float* bpartial = (float*)(e->ws + e->bpartial_off);
  const long long M = (long long)F * y.H * y.W;
  float* dbp = (e->db.size() && e->db[o.conv]) ? e->db[o.conv] : nullptr;
  if (e->tc) {
    // EXACT_TC: fp32 mask + bias gradient (as EXACT), then dz * grad_scale as hi/lo planes for the tensor-core products
    const float gst = e->cfg.grad_scale;
    const bool want_w = e->dw.size() && e->dw[o.conv];
    const bool want_x = e->vals[o.in_val].name != "data" && !skip_dgrad;
    const bool tc_w = want_w && o.umma_wgrad.enabled, tc_x = want_x && o.umma_dgrad.enabled;
    const bool pre = full && e->fold_pools && o.dy_premasked;      // the last writer of dy masked it and wrote its operand planes
    const bool bias_w = pre && o.bias_in_wgrad && dbp && tc_w;     // ... and the column sums ride on the weight-gradient MMAs
    if (o.raw) {
      // the training-mode BatchNorm behind this convolution produced dz and its planes: only the bias-gradient column sums are left
      if (dbp)
        if ((rc = launch_mask_bias_split_f4(dy, View(), View(), gst, 0, nullptr, F, scale, 1.0f, bpartial, (1024 * 512 - 64) / y.C, dbp, e->grad_accumulate, s))) return rc;
    } else if (pre) {
      if (!bias_w && dbp)       // bias gradient only: column sums of the (already masked) fp32 dz, no planes, nothing written back
        if ((rc = launch_mask_bias_split_f4(dy, y, View(), gst, 0, nullptr, F, scale, 1.0f, bpartial, (1024 * 512 - 64) / y.C, dbp, e->grad_accumulate, s))) return rc;
    } else if (full && e->fold_pools && o.pool_consumer >= 0) {
      // the consuming max pool's backward gather + ReLU mask + bias sums + planes in one pass (the fp32 dy is never materialised)
      const Op& po = e->ops[o.pool_consumer];
      const bool need_f32 = (want_w && !tc_w) || (want_x && !tc_x);
      View pl = (tc_w || tc_x) ? e->planes(o.out_val, true) : View();
      if ((rc = launch_pool_mask_bias_split_f4(dy, y, e->view(po.out_val, true), pl, gst, need_f32 ? 1 : 0, e->tc_flag, F,
                                               (const uint8_t*)(e->ws + po.argmax_off), scale, 1.0f, bpartial, (1024 * 512 - 64) / y.C, dbp,
                                               e->grad_accumulate, s))) return rc;
    } else {
      // one pass over dy: ReLU mask, bias-gradient column sums and the hi/lo planes of dz * grad_scale; the masked fp32 dz is
      // written back only when a SIMT kernel will read it
      const bool need_f32 = (want_w && !tc_w) || (want_x && !tc_x) || !full;
      View pl = (tc_w || tc_x) ? e->planes(o.out_val, true) : View();
      if ((rc = launch_mask_bias_split_f4(dy, y, pl, gst, need_f32 ? 1 : 0, e->tc_flag, F, scale, 1.0f, bpartial, (1024 * 512 - 64) / y.C, dbp,
                                          e->grad_accumulate, s))) return rc;
    }
    if (tc_x && c.stride == 2 && o.conv != 0) {              // dz at input resolution (zero-upsampled), both planes
      const View dzp = e->planes(o.out_val, true);
      View lo = dzp; lo.base = (char*)dzp.base + dzp.lo_off;
      if ((rc = launch_upsample2_zero(dzp, (__half*)(e->ws + e->up_off), x.H, x.W, F, s))) return rc;
      if ((rc = launch_upsample2_zero(lo, (__half*)(e->ws + e->up_off + e->up_plane), x.H, x.W, F, s))) return rc;
    }
    if (tc_w) {
      tag_next(2, conv_flops(e, o));
      if ((rc = umma_wgrad_launch(e->umma_ctx, o.umma_wgrad, s, bias_w ? (float*)(e->ws + o.bias_partial_off) : nullptr))) return rc;
      if (full && o.conv != 0) { e->pending_finalize.push_back((int)(&o - e->ops.data())); rc = 0; }     // batched at the end of the backward
      else if (o.conv == 0) rc = launch_wgrad_finalize_s2d(partial, o.umma_wgrad.p.splits, c.cout, c.cin, e->Cs, scale, 1.0f / gst, e->dw[o.conv], e->grad_accumulate, s);
      else rc = launch_wgrad_finalize(partial, o.umma_wgrad.p.splits, c.k * c.k, c.cout, c.cin, scale, 1.0f / gst, e->dw[o.conv], e->grad_accumulate, s);
      if (rc) return rc;
    } else if (want_w) {
      WgradArgs w;
      w.dz = dy.base; w.OH = y.H; w.OW = y.W; w.Cout = y.C; w.dz_pitch = dy.pitch; w.dz_coff = dy.coff;
      w.x = x.base; w.IH = x.H; w.IW = x.W; w.Cin = x.C; w.x_pitch = x.pitch; w.x_coff = x.coff;
      w.partial = partial; w.F = F; w.k = c.k; w.stride = c.stride; w.pad = c.pad;
      w.rows_per_split = o.wrows; w.splits = o.wsplits;
      tag_next(2, conv_flops(e, o));
      if ((rc = launch_wgrad<float>(w, s))) return rc;
      if ((rc = launch_wgrad_finalize(partial, o.wsplits, c.k * c.k, c.cout, c.cin, scale, 1.0f, e->dw[o.conv], e->grad_accumulate, s))) return rc;
    }
    tag_next(1, conv_flops(e, o));
    if (tc_x) return umma_conv_launch(e->umma_ctx, o.umma_dgrad, s, full && e->fold_pools && o.dgrad_masks);
    if (want_x) {
      ConvArgs a;
      a.src = dy.base; a.SH = dy.H; a.SW = dy.W; a.Csrc = dy.C; a.src_pitch = dy.pitch; a.src_coff = dy.coff;
      a.dst = dx.base; a.DH = dx.H; a.DW = dx.W; a.Cdst = dx.C; a.dst_pitch = dx.pitch; a.dst_coff = dx.coff;
      a.wgt = e->ws + e->packed[o.conv].wd; a.bias = nullptr;
      a.F = F; a.k = c.k; a.stride = c.stride; a.pad = c.pad; a.relu = 0; a.accumulate = o.grad_accumulate; a.dgrad = 1;
      rc = launch_conv<float>(a, s);
    }
    return rc;
  }
  if (e->fp16 && full && e->fold_pools && o.pool_consumer >= 0) {
    // max-pool backward gather + ReLU mask + bias-gradient column sums in one pass (dy is never materialised)
    const Op& po = e->ops[o.pool_consumer];
    if ((rc = launch_pool_mask_bias_h8(dy, y, e->view(po.out_val, true), F, po.k, po.stride, po.pad, (const uint8_t*)(e->ws + po.argmax_off),
                                       scale, 1.0f / gs, bpartial, (1024 * 512 - 64) / y.C, dbp, e->grad_accumulate, s))) return rc;
  } else if (e->fp16) {
    // one pass: ReLU gradient mask in place + bias-gradient column sums (mask skipped when the producer of dy applied it)
    const bool pre = full && e->fold_pools && o.dy_premasked;
    const bool bias_w = pre && o.bias_in_wgrad && dbp && e->dw.size() && e->dw[o.conv] && o.umma_wgrad.enabled;
    if (bias_w) { /* no pass at all: dy is already masked and the column sums ride on the weight-gradient MMAs */ }
    else if ((rc = launch_mask_bias_h8(dy, pre ? View() : y, F, scale, 1.0f / gs, bpartial, (1024 * 512 - 64) / y.C, dbp, e->grad_accumulate, s))) return rc;
  } else {
    if (!o.raw && (rc = launch_relu_mask<float>(dy, y, F, s))) return rc;
    if (dbp) {
      int bs = (int)((M + 4095) / 4096); if (bs > 64) bs = 64; if (bs < 1) bs = 1;
      if ((rc = launch_bias_grad<float>(dy.base, (int)M, y.C, dy.pitch, dy.coff, scale, 1.0f / gs, bpartial, bs, dbp, e->grad_accumulate, s))) return rc;
    }
  }
  if (e->fp16 && c.stride == 2 && o.conv != 0 && o.umma_dgrad.enabled && !skip_dgrad)
    if ((rc = launch_upsample2_zero(dy, (__half*)(e->ws + e->up_off), x.H, x.W, F, s))) return rc;   // dz at input resolution
  if (e->dw.size() && e->dw[o.conv] && e->fp16 && o.umma_wgrad.enabled) {
    const bool bias_w = full && e->fold_pools && o.dy_premasked && o.bias_in_wgrad && dbp;
    float* bp = bias_w ? (float*)(e->ws + o.bias_partial_off) : nullptr;
    tag_next(2, conv_flops(e, o));
    if ((rc = umma_wgrad_launch(e->umma_ctx, o.umma_wgrad, s, bp))) return rc;
    if (full && e->fold_pools && o.conv != 0) { e->pending_finalize.push_back((int)(&o - e->ops.data())); rc = 0; }   // batched at the end of the backward
    else if (o.conv == 0) rc = launch_wgrad_finalize_s2d(partial, o.umma_wgrad.p.splits, c.cout, c.cin, e->Cs, scale, 1.0f / gs, e->dw[o.conv], e->grad_accumulate, s);
    else rc = launch_wgrad_finalize(partial, o.umma_wgrad.p.splits, c.k * c.k, c.cout, c.cin, scale, 1.0f / gs, e->dw[o.conv], e->grad_accumulate, s, bp, dbp, e->tc_flag);
    if (rc) return rc;
  } else if (e->dw.size() && e->dw[o.conv]) {
    WgradArgs w;
    w.dz = dy.base; w.OH = y.H; w.OW = y.W; w.Cout = y.C; w.dz_pitch = dy.pitch; w.dz_coff = dy.coff;
    w.x = x.base; w.IH = x.H; w.IW = x.W; w.Cin = x.C; w.x_pitch = x.pitch; w.x_coff = x.coff;
    w.partial = partial; w.F = F; w.k = c.k; w.stride = c.stride; w.pad = c.pad;
    w.rows_per_split = o.wrows; w.splits = o.wsplits;
    tag_next(2, conv_flops(e, o));
    if ((rc = DISPATCH(e, launch_wgrad<float>(w, s), launch_wgrad<__half>(w, s)))) return rc;
    if ((rc = launch_wgrad_finalize(partial, o.wsplits, c.k * c.k, c.cout, c.cin, scale, 1.0f / gs, e->dw[o.conv], e->grad_accumulate, s))) return rc;
  }
  if (e->vals[o.in_val].name != "data" && !skip_dgrad) {
    tag_next(1, conv_flops(e, o));
    if (e->fp16 && o.umma_dgrad.enabled) return umma_conv_launch(e->umma_ctx, o.umma_dgrad, s, full && e->fold_pools && o.dgrad_masks);
    ConvArgs a;
    a.src = dy.base; a.SH = dy.H; a.SW = dy.W; a.Csrc = dy.C; a.src_pitch = dy.pitch; a.src_coff = dy.coff;
    a.dst = dx.base; a.DH = dx.H; a.DW = dx.W; a.Cdst = dx.C; a.dst_pitch = dx.pitch; a.dst_coff = dx.coff;
    a.wgt = e->ws + e->packed[o.conv].wd; a.bias = nullptr;
    a.F = F; a.k = c.k; a.stride = c.stride; a.pad = c.pad; a.relu = 0; a.accumulate = o.grad_accumulate; a.dgrad = 1;
    rc = DISPATCH(e, launch_conv<float>(a, s), launch_conv<__half>(a, s));
  }
  return rc;
}

int engine_tail_view(ssnb_handle h, View* v, int* F, int* fp16) {
  if (!h->ws || !h->weights_ready) return h->fail(SSNB_ESTATE, "workspace/weights not set");
  *v = h->view(h->ops.back().in_val, false);
  *F = h->F; *fp16 = h->fp16 ? 1 : 0;
  return 0;
}

}  // namespace ssnb

// ---- C ABI -----------------------------------------------------------------------------------------
extern "C" {

const char* ssnb_version(void) { return "libssn_b200 0.2 (sm_100a)"; }

const char* ssnb_last_error(ssnb_handle h) { return h ? h->error.c_str() : ssnb::thread_error().c_str(); }

int ssnb_num_convs(void) { return 69; }

int ssnb_conv_info(int idx, int in_channels, char* name, int name_cap, int* cin, int* cout, int* k, int* stride, int* pad) {
  std::vector<ConvSpec> t = conv_table(in_channels);
  if (idx < 0 || idx >= (int)t.size()) { set_thread_error("ssnb_conv_info: index out of range"); return SSNB_EINVAL; }
  if (name && name_cap > 0) { snprintf(name, name_cap, "%s", t[idx].id.c_str()); }
  if (cin) *cin = t[idx].cin; if (cout) *cout = t[idx].cout; if (k) *k = t[idx].k;
  if (stride) *stride = t[idx].stride; if (pad) *pad = t[idx].pad;
  return SSNB_OK;
}

int ssnb_create(const ssnb_config* cfg, ssnb_handle* out) {
  if (!cfg || !out) { set_thread_error("ssnb_create: null argument"); return SSNB_EINVAL; }
  if (cfg->frames <= 0 || cfg->in_channels <= 0 || cfg->in_channels > 64) { set_thread_error("ssnb_create: bad frames/in_channels"); return SSNB_EINVAL; }
  if (cfg->precision != SSNB_EXACT_FP32 && cfg->precision != SSNB_FAST_FP16 && cfg->precision != SSNB_EXACT_TC) { set_thread_error("ssnb_create: unknown precision"); return SSNB_EINVAL; }
  ssnb_engine* e = new ssnb_engine();
  e->cfg = *cfg;
  if (!(e->cfg.grad_scale > 0.f)) e->cfg.grad_scale = 1.0f;
  e->F = cfg->frames;
  e->fp16 = cfg->precision == SSNB_FAST_FP16;
  e->tc = cfg->precision == SSNB_EXACT_TC;
  e->bn1_train = cfg->bn1_train != 0;
  if (e->bn1_train && e->fp16) { delete e; set_thread_error("ssnb_create: bn1_train (bn_mode='partial') needs EXACT_FP32 or EXACT_TC"); return SSNB_ENOSUPPORT; }
  e->esz = e->fp16 ? 2 : 4;
  build_graph(e);
  if ((int)e->convs.size() != 69) { delete e; set_thread_error("internal: conv table size"); return SSNB_ESTATE; }
  umma_context_init(e->umma_ctx, e->fp16 || e->tc);
  plan(e);
  e->launches0 = g_launches.load();
  *out = e;
  return SSNB_OK;
}

int ssnb_destroy(ssnb_handle h) {
  if (!h) return SSNB_OK;
  umma_context_destroy(h->umma_ctx);
  delete h;
  return SSNB_OK;
}

size_t ssnb_workspace_bytes(ssnb_handle h) { return h ? h->ws_bytes : 0; }

int ssnb_set_workspace(ssnb_handle h, void* dev_ptr, size_t bytes) {
  if (!h) return SSNB_EINVAL;
  if (!dev_ptr || bytes < h->ws_bytes) return h->fail(SSNB_EINVAL, "workspace too small");
  if (((uintptr_t)dev_ptr) % 1024) return h->fail(SSNB_EINVAL, "workspace must be 1024-byte aligned");
  h->ws = (char*)dev_ptr;
  h->weights_ready = false;
  if ((h->fp16 || h->tc) && cudaMemset(h->ws + h->bpartial_off, 0, 256) != cudaSuccess) { cudaGetLastError(); /* no device (CPU-only planning) */ }
  h->tc_flag = (int*)(h->ws + h->tc_flag_off);
  if (cudaMemset(h->tc_flag, 0, 256) != cudaSuccess) cudaGetLastError();
  if (h->tc) {
    // SSNB_EXACT_TC: split-operand plans over the hi/lo planes.  SSNB_DISABLE_UMMA=1 leaves every convolution on the fp32
    // SIMT kernels (= SSNB_EXACT_FP32 arithmetic; what the tensor-core launches are diffed against).
    const char* dis_tc = getenv("SSNB_DISABLE_UMMA");
    const bool use_tc = !(dis_tc && dis_tc[0] == '1');
    const char* disw_tc = getenv("SSNB_DISABLE_UMMA_WGRAD");
    const bool use_wgrad_tc = h->cfg.training && !(disw_tc && disw_tc[0] == '1');
    const float gs = h->cfg.grad_scale;
    for (Op& o : h->ops) {
      o.umma.enabled = false; o.umma_dgrad.enabled = false; o.umma_wgrad.enabled = false;
      o.fuse_role = 0; o.fuse_block = -1; o.dgrad_masks = false; o.dy_premasked = false; o.bias_in_wgrad = false;
      if (o.kind != OP_CONV || !use_tc) continue;
      const ConvSpec& c = h->convs[o.conv];
      const PackedConv& pk = h->packed[o.conv];
      const View out32 = h->view(o.out_val, false);
      int rc = 0;
      if (o.conv == 0) {
        // conv1 7x7/2: four vertical taps over the packed space-to-depth input planes (see the FAST binding below)
        const int Ck = 4 * h->Cs;
        View xs; xs.base = h->ws + h->s2d_off; xs.H = 112; xs.W = 112; xs.C = Ck; xs.pitch = Ck; xs.coff = 0; xs.lo_off = (long long)h->s2d_plane;
        int dy[4], dx[4];
        for (int t = 0; t < 4; ++t) { dy[t] = t - 2; dx[t] = 0; }
        UmmaTcOpts t; t.w_lo_off = (long long)h->s2d_w_plane; t.out32 = (float*)out32.base; t.alpha = 1.0f; t.alpha_dev = (const float*)(h->ws + pk.wmax) + 1;
        rc = umma_conv_bind_taps(h->umma_ctx, o.umma, xs, h->planes(o.out_val, false), h->F, Ck, c.cout, 4, dy, dx,
                                 (const __half*)(h->ws + h->s2d_w_off), (const float*)(h->ws + pk.bias), o.raw ? 0 : 1, &t);
        if (rc) return h->fail(rc, "tc conv1 bind: " + ssnb::thread_error());
        if (use_wgrad_tc) {
          rc = umma_wgrad_bind_taps(h->umma_ctx, o.umma_wgrad, h->planes(o.out_val, true), xs, h->F, Ck, c.cout, 4, dy, dx,
                                    (float*)(h->ws + o.partial_off), 128);
          if (rc) return h->fail(rc, "tc conv1 wgrad bind: " + ssnb::thread_error());
        }
        continue;
      }
      if (c.cin % 8 != 0 || c.k * c.k > UMMA_MAX_TAPS) continue;
      UmmaTcOpts t; t.w_lo_off = (long long)pk.wplane; t.out32 = (float*)out32.base; t.alpha = 1.0f; t.alpha_dev = (const float*)(h->ws + pk.wmax) + 1;
      rc = umma_conv_bind_fwd(h->umma_ctx, o.umma, h->planes(o.in_val, false), h->planes(o.out_val, false), h->F, c.cin, c.cout, c.k, c.pad,
                              c.stride, (const __half*)(h->ws + pk.wd16), (const float*)(h->ws + pk.bias), &t);
      if (rc) return h->fail(rc, "tc bind_fwd(" + c.id + "): " + ssnb::thread_error());
      if (!h->cfg.training) continue;
      View dz = h->planes(o.out_val, true);
      const View in = h->view(o.in_val, false);
      if (c.stride == 2) { dz.base = h->ws + h->up_off; dz.H = in.H; dz.W = in.W; dz.C = c.cout; dz.pitch = c.cout; dz.coff = 0; dz.lo_off = (long long)h->up_plane; }
      View dxp = h->planes(o.in_val, true); dxp.base = nullptr; dxp.lo_off = 0;          // data gradients: fp32 only (masked and split by their consumer)
      UmmaTcOpts tg; tg.w_lo_off = (long long)pk.wplane; tg.out32 = (float*)h->view(o.in_val, true).base; tg.alpha = 1.0f / gs; tg.alpha_dev = (const float*)(h->ws + pk.wmax) + 1;
      rc = umma_conv_bind_dgrad(h->umma_ctx, o.umma_dgrad, dz, dxp, h->F, c.cin, c.cout, c.k, c.pad, (const __half*)(h->ws + pk.wf16),
                                o.grad_accumulate, &tg);
      if (rc) return h->fail(rc, "tc bind_dgrad(" + c.id + "): " + ssnb::thread_error());
      if (use_wgrad_tc) {
        rc = umma_wgrad_bind(h->umma_ctx, o.umma_wgrad, h->planes(o.out_val, true), h->planes(o.in_val, false), h->F, c.cin, c.cout, c.k, c.pad,
                             (float*)(h->ws + o.partial_off), o.tsplits, c.stride);
        if (rc) return h->fail(rc, "tc wgrad_bind(" + c.id + "): " + ssnb::thread_error());
      }
    }
    h->fold_pools = false;
    for (FusedBlock& fb : h->fused) fb.enabled = false;
    const char* disf_sib = getenv("SSNB_DISABLE_FUSION");
    if (use_tc && !(disf_sib && disf_sib[0] == '1')) {
      // horizontal fusion of the sibling 1x1 convolutions of each inception block: ONE forward launch (stacked weights; the first
      // c1 columns land in the concat buffer, the rest in the shared reduce buffer) and ONE data-gradient launch (K-concatenated
      // dz planes from two sources) instead of three read-modify-write passes over the block input's gradient
      for (size_t bi = 0; bi < h->fused.size(); ++bi) {
        FusedBlock& fb = h->fused[bi];
        Op& o3 = h->ops[fb.op_r3]; Op& od = h->ops[fb.op_rd];
        if (!o3.umma.enabled || !od.umma.enabled) continue;
        const View xp = h->planes(o3.in_val, false);
        View redp = h->planes(o3.out_val, false); redp.C = fb.c3r + fb.cdr;
        const View red32 = h->view(o3.out_val, false);
        const float* alpha_dev = (const float*)(h->ws + fb.wmax) + 1;
        int rc;
        UmmaTcOpts t; t.w_lo_off = (long long)fb.w_fwd_plane; t.alpha = 1.0f; t.alpha_dev = alpha_dev;
        if (fb.op1 >= 0) {
          t.out32 = (float*)h->view(h->ops[fb.op1].out_val, false).base; t.out32_2 = (float*)red32.base;
          rc = umma_conv_bind_fused_fwd(h->umma_ctx, fb.fwd, xp, h->planes(h->ops[fb.op1].out_val, false), redp, h->F, fb.cx, fb.c1, fb.c3r + fb.cdr,
                                        (const __half*)(h->ws + fb.w_fwd), (const float*)(h->ws + fb.bias), &t);
        } else {
          t.out32 = (float*)red32.base;
          rc = umma_conv_bind_fwd(h->umma_ctx, fb.fwd, xp, redp, h->F, fb.cx, fb.c3r + fb.cdr, 1, 0, 1, (const __half*)(h->ws + fb.w_fwd),
                                  (const float*)(h->ws + fb.bias), &t);
        }
        if (rc) return h->fail(rc, "tc fused fwd bind(" + o3.id + "): " + ssnb::thread_error());
        if (h->cfg.training) {
          View dredp = h->planes(o3.out_val, true); dredp.C = fb.c3r + fb.cdr;
          View d1p = fb.op1 >= 0 ? h->planes(h->ops[fb.op1].out_val, true) : dredp;
          View dxp = h->planes(o3.in_val, true); dxp.base = nullptr; dxp.lo_off = 0;
          UmmaTcOpts tg; tg.w_lo_off = (long long)fb.w_dg_plane; tg.out32 = (float*)h->view(o3.in_val, true).base; tg.alpha = 1.0f / gs; tg.alpha_dev = alpha_dev;
          rc = umma_conv_bind_fused_dgrad(h->umma_ctx, fb.dgrad, d1p, dredp, dxp, h->F, fb.cx, fb.c1, fb.c3r + fb.cdr, (const __half*)(h->ws + fb.w_dg),
                                          od.grad_accumulate, &tg);
          if (rc) return h->fail(rc, "tc fused dgrad bind(" + o3.id + "): " + ssnb::thread_error());
          // zero the K padding of the concatenated data-gradient weights once (both planes); split_all_kernel never writes it
          if (cudaMemset(h->ws + fb.w_dg, 0, 2 * fb.w_dg_plane) != cudaSuccess) cudaGetLastError();
        }
        fb.enabled = true;
        const int leader = fb.op1 >= 0 ? fb.op1 : fb.op_r3;
        for (int j : {fb.op1, fb.op_r3, fb.op_rd})
          if (j >= 0) { h->ops[j].fuse_block = (int)bi; h->ops[j].fuse_role = (j == leader) ? 1 : 2; }
      }
    }
    // ReLU-mask fusion (same rule as the FAST schedule below): the consumer with the smallest forward index is the LAST writer
    // of a value's gradient in the reverse schedule; when that is a tensor-core data gradient its fp32 epilogue applies
    // dz = dy * (y > 0) and emits the value's gradient operand planes (dz * grad_scale), so the producing convolutions run
    // neither a mask pass nor a split pass: their bias gradients ride on the weight-gradient MMAs (ones operand).
    // SSNB_DISABLE_FUSION=1 keeps one mask + bias + split pass per convolution.
    const char* disf_tc = getenv("SSNB_DISABLE_FUSION");
    if (use_tc && h->cfg.training && !(disf_tc && disf_tc[0] == '1')) {
      h->fold_pools = true;
      std::vector<int> first_consumer(h->vals.size(), -1);
      for (int i = 0; i < (int)h->ops.size(); ++i)
        if (first_consumer[h->ops[i].in_val] < 0) first_consumer[h->ops[i].in_val] = i;
      for (size_t v = 0; v < h->vals.size(); ++v) {
        const int fc = first_consumer[v];
        if (fc < 0 || h->vals[v].name == "data" || !h->bufs[h->vals[v].buf].plane) continue;
        bool conv_made = false;                    // only buffers that hold convolution outputs have a ReLU to differentiate
        for (const Op& q : h->ops) conv_made = conv_made || (q.kind == OP_CONV && h->vals[q.out_val].buf == h->vals[v].buf);
        if (!conv_made) continue;
        Op& c = h->ops[fc];
        if (c.kind == OP_CONV && c.fuse_role == 1 && h->fused[c.fuse_block].enabled) {
          c.dgrad_masks = true;
          umma_conv_set_mask_tc(h->fused[c.fuse_block].dgrad, h->view((int)v, false), h->planes((int)v, true), gs, h->tc_flag);
        } else if (c.kind == OP_CONV && c.fuse_role == 0 && c.umma_dgrad.enabled) {
          c.dgrad_masks = true;
          umma_conv_set_mask_tc(c.umma_dgrad, h->view((int)v, false), h->planes((int)v, true), gs, h->tc_flag);
        }
      }
      for (Op& o : h->ops) {
        if (o.kind != OP_CONV) continue;
        int w = o.out_val;
        if (first_consumer[w] < 0) {               // a slice of a concat buffer: gradients are written through the whole-buffer value
          const Value& ov = h->vals[o.out_val];
          for (size_t v = 0; v < h->vals.size(); ++v)
            if (h->vals[v].buf == ov.buf && h->vals[v].coff == 0 && h->vals[v].C == h->bufs[ov.buf].C && first_consumer[v] >= 0) { w = (int)v; break; }
        }
        if (first_consumer[w] >= 0 && h->ops[first_consumer[w]].dgrad_masks) o.dy_premasked = true;
        o.bias_in_wgrad = o.dy_premasked && o.conv != 0 && o.umma_wgrad.enabled && o.umma_wgrad.p.taps_per_cta * o.umma_wgrad.p.mma_n + 16 <= 512;
      }
    }
    return SSNB_OK;
  }
  // bind tcgen05 plans (tensor maps need final addresses); SSNB_DISABLE_UMMA=1 keeps FAST mode on the SIMT kernels
  const char* dis = getenv("SSNB_DISABLE_UMMA");
  const bool use_umma = h->fp16 && !(dis && dis[0] == '1');
  for (Op& o : h->ops) {
    o.umma.enabled = false; o.umma_dgrad.enabled = false; o.umma_wgrad.enabled = false;
    if (o.kind != OP_CONV || !use_umma) continue;
    const ConvSpec& c = h->convs[o.conv];
    const char* disw = getenv("SSNB_DISABLE_UMMA_WGRAD");
    const bool use_wgrad = h->cfg.training && !(disw && disw[0] == '1');
    const View in = h->view(o.in_val, false), out = h->view(o.out_val, false);
    int rc = 0;
    if (o.conv == 0) {
      // conv1 7x7/2: four vertical taps over the packed space-to-depth input (r = 2*dr + a - 1, s = 2*ds + b - 1)
      const int Ck = 4 * h->Cs;
      View xs; xs.base = h->ws + h->s2d_off; xs.H = 112; xs.W = 112; xs.C = Ck; xs.pitch = Ck; xs.coff = 0;
      int dy[4], dx[4];
      for (int t = 0; t < 4; ++t) { dy[t] = t - 2; dx[t] = 0; }
      rc = umma_conv_bind_taps(h->umma_ctx, o.umma, xs, out, h->F, Ck, c.cout, 4, dy, dx, (const __half*)(h->ws + h->s2d_w_off),
                               (const float*)(h->ws + h->packed[0].bias), 1);
      if (rc) return h->fail(rc, "umma conv1 bind: " + ssnb::thread_error());
      if (use_wgrad) {
        rc = umma_wgrad_bind_taps(h->umma_ctx, o.umma_wgrad, h->view(o.out_val, true), xs, h->F, Ck, c.cout, 4, dy, dx,
                                  (float*)(h->ws + o.partial_off), 128);
        if (rc) return h->fail(rc, "umma conv1 wgrad bind: " + ssnb::thread_error());
      }
      continue;
    }
    if (c.cin % 8 != 0 || c.k * c.k > UMMA_MAX_TAPS) continue;
    rc = umma_conv_bind_fwd(h->umma_ctx, o.umma, in, out, h->F, c.cin, c.cout, c.k, c.pad, c.stride,
                            (const __half*)(h->ws + h->packed[o.conv].wd), (const float*)(h->ws + h->packed[o.conv].bias));
    if (rc) return h->fail(rc, "umma_conv_bind_fwd(" + c.id + "): " + ssnb::thread_error());
    if (!h->cfg.training) continue;
    // backward operands: the output gradient (stride-2 layers: its zero-upsampled copy at input resolution)
    View dz = h->view(o.out_val, true);
    if (c.stride == 2) { dz.base = h->ws + h->up_off; dz.H = in.H; dz.W = in.W; dz.C = c.cout; dz.pitch = c.cout; dz.coff = 0; }
    rc = umma_conv_bind_dgrad(h->umma_ctx, o.umma_dgrad, dz, h->view(o.in_val, true), h->F, c.cin, c.cout, c.k, c.pad,
                              (const __half*)(h->ws + h->packed[o.conv].wf), o.grad_accumulate);
    if (rc) return h->fail(rc, "umma_conv_bind_dgrad(" + c.id + "): " + ssnb::thread_error());
    if (use_wgrad) {
      // stride-2 layers: dz at its own (output) resolution, the x boxes step over the input with element stride 2
      rc = umma_wgrad_bind(h->umma_ctx, o.umma_wgrad, h->view(o.out_val, true), in, h->F, c.cin, c.cout, c.k, c.pad,
                           (float*)(h->ws + o.partial_off), o.tsplits, c.stride);
      if (rc) return h->fail(rc, "umma_wgrad_bind(" + c.id + "): " + ssnb::thread_error());
    }
  }
  // horizontal fusion of the sibling 1x1 convolutions of each inception block (SSNB_DISABLE_FUSION=1 turns it off)
  const char* disf = getenv("SSNB_DISABLE_FUSION");
  h->fold_pools = !(disf && disf[0] == '1');
  for (Op& o : h->ops) { o.fuse_role = 0; o.fuse_block = -1; }
  for (size_t bi = 0; bi < h->fused.size(); ++bi) {
    FusedBlock& fb = h->fused[bi];
    fb.enabled = false;
    if (!use_umma || (disf && disf[0] == '1')) continue;
    Op& o3 = h->ops[fb.op_r3]; Op& od = h->ops[fb.op_rd];
    const View x = h->view(o3.in_val, false);
    View red = h->view(o3.out_val, false); red.C = fb.c3r + fb.cdr;          // both reduce outputs: adjacent slices of one buffer
    int rc;
    if (fb.op1 >= 0) rc = umma_conv_bind_fused_fwd(h->umma_ctx, fb.fwd, x, h->view(h->ops[fb.op1].out_val, false), red, h->F, fb.cx, fb.c1,
                                                  fb.c3r + fb.cdr, (const __half*)(h->ws + fb.w_fwd), (const float*)(h->ws + fb.bias));
    else rc = umma_conv_bind_fwd(h->umma_ctx, fb.fwd, x, red, h->F, fb.cx, fb.c3r + fb.cdr, 1, 0, 1, (const __half*)(h->ws + fb.w_fwd),
                                 (const float*)(h->ws + fb.bias));
    if (rc) return h->fail(rc, "fused fwd bind(" + o3.id + "): " + ssnb::thread_error());
    if (h->cfg.training) {
      View dred = h->view(o3.out_val, true); dred.C = fb.c3r + fb.cdr;
      View d1 = fb.op1 >= 0 ? h->view(h->ops[fb.op1].out_val, true) : dred;
      rc = umma_conv_bind_fused_dgrad(h->umma_ctx, fb.dgrad, d1, dred, h->view(o3.in_val, true), h->F, fb.cx, fb.c1, fb.c3r + fb.cdr,
                                      (const __half*)(h->ws + fb.w_dg), od.grad_accumulate);
      if (rc) return h->fail(rc, "fused dgrad bind(" + o3.id + "): " + ssnb::thread_error());
    }
    fb.enabled = true;
    const int leader = fb.op1 >= 0 ? fb.op1 : fb.op_r3;
    for (int j : {fb.op1, fb.op_r3, fb.op_rd})
      if (j >= 0) { h->ops[j].fuse_block = (int)bi; h->ops[j].fuse_role = (j == leader) ? 1 : 2; }
  }
  // ReLU-mask fusion: the consumer with the smallest forward index is the last writer of a value's gradient in the
  // reverse schedule (sibling followers are folded into their leader); if that writer is a tcgen05 data gradient or the
  // global pool, it applies dz = dy * (y > 0) in its epilogue and the producing conv skips its own mask pass.
  for (Op& o : h->ops) { o.dgrad_masks = false; o.dy_premasked = false; }
  if (use_umma && h->cfg.training) {
    std::vector<int> first_consumer(h->vals.size(), -1);
    for (int i = 0; i < (int)h->ops.size(); ++i)
      if (first_consumer[h->ops[i].in_val] < 0) first_consumer[h->ops[i].in_val] = i;
    for (size_t v = 0; v < h->vals.size(); ++v) {
      const int fc = first_consumer[v];
      if (fc < 0 || h->vals[v].name == "data") continue;
      bool conv_made = false;                    // only buffers that hold convolution outputs have a ReLU to differentiate
      for (const Op& q : h->ops) conv_made = conv_made || (q.kind == OP_CONV && h->vals[q.out_val].buf == h->vals[v].buf);
      if (!conv_made) continue;
      Op& c = h->ops[fc];
      if (c.kind == OP_GPOOL) c.dgrad_masks = true;
      else if (c.kind == OP_CONV && (c.fuse_role == 1 ? h->fused[c.fuse_block].enabled : (c.fuse_role == 0 && c.umma_dgrad.enabled))) {
        c.dgrad_masks = true;
        UmmaConvPlan& dg = c.fuse_role == 1 ? h->fused[c.fuse_block].dgrad : c.umma_dgrad;
        if (int rc = umma_conv_set_mask(h->umma_ctx, dg, h->view((int)v, false))) return h->fail(rc, "mask fusion(" + c.id + "): " + ssnb::thread_error());
      }
    }
    for (Op& o : h->ops) {
      if (o.kind != OP_CONV) continue;
      int w = o.out_val;
      if (first_consumer[w] < 0) {               // a slice of a concat buffer: gradients are written through the whole-buffer value
        const Value& ov = h->vals[o.out_val];
        for (size_t v = 0; v < h->vals.size(); ++v)
          if (h->vals[v].buf == ov.buf && h->vals[v].coff == 0 && h->vals[v].C == h->bufs[ov.buf].C && first_consumer[v] >= 0) { w = (int)v; break; }
      }
      if (first_consumer[w] >= 0 && h->ops[first_consumer[w]].dgrad_masks) o.dy_premasked = true;
      o.bias_in_wgrad = o.dy_premasked && o.conv != 0 && o.umma_wgrad.enabled && o.umma_wgrad.p.taps_per_cta * o.umma_wgrad.p.mma_n + 16 <= 512;
    }
  }
  return SSNB_OK;
}

int ssnb_pack_weights(ssnb_handle h, const float* const* w, const float* const* b, const float* const* gamma,
                      const float* const* beta, const float* const* mean, const float* const* var, void* stream) {
  if (!h || !h->ws) return h ? h->fail(SSNB_ESTATE, "set_workspace first") : SSNB_EINVAL;
  cudaStream_t s = (cudaStream_t)stream;
  if (h->tc && cudaMemsetAsync(h->ws + h->wmax_off, 0, (h->convs.size() + 16) * 8, s) != cudaSuccess) return h->fail(SSNB_ECUDA, "pack_weights: memset");
  {
    // fold + re-layout of all 69 layers in a few launches (PACK_MAX entries per launch); EXACT_TC: every fold launch first (the
    // layers of a fused sibling block share one absmax slot), then the hi/lo splits
    struct Member { int block = -1, row = 0, col = 0; };
    std::vector<Member> member(h->convs.size());
    for (size_t bi = 0; bi < h->fused.size(); ++bi) {
      const FusedBlock& fb = h->fused[bi];
      if (!fb.enabled) continue;
      const int k1p = (fb.c1 + 63) / 64 * 64;
      int row = 0, col = 0;
      for (int j : {fb.op1, fb.op_r3, fb.op_rd}) {
        if (j < 0) continue;
        const int ci = h->ops[j].conv;
        member[ci].block = (int)bi; member[ci].row = row; member[ci].col = col;
        row += h->convs[ci].cout;
        col += (j == fb.op1) ? k1p : h->convs[ci].cout;
      }
    }
    std::vector<PackTable> pt(1);
    std::vector<SplitTable> stt(1);
    std::vector<int> pblocks(1, 0), sblocks(1, 0);
    pt[0].n = 0; pt[0].pad_ = 0; stt[0].n = 0; stt[0].pad_ = 0;
    for (size_t i = 0; i < h->convs.size(); ++i) {
      const ConvSpec& c = h->convs[i];
      const PackedConv& p = h->packed[i];
      const long long n = (long long)c.cout * c.cin * c.k * c.k;
      if (pt.back().n == PACK_MAX) { pt.emplace_back(); pt.back().n = 0; pt.back().pad_ = 0; pblocks.push_back(0); stt.emplace_back(); stt.back().n = 0; stt.back().pad_ = 0; sblocks.push_back(0); }
      const Member& mb = member[i];
      const FusedBlock* fb = mb.block >= 0 ? &h->fused[mb.block] : nullptr;
      PackEntry& q = pt.back().e[pt.back().n++];
      q.w = w[i]; q.b = b[i]; q.gamma = gamma[i]; q.beta = beta[i]; q.mean = mean[i]; q.var = var[i];
      q.wf = h->ws + p.wf; q.wd = h->ws + p.wd; q.bias = (float*)(h->ws + p.bias); q.scale = (float*)(h->ws + p.scale);
      q.absmax = h->tc ? (float*)(h->ws + p.wmax) : nullptr;
      q.cout = c.cout; q.cin = c.cin; q.k = c.k; q.block0 = pblocks.back();
      q.nofold = (h->bn1_train && i == 0) ? 1 : 0; q.pad_[0] = q.pad_[1] = q.pad_[2] = 0;
      q.bias_b = (h->tc && fb) ? (float*)(h->ws + fb->bias) + mb.row : nullptr;
      pblocks.back() += pack_ctas(c.cout, c.cin, c.k);
      if (h->tc) {
        SplitEntry& e = stt.back().e[stt.back().n++];
        e.wf = (const float*)(h->ws + p.wf); e.wd = (const float*)(h->ws + p.wd);
        e.wf16 = (__half*)(h->ws + p.wf16); e.wd16 = (__half*)(h->ws + p.wd16); e.plane_bytes = (long long)p.wplane; e.n = n;
        e.absmax = (const float*)(h->ws + p.wmax); e.inv_scale = (float*)(h->ws + p.wmax) + 1; e.block0 = sblocks.back(); e.pad_ = 0;
        e.wd16_b = nullptr; e.wf16_b = nullptr; e.b_plane_bytes = 0; e.b_pitch = 0; e.cout = c.cout;
        if (fb) {
          const int kf = (fb->c1 + 63) / 64 * 64 + fb->c3r + fb->cdr;
          e.wd16_b = (__half*)(h->ws + fb->w_fwd) + (size_t)mb.row * fb->cx;      // stacked forward rows [n][cx]
          e.wf16_b = (__half*)(h->ws + fb->w_dg) + mb.col;                         // column block of [cx][kf]
          e.b_pitch = kf;
          // both fused buffers are written through ONE plane distance per entry: the kernel applies it to wd16_b and wf16_b alike,
          // so the two buffers are planned with equal plane sizes (max of the two)
          e.b_plane_bytes = (long long)std::max(fb->w_fwd_plane, fb->w_dg_plane);
        }
        sblocks.back() += (int)((n + 255) / 256);
      }
    }
    for (size_t k = 0; k < pt.size(); ++k) {
      int rc = h->fp16 ? launch_pack_all<__half>(pt[k], pblocks[k], s) : launch_pack_all<float>(pt[k], pblocks[k], s);
      if (rc) return h->fail(rc, "pack_weights: " + ssnb::thread_error());
    }
    if (h->tc)
      for (size_t k = 0; k < stt.size(); ++k)
        if (int rc = launch_split_all(stt[k], sblocks[k], s)) return h->fail(rc, "pack_weights split: " + ssnb::thread_error());
  }
  if (h->tc && h->ops.size() && h->ops[0].umma.enabled) {
    for (int pl = 0; pl < 2; ++pl) {
      int rc = launch_pack_conv1_s2d((const __half*)(h->ws + h->packed[0].wd16 + pl * h->packed[0].wplane), h->convs[0].cout, h->convs[0].cin, h->Cs,
                                     (__half*)(h->ws + h->s2d_w_off + pl * h->s2d_w_plane), s);
      if (rc) return h->fail(rc, "pack conv1 s2d (tc): " + ssnb::thread_error());
    }
  }
  if (h->fp16 && h->ops.size() && h->ops[0].umma.enabled) {
    int rc = launch_pack_conv1_s2d((const __half*)(h->ws + h->packed[0].wd), h->convs[0].cout, h->convs[0].cin, h->Cs,
                                   (__half*)(h->ws + h->s2d_w_off), s);
    if (rc) return h->fail(rc, "pack conv1 s2d: " + ssnb::thread_error());
  }
  for (FusedBlock& fb : h->fused) {
    if (!fb.enabled || !h->fp16) continue;          // EXACT_TC: split_all_kernel wrote the fused operands directly
    // forward: rows of wd ([co][ci]) stacked; bias stacked.  data gradient: wf ([ci][co]) concatenated along K,
    // the 1x1 part padded to a multiple of 64 so each K chunk has a single activation source.
    const int k1p = (fb.c1 + 63) / 64 * 64, kf = k1p + fb.c3r + fb.cdr;
    __half* wfwd = (__half*)(h->ws + fb.w_fwd); float* bias = (float*)(h->ws + fb.bias); __half* wdg = (__half*)(h->ws + fb.w_dg);
    if (cudaMemsetAsync(wdg, 0, (size_t)fb.cx * kf * 2, s) != cudaSuccess) return h->fail(SSNB_ECUDA, "fused pack: memset");
    int row = 0, col = 0;
    for (int j : {fb.op1, fb.op_r3, fb.op_rd}) {
      if (j < 0) { continue; }
      const int ci = h->ops[j].conv, co = h->convs[ci].cout;
      cudaError_t e1 = cudaMemcpyAsync(wfwd + (size_t)row * fb.cx, h->ws + h->packed[ci].wd, (size_t)co * fb.cx * 2, cudaMemcpyDeviceToDevice, s);
      cudaError_t e2 = cudaMemcpyAsync(bias + row, h->ws + h->packed[ci].bias, (size_t)co * 4, cudaMemcpyDeviceToDevice, s);
      cudaError_t e3 = cudaMemcpy2DAsync(wdg + col, (size_t)kf * 2, h->ws + h->packed[ci].wf, (size_t)co * 2, (size_t)co * 2, fb.cx,
                                         cudaMemcpyDeviceToDevice, s);
      if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) return h->fail(SSNB_ECUDA, "fused pack: copy failed");
      row += co;
      col += (j == fb.op1) ? k1p : co;
    }
  }
  h->weights_ready = true;
  return SSNB_OK;
}

int ssnb_set_bn1(ssnb_handle h, const float* gamma, const float* beta, float* running_mean, float* running_var, float* dgamma, float* dbeta,
                 float momentum, float eps) {
  if (!h) return SSNB_EINVAL;
  if (!h->bn1_train) return h->fail(SSNB_ESTATE, "engine created without bn1_train");
  if (!gamma || !beta) return h->fail(SSNB_EINVAL, "set_bn1: gamma / beta are required");
  h->bn1_gamma = gamma; h->bn1_beta = beta; h->bn1_rmean = running_mean; h->bn1_rvar = running_var; h->bn1_dgamma = dgamma; h->bn1_dbeta = dbeta;
  h->bn1_momentum = momentum; h->bn1_eps = eps;
  return SSNB_OK;
}

int ssnb_backbone_fwd(ssnb_handle h, const float* input_nchw, float* feat, void* stream) {
  if (!h || !input_nchw || !feat) return h ? h->fail(SSNB_EINVAL, "null argument") : SSNB_EINVAL;
  if (!h->ws || !h->weights_ready) return h->fail(SSNB_ESTATE, "workspace/weights not set");
  cudaStream_t s = (cudaStream_t)stream;
  const View d = h->view(h->val_by_name["data"], false);
  int rc;
  h->s2d_ready = (h->fp16 || h->tc) && h->ops[0].umma.enabled;
  if (h->s2d_ready && h->tc) rc = launch_nchw_to_s2d_split(input_nchw, h->F, d.C, d.H, d.W, (__half*)(h->ws + h->s2d_off), (long long)h->s2d_plane, h->Cs, s);
  else if (h->s2d_ready) rc = launch_nchw_to_s2d(input_nchw, h->F, d.C, d.H, d.W, (__half*)(h->ws + h->s2d_off), h->Cs, s);
  else rc = h->fp16 ? launch_nchw_to_nhwc<__half>(input_nchw, h->F, d.C, d.H, d.W, d, 1.0f, s)
                    : launch_nchw_to_nhwc<float>(input_nchw, h->F, d.C, d.H, d.W, d, 1.0f, s);
  if (rc) { h->s2d_ready = false; return h->fail(rc, "input layout: " + ssnb::thread_error()); }
  for (size_t i = 0; i < h->ops.size(); ++i) {
    const Op& o = h->ops[i];
    if (o.fuse_role == 2) continue;                       // computed by its block's fused launch
    const bool prof = profiled_op("SSNB_PROFILE_FWD_OPS", o.id);
    if (prof) cudaProfilerStart();
    int r;
    if (o.fuse_role == 1) {
      const FusedBlock& fb = h->fused[o.fuse_block];
      double fl = 0.0;
      for (int j : {fb.op1, fb.op_r3, fb.op_rd}) if (j >= 0) fl += conv_flops(h, h->ops[j]);
      tag_next(0, fl);
      r = umma_conv_launch(h->umma_ctx, fb.fwd, s);
    } else r = run_fwd(h, o, input_nchw, feat, s);
    if (prof) cudaProfilerStop();
    if (r) { h->s2d_ready = false; return h->fail(r, "fwd " + o.id + ": " + ssnb::thread_error()); }
  }
  h->s2d_ready = false;
  return SSNB_OK;
}

int ssnb_bind_grads(ssnb_handle h, float* const* dw, float* const* db) {
  if (!h) return SSNB_EINVAL;
  h->dw.assign(h->convs.size(), nullptr); h->db.assign(h->convs.size(), nullptr);
  for (size_t i = 0; i < h->convs.size(); ++i) { if (dw) h->dw[i] = dw[i]; if (db) h->db[i] = db[i]; }
  return SSNB_OK;
}

int ssnb_backbone_bwd(ssnb_handle h, const float* dfeat, float* const* dw, float* const* db, void* stream) {
  return ssnb_backbone_bwd_range(h, dfeat, dw, db, -1, 0, stream);
}

int ssnb_backbone_bwd_range(ssnb_handle h, const float* dfeat, float* const* dw, float* const* db, int op_hi, int op_lo, void* stream) {
  if (!h || (!dfeat && (op_hi < 0 || op_hi >= (int)h->ops.size() - 1))) return h ? h->fail(SSNB_EINVAL, "null argument") : SSNB_EINVAL;
  if (!h->cfg.training) return h->fail(SSNB_ESTATE, "engine created without training=1");
  if (!h->ws || !h->weights_ready) return h->fail(SSNB_ESTATE, "workspace/weights not set");
  ssnb_bind_grads(h, dw, db);
  h->pending_finalize.clear();
  cudaStream_t s = (cudaStream_t)stream;
  // ops [first, last] of the reverse schedule; the global pool's backward (the first of them) reads the caller's dfeat
  auto run_range = [&](int hi, int lo) -> int {
    for (int i = hi; i >= lo; --i) {
      const Op& o = h->ops[i];
      const bool prof = profiled_op("SSNB_PROFILE_BWD_OPS", o.id);
      if (prof) cudaProfilerStart();
      int rc = run_bwd(h, o, dfeat, s, o.fuse_role != 0, true);   // siblings: mask/bias/wgrad only ...
      if (!rc && o.fuse_role == 1) {                                   // ... one fused data gradient
        const FusedBlock& fb = h->fused[o.fuse_block];
        double fl = 0.0;
        for (int j : {fb.op1, fb.op_r3, fb.op_rd}) if (j >= 0) fl += conv_flops(h, h->ops[j]);
        tag_next(1, fl);
        rc = umma_conv_launch(h->umma_ctx, fb.dgrad, s, h->fold_pools && o.dgrad_masks);
      }
      if (prof) cudaProfilerStop();
      if (rc) return h->fail(rc, "bwd " + o.id + ": " + ssnb::thread_error());
    }
    return 0;
  };
  auto finalize = [&]() -> int {
    const float gs = (h->fp16 || h->tc) ? h->cfg.grad_scale : 1.0f;
    FinalizeTable t; t.n = 0; t.total_blocks = 0; t.flag = h->tc_flag;
    auto flush = [&]() -> int { int rc = launch_wgrad_finalize_all(t, 1.0f / gs, h->grad_accumulate, s); t.n = 0; t.total_blocks = 0; return rc; };
    for (int oi : h->pending_finalize) {
      const Op& o = h->ops[oi];
      const ConvSpec& c = h->convs[o.conv];
      FinalizeEntry& q = t.e[t.n];
      q.partial = (const float*)(h->ws + o.partial_off); q.mult = (const float*)(h->ws + h->packed[o.conv].scale); q.dw = h->dw[o.conv];
      const bool bias_w = o.dy_premasked && o.bias_in_wgrad && h->db.size() && h->db[o.conv];
      q.bias_partial = bias_w ? (const float*)(h->ws + o.bias_partial_off) : nullptr; q.db = bias_w ? h->db[o.conv] : nullptr;
      q.splits = o.umma_wgrad.p.splits; q.taps = c.k * c.k; q.Cout = c.cout; q.Cin = c.cin; q.block0 = t.total_blocks; q.pad_ = 0;
      t.total_blocks += (int)(((long long)q.taps * q.Cout * q.Cin + 255) / 256);
      if (++t.n == FIN_MAX) if (int rc = flush()) { h->pending_finalize.clear(); return h->fail(rc, "finalize: " + ssnb::thread_error()); }
    }
    h->pending_finalize.clear();
    if (int rc = flush()) return h->fail(rc, "finalize: " + ssnb::thread_error());
    return 0;
  };
  const int last = (int)h->ops.size() - 1;
  if (op_hi < 0 || op_hi > last) op_hi = last;
  if (op_lo < 0 || op_lo > op_hi) return h->fail(SSNB_EINVAL, "backbone_bwd_range: bad op range");
  if (int rc = run_range(op_hi, op_lo)) return rc;
  return finalize();
}

int ssnb_set_grad_accumulate(ssnb_handle h, int accumulate) {
  if (!h) return SSNB_EINVAL;
  h->grad_accumulate = accumulate ? 1 : 0;
  return SSNB_OK;
}

int ssnb_num_ops(ssnb_handle h) { return h ? (int)h->ops.size() : 0; }

int ssnb_op_info(ssnb_handle h, int op, char* kind, int kind_cap, char* in_name, int in_cap, char* out_name, int out_cap) {
  if (!h || op < 0 || op >= (int)h->ops.size()) return SSNB_EINVAL;
  static const char* kn[] = {"conv", "maxpool", "avgpool", "gpool", "bn"};
  const Op& o = h->ops[op];
  if (kind) snprintf(kind, kind_cap, "%s", kn[o.kind]);
  if (in_name) snprintf(in_name, in_cap, "%s", h->vals[o.in_val].name.c_str());
  if (out_name) snprintf(out_name, out_cap, "%s", o.out_val >= 0 ? h->vals[o.out_val].name.c_str() : "feat");
  return SSNB_OK;
}

int ssnb_value_shape(ssnb_handle h, const char* name, int* c, int* hh, int* ww) {
  if (!h || !name) return SSNB_EINVAL;
  auto it = h->val_by_name.find(name);
  if (it == h->val_by_name.end()) return h->fail(SSNB_EINVAL, std::string("unknown value ") + name);
  const View v = h->view(it->second, false);
  if (c) *c = v.C; if (hh) *hh = v.H; if (ww) *ww = v.W;
  return SSNB_OK;
}

int ssnb_value_write(ssnb_handle h, const char* name, int grad, const float* src_nchw, void* stream) {
  if (!h || !name || !src_nchw || !h->ws) return SSNB_EINVAL;
  auto it = h->val_by_name.find(name);
  if (it == h->val_by_name.end()) return h->fail(SSNB_EINVAL, std::string("unknown value ") + name);
  if (grad && !h->cfg.training) return h->fail(SSNB_ESTATE, "no gradient buffers");
  const View v = h->view(it->second, grad != 0);
  const float sc = (grad && h->fp16) ? h->cfg.grad_scale : 1.0f;
  int rc = h->fp16 ? launch_nchw_to_nhwc<__half>(src_nchw, h->F, v.C, v.H, v.W, v, sc, (cudaStream_t)stream)
                   : launch_nchw_to_nhwc<float>(src_nchw, h->F, v.C, v.H, v.W, v, sc, (cudaStream_t)stream);
  if (!rc && h->tc && !grad) rc = tc_split_value(h, it->second, false, 1.0f, (cudaStream_t)stream);   // activation planes follow the fp32 value
  return rc ? h->fail(rc, ssnb::thread_error()) : SSNB_OK;
}

int ssnb_value_read(ssnb_handle h, const char* name, int grad, float* dst_nchw, void* stream) {
  if (!h || !name || !dst_nchw || !h->ws) return SSNB_EINVAL;
  auto it = h->val_by_name.find(name);
  if (it == h->val_by_name.end()) return h->fail(SSNB_EINVAL, std::string("unknown value ") + name);
  if (grad && !h->cfg.training) return h->fail(SSNB_ESTATE, "no gradient buffers");
  if (grad & 2) {       // diagnostic: read hi + lo of the value's EXACT_TC operand planes (bit 0: gradient planes, un-scaled)
    if (!h->tc || !h->bufs[h->vals[it->second].buf].plane) return h->fail(SSNB_ESTATE, "value has no operand planes");
    int rc = launch_planes_to_nchw(h->planes(it->second, (grad & 1) != 0), h->F, (grad & 1) ? 1.0f / h->cfg.grad_scale : 1.0f, dst_nchw, (cudaStream_t)stream);
    return rc ? h->fail(rc, ssnb::thread_error()) : SSNB_OK;
  }
  const View v = h->view(it->second, grad != 0);
  const float sc = (grad && h->fp16) ? 1.0f / h->cfg.grad_scale : 1.0f;
  int rc = h->fp16 ? launch_nhwc_to_nchw<__half>(v, h->F, sc, dst_nchw, (cudaStream_t)stream)
                   : launch_nhwc_to_nchw<float>(v, h->F, sc, dst_nchw, (cudaStream_t)stream);
  return rc ? h->fail(rc, ssnb::thread_error()) : SSNB_OK;
}

int ssnb_run_op(ssnb_handle h, int op, int backward, void* stream) {
  if (!h || op < 0 || op >= (int)h->ops.size()) return SSNB_EINVAL;
  if (!h->ws || !h->weights_ready) return h->fail(SSNB_ESTATE, "workspace/weights not set");
  const Op& o = h->ops[op];
  if (o.kind == OP_GPOOL) return h->fail(SSNB_ENOSUPPORT, "run_op: global_pool runs through backbone_fwd/bwd");
  int rc = backward ? run_bwd(h, o, nullptr, (cudaStream_t)stream) : run_fwd(h, o, nullptr, nullptr, (cudaStream_t)stream);
  return rc ? h->fail(rc, o.id + ": " + ssnb::thread_error()) : SSNB_OK;
}

int ssnb_grad_overflow(ssnb_handle h, int clear) {
  // did a gradient leave the fp16 range under the loss scale since the last clear?  EXACT_TC: an operand plane saw
  // |dz * grad_scale| > 65504 or NaN; FAST: a weight-gradient sum came out inf / NaN (fp16 gradient storage overflowed).
  // Synchronises the device (one 4-byte read).
  if (!h) return -1;
  if (!h->tc_flag) return 0;
  int v = 0;
  if (cudaMemcpy(&v, h->tc_flag, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return -1; }
  if (v && clear) cudaMemset(h->tc_flag, 0, sizeof(int));
  return v ? 1 : 0;
}

int ssnb_timing_begin(void* stream) {
  for (TimingMark& m : ssnb::t_marks) ssnb::t_event_pool.push_back(m.ev);
  ssnb::t_marks.clear();
  ssnb::t_tag = LaunchTag();
  ssnb::t_timing = true;
  ssnb::timing_mark("(begin)", (cudaStream_t)stream);
  return SSNB_OK;
}

const char* ssnb_timing_report(void) {
  // closes the session, waits for the last launch and aggregates by (kernel, phase): "kernel\tphase\tlaunches\tms\tflop\n"
  ssnb::t_timing = false;
  ssnb::t_report.clear();
  if (ssnb::t_marks.empty()) return ssnb::t_report.c_str();
  if (cudaEventSynchronize(ssnb::t_marks.back().ev) != cudaSuccess) { cudaGetLastError(); return ssnb::t_report.c_str(); }
  struct Agg { int n = 0; double ms = 0, flop = 0; };
  std::map<std::pair<std::string, int>, Agg> agg;
  for (size_t i = 1; i < ssnb::t_marks.size(); ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ssnb::t_marks[i - 1].ev, ssnb::t_marks[i].ev) != cudaSuccess) { cudaGetLastError(); continue; }
    Agg& a = agg[{ssnb::t_marks[i].what, ssnb::t_marks[i].tag.phase}];
    a.n += 1; a.ms += ms; a.flop += ssnb::t_marks[i].tag.flop;
  }
  char line[256];
  for (const auto& kv : agg) {
    snprintf(line, sizeof line, "%s\t%d\t%d\t%.6f\t%.0f\n", kv.first.first.c_str(), kv.first.second, kv.second.n, kv.second.ms, kv.second.flop);
    ssnb::t_report += line;
  }
  return ssnb::t_report.c_str();
}

int64_t ssnb_launch_count(ssnb_handle h) { return h ? (int64_t)(g_launches.load() - h->launches0) : 0; }
int64_t ssnb_global_launch_count(void) { return (int64_t)g_launches.load(); }

}  // extern "C"
