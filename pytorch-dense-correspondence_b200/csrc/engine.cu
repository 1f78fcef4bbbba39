// Network-level orchestration of Resnet34_8s forward/backward behind the C ABI, plus the single-operator
// entry points.  The structure restated here is the reference's
//   PSD/vision/torchvision/models/resnet.py:112-265  (ResNet.__init__/_make_layer/forward, BasicBlock)
//   PSD/pytorch_segmentation_detection/models/resnet_dilated.py:283-322 (Resnet34_8s)
// configured as resnet34(fully_conv=True, output_stride=8, remove_avg_pool_layer=True).
#include <algorithm>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "conv.cuh"
#include "conv_tc.cuh"

namespace ddn {

std::atomic<long long> g_launches{0};
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

// ------------------------------------------------------------------------------------------------ profiler
static const char* kProfNames[PROF_NUM_CLASSES] = {"conv_fwd_simt", "conv_dgrad_simt", "conv_wgrad_simt", "conv_fwd_tc",
                                                   "conv_dgrad_tc", "conv_wgrad_tc", "loss_fwd", "loss_bwd"};
struct ProfRec { int cls; double work; cudaEvent_t a, b; };
static std::mutex g_prof_mu;
static std::vector<ProfRec> g_prof;
static size_t g_prof_used = 0;
static std::atomic<int> g_prof_on{0};

ProfScope::ProfScope(int cls, double work, cudaStream_t s) : slot(-1), st(s) {
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (g_prof_used == g_prof.size()) {
    if (g_prof.size() >= (1u << 17)) return;
    ProfRec r; r.cls = cls; r.work = work;
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
    g_prof.push_back(r);
  }
  slot = (int)g_prof_used++;
  g_prof[slot].cls = cls; g_prof[slot].work = work;
  cudaEventRecord(g_prof[slot].a, st);
}
ProfScope::~ProfScope() {
  if (slot < 0) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  cudaEventRecord(g_prof[slot].b, st);
}

// ------------------------------------------------------------------------------------------------ network description
struct ConvSpec { int cin, cout, k, stride, pad, dil; int64_t w_off; };
struct BnSpec { int C; int64_t g_off, b_off, rm_off, rv_off; };
struct BlockSpec { ConvSpec c1, c2, ds; BnSpec b1, b2, bd; bool has_ds; };

struct NetSpec {
  int D = 0;
  ConvSpec stem; BnSpec stem_bn;
  std::vector<BlockSpec> blocks;
  int64_t fc_w = 0, fc_b = 0, n_params = 0, n_buffers = 0;
  std::vector<ddn_tensor_entry> ptab, btab;
};

static void add_entry(std::vector<ddn_tensor_entry>& tab, int64_t& cursor, const std::string& name,
                      std::initializer_list<int> shape, int64_t* off_out) {
  ddn_tensor_entry e;
  memset(&e, 0, sizeof(e));
  snprintf(e.name, sizeof(e.name), "%s", name.c_str());
  e.ndim = (int)shape.size();
  int64_t n = 1; int i = 0;
  for (int s : shape) { e.shape[i++] = s; n *= s; }
  e.offset = cursor; e.numel = n;
  *off_out = cursor;
  cursor += (n + 3) / 4 * 4;   // keep every tensor 16-byte aligned inside the flat array
  tab.push_back(e);
}

static NetSpec build_spec(int D) {
  NetSpec s; s.D = D;
  int64_t pc = 0, bc = 0;
  auto conv = [&](const std::string& name, int cin, int cout, int k, int stride, int pad, int dil) {
    ConvSpec c{cin, cout, k, stride, pad, dil, 0};
    add_entry(s.ptab, pc, name + ".weight", {cout, cin, k, k}, &c.w_off);
    return c;
  };
  auto bn = [&](const std::string& name, int C) {
    BnSpec b{C, 0, 0, 0, 0};
    add_entry(s.ptab, pc, name + ".weight", {C}, &b.g_off);
    add_entry(s.ptab, pc, name + ".bias", {C}, &b.b_off);
    add_entry(s.btab, bc, name + ".running_mean", {C}, &b.rm_off);
    add_entry(s.btab, bc, name + ".running_var", {C}, &b.rv_off);
    return b;
  };
  s.stem = conv("conv1", 3, 64, 7, 2, 3, 1);
  s.stem_bn = bn("bn1", 64);
  // resnet.py:183-229 with output_stride = 8
  const int layers[4] = {3, 4, 6, 3}, planes[4] = {64, 128, 256, 512}, strides[4] = {1, 2, 2, 2};
  int inplanes = 64, current_stride = 4, current_dilation = 1;
  for (int L = 0; L < 4; ++L) {
    int stride = strides[L];
    bool ds = stride != 1 || inplanes != planes[L];
    if (ds) {
      if (current_stride == 8) { current_dilation *= stride; stride = 1; }
      else current_stride *= stride;
    }
    for (int i = 0; i < layers[L]; ++i) {
      std::string p = "layer" + std::to_string(L + 1) + "." + std::to_string(i);
      BlockSpec b; memset(&b, 0, sizeof(b));
      int st = i == 0 ? stride : 1;
      int dil = current_dilation;
      b.c1 = conv(p + ".conv1", inplanes, planes[L], 3, st, dil, dil);
      b.b1 = bn(p + ".bn1", planes[L]);
      b.c2 = conv(p + ".conv2", planes[L], planes[L], 3, 1, dil, dil);
      b.b2 = bn(p + ".bn2", planes[L]);
      b.has_ds = (i == 0) && ds;
      if (b.has_ds) {
        b.ds = conv(p + ".downsample.0", inplanes, planes[L], 1, st, 0, 1);
        b.bd = bn(p + ".downsample.1", planes[L]);
      }
      s.blocks.push_back(b);
      inplanes = planes[L];
    }
  }
  add_entry(s.ptab, pc, "fc.weight", {D, 512, 1, 1}, &s.fc_w);
  add_entry(s.ptab, pc, "fc.bias", {D}, &s.fc_b);
  s.n_params = pc; s.n_buffers = bc;
  return s;
}

static const NetSpec& get_spec(int D) {
  static std::mutex mu;
  static std::vector<NetSpec> cache;
  std::lock_guard<std::mutex> lk(mu);
  for (auto& s : cache) if (s.D == D) return s;
  cache.push_back(build_spec(D));
  return cache.back();
}

// ------------------------------------------------------------------------------------------------ workspace plan
// mode: DDN_MODE_INFER (eval statistics, BatchNorm folded into the conv epilogues, nothing kept), DDN_MODE_TRAIN (batch
// statistics, activations kept for backward), DDN_MODE_EVAL_SAVE (frozen running statistics, activations kept: the reference
// backpropagates through an eval()-mode network this way).
struct ConvBufs { size_t raw, stats; int Hin, Win, Hout, Wout; };   // stats: [G][C] mean, then [G][C] 1/sqrt(var+eps)
struct PlaneBufs { size_t hi, lo; };   // bf16 operand planes of an activation (tensor-core modes only)
struct BlockBufs { ConvBufs c1, c2, ds; size_t act1, out; PlaneBufs act1_p, out_p; };
struct Plan {
  int B, H, W, D, mode, precision;
  int H1, W1, Hp, Wp;
  size_t x4, stem_raw, stem_stats, pool_out, argmax;
  PlaneBufs pool_p, grad_p, patch_p;  // pooled stem output; current d(raw conv output); 7x7/2 stem patches [B,H1,W1,192]
  size_t wws;                         // packed-weight staging of the tensor-core convs
  bool tc;
  std::vector<BlockBufs> blk;
  size_t low, dlow;
  size_t wpack, wpack2, dwp, scratch[4];
  size_t acc, sums;                   // BatchNorm accumulator (bn_stats.cuh) and the backward's per-group sums
  size_t dwp_all;                     // [n_params + 64*192] floats: every conv's [taps][Cout][Cin] gradient accumulator (tensor-core modes)
  size_t scratch_elems;
  size_t total;
};

static float* stat_mean(char* ws, const ConvBufs& cb) { return reinterpret_cast<float*>(ws + cb.stats); }

static int make_plan(Plan* p, int B, int H, int W, int D, int mode, int precision) {
  DDN_CHECK_ARG(B >= 1 && H >= 32 && W >= 32 && H % 8 == 0 && W % 8 == 0, "need B>=1 and H, W multiples of 8 (>=32); got B=%d H=%d W=%d", B, H, W);
  DDN_CHECK_ARG(D >= 1 && D <= 32, "descriptor dimension must be in [1,32] (got %d)", D);
  DDN_CHECK_ARG(precision >= DDN_PRECISION_FP32_SIMT && precision <= DDN_PRECISION_BF16, "unknown precision %d", precision);
  DDN_CHECK_ARG(mode >= DDN_MODE_INFER && mode <= DDN_MODE_EVAL_SAVE, "unknown mode %d", mode);
  if (precision != DDN_PRECISION_FP32_SIMT && !tc_available()) {
    set_error("precision %d needs the tcgen05 conv path, which this build does not contain", precision);
    return DDN_EUNSUPPORTED;
  }
  const NetSpec& s = get_spec(D);
  p->B = B; p->H = H; p->W = W; p->D = D; p->mode = mode; p->precision = precision;
  const int G = BN_MAX_GROUPS;
  size_t cur = 0;
  auto alloc = [&](size_t bytes) { size_t o = cur; cur += align_up(bytes, 256); return o; };
  auto f32 = [&](int64_t n) { return alloc(sizeof(float) * (size_t)n); };
  p->H1 = (H + 6 - 7) / 2 + 1; p->W1 = (W + 6 - 7) / 2 + 1;
  p->Hp = (p->H1 - 1) / 2 + 1; p->Wp = (p->W1 - 1) / 2 + 1;
  p->tc = precision != DDN_PRECISION_FP32_SIMT;
  p->x4 = p->tc ? 0 : f32((int64_t)B * H * W * 4);
  p->stem_raw = f32((int64_t)B * p->H1 * p->W1 * 64);
  p->stem_stats = f32(2 * G * 64);
  // fp32 pooled output: the SIMT instrument's activations, and the first residual of the folded inference path
  p->pool_out = (p->tc && mode != DDN_MODE_INFER) ? 0 : f32((int64_t)B * p->Hp * p->Wp * 64);
  p->argmax = alloc((size_t)B * p->Hp * p->Wp * 64);
  auto planes = [&](int64_t n) { PlaneBufs pb{0, 0}; if (p->tc) { pb.hi = alloc(2 * (size_t)n); pb.lo = alloc(2 * (size_t)n); } return pb; };
  p->pool_p = planes((int64_t)B * p->Hp * p->Wp * 64);
  p->patch_p = planes((int64_t)B * p->H1 * p->W1 * 192);
  int h = p->Hp, w = p->Wp;
  size_t max_w = 0;
  int64_t max_act = (int64_t)B * p->H1 * p->W1 * 64;
  p->blk.clear();
  for (const BlockSpec& b : s.blocks) {
    BlockBufs bb;
    memset(&bb, 0, sizeof(bb));
    auto conv_bufs = [&](const ConvSpec& c, int hin, int win) {
      ConvBufs cb; cb.Hin = hin; cb.Win = win;
      cb.Hout = (hin + 2 * c.pad - c.dil * (c.k - 1) - 1) / c.stride + 1;
      cb.Wout = (win + 2 * c.pad - c.dil * (c.k - 1) - 1) / c.stride + 1;
      cb.raw = f32((int64_t)B * cb.Hout * cb.Wout * c.cout);
      cb.stats = f32(2 * G * c.cout);
      max_w = std::max(max_w, (size_t)c.k * c.k * c.cin * c.cout);
      max_act = std::max(max_act, (int64_t)B * cb.Hout * cb.Wout * c.cout);
      return cb;
    };
    bb.c1 = conv_bufs(b.c1, h, w);
    // tensor-core modes keep activations only as bf16 hi/lo planes; the fp32 SIMT instrument keeps fp32 tensors
    if (!p->tc) bb.act1 = f32((int64_t)B * bb.c1.Hout * bb.c1.Wout * b.c1.cout);
    bb.act1_p = planes((int64_t)B * bb.c1.Hout * bb.c1.Wout * b.c1.cout);
    bb.c2 = conv_bufs(b.c2, bb.c1.Hout, bb.c1.Wout);
    if (b.has_ds) bb.ds = conv_bufs(b.ds, h, w);
    if (!p->tc) bb.out = f32((int64_t)B * bb.c2.Hout * bb.c2.Wout * b.c2.cout);
    bb.out_p = planes((int64_t)B * bb.c2.Hout * bb.c2.Wout * b.c2.cout);
    h = bb.c2.Hout; w = bb.c2.Wout;
    p->blk.push_back(bb);
  }
  DDN_CHECK_ARG(h * 8 == H && w * 8 == W, "internal: trunk output %dx%d is not H/8 x W/8", h, w);
  p->low = f32((int64_t)B * D * h * w);
  p->dlow = f32((int64_t)B * D * h * w);
  max_w = std::max(max_w, (size_t)7 * 7 * 4 * 64);
  p->wpack = f32((int64_t)max_w); p->wpack2 = f32((int64_t)max_w); p->dwp = f32((int64_t)max_w);
  p->acc = alloc(bn_accum_bytes(512));
  p->sums = f32(3 * 2 * G * 512);     // [0]: standalone column-sum pass, [1], [2]: sums produced by a data-gradient epilogue
  p->scratch_elems = (size_t)max_act;
  for (int i = 0; i < 4; ++i) p->scratch[i] = f32((int64_t)max_act);
  p->grad_p = planes(max_act);
  p->wws = alloc(p->tc ? tc_weight_ws_bytes() : 0);
  p->dwp_all = (p->tc && mode != DDN_MODE_INFER) ? f32(s.n_params + 64 * 192) : 0;
  p->total = cur;
  return 0;
}

struct Ctx {
  const NetSpec* s; const Plan* p; char* ws; const float* params; float* buffers; float* grads;
  cudaStream_t st; float momentum, eps; int mode; int G;
  float* f(size_t off) const { return reinterpret_cast<float*>(ws + off); }
  __nv_bfloat16* h(size_t off) const { return reinterpret_cast<__nv_bfloat16*>(ws + off); }
  TcPlanes planes(const PlaneBufs& b) const { return TcPlanes{h(b.hi), h(b.lo)}; }
  float* mean(size_t stats) const { return f(stats); }
  float* invstd(size_t stats, int C) const { return f(stats) + (size_t)G * C; }
  BnAccum accum() const { return bn_accum_at(ws + p->acc, 512); }
  bool training() const { return mode == DDN_MODE_TRAIN; }
};

// Optional caller-owned caches of the packed bf16 weights (forward and data-gradient packs of every conv), registered with
// ddn_resnet34_8s_set_weight_cache(), one slot per parameter array (two networks in one process do not evict each other).
// Validity is decided on the device: every forward fingerprints the parameter array and re-packs only when it changed
// (tc_pack_all), so no host-side version bookkeeping can go stale.  Layout: [tensor][forward | dgrad][hi | lo] at byte
// offset w_off * 8, then the two fingerprints in the last 256 bytes.
struct WeightCache {
  char* base = nullptr; size_t bytes = 0; uint64_t version = 0; const float* params = nullptr; int precision = -1;
  bool fresh = true;
};
static std::vector<WeightCache> g_wcaches;
static std::mutex g_wcache_mu;

static WeightCache* find_cache(const float* params) {
  for (auto& wc : g_wcaches) if (wc.params == params && wc.base) return &wc;
  return nullptr;
}
static size_t pack_offset(const ConvSpec& cs, int dgrad) {
  const size_t slot = (size_t)cs.cout * cs.cin * cs.k * cs.k;                 // the cache reserves 4 x numel bf16 per tensor
  return ((size_t)cs.w_off * 2 + (size_t)dgrad * slot) * 2 * sizeof(__nv_bfloat16);
}

// start of every tensor-core forward: make the cached packs match the parameters (3 launches; packs only when they changed)
static int ensure_packs(const Ctx& c) {
  std::lock_guard<std::mutex> lk(g_wcache_mu);
  WeightCache* wc = find_cache(c.params);
  if (!wc || wc->precision != c.p->precision) return 0;
  const NetSpec& s = *c.s;
  if (wc->bytes < (size_t)s.n_params * 8 + 512) { set_error("weight cache too small"); return DDN_EWORKSPACE; }
  std::vector<TcPackEntry> tab;
  auto add = [&](const ConvSpec& cs, int dgrad, int kind) {
    TcPackEntry e; e.w_off = cs.w_off; e.dst_off = (int64_t)pack_offset(cs, dgrad); e.Cout = cs.cout; e.Cin = cs.cin; e.k = cs.k;
    e.dgrad = dgrad; e.kind = kind;
    tab.push_back(e);
  };
  add(s.stem, 0, 1);
  for (const BlockSpec& b : s.blocks) {
    add(b.c1, 0, 0); add(b.c1, 1, 0); add(b.c2, 0, 0); add(b.c2, 1, 0);
    if (b.has_ds) { add(b.ds, 0, 0); add(b.ds, 1, 0); }
  }
  unsigned long long* fp_new = reinterpret_cast<unsigned long long*>(wc->base + wc->bytes - 256);
  unsigned long long* fp_old = reinterpret_cast<unsigned long long*>(wc->base + wc->bytes - 128);
  int force = 0;
  if (wc->fresh) {
    DDN_CUDA(cudaMemsetAsync(wc->base + wc->bytes - 256, 0, 256, c.st));
    force = 1; wc->fresh = false;
  }
  return tc_pack_all(c.params, s.n_params, wc->base, tab.data(), (int)tab.size(), fp_new, fp_old, force, c.p->precision, c.st);
}

// packed planes of conv `cs` (mode 0 = forward, 1 = data gradient; stem: [64][192] patch-GEMM layout) from the cache, or
// nullptr when no cache is registered for this parameter array (the conv then packs into the staging area per call)
static const TcPlanes* cached_pack(const Ctx& c, const ConvSpec& cs, int dgrad, TcPlanes* out) {
  std::lock_guard<std::mutex> lk(g_wcache_mu);
  WeightCache* wc = find_cache(c.params);
  if (!wc || wc->precision != c.p->precision || wc->fresh) return nullptr;
  const size_t wel = cs.k == 7 ? (size_t)64 * 192 : (size_t)cs.cout * cs.cin * cs.k * cs.k;
  __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(wc->base + pack_offset(cs, dgrad));
  out->hi = hi; out->lo = hi + wel;
  return out;
}

static bool conv_on_tc(const Ctx& c, const ConvSpec& cs, int Hin, int Win) {
  return c.p->tc && tc_conv_supported(cs.cin, cs.cout, cs.k, cs.stride, cs.pad, cs.dil, Hin, Win);
}

// BatchNorm statistics request of a forward conv: batch statistics accumulated by the conv epilogue (training), or none
// (the statistics slots were filled from the running estimates by bn_eval_stats_all before the first conv)
static BnFwdFinal stats_request(const Ctx& c, const BnSpec& bs, const ConvBufs& cb, int64_t M) {
  BnFwdFinal f;
  f.a = c.accum();
  f.mean = c.mean(cb.stats); f.invstd = c.invstd(cb.stats, bs.C);
  f.running_mean = c.buffers + bs.rm_off; f.running_var = c.buffers + bs.rv_off;
  f.count = M / c.G; f.G = c.G; f.C = bs.C; f.momentum = c.momentum; f.eps = c.eps;
  return f;
}

// one conv (forward) + the statistics of the BatchNorm that follows it.
// Tensor-core convs read the bf16 planes of their input and accumulate the BN sums in their epilogue (the last CTA writes
// mean / invstd / running statistics); the fp32 SIMT convs read the fp32 tensor and the column sums come from a separate pass.
static int conv_bn_forward(const Ctx& c, const ConvSpec& cs, const BnSpec& bs, const float* in, const PlaneBufs& in_p,
                           const ConvBufs& cb, int N, int cin_eff) {
  const float* w = c.params + cs.w_off;
  float* raw = c.f(cb.raw);
  const int64_t M = (int64_t)N * cb.Hout * cb.Wout;
  const BnFwdFinal fin = stats_request(c, bs, cb, M);
  if (conv_on_tc(c, cs, cb.Hin, cb.Win)) {
    TcPlanes wpk_s; const TcPlanes* wpk = cached_pack(c, cs, 0, &wpk_s);
    return tc_conv_planes(c.planes(in_p), w, wpk, raw, nullptr, c.training() ? &fin : nullptr, N, cb.Hin, cb.Win, cs.cin, cs.cout, cs.k,
                          cs.stride, cs.dil, 0, c.p->precision, c.ws + c.p->wws, tc_weight_ws_bytes(), c.st);
  }
  ConvGeom g;
  DDN_TRY(conv_geom_init(&g, N, cb.Hin, cb.Win, cin_eff, cb.Hout, cb.Wout, cs.cout, cs.k, cs.k, cs.stride, 1, cs.pad, cs.dil));
  DDN_TRY(launch_pack_weights(w, c.f(c.p->wpack), cs.cout, cs.cin, cin_eff, cs.k, cs.k, 0, c.st));
  {
    ProfScope ps(PROF_CONV_FWD_SIMT, 2.0 * M * (double)cs.cout * cs.k * cs.k * cs.cin, c.st);
    DDN_TRY(launch_conv_gather_f32(in, c.f(c.p->wpack), nullptr, raw, g, c.st));
  }
  if (c.training())
    return launch_bn_stats(raw, M, bs.C, c.G, fin.a, fin.mean, fin.invstd, fin.running_mean, fin.running_var, c.momentum, c.eps, c.st);
  return 0;
}

// Inference (eval-mode BN) on the tensor-core path: BN is a per-channel multiply-add of the conv accumulator, so the conv
// epilogue applies it together with the residual add and the ReLU and writes the next conv's operand planes itself; no
// un-normalised conv output and no separate BN pass exist.  `out` / `out_p` may be absent (null / {0,0}).
static int conv_bn_folded(const Ctx& c, const ConvSpec& cs, const BnSpec& bs, const PlaneBufs& in_p, const ConvBufs& cb, int N,
                          float* out, const PlaneBufs* out_p, const float* addend, int relu) {
  float* scale = c.f(cb.stats); float* shift = c.f(cb.stats) + bs.C;     // the per-conv statistics slots hold scale / shift here
  DDN_TRY(launch_bn_fold(c.buffers + bs.rm_off, c.buffers + bs.rv_off, c.params + bs.g_off, c.params + bs.b_off, bs.C, c.eps,
                         scale, shift, c.st));
  TcPlanes wpk_s; const TcPlanes* wpk = cached_pack(c, cs, 0, &wpk_s);
  TcFoldedEpilogue ep = {scale, shift, relu, out_p ? c.h(out_p->hi) : nullptr, out_p ? c.h(out_p->lo) : nullptr};
  return tc_conv_planes(c.planes(in_p), c.params + cs.w_off, wpk, out, addend, nullptr, N, cb.Hin, cb.Win, cs.cin, cs.cout, cs.k,
                        cs.stride, cs.dil, 0, c.p->precision, c.ws + c.p->wws, tc_weight_ws_bytes(), c.st, &ep);
}

// every BatchNorm's statistics slots <- running estimates, in one launch (modes without batch statistics)
static int fill_eval_stats(const Ctx& c) {
  const NetSpec& s = *c.s; const Plan& p = *c.p;
  std::vector<BnEvalSeg> segs;
  auto add = [&](const BnSpec& bs, size_t stats_off) {
    BnEvalSeg sg; sg.rm_off = bs.rm_off; sg.rv_off = bs.rv_off; sg.stat_off = (int64_t)(stats_off / sizeof(float)); sg.C = bs.C;
    segs.push_back(sg);
  };
  add(s.stem_bn, p.stem_stats);
  for (size_t i = 0; i < s.blocks.size(); ++i) {
    add(s.blocks[i].b1, p.blk[i].c1.stats); add(s.blocks[i].b2, p.blk[i].c2.stats);
    if (s.blocks[i].has_ds) add(s.blocks[i].bd, p.blk[i].ds.stats);
  }
  return launch_bn_eval_stats_all(c.buffers, reinterpret_cast<float*>(c.ws), segs.data(), (int)segs.size(), c.G, c.eps, c.st);
}

static int net_forward(const Ctx& c, const float* x, float* y, float* low_nhwc) {
  const NetSpec& s = *c.s; const Plan& p = *c.p;
  const int B = p.B, G = c.G;
  const bool want_lo = p.precision == DDN_PRECISION_BF16X3;
  const bool fold = c.mode == DDN_MODE_INFER && p.tc;
  DDN_CUDA(cudaMemsetAsync(c.ws + p.acc, 0, bn_accum_bytes(512), c.st));     // the workspace arrives uninitialised
  if (p.tc) DDN_TRY(ensure_packs(c));
  if (!c.training() && !fold) DDN_TRY(fill_eval_stats(c));
  // stem: conv1 7x7/2 -> bn1 -> relu -> maxpool 3x3/2          (resnet.py:232-235)
  ConvBufs stem_cb{p.stem_raw, p.stem_stats, p.H, p.W, p.H1, p.W1};
  if (p.tc) {   // conv1 as a K = 192 GEMM over 7x7/2 patch planes, BN statistics from the conv epilogue
    DDN_TRY(tc_stem_patches(x, c.h(p.patch_p.hi), c.h(p.patch_p.lo), B, p.H, p.W, p.precision, c.st));
    const BnFwdFinal fin = stats_request(c, s.stem_bn, stem_cb, (int64_t)B * p.H1 * p.W1);
    TcPlanes wpk_s; const TcPlanes* wpk = cached_pack(c, s.stem, 0, &wpk_s);
    DDN_TRY(tc_stem_forward(c.planes(p.patch_p), c.params + s.stem.w_off, wpk, c.f(p.stem_raw), c.training() ? &fin : nullptr, B, p.H1,
                            p.W1, p.precision, c.ws + p.wws, tc_weight_ws_bytes(), c.st));
    if (fold) DDN_TRY(launch_bn_eval_stats(c.buffers + s.stem_bn.rm_off, c.buffers + s.stem_bn.rv_off, 64, G, c.eps,
                                           c.mean(p.stem_stats), c.invstd(p.stem_stats, 64), c.st));
  } else {
    DDN_TRY(launch_nchw_to_nhwc4(x, c.f(p.x4), B, p.H, p.W, c.st));
    DDN_TRY(conv_bn_forward(c, s.stem, s.stem_bn, c.f(p.x4), PlaneBufs{0, 0}, stem_cb, B, 4));
  }
  DDN_TRY(launch_stem_bn_relu_pool(c.f(p.stem_raw), c.mean(p.stem_stats), c.invstd(p.stem_stats, 64), c.params + s.stem_bn.g_off,
                                   c.params + s.stem_bn.b_off, (p.tc && c.mode != DDN_MODE_INFER) ? nullptr : c.f(p.pool_out), reinterpret_cast<uint8_t*>(c.ws + p.argmax),
                                   p.tc ? c.h(p.pool_p.hi) : nullptr, (p.tc && want_lo) ? c.h(p.pool_p.lo) : nullptr,
                                   B, p.H1, p.W1, 64, G, c.st));
  const float* cur = p.tc ? nullptr : c.f(p.pool_out);      // fp32 activations exist only in the SIMT instrument
  PlaneBufs cur_p = p.pool_p;
  for (size_t i = 0; i < s.blocks.size(); ++i) {        // BasicBlock.forward, resnet.py:53-69
    const BlockSpec& b = s.blocks[i]; const BlockBufs& bb = p.blk[i];
    int64_t M1 = (int64_t)B * bb.c1.Hout * bb.c1.Wout;
    if (fold && conv_on_tc(c, b.c1, bb.c1.Hin, bb.c1.Win) && conv_on_tc(c, b.c2, bb.c2.Hin, bb.c2.Win) &&
        (!b.has_ds || conv_on_tc(c, b.ds, bb.ds.Hin, bb.ds.Win))) {
      DDN_TRY(conv_bn_folded(c, b.c1, b.b1, cur_p, bb.c1, B, nullptr, &bb.act1_p, nullptr, 1));       // act1: planes only
      // the epilogue's residual addend is fp32: the pooled stem output for the first block, else the previous block's fp32
      // output, which the folded path keeps in that block's (otherwise unused) c2.raw slot
      const float* res = i == 0 ? c.f(p.pool_out) : c.f(p.blk[i - 1].c2.raw);
      if (b.has_ds) {
        DDN_TRY(conv_bn_folded(c, b.ds, b.bd, cur_p, bb.ds, B, c.f(bb.ds.raw), nullptr, nullptr, 0));  // bn_d(conv_d(x)), fp32
        res = c.f(bb.ds.raw);
      }
      DDN_TRY(conv_bn_folded(c, b.c2, b.b2, bb.act1_p, bb.c2, B, c.f(bb.c2.raw), &bb.out_p, res, 1));   // fp32 block output in c2.raw
      cur = c.f(bb.c2.raw);
      cur_p = bb.out_p;
      continue;
    }
    DDN_TRY(conv_bn_forward(c, b.c1, b.b1, cur, cur_p, bb.c1, B, b.c1.cin));
    BnApplyArgs a1;
    memset(&a1, 0, sizeof(a1));
    a1.x = c.f(bb.c1.raw); a1.mean = c.mean(bb.c1.stats); a1.invstd = c.invstd(bb.c1.stats, b.b1.C);
    a1.gamma = c.params + b.b1.g_off; a1.beta = c.params + b.b1.b_off;
    a1.y = p.tc ? nullptr : c.f(bb.act1); a1.hi = p.tc ? c.h(bb.act1_p.hi) : nullptr; a1.lo = (p.tc && want_lo) ? c.h(bb.act1_p.lo) : nullptr;
    a1.M = M1; a1.C = b.b1.C; a1.relu = 1; a1.G = G;
    DDN_TRY(launch_bn_apply(a1, c.st));
    DDN_TRY(conv_bn_forward(c, b.c2, b.b2, p.tc ? nullptr : c.f(bb.act1), bb.act1_p, bb.c2, B, b.c2.cin));
    BnApplyArgs a2;
    memset(&a2, 0, sizeof(a2));
    a2.x = c.f(bb.c2.raw); a2.mean = c.mean(bb.c2.stats); a2.invstd = c.invstd(bb.c2.stats, b.b2.C);
    a2.gamma = c.params + b.b2.g_off; a2.beta = c.params + b.b2.b_off;
    a2.y = p.tc ? nullptr : c.f(bb.out); a2.hi = p.tc ? c.h(bb.out_p.hi) : nullptr; a2.lo = (p.tc && want_lo) ? c.h(bb.out_p.lo) : nullptr;
    a2.M = M1; a2.C = b.b2.C; a2.relu = 1; a2.G = G;
    if (b.has_ds) {
      DDN_TRY(conv_bn_forward(c, b.ds, b.bd, cur, cur_p, bb.ds, B, b.ds.cin));
      a2.r = c.f(bb.ds.raw); a2.rmean = c.mean(bb.ds.stats); a2.rinvstd = c.invstd(bb.ds.stats, b.bd.C);
      a2.rgamma = c.params + b.bd.g_off; a2.rbeta = c.params + b.bd.b_off;
    } else if (p.tc) {           // identity residual straight from the block input's operand planes
      a2.r_hi = c.h(cur_p.hi); a2.r_lo = want_lo ? c.h(cur_p.lo) : nullptr;
    } else {
      a2.r = cur;
    }
    DDN_TRY(launch_bn_apply(a2, c.st));
    cur = p.tc ? nullptr : c.f(bb.out);
    cur_p = bb.out_p;
  }
  // fc (1x1 conv + bias) and the bilinear upsample back to the input size      (resnet.py:263, resnet_dilated.py:320)
  const int h8 = p.H / 8, w8 = p.W / 8;
  const bool feat_planes = p.tc;       // the features are read from the operand planes (hi + lo)
  DDN_TRY(launch_fc_forward(feat_planes ? nullptr : cur, feat_planes ? c.h(cur_p.hi) : nullptr,
                            (feat_planes && want_lo) ? c.h(cur_p.lo) : nullptr, c.params + s.fc_w, c.params + s.fc_b, c.f(p.low),
                            low_nhwc, (int64_t)h8 * w8, B, 512, p.D, c.st));
  DDN_TRY(launch_upsample_fwd(c.f(p.low), y, B * p.D, h8, w8, p.H, p.W, c.st));
  return 0;
}

// conv backward: dw -> grads (SIMT: immediately; tensor core: accumulated in dwp_all, converted per bucket), dx -> `dx`
// (+ addend) when dx != nullptr.  Tensor-core convs take the saved bf16 planes of their input and the planes of dY
// (p.grad_p, written by the BN backward that precedes this call); the fp32 SIMT convs take the fp32 tensors.
static int conv_backward(const Ctx& c, const ConvSpec& cs, const float* in, const PlaneBufs& in_p, const float* dy, float* dx,
                         const float* addend, int N, int Hin, int Win, int Hout, int Wout, int cin_eff, const TcBwdStats* bst = nullptr) {
  const Plan& p = *c.p;
  const float* w = c.params + cs.w_off;
  float* dw = c.grads + cs.w_off;
  const double fl = 2.0 * N * Hout * Wout * (double)cs.cout * cs.k * cs.k * cs.cin;
  if (conv_on_tc(c, cs, Hin, Win)) {
    DDN_TRY(tc_wgrad_planes(c.planes(in_p), c.planes(p.grad_p), nullptr, N, Hin, Win, cs.cin, cs.cout, cs.k, cs.stride, cs.dil,
                            p.precision, c.f(p.dwp_all) + cs.w_off, c.st));
    if (dx) {
      TcPlanes wpk_s; const TcPlanes* wpk = cached_pack(c, cs, 1, &wpk_s);
      if (cs.stride == 2)   // zero-insert the fp32 dY into the (now free) gradient planes, then an ordinary stride-1 dgrad
        DDN_TRY(tc_dgrad_strided(dy, c.planes(p.grad_p), w, wpk, dx, addend, N, Hin, Win, cs.cin, cs.cout, cs.k, p.precision,
                                 c.ws + p.wws, tc_weight_ws_bytes(), c.st, bst));
      else
        DDN_TRY(tc_conv_planes(c.planes(p.grad_p), w, wpk, dx, addend, nullptr, N, Hin, Win, cs.cin, cs.cout, cs.k, 1, cs.dil, 1,
                               p.precision, c.ws + p.wws, tc_weight_ws_bytes(), c.st, nullptr, bst));
    }
    return 0;
  }
  DDN_CHECK_ARG(bst == nullptr, "backward statistics can only ride on a tensor-core data gradient");
  ConvGeom g;
  DDN_TRY(conv_geom_init(&g, N, Hin, Win, cin_eff, Hout, Wout, cs.cout, cs.k, cs.k, cs.stride, 1, cs.pad, cs.dil));
  size_t wbytes = sizeof(float) * (size_t)cs.k * cs.k * cin_eff * cs.cout;
  DDN_TRY(launch_fill_zero(c.f(p.dwp), wbytes, c.st));
  {
    ProfScope ps(PROF_CONV_WGRAD_SIMT, fl, c.st);
    DDN_TRY(launch_conv_wgrad_f32(in, dy, c.f(p.dwp), g, c.st));
  }
  DDN_TRY(launch_unpack_wgrad(c.f(p.dwp), dw, cs.cout, cs.cin, cin_eff, cs.k, cs.k, c.st));
  if (dx) {
    ConvGeom gd;
    DDN_TRY(conv_geom_init(&gd, N, Hout, Wout, cs.cout, Hin, Win, cs.cin, cs.k, cs.k, 1, cs.stride, cs.dil * (cs.k - 1) - cs.pad, cs.dil));
    DDN_TRY(launch_pack_weights(w, c.f(p.wpack2), cs.cout, cs.cin, cs.cin, cs.k, cs.k, 1, c.st));
    ProfScope ps(PROF_CONV_DGRAD_SIMT, fl, c.st);
    DDN_TRY(launch_conv_gather_f32(dy, c.f(p.wpack2), addend, dx, gd, c.st));
  }
  return 0;
}

// BN backward of `bs` (output y = relu?(bn(raw) + res)) whose dx feeds conv `cs`'s backward: planes for a tensor-core conv,
// fp32 for a SIMT conv.  mask: the bf16 hi plane of y / the fp32 y / recomputed from raw (no residual) -- see BnBwdArgs.
// fused_slot > 0: the column sums were produced by the data-gradient epilogue that wrote `dy` (bwd_stats_for) -- skip that pass.
static int bn_backward_for(const Ctx& c, const BnSpec& bs, const ConvBufs& cb, const float* dy, const float* y_f32,
                           const __nv_bfloat16* y_hi, int relu, float* g_out, const ConvSpec& cs, int Hin, int Win, float* dx_f32, int64_t M,
                           int fused_slot = 0) {
  BnBwdArgs a;
  memset(&a, 0, sizeof(a));
  a.dy = dy; a.x = c.f(cb.raw); a.mean = c.mean(cb.stats); a.invstd = c.invstd(cb.stats, bs.C);
  a.gamma = c.params + bs.g_off; a.beta = c.params + bs.b_off;
  a.y = y_f32; a.y_hi = y_hi; a.g_out = g_out;
  a.dgamma = c.grads + bs.g_off; a.dbeta = c.grads + bs.b_off;
  a.acc = c.accum(); a.sums = c.f(c.p->sums) + (size_t)fused_slot * 2 * c.G * 512;
  a.sums_ready = fused_slot > 0;
  a.M = M; a.C = bs.C; a.relu = relu; a.training = c.training() ? 1 : 0; a.G = c.G;
  if (conv_on_tc(c, cs, Hin, Win)) {
    a.dx = cs.stride == 2 ? dx_f32 : nullptr;      // the strided data gradient re-reads dY in fp32 (zero insertion)
    a.dx_hi = c.h(c.p->grad_p.hi);
    a.dx_lo = c.p->precision == DDN_PRECISION_BF16X3 ? c.h(c.p->grad_p.lo) : nullptr;
  } else {
    a.dx = dx_f32;
  }
  return launch_bn_backward(a, c.st);
}

// Column sums of BatchNorm `bs` (y = relu(bn(raw) [+ residual])) computed by the epilogue of the tensor-core data gradient that
// produces its dY (conv_tc.cuh TcBwdStats) instead of a separate pass over dY and raw.
static bool bwd_stats_for(const Ctx& c, const BnSpec& bs, const ConvBufs& cb, const __nv_bfloat16* y_hi, int slot, TcBwdStats* out) {
  if (!c.p->tc) return false;
  memset(out, 0, sizeof(*out));
  out->raw = c.f(cb.raw); out->y_hi = y_hi; out->mean = c.mean(cb.stats); out->invstd = c.invstd(cb.stats, bs.C);
  out->gamma = c.params + bs.g_off; out->beta = c.params + bs.b_off; out->relu = 1;
  out->fin.a = c.accum(); out->fin.sums = c.f(c.p->sums) + (size_t)slot * 2 * c.G * 512;
  out->fin.dgamma = c.grads + bs.g_off; out->fin.dbeta = c.grads + bs.b_off; out->fin.G = c.G; out->fin.C = bs.C;
  return true;
}

// gradient buckets, in the order the backward completes them (ddn_grad_bucket_fn): [first block of the layer .. next bucket)
struct Bucket { int64_t begin, end; };

static int net_backward(const Ctx& c, const float* dy, const float* dlow_nhwc, ddn_grad_bucket_fn on_bucket, void* user) {
  const NetSpec& s = *c.s; const Plan& p = *c.p;
  const int B = p.B, h8 = p.H / 8, w8 = p.W / 8;
  const bool want_lo = p.precision == DDN_PRECISION_BF16X3;
  float* S[4] = {c.f(p.scratch[0]), c.f(p.scratch[1]), c.f(p.scratch[2]), c.f(p.scratch[3])};
  DDN_CUDA(cudaMemsetAsync(c.ws + p.acc, 0, bn_accum_bytes(512), c.st));
  if (p.tc) DDN_CUDA(cudaMemsetAsync(c.f(p.dwp_all), 0, sizeof(float) * (size_t)(s.n_params + 64 * 192), c.st));
  const BlockBufs& last = p.blk.back();
  // d(low) = upsample^T(dy) [+ the gradient the fused loss scattered straight into the low-resolution map]
  if (dy) DDN_TRY(launch_upsample_bwd(dy, c.f(p.dlow), B * p.D, h8, w8, p.H, p.W, c.st));
  if (dlow_nhwc) DDN_TRY(launch_add_lowres_nhwc(dlow_nhwc, c.f(p.dlow), (int64_t)h8 * w8, B, p.D, dy ? 1 : 0, c.st));
  int cur = 0;   // index of the scratch buffer holding d(block output)
  DDN_TRY(launch_fc_backward(c.f(p.dlow), p.tc ? nullptr : c.f(last.out), p.tc ? c.h(last.out_p.hi) : nullptr,
                             (p.tc && want_lo) ? c.h(last.out_p.lo) : nullptr, c.params + s.fc_w, S[cur], c.grads + s.fc_w,
                             c.grads + s.fc_b, (int64_t)h8 * w8, B, 512, p.D, c.st));
  std::vector<TcUnpackEntry> pending;      // tensor-core weight gradients waiting in dwp_all for the bucket's conversion
  auto defer = [&](const ConvSpec& cs, int Hin, int Win) {
    if (!conv_on_tc(c, cs, Hin, Win)) return;
    TcUnpackEntry e; e.src_off = cs.w_off; e.dst_off = cs.w_off; e.Cout = cs.cout; e.Cin = cs.cin; e.taps = cs.k * cs.k; e.kind = 0;
    pending.push_back(e);
  };
  int64_t bucket_end = s.n_params;
  int bucket_id = 0;
  auto close_bucket = [&](int64_t begin) -> int {
    if (!pending.empty()) DDN_TRY(tc_unpack_wgrads(pending.data(), (int)pending.size(), c.f(p.dwp_all), c.grads, c.st));
    pending.clear();
    if (on_bucket) on_bucket(user, bucket_id, begin, bucket_end - begin);
    ++bucket_id; bucket_end = begin;
    return 0;
  };
  bool b2_fused = false;    // the column sums of this block's bn2 came out of the next block's conv1 data gradient (slot 2)
  for (int i = (int)s.blocks.size() - 1; i >= 0; --i) {
    const BlockSpec& b = s.blocks[i]; const BlockBufs& bb = p.blk[i];
    const float* xin = p.tc ? nullptr : (i == 0 ? c.f(p.pool_out) : c.f(p.blk[i - 1].out));
    const PlaneBufs xin_p = i == 0 ? p.pool_p : p.blk[i - 1].out_p;
    int64_t M1 = (int64_t)B * bb.c1.Hout * bb.c1.Wout;
    int t1 = (cur + 1) & 3, t2 = (cur + 2) & 3, t3 = (cur + 3) & 3;
    // out = relu(bn2(raw2) + residual):  g = dOut*(out>0) -> S[t2];  d raw2 -> planes (tensor core) or S[t1] (fp32)
    DDN_TRY(bn_backward_for(c, b.b2, bb.c2, S[cur], p.tc ? nullptr : c.f(bb.out), p.tc ? c.h(bb.out_p.hi) : nullptr, 1, S[t2], b.c2,
                            bb.c2.Hin, bb.c2.Win, S[t1], M1, b2_fused ? 2 : 0));
    // conv2: dW, d act1 -> S[t3] (+ the column sums of bn1's backward, in the same epilogue)
    TcBwdStats st1, st2;
    const bool b1_fused = conv_on_tc(c, b.c2, bb.c2.Hin, bb.c2.Win) && bwd_stats_for(c, b.b1, bb.c1, nullptr, 1, &st1);
    DDN_TRY(conv_backward(c, b.c2, p.tc ? nullptr : c.f(bb.act1), bb.act1_p, S[t1], S[t3], nullptr, B, bb.c2.Hin, bb.c2.Win, bb.c2.Hout,
                          bb.c2.Wout, b.c2.cin, b1_fused ? &st1 : nullptr));
    defer(b.c2, bb.c2.Hin, bb.c2.Win);
    // conv1's data gradient completes d(block input) = dOut of the previous block: bn2 of that block gets its column sums there
    b2_fused = i > 0 && conv_on_tc(c, b.c1, bb.c1.Hin, bb.c1.Win) &&
               bwd_stats_for(c, s.blocks[i - 1].b2, p.blk[i - 1].c2, c.h(p.blk[i - 1].out_p.hi), 2, &st2);
    // act1 = relu(bn1(raw1)), no residual: the mask is recomputed from raw1 in the tensor-core modes
    if (!b.has_ds) {
      DDN_TRY(bn_backward_for(c, b.b1, bb.c1, S[t3], p.tc ? nullptr : c.f(bb.act1), nullptr, 1, nullptr, b.c1, bb.c1.Hin, bb.c1.Win, S[t1], M1,
                              b1_fused ? 1 : 0));
      // dX = dgrad(conv1) + g
      DDN_TRY(conv_backward(c, b.c1, xin, xin_p, S[t1], S[t3], S[t2], B, bb.c1.Hin, bb.c1.Win, bb.c1.Hout, bb.c1.Wout, b.c1.cin,
                            b2_fused ? &st2 : nullptr));
      defer(b.c1, bb.c1.Hin, bb.c1.Win);
      cur = t3;
    } else {
      // residual branch first (its dY planes are consumed before conv1's overwrite them):
      // bn_d(raw_d): d raw_d; ds conv: dW, dX_ds -> S[cur]
      DDN_TRY(bn_backward_for(c, b.bd, bb.ds, S[t2], nullptr, nullptr, 0, nullptr, b.ds, bb.ds.Hin, bb.ds.Win, S[t1], M1));
      DDN_TRY(conv_backward(c, b.ds, xin, xin_p, S[t1], S[cur], nullptr, B, bb.ds.Hin, bb.ds.Win, bb.ds.Hout, bb.ds.Wout, b.ds.cin));
      defer(b.ds, bb.ds.Hin, bb.ds.Win);
      // main branch: d raw1, then dX = dgrad(conv1) + dX_ds -> S[t2]
      DDN_TRY(bn_backward_for(c, b.b1, bb.c1, S[t3], p.tc ? nullptr : c.f(bb.act1), nullptr, 1, nullptr, b.c1, bb.c1.Hin, bb.c1.Win, S[t1], M1,
                              b1_fused ? 1 : 0));
      DDN_TRY(conv_backward(c, b.c1, xin, xin_p, S[t1], S[t2], S[cur], B, bb.c1.Hin, bb.c1.Win, bb.c1.Hout, bb.c1.Wout, b.c1.cin,
                            b2_fused ? &st2 : nullptr));
      defer(b.c1, bb.c1.Hin, bb.c1.Win);
      cur = t2;
      // a block with a downsample branch opens a residual layer: everything from its first parameter up is final now
      DDN_TRY(close_bucket(b.c1.w_off));     // layer4 (+fc), layer3, layer2; layer1 + stem close at the end
    }
  }
  // stem: maxpool -> relu -> bn1 -> conv1 (weight gradient only; the image is not differentiated)
  int t1 = (cur + 1) & 3, t2 = (cur + 2) & 3;
  DDN_TRY(launch_stem_pool_relu_backward(S[cur], reinterpret_cast<const uint8_t*>(c.ws + p.argmax), c.f(p.stem_raw),
                                         c.mean(p.stem_stats), c.invstd(p.stem_stats, 64), c.params + s.stem_bn.g_off,
                                         c.params + s.stem_bn.b_off, S[t1], B, p.H1, p.W1, 64, c.G, c.st));
  BnBwdArgs ks;
  memset(&ks, 0, sizeof(ks));
  ks.dy = S[t1]; ks.x = c.f(p.stem_raw); ks.mean = c.mean(p.stem_stats); ks.invstd = c.invstd(p.stem_stats, 64);
  ks.gamma = c.params + s.stem_bn.g_off; ks.beta = c.params + s.stem_bn.b_off;
  ks.dgamma = c.grads + s.stem_bn.g_off; ks.dbeta = c.grads + s.stem_bn.b_off;
  ks.acc = c.accum(); ks.sums = c.f(p.sums);
  ks.M = (int64_t)B * p.H1 * p.W1; ks.C = 64; ks.relu = 0; ks.training = c.training() ? 1 : 0; ks.G = c.G;
  if (p.tc) {
    ks.dx_hi = c.h(p.grad_p.hi); ks.dx_lo = want_lo ? c.h(p.grad_p.lo) : nullptr;
    DDN_TRY(launch_bn_backward(ks, c.st));
    DDN_TRY(tc_stem_wgrad(c.planes(p.patch_p), c.planes(p.grad_p), nullptr, B, p.H1, p.W1, p.precision, c.f(p.dwp_all) + s.n_params, c.st));
    TcUnpackEntry e; e.src_off = s.n_params; e.dst_off = s.stem.w_off; e.Cout = 64; e.Cin = 3; e.taps = 49; e.kind = 1;
    pending.push_back(e);
  } else {
    ks.dx = S[t2];
    DDN_TRY(launch_bn_backward(ks, c.st));
    DDN_TRY(conv_backward(c, s.stem, c.f(p.x4), PlaneBufs{0, 0}, S[t2], nullptr, nullptr, B, p.H, p.W, p.H1, p.W1, 4));
  }
  return close_bucket(0);
}

}  // namespace ddn

using namespace ddn;

extern "C" int ddn_abi_version(void) { return DDN_ABI_VERSION; }
extern "C" const char* ddn_last_error(void) { return g_err; }
extern "C" int64_t ddn_kernel_launch_count(void) { return g_launches.load(); }

extern "C" int ddn_profile_enable(int on) { g_prof_on.store(on ? 1 : 0); return 0; }
extern "C" int ddn_profile_reset(void) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_used = 0;
  return 0;
}
extern "C" int ddn_profile_read(ddn_profile_entry* out, int cap) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  double ms[PROF_NUM_CLASSES] = {0}, work[PROF_NUM_CLASSES] = {0};
  int64_t n[PROF_NUM_CLASSES] = {0};
  for (size_t i = 0; i < g_prof_used; ++i) {
    float t = 0.f;
    if (cudaEventSynchronize(g_prof[i].b) != cudaSuccess || cudaEventElapsedTime(&t, g_prof[i].a, g_prof[i].b) != cudaSuccess) continue;
    ms[g_prof[i].cls] += t; work[g_prof[i].cls] += g_prof[i].work; n[g_prof[i].cls]++;
  }
  int k = 0;
  for (int c = 0; c < PROF_NUM_CLASSES; ++c) {
    if (!n[c]) continue;
    if (out && k < cap) {
      memset(&out[k], 0, sizeof(out[k]));
      snprintf(out[k].name, sizeof(out[k].name), "%s", kProfNames[c]);
      out[k].launches = n[c]; out[k].ms = ms[c]; out[k].work = work[c];
    }
    ++k;
  }
  return k;
}

extern "C" int ddn_resnet34_8s_param_table(int D, ddn_tensor_entry* out, int cap) {
  if (D < 1 || D > 32) return DDN_EINVAL;
  const NetSpec& s = get_spec(D);
  for (int i = 0; i < (int)s.ptab.size() && i < cap && out; ++i) out[i] = s.ptab[i];
  return (int)s.ptab.size();
}
extern "C" int ddn_resnet34_8s_buffer_table(ddn_tensor_entry* out, int cap) {
  const NetSpec& s = get_spec(3);
  for (int i = 0; i < (int)s.btab.size() && i < cap && out; ++i) out[i] = s.btab[i];
  return (int)s.btab.size();
}
extern "C" int64_t ddn_resnet34_8s_param_count(int D) { return (D < 1 || D > 32) ? DDN_EINVAL : get_spec(D).n_params; }
extern "C" int64_t ddn_resnet34_8s_buffer_count(void) { return get_spec(3).n_buffers; }

extern "C" size_t ddn_resnet34_8s_weight_cache_bytes(int D) {
  if (D < 1 || D > 32) return 0;
  return (size_t)get_spec(D).n_params * 2 * 2 * sizeof(__nv_bfloat16) + 4096;
}

extern "C" int ddn_resnet34_8s_set_weight_cache(void* cache, size_t bytes, const float* params, uint64_t version, int precision) {
  std::lock_guard<std::mutex> lk(g_wcache_mu);
  WeightCache* wc = nullptr;
  for (auto& w : g_wcaches) if (w.params == params) wc = &w;
  if (!wc) {
    if (!cache) return 0;
    for (auto& w : g_wcaches) if (!w.base) wc = &w;          // reuse a retired slot
    if (!wc) {
      if (g_wcaches.size() >= 64) g_wcaches.erase(g_wcaches.begin());
      g_wcaches.emplace_back();
      wc = &g_wcaches.back();
    }
    wc->params = params; wc->base = nullptr;
  }
  const bool same = wc->base == (char*)cache && wc->bytes == bytes && wc->version == version && wc->precision == precision;
  if (!same) {
    wc->base = (char*)cache; wc->bytes = bytes; wc->version = version; wc->precision = precision;
    wc->fresh = true;           // first use re-packs unconditionally and (re)initialises the device-side fingerprints
  }
  if (!cache) wc->params = nullptr;
  return 0;
}

extern "C" size_t ddn_resnet34_8s_workspace_bytes(int B, int H, int W, int D, int mode, int precision) {
  Plan p;
  if (make_plan(&p, B, H, W, D, mode, precision) != 0) return 0;
  return p.total;
}

static int check_ws(const Plan& p, void* ws, size_t bytes) {
  DDN_CHECK_ARG(ws && (reinterpret_cast<uintptr_t>(ws) & 255) == 0, "workspace must be non-null and 256-byte aligned");
  if (bytes < p.total) { set_error("workspace too small: %zu < %zu", bytes, p.total); return DDN_EWORKSPACE; }
  return 0;
}
static int check_groups(int B, int G) {
  DDN_CHECK_ARG(G >= 1 && G <= BN_MAX_GROUPS && B % G == 0, "bn_groups must be 1 or %d and divide the batch (got %d for B=%d)", BN_MAX_GROUPS, G, B);
  return 0;
}

extern "C" int ddn_resnet34_8s_forward(const float* x, const float* params, float* buffers, float* y,
                                       void* workspace, size_t workspace_bytes, int B, int H, int W, int D,
                                       int mode, int bn_groups, float momentum, float eps, int precision, float* low_nhwc_out,
                                       void* stream) {
  DDN_CHECK_ARG(x && params && buffers && y, "null tensor");
  DDN_TRY(check_groups(B, bn_groups));
  Plan p;
  DDN_TRY(make_plan(&p, B, H, W, D, mode, precision));
  DDN_TRY(check_ws(p, workspace, workspace_bytes));
  Ctx c = {&get_spec(D), &p, (char*)workspace, params, buffers, nullptr, (cudaStream_t)stream, momentum, eps, mode, bn_groups};
  return net_forward(c, x, y, low_nhwc_out);
}

extern "C" int ddn_resnet34_8s_backward(const float* dy, const float* dlow_nhwc, const float* params, float* grads,
                                        void* workspace, size_t workspace_bytes, int B, int H, int W, int D,
                                        int mode, int bn_groups, float eps, int precision,
                                        ddn_grad_bucket_fn on_bucket, void* user, void* stream) {
  DDN_CHECK_ARG((dy || dlow_nhwc) && params && grads, "null tensor");
  DDN_CHECK_ARG(mode == DDN_MODE_TRAIN || mode == DDN_MODE_EVAL_SAVE, "backward needs a forward that kept its activations (mode %d)", mode);
  DDN_TRY(check_groups(B, bn_groups));
  Plan p;
  DDN_TRY(make_plan(&p, B, H, W, D, mode, precision));
  DDN_TRY(check_ws(p, workspace, workspace_bytes));
  Ctx c = {&get_spec(D), &p, (char*)workspace, params, nullptr, grads, (cudaStream_t)stream, 0.f, eps, mode, bn_groups};
  return net_backward(c, dy, dlow_nhwc, on_bucket, user);
}

extern "C" int ddn_resnet34_8s_grad_buckets(int D, int64_t* offsets, int cap) {
  if (D < 1 || D > 32) return DDN_EINVAL;
  const NetSpec& s = get_spec(D);
  const int64_t b[5] = {s.blocks[13].c1.w_off, s.blocks[7].c1.w_off, s.blocks[3].c1.w_off, 0, s.n_params};
  for (int i = 0; i < 5 && i < cap && offsets; ++i) offsets[i] = b[i];
  return 4;
}

// ------------------------------------------------------------------------------------------------ single operators
static int conv_out(int in, int k, int stride, int pad, int dil) { return (in + 2 * pad - dil * (k - 1) - 1) / stride + 1; }

extern "C" size_t ddn_conv2d_workspace_bytes(int N, int H, int W, int Cin, int Cout, int k, int stride, int pad, int dil, int precision) {
  size_t wb = align_up(sizeof(float) * (size_t)k * k * Cin * Cout, 256);
  size_t tc = precision == DDN_PRECISION_FP32_SIMT ? 0 : tc_workspace_bytes((size_t)N * H * W * (Cin > Cout ? Cin : Cout));
  return 3 * wb + align_up(tc, 256) + 256;
}

extern "C" int ddn_conv2d_forward(const float* x, const float* w, float* y, int N, int H, int W, int Cin, int Cout,
                                  int k, int stride, int pad, int dil, int precision, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  DDN_CHECK_ARG(x && w && y && workspace, "null tensor");
  DDN_CHECK_ARG(workspace_bytes >= ddn_conv2d_workspace_bytes(N, H, W, Cin, Cout, k, stride, pad, dil, precision), "workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  size_t wb = align_up(sizeof(float) * (size_t)k * k * Cin * Cout, 256);
  int Ho = conv_out(H, k, stride, pad, dil), Wo = conv_out(W, k, stride, pad, dil);
  if (precision != DDN_PRECISION_FP32_SIMT) {
    DDN_CHECK_ARG(tc_conv_supported(Cin, Cout, k, stride, pad, dil, H, W), "shape not supported by the tcgen05 path");
    return tc_conv_forward(x, w, y, N, H, W, Cin, Cout, k, stride, pad, dil, precision, (char*)workspace + 3 * wb,
                           workspace_bytes - 3 * wb, st);
  }
  ConvGeom g;
  DDN_TRY(conv_geom_init(&g, N, H, W, Cin, Ho, Wo, Cout, k, k, stride, 1, pad, dil));
  float* wp = (float*)workspace;
  DDN_TRY(launch_pack_weights(w, wp, Cout, Cin, Cin, k, k, 0, st));
  return launch_conv_gather_f32(x, wp, nullptr, y, g, st);
}

extern "C" int ddn_conv2d_backward(const float* x, const float* w, const float* dy, float* dx, float* dw,
                                   int N, int H, int W, int Cin, int Cout, int k, int stride, int pad, int dil,
                                   int precision, void* workspace, size_t workspace_bytes, void* stream) {
  DDN_CHECK_ARG(x && w && dy && dw && workspace, "null tensor");
  DDN_CHECK_ARG(workspace_bytes >= ddn_conv2d_workspace_bytes(N, H, W, Cin, Cout, k, stride, pad, dil, precision), "workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  size_t wb = align_up(sizeof(float) * (size_t)k * k * Cin * Cout, 256);
  int Ho = conv_out(H, k, stride, pad, dil), Wo = conv_out(W, k, stride, pad, dil);
  float* wp = (float*)workspace; float* dwp = (float*)((char*)workspace + wb);
  if (precision != DDN_PRECISION_FP32_SIMT) {
    DDN_CHECK_ARG(tc_conv_supported(Cin, Cout, k, stride, pad, dil, H, W), "shape not supported by the tcgen05 path");
    return tc_conv_backward(x, w, dy, dx, nullptr, dw, N, H, W, Cin, Cout, k, stride, pad, dil, precision,
                            (char*)workspace + 3 * wb, workspace_bytes - 3 * wb, dwp, st);
  }
  ConvGeom g;
  DDN_TRY(conv_geom_init(&g, N, H, W, Cin, Ho, Wo, Cout, k, k, stride, 1, pad, dil));
  DDN_TRY(launch_fill_zero(dwp, sizeof(float) * (size_t)k * k * Cin * Cout, st));
  DDN_TRY(launch_conv_wgrad_f32(x, dy, dwp, g, st));
  DDN_TRY(launch_unpack_wgrad(dwp, dw, Cout, Cin, Cin, k, k, st));
  if (dx) {
    ConvGeom gd;
    DDN_TRY(conv_geom_init(&gd, N, Ho, Wo, Cout, H, W, Cin, k, k, 1, stride, dil * (k - 1) - pad, dil));
    DDN_TRY(launch_pack_weights(w, wp, Cout, Cin, Cin, k, k, 1, st));
    DDN_TRY(launch_conv_gather_f32(dy, wp, nullptr, dx, gd, st));
  }
  return 0;
}

extern "C" size_t ddn_batchnorm_workspace_bytes(int64_t M, int C) {
  (void)M;
  if (C < 4 || C % 4 || 256 % (C / 4)) return 0;
  return bn_accum_bytes(C) + sizeof(float) * 2 * BN_MAX_GROUPS * C + 256;
}

extern "C" int ddn_batchnorm_forward(const float* x, const float* gamma, const float* beta, const float* residual,
                                     float* y, float* save_mean, float* save_invstd, float* running_mean, float* running_var,
                                     int64_t M, int C, int relu, int training, float momentum, float eps,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  DDN_CHECK_ARG(x && gamma && beta && y && save_mean && save_invstd && workspace, "null tensor");
  DDN_CHECK_ARG(workspace_bytes >= ddn_batchnorm_workspace_bytes(M, C) && ddn_batchnorm_workspace_bytes(M, C) > 0, "bad C or workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  if (training) {
    DDN_CUDA(cudaMemsetAsync(workspace, 0, bn_accum_bytes(C), st));
    DDN_TRY(launch_bn_stats(x, M, C, 1, bn_accum_at(workspace, C), save_mean, save_invstd, running_mean, running_var, momentum, eps, st));
  } else {
    DDN_CHECK_ARG(running_mean && running_var, "eval mode needs running statistics");
    DDN_TRY(launch_bn_eval_stats(running_mean, running_var, C, 1, eps, save_mean, save_invstd, st));
  }
  BnApplyArgs a;
  memset(&a, 0, sizeof(a));
  a.x = x; a.mean = save_mean; a.invstd = save_invstd; a.gamma = gamma; a.beta = beta; a.r = residual; a.y = y;
  a.M = M; a.C = C; a.relu = relu; a.G = 1;
  return launch_bn_apply(a, st);
}

extern "C" int ddn_batchnorm_backward(const float* dy, const float* x, const float* y, const float* gamma,
                                      const float* save_mean, const float* save_invstd, float* dx, float* dgamma, float* dbeta,
                                      float* d_residual, int64_t M, int C, int relu, void* workspace, size_t workspace_bytes, void* stream) {
  DDN_CHECK_ARG(dy && x && gamma && save_mean && save_invstd && dx && dgamma && dbeta && workspace, "null tensor");
  DDN_CHECK_ARG(!relu || y, "relu backward needs the forward output");
  DDN_CHECK_ARG(workspace_bytes >= ddn_batchnorm_workspace_bytes(M, C) && ddn_batchnorm_workspace_bytes(M, C) > 0, "bad C or workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  DDN_CUDA(cudaMemsetAsync(workspace, 0, bn_accum_bytes(C), st));
  BnBwdArgs a;
  memset(&a, 0, sizeof(a));
  a.dy = dy; a.x = x; a.mean = save_mean; a.invstd = save_invstd; a.gamma = gamma; a.y = y;
  a.dx = dx; a.g_out = d_residual; a.dgamma = dgamma; a.dbeta = dbeta;
  a.acc = bn_accum_at(workspace, C); a.sums = reinterpret_cast<float*>((char*)workspace + bn_accum_bytes(C));
  a.M = M; a.C = C; a.relu = relu; a.training = 1; a.G = 1;
  return launch_bn_backward(a, st);
}
