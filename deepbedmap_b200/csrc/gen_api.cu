// Model-level C entry points of the generator (SURVEY 8b): a host in any language runs
// GeneratorModel.forward (srgan_train.py:525-576) with
//   dbm_gen_create -> dbm_gen_set_param (x every array of the Chainer .npz, App. C keys) -> dbm_gen_workspace_bytes ->
//   dbm_gen_forward
// and nothing of the Python shim. The handle owns the fp32 master weights (or views a caller-owned flat buffer,
// dbm_gen_bind_params), their re-packed bf16 UMMA operand images and the pass table of the persistent trunk kernel;
// activations live in the caller's workspace; all work is enqueued on the caller's stream. The forward is the
// tensor-core inference path (bf16 operands, fp32 accumulation, fp32 residual stream): the same kernels, in the same
// order, with the same tables as deepbedmap_b200/model.py builds for its tiled path -- which now calls this file.
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "umma_common.cuh"

namespace dbm {

struct GenParam {
  std::string key;
  int ndim;
  int dims[4];
  long off, n;
};

// The packed operand images of one precision in one device arena, and the table dbm_pack_conv3x3_table executes to
// (re)build them from the master weights
struct PackArena {
  uint8_t* base = nullptr;
  PackEntry* dev = nullptr;   // pack table
  int n = 0;                  // its entries
  long max = 0;               // elements of the largest image
  bool stale = true;          // the master weights changed since the last pack
  std::map<std::string, size_t> img;   // image offsets by name
  const __nv_bfloat16* image(const std::string& name) const { return (const __nv_bfloat16*)(base + img.at(name)); }
};

struct Gen {
  int nb = 12, inter = 32;
  float beta = 0.1f;
  int dev = 0;
  std::vector<GenParam> params;
  std::map<std::string, int> index;
  long total = 0;
  float* flat = nullptr;     // device fp32 master weights, App. C order
  bool owns_flat = false;
  // re-packed bf16 operands, and offsets of the stem / head regions of that arena
  PackArena pack;
  size_t off_wts = 0, off_bias128 = 0, off_w1tc = 0, off_bias_off1 = 0, off_bias_off2 = 0;
  // precision: 0 = bf16 tensor-core path, 1 = "bf16x3" (split-bf16 trunk + upsample convs, fp32 stem and deformable
  // layers; dbm_gen_set_precision). The split operand images live in their own arena, built on first use.
  int precision = 0;
  PackArena pack_s;
  // pass-table cache: rebuilt when the workspace or the shape changes
  const void* tab_ws = nullptr;
  int tab_n = 0, tab_h = 0, tab_w = 0, tab_layers = 0, tab_precision = -1;
  bool tab_paired = false;
  std::vector<TrunkLayer> tab_host;
};

static const float* P(const Gen* g, const std::string& key) {
  auto it = g->index.find(key);
  return it == g->index.end() ? nullptr : g->flat + g->params[it->second].off;
}

static void add_param(Gen* g, const std::string& key, int d0, int d1 = 0, int d2 = 0, int d3 = 0) {
  GenParam p;
  p.key = key;
  p.dims[0] = d0; p.dims[1] = d1; p.dims[2] = d2; p.dims[3] = d3;
  p.ndim = d1 == 0 ? 1 : 4;
  p.n = p.ndim == 1 ? d0 : (long)d0 * d1 * d2 * d3;
  p.off = g->total;
  g->total += p.n;
  g->index[key] = (int)g->params.size();
  g->params.push_back(p);
}

// Parameter inventory in the reference's Chainer .npz order (srgan_train.py:218-523; SURVEY App. C;
// deepbedmap_b200/layout.py generator_shapes)
static void build_inventory(Gen* g) {
  const int ic = g->inter;
  const char* stem[4] = {"X", "W1", "W2", "W3"};
  const int sc[4] = {1, 1, 2, 1}, sk[4] = {3, 30, 6, 3};
  for (int i = 0; i < 4; ++i) {
    add_param(g, std::string("input_block/conv_on_") + stem[i] + "/W", 32, sc[i], sk[i], sk[i]);
    add_param(g, std::string("input_block/conv_on_") + stem[i] + "/b", 32);
  }
  add_param(g, "pre_residual_conv_layer/W", 64, 128, 3, 3);
  add_param(g, "pre_residual_conv_layer/b", 64);
  for (int i = 0; i < g->nb; ++i)
    for (int r = 1; r <= 3; ++r) {
      const std::string pre = "residual_network/" + std::to_string(i) + "/residual_dense_block" + std::to_string(r);
      for (int k = 1; k <= 4; ++k) {
        add_param(g, pre + "/conv_layer" + std::to_string(k) + "/W", ic, 64 + (k - 1) * ic, 3, 3);
        add_param(g, pre + "/conv_layer" + std::to_string(k) + "/b", ic);
      }
      add_param(g, pre + "/conv_layer5/W", 64, 64 + 4 * ic, 3, 3);
      add_param(g, pre + "/conv_layer5/b", 64);
    }
  const char* plain[3] = {"post_residual_conv_layer", "post_upsample_conv_layer_1", "post_upsample_conv_layer_2"};
  for (int i = 0; i < 3; ++i) {
    add_param(g, std::string(plain[i]) + "/W", 64, 64, 3, 3);
    add_param(g, std::string(plain[i]) + "/b", 64);
  }
  const char* fin[2] = {"final_conv_layer1", "final_conv_layer2"};
  const int oc[2] = {64, 1};
  for (int i = 0; i < 2; ++i) {
    add_param(g, std::string(fin[i]) + "/offset_conv/W", 18, 64, 3, 3);
    add_param(g, std::string(fin[i]) + "/offset_conv/b", 18);
    add_param(g, std::string(fin[i]) + "/deform_conv/W", oc[i], 64, 3, 3);
    add_param(g, std::string(fin[i]) + "/deform_conv/b", oc[i]);
  }
}

static std::string rdb_prefix(int i, int r) {
  return "residual_network/" + std::to_string(i) + "/residual_dense_block" + std::to_string(r);
}

// Lays packed operand images out in an arena and collects the entries of its pack table. elem: bf16 elements of an
// image per filter element (1, or 3 for split-bf16's [w_hi | w_hi | w_lo]); mode: the pack mode of every entry.
struct PackPlan {
  const Gen* g;
  PackArena& a;
  int elem, mode;
  std::vector<PackEntry> ent;
  size_t off = 0;
  size_t raw(size_t bytes) {
    const size_t o = off;
    off += (bytes + 255) & ~(size_t)255;
    return o;
  }
  size_t image(const std::string& name, int cin, int coutp) {
    return a.img[name] = raw((size_t)elem * 9 * cin * coutp * 2);
  }
  void entry(const std::string& wkey, size_t img_off, int O, int o0, int cin, int cin_total, int c0, int coutp, int ck) {
    PackEntry e;
    e.w = P(g, wkey);
    e.out = (__nv_bfloat16*)img_off;   // arena-relative until upload()
    e.O = O; e.o0 = o0; e.Cin = cin; e.CinTotal = cin_total; e.c0 = c0; e.COUTP = coutp; e.CK = ck; e.mode = mode;
    ent.push_back(e);
  }
};

// The trunk's filters in 16-channel chunks: pre-residual conv; per dense block conv1..4 (plain_dense), conv5 and, for
// inter_channels 32, the pair / tail images of dense-block pairing (layout.trunk_plan); post-residual conv
static void trunk_pack_entries(PackPlan& p, bool plain_dense) {
  const int ic = p.g->inter, cc = 64 + 4 * ic;
  p.entry("pre_residual_conv_layer/W", p.image("pre", 128, 64), 64, 0, 128, 128, 0, 64, 16);
  for (int i = 0; i < p.g->nb; ++i)
    for (int r = 1; r <= 3; ++r) {
      const std::string pre = rdb_prefix(i, r);
      for (int k = 1; plain_dense && k <= 4; ++k) {
        const int cin = 64 + (k - 1) * ic;
        p.entry(pre + "/conv_layer" + std::to_string(k) + "/W", p.image(pre + "/c" + std::to_string(k), cin, ic), ic, 0,
                cin, cin, 0, ic, 16);
      }
      p.entry(pre + "/conv_layer5/W", p.image(pre + "/c5", cc, 64), 64, 0, cc, cc, 0, 64, 16);
      if (ic == 32)
        for (int k = 1; k <= 3; k += 2) {   // head = conv_k | conv_{k+1} over their shared inputs, tail = conv_{k+1} over a_k
          const int cin = 64 + (k - 1) * 32;
          const std::string wa = pre + "/conv_layer" + std::to_string(k) + "/W";
          const std::string wb = pre + "/conv_layer" + std::to_string(k + 1) + "/W";
          const size_t both = p.image(pre + "/pair" + std::to_string(k), cin, 64);
          p.entry(wa, both, 32, 0, cin, cin, 0, 64, 16);
          p.entry(wb, both, 32, 32, cin, cin + 32, 0, 64, 16);
          p.entry(wb, p.image(pre + "/tail" + std::to_string(k + 1), 32, 32), 32, 0, 32, cin + 32, cin, 32, 16);
        }
    }
  p.entry("post_residual_conv_layer/W", p.image("post", 64, 64), 64, 0, 64, 64, 0, 64, 16);
}

// Allocates the arena (zeroed: padded rows and biases stay zero), rebases the entries onto it and uploads the table
static int upload(PackPlan& p) {
  PackArena& a = p.a;
  DBM_CUDA(cudaMalloc(&a.base, p.off));
  DBM_CUDA(cudaMemset(a.base, 0, p.off));
  a.max = 0;
  for (auto& e : p.ent) {
    e.out = (__nv_bfloat16*)(a.base + (size_t)e.out);
    a.max = std::max(a.max, (long)9 * e.Cin * e.COUTP);
  }
  a.n = (int)p.ent.size();
  DBM_CUDA(cudaMalloc(&a.dev, p.ent.size() * sizeof(PackEntry)));
  DBM_CUDA(cudaMemcpy(a.dev, p.ent.data(), p.ent.size() * sizeof(PackEntry), cudaMemcpyHostToDevice));
  a.stale = true;
  return DBM_OK;
}

// Points the table's filter pointers at a new master-weight buffer
static int rebase_weights(PackArena& a, const float* from, const float* to) {
  if (!a.dev) return DBM_OK;
  std::vector<PackEntry> ent(a.n);
  DBM_CUDA(cudaMemcpy(ent.data(), a.dev, ent.size() * sizeof(PackEntry), cudaMemcpyDeviceToHost));
  for (auto& e : ent) e.w = to + (e.w - from);
  DBM_CUDA(cudaMemcpy(a.dev, ent.data(), ent.size() * sizeof(PackEntry), cudaMemcpyHostToDevice));
  return DBM_OK;
}

static int refresh(PackArena& a, cudaStream_t st) {
  if (!a.stale) return DBM_OK;
  const int rc = dbm_pack_conv3x3_table(a.dev, a.n, a.max, st);
  if (rc) return rc;
  a.stale = false;
  return DBM_OK;
}

static void free_arena(PackArena& a) {
  if (a.base) cudaFree(a.base);
  if (a.dev) cudaFree(a.dev);
}

// The bf16 arena: the trunk's images, the upsample / offset / first deformable convs, and the stem's and heads' operands
static int build_pack_plan(Gen* g) {
  PackPlan p{g, g->pack, 1, 0};
  trunk_pack_entries(p, true);
  p.entry("post_upsample_conv_layer_1/W", p.image("up1", 64, 64), 64, 0, 64, 64, 0, 64, 32);
  p.entry("post_upsample_conv_layer_2/W", p.image("up2", 64, 64), 64, 0, 64, 64, 0, 64, 32);
  p.entry("final_conv_layer1/offset_conv/W", p.image("off1", 64, 32), 18, 0, 64, 64, 0, 32, 32);
  p.entry("final_conv_layer2/offset_conv/W", p.image("off2", 64, 32), 18, 0, 64, 64, 0, 32, 32);
  p.entry("final_conv_layer1/deform_conv/W", p.image("dc1", 64, 64), 64, 0, 64, 64, 0, 64, 64);
  g->off_wts = p.raw(90 * 32 * 4);
  g->off_bias128 = p.raw(128 * 4);
  g->off_w1tc = p.raw((size_t)9 * 320 * 32 * 2);
  g->off_bias_off1 = p.raw(32 * 4);
  g->off_bias_off2 = p.raw(32 * 4);
  return upload(p);
}

static int refresh_packed(Gen* g, cudaStream_t st) {
  if (!g->pack.stale) return DBM_OK;
  uint8_t* arena = g->pack.base;
  float* wts = (float*)(arena + g->off_wts);
  float* bias128 = (float*)(arena + g->off_bias128);
  int rc;
  // conv_on_X (9 taps) | conv_on_W2 (72) | conv_on_W3 (9), tap-major [taps][32]
  if ((rc = dbm_transpose_f32(P(g, "input_block/conv_on_X/W"), wts, 32, 9, st))) return rc;
  if ((rc = dbm_transpose_f32(P(g, "input_block/conv_on_W2/W"), wts + 9 * 32, 32, 72, st))) return rc;
  if ((rc = dbm_transpose_f32(P(g, "input_block/conv_on_W3/W"), wts + 81 * 32, 32, 9, st))) return rc;
  const char* stem[4] = {"X", "W1", "W2", "W3"};
  for (int i = 0; i < 4; ++i)
    DBM_CUDA(cudaMemcpyAsync(bias128 + 32 * i, P(g, std::string("input_block/conv_on_") + stem[i] + "/b"), 32 * 4,
                             cudaMemcpyDeviceToDevice, st));
  DBM_CUDA(cudaMemcpyAsync(arena + g->off_bias_off1, P(g, "final_conv_layer1/offset_conv/b"), 18 * 4,
                           cudaMemcpyDeviceToDevice, st));
  DBM_CUDA(cudaMemcpyAsync(arena + g->off_bias_off2, P(g, "final_conv_layer2/offset_conv/b"), 18 * 4,
                           cudaMemcpyDeviceToDevice, st));
  if ((rc = dbm_pack_stem_w1(P(g, "input_block/conv_on_W1/W"), arena + g->off_w1tc, st))) return rc;
  return refresh(g->pack, st);   // the filter images, last: it clears the stale mark
}

// ---- workspace layout ------------------------------------------------------------------------------------------
struct WsLayout {
  size_t s2d, s0, cat[2], a1, f32[3], u1, u2, f1, offs, proj, flags, table, total;
  int num_layers, units;
  bool paired;
};

static WsLayout ws_layout(const Gen* g, int n, int h, int w) {
  WsLayout L;
  const size_t H = h - 2, W = w - 2;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += (bytes + 1023) & ~(size_t)1023;
    return o;
  };
  const size_t px = (size_t)n * H * W;
  const int ccs = (64 + 4 * g->inter) / 8;
  L.s2d = take((size_t)n * 40 * h * w * 16);
  L.s0 = take(px * 16 * 16);
  L.cat[0] = take(px * ccs * 16);
  L.cat[1] = take(px * ccs * 16);
  L.a1 = take(px * 64 * 4);
  for (int i = 0; i < 3; ++i) L.f32[i] = take(px * 64 * 4);
  L.u1 = take(px * 4 * 8 * 16);
  L.u2 = take(px * 16 * 8 * 16);     // also the first deformable layer's output (the upsample-conv input is dead by then)
  L.f1 = take(px * 16 * 8 * 16);
  L.offs = take(px * 16 * 8 * 16);   // offset fields, fp32 slab4 x 8 slabs (18 of 32 channels used)
  L.proj = take(px * 16 * 9 * 4);
  L.paired = g->inter == 32 && ((int)W + 15) / 16 + 2 <= 128;
  L.num_layers = 2 + g->nb * 3 * 5;
  L.units = n * (((int)H + 31) / 32) * (((int)W + 15) / 16);
  L.flags = take((size_t)L.num_layers * L.units * 4);
  L.table = take((size_t)L.num_layers * sizeof(TrunkLayer));
  L.total = off;
  return L;
}

static void add_pass(std::vector<TrunkLayer>& T, const __nv_bfloat16* wq, const float* bias, int cin, int cout, int in_map,
                     int act, float beta, __nv_bfloat16* out, int out_cs_total, int out_cs0, float* out_f32,
                     const float* res1, const float* res2, int up2, int in_cs0, int cout_main, int mode) {
  TrunkLayer t;
  memset(&t, 0, sizeof(t));
  t.wpacked = wq; t.bias = bias; t.out_bf16 = out; t.out_f32 = out_f32; t.res1 = res1; t.res2 = res2;
  t.stash_out = nullptr;
  t.cin = cin; t.cout = cout; t.in_map = in_map; t.in_cs0 = in_cs0; t.act = act; t.up2 = up2;
  t.out_cs_total = out_cs_total; t.out_cs0 = out_cs0; t.cout_main = cout_main; t.res1_cs_total = 16;
  t.beta = beta; t.mode = mode;
  T.push_back(t);
}

// Pass table of the trunk kernels with the filter images of arena a and the buffers of workspace layout L (WsLayout or
// WsSplit; cs fields are logical, the same for both): the C++ twin of layout.trunk_plan as model.py's
// _trunk_workspace / _split_workspace bind it
template <class Layout>
static void build_trunk_passes(const Gen* g, const PackArena& a, const Layout& L, uint8_t* ws, std::vector<TrunkLayer>& T) {
  T.clear();
  auto bf = [&](size_t o) { return (__nv_bfloat16*)(ws + o); };
  auto f32 = [&](size_t o) { return (float*)(ws + o); };
  const int ic = g->inter, cc = 64 + 4 * ic, ccs = cc / 8;
  __nv_bfloat16* cat[2] = {bf(L.cat[0]), bf(L.cat[1])};
  float* a1 = f32(L.a1);
  float* fb[3] = {f32(L.f32[0]), f32(L.f32[1]), f32(L.f32[2])};
  add_pass(T, a.image("pre"), P(g, "pre_residual_conv_layer/b"), 128, 64, 0, 1, 0.f, cat[0], ccs, 0, a1, nullptr,
           nullptr, 0, 0, 64, 0);
  int cur = 0, fi = 0;
  float* cur_f32 = a1;
  for (int i = 0; i < g->nb; ++i) {
    float* rrdb_in = cur_f32;
    for (int r = 1; r <= 3; ++r) {
      const std::string pre = rdb_prefix(i, r);
      auto bias = [&](int k) { return P(g, pre + "/conv_layer" + std::to_string(k) + "/b"); };
      if (L.paired) {
        for (int k = 1; k <= 3; k += 2) {
          const int cin = 64 + (k - 1) * ic;
          add_pass(T, a.image(pre + "/pair" + std::to_string(k)), bias(k), cin, 64, 1 + cur, 1, 0.f, cat[cur], ccs,
                   cin / 8, nullptr, nullptr, nullptr, 0, 0, 32, 1);
          add_pass(T, a.image(pre + "/tail" + std::to_string(k + 1)), bias(k + 1), 32, 32, 1 + cur, 1, 0.f, cat[cur],
                   ccs, cin / 8 + 4, nullptr, nullptr, nullptr, 0, cin / 8, 32, 2);
        }
      } else {
        for (int k = 1; k <= 4; ++k) {
          const int cin = 64 + (k - 1) * ic;
          add_pass(T, a.image(pre + "/c" + std::to_string(k)), bias(k), cin, ic, 1 + cur, 1, 0.f, cat[cur], ccs, cin / 8,
                   nullptr, nullptr, nullptr, 0, 0, ic, 0);
        }
      }
      while (fb[fi] == cur_f32 || fb[fi] == rrdb_in) fi = (fi + 1) % 3;
      float* nxt = fb[fi];
      add_pass(T, a.image(pre + "/c5"), bias(5), cc, 64, 1 + cur, 0, g->beta, cat[1 - cur], ccs, 0, nxt, cur_f32,
               r == 3 ? rrdb_in : nullptr, 0, 0, 64, 0);
      cur = 1 - cur;
      cur_f32 = nxt;
    }
  }
  add_pass(T, a.image("post"), P(g, "post_residual_conv_layer/b"), 64, 64, 1 + cur, 0, 1.f, bf(L.u1), 8, 0, nullptr, a1,
           nullptr, 1, 0, 64, 0);
}

// ---- precision "bf16x3": split-bf16 operand images, workspace and pass tables ---------------------------------------
// (the C++ twin of model.py's _pack("split") / _split_workspace / _forward_split)
static int build_split_pack_plan(Gen* g) {
  if (g->pack_s.base) return DBM_OK;
  PackPlan p{g, g->pack_s, 3, 16};
  trunk_pack_entries(p, g->inter != 32);   // inter_channels 32: the paired images only
  p.entry("post_upsample_conv_layer_1/W", p.image("up1", 64, 64), 64, 0, 64, 64, 0, 64, 16);
  p.entry("post_upsample_conv_layer_2/W", p.image("up2", 64, 64), 64, 0, 64, 64, 0, 64, 16);
  return upload(p);
}

struct WsSplit {
  size_t a0, s0, cat[2], a1, f32[3], u1, u2, c2f, c2, off, cols, d1, proj, flags[3], table[3], total;
  int num_layers, units[3];
  bool paired;
};

static WsSplit ws_layout_split(const Gen* g, int n, int h, int w) {
  WsSplit L;
  const size_t H = h - 2, W = w - 2;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += (bytes + 1023) & ~(size_t)1023;
    return o;
  };
  const size_t px = (size_t)n * H * W, px1 = 16 * H * W;   // trunk pixels of the batch; output pixels of ONE image
  const int ccs = (64 + 4 * g->inter) / 8;
  L.a0 = take(px * 128 * 4);
  L.s0 = take(px * 32 * 16);
  L.cat[0] = take(px * 2 * ccs * 16);
  L.cat[1] = take(px * 2 * ccs * 16);
  L.a1 = take(px * 64 * 4);
  for (int i = 0; i < 3; ++i) L.f32[i] = take(px * 64 * 4);
  L.u1 = take(px * 4 * 16 * 16);
  L.u2 = take(px * 16 * 16 * 16);
  L.c2f = take(px * 16 * 64 * 4);
  L.c2 = take(px1 * 64 * 4);          // the deformable layers run image by image (the fp32 sampler keeps 576 planes)
  L.off = take(px1 * 18 * 4);
  L.cols = take(px1 * 576 * 4);
  L.d1 = take(px1 * 64 * 4);
  L.proj = take(px1 * 9 * 4);
  L.paired = g->inter == 32 && ((int)W + 15) / 16 + 2 <= 128;
  L.num_layers = 2 + g->nb * 3 * 5;
  for (int i = 0; i < 3; ++i) {
    const int hh = (int)H << i, ww = (int)W << i;
    L.units[i] = n * ((hh + 31) / 32) * ((ww + 15) / 16);
  }
  L.flags[0] = take((size_t)L.num_layers * L.units[0] * 4);
  L.flags[1] = take((size_t)L.units[1] * 4);
  L.flags[2] = take((size_t)L.units[2] * 4);
  L.table[0] = take((size_t)L.num_layers * sizeof(TrunkLayer));
  L.table[1] = take(sizeof(TrunkLayer));
  L.table[2] = take(sizeof(TrunkLayer));
  L.total = off;
  return L;
}

// Pass tables of the split path: the trunk's (same passes as the bf16 table) followed by the two single-pass tables of
// the upsample convs
static int build_split_tables(Gen* g, const WsSplit& L, uint8_t* ws, std::vector<TrunkLayer>& T) {
  DBM_REQUIRE(L.paired || g->inter != 32, "gen_forward (bf16x3): tiles wider than ~2000 px are not supported");
  build_trunk_passes(g, g->pack_s, L, ws, T);
  // upsample convs: single-pass tables of the same kernel at 2x / 4x the resolution (input = "stem" map 0)
  add_pass(T, g->pack_s.image("up1"), P(g, "post_upsample_conv_layer_1/b"), 64, 64, 0, 1, 0.f,
           (__nv_bfloat16*)(ws + L.u2), 8, 0, nullptr, nullptr, nullptr, 1, 0, 64, 0);
  add_pass(T, g->pack_s.image("up2"), P(g, "post_upsample_conv_layer_2/b"), 64, 64, 0, 1, 0.f, nullptr, 0, 0,
           (float*)(ws + L.c2f), nullptr, nullptr, 0, 0, 64, 0);
  return DBM_OK;
}

static int gen_forward_split(Gen* g, const float* x, const float* w1, const float* w2, const float* w3, int n, int h_in,
                             int w_in, float* y_out, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  int rc = build_split_pack_plan(g);
  if (rc) return rc;
  const WsSplit L = ws_layout_split(g, n, h_in, w_in);
  DBM_REQUIRE(workspace_bytes >= L.total, "gen_forward: workspace of %zu bytes, need %zu (dbm_gen_workspace_bytes)",
              workspace_bytes, L.total);
  uint8_t* ws = (uint8_t*)workspace;
  const int H = h_in - 2, W = w_in - 2;
  if ((rc = refresh(g->pack_s, st))) return rc;
  if (g->tab_ws != workspace || g->tab_n != n || g->tab_h != h_in || g->tab_w != w_in || g->tab_precision != 1) {
    if ((rc = build_split_tables(g, L, ws, g->tab_host))) return rc;
    DBM_REQUIRE((int)g->tab_host.size() == L.num_layers + 2, "gen_forward: split pass tables have %zu entries, expected %d",
                g->tab_host.size(), L.num_layers + 2);
    const TrunkLayer* T = g->tab_host.data();
    DBM_CUDA(cudaMemcpyAsync(ws + L.table[0], T, (size_t)L.num_layers * sizeof(TrunkLayer), cudaMemcpyHostToDevice, st));
    DBM_CUDA(cudaMemcpyAsync(ws + L.table[1], T + L.num_layers, sizeof(TrunkLayer), cudaMemcpyHostToDevice, st));
    DBM_CUDA(cudaMemcpyAsync(ws + L.table[2], T + L.num_layers + 1, sizeof(TrunkLayer), cudaMemcpyHostToDevice, st));
    DBM_CUDA(cudaStreamSynchronize(st));
    g->tab_ws = workspace; g->tab_n = n; g->tab_h = h_in; g->tab_w = w_in; g->tab_precision = 1;
  }
  // ---- input block in fp32 (srgan_train.py:256-266), concatenated along channels ----
  float* a0 = (float*)(ws + L.a0);
  const long hw = (long)H * W, a0_bs = 128 * hw;
  struct Stem { const char* key; const float* in; int c, k, s; };
  const Stem stem[4] = {{"X", x, 1, 3, 1}, {"W1", w1, 1, 30, 10}, {"W2", w2, 2, 6, 2}, {"W3", w3, 1, 3, 1}};
  for (int i = 0; i < 4; ++i) {
    const std::string key = std::string("input_block/conv_on_") + stem[i].key;
    const int sc = stem[i].s;   // the input of stem i is sc times the size of x (s10 <- 10h, s2 <- 2h, s1 <- h)
    if ((rc = dbm_conv2d_fwd_f32(stem[i].in, (long)stem[i].c * (sc * h_in) * (sc * w_in), P(g, key + "/W"), P(g, key + "/b"),
                                 a0 + 32 * i * hw, a0_bs, n, stem[i].c, sc * h_in, sc * w_in, 32, stem[i].k, stem[i].s, 0,
                                 0, st)))
      return rc;
  }
  if ((rc = dbm_nchw_to_slab8_split(a0, 0, ws + L.s0, n, 128, H, W, st))) return rc;
  // ---- trunk and both upsample convs in split-bf16 ----
  const int ccs = (64 + 4 * g->inter) / 8;
  if ((rc = dbm_trunk_umma_split(ws + L.table[0], L.num_layers, n, H, W, ws + L.s0, 16, ws + L.cat[0], ws + L.cat[1], ccs,
                                 (unsigned int*)(ws + L.flags[0]), st)))
    return rc;
  if ((rc = dbm_trunk_umma_split(ws + L.table[1], 1, n, 2 * H, 2 * W, ws + L.u1, 8, ws + L.u1, ws + L.u1, 8,
                                 (unsigned int*)(ws + L.flags[1]), st)))
    return rc;
  if ((rc = dbm_trunk_umma_split(ws + L.table[2], 1, n, 4 * H, 4 * W, ws + L.u2, 8, ws + L.u2, ws + L.u2, 8,
                                 (unsigned int*)(ws + L.flags[2]), st)))
    return rc;
  // ---- deformable layers in fp32, image by image (srgan_train.py:572-574) ----
  const int Ho = 4 * H, Wo = 4 * W;
  const long hwo = (long)Ho * Wo;
  float* c2 = (float*)(ws + L.c2);
  float* off = (float*)(ws + L.off);
  float* cols = (float*)(ws + L.cols);
  float* d1 = (float*)(ws + L.d1);
  float* proj = (float*)(ws + L.proj);
  for (int i = 0; i < n; ++i) {
    if ((rc = dbm_slab8f_to_nchw((const float*)(ws + L.c2f) + (size_t)i * 64 * hwo, c2, 0, 1, 64, Ho, Wo, st))) return rc;
    if ((rc = dbm_conv2d_fwd_f32(c2, 64 * hwo, P(g, "final_conv_layer1/offset_conv/W"), P(g, "final_conv_layer1/offset_conv/b"),
                                 off, 18 * hwo, 1, 64, Ho, Wo, 18, 3, 1, 1, 0, st)))
      return rc;
    if ((rc = dbm_deform_sample_f32(c2, off, cols, 1, 64, Ho, Wo, st))) return rc;
    // d1[o, p] = lrelu(sum_k cols[k, p] w[o, k] + b[o])   (M = pixels, N = 64, K = 576)
    if ((rc = dbm_gemm_f32(cols, 1, hwo, 576 * hwo, P(g, "final_conv_layer1/deform_conv/W"), 1, 576, 0, d1, 1, hwo, 64 * hwo,
                           P(g, "final_conv_layer1/deform_conv/b"), (int)hwo, 64, 576, 1, 1, 0, st)))
      return rc;
    if ((rc = dbm_conv2d_fwd_f32(d1, 64 * hwo, P(g, "final_conv_layer2/offset_conv/W"), P(g, "final_conv_layer2/offset_conv/b"),
                                 off, 18 * hwo, 1, 64, Ho, Wo, 18, 3, 1, 1, 0, st)))
      return rc;
    if ((rc = dbm_deform1_fwd_f32(d1, off, P(g, "final_conv_layer2/deform_conv/W"), P(g, "final_conv_layer2/deform_conv/b"),
                                  y_out + (size_t)i * hwo, proj, 1, 64, Ho, Wo, st)))
      return rc;
  }
  return DBM_OK;
}

}  // namespace dbm

using namespace dbm;

struct dbm_gen {
  Gen g;
};

extern "C" int dbm_gen_create(int num_residual_blocks, float residual_scaling, int inter_channels, dbm_gen** out) {
  DBM_REQUIRE(out != nullptr, "gen_create: null output");
  DBM_REQUIRE(num_residual_blocks >= 1 && 2 + 15 * num_residual_blocks <= 512, "gen_create: %d residual blocks",
              num_residual_blocks);
  DBM_REQUIRE(inter_channels == 32 || inter_channels == 64, "gen_create: inter_channels must be 32 or 64 (the "
              "reference's search space, srgan_train.py:283-284); got %d", inter_channels);
  dbm_gen* h = new dbm_gen();
  Gen* g = &h->g;
  g->nb = num_residual_blocks; g->beta = residual_scaling; g->inter = inter_channels;
  cudaGetDevice(&g->dev);
  build_inventory(g);
  cudaError_t e = cudaMalloc(&g->flat, (size_t)g->total * 4);
  if (e != cudaSuccess) {
    delete h;
    set_error("gen_create: cudaMalloc of %ld parameters failed: %s", g->total, cudaGetErrorString(e));
    return DBM_ERR_CUDA;
  }
  cudaMemset(g->flat, 0, (size_t)g->total * 4);
  g->owns_flat = true;
  int rc = build_pack_plan(g);
  if (rc) {
    cudaFree(g->flat);
    delete h;
    return rc;
  }
  *out = h;
  return DBM_OK;
}

extern "C" int dbm_gen_destroy(dbm_gen* h) {
  if (!h) return DBM_OK;
  Gen* g = &h->g;
  if (g->owns_flat && g->flat) cudaFree(g->flat);
  free_arena(g->pack);
  free_arena(g->pack_s);
  delete h;
  return DBM_OK;
}

extern "C" long dbm_gen_count_params(const dbm_gen* h) { return h ? h->g.total : -1; }
extern "C" int dbm_gen_num_arrays(const dbm_gen* h) { return h ? (int)h->g.params.size() : -1; }

extern "C" int dbm_gen_array_info(const dbm_gen* h, int index, const char** key, int* ndim, int* dims4,
                                  long* flat_offset) {
  DBM_REQUIRE(h && index >= 0 && index < (int)h->g.params.size(), "gen_array_info: bad index %d", index);
  const GenParam& p = h->g.params[index];
  if (key) *key = p.key.c_str();
  if (ndim) *ndim = p.ndim;
  if (dims4)
    for (int i = 0; i < 4; ++i) dims4[i] = p.dims[i];
  if (flat_offset) *flat_offset = p.off;
  return DBM_OK;
}

extern "C" int dbm_gen_set_param(dbm_gen* h, const char* key, const float* host_values, int ndim, const int* dims) {
  DBM_REQUIRE(h && key && host_values && dims, "gen_set_param: null argument");
  Gen* g = &h->g;
  auto it = g->index.find(key);
  DBM_REQUIRE(it != g->index.end(), "gen_set_param: unknown key '%s'", key);
  const GenParam& p = g->params[it->second];
  bool ok = ndim == p.ndim;
  for (int i = 0; ok && i < ndim; ++i) ok = dims[i] == p.dims[i];
  DBM_REQUIRE(ok, "gen_set_param: '%s' has shape (%d,%d,%d,%d), got %d-d (%d,...)", key, p.dims[0], p.dims[1],
              p.dims[2], p.dims[3], ndim, ndim > 0 ? dims[0] : 0);
  DBM_CUDA(cudaMemcpy(g->flat + p.off, host_values, (size_t)p.n * 4, cudaMemcpyHostToDevice));
  g->pack.stale = g->pack_s.stale = true;
  return DBM_OK;
}

// View a caller-owned device buffer of dbm_gen_count_params floats (App. C order) as the master weights -- the Python
// shim shares its flat parameter buffer (the one Adam updates) this way. Call dbm_gen_mark_updated after changing it.
extern "C" int dbm_gen_bind_params(dbm_gen* h, float* device_flat) {
  DBM_REQUIRE(h && device_flat, "gen_bind_params: null argument");
  Gen* g = &h->g;
  DBM_REQUIRE(g->owns_flat, "gen_bind_params: parameters are already bound");
  cudaFree(g->flat);
  int rc;
  if ((rc = rebase_weights(g->pack, g->flat, device_flat)) || (rc = rebase_weights(g->pack_s, g->flat, device_flat)))
    return rc;
  g->flat = device_flat;
  g->owns_flat = false;
  g->pack.stale = g->pack_s.stale = true;
  g->tab_ws = nullptr;
  return DBM_OK;
}

extern "C" int dbm_gen_mark_updated(dbm_gen* h) {
  DBM_REQUIRE(h != nullptr, "gen_mark_updated: null handle");
  h->g.pack.stale = h->g.pack_s.stale = true;
  return DBM_OK;
}

// 0 = bf16 tensor-core path (default), 1 = "bf16x3": split-bf16 trunk and upsample convs on the tensor cores, stem and
// deformable layers fp32 -- fp32-grade results (GeneratorModel(precision="bf16x3") of the Python shim)
extern "C" int dbm_gen_set_precision(dbm_gen* h, int precision) {
  DBM_REQUIRE(h != nullptr, "gen_set_precision: null handle");
  DBM_REQUIRE(precision == 0 || precision == 1, "gen_set_precision: %d (0 = bf16, 1 = bf16x3)", precision);
  h->g.precision = precision;
  h->g.tab_ws = nullptr;
  return DBM_OK;
}

extern "C" size_t dbm_gen_workspace_bytes(const dbm_gen* h, int n, int h_in, int w_in) {
  if (!h || n <= 0 || h_in < 3 || w_in < 3) return 0;
  if (h->g.precision == 1) return ws_layout_split(&h->g, n, h_in, w_in).total;
  return ws_layout(&h->g, n, h_in, w_in).total;
}

extern "C" int dbm_gen_forward(dbm_gen* h, const float* x, const float* w1, const float* w2, const float* w3, int n,
                               int h_in, int w_in, float* y_out, void* workspace, size_t workspace_bytes,
                               cudaStream_t st) {
  DBM_REQUIRE(h && x && w1 && w2 && w3 && y_out && workspace, "gen_forward: null argument");
  // Chainer raises InvalidType from F.concat for inconsistent input sizes (srgan_train.py:265): shapes are implied here
  // by (n, h, w): x (n,1,h,w), w1 (n,1,10h,10w), w2 (n,2,2h,2w), w3 (n,1,h,w) -> y (n,1,4(h-2),4(w-2))
  DBM_REQUIRE(n > 0 && h_in >= 3 && w_in >= 3, "gen_forward: input %d x %d x %d too small (need >= 3 x 3)", n, h_in, w_in);
  Gen* g = &h->g;
  DBM_REQUIRE(((uintptr_t)workspace & 1023) == 0, "gen_forward: workspace must be 1024-byte aligned");
  if (g->precision == 1)
    return gen_forward_split(g, x, w1, w2, w3, n, h_in, w_in, y_out, workspace, workspace_bytes, st);
  const WsLayout L = ws_layout(g, n, h_in, w_in);
  DBM_REQUIRE(workspace_bytes >= L.total, "gen_forward: workspace of %zu bytes, need %zu (dbm_gen_workspace_bytes)",
              workspace_bytes, L.total);
  DBM_REQUIRE(((uintptr_t)workspace & 1023) == 0, "gen_forward: workspace must be 1024-byte aligned");
  uint8_t* ws = (uint8_t*)workspace;
  const int H = h_in - 2, W = w_in - 2;
  int rc = refresh_packed(g, st);
  if (rc) return rc;
  if (g->tab_ws != workspace || g->tab_n != n || g->tab_h != h_in || g->tab_w != w_in || g->tab_precision != 0) {
    build_trunk_passes(g, g->pack, L, ws, g->tab_host);
    DBM_REQUIRE((int)g->tab_host.size() == L.num_layers, "gen_forward: pass table has %zu entries, expected %d",
                g->tab_host.size(), L.num_layers);
    // the table is read by this very stream's kernels only: an ordered copy is enough
    DBM_CUDA(cudaMemcpyAsync(ws + L.table, g->tab_host.data(), g->tab_host.size() * sizeof(TrunkLayer),
                             cudaMemcpyHostToDevice, st));
    DBM_CUDA(cudaStreamSynchronize(st));   // tab_host is pageable: the copy must have left it before it is reused
    g->tab_ws = workspace; g->tab_n = n; g->tab_h = h_in; g->tab_w = w_in; g->tab_precision = 0;
  }
  void* s2d = ws + L.s2d;
  void* s0 = ws + L.s0;
  const uint8_t* arena = g->pack.base;
  const float* wts = (const float*)(arena + g->off_wts);
  const float* bias128 = (const float*)(arena + g->off_bias128);
  auto image = [&](const char* name) { return (const void*)g->pack.image(name); };
  // ---- input block (srgan_train.py:256-266) ----
  if ((rc = dbm_stem_w1_s2d(w1, s2d, n, h_in, w_in, st))) return rc;
  if ((rc = dbm_stem_fwd_slab8(x, nullptr, w2, w3, nullptr, wts, bias128, s0, 16, 0, n, h_in, w_in, st))) return rc;
  if ((rc = dbm_conv3x3_umma_valid(s2d, 40, 320, arena + g->off_w1tc, P(g, "input_block/conv_on_W1/b"), n, h_in, w_in,
                                   s0, 16, 4, st)))
    return rc;
  // ---- pre-residual conv, 12 x RRDB, post-residual conv + skip + nearest x2 (:541-558) ----
  const int ccs = (64 + 4 * g->inter) / 8;
  if ((rc = dbm_trunk_umma(ws + L.table, L.num_layers, n, H, W, s0, 16, ws + L.cat[0], ws + L.cat[1], ccs,
                           (unsigned int*)(ws + L.flags), st)))
    return rc;
  // ---- upsample convs (:556-568) ----
  void* u1 = ws + L.u1;
  void* u2 = ws + L.u2;
  void* f1 = ws + L.f1;
  float* offs = (float*)(ws + L.offs);
  if ((rc = dbm_conv3x3_umma(u1, 8, 64, image("up1"), P(g, "post_upsample_conv_layer_1/b"), 64, n, 2 * H, 2 * W, 0.f, 1, 1,
                             u2, 8, 0, nullptr, 0, 0, nullptr, nullptr, st)))
    return rc;
  if ((rc = dbm_conv3x3_umma(u2, 8, 64, image("up2"), P(g, "post_upsample_conv_layer_2/b"), 64, n, 4 * H, 4 * W, 0.f, 1, 0,
                             f1, 8, 0, nullptr, 0, 0, nullptr, nullptr, st)))
    return rc;
  // ---- deformable layers (:572-574) ----
  if ((rc = dbm_conv3x3_umma(f1, 8, 64, image("off1"), (const float*)(arena + g->off_bias_off1), 32, n, 4 * H, 4 * W,
                             0.f, 0, 0, nullptr, 0, 0, offs, 8, 0, nullptr, nullptr, st)))
    return rc;
  void* d1 = u2;
  if ((rc = dbm_deform_conv_umma(f1, offs, 8, image("dc1"), P(g, "final_conv_layer1/deform_conv/b"), n, 4 * H, 4 * W, 1, d1,
                                 8, 0, nullptr, nullptr, st)))
    return rc;
  if ((rc = dbm_conv3x3_umma(d1, 8, 64, image("off2"), (const float*)(arena + g->off_bias_off2), 32, n, 4 * H, 4 * W,
                             0.f, 0, 0, nullptr, 0, 0, offs, 8, 0, nullptr, nullptr, st)))
    return rc;
  return dbm_deform_conv_out1(d1, offs, 8, P(g, "final_conv_layer2/deform_conv/W"), P(g, "final_conv_layer2/deform_conv/b"),
                              y_out, (float*)(ws + L.proj), n, 4 * H, 4 * W, st);
}
