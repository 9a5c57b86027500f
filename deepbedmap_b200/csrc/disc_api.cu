// Model-level C entry points of the discriminator (SURVEY 8b): a host in any language trains DiscriminatorModel
// (srgan_train.py:591-699) with
//   dbm_disc_create -> dbm_disc_set_param (x every array of the Chainer .npz) -> dbm_disc_workspace_bytes ->
//   dbm_disc_zero_grads -> dbm_disc_forward(save = 1) -> (loss gradient) -> dbm_disc_backward -> (optimizer)
// and nothing of the Python shim. The handle owns the fp32 master weights and gradients (or views caller-owned flat
// buffers, dbm_disc_bind_params / _grads), the BatchNormalization running statistics and counters, the packed bf16
// operand images of conv_layer1..9 and every device table; activations live in the caller's workspace; all work is
// enqueued on the caller's stream. Forward and backward are DiscriminatorModel.forward / .backward of
// deepbedmap_b200/model.py with flat.FlatConv: the same entry points, with the same arguments, in the same order, on one
// stream (the class moves the weight gradients to a side stream; that changes when they run, not what they compute).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "flat_records.cuh"
#include "umma_common.cuh"

namespace dbm {

// (out_channels, ksize, stride) of conv_layer0..9 (srgan_train.py:617-634; deepbedmap_b200/layout.py DISC_CONVS)
static const int kConv[10][3] = {{64, 3, 1},  {64, 4, 2},  {128, 3, 1}, {128, 4, 2}, {128, 3, 1},
                                 {256, 4, 2}, {256, 3, 1}, {512, 4, 2}, {512, 3, 1}, {512, 4, 2}};
constexpr int kImg = 36;                          // linear_1 takes 512 inputs: 36 x 36 images (srgan_train.py:646, 693)
constexpr float kBnEps = 1e-5f, kBnDecay = 0.9f;  // L.BatchNormalization(eps=1e-5), Chainer's decay (:636)
constexpr long kPartialFloats = 9 * 32 * 128;     // one weight-gradient unit's partial sums (flat.PARTIAL_FLOATS)
constexpr int kTargetUnits = 296;                 // flat.FlatConv.TARGET_UNITS
constexpr int kMaxTables = 4;                     // cached (workspace, n, precision) table sets

enum ArrayKind { kParam = 0, kStat = 1, kCount = 2 };

struct DiscArray {
  std::string key;
  int ndim;
  int dims[4];
  long off, n;   // kParam: offset into the parameter buffer; kStat: into the running statistics; kCount: layer
  int kind;
};

// One convolution i = 1..9 on the flat tensor-core kernels (flat.ConvImages / flat.FlatConv) for a batch of n
struct ConvShape {
  int C, O, k, s, h, ho;              // NCHW: (n, C, h, h) -> (n, O, ho, ho)
  int s2d, Cg, Opad, Nf, ny_f, Nd, ny_d;
  int gh, P, tiles, Pg;               // flat geometry of the GEMM input (h, or h / 2 after space-to-depth)
  int nchunks, nsplit, units;         // weight-gradient units: nchunks x Opad / 32 x nsplit
};

struct WsLayout {
  size_t x, a0, z[10], y[10], mean[10], invstd[10], l1, r0, r1, dl1, bn_scratch;
  size_t xin[10], zf[10], gin[10], dxf[10], partial;   // precision 0 only
  size_t total;
  ConvShape L[10];
};

// Cached per (workspace, n, precision): the host launch records of dbm_flat_conv3x3_seq and the device unit / reduce
// tables of dbm_flat_wgrad(_reduce), whose pointers lead into that workspace; and whether the workspace holds a saved
// forward pass for backward.
struct Tables {
  const void* ws = nullptr;
  int n = 0, precision = 0;
  FlatLaunch rec_f[10], rec_d[10];
  uint8_t* dev = nullptr;
  int unit0[10], reduce0[10], n_reduce[10];   // record offsets into dev
  bool saved = false;
  int groups = 1;
  unsigned long long used = 0;
};

struct Disc {
  int dev = 0, precision = 0;
  std::vector<DiscArray> arrays;
  std::map<std::string, int> index;
  long total = 0;
  float* flat = nullptr;
  bool owns_flat = false;
  float* grad = nullptr;
  bool owns_grad = false;
  float* stats = nullptr;   // avg_mean, avg_var of batch_norm1..9
  long stats_total = 0;
  long bn_N[10] = {0};      // batch_norm{i}/N: kept as loaded (model.py:1183)
  // packed operand images of conv_layer1..9 (forward and data-gradient) in one arena; pack table on the device
  uint8_t* arena = nullptr;
  size_t img_fwd[10], img_dgrad[10];
  PackEntry* pack_dev = nullptr;
  int pack_n = 0;
  long pack_max = 0;
  bool stale = true;
  std::vector<Tables*> tables;
  unsigned long long tick = 0;
};

static const DiscArray* find(const Disc* d, const std::string& key) {
  auto it = d->index.find(key);
  return it == d->index.end() ? nullptr : &d->arrays[it->second];
}
static float* P(const Disc* d, const std::string& key) { return d->flat + find(d, key)->off; }
static float* G(const Disc* d, const std::string& key) { return d->grad + find(d, key)->off; }
static float* S(const Disc* d, const std::string& key) { return d->stats + find(d, key)->off; }
static std::string L_(const char* pre, int i, const char* post) { return pre + std::to_string(i) + post; }

static void add_array(Disc* d, const std::string& key, int kind, int ndim, int d0 = 0, int d1 = 0, int d2 = 0,
                      int d3 = 0) {
  DiscArray a;
  a.key = key; a.kind = kind; a.ndim = ndim;
  a.dims[0] = d0; a.dims[1] = d1; a.dims[2] = d2; a.dims[3] = d3;
  a.n = ndim == 0 ? 1 : ndim == 1 ? d0 : ndim == 2 ? (long)d0 * d1 : (long)d0 * d1 * d2 * d3;
  if (kind == kParam) { a.off = d->total; d->total += a.n; }
  else if (kind == kStat) { a.off = d->stats_total; d->stats_total += a.n; }
  else a.off = -1;
  d->index[key] = (int)d->arrays.size();
  d->arrays.push_back(a);
}

// The 33 parameters in layout.discriminator_shapes() order (= DiscriminatorModel.flat), then avg_mean / avg_var / N of
// batch_norm1..9 (the 27 persistents serialised next to them, SURVEY App. C)
static void build_inventory(Disc* d) {
  int cin = 1;
  for (int i = 0; i < 10; ++i) {
    const int cout = kConv[i][0], k = kConv[i][1];
    add_array(d, L_("conv_layer", i, "/W"), kParam, 4, cout, cin, k, k);
    if (i == 0) {
      add_array(d, "conv_layer0/b", kParam, 1, cout);
    } else {
      add_array(d, L_("batch_norm", i, "/gamma"), kParam, 1, cout);
      add_array(d, L_("batch_norm", i, "/beta"), kParam, 1, cout);
    }
    cin = cout;
  }
  add_array(d, "linear_1/W", kParam, 2, 100, 512);
  add_array(d, "linear_1/b", kParam, 1, 100);
  add_array(d, "linear_2/W", kParam, 2, 1, 100);
  add_array(d, "linear_2/b", kParam, 1, 1);
  for (int i = 1; i < 10; ++i) {
    add_array(d, L_("batch_norm", i, "/avg_mean"), kStat, 1, kConv[i][0]);
    add_array(d, L_("batch_norm", i, "/avg_var"), kStat, 1, kConv[i][0]);
    add_array(d, L_("batch_norm", i, "/N"), kCount, 0);
  }
}

// ---- flat.ConvImages: operand images of conv_layer1..9 and their pack table ------------------------------------
static void image_shape(int i, ConvShape& c) {
  c.O = kConv[i][0]; c.C = kConv[i - 1][0]; c.k = kConv[i][1]; c.s = kConv[i][2];
  c.s2d = c.k == 4;
  c.Cg = c.s2d ? 4 * c.C : c.C;
  c.Opad = (c.O + 31) / 32 * 32;
  c.Nf = c.Opad < 128 ? c.Opad : 128;
  c.ny_f = c.Opad / c.Nf;
  c.Nd = c.Cg < 128 ? c.Cg : 128;
  c.ny_d = c.Cg / c.Nd;
}

static std::vector<PackEntry> pack_entries(const Disc* d) {
  std::vector<PackEntry> ent;
  for (int i = 1; i < 10; ++i) {
    ConvShape c;
    image_shape(i, c);
    const float* w = P(d, L_("conv_layer", i, "/W"));
    __nv_bfloat16* fwd = (__nv_bfloat16*)(d->arena + d->img_fwd[i]);
    __nv_bfloat16* dgr = (__nv_bfloat16*)(d->arena + d->img_dgrad[i]);
    for (int y = 0; y < c.ny_f; ++y) {
      const int rows = c.O - y * c.Nf < c.Nf ? c.O - y * c.Nf : c.Nf;
      ent.push_back(PackEntry{w + (long)y * c.Nf * c.C * c.k * c.k, fwd + (long)y * 9 * c.Cg * c.Nf, rows, 0, c.Cg, c.C,
                              0, c.Nf, 16, c.s2d ? 2 : 0});
    }
    for (int y = 0; y < c.ny_d; ++y)
      ent.push_back(PackEntry{w, dgr + (long)y * 9 * c.Opad * c.Nd, c.Nd, c.O < c.Opad ? c.O : 0, c.Opad, c.C, y * c.Nd,
                              c.Nd, 16, c.s2d ? 3 : 1});
  }
  return ent;
}

static int build_pack_plan(Disc* d) {
  size_t off = 0;
  long mx = 0;
  for (int i = 1; i < 10; ++i) {
    ConvShape c;
    image_shape(i, c);
    d->img_fwd[i] = off;
    off += ((size_t)c.ny_f * 9 * c.Cg * c.Nf * 2 + 1023) & ~(size_t)1023;
    d->img_dgrad[i] = off;
    off += ((size_t)c.ny_d * 9 * c.Opad * c.Nd * 2 + 1023) & ~(size_t)1023;
    const long e = (long)9 * c.Cg * c.Nf > (long)9 * c.Opad * c.Nd ? (long)9 * c.Cg * c.Nf : (long)9 * c.Opad * c.Nd;
    if (e > mx) mx = e;
  }
  DBM_CUDA(cudaMalloc(&d->arena, off));
  DBM_CUDA(cudaMemset(d->arena, 0, off));   // rows the pack leaves alone stay zero (flat.ConvImages: ops.zeros)
  const std::vector<PackEntry> ent = pack_entries(d);
  d->pack_n = (int)ent.size();
  d->pack_max = mx;
  DBM_CUDA(cudaMalloc(&d->pack_dev, ent.size() * sizeof(PackEntry)));
  DBM_CUDA(cudaMemcpy(d->pack_dev, ent.data(), ent.size() * sizeof(PackEntry), cudaMemcpyHostToDevice));
  return DBM_OK;
}

// ---- workspace layout ------------------------------------------------------------------------------------------
static void split_blocks(int tiles, int nsplit, std::vector<std::pair<int, int>>& out) {   // flat.split_blocks
  if (nsplit > tiles) nsplit = tiles;
  if (nsplit < 1) nsplit = 1;
  const int base = tiles / nsplit, rem = tiles % nsplit;
  out.clear();
  for (int s = 0, b = 0; s < nsplit; ++s) {
    const int k = base + (s < rem ? 1 : 0);
    out.emplace_back(b, k);
    b += k;
  }
}

static int s2d_tap_mask(int c0, int nch, int C) {   // flat.s2d_tap_mask
  int mask = 0;
  for (int ph = c0 / C; ph <= (c0 + nch - 1) / C; ++ph) {
    const int py = ph >> 1, px = ph & 1;
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b) {
        const int ky = py == 0 ? 1 + a : a, kx = px == 0 ? 1 + b : b;
        mask |= 1 << (ky * 3 + kx);
      }
  }
  return mask;
}

static WsLayout ws_layout(int n, int precision) {
  WsLayout L;
  memset(&L, 0, sizeof(L));
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += (bytes + 1023) & ~(size_t)1023;
    return o;
  };
  const size_t N = (size_t)n;
  L.x = take(N * kImg * kImg * 4);                    // the input, kept for conv_layer0's weight gradient
  L.a0 = take(N * 64 * kImg * kImg * 4);
  size_t zmax = 0, dxmax = N * 512 * 4;               // dx of every conv and d(loss)/d(flat)
  int h = kImg;
  long partial_max = 0;
  for (int i = 1; i < 10; ++i) {
    ConvShape& c = L.L[i];
    image_shape(i, c);
    c.h = h;
    c.ho = (h + 2 - c.k) / c.s + 1;
    const size_t zb = N * c.O * c.ho * c.ho * 4;
    L.z[i] = take(zb);
    L.y[i] = take(zb);
    L.mean[i] = take(N * c.O * 4);                    // [groups][O], groups <= n
    L.invstd[i] = take(N * c.O * 4);
    if (zb > zmax) zmax = zb;
    if (N * c.C * h * h * 4 > dxmax) dxmax = N * c.C * h * h * 4;
    if (precision == 0) {
      c.gh = c.s2d ? (h + 1) / 2 : h;
      int g5[5];
      dbm_flat_geometry(n, c.gh, c.gh, g5);
      c.P = g5[0]; c.tiles = g5[1]; c.Pg = g5[3];
      const size_t pg = (size_t)c.Pg;
      L.xin[i] = take(c.Cg * pg * 2);
      L.zf[i] = take(c.Opad * pg * 4);
      L.gin[i] = take(c.Opad * pg * 2);
      L.dxf[i] = take(c.Cg * pg * 4);
      c.nchunks = (c.Cg + 127) / 128;
      // Python's round(): half to even, as nearbyint in the default rounding mode
      int ns = (int)std::nearbyint((double)kTargetUnits / (c.nchunks * (c.Opad / 32)));
      if (ns > c.tiles) ns = c.tiles;
      c.nsplit = ns < 1 ? 1 : ns;
      c.units = c.nchunks * (c.Opad / 32) * c.nsplit;
      if (c.units > partial_max) partial_max = c.units;
    }
    h = c.ho;
  }
  L.l1 = take(N * 100 * 4);
  L.r0 = take(dxmax);                                 // backward: d(loss)/d(conv input), in turn
  L.r1 = take(zmax);                                  // backward: d(loss)/d(conv output)
  L.dl1 = take(N * 100 * 4);
  L.bn_scratch = take(N * 2 * 512 * 4);               // [groups][2 O]
  if (precision == 0) L.partial = take((size_t)partial_max * kPartialFloats * 4);   // shared: layers run in turn
  L.total = off;
  return L;
}

// flat.FlatConv's launch records and weight-gradient tables for one workspace
static int build_tables(Disc* d, const WsLayout& L, uint8_t* ws, Tables* t, cudaStream_t st) {
  std::vector<WgradUnit> units;
  std::vector<WgradReduce> reduces;
  std::vector<std::pair<int, int>> splits;
  float* partial = (float*)(ws + L.partial);
  for (int i = 1; i < 10; ++i) {
    const ConvShape& c = L.L[i];
    const long Pg = c.Pg;
    __nv_bfloat16* xin = (__nv_bfloat16*)(ws + L.xin[i]);
    __nv_bfloat16* gin = (__nv_bfloat16*)(ws + L.gin[i]);
    auto epi = [](float* out_f32) {
      FlatEpiBlock e;
      memset(&e, 0, sizeof(e));
      e.s1 = e.beta = e.beta2 = e.out_scale = 1.f;
      e.out_f32 = out_f32;
      return e;
    };
    FlatLaunch& f = t->rec_f[i];
    memset(&f, 0, sizeof(f));
    f.in = xin;
    f.wpacked = (const __nv_bfloat16*)(d->arena + d->img_fwd[i]);
    f.cin = c.Cg; f.nout = c.Nf; f.ny = c.ny_f;
    f.w_chunk_stride = (long)9 * c.Cg * c.Nf;
    for (int b = 0; b < c.Nf / 32; ++b) f.blk[b] = epi((float*)(ws + L.zf[i]) + 32 * b * Pg);
    FlatLaunch& g = t->rec_d[i];
    memset(&g, 0, sizeof(g));
    g.in = gin;
    g.wpacked = (const __nv_bfloat16*)(d->arena + d->img_dgrad[i]);
    g.cin = c.Opad; g.nout = c.Nd; g.ny = c.ny_d;
    g.w_chunk_stride = (long)9 * c.Opad * c.Nd;
    for (int b = 0; b < c.Nd / 32; ++b) g.blk[b] = epi((float*)(ws + L.dxf[i]) + 32 * b * Pg);
    split_blocks(c.tiles, c.nsplit, splits);
    t->unit0[i] = (int)units.size();
    t->reduce0[i] = (int)reduces.size();
    int u = 0;
    for (int og = 0; og < c.Opad / 32; ++og)
      for (int c0 = 0; c0 < c.Cg; c0 += 128) {
        const int nch = c.Cg - c0 < 128 ? c.Cg - c0 : 128;
        const int first = u;
        for (const auto& sp : splits) {
          WgradUnit w;
          memset(&w, 0, sizeof(w));
          w.act = xin + (long)c0 * Pg;
          w.gout = gin + (long)32 * og * Pg;
          w.partial = partial + (long)u * kPartialFloats;
          w.blk0 = sp.first; w.nblk = sp.second; w.nslab = nch / 8;
          w.tapmask = c.s2d ? s2d_tap_mask(c0, nch, c.C) : 0;
          units.push_back(w);
          ++u;
        }
        const int ovalid = c.O - 32 * og < 32 ? c.O - 32 * og : 32;
        WgradReduce r;
        memset(&r, 0, sizeof(r));
        r.partial = partial + (long)first * kPartialFloats;
        r.dw = G(d, L_("conv_layer", i, "/W"));
        r.split_stride = kPartialFloats;
        r.nsplit = (int)splits.size(); r.cin_total = c.C; r.c0 = c0; r.o0 = 32 * og; r.nch = nch;
        r.mode = (c.s2d ? 1 : 0) | ((ovalid < 32 ? ovalid : 0) << 8);
        reduces.push_back(r);
      }
    DBM_REQUIRE(u == c.units, "disc_forward: conv_layer%d has %d weight-gradient units, expected %d", i, u, c.units);
    t->n_reduce[i] = (int)reduces.size() - t->reduce0[i];
  }
  const size_t ub = units.size() * sizeof(WgradUnit), rb = reduces.size() * sizeof(WgradReduce);
  DBM_CUDA(cudaMalloc(&t->dev, ub + rb));
  DBM_CUDA(cudaMemcpyAsync(t->dev, units.data(), ub, cudaMemcpyHostToDevice, st));
  DBM_CUDA(cudaMemcpyAsync(t->dev + ub, reduces.data(), rb, cudaMemcpyHostToDevice, st));
  DBM_CUDA(cudaStreamSynchronize(st));   // the host vectors are pageable: the copies must have left them
  for (int i = 1; i < 10; ++i) t->reduce0[i] = (int)(ub / sizeof(WgradReduce)) + t->reduce0[i];
  return DBM_OK;
}

static void free_tables(Disc* d) {
  for (Tables* t : d->tables) {
    if (t->dev) cudaFree(t->dev);
    delete t;
  }
  d->tables.clear();
}

static Tables* lookup(Disc* d, const void* ws) {
  for (Tables* t : d->tables)
    if (t->ws == ws && t->precision == d->precision) return t;
  return nullptr;
}

// The tables of (workspace, n, precision): built and uploaded on first use (one stream synchronisation), afterwards only
// looked up. The batch split into `groups` does not enter them.
static int tables_for(Disc* d, const WsLayout& L, const void* ws, int n, cudaStream_t st, Tables** out) {
  Tables* t = lookup(d, ws);
  if (t && t->n != n) {
    if (t->dev) cudaFree(t->dev);
    d->tables.erase(std::find(d->tables.begin(), d->tables.end(), t));
    delete t;
    t = nullptr;
  }
  if (!t) {
    if ((int)d->tables.size() >= kMaxTables) {   // evict the least recently used set (cudaFree waits for the device)
      size_t lru = 0;
      for (size_t k = 1; k < d->tables.size(); ++k)
        if (d->tables[k]->used < d->tables[lru]->used) lru = k;
      if (d->tables[lru]->dev) cudaFree(d->tables[lru]->dev);
      delete d->tables[lru];
      d->tables.erase(d->tables.begin() + lru);
    }
    t = new Tables();
    t->ws = ws; t->n = n; t->precision = d->precision;
    if (d->precision == 0) {
      const int rc = build_tables(d, L, (uint8_t*)ws, t, st);
      if (rc) {
        if (t->dev) cudaFree(t->dev);
        delete t;
        return rc;
      }
    }
    d->tables.push_back(t);
  }
  t->used = ++d->tick;
  *out = t;
  return DBM_OK;
}

static int check_device(const Disc* d, const char* who) {
  int cur = -1;
  DBM_CUDA(cudaGetDevice(&cur));
  DBM_REQUIRE(cur == d->dev, "%s: the handle belongs to device %d, the current device is %d", who, d->dev, cur);
  return DBM_OK;
}

#define DBM_TRY(expr)          \
  do {                         \
    const int rc_ = (expr);    \
    if (rc_) return rc_;       \
  } while (0)

static int disc_forward(Disc* d, const float* x, int n, int groups, int train, int save, float* logits, void* workspace,
                        size_t bytes, cudaStream_t st) {
  DBM_REQUIRE(x && logits && workspace, "disc_forward: null argument");
  DBM_REQUIRE(n >= 1, "disc_forward: batch of %d", n);
  DBM_REQUIRE(groups >= 1 && n % groups == 0, "disc_forward: batch of %d does not split into %d groups", n, groups);
  DBM_REQUIRE(!save || train, "disc_forward: backward through eval-mode BatchNormalization is not needed by the reference");
  DBM_REQUIRE(((uintptr_t)workspace & 1023) == 0, "disc_forward: workspace must be 1024-byte aligned");
  const WsLayout L = ws_layout(n, d->precision);
  DBM_REQUIRE(bytes >= L.total, "disc_forward: workspace of %zu bytes, need %zu (dbm_disc_workspace_bytes)", bytes,
              L.total);
  DBM_TRY(check_device(d, "disc_forward"));
  Tables* t = nullptr;
  DBM_TRY(tables_for(d, L, workspace, n, st, &t));
  t->saved = false;   // this pass overwrites whatever the workspace kept
  uint8_t* ws = (uint8_t*)workspace;
  const bool tc = d->precision == 0;
  const int ng = n / groups;
  if (tc)   // flat operands are read with their one-pixel zero border, which no kernel writes (flat.alloc_bf16)
    for (int i = 1; i < 10; ++i) {
      const ConvShape& c = L.L[i];
      DBM_CUDA(cudaMemsetAsync(ws + L.xin[i], 0, (size_t)c.Cg * c.Pg * 2, st));
      DBM_CUDA(cudaMemsetAsync(ws + L.gin[i], 0, (size_t)c.Opad * c.Pg * 2, st));
    }
  if (save) DBM_CUDA(cudaMemcpyAsync(ws + L.x, x, (size_t)n * kImg * kImg * 4, cudaMemcpyDeviceToDevice, st));
  float* a0 = (float*)(ws + L.a0);
  DBM_TRY(dbm_conv2d_fwd_f32(x, kImg * kImg, P(d, "conv_layer0/W"), P(d, "conv_layer0/b"), a0, 64 * kImg * kImg, n, 1,
                             kImg, kImg, 64, 3, 1, 1, 1, st));
  if (tc && d->stale) {
    DBM_TRY(dbm_pack_conv3x3_table(d->pack_dev, d->pack_n, d->pack_max, st));
    d->stale = false;
  }
  const float* cur = a0;
  for (int i = 1; i < 10; ++i) {
    const ConvShape& c = L.L[i];
    float* z = (float*)(ws + L.z[i]);
    float* y = (float*)(ws + L.y[i]);
    if (tc) {
      DBM_TRY(dbm_flat_from_nchw_ex(cur, c.C, c.h, c.h, c.s2d, ws + L.xin[i], nullptr, 1.f, n, c.gh, c.gh, st));
      DBM_TRY(dbm_flat_conv3x3_seq(&t->rec_f[i], 1, n, c.gh, c.gh, c.ho, c.ho, st));
      DBM_TRY(dbm_flat_to_nchw_ex((const float*)(ws + L.zf[i]), nullptr, z, c.O, c.ho, c.ho, 0, n, c.gh, c.gh, st));
    } else {
      DBM_TRY(dbm_conv2d_fwd_f32(cur, (long)c.C * c.h * c.h, P(d, L_("conv_layer", i, "/W")), nullptr, z,
                                 (long)c.O * c.ho * c.ho, n, c.C, c.h, c.h, c.O, c.k, c.s, 1, 0, st));
    }
    DBM_TRY(dbm_bn_lrelu_fwd_groups_f32(z, y, P(d, L_("batch_norm", i, "/gamma")), P(d, L_("batch_norm", i, "/beta")),
                                        S(d, L_("batch_norm", i, "/avg_mean")), S(d, L_("batch_norm", i, "/avg_var")),
                                        (float*)(ws + L.mean[i]), (float*)(ws + L.invstd[i]), groups, ng, c.O,
                                        c.ho * c.ho, kBnEps, kBnDecay, train, st));
    cur = y;
  }
  float* l1 = (float*)(ws + L.l1);
  DBM_TRY(dbm_gemm_f32(cur, 512, 1, 0, P(d, "linear_1/W"), 1, 512, 0, l1, 100, 1, 0, P(d, "linear_1/b"), n, 100, 512, 1,
                       1, 0, st));
  DBM_TRY(dbm_gemm_f32(l1, 100, 1, 0, P(d, "linear_2/W"), 1, 100, 0, logits, 1, 1, 0, P(d, "linear_2/b"), n, 1, 100, 1, 0,
                       0, st));
  if (save) {
    t->saved = true;
    t->groups = groups;
  }
  return DBM_OK;
}

static int disc_backward(Disc* d, const float* dlogit, void* workspace, size_t bytes, cudaStream_t st) {
  DBM_REQUIRE(dlogit && workspace, "disc_backward: null argument");
  DBM_REQUIRE(((uintptr_t)workspace & 1023) == 0, "disc_backward: workspace must be 1024-byte aligned");
  Tables* t = lookup(d, workspace);
  DBM_REQUIRE(t && t->saved, "disc_backward: this workspace holds no saved pass (run dbm_disc_forward with save = 1 on "
              "it first; each pass is consumed by one backward)");
  const int n = t->n, groups = t->groups, ng = n / groups;
  const WsLayout L = ws_layout(n, d->precision);
  DBM_REQUIRE(bytes >= L.total, "disc_backward: workspace of %zu bytes, need %zu (dbm_disc_workspace_bytes)", bytes,
              L.total);
  DBM_TRY(check_device(d, "disc_backward"));
  t->saved = false;
  uint8_t* ws = (uint8_t*)workspace;
  const bool tc = d->precision == 0;
  const float* l1 = (const float*)(ws + L.l1);
  float* dl1 = (float*)(ws + L.dl1);
  float* r0 = (float*)(ws + L.r0);
  float* r1 = (float*)(ws + L.r1);
  // linear_2
  DBM_TRY(dbm_gemm_f32(dlogit, 1, 1, 0, l1, 100, 1, 0, G(d, "linear_2/W"), 100, 1, 0, nullptr, 1, 100, n, 1, 0, 1, st));
  DBM_TRY(dbm_bias_grad_f32(dlogit, 1, G(d, "linear_2/b"), n, 1, 1, st));
  DBM_TRY(dbm_gemm_f32(dlogit, 1, 1, 0, P(d, "linear_2/W"), 100, 1, 0, dl1, 100, 1, 0, nullptr, n, 100, 1, 1, 0, 0, st));
  DBM_TRY(dbm_lrelu_bwd_f32(dl1, 100, l1, 100, dl1, 100, n, 100, 0, st));
  // linear_1: dW[o, i] += sum_n dl1[n, o] * flat[n, i]
  const float* flat = (const float*)(ws + L.y[9]);
  DBM_TRY(dbm_gemm_f32(dl1, 1, 100, 0, flat, 512, 1, 0, G(d, "linear_1/W"), 512, 1, 0, nullptr, 100, 512, n, 1, 0, 1, st));
  DBM_TRY(dbm_bias_grad_f32(dl1, 100, G(d, "linear_1/b"), n, 100, 1, st));
  DBM_TRY(dbm_gemm_f32(dl1, 100, 1, 0, P(d, "linear_1/W"), 512, 1, 0, r0, 512, 1, 0, nullptr, n, 512, 100, 1, 0, 0, st));
  // conv_layer9 .. 1 with their BatchNormalization + LeakyReLU; d(loss)/d(input) of each conv lands in r0
  for (int i = 9; i >= 1; --i) {
    const ConvShape& c = L.L[i];
    const float* z = (const float*)(ws + L.z[i]);
    const float* y = (const float*)(ws + L.y[i]);
    const float* xin = i == 1 ? (const float*)(ws + L.a0) : (const float*)(ws + L.y[i - 1]);
    DBM_TRY(dbm_bn_lrelu_bwd_groups_f32(z, y, r0, r1, P(d, L_("batch_norm", i, "/gamma")), (const float*)(ws + L.mean[i]),
                                        (const float*)(ws + L.invstd[i]), G(d, L_("batch_norm", i, "/gamma")),
                                        G(d, L_("batch_norm", i, "/beta")), (float*)(ws + L.bn_scratch), groups, ng,
                                        c.O, c.ho * c.ho, st));
    if (tc) {
      DBM_TRY(dbm_flat_from_nchw_ex(r1, c.O, c.ho, c.ho, 0, ws + L.gin[i], nullptr, 1.f, n, c.gh, c.gh, st));
      DBM_TRY(dbm_flat_wgrad(t->dev + (size_t)t->unit0[i] * sizeof(WgradUnit), c.units, n, c.gh, c.gh, st));
      DBM_TRY(dbm_flat_wgrad_reduce(t->dev + (size_t)t->reduce0[i] * sizeof(WgradReduce), t->n_reduce[i], st));
      DBM_TRY(dbm_flat_conv3x3_seq(&t->rec_d[i], 1, n, c.gh, c.gh, 0, 0, st));
      DBM_TRY(dbm_flat_to_nchw_ex((const float*)(ws + L.dxf[i]), nullptr, r0, c.C, c.h, c.h, c.s2d, n, c.gh, c.gh, st));
    } else {
      DBM_TRY(dbm_conv2d_bwd_weight_f32(xin, (long)c.C * c.h * c.h, r1, (long)c.O * c.ho * c.ho,
                                        G(d, L_("conv_layer", i, "/W")), n, c.C, c.h, c.h, c.O, c.k, c.s, 1, st));
      DBM_TRY(dbm_conv2d_bwd_data_f32(r1, (long)c.O * c.ho * c.ho, P(d, L_("conv_layer", i, "/W")), r0,
                                      (long)c.C * c.h * c.h, n, c.C, c.h, c.h, c.O, c.k, c.s, 1, 0, st));
    }
  }
  // conv_layer0 + LeakyReLU
  const long a0_bs = 64L * kImg * kImg;
  DBM_TRY(dbm_lrelu_bwd_f32(r0, a0_bs, (const float*)(ws + L.a0), a0_bs, r0, a0_bs, n, a0_bs, 0, st));
  DBM_TRY(dbm_conv2d_bwd_weight_f32((const float*)(ws + L.x), kImg * kImg, r0, a0_bs, G(d, "conv_layer0/W"), n, 1, kImg,
                                    kImg, 64, 3, 1, 1, st));
  return dbm_bias_grad_f32(r0, a0_bs, G(d, "conv_layer0/b"), n, 64, kImg * kImg, st);
}

}  // namespace dbm

using namespace dbm;

struct dbm_disc {
  Disc d;
};

extern "C" int dbm_disc_destroy(dbm_disc* h);

extern "C" int dbm_disc_create(dbm_disc** out) {
  DBM_REQUIRE(out != nullptr, "disc_create: null output");
  *out = nullptr;
  dbm_disc* h = new dbm_disc();
  Disc* d = &h->d;
  cudaGetDevice(&d->dev);
  build_inventory(d);
  // DiscriminatorModel's fixed initial values: BatchNormalization gamma = 1, avg_var = 1, everything else 0
  std::vector<float> p(d->total, 0.f), s(d->stats_total, 0.f);
  for (const DiscArray& a : d->arrays) {
    const bool gamma = a.key.size() > 6 && a.key.compare(a.key.size() - 6, 6, "/gamma") == 0;
    const bool var = a.key.size() > 8 && a.key.compare(a.key.size() - 8, 8, "/avg_var") == 0;
    if (gamma) std::fill(p.begin() + a.off, p.begin() + a.off + a.n, 1.f);
    if (var) std::fill(s.begin() + a.off, s.begin() + a.off + a.n, 1.f);
  }
  cudaError_t e = cudaMalloc(&d->flat, (size_t)d->total * 4);
  if (e == cudaSuccess) { d->owns_flat = true; e = cudaMalloc(&d->grad, (size_t)d->total * 4); }
  if (e == cudaSuccess) { d->owns_grad = true; e = cudaMalloc(&d->stats, (size_t)d->stats_total * 4); }
  if (e == cudaSuccess) e = cudaMemcpy(d->flat, p.data(), p.size() * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(d->grad, 0, (size_t)d->total * 4);
  if (e == cudaSuccess) e = cudaMemcpy(d->stats, s.data(), s.size() * 4, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    set_error("disc_create: %s", cudaGetErrorString(e));
    dbm_disc_destroy(h);
    return DBM_ERR_CUDA;
  }
  const int rc = build_pack_plan(d);
  if (rc) {
    dbm_disc_destroy(h);
    return rc;
  }
  *out = h;
  return DBM_OK;
}

extern "C" int dbm_disc_destroy(dbm_disc* h) {
  if (!h) return DBM_OK;
  Disc* d = &h->d;
  free_tables(d);
  if (d->owns_flat && d->flat) cudaFree(d->flat);
  if (d->owns_grad && d->grad) cudaFree(d->grad);
  if (d->stats) cudaFree(d->stats);
  if (d->arena) cudaFree(d->arena);
  if (d->pack_dev) cudaFree(d->pack_dev);
  delete h;
  return DBM_OK;
}

extern "C" int dbm_disc_set_precision(dbm_disc* h, int precision) {
  DBM_REQUIRE(h != nullptr, "disc_set_precision: null handle");
  DBM_REQUIRE(precision == 0 || precision == 1, "disc_set_precision: %d (0 = bf16, 1 = fp32)", precision);
  if (precision != h->d.precision) free_tables(&h->d);   // the workspace layout changes; saved passes are dropped
  h->d.precision = precision;
  return DBM_OK;
}

extern "C" long dbm_disc_count_params(const dbm_disc* h) { return h ? h->d.total : -1; }
extern "C" int dbm_disc_num_arrays(const dbm_disc* h) { return h ? (int)h->d.arrays.size() : -1; }

extern "C" int dbm_disc_array_info(const dbm_disc* h, int index, const char** key, int* ndim, int* dims4,
                                   long* flat_offset) {
  DBM_REQUIRE(h && index >= 0 && index < (int)h->d.arrays.size(), "disc_array_info: bad index %d", index);
  const DiscArray& a = h->d.arrays[index];
  if (key) *key = a.key.c_str();
  if (ndim) *ndim = a.ndim;
  if (dims4)
    for (int i = 0; i < 4; ++i) dims4[i] = a.dims[i];
  if (flat_offset) *flat_offset = a.kind == kParam ? a.off : -1;
  return DBM_OK;
}

static int check_array(const Disc* d, const char* who, const char* key, int ndim, const int* dims, const DiscArray** out) {
  const DiscArray* a = find(d, key);
  DBM_REQUIRE(a != nullptr, "%s: unknown key '%s'", who, key);
  bool ok = ndim == a->ndim;
  for (int i = 0; ok && i < ndim; ++i) ok = dims[i] == a->dims[i];
  DBM_REQUIRE(ok, "%s: '%s' has shape (%d,%d,%d,%d) of %d dims, got %d-d (%d,...)", who, key, a->dims[0], a->dims[1],
              a->dims[2], a->dims[3], a->ndim, ndim, ndim > 0 ? dims[0] : 0);
  *out = a;
  return DBM_OK;
}

extern "C" int dbm_disc_set_param(dbm_disc* h, const char* key, const float* host_values, int ndim, const int* dims) {
  DBM_REQUIRE(h && key && host_values && (dims || ndim == 0), "disc_set_param: null argument");
  Disc* d = &h->d;
  const DiscArray* a = nullptr;
  DBM_TRY(check_array(d, "disc_set_param", key, ndim, dims, &a));
  if (a->kind == kCount) {
    d->bn_N[std::stoi(a->key.substr(10))] = (long)host_values[0];
    return DBM_OK;
  }
  float* dst = a->kind == kParam ? d->flat + a->off : d->stats + a->off;
  DBM_CUDA(cudaMemcpy(dst, host_values, (size_t)a->n * 4, cudaMemcpyHostToDevice));
  if (a->kind == kParam) d->stale = true;
  return DBM_OK;
}

extern "C" int dbm_disc_get_param(const dbm_disc* h, const char* key, float* host_values) {
  DBM_REQUIRE(h && key && host_values, "disc_get_param: null argument");
  const Disc* d = &h->d;
  const DiscArray* a = find(d, key);
  DBM_REQUIRE(a != nullptr, "disc_get_param: unknown key '%s'", key);
  if (a->kind == kCount) {
    host_values[0] = (float)d->bn_N[std::stoi(a->key.substr(10))];
    return DBM_OK;
  }
  const float* src = a->kind == kParam ? d->flat + a->off : d->stats + a->off;
  DBM_CUDA(cudaMemcpy(host_values, src, (size_t)a->n * 4, cudaMemcpyDeviceToHost));
  return DBM_OK;
}

// View a caller-owned device buffer of dbm_disc_count_params floats (layout.discriminator_shapes() order) as the master
// weights; call dbm_disc_mark_updated after changing it.
extern "C" int dbm_disc_bind_params(dbm_disc* h, float* device_flat) {
  DBM_REQUIRE(h && device_flat, "disc_bind_params: null argument");
  Disc* d = &h->d;
  DBM_REQUIRE(d->owns_flat, "disc_bind_params: parameters are already bound");
  cudaFree(d->flat);
  d->flat = device_flat;
  d->owns_flat = false;
  const std::vector<PackEntry> ent = pack_entries(d);   // the pack table reads the filters from the new buffer
  DBM_CUDA(cudaMemcpy(d->pack_dev, ent.data(), ent.size() * sizeof(PackEntry), cudaMemcpyHostToDevice));
  d->stale = true;
  return DBM_OK;
}

// The same for the gradient buffer (backward accumulates into it). Drops the cached tables and any saved pass.
extern "C" int dbm_disc_bind_grads(dbm_disc* h, float* device_flat) {
  DBM_REQUIRE(h && device_flat, "disc_bind_grads: null argument");
  Disc* d = &h->d;
  DBM_REQUIRE(d->owns_grad, "disc_bind_grads: gradients are already bound");
  free_tables(d);   // the weight-gradient reduce tables point into the gradient buffer
  cudaFree(d->grad);
  d->grad = device_flat;
  d->owns_grad = false;
  return DBM_OK;
}

extern "C" int dbm_disc_mark_updated(dbm_disc* h) {
  DBM_REQUIRE(h != nullptr, "disc_mark_updated: null handle");
  h->d.stale = true;
  return DBM_OK;
}

extern "C" int dbm_disc_zero_grads(dbm_disc* h, cudaStream_t st) {
  DBM_REQUIRE(h != nullptr, "disc_zero_grads: null handle");
  return dbm_fill_f32(h->d.grad, 0.f, h->d.total, st);
}

extern "C" size_t dbm_disc_workspace_bytes(const dbm_disc* h, int n) {
  if (!h || n < 1) return 0;
  return ws_layout(n, h->d.precision).total;
}

extern "C" int dbm_disc_forward(dbm_disc* h, const float* x, int n, int groups, int train, int save, float* logits,
                                void* workspace, size_t workspace_bytes, cudaStream_t st) {
  DBM_REQUIRE(h != nullptr, "disc_forward: null handle");
  return disc_forward(&h->d, x, n, groups, train, save, logits, workspace, workspace_bytes, st);
}

extern "C" int dbm_disc_backward(dbm_disc* h, const float* dlogit, void* workspace, size_t workspace_bytes,
                                 cudaStream_t st) {
  DBM_REQUIRE(h != nullptr, "disc_backward: null handle");
  return disc_backward(&h->d, dlogit, workspace, workspace_bytes, st);
}
