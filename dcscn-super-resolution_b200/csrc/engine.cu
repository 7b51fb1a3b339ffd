// DCSCN engine: graph plan, parameter storage / packing, workspace, launch orchestration and the C-ABI
// declared in include/dcscn_b200.h.  Stands in for what `sess.run(self.y_)` executed in the reference
// (DCSCN.py:565; graph built by DCSCN.py:222-332 and helper/tf_graph.py:104-249).
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/dcscn_b200.h"
#include "common.h"
#include "conv_aux.cuh"
#include "conv_tc.cuh"
#include "conv_tc_pair.cuh"
#include "conv_tc_halo2.cuh"
#include "conv_ds.cuh"
#include "conv_ds_tile.cuh"
#include "train.cuh"
#include "wgrad_tc.cuh"
#include "train_ds.cuh"
#include "umma_probe.cuh"

using namespace dcscn;

// ----------------------------------------------------------------------------------------- errors ----
static thread_local std::string g_last_error;

static int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return 1;
}

#define CUDA_TRY(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return fail("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e)); \
  } while (0)

static inline int pad16(int v) { return (v + 15) & ~15; }

// ------------------------------------------------------------------------------------- graph plan ----
struct LayerDef {
  std::string scope;  // TF variable scope, e.g. "CNN3", "Up-PS/Up-PS_CNN"
  int k, cin, cout;
  bool bias, prelu;
};

struct ParamDef {
  std::string name;
  std::vector<int64_t> shape;
  std::vector<float> host;
  std::vector<float> shadow;    // flat index + 2 of every element (float-coded), see build_refresh_maps
  int64_t numel() const {
    int64_t n = 1;
    for (auto d : shape) n *= d;
    return n;
  }
};

// device-side packed form of one tensor-core layer (possibly a fusion of several TF layers)
struct TcLayer {
  std::string name;
  int ksz = 3;
  int cin_pad = 0;              // channel extent of the source region
  int n_tiles = 1, n_pad = 16;  // column tiling
  int n_valid = 0;
  std::vector<int> in_map;      // logical cin -> channel position in the source region
  std::vector<float> w_host;    // fused HWIO fp32 [taps][cin][cout]
  std::vector<float> bias_host, alpha_host;  // [n_tiles*n_pad]
  int cin = 0, cout = 0;
  float wscale = 1.f;
  float* d_bias = nullptr;
  float* d_alpha = nullptr;
  float* d_wref = nullptr;      // fp32 HWIO for the validation kernel
  int* d_in_map = nullptr;
  __half* d_wpair = nullptr;    // CTA-pair layout [n_tile][block][rank][plane][n_pad/2 x 64], blocks as in pair_image
  CUtensorMap tm_w;             // 2-D map over d_wpair (rows of 128 bytes)
  bool h2 = false;              // streaming 3x3 kernel (conv_tc_halo2.cuh): d_wpair is in its [chunk][dx][dy] stage order
  int h2_nseg = 0;              // its fp32-promotion segments per item
  int h2_seg_units = 1;         // its promotion period, in (chunk, dx) units
  int* d_pair_src = nullptr;    // training: flat parameter index behind every hi-plane element of d_wpair (-1 = zero)
  size_t pair_src_n = 0;
};

struct GatherJob {   // training: dst[i] = d_w[map[i]] where map[i] >= 0 (biases, PReLU slopes, CNN1 / R-CNN1 filters)
  float* dst;
  int* map;
  int n;
};

struct TcLaunch {
  int layer_index = -1;          // index into dcscn_handle::tcl (forward) or ::bwd (dgrad twins): the layer whose CURRENT
  bool layer_bwd = false;        // power-of-two weight scale the epilogue has to undo (it changes when a layer is re-packed)
  CUtensorMap tm_hi, tm_lo, tm_w;
  int pair_grid = 0, pair_stages = 0, pair_seg = 1;
  bool pair_stream = false;
  size_t pair_smem = 0;
  bool halo2 = false;            // 3x3 layers: streaming halo kernel on 16 x 8 pixel patches
  ConvGeom hg;
  int halo_grid = 0;
  CUtensorMap t1_hi, t1_lo;      // A maps with box {64, 10, 18, 1}
  int halo2_na = 0, halo2_nb = 0, halo2_seg = 1;
  size_t halo2_smem = 0;
  ConvTCParams p;
  ConvRefParams ref;
};

struct Plan {
  int n = 0, h = 0, w = 0;
  ConvFirstParams first;
  std::vector<TcLaunch> tc;      // in execution order
  ConvLastParams last;
  bool fused_last = false;       // Up-PS epilogue computes the per-pixel half of R-CNN1 (EPI_D2S_RDOT)
  int fused_index = -1;          // index into tc of the launch that carries the fused epilogue
  TcLaunch unfused;              // same layer with the plain depth_to_space epilogue (validation path)
  ConvGatherParams gather;
  bool ran_fused = false;
  std::vector<TcLaunch> bwd;     // dgrad launches (built lazily by the train step)
  bool bwd_built = false;
  // CUDA graph of CNN1 + the tensor-core layers (everything but the last kernel, the only one that reads x2 / writes y):
  // instantiated after the plan ran eagerly once, replayed while the input pointer and the option epoch stay the same
  cudaGraphExec_t gexec = nullptr;
  const float* g_x = nullptr;
  uint64_t g_epoch = 0;
  bool g_fused = false;
  int g_launches = 0;
  int eager_runs = 0;
  const float* last_x = nullptr; // input of the previous forward on this plan: a graph is only built for a pointer seen twice in a row
  ~Plan() { if (gexec) cudaGraphExecDestroy(gexec); }
};

struct dcscn_handle {
  dcscn_config cfg;
  int sm_count = 148;
  std::vector<int> filters;          // feature-extraction filter schedule
  std::vector<LayerDef> layers;      // graph-construction order (self.Weights order)
  std::vector<ParamDef> params;
  std::map<std::string, int> param_index;
  bool params_dirty = true;

  // layout
  std::vector<int> feat_off, feat_w;
  int feat_pitch = 0;
  int a1_w = 0, b1_w = 0, nin_pitch = 0;
  int ps_out = 0;                    // channels after the last depth_to_space
  int mid_pitch = 0;                 // x4: channels after the first depth_to_space (padded)

  // packed layers
  std::vector<TcLayer> tcl;          // CNN2..CNNL, A1+B1, B2, Up-PS [, Up-PS2]
  std::vector<TcLayer> bwd;          // data-gradient twins (transposed, flipped filters), see build_bwd_layers
  bool train_enabled = false;
  float *ens_x = nullptr, *ens_x2 = nullptr, *ens_y = nullptr;   // self-ensemble: transformed copies / per-flip outputs
  size_t ens_cap = 0;
  float *ensio_x = nullptr, *ensio_x2 = nullptr;                  // host-call staging of the ensemble entry point
  double* ensio_y = nullptr;
  size_t ensio_cap = 0;
  int l1_loss = 0;                   // --use_l1_loss: image_loss = mean |y_ - y| (DCSCN.py:342-344)
  int wgrad_taps = 0;                // 0 = automatic (up to 3 filter taps per wgrad CTA), else the cap
  int wgrad_impl = 0;                // 0 = tcgen05 (wgrad_tc.cuh), 1 = CUDA cores (validation)
  int host_repack = 0;               // option: always re-pack on the host after an update (validation of the device path)
  bool shadow_mode = false;          // P() returns index-coded shadows (build_refresh_maps)
  bool refresh_ready = false;        // device-side weight refresh maps are valid for the current packing
  std::vector<struct GatherJob> gather_jobs;
  struct TrainState* train = nullptr;
  float* d_first_w = nullptr;        // CNN1 [taps][n_pad]
  float* d_first_bias = nullptr;
  float* d_first_alpha = nullptr;
  float* d_last_w = nullptr;         // R-CNN1 [taps][C]

  // workspace (grow-only)
  size_t cap_px = 0;                 // LR pixels the buffers can hold
  __half *feat_hi = nullptr, *feat_lo = nullptr;
  __half *b1_hi = nullptr, *b1_lo = nullptr;
  __half *nin_hi = nullptr, *nin_lo = nullptr;
  __half *mid_hi = nullptr, *mid_lo = nullptr;
  float* hr = nullptr;
  float* vbuf = nullptr;             // tap-planar partial products of the fused R-CNN1 [9][N][sH][sW]
  float *io_x = nullptr, *io_x2 = nullptr, *io_y = nullptr;  // staging for forward_host
  size_t io_cap = 0;
  // training patch store (dcscn_patch_store_set): uint8 patches resident in HBM + the mini-batch's index list
  uint8_t *ps_lr = nullptr, *ps_bic = nullptr, *ps_true = nullptr;
  int64_t ps_count = 0;
  int ps_h = 0, ps_w = 0;
  int* ps_idx = nullptr;
  int ps_idx_cap = 0;
  // Pillow-bicubic resampling tables per (input size, output size) and the float32 intermediate of the two passes
  struct PilTable { int in = 0, out = 0, ksize = 0; double* k = nullptr; int* bounds = nullptr; };
  std::vector<PilTable> pil_tables;
  float* pil_tmp = nullptr;
  size_t pil_tmp_cap = 0;
  cudaStream_t copy_stream = nullptr;  // forward_host: x2 (only read by the last kernel) rides in beside the conv stack
  cudaEvent_t x2_ready = nullptr;
  bool wait_x2 = false;                // the next forward's last kernel waits for x2_ready
  int64_t device_bytes = 0;

  // depthwise-separable graphs: fp32 buffers + per-layer device filters
  struct DsDev { float *dw = nullptr, *pw = nullptr, *bias = nullptr, *alpha = nullptr; };
  std::vector<DsDev> ds;             // same order as `layers`
  DsDev ds_ab;                       // fused A1 | B1 1x1 layer of the tile kernels: [concat positions][A1 cols | B1 cols], scales folded
  int ds_impl = 0;                   // 0 = tile kernels (conv_ds_tile.cuh), 1 = first-generation kernels (cross-check)
  int ds_cache = 1;                  // option "ds_cache": pixel-shuffler layers keep their depthwise values across column groups
  float *ds_feat = nullptr, *ds_b1 = nullptr, *ds_nin = nullptr, *ds_mid = nullptr, *ds_hr = nullptr;
  int ds_total = 0;                  // channels of the (unpadded) concat buffer
  int ds_n = 0, ds_h = 0, ds_w = 0;  // geometry of the last DS forward
  std::vector<int> ds_off;

  std::vector<std::unique_ptr<Plan>> plans;
  Plan* last_plan = nullptr;
  int gather_impl = 0;               // option "gather_impl": 0 = four pixels per thread when the shape allows, 1 = generic kernel
  int wide_tiles = 1;                // option "wide_tiles": streaming 3x3 kernel with column tiles up to 256 (two TMEM buffers above 160)
  int store_mode = 2;                // option "store_mode": EpiParams::store_mode of every tensor-core launch
  int use_graph = 1;                 // option "graph": replay the per-(n,h,w) launch sequence of a forward as one CUDA graph
  uint64_t graph_epoch = 1;          // bumped by everything a captured launch bakes in (options, weight re-packs)
  cudaStream_t cap_stream = nullptr; // capture happens on a private stream (the caller's may be the legacy default stream)
  int64_t graph_replays = 0;

  int conv_impl = 0;
  int seg_chunks = 0;                // pipeline stages per fp32-promotion segment; 0 = automatic
  int act_grad_impl = 0;             // 0: 16-byte activation-gradient kernel, 1: channel-pair kernel (cross-check)
  int timing = 0;
  int fuse_last = 1;                 // fold the per-pixel half of R-CNN1 into the last Up-PS epilogue
  std::vector<cudaEvent_t> ev;       // timing events (launch boundaries of the last forward)
  int ev_used = 0;
  int64_t launches = 0;
  PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
};

static int planes(const dcscn_handle* h) { return h->cfg.precision == DCSCN_PRECISION_F16X1 ? 1 : 2; }

// Filter-count schedule of the feature-extraction stack (DCSCN.py:240-244).
static std::vector<int> feature_filters(const dcscn_config& c) {
  std::vector<int> out;
  const int minf = std::min(c.filters, c.min_filters);  // DCSCN.py:37
  int n = c.filters;
  for (int i = 0; i < c.layers; ++i) {
    if (minf != 0 && i > 0) {
      double x1 = (double)i / (double)(c.layers - 1);
      double y1 = std::pow(x1, 1.0 / (double)c.filters_decay_gamma);
      n = (int)((c.filters - minf) * (1 - y1) + minf);
    }
    out.push_back(n);
  }
  return out;
}

static void add_param(dcscn_handle* h, const std::string& name, std::vector<int64_t> shape, float fill) {
  ParamDef p;
  p.name = name;
  p.shape = shape;
  p.host.assign((size_t)p.numel(), fill);
  h->param_index[name] = (int)h->params.size();
  h->params.push_back(std::move(p));
}

static int build_graph(dcscn_handle* h) {
  const dcscn_config& c = h->cfg;
  if (!c.use_nin) return fail("use_nin=false is not supported (no shipped checkpoint uses it)");
  if (c.channels != 1) return fail("channels must be 1 (helper/args.py: 'Now it should be 1')");
  if (std::max(c.reconstruct_layers, 1) != 1) return fail("reconstruct_layers > 1 is not supported");
  if (c.scale < 2 || c.scale > 4) return fail("scale must be 2, 3 or 4");
  if (c.cnn_size != 3 && c.cnn_size != 1 && c.cnn_size != 5) return fail("cnn_size %d is not supported", c.cnn_size);
  if (c.layers < 2) return fail("layers must be >= 2");

  h->filters = feature_filters(c);
  int cin = c.channels, total = 0;
  for (int i = 0; i < c.layers; ++i) {
    h->layers.push_back({"CNN" + std::to_string(i + 1), c.cnn_size, cin, h->filters[i], true, true});
    cin = h->filters[i];
    total += cin;
  }
  h->layers.push_back({"A1", 1, total, c.nin_filters, true, true});
  h->layers.push_back({"B1", 1, total, c.nin_filters2, true, true});
  h->layers.push_back({"B2", 3, c.nin_filters2, c.nin_filters2, true, true});
  cin = c.nin_filters + c.nin_filters2;
  h->ps_out = c.pixel_shuffler_filters != 0 ? c.pixel_shuffler_filters : cin;
  if (c.scale == 4) {  // DCSCN.py:298-304
    h->layers.push_back({"Up-PS/Up-PS_CNN", c.cnn_size, cin, 4 * cin, true, false});
    h->layers.push_back({"Up-PS2/Up-PS2_CNN", c.cnn_size, cin, 4 * h->ps_out, true, false});
  } else {
    h->layers.push_back({"Up-PS/Up-PS_CNN", c.cnn_size, cin, c.scale * c.scale * h->ps_out, true, false});
  }
  h->layers.push_back({"R-CNN1", c.cnn_size, h->ps_out, 1, false, false});

  for (const LayerDef& l : h->layers) {
    std::string base = l.scope.substr(l.scope.find_last_of('/') == std::string::npos ? 0 : l.scope.find_last_of('/') + 1);
    add_param(h, l.scope + "/conv_W", {l.k, l.k, l.cin, l.cout}, 0.f);
    if (c.depthwise_separable) {  // tf_graph.py:157-160; conv_W stays as the (dead) variable the reference also creates
      add_param(h, l.scope + "/depthwise_W", {l.k, l.k, l.cin, 1}, 0.f);
      add_param(h, l.scope + "/pointwise_W", {1, 1, l.cin, l.cout}, 0.f);
    }
    if (l.bias) add_param(h, l.scope + "/conv_B", {l.cout}, 0.f);                 // util.bias: zeros
    if (l.prelu) add_param(h, l.scope + "/prelu/" + base + "_prelu", {l.cout}, 0.1f);  // tf_graph.py:91
  }

  // channel layout of the shared feature ("concat") buffer: 16-aligned slot per CNN layer
  int off = 0;
  for (int f : h->filters) {
    h->feat_off.push_back(off);
    h->feat_w.push_back(pad16(f));
    off += pad16(f);
  }
  h->feat_pitch = off;
  h->b1_w = pad16(c.nin_filters2);
  h->a1_w = pad16(c.nin_filters);
  h->nin_pitch = h->b1_w + h->a1_w;  // [B2 | A1]  (Concat2 order, DCSCN.py:281)
  h->mid_pitch = pad16(cin);
  return 0;
}

static const LayerDef* find_layer(const dcscn_handle* h, const std::string& scope) {
  for (const LayerDef& l : h->layers)
    if (l.scope == scope) return &l;
  return nullptr;
}
static const std::vector<float>& P(const dcscn_handle* h, const std::string& name) {
  const ParamDef& p = h->params[h->param_index.at(name)];
  return h->shadow_mode ? p.shadow : p.host;
}

// ------------------------------------------------------------------------------ weight packing ----
// Device copies of host vectors.  Re-uploading the same number of bytes reuses the allocation, so cached launch
// plans (which embed these pointers) stay valid across weight updates; `g_upload_realloc` records when that failed.
static std::map<void*, size_t> g_upload_bytes;
static bool g_upload_realloc = false;

static void dev_free(void* p) {
  if (!p) return;
  g_upload_bytes.erase(p);
  cudaFree(p);
}

template <typename T>
static int upload(T** dptr, const std::vector<T>& host, dcscn_handle* h) {
  (void)h;
  const size_t bytes = host.size() * sizeof(T);
  if (*dptr) {
    auto it = g_upload_bytes.find((void*)*dptr);
    if (it != g_upload_bytes.end() && it->second == bytes && bytes > 0) {
      CUDA_TRY(cudaMemcpy(*dptr, host.data(), bytes, cudaMemcpyHostToDevice));
      return 0;
    }
    dev_free(*dptr);
    *dptr = nullptr;
    g_upload_realloc = true;
  }
  if (host.empty()) return 0;
  CUDA_TRY(cudaMalloc((void**)dptr, bytes));
  g_upload_bytes[(void*)*dptr] = bytes;
  g_upload_realloc = true;
  CUDA_TRY(cudaMemcpy(*dptr, host.data(), bytes, cudaMemcpyHostToDevice));
  return 0;
}

// Appends the TF layer `scope` as columns [col0, col0+cout) of a fused tensor-core layer.
static void fuse_columns(const dcscn_handle* h, TcLayer& t, const std::string& scope, int col0, int n_total_pad) {
  const LayerDef* l = find_layer(h, scope);
  const std::vector<float>& W = P(h, scope + "/conv_W");
  const int taps = l->k * l->k;
  for (int tp = 0; tp < taps; ++tp)
    for (int ci = 0; ci < l->cin; ++ci)
      for (int co = 0; co < l->cout; ++co)
        t.w_host[((size_t)tp * t.cin + ci) * t.cout + col0 + co] = W[((size_t)tp * l->cin + ci) * l->cout + co];
  std::string base = scope.substr(scope.find_last_of('/') == std::string::npos ? 0 : scope.find_last_of('/') + 1);
  (void)n_total_pad;
  if (l->bias) {
    const std::vector<float>& B = P(h, scope + "/conv_B");
    for (int co = 0; co < l->cout; ++co) t.bias_host[col0 + co] = B[co];
  }
  if (l->prelu) {
    const std::vector<float>& A = P(h, scope + "/prelu/" + base + "_prelu");
    for (int co = 0; co < l->cout; ++co) t.alpha_host[col0 + co] = A[co];
  }
}

static void choose_tiling(int n_total_pad16, int* n_tiles, int* n_pad, int cap = 256) {
  int nt = (n_total_pad16 + cap - 1) / cap;
  int np = pad16((n_total_pad16 + nt - 1) / nt);
  *n_tiles = nt;
  *n_pad = np;
}

// Column-tile cap of a layer.  The streaming 3x3 kernel rotates TMEM buffers of n_pad columns: 160 keeps three of them
// (3 * n_pad <= 512).  Option "wide_tiles" lifts it to 256: layers wider than 160 columns then run with TWO buffers (the
// issuer waits for a drain at every segment end) but read every A box once per pixel tile instead of once per column
// tile - CNN2 is one tile of 176 columns instead of 2 x 96, Up-PS 2 x 192 instead of 4 x 96.
static int tile_cap(const dcscn_handle* h, int ksz) { return ksz == 3 ? (h->wide_tiles ? 256 : 160) : 256; }

// Experiments: DCSCN_SEG="CNN2=1,A1=6" overrides the fp32-promotion period of single layers.
static int seg_override(const std::string& name, int seg) {
  if (const char* ov = getenv("DCSCN_SEG")) {
    const std::string key = name + "=";
    const char* hit = strstr(ov, key.c_str());
    if (hit && (hit == ov || hit[-1] == ',')) seg = atoi(hit + key.size());
  }
  return std::max(1, seg);
}

// fp32-promotion segments of one item of the streaming 3x3 kernel: a segment ends after `seg_units` (chunk, dx) units of
// 12 dominant UMMAs (3 taps x 4 slices), or with the last unit - the rule of the kernel's seg_end.
static int h2_segments(int cin_pad, int seg_units) {
  const int units = 3 * ((cin_pad + 63) / 64);
  return (units + seg_units - 1) / seg_units;
}

// Values (unscaled fp32) of the CTA-pair operand image of a layer, one per hi-plane element, in image order:
// [n_tile][block][rank][n_pad/2 rows x 64 halves], each row 128-byte swizzled (16-byte chunk j of row r at j ^ (r & 7)).
// A block holds one filter tap of one 64-channel chunk.  Blocks are in [tap][chunk] order for conv_tc_pair_kernel, and in
// the streaming kernel's stage order [chunk][dx][dy] when t.h2 is set.
static void pair_image(const TcLayer& t, std::vector<float>& img) {
  const int taps = t.ksz * t.ksz, chunks = (t.cin_pad + 63) / 64, n_total = t.n_tiles * t.n_pad;
  std::vector<float> wq((size_t)taps * t.cin_pad * n_total, 0.f);   // dense, channel-position-indexed  Wq[tap][q][n]
  for (int tp = 0; tp < taps; ++tp)
    for (int ci = 0; ci < t.cin; ++ci) {
      const int q = t.in_map[ci];
      for (int co = 0; co < t.cout; ++co)
        wq[((size_t)tp * t.cin_pad + q) * n_total + co] = t.w_host[((size_t)tp * t.cin + ci) * t.cout + co];
    }
  const int half_rows = t.n_pad / 2;
  const size_t half_elems = (size_t)half_rows * 64;
  img.assign((size_t)t.n_tiles * taps * chunks * 2 * half_elems, 0.f);
  for (int nt = 0; nt < t.n_tiles; ++nt)
    for (int tp = 0; tp < taps; ++tp)
      for (int ch = 0; ch < chunks; ++ch) {
        // HWIO tap tp = dy * 3 + dx is stage dx * 3 + dy of its chunk in the streaming order
        const int blk = t.h2 ? ch * 9 + (tp % 3) * 3 + tp / 3 : tp * chunks + ch;
        for (int rk = 0; rk < 2; ++rk) {
          float* base = img.data() + (((size_t)nt * taps * chunks + blk) * 2 + rk) * half_elems;
          for (int r = 0; r < half_rows; ++r) {
            const int n = nt * t.n_pad + rk * half_rows + r;
            const int sw = r & 7;
            for (int kk = 0; kk < 64; ++kk) {
              const int q = ch * 64 + kk;
              if (q < t.cin_pad) base[(size_t)r * 64 + (size_t)((kk / 8) ^ sw) * 8 + (kk % 8)] = wq[((size_t)tp * t.cin_pad + q) * n_total + n];
            }
          }
        }
      }
}

static int pack_tc_layer(dcscn_handle* h, TcLayer& t) {
  const int NPL = planes(h);

  float maxw = 0.f;
  for (float v : t.w_host) maxw = std::max(maxw, std::fabs(v));
  t.wscale = 1.f;
  if (maxw > 0.f) t.wscale = std::ldexp(1.0f, (int)std::floor(std::log2(16384.0 / (double)maxw)));

  t.h2 = t.ksz == 3 && (h->wide_tiles ? 2 : 3) * t.n_pad <= 512;   // streaming kernel: stage-ordered image
  t.h2_nseg = 0;
  if (t.h2) {
    // Promotion period in (chunk, dx) units of K = 192.  Measured (gpurun_out/seg15.log): with three TMEM buffers
    // (n_pad >= 144) a period of 1 leaves the epilogue one segment (~1.5 us) to drain a slot and the issuer stalls -
    // CNN3 0.85 -> 0.63 ms, CNN4 0.74 -> 0.52 ms at 4; the noise-tile error is flat in this range (1.2-1.35e-3).
    // Two-buffer tiles (3 * n_pad > 512, option "wide_tiles") stall the issuer at every segment end, so the longer period
    // pays twice there: CNN2 as one 176-column tile 0.93 -> 0.88 ms at 4 units, noise-tile error unchanged (1.27 -> 1.28e-3).
    const int seg = seg_override(t.name, h->seg_chunks > 0 ? h->seg_chunks : (t.n_pad >= 144 ? 4 : 3));
    t.h2_seg_units = seg;
    t.h2_nseg = h2_segments(t.cin_pad, seg);
  }
  const int half_rows = t.n_pad / 2;
  const size_t half_elems = (size_t)half_rows * 64;
  std::vector<float> img;
  pair_image(t, img);
  std::vector<__half> pp(img.size() * NPL);
  for (size_t i = 0; i < img.size(); ++i) {
    const size_t blk = i / half_elems, pos = i - blk * half_elems;
    const float v = img[i] * t.wscale;
    const __half hi = __float2half_rn(v);
    pp[blk * NPL * half_elems + pos] = hi;
    if (NPL == 2) pp[blk * NPL * half_elems + half_elems + pos] = __float2half_rn(v - __half2float(hi));
  }
  if (upload(&t.d_wpair, pp, h)) return 1;
  const size_t total_rows = pp.size() / 64;
  cuuint64_t dims[2] = {64, (cuuint64_t)total_rows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, (cuuint32_t)(NPL * half_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = h->encode(&t.tm_w, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)t.d_wpair, dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled (weights, layer %s) failed: %d", t.name.c_str(), (int)r);
  if (upload(&t.d_bias, t.bias_host, h)) return 1;
  if (upload(&t.d_alpha, t.alpha_host, h)) return 1;
  if (upload(&t.d_wref, t.w_host, h)) return 1;
  if (upload(&t.d_in_map, t.in_map, h)) return 1;
  return 0;
}

static TcLayer make_tc(const dcscn_handle* h, const std::string& name, int ksz, int cin, int cout_cols, int cin_pad,
                       int tile_unit = 0) {
  const int cap = tile_cap(h, ksz);
  TcLayer t;
  t.name = name;
  t.ksz = ksz;
  t.cin = cin;
  t.cout = cout_cols;
  t.cin_pad = cin_pad;
  choose_tiling(pad16(cout_cols), &t.n_tiles, &t.n_pad, cap);
  if (tile_unit > 0 && cap < 256 && ksz == 3 && t.n_tiles > 1 && tile_unit % 16 == 0 && tile_unit <= cap && cout_cols % tile_unit == 0) {
    t.n_pad = tile_unit;               // pixel-shuffler layers: one column tile per sub-pixel (fused R-CNN1 epilogue)
    t.n_tiles = cout_cols / tile_unit;
  }
  t.n_valid = cout_cols;
  t.w_host.assign((size_t)ksz * ksz * cin * cout_cols, 0.f);
  t.bias_host.assign((size_t)t.n_tiles * t.n_pad, 0.f);
  t.alpha_host.assign((size_t)t.n_tiles * t.n_pad, 1.f);
  return t;
}

static void free_tc(TcLayer& t) {
  dev_free(t.d_wpair);
  dev_free(t.d_bias);
  dev_free(t.d_alpha);
  dev_free(t.d_wref);
  dev_free(t.d_in_map);
  dev_free(t.d_pair_src);
  t.d_pair_src = nullptr;
  t.d_wpair = nullptr;
  t.d_bias = t.d_alpha = t.d_wref = nullptr;
  t.d_in_map = nullptr;
}

static void adopt_tc(TcLayer& t, const TcLayer& old) {  // keep the device allocations of the previous packing
  t.d_wpair = old.d_wpair; t.d_bias = old.d_bias; t.d_alpha = old.d_alpha;
  t.d_wref = old.d_wref; t.d_in_map = old.d_in_map; t.d_pair_src = old.d_pair_src;
}

// (Re)builds every device-side weight image from the host fp32 parameters.
static int finalize_params_ds(dcscn_handle* h) {
  for (auto& d : h->ds) {
    cudaFree(d.dw); cudaFree(d.pw); cudaFree(d.bias); cudaFree(d.alpha);
  }
  cudaFree(h->ds_ab.pw); cudaFree(h->ds_ab.bias); cudaFree(h->ds_ab.alpha);
  h->ds_ab = dcscn_handle::DsDev();
  h->ds.assign(h->layers.size(), dcscn_handle::DsDev());
  // concat buffer: every CNNi slot starts on a multiple of 4 channels (16-byte loads / stores); the pad channels are never
  // written (the buffer is zero-filled once) and meet zero rows in the A1 / B1 filters
  h->ds_off.clear();
  int off = 0;
  for (int f : h->filters) {
    h->ds_off.push_back(off);
    off += (f + 3) & ~3;
  }
  h->ds_total = off;
  const int T = h->ds_total, L = h->cfg.layers;
  std::vector<float> ab_pw, ab_bias, ab_alpha;
  const int na = h->cfg.nin_filters, nb = h->cfg.nin_filters2;
  ab_pw.assign((size_t)T * (na + nb), 0.f);
  ab_bias.assign(na + nb, 0.f);
  ab_alpha.assign(na + nb, 1.f);
  for (size_t i = 0; i < h->layers.size(); ++i) {
    const LayerDef& l = h->layers[i];
    std::string base = l.scope.substr(l.scope.find_last_of('/') == std::string::npos ? 0 : l.scope.find_last_of('/') + 1);
    const std::vector<float>& dwv = P(h, l.scope + "/depthwise_W");   // [k,k,cin,1] == [taps][cin]
    const std::vector<float>& pwv = P(h, l.scope + "/pointwise_W");   // [1,1,cin,cout] == [cin][cout]
    if (l.scope == "A1" || l.scope == "B1") {
      // these read the whole concat buffer: spread their rows over the 4-aligned slot positions
      std::vector<float> dwp((size_t)l.k * l.k * T, 0.f), pwp((size_t)T * l.cout, 0.f);
      const int col0 = l.scope == "A1" ? 0 : na;
      int ci = 0;
      for (int li = 0; li < L; ++li)
        for (int k = 0; k < h->filters[li]; ++k, ++ci) {
          const int pos = h->ds_off[li] + k;
          for (int t = 0; t < l.k * l.k; ++t) dwp[(size_t)t * T + pos] = dwv[(size_t)t * l.cin + ci];
          for (int co = 0; co < l.cout; ++co) {
            pwp[(size_t)pos * l.cout + co] = pwv[(size_t)ci * l.cout + co];
            if (l.k == 1) ab_pw[(size_t)pos * (na + nb) + col0 + co] = dwv[ci] * pwv[(size_t)ci * l.cout + co];
          }
        }
      const auto& B = P(h, l.scope + "/conv_B");
      const auto& A = P(h, l.scope + "/prelu/" + base + "_prelu");
      for (int co = 0; co < l.cout; ++co) {
        ab_bias[col0 + co] = B[co];
        ab_alpha[col0 + co] = A[co];
      }
      if (upload(&h->ds[i].dw, dwp, h) || upload(&h->ds[i].pw, pwp, h)) return 1;
    } else {
      if (upload(&h->ds[i].dw, dwv, h) || upload(&h->ds[i].pw, pwv, h)) return 1;
    }
    if (l.bias && upload(&h->ds[i].bias, P(h, l.scope + "/conv_B"), h)) return 1;
    if (l.prelu && upload(&h->ds[i].alpha, P(h, l.scope + "/prelu/" + base + "_prelu"), h)) return 1;
  }
  if (upload(&h->ds_ab.pw, ab_pw, h) || upload(&h->ds_ab.bias, ab_bias, h) || upload(&h->ds_ab.alpha, ab_alpha, h)) return 1;
  h->params_dirty = false;
  return 0;
}

static int build_bwd_layers(dcscn_handle* h);
static int sync_host_params(dcscn_handle* h);   // train_engine.inc: device master copy -> host, when newer

// CNN1's device vectors (CUDA cores): filter [taps][n_pad], bias, PReLU slope, padded to the slot width.
static void first_layer_vectors(const dcscn_handle* h, std::vector<float>& w, std::vector<float>& b, std::vector<float>& a) {
  const LayerDef* l = find_layer(h, "CNN1");
  const int taps = l->k * l->k, np = h->feat_w[0];
  w.assign((size_t)taps * np, 0.f);
  b.assign(np, 0.f);
  a.assign(np, 1.f);
  const auto& W = P(h, "CNN1/conv_W");
  for (int tp = 0; tp < taps; ++tp)
    for (int co = 0; co < l->cout; ++co) w[(size_t)tp * np + co] = W[(size_t)tp * l->cout + co];
  const auto& B = P(h, "CNN1/conv_B");
  const auto& A = P(h, "CNN1/prelu/CNN1_prelu");
  for (int co = 0; co < l->cout; ++co) {
    b[co] = B[co];
    a[co] = A[co];
  }
}

// Fills h->tcl (forward tensor-core layers) and, when training, h->bwd (their dgrad twins) from the parameters P().
static int construct_tc_layers(dcscn_handle* h) {
  const dcscn_config& c = h->cfg;
  const int L = c.layers;
  // CNN2..CNNL
  for (int i = 1; i < L; ++i) {
    const std::string scope = "CNN" + std::to_string(i + 1);
    const LayerDef* l = find_layer(h, scope);
    TcLayer t = make_tc(h, scope, l->k, l->cin, l->cout, h->feat_w[i - 1]);
    for (int ci = 0; ci < l->cin; ++ci) t.in_map.push_back(ci);
    fuse_columns(h, t, scope, 0, 0);
    h->tcl.push_back(std::move(t));
  }
  // A1 || B1 fused 1x1 over the whole concat buffer: columns [A1 (padded to 16) | B1]
  {
    const LayerDef* a1 = find_layer(h, "A1");
    const LayerDef* b1 = find_layer(h, "B1");
    TcLayer t = make_tc(h, "A1+B1", 1, a1->cin, h->a1_w + b1->cout, h->feat_pitch);
    for (int li = 0; li < L; ++li)
      for (int ci = 0; ci < h->filters[li]; ++ci) t.in_map.push_back(h->feat_off[li] + ci);
    fuse_columns(h, t, "A1", 0, 0);
    fuse_columns(h, t, "B1", h->a1_w, 0);
    h->tcl.push_back(std::move(t));
  }
  // B2
  {
    const LayerDef* l = find_layer(h, "B2");
    TcLayer t = make_tc(h, "B2", l->k, l->cin, l->cout, h->b1_w);
    for (int ci = 0; ci < l->cin; ++ci) t.in_map.push_back(ci);
    fuse_columns(h, t, "B2", 0, 0);
    h->tcl.push_back(std::move(t));
  }
  // Up-PS (+ Up-PS2): input = Concat2 = [B2 | A1]
  {
    const LayerDef* l = find_layer(h, "Up-PS/Up-PS_CNN");
    // the LAST depth_to_space layer carries the fused R-CNN1 epilogue: one column tile per sub-pixel
    TcLayer t = make_tc(h, "Up-PS", l->k, l->cin, l->cout, h->nin_pitch, c.scale == 4 ? 0 : h->ps_out);
    for (int ci = 0; ci < c.nin_filters2; ++ci) t.in_map.push_back(ci);
    for (int ci = 0; ci < c.nin_filters; ++ci) t.in_map.push_back(h->b1_w + ci);
    fuse_columns(h, t, "Up-PS/Up-PS_CNN", 0, 0);
    h->tcl.push_back(std::move(t));
    if (c.scale == 4) {
      const LayerDef* l2 = find_layer(h, "Up-PS2/Up-PS2_CNN");
      TcLayer t2 = make_tc(h, "Up-PS2", l2->k, l2->cin, l2->cout, h->mid_pitch, h->ps_out);
      for (int ci = 0; ci < l2->cin; ++ci) t2.in_map.push_back(ci);
      fuse_columns(h, t2, "Up-PS2/Up-PS2_CNN", 0, 0);
      h->tcl.push_back(std::move(t2));
    }
  }
  if (h->train_enabled && build_bwd_layers(h)) return 1;
  return 0;
}

static int finalize_params(dcscn_handle* h) {
  const dcscn_config& c = h->cfg;
  if (sync_host_params(h)) return 1;
  if (c.depthwise_separable) return finalize_params_ds(h);
  std::vector<TcLayer> old_tcl = std::move(h->tcl);
  std::vector<TcLayer> old_bwd = std::move(h->bwd);
  h->tcl.clear();
  h->bwd.clear();
  h->refresh_ready = false;
  g_upload_realloc = false;
  {
    std::vector<float> w, b, a;
    first_layer_vectors(h, w, b, a);
    if (upload(&h->d_first_w, w, h) || upload(&h->d_first_bias, b, h) || upload(&h->d_first_alpha, a, h)) return 1;
  }
  if (construct_tc_layers(h)) return 1;
  for (size_t i = 0; i < h->tcl.size(); ++i) {
    if (i < old_tcl.size()) adopt_tc(h->tcl[i], old_tcl[i]);
    if (pack_tc_layer(h, h->tcl[i])) return 1;
  }
  for (size_t i = h->tcl.size(); i < old_tcl.size(); ++i) free_tc(old_tcl[i]);
  for (size_t i = 0; i < h->bwd.size(); ++i) {
    if (i < old_bwd.size()) adopt_tc(h->bwd[i], old_bwd[i]);
    if (pack_tc_layer(h, h->bwd[i])) return 1;
  }
  for (size_t i = h->bwd.size(); i < old_bwd.size(); ++i) free_tc(old_bwd[i]);
  // R-CNN1 (CUDA cores): [taps][C]
  {
    const LayerDef* l = find_layer(h, "R-CNN1");
    const auto& W = P(h, "R-CNN1/conv_W");  // [k,k,C,1]
    std::vector<float> w(W.begin(), W.end());
    (void)l;
    if (upload(&h->d_last_w, w, h)) return 1;
  }
  if (g_upload_realloc) {  // some device pointer moved: cached plans embed stale pointers
    h->plans.clear();
    h->last_plan = nullptr;
  }
  h->graph_epoch++;          // captured launches bake the epilogue's 1 / weight-scale
  h->params_dirty = false;
  return 0;
}

// Partial plane sets of the fused R-CNN1 epilogue: an epilogue thread owns n_pad / kColSplit GEMM columns; when that share
// is a fraction of one sub-pixel's `cout` channels, `cout / share` threads each write their own tap-planar partials.
static int rdot_parts(int n_pad, int cout) {
  const int nch = n_pad >> 4, per16 = ((nch + kColSplit - 1) / kColSplit) * 16;
  if (cout <= 0 || per16 % cout == 0) return 1;
  return (cout % per16 == 0) ? cout / per16 : 1;
}

// ----------------------------------------------------------------------------------- workspace ----
template <typename T>
static int dev_alloc(dcscn_handle* h, T** p, size_t count, bool zero) {
  if (*p) {
    cudaFree(*p);
    *p = nullptr;
  }
  if (count == 0) return 0;
  CUDA_TRY(cudaMalloc((void**)p, count * sizeof(T)));
  if (zero) CUDA_TRY(cudaMemset(*p, 0, count * sizeof(T)));
  h->device_bytes += (int64_t)(count * sizeof(T));
  return 0;
}

static int ensure_workspace(dcscn_handle* h, size_t lr_px) {
  if (lr_px <= h->cap_px) return 0;
  const dcscn_config& c = h->cfg;
  if (c.depthwise_separable) {
    h->device_bytes = 0;
    const size_t s2 = (size_t)c.scale * c.scale;
    const int cps = c.nin_filters + c.nin_filters2;
    if (dev_alloc(h, &h->ds_feat, lr_px * h->ds_total, true)) return 1;   // pad channels must stay zero
    if (dev_alloc(h, &h->ds_b1, lr_px * c.nin_filters2, false)) return 1;
    if (dev_alloc(h, &h->ds_nin, lr_px * cps, false)) return 1;
    if (c.scale == 4 && dev_alloc(h, &h->ds_mid, lr_px * 4 * cps, false)) return 1;
    if (dev_alloc(h, &h->ds_hr, lr_px * s2 * h->ps_out, false)) return 1;
    h->cap_px = lr_px;
    return 0;
  }
  h->plans.clear();
  h->last_plan = nullptr;
  h->device_bytes = 0;
  const bool two = planes(h) == 2;
  const size_t s2 = (size_t)c.scale * c.scale;
  if (dev_alloc(h, &h->feat_hi, lr_px * h->feat_pitch, true)) return 1;
  if (dev_alloc(h, &h->feat_lo, two ? lr_px * h->feat_pitch : 0, true)) return 1;
  if (dev_alloc(h, &h->b1_hi, lr_px * h->b1_w, true)) return 1;
  if (dev_alloc(h, &h->b1_lo, two ? lr_px * h->b1_w : 0, true)) return 1;
  if (dev_alloc(h, &h->nin_hi, lr_px * h->nin_pitch, true)) return 1;
  if (dev_alloc(h, &h->nin_lo, two ? lr_px * h->nin_pitch : 0, true)) return 1;
  if (c.scale == 4) {
    if (dev_alloc(h, &h->mid_hi, lr_px * 4 * h->mid_pitch, true)) return 1;
    if (dev_alloc(h, &h->mid_lo, two ? lr_px * 4 * h->mid_pitch : 0, true)) return 1;
  }
  if (dev_alloc(h, &h->hr, lr_px * s2 * h->ps_out, true)) return 1;
  if (dev_alloc(h, &h->vbuf, lr_px * s2 * 9 * (size_t)rdot_parts(h->tcl.empty() ? 16 : h->tcl.back().n_pad, h->ps_out), true)) return 1;
  h->cap_px = lr_px;
  return 0;
}

// --------------------------------------------------------------------------------------- plans ----
static void choose_patch(int H, int W, int* TH, int* TW) {
  // 128-pixel rectangular patches; minimise padded area, prefer wide patches (contiguous TMA rows)
  static const int cand[][2] = {{8, 16}, {4, 32}, {16, 8}, {2, 64}, {32, 4}, {1, 128}, {64, 2}, {128, 1}};
  long long best = -1;
  for (auto& c : cand) {
    const int th = c[0], tw = c[1];
    long long area = (long long)((H + th - 1) / th) * th * ((W + tw - 1) / tw) * tw;
    if (best < 0 || area < best) {
      best = area;
      *TH = th;
      *TW = tw;
    }
  }
}

static int encode_map(dcscn_handle* h, CUtensorMap* tm, const __half* base, int cin_pad, int pitch, int n, int H,
                      int W, int TH, int TW) {
  cuuint64_t dims[4] = {(cuuint64_t)cin_pad, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)pitch * 2, (cuuint64_t)W * pitch * 2, (cuuint64_t)H * W * pitch * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)TW, (cuuint32_t)TH, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = h->encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)base, dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail("cuTensorMapEncodeTiled failed (%d) cin_pad=%d pitch=%d n=%d H=%d W=%d box=%dx%d", (int)r, cin_pad,
                pitch, n, H, W, TH, TW);
  return 0;
}

static int add_tc_launch(dcscn_handle* h, Plan* pl, const TcLayer& t, const __half* src_hi, const __half* src_lo,
                         int src_pitch, int n, int H, int W, const EpiParams& epi) {
  TcLaunch L;
  memset(&L, 0, sizeof(L));
  int TH, TW;
  choose_patch(H, W, &TH, &TW);
  ConvGeom g{n, H, W, (W + TW - 1) / TW, (H + TH - 1) / TH, TW, TH};
  if (encode_map(h, &L.tm_hi, src_hi, t.cin_pad, src_pitch, n, H, W, TH, TW)) return 1;
  if (planes(h) == 2) {
    if (encode_map(h, &L.tm_lo, src_lo, t.cin_pad, src_pitch, n, H, W, TH, TW)) return 1;
  } else {
    L.tm_lo = L.tm_hi;
  }
  L.p.g = g;
  L.p.ksz = t.ksz;
  L.p.cin_pad = t.cin_pad;
  L.p.chunks = (t.cin_pad + 63) / 64;
  L.p.n_tiles = t.n_tiles;
  L.p.n_pad = t.n_pad;
  L.p.seg_chunks = h->seg_chunks;  // finalised per kernel at launch
  L.p.epi = epi;
  L.p.epi.bias = t.d_bias;
  L.p.epi.alpha = t.d_alpha;
  L.p.epi.out_scale = 1.0f / t.wscale;   // refreshed at every launch (launch_tc): a re-pack may pick another scale
  if (!h->tcl.empty() && &t >= h->tcl.data() && &t < h->tcl.data() + h->tcl.size()) {
    L.layer_index = (int)(&t - h->tcl.data());
    L.layer_bwd = false;
  } else if (!h->bwd.empty() && &t >= h->bwd.data() && &t < h->bwd.data() + h->bwd.size()) {
    L.layer_index = (int)(&t - h->bwd.data());
    L.layer_bwd = true;
  }
  L.p.epi.n_valid = t.n_valid;
  L.p.epi.drop_ntotal = pad16(t.cout);   // keep-mask index stride = slot width, whatever the column tiling

  // CTA-pair launch shape
  const size_t budget = 227 * 1024 - 2048 - kRdotSmemBytes;
  const long long tiles = (long long)n * g.tiles_x * g.tiles_y;
  L.tm_w = t.tm_w;
  const size_t pstage = tc_pair_stage_bytes(planes(h), t.n_pad);
  L.pair_stages = (int)std::min<size_t>(kMaxStages, budget / pstage);
  if (L.pair_stages < 2) return fail("layer %s: pipeline stage of %zu bytes does not fit twice in shared memory", t.name.c_str(), pstage);
  L.pair_smem = L.pair_stages * pstage + 1024 + kPairBarBytes + kRdotSmemBytes;
  const long long pitems = ((tiles + 1) / 2) * t.n_tiles;
  L.pair_grid = (int)std::min<long long>(pitems, h->sm_count / 2) * 2;
  {
    int seg = h->seg_chunks > 0 ? h->seg_chunks : (t.n_pad >= 112 ? 2 : 3);
    L.pair_seg = std::max(1, std::min(seg, L.pair_stages - 1));   // a segment's stages stay resident until its 2nd pass
  }
  // 1x1 layers stream (split accumulators over four TMEM buffers): nothing is held, the promotion period is free
  L.pair_stream = t.ksz == 1 && planes(h) == 2 && t.n_pad <= kPairStreamStride;
  if (L.pair_stream) L.pair_seg = seg_override(t.name, h->seg_chunks > 0 ? h->seg_chunks : 4);

  // streaming halo kernel (3x3 layers, 16 x 8 pixel patches): every ring slot is prefetch depth; two, three (n_pad > 128)
  // or four TMEM accumulation buffers
  if (t.h2) {
    ConvGeom hg{n, H, W, (W + kHaloTW - 1) / kHaloTW, (H + kHaloTH - 1) / kHaloTH, kHaloTW, kHaloTH};
    L.hg = hg;
    const long long htiles = (long long)n * hg.tiles_x * hg.tiles_y;
    const long long hitems = ((htiles + 1) / 2) * t.n_tiles;
    L.halo_grid = (int)std::min<long long>(hitems, h->sm_count / 2) * 2;
    const size_t a_slot = tc_halo1_a_slot_bytes(planes(h)), b_stage = tc_halo_b_stage_bytes(planes(h), t.n_pad);
    const long long total = 227 * 1024 - (long long)tc_halo2_misc_bytes();
    const int nst = 9 * L.p.chunks;
    int na = 2;
    long long nb = (total - na * (long long)a_slot) / (long long)b_stage;
    bool resident = false;
    if (t.n_tiles == 1 && nst <= kH2MaxStages && (long long)nst * (long long)b_stage + 2 * (long long)a_slot <= total) {
      // thin layers: the whole weight image of this CTA half stays in shared memory, every other byte goes to A boxes
      resident = true;
      nb = nst;
      na = (int)std::min<long long>(4, (total - (long long)nst * (long long)b_stage) / (long long)a_slot);
    } else if ((total - 3 * (long long)a_slot) / (long long)b_stage >= 9) {   // a third A slot, still >= 9 weight stages
      na = 3;
      nb = (total - 3 * (long long)a_slot) / (long long)b_stage;
    }
    nb = std::min<long long>(nb, kH2MaxStages);
    if (nb >= 3 || resident) {
      L.halo2 = true;
      L.halo2_seg = t.h2_seg_units;
      L.halo2_na = na;
      L.halo2_nb = (int)nb;
      L.halo2_smem = na * a_slot + (size_t)nb * b_stage + tc_halo2_misc_bytes();
      L.p.h2_nstages = nst;
      L.p.h2_nseg = t.h2_nseg;
      L.p.h2_resident = resident ? 1 : 0;
      if (encode_map(h, &L.t1_hi, src_hi, t.cin_pad, src_pitch, n, H, W, kHaloTH + 2, kHalo1W)) return 1;
      if (planes(h) == 2) {
        if (encode_map(h, &L.t1_lo, src_lo, t.cin_pad, src_pitch, n, H, W, kHaloTH + 2, kHalo1W)) return 1;
      } else {
        L.t1_lo = L.t1_hi;
      }
    }
  }

  // validation twin
  L.ref.g = g;
  L.ref.ksz = t.ksz;
  L.ref.cin = t.cin;
  L.ref.cout = t.cout;
  L.ref.src_hi = src_hi;
  L.ref.src_lo = planes(h) == 2 ? src_lo : nullptr;
  L.ref.src_pitch = src_pitch;
  L.ref.in_map = t.d_in_map;
  L.ref.w = t.d_wref;
  L.ref.n_total_pad = t.n_tiles * t.n_pad;
  L.ref.epi = L.p.epi;
  L.ref.epi.out_scale = 1.0f;
  pl->tc.push_back(L);
  return 0;
}

static EpiParams epi_planes(__half* hi, __half* lo, int pitch, int col_begin, int col_end) {
  EpiParams e;
  memset(&e, 0, sizeof(e));
  e.mode = EPI_PLANES;
  e.num_seg = 1;
  e.seg[0] = {col_begin, col_end, hi, lo, pitch};
  e.keep_prob = 1.0f;
  e.out_scale = 1.0f;
  return e;
}

static Plan* get_plan(dcscn_handle* h, int n, int H, int W) {
  for (auto& p : h->plans)
    if (p->n == n && p->h == H && p->w == W) return p.get();
  const dcscn_config& c = h->cfg;
  std::unique_ptr<Plan> pl(new Plan());
  pl->n = n;
  pl->h = H;
  pl->w = W;
  const bool two = planes(h) == 2;
  auto lo = [&](__half* p, size_t off) -> __half* { return two ? p + off : nullptr; };

  // CNN1
  memset(&pl->first, 0, sizeof(pl->first));
  pl->first.g = ConvGeom{n, H, W, 1, 1, 1, 1};
  pl->first.ksz = find_layer(h, "CNN1")->k;
  pl->first.n_pad = h->feat_w[0];
  pl->first.w = h->d_first_w;
  pl->first.epi = epi_planes(h->feat_hi, lo(h->feat_lo, 0), h->feat_pitch, 0, h->feat_w[0]);
  pl->first.epi.bias = h->d_first_bias;
  pl->first.epi.alpha = h->d_first_alpha;
  pl->first.epi.n_valid = h->filters[0];

  size_t ti = 0;
  for (int i = 1; i < c.layers; ++i, ++ti) {
    EpiParams e = epi_planes(h->feat_hi + h->feat_off[i], lo(h->feat_lo, h->feat_off[i]), h->feat_pitch, 0, h->feat_w[i]);
    if (add_tc_launch(h, pl.get(), h->tcl[ti], h->feat_hi + h->feat_off[i - 1], lo(h->feat_lo, h->feat_off[i - 1]),
                      h->feat_pitch, n, H, W, e))
      return nullptr;
  }
  {  // A1+B1: columns [0,a1_w) -> nin[:, b1_w:], columns [a1_w, a1_w+b1_w) -> b1
    EpiParams e = epi_planes(h->nin_hi + h->b1_w, lo(h->nin_lo, h->b1_w), h->nin_pitch, 0, h->a1_w);
    e.num_seg = 2;
    e.seg[1] = {h->a1_w, h->a1_w + h->b1_w, h->b1_hi, two ? h->b1_lo : nullptr, h->b1_w};
    if (add_tc_launch(h, pl.get(), h->tcl[ti++], h->feat_hi, lo(h->feat_lo, 0), h->feat_pitch, n, H, W, e)) return nullptr;
  }
  {  // B2 -> nin[:, 0:b1_w]
    EpiParams e = epi_planes(h->nin_hi, lo(h->nin_lo, 0), h->nin_pitch, 0, h->b1_w);
    if (add_tc_launch(h, pl.get(), h->tcl[ti++], h->b1_hi, two ? h->b1_lo : nullptr, h->b1_w, n, H, W, e)) return nullptr;
  }
  int HR_H = H, HR_W = W;
  {  // Up-PS
    EpiParams e;
    memset(&e, 0, sizeof(e));
    e.keep_prob = 1.0f;
    if (c.scale == 4) {
      e.mode = EPI_D2S_PLANES;
      e.d2s_r = 2;
      e.d2s_cout = c.nin_filters + c.nin_filters2;
      e.num_seg = 1;
      e.seg[0] = {0, 0, h->mid_hi, two ? h->mid_lo : nullptr, h->mid_pitch};
    } else {
      e.mode = EPI_D2S_F32;
      e.d2s_r = c.scale;
      e.d2s_cout = h->ps_out;
      e.dst_f32 = h->hr;
      e.d2s_pitch = h->ps_out;
    }
    if (add_tc_launch(h, pl.get(), h->tcl[ti++], h->nin_hi, two ? h->nin_lo : nullptr, h->nin_pitch, n, H, W, e)) return nullptr;
    HR_H = H * (c.scale == 4 ? 2 : c.scale);
    HR_W = W * (c.scale == 4 ? 2 : c.scale);
  }
  if (c.scale == 4) {  // Up-PS2 at 2x resolution
    EpiParams e;
    memset(&e, 0, sizeof(e));
    e.keep_prob = 1.0f;
    e.mode = EPI_D2S_F32;
    e.d2s_r = 2;
    e.d2s_cout = h->ps_out;
    e.dst_f32 = h->hr;
    e.d2s_pitch = h->ps_out;
    if (add_tc_launch(h, pl.get(), h->tcl[ti++], h->mid_hi, two ? h->mid_lo : nullptr, h->mid_pitch, n, HR_H, HR_W, e))
      return nullptr;
    HR_H *= 2;
    HR_W *= 2;
  }
  {  // the last depth_to_space layer can carry the per-pixel half of R-CNN1 in its epilogue
    TcLaunch& L = pl->tc.back();
    const int cout = h->ps_out, nch = L.p.n_pad >> 4, per = (nch + kColSplit - 1) / kColSplit;
    const int klast = find_layer(h, "R-CNN1")->k;
    pl->unfused = L;
    pl->fused_index = (int)pl->tc.size() - 1;
    const int parts = rdot_parts(L.p.n_pad, cout);
    pl->fused_last = (klast == 3) && (cout % 16 == 0) && (cout <= 128) && (nch % kColSplit == 0) &&
                     (((per * 16) % cout == 0) || (parts > 1 && L.halo2 && L.p.n_pad % (per * 16) == 0));
    if (pl->fused_last) {
      L.p.epi.rdot_parts = ((per * 16) % cout == 0) ? 1 : parts;
      L.p.epi.mode = EPI_D2S_RDOT;
      L.p.epi.rdot_w = h->d_last_w;
      L.p.epi.rdot_out = h->vbuf;
      L.p.epi.rdot_taps = klast * klast;
    }
    const int gparts = pl->fused_last ? L.p.epi.rdot_parts : 1;
    memset(&pl->gather, 0, sizeof(pl->gather));
    pl->gather.parts = gparts;
    pl->gather.n_img = n;
    pl->gather.H = HR_H;
    pl->gather.W = HR_W;
    pl->gather.ksz = klast;
    pl->gather.v = h->vbuf;
  }
  memset(&pl->last, 0, sizeof(pl->last));
  pl->last.n_img = n;
  pl->last.H = HR_H;
  pl->last.W = HR_W;
  pl->last.ksz = find_layer(h, "R-CNN1")->k;
  pl->last.C = h->ps_out;
  pl->last.pitch = h->ps_out;
  pl->last.src = h->hr;
  pl->last.w = h->d_last_w;
  pl->last.bias = 0.f;
  if (h->plans.size() >= 64) h->plans.erase(h->plans.begin());
  h->plans.push_back(std::move(pl));
  return h->plans.back().get();
}

// ------------------------------------------------------------------------------------- forward ----
template <int NPL>
static int launch_tc_pair(dcscn_handle* h, const TcLaunch& L, cudaStream_t st) {
  static bool attr_set_dev[64] = {};   // function attributes are per device
  bool& attr_set = attr_set_dev[h->cfg.device_id & 63];
  if (!attr_set) {
    CUDA_TRY(cudaFuncSetAttribute(conv_tc_pair_kernel<NPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(L.pair_grid);
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = L.pair_smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ConvTCParams p = L.p;
  p.seg_chunks = L.pair_seg;
  p.pair_stream = L.pair_stream ? 1 : 0;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, conv_tc_pair_kernel<NPL>, L.tm_hi, L.tm_lo, L.tm_w, p, L.pair_stages));
  return 0;
}

#ifdef DCSCN_H2_DEBUG
static unsigned long long* g_h2_dbg = nullptr;
static int g_h2_dbg_launch = 0;
static std::string g_h2_dbg_names[64];
// Prints, per launch since the last dump: issuer cycles (total / waiting for A boxes / weight stages / free TMEM buffers)
// and epilogue cycles (total / waiting for full accumulators / bias-PReLU-store phase), averaged over clusters.
extern "C" int dcscn_h2_debug_dump(void) {
  if (!g_h2_dbg) return 0;
  cudaDeviceSynchronize();
  std::vector<unsigned long long> hbuf((size_t)8 * 128 * 64);
  cudaMemcpy(hbuf.data(), g_h2_dbg, hbuf.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
  for (int l = 0; l < std::min(g_h2_dbg_launch, 64); ++l) {
    double a[8] = {0};
    int n = 0;
    for (int c = 0; c < 128; ++c) {
      const unsigned long long* d = hbuf.data() + ((size_t)l * 128 + c) * 8;
      if (d[0] == 0) continue;
      for (int k = 0; k < 8; ++k) a[k] += (double)d[k];
      ++n;
    }
    if (!n) continue;
    for (int k = 0; k < 8; ++k) a[k] /= n;
    printf("%-70s clusters %3d | issuer total %9.0f  wait A %5.1f%%  wait W %5.1f%%  wait TMEM %5.1f%% | epilogue total %9.0f  wait acc %5.1f%%  store %5.1f%%\n",
           g_h2_dbg_names[l].c_str(), n, a[0], 100 * a[1] / a[0], 100 * a[2] / a[0], 100 * a[3] / a[0], a[4], 100 * a[5] / a[4], 100 * a[6] / a[4]);
  }
  cudaMemset(g_h2_dbg, 0, hbuf.size() * sizeof(unsigned long long));
  g_h2_dbg_launch = 0;
  fflush(stdout);
  return 0;
}
#endif

template <int NPL>
static int launch_tc_halo2(dcscn_handle* h, const TcLaunch& L, cudaStream_t st) {
  static bool attr_set_dev[64] = {};   // function attributes are per device
  bool& attr_set = attr_set_dev[h->cfg.device_id & 63];
  if (!attr_set) {
    CUDA_TRY(cudaFuncSetAttribute(conv_tc_halo2_kernel<NPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(L.halo_grid);
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = L.halo2_smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ConvTCParams p = L.p;
  p.g = L.hg;
  p.seg_chunks = L.halo2_seg;
#ifdef DCSCN_H2_DEBUG
  {  // diagnostic build: one counter block per launch, dumped by h2_debug_dump() (scripts/r2_h2_timeline.sh)
    static unsigned long long* d_dbg = nullptr;
    if (!d_dbg) {
      CUDA_TRY(cudaMalloc(&d_dbg, sizeof(unsigned long long) * 8 * 128 * 64));
      CUDA_TRY(cudaMemset(d_dbg, 0, sizeof(unsigned long long) * 8 * 128 * 64));
    }
    g_h2_dbg = d_dbg;
    p.dbg = d_dbg + (size_t)(g_h2_dbg_launch % 64) * 8 * 128;
    const std::string lname = L.layer_index >= 0 ? (L.layer_bwd ? h->bwd : h->tcl)[L.layer_index].name : std::string("?");
    g_h2_dbg_names[g_h2_dbg_launch % 64] = lname + (L.layer_bwd ? "(bwd)" : "") + " n_pad=" + std::to_string(L.p.n_pad) +
        " cin_pad=" + std::to_string(L.p.cin_pad) + " nst=" + std::to_string(L.p.h2_nstages) + " res=" + std::to_string(L.p.h2_resident) +
        " na=" + std::to_string(L.halo2_na) + " nb=" + std::to_string(L.halo2_nb) + " grid=" + std::to_string(L.halo_grid);
    ++g_h2_dbg_launch;
  }
#endif
  CUDA_TRY(cudaLaunchKernelEx(&cfg, conv_tc_halo2_kernel<NPL>, L.t1_hi, L.t1_lo, L.tm_w, p, L.halo2_na, L.halo2_nb));
  return 0;
}

static int launch_tc(dcscn_handle* h, const TcLaunch& Lc, cudaStream_t st) {
  h->launches++;
  // Cached plans outlive weight re-packs.  A re-pack keeps the device allocations (so the plan's pointers stay valid) but
  // may choose a different power-of-two weight scale: take the epilogue's 1 / scale from the layer as it is NOW.
  TcLaunch& L = const_cast<TcLaunch&>(Lc);
  if (L.layer_index >= 0) {
    const std::vector<TcLayer>& ls = L.layer_bwd ? h->bwd : h->tcl;
    if (L.layer_index < (int)ls.size()) L.p.epi.out_scale = 1.0f / ls[L.layer_index].wscale;
  }
  L.p.epi.store_mode = h->store_mode;
  if (h->conv_impl == 1) {
    const long long total = (long long)L.ref.g.n_img * L.ref.g.H * L.ref.g.W * (L.ref.n_total_pad >> 4);
    const int grid = (int)std::min<long long>((total + 127) / 128, (long long)h->sm_count * 16);
    conv_ref_kernel<<<grid, 128, 0, st>>>(L.ref);
    CUDA_TRY(cudaGetLastError());
    return 0;
  }
  const int npl = planes(h);
  if (L.halo2) return npl == 2 ? launch_tc_halo2<2>(h, L, st) : launch_tc_halo2<1>(h, L, st);
  if (L.p.ksz == 3) return fail("internal: 3x3 layer has no streaming launch shape");
  return npl == 2 ? launch_tc_pair<2>(h, L, st) : launch_tc_pair<1>(h, L, st);
}

static int mark(dcscn_handle* h, cudaStream_t st) {
  if (!h->timing) return 0;
  if (h->ev_used >= (int)h->ev.size()) {
    cudaEvent_t e;
    CUDA_TRY(cudaEventCreate(&e));
    h->ev.push_back(e);
  }
  CUDA_TRY(cudaEventRecord(h->ev[h->ev_used++], st));
  return 0;
}

static int mark(dcscn_handle* h, cudaStream_t st);
static int launch_ds(dcscn_handle* h, const LayerDef& l, const dcscn_handle::DsDev& d, const float* src, int src_pitch,
                     float* dst, int dst_pitch, int dst_off, int n, int H, int W, int d2s_r, int d2s_cout,
                     const float* add, cudaStream_t st) {
  DsLayerParams p;
  memset(&p, 0, sizeof(p));
  p.n_img = n; p.H = H; p.W = W; p.ksz = l.k; p.cin = l.cin; p.cout = l.cout;
  p.src = src; p.src_pitch = src_pitch; p.dw = d.dw; p.pw = d.pw; p.bias = d.bias; p.alpha = d.alpha;
  p.dst = dst; p.dst_pitch = dst_pitch; p.dst_off = dst_off; p.d2s_r = d2s_r; p.d2s_cout = d2s_cout; p.add = add;
  if (l.k != 1 && l.k != 3) return fail("depthwise-separable layer %s: kernel size %d is not supported (1 or 3)", l.scope.c_str(), l.k);
  const long long total = (long long)n * H * W;
  if (l.cin == 1 && l.cout == 1 && d2s_r == 0 && total < (1ll << 32)) {
    const int grid = (int)std::min<long long>((total + 255) / 256, (long long)h->sm_count * 16);
    if (l.k == 3) ds_single_kernel<3><<<grid, 256, 0, st>>>(p); else ds_single_kernel<1><<<grid, 256, 0, st>>>(p);
  } else {
    const size_t smem = ds_smem_bytes(l.k, l.cin, l.cout);
    if (smem > 200 * 1024) return fail("depthwise-separable layer %s: %d -> %d channels exceed the kernel's shared memory", l.scope.c_str(), l.cin, l.cout);
    static size_t ds_smem_attr_dev[64] = {};  // current opt-in limit of the DS kernels per device (only ever raised)
    size_t& ds_smem_attr = ds_smem_attr_dev[h->cfg.device_id & 63];
    if (ds_smem_attr == 0) ds_smem_attr = 48 * 1024;
    if (smem > ds_smem_attr) {   // raise the opt-in limit only as far as needed (keeps the L1 carve-out large)
      CUDA_TRY(cudaFuncSetAttribute(ds_layer_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      CUDA_TRY(cudaFuncSetAttribute(ds_layer_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      ds_smem_attr = smem;
    }
    const unsigned grid = (unsigned)((total + kDsPix - 1) / kDsPix);
    if (l.k == 3) ds_layer_kernel<3><<<grid, kDsThreads, smem, st>>>(p); else ds_layer_kernel<1><<<grid, kDsThreads, smem, st>>>(p);
  }
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return mark(h, st);
}

// ---- second-generation depthwise-separable kernels (conv_ds_tile.cuh) ----
template <int KSZ>
static int launch_ds_tile_k(dcscn_handle* h, const DsTileParams& p, unsigned grid, size_t smem, cudaStream_t st) {
  const int cols = p.cout < 32 ? ((p.cout + 3) & ~3) : 32;
  static size_t attr_dev[64][2] = {};
  size_t& cur = attr_dev[h->cfg.device_id & 63][KSZ == 3 ? 1 : 0];
  if (cur == 0) cur = 48 * 1024;
  if (smem > cur) {
    const int b = (int)smem;
    CUDA_TRY(cudaFuncSetAttribute(ds_tile_kernel<KSZ, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
    CUDA_TRY(cudaFuncSetAttribute(ds_tile_kernel<KSZ, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
    CUDA_TRY(cudaFuncSetAttribute(ds_tile_kernel<KSZ, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
    CUDA_TRY(cudaFuncSetAttribute(ds_tile_kernel<KSZ, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
    CUDA_TRY(cudaFuncSetAttribute(ds_tile_kernel<KSZ, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, b));
    cur = smem;
  }
  if (cols <= 4) ds_tile_kernel<KSZ, 1><<<grid, kDtThreads, smem, st>>>(p);
  else if (cols <= 8) ds_tile_kernel<KSZ, 2><<<grid, kDtThreads, smem, st>>>(p);
  else if (cols <= 16) ds_tile_kernel<KSZ, 4><<<grid, kDtThreads, smem, st>>>(p);
  else if (cols <= 24) ds_tile_kernel<KSZ, 6><<<grid, kDtThreads, smem, st>>>(p);
  else ds_tile_kernel<KSZ, 8><<<grid, kDtThreads, smem, st>>>(p);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

static int launch_ds_tile(dcscn_handle* h, DsTileParams p, int ksz, cudaStream_t st) {
  if (ksz != 1 && ksz != 3) return fail("depthwise-separable layer: kernel size %d is not supported (1 or 3)", ksz);
  if (p.cout > 32 && p.cin > kDtCC) return fail("depthwise-separable layer %d -> %d: more than 32 output columns need <= 32 input channels", p.cin, p.cout);
  const int cols = p.cout < 32 ? ((p.cout + 3) & ~3) : 32;
  // the kernel's shared-memory carve-up uses the per-pass column count of the instantiated template
  const int tcols = cols <= 4 ? 4 : cols <= 8 ? 8 : cols <= 16 ? 16 : cols <= 24 ? 24 : 32;
  const size_t in_px = ksz == 3 ? (size_t)(kDtT + 2) * kDtS : (size_t)kDtThreads;
  p.cache_u = (h->ds_cache && ds_tile_caches_depthwise(ksz, p.cin, p.cout)) ? 1 : 0;
  const size_t cache = p.cache_u ? (size_t)kDtThreads * kDtCP : 0;   // private depthwise rows
  const size_t smem = (in_px * kDtCP + (size_t)p.cin * tcols + (size_t)ksz * ksz * p.cin + cache) * sizeof(float);
  if (smem > 200 * 1024) return fail("depthwise-separable layer %d -> %d exceeds the kernel's shared memory", p.cin, p.cout);
  unsigned grid;
  if (ksz == 3) {
    p.tiles_x = (p.W + kDtT - 1) / kDtT;
    p.tiles_y = (p.H + kDtT - 1) / kDtT;
    grid = (unsigned)((long long)p.n_img * p.tiles_x * p.tiles_y);
  } else {
    grid = (unsigned)(((long long)p.n_img * p.H * p.W + kDtThreads - 1) / kDtThreads);
  }
  const int rc = ksz == 3 ? launch_ds_tile_k<3>(h, p, grid, smem, st) : launch_ds_tile_k<1>(h, p, grid, smem, st);
  if (rc) return rc;
  h->launches++;
  return mark(h, st);
}

static DsTileParams ds_tile_params(const LayerDef& l, const dcscn_handle::DsDev& d, const float* src, int src_pitch, float* dst,
                                   int dst_pitch, int dst_off, int n, int H, int W) {
  DsTileParams p;
  memset(&p, 0, sizeof(p));
  p.n_img = n; p.H = H; p.W = W; p.cin = l.cin; p.cout = l.cout;
  p.src = src; p.src_pitch = src_pitch; p.dw = d.dw; p.pw = d.pw; p.bias = d.bias; p.alpha = d.alpha;
  p.dst = dst; p.dst_pitch = dst_pitch; p.dst_off = dst_off;
  return p;
}

static int forward_ds_tile(dcscn_handle* h, const float* x, const float* x2, float* y, int n, int H, int W, cudaStream_t st) {
  const dcscn_config& c = h->cfg;
  const int L = c.layers, T = h->ds_total, na = c.nin_filters, nb = c.nin_filters2, cps = na + nb;
  h->ev_used = 0;
  if (mark(h, st)) return 1;
  size_t li = 0;
  for (int i = 0; i < L; ++i, ++li) {
    const float* src = i == 0 ? x : h->ds_feat + h->ds_off[i - 1];
    DsTileParams p = ds_tile_params(h->layers[li], h->ds[li], src, i == 0 ? c.channels : T, h->ds_feat, T, h->ds_off[i], n, H, W);
    if (launch_ds_tile(h, p, h->layers[li].k, st)) return 1;
  }
  {  // A1 | B1: both are 1x1 over the whole concat buffer -> ONE pass; the per-channel depthwise scales are folded into the
     // pointwise rows.  Columns [0, na) = A1 -> [B2 | A1] buffer at channel nb; columns [na, na+nb) = B1 -> B1 buffer.
    if (h->layers[li].k != 1 || h->layers[li + 1].k != 1) return fail("depthwise-separable A1 / B1 must be 1x1");
    LayerDef ab = h->layers[li];
    ab.k = 1; ab.cin = T; ab.cout = cps;
    DsTileParams p = ds_tile_params(ab, h->ds_ab, h->ds_feat, T, h->ds_nin, cps, nb, n, H, W);
    p.dw = nullptr;
    p.split = na;
    p.dst2 = h->ds_b1; p.dst2_pitch = nb; p.dst2_off = 0;
    if (cps > 32) return fail("depthwise-separable graph: nin_filters + nin_filters2 = %d > 32 is not supported by the fused A1|B1 kernel", cps);
    if (launch_ds_tile(h, p, 1, st)) return 1;
    li += 2;
  }
  {  // B2
    DsTileParams p = ds_tile_params(h->layers[li], h->ds[li], h->ds_b1, nb, h->ds_nin, cps, 0, n, H, W);
    if (launch_ds_tile(h, p, h->layers[li].k, st)) return 1;
    ++li;
  }
  int HH = H, WW = W;
  if (c.scale == 4) {
    DsTileParams p = ds_tile_params(h->layers[li], h->ds[li], h->ds_nin, cps, h->ds_mid, cps, 0, n, H, W);
    p.d2s_r = 2; p.d2s_cout = cps;
    if (launch_ds_tile(h, p, h->layers[li].k, st)) return 1;
    ++li;
    HH = 2 * H; WW = 2 * W;
    DsTileParams q = ds_tile_params(h->layers[li], h->ds[li], h->ds_mid, cps, h->ds_hr, h->ps_out, 0, n, HH, WW);
    q.d2s_r = 2; q.d2s_cout = h->ps_out;
    if (launch_ds_tile(h, q, h->layers[li].k, st)) return 1;
    ++li;
    HH *= 2; WW *= 2;
  } else {
    DsTileParams p = ds_tile_params(h->layers[li], h->ds[li], h->ds_nin, cps, h->ds_hr, h->ps_out, 0, n, H, W);
    p.d2s_r = c.scale; p.d2s_cout = h->ps_out;
    if (launch_ds_tile(h, p, h->layers[li].k, st)) return 1;
    ++li;
    HH = c.scale * H; WW = c.scale * W;
  }
  if (h->wait_x2) {
    CUDA_TRY(cudaStreamWaitEvent(st, h->x2_ready, 0));
    h->wait_x2 = false;
  }
  // R-CNN1 (no bias / activation) + x2
  const LayerDef& lr = h->layers[li];
  const dcscn_handle::DsDev& d = h->ds[li];
  const long long total = (long long)n * HH * WW;
  if (lr.cin == 1 && lr.cout == 1 && lr.k == 3 && (WW & 3) == 0 && total < (1ll << 32) &&
      ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(x2)) & 15) == 0) {
    const int grid = (int)std::min<long long>((total / 4 + 255) / 256, (long long)h->sm_count * 16);
    ds_single4_kernel<<<grid, 256, 0, st>>>(h->ds_hr, x2, y, n, HH, WW, d.dw, d.pw, d.bias, d.alpha);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return mark(h, st);
  }
  if (lr.cin == 1 && lr.cout == 1) return launch_ds(h, lr, d, h->ds_hr, h->ps_out, y, 1, 0, n, HH, WW, 0, 0, x2, st);
  DsTileParams p = ds_tile_params(lr, d, h->ds_hr, h->ps_out, y, 1, 0, n, HH, WW);
  p.add = x2;
  return launch_ds_tile(h, p, lr.k, st);
}

// Depthwise-separable graph (DCSCN.py:246-249, 264-271, 318-320; tf_graph.py:240-243): fp32 NHWC, CUDA cores.
static int forward_ds(dcscn_handle* h, const float* x, const float* x2, float* y, int n, int H, int W, cudaStream_t st) {
  if (h->ds_impl == 0) return forward_ds_tile(h, x, x2, y, n, H, W, st);
  const dcscn_config& c = h->cfg;
  const int L = c.layers, T = h->ds_total, cps = c.nin_filters + c.nin_filters2;
  h->ev_used = 0;
  if (mark(h, st)) return 1;
  size_t li = 0;
  for (int i = 0; i < L; ++i, ++li) {
    const float* src = i == 0 ? x : h->ds_feat + h->ds_off[i - 1];
    if (launch_ds(h, h->layers[li], h->ds[li], src, i == 0 ? c.channels : T, h->ds_feat, T, h->ds_off[i], n, H, W, 0, 0, nullptr, st)) return 1;
  }
  LayerDef la = h->layers[li], lb = h->layers[li + 1];
  la.cin = lb.cin = T;   // their filters are spread over the 4-aligned concat positions (finalize_params_ds)
  if (launch_ds(h, la, h->ds[li], h->ds_feat, T, h->ds_nin, cps, c.nin_filters2, n, H, W, 0, 0, nullptr, st)) return 1;  // A1
  ++li;
  if (launch_ds(h, lb, h->ds[li], h->ds_feat, T, h->ds_b1, c.nin_filters2, 0, n, H, W, 0, 0, nullptr, st)) return 1;     // B1
  ++li;
  if (launch_ds(h, h->layers[li], h->ds[li], h->ds_b1, c.nin_filters2, h->ds_nin, cps, 0, n, H, W, 0, 0, nullptr, st)) return 1;     // B2
  ++li;
  int HH = H, WW = W;
  if (c.scale == 4) {
    if (launch_ds(h, h->layers[li], h->ds[li], h->ds_nin, cps, h->ds_mid, cps, 0, n, H, W, 2, cps, nullptr, st)) return 1;           // Up-PS
    ++li;
    HH = 2 * H; WW = 2 * W;
    if (launch_ds(h, h->layers[li], h->ds[li], h->ds_mid, cps, h->ds_hr, h->ps_out, 0, n, HH, WW, 2, h->ps_out, nullptr, st)) return 1;  // Up-PS2
    ++li;
    HH *= 2; WW *= 2;
  } else {
    if (launch_ds(h, h->layers[li], h->ds[li], h->ds_nin, cps, h->ds_hr, h->ps_out, 0, n, H, W, c.scale, h->ps_out, nullptr, st)) return 1;
    ++li;
    HH = c.scale * H; WW = c.scale * W;
  }
  // R-CNN1 (no bias / activation) + x2
  if (h->wait_x2) {
    CUDA_TRY(cudaStreamWaitEvent(st, h->x2_ready, 0));
    h->wait_x2 = false;
  }
  if (launch_ds(h, h->layers[li], h->ds[li], h->ds_hr, h->ps_out, y, 1, 0, n, HH, WW, 0, 0, x2, st)) return 1;
  return 0;
}

// CNN1 and the tensor-core layers of one forward, in execution order, on `st` (a capturing stream when the plan's graph is
// being built).  The last kernel (R-CNN1 gather / R-CNN1) is issued by forward_impl: it alone touches x2 and y.
static int issue_front(dcscn_handle* h, Plan* pl, const float* x, int n, int H, int W, bool fused, cudaStream_t st) {
  {  // CNN1
    ConvFirstParams p = pl->first;
    p.x = x;
    if (p.ksz > 5) return fail("cnn_size %d is not supported by the first-layer kernel", p.ksz);
    const long long total = (long long)n * H * W;
    const int grid = (int)std::min<long long>((total + 255) / 256, (long long)h->sm_count * 8);
    const size_t smem = (size_t)p.ksz * p.ksz * p.n_pad * sizeof(float);
    if (p.ksz == 3 && p.n_pad <= 256) {
      const int first_grid = (int)std::min<long long>((total + 7) / 8, (long long)h->sm_count * 8);
      if (p.epi.seg[0].dst_zneg != nullptr) conv_first3x3_kernel<true><<<first_grid, 256, 0, st>>>(p);
      else conv_first3x3_kernel<false><<<first_grid, 256, 0, st>>>(p);
    } else {
      conv_first_kernel<<<grid, 256, smem, st>>>(p);
    }
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    if (mark(h, st)) return 1;
  }
  for (size_t i = 0; i < pl->tc.size(); ++i) {
    const TcLaunch& L = ((int)i == pl->fused_index && !fused) ? pl->unfused : pl->tc[i];
    if (launch_tc(h, L, st)) return 1;
    if (mark(h, st)) return 1;
  }
  return 0;
}

static int forward_impl(dcscn_handle* h, const float* x, const float* x2, float* y, int n, int H, int W,
                        cudaStream_t st) {
  if (n <= 0 || H <= 0 || W <= 0) return fail("forward: bad shape n=%d h=%d w=%d", n, H, W);
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  if (h->params_dirty && finalize_params(h)) return 1;
  if (ensure_workspace(h, (size_t)n * H * W)) return 1;
  if (h->cfg.depthwise_separable) {
    h->ds_n = n; h->ds_h = H; h->ds_w = W;
    return forward_ds(h, x, x2, y, n, H, W, st);
  }
  Plan* pl = get_plan(h, n, H, W);
  if (!pl) return 1;
  h->last_plan = pl;
  h->ev_used = 0;
  if (mark(h, st)) return 1;
  const bool fused = pl->fused_last && h->fuse_last && h->conv_impl == 0;

  // ---- graph replay / capture of the launches in front of the last kernel (SURVEY 7 step 5: 15 launches per step)
  const bool graphable = h->use_graph && !h->timing && h->conv_impl == 0;
  if (graphable && pl->gexec && pl->g_x == x && pl->g_epoch == h->graph_epoch && pl->g_fused == fused) {
    CUDA_TRY(cudaGraphLaunch(pl->gexec, st));
    h->launches += pl->g_launches;
    h->graph_replays++;
  } else if (graphable && pl->eager_runs >= 1 && pl->last_x == x) {
    if (!h->cap_stream) CUDA_TRY(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
    if (pl->gexec) { cudaGraphExecDestroy(pl->gexec); pl->gexec = nullptr; }
    const int64_t before = h->launches;
    CUDA_TRY(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal));
    const int rc = issue_front(h, pl, x, n, H, W, fused, h->cap_stream);
    cudaGraph_t g = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(h->cap_stream, &g);
    h->launches = before;
    if (rc) { if (g) cudaGraphDestroy(g); return 1; }
    if (ce != cudaSuccess || g == nullptr) return fail("forward: stream capture failed: %s", cudaGetErrorString(ce));
    const cudaError_t ie = cudaGraphInstantiate(&pl->gexec, g, 0);
    cudaGraphDestroy(g);
    if (ie != cudaSuccess) { pl->gexec = nullptr; return fail("forward: cudaGraphInstantiate failed: %s", cudaGetErrorString(ie)); }
    pl->g_x = x; pl->g_epoch = h->graph_epoch; pl->g_fused = fused;
    pl->g_launches = 1 + (int)pl->tc.size();
    CUDA_TRY(cudaGraphLaunch(pl->gexec, st));
    h->launches += pl->g_launches;
    h->graph_replays++;
  } else {
    if (issue_front(h, pl, x, n, H, W, fused, st)) return 1;
    pl->eager_runs++;
  }
  pl->last_x = x;
  pl->ran_fused = fused;
  if (h->wait_x2) {  // forward_host: x2 was copied on the side stream
    CUDA_TRY(cudaStreamWaitEvent(st, h->x2_ready, 0));
    h->wait_x2 = false;
  }
  if (fused) {  // R-CNN1 second half: 9-tap gather of the tap-planar partial products + x2
    ConvGatherParams p = pl->gather;
    p.x2 = x2;
    p.y = y;
    const size_t total = (size_t)p.n_img * p.H * p.W;
    const bool vec4 = p.ksz == 3 && (p.W & 3) == 0 && ((reinterpret_cast<uintptr_t>(x2) | reinterpret_cast<uintptr_t>(y)) & 15) == 0 && h->gather_impl == 0;
    if (vec4) {
      const int grid = (int)std::min<size_t>((total / 4 + 255) / 256, (size_t)h->sm_count * 16);
      conv_last_gather4_kernel<<<grid, 256, 0, st>>>(p);
    } else {
      const int grid = (int)std::min<size_t>((total + 255) / 256, (size_t)h->sm_count * 16);
      conv_last_gather_kernel<<<grid, 256, 0, st>>>(p);
    }
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    if (mark(h, st)) return 1;
    return 0;
  }
  {  // R-CNN1 + x2
    ConvLastParams p = pl->last;
    p.x2 = x2;
    p.y = y;
    const int half = p.ksz >> 1;
    const int tiles = ((p.W + kLastTW - 1) / kLastTW) * ((p.H + kLastTH - 1) / kLastTH) * p.n_img;
    const size_t smem = ((size_t)p.ksz * p.ksz * p.C + (size_t)(kLastTH + 2 * half) * (kLastTW + 2 * half) * kLastCC) * sizeof(float);
    conv_last_kernel<<<tiles, 256, smem, st>>>(p);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    if (mark(h, st)) return 1;
  }
  return 0;
}

// ------------------------------------------------------------------------- Pillow bicubic on the device ----
static double pil_bicubic_filter(double x) {   // Pillow Resample.c bicubic_filter, a = -0.5
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

// Pillow's precompute_coeffs for one axis (helper/pil_resample.py is the Python statement of the same arithmetic).
static int pil_axis(dcscn_handle* h, int in_size, int out_size, PilAxis* ax) {
  for (const auto& t : h->pil_tables)
    if (t.in == in_size && t.out == out_size) {
      *ax = PilAxis{t.k, t.bounds, t.ksize};
      return 0;
    }
  double scale = (double)in_size / (double)out_size, filterscale = scale;
  if (filterscale < 1.0) filterscale = 1.0;
  const double support = 2.0 * filterscale;
  const int ksize = (int)std::ceil(support) * 2 + 1;
  std::vector<double> kk((size_t)out_size * ksize, 0.0);
  std::vector<int> bounds((size_t)out_size * 2, 0);
  const double ss = 1.0 / filterscale;
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = (xx + 0.5) * scale;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    double* k = kk.data() + (size_t)xx * ksize;
    double ww = 0.0;
    for (int x = 0; x < xmax; ++x) {
      const double w = pil_bicubic_filter((x + xmin - center + 0.5) * ss);
      k[x] = w;
      ww += w;
    }
    for (int x = 0; x < xmax; ++x)
      if (ww != 0.0) k[x] /= ww;
    bounds[2 * xx] = xmin;
    bounds[2 * xx + 1] = xmax;
  }
  dcscn_handle::PilTable t;
  t.in = in_size; t.out = out_size; t.ksize = ksize;
  CUDA_TRY(cudaMalloc((void**)&t.k, kk.size() * sizeof(double)));
  CUDA_TRY(cudaMalloc((void**)&t.bounds, bounds.size() * sizeof(int)));
  CUDA_TRY(cudaMemcpy(t.k, kk.data(), kk.size() * sizeof(double), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(t.bounds, bounds.data(), bounds.size() * sizeof(int), cudaMemcpyHostToDevice));
  if (h->pil_tables.size() >= 64) {
    cudaFree(h->pil_tables.front().k);
    cudaFree(h->pil_tables.front().bounds);
    h->pil_tables.erase(h->pil_tables.begin());
  }
  h->pil_tables.push_back(t);
  *ax = PilAxis{t.k, t.bounds, t.ksize};
  return 0;
}

// dst [n, OH, OW] = Pillow-bicubic resize of src [n, H, W] (both fp32 device tensors), horizontal pass first.
static int pil_resize_impl(dcscn_handle* h, const float* src, float* dst, int n, int H, int W, int OH, int OW, cudaStream_t st) {
  if (n <= 0 || H <= 0 || W <= 0 || OH <= 0 || OW <= 0) return fail("bicubic_resize: bad shape");
  PilAxis ax, ay;
  if (pil_axis(h, W, OW, &ax) || pil_axis(h, H, OH, &ay)) return 1;
  const size_t need = (size_t)n * H * OW;
  if (need > h->pil_tmp_cap) {
    cudaFree(h->pil_tmp);
    h->pil_tmp = nullptr;
    h->pil_tmp_cap = 0;
    CUDA_TRY(cudaMalloc((void**)&h->pil_tmp, need * sizeof(float)));
    h->pil_tmp_cap = need;
  }
  const long long t1 = (long long)need, t2 = (long long)n * OH * OW;
  pil_resample_h_kernel<<<(int)std::min<long long>((t1 + 255) / 256, (long long)h->sm_count * 16), 256, 0, st>>>(
      src, h->pil_tmp, (long long)n * H, W, OW, ax);
  pil_resample_v_kernel<<<(int)std::min<long long>((t2 + 255) / 256, (long long)h->sm_count * 16), 256, 0, st>>>(
      h->pil_tmp, dst, n, H, OH, OW, ay);
  CUDA_TRY(cudaGetLastError());
  h->launches += 2;
  return 0;
}

#include "train_engine.inc"
#include "train_ds.inc"

// --------------------------------------------------------------------------------------- C ABI ----
extern "C" {

const char* dcscn_last_error(void) { return g_last_error.c_str(); }

int dcscn_create(const dcscn_config* cfg, dcscn_handle** out) {
  if (!cfg || !out) return fail("dcscn_create: null argument");
  if (cfg->struct_size != (int32_t)sizeof(dcscn_config))
    return fail("dcscn_create: dcscn_config size mismatch (got %d, expected %d)", cfg->struct_size, (int)sizeof(dcscn_config));
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail("dcscn_create: no CUDA device available (%s); this library has no CPU path", cudaGetErrorString(e));
  if (cfg->device_id < 0 || cfg->device_id >= ndev) return fail("dcscn_create: device %d out of range (%d devices)", cfg->device_id, ndev);
  CUDA_TRY(cudaSetDevice(cfg->device_id));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, cfg->device_id));
  if (prop.major != 10) return fail("dcscn_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", cfg->device_id, prop.major, prop.minor);
  if (prop.multiProcessorCount % 2 != 0)   // the tensor-core kernels run on CTA pairs (two SMs of one TPC)
    return fail("dcscn_create: device %d has an odd SM count (%d); the CTA-pair tensor-core kernels need an even one", cfg->device_id, prop.multiProcessorCount);

  std::unique_ptr<dcscn_handle> h(new dcscn_handle());
  h->cfg = *cfg;
  h->sm_count = prop.multiProcessorCount;
  if (build_graph(h.get())) return 1;

  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (qres != cudaDriverEntryPointSuccess || fn == nullptr) return fail("cuTensorMapEncodeTiled is not available in this driver");
  h->encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
  *out = h.release();
  return 0;
}

int dcscn_destroy(dcscn_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->cfg.device_id);
  cudaDeviceSynchronize();
  for (TcLayer& t : h->tcl) free_tc(t);
  for (TcLayer& t : h->bwd) free_tc(t);
  train_free(h);
  cudaFree(h->ens_x); cudaFree(h->ens_x2); cudaFree(h->ens_y); cudaFree(h->ensio_x); cudaFree(h->ensio_x2); cudaFree(h->ensio_y);
  cudaFree(h->d_first_w);
  cudaFree(h->d_first_bias);
  cudaFree(h->d_first_alpha);
  cudaFree(h->d_last_w);
  cudaFree(h->feat_hi);
  cudaFree(h->feat_lo);
  cudaFree(h->b1_hi);
  cudaFree(h->b1_lo);
  cudaFree(h->nin_hi);
  cudaFree(h->nin_lo);
  cudaFree(h->mid_hi);
  cudaFree(h->mid_lo);
  cudaFree(h->hr);
  cudaFree(h->vbuf);
  cudaFree(h->ds_feat); cudaFree(h->ds_b1); cudaFree(h->ds_nin); cudaFree(h->ds_mid); cudaFree(h->ds_hr);
  for (auto& d : h->ds) { cudaFree(d.dw); cudaFree(d.pw); cudaFree(d.bias); cudaFree(d.alpha); }
  cudaFree(h->ds_ab.pw); cudaFree(h->ds_ab.bias); cudaFree(h->ds_ab.alpha);
  cudaFree(h->io_x);
  cudaFree(h->io_x2);
  cudaFree(h->io_y);
  for (auto& pt : h->pil_tables) { cudaFree(pt.k); cudaFree(pt.bounds); }
  cudaFree(h->pil_tmp);
  cudaFree(h->ps_lr); cudaFree(h->ps_bic); cudaFree(h->ps_true); cudaFree(h->ps_idx);
  h->plans.clear();
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->x2_ready) cudaEventDestroy(h->x2_ready);
  delete h;
  return 0;
}

int dcscn_num_params(dcscn_handle* h) { return h ? (int)h->params.size() : 0; }

int dcscn_param_info(dcscn_handle* h, int index, char* name_buf, int name_buf_len, int64_t* dims4, int* ndim) {
  if (!h || index < 0 || index >= (int)h->params.size()) return fail("dcscn_param_info: bad index %d", index);
  const ParamDef& p = h->params[index];
  if (name_buf && name_buf_len > 0) snprintf(name_buf, name_buf_len, "%s", p.name.c_str());
  if (ndim) *ndim = (int)p.shape.size();
  if (dims4)
    for (size_t i = 0; i < p.shape.size() && i < 4; ++i) dims4[i] = p.shape[i];
  return 0;
}

int dcscn_set_param(dcscn_handle* h, const char* name, const float* host_data, int64_t numel) {
  if (!h || !name || !host_data) return fail("dcscn_set_param: null argument");
  auto it = h->param_index.find(name);
  if (it == h->param_index.end()) return fail("dcscn_set_param: unknown variable '%s'", name);
  if (sync_host_params(h)) return 1;
  ParamDef& p = h->params[it->second];
  if (numel != p.numel()) return fail("dcscn_set_param: '%s' has %lld elements, got %lld", name, (long long)p.numel(), (long long)numel);
  memcpy(p.host.data(), host_data, (size_t)numel * sizeof(float));
  h->params_dirty = true;
  if (h->train) h->train->w_synced = false;
  return 0;
}

int dcscn_get_param(dcscn_handle* h, const char* name, float* host_data, int64_t numel) {
  if (!h || !name || !host_data) return fail("dcscn_get_param: null argument");
  auto it = h->param_index.find(name);
  if (it == h->param_index.end()) return fail("dcscn_get_param: unknown variable '%s'", name);
  if (sync_host_params(h)) return 1;
  const ParamDef& p = h->params[it->second];
  if (numel != p.numel()) return fail("dcscn_get_param: '%s' has %lld elements, got %lld", name, (long long)p.numel(), (long long)numel);
  memcpy(host_data, p.host.data(), (size_t)numel * sizeof(float));
  return 0;
}

int dcscn_forward(dcscn_handle* h, const float* x_dev, const float* x2_dev, float* y_dev, int n, int height, int width,
                  void* stream) {
  if (!h || !x_dev || !x2_dev || !y_dev) return fail("dcscn_forward: null argument");
  return forward_impl(h, x_dev, x2_dev, y_dev, n, height, width, (cudaStream_t)stream);
}

int dcscn_bicubic_resize(dcscn_handle* h, const float* src_dev, float* dst_dev, int n, int height, int width, int out_height,
                         int out_width, void* stream) {
  if (!h || !src_dev || !dst_dev) return fail("dcscn_bicubic_resize: null argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  return pil_resize_impl(h, src_dev, dst_dev, n, height, width, out_height, out_width, (cudaStream_t)stream);
}

int dcscn_forward_host(dcscn_handle* h, const float* x, const float* x2, float* y, int n, int height, int width) {
  if (!h || !x || !y) return fail("dcscn_forward_host: null argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  const size_t lr = (size_t)n * height * width;
  const size_t hr = lr * h->cfg.scale * h->cfg.scale;
  if (hr > h->io_cap) {
    cudaFree(h->io_x);
    cudaFree(h->io_x2);
    cudaFree(h->io_y);
    h->io_x = h->io_x2 = h->io_y = nullptr;
    CUDA_TRY(cudaMalloc((void**)&h->io_x, lr * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->io_x2, hr * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->io_y, hr * sizeof(float)));
    h->io_cap = hr;
  }
  cudaStream_t st = 0;
  if (!h->copy_stream) {
    CUDA_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&h->x2_ready, cudaEventDisableTiming));
  }
  // x feeds the first kernel; x2 (4x / 9x / 16x the bytes) is only read by the very last one, so it is copied on a second
  // stream while the conv stack runs and the last kernel waits for it
  CUDA_TRY(cudaMemcpyAsync(h->io_x, x, lr * sizeof(float), cudaMemcpyHostToDevice, st));
  if (x2) {
    CUDA_TRY(cudaMemcpyAsync(h->io_x2, x2, hr * sizeof(float), cudaMemcpyHostToDevice, h->copy_stream));
    CUDA_TRY(cudaEventRecord(h->x2_ready, h->copy_stream));
    h->wait_x2 = true;
  } else {
    // x2 = Pillow-bicubic up-scale of x, formed in HBM (what util.resize_image_by_pil does on the host, bit for bit)
    const int s = h->cfg.scale;
    if (pil_resize_impl(h, h->io_x, h->io_x2, n, height, width, s * height, s * width, st)) return 1;
  }
  const int rc = forward_impl(h, h->io_x, h->io_x2, h->io_y, n, height, width, st);
  h->wait_x2 = false;
  if (rc) {
    cudaStreamSynchronize(h->copy_stream);
    return 1;
  }
  CUDA_TRY(cudaMemcpyAsync(y, h->io_y, hr * sizeof(float), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

// Self-ensemble entirely on the device (DCSCN.py:547-586 `do` with self_ensemble = flips): the transformed copies of x
// and x2 are produced by a kernel, transforms 0..3 run as ONE batched forward (n = up to 4, shape [h][w]) and 4..7 as
// another (shape [w][h]), and the inverse transforms + the float64 mean are one more kernel.
static int ensemble_impl(dcscn_handle* h, const float* x, const float* x2, double* y, int height, int width, int mask,
                         double divisor, cudaStream_t st) {
  if (mask <= 0 || mask > 255) return fail("forward_ensemble: transform mask must select 1..8 of the 8 transforms (got 0x%x)", mask);
  if (height <= 0 || width <= 0) return fail("forward_ensemble: bad shape h=%d w=%d", height, width);
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  const int s = h->cfg.scale;
  const size_t lr = (size_t)height * width, hr = lr * s * s;
  if (hr > h->ens_cap) {
    cudaFree(h->ens_x); cudaFree(h->ens_x2); cudaFree(h->ens_y);
    h->ens_x = h->ens_x2 = h->ens_y = nullptr;
    h->ens_cap = 0;
    CUDA_TRY(cudaMalloc((void**)&h->ens_x, 4 * lr * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->ens_x2, 4 * hr * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->ens_y, 8 * hr * sizeof(float)));
    h->ens_cap = hr;
  }
  const int grid_lr = (int)std::min<size_t>((4 * lr + 255) / 256, (size_t)h->sm_count * 8);
  const int grid_hr = (int)std::min<size_t>((4 * hr + 255) / 256, (size_t)h->sm_count * 8);
  for (int grp = 0; grp < 2; ++grp) {
    EnsembleSel sel;
    memset(&sel, 0, sizeof(sel));
    for (int t = 4 * grp; t < 4 * grp + 4; ++t)
      if ((mask >> t) & 1) sel.t[sel.count++] = t;
    if (sel.count == 0) continue;
    ensemble_flip_kernel<<<grid_lr, 256, 0, st>>>(x, h->ens_x, height, width, sel);
    ensemble_flip_kernel<<<grid_hr, 256, 0, st>>>(x2, h->ens_x2, s * height, s * width, sel);
    CUDA_TRY(cudaGetLastError());
    h->launches += 2;
    const int fh = grp == 0 ? height : width, fw = grp == 0 ? width : height;
    if (forward_impl(h, h->ens_x, h->ens_x2, h->ens_y + (size_t)grp * 4 * hr, sel.count, fh, fw, st)) return 1;
  }
  ensemble_reduce_kernel<<<(int)std::min<size_t>((hr + 255) / 256, (size_t)h->sm_count * 8), 256, 0, st>>>(
      h->ens_y, h->ens_y + 4 * hr, y, s * height, s * width, mask, divisor);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return 0;
}

int dcscn_forward_ensemble(dcscn_handle* h, const float* x_dev, const float* x2_dev, double* y_dev, int height, int width,
                           int flips, void* stream) {
  if (!h || !x_dev || !x2_dev || !y_dev) return fail("dcscn_forward_ensemble: null argument");
  if (flips < 1 || flips > 8) return fail("forward_ensemble: flips must be 1..8 (got %d)", flips);
  return ensemble_impl(h, x_dev, x2_dev, y_dev, height, width, (1 << flips) - 1, (double)flips, (cudaStream_t)stream);
}

int dcscn_forward_ensemble_partial(dcscn_handle* h, const float* x_dev, const float* x2_dev, double* y_dev, int height,
                                   int width, int transform_mask, void* stream) {
  if (!h || !x_dev || !x2_dev || !y_dev) return fail("dcscn_forward_ensemble_partial: null argument");
  return ensemble_impl(h, x_dev, x2_dev, y_dev, height, width, transform_mask, 1.0, (cudaStream_t)stream);
}

int dcscn_forward_ensemble_host(dcscn_handle* h, const float* x, const float* x2, double* y, int height, int width, int flips) {
  if (!h || !x || !y) return fail("dcscn_forward_ensemble_host: null argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  const size_t lr = (size_t)height * width;
  const size_t hr = lr * h->cfg.scale * h->cfg.scale;
  if (hr > h->ensio_cap) {
    cudaFree(h->ensio_x); cudaFree(h->ensio_x2); cudaFree(h->ensio_y);
    h->ensio_x = h->ensio_x2 = nullptr;
    h->ensio_y = nullptr;
    h->ensio_cap = 0;
    CUDA_TRY(cudaMalloc((void**)&h->ensio_x, lr * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->ensio_x2, hr * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->ensio_y, hr * sizeof(double)));
    h->ensio_cap = hr;
  }
  cudaStream_t st = 0;
  CUDA_TRY(cudaMemcpyAsync(h->ensio_x, x, lr * sizeof(float), cudaMemcpyHostToDevice, st));
  if (x2) {
    CUDA_TRY(cudaMemcpyAsync(h->ensio_x2, x2, hr * sizeof(float), cudaMemcpyHostToDevice, st));
  } else if (pil_resize_impl(h, h->ensio_x, h->ensio_x2, 1, height, width, h->cfg.scale * height, h->cfg.scale * width, st)) {
    return 1;
  }
  if (flips < 1 || flips > 8) return fail("forward_ensemble: flips must be 1..8 (got %d)", flips);
  if (ensemble_impl(h, h->ensio_x, h->ensio_x2, h->ensio_y, height, width, (1 << flips) - 1, (double)flips, st)) return 1;
  CUDA_TRY(cudaMemcpyAsync(y, h->ensio_y, hr * sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

int dcscn_get_activation(dcscn_handle* h, const char* tensor, float* host_data, int64_t numel) {
  if (!h || !tensor || !host_data) return fail("dcscn_get_activation: null argument");
  if (h->cfg.depthwise_separable) {
    if (h->ds_n == 0) return fail("dcscn_get_activation: no forward has run yet");
    CUDA_TRY(cudaSetDevice(h->cfg.device_id));
    CUDA_TRY(cudaDeviceSynchronize());
    const dcscn_config& c = h->cfg;
    const std::string t(tensor);
    const int cps = c.nin_filters + c.nin_filters2;
    const float* src = nullptr;
    int pitch = 0, off = 0, ch = 0;
    size_t px = (size_t)h->ds_n * h->ds_h * h->ds_w;
    if (t.rfind("CNN", 0) == 0) {
      int i = atoi(t.c_str() + 3) - 1;
      if (i < 0 || i >= c.layers) return fail("dcscn_get_activation: no tensor '%s'", tensor);
      src = h->ds_feat; pitch = h->ds_total; off = h->ds_off[i]; ch = h->filters[i];
    } else if (t == "A1") { src = h->ds_nin; pitch = cps; off = c.nin_filters2; ch = c.nin_filters;
    } else if (t == "B2") { src = h->ds_nin; pitch = cps; off = 0; ch = c.nin_filters2;
    } else if (t == "B1") { src = h->ds_b1; pitch = c.nin_filters2; off = 0; ch = c.nin_filters2;
    } else if (t == "Up-PS" && c.scale == 4) { src = h->ds_mid; pitch = cps; off = 0; ch = cps; px *= 4;
    } else if ((t == "Up-PS" && c.scale != 4) || (t == "Up-PS2" && c.scale == 4)) {
      src = h->ds_hr; pitch = h->ps_out; off = 0; ch = h->ps_out; px *= (size_t)c.scale * c.scale;
    } else return fail("dcscn_get_activation: no tensor '%s'", tensor);
    if (numel != (int64_t)(px * ch)) return fail("dcscn_get_activation: '%s' has %lld elements, got %lld", tensor, (long long)(px * ch), (long long)numel);
    std::vector<float> full(px * pitch);
    CUDA_TRY(cudaMemcpy(full.data(), src, full.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (size_t p = 0; p < px; ++p)
      for (int k = 0; k < ch; ++k) host_data[p * ch + k] = full[p * pitch + off + k];
    return 0;
  }
  Plan* pl = h->last_plan;
  if (!pl) return fail("dcscn_get_activation: no forward has run yet");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  CUDA_TRY(cudaDeviceSynchronize());
  const dcscn_config& c = h->cfg;
  const std::string t(tensor);
  const __half *hi = nullptr, *lo = nullptr;
  const float* f32 = nullptr;
  int pitch = 0, off = 0, ch = 0;
  size_t px = (size_t)pl->n * pl->h * pl->w;
  if (t.rfind("CNN", 0) == 0) {
    int i = atoi(t.c_str() + 3) - 1;
    if (i < 0 || i >= c.layers) return fail("dcscn_get_activation: no tensor '%s'", tensor);
    hi = h->feat_hi; lo = h->feat_lo; pitch = h->feat_pitch; off = h->feat_off[i]; ch = h->filters[i];
  } else if (t == "A1") {
    hi = h->nin_hi; lo = h->nin_lo; pitch = h->nin_pitch; off = h->b1_w; ch = c.nin_filters;
  } else if (t == "B2") {
    hi = h->nin_hi; lo = h->nin_lo; pitch = h->nin_pitch; off = 0; ch = c.nin_filters2;
  } else if (t == "B1") {
    hi = h->b1_hi; lo = h->b1_lo; pitch = h->b1_w; off = 0; ch = c.nin_filters2;
  } else if (t == "Up-PS" && c.scale == 4) {
    hi = h->mid_hi; lo = h->mid_lo; pitch = h->mid_pitch; off = 0; ch = c.nin_filters + c.nin_filters2; px *= 4;
  } else if (((t == "Up-PS" && c.scale != 4) || (t == "Up-PS2" && c.scale == 4)) && pl->ran_fused) {
    return fail("dcscn_get_activation: '%s' is not materialised when the R-CNN1 fusion is on (set option fuse_last=0)", tensor);
  } else if ((t == "Up-PS" && c.scale != 4) || (t == "Up-PS2" && c.scale == 4)) {
    f32 = h->hr; pitch = h->ps_out; ch = h->ps_out; px *= (size_t)c.scale * c.scale;
  } else {
    return fail("dcscn_get_activation: no tensor '%s'", tensor);
  }
  if (numel != (int64_t)(px * ch)) return fail("dcscn_get_activation: '%s' has %lld elements, got %lld", tensor, (long long)(px * ch), (long long)numel);
  std::vector<float> full(px * pitch);
  if (f32) {
    CUDA_TRY(cudaMemcpy(full.data(), f32, full.size() * sizeof(float), cudaMemcpyDeviceToHost));
  } else {
    float* tmp = nullptr;
    CUDA_TRY(cudaMalloc((void**)&tmp, full.size() * sizeof(float)));
    planes_to_f32_kernel<<<1024, 256>>>(hi, planes(h) == 2 ? lo : nullptr, tmp, full.size());
    cudaError_t e = cudaMemcpy(full.data(), tmp, full.size() * sizeof(float), cudaMemcpyDeviceToHost);
    cudaFree(tmp);
    if (e != cudaSuccess) return fail("dcscn_get_activation: copy failed: %s", cudaGetErrorString(e));
  }
  for (size_t p = 0; p < px; ++p)
    for (int k = 0; k < ch; ++k) host_data[p * ch + k] = full[p * pitch + off + k];
  return 0;
}

int dcscn_set_option(dcscn_handle* h, const char* key, int64_t value) {
  if (!h || !key) return fail("dcscn_set_option: null argument");
  const std::string k(key);
  h->graph_epoch++;          // whatever changes, captured launch sequences are rebuilt
  if (k == "graph") {
    h->use_graph = value ? 1 : 0;
    return 0;
  }
  if (k == "gather_impl") {
    h->gather_impl = value ? 1 : 0;
    return 0;
  }
  if (k == "ds_cache") {
    h->ds_cache = value ? 1 : 0;
    return 0;
  }
  if (k == "wide_tiles") {
    if (h->wide_tiles != (value ? 1 : 0)) {
      h->wide_tiles = value ? 1 : 0;
      h->params_dirty = true;               // other column tiles: re-tile and re-pack
      h->cap_px = 0;                        // the fused R-CNN1 partial planes change size
      h->plans.clear();
      h->last_plan = nullptr;
    }
    return 0;
  }
  if (k == "store_mode") {
    if (value < 0 || value > 2) return fail("store_mode must be 0 (32-byte stores), 1 (16-byte stores) or 2 (lane-pair 64-byte runs)");
    h->store_mode = (int)value;
    return 0;
  }
  if (k == "conv_impl") {
    if (value != 0 && value != 1) return fail("conv_impl must be 0 (tcgen05) or 1 (CUDA-core validation)");
    h->conv_impl = (int)value;
  } else if (k == "ds_impl") {
    if (value != 0 && value != 1) return fail("ds_impl must be 0 (tile kernels) or 1 (first-generation kernels)");
    h->ds_impl = (int)value;
  } else if (k == "fuse_last") {
    h->fuse_last = value ? 1 : 0;
  } else if (k == "timing") {
    h->timing = value ? 1 : 0;
  } else if (k == "wgrad_impl") {
    if (value != 0 && value != 1) return fail("wgrad_impl must be 0 (tensor cores) or 1 (CUDA cores)");
    h->wgrad_impl = (int)value;
  } else if (k == "l1_loss") {
    h->l1_loss = value ? 1 : 0;
  } else if (k == "wgrad_taps") {
    if (value < 0 || value > 3) return fail("wgrad_taps must be 0 (automatic) .. 3");
    h->wgrad_taps = (int)value;
  } else if (k == "host_repack") {
    h->host_repack = value ? 1 : 0;
  } else if (k == "act_grad_impl") {
    if (value < 0 || value > 1) return fail("act_grad_impl must be 0 or 1");
    h->act_grad_impl = (int)value;
  } else if (k == "seg_chunks") {
    if (value < 0 || value > 4096) return fail("seg_chunks must be >= 0 (0 = automatic)");
    h->seg_chunks = (int)value;
    h->params_dirty = true;     // the streaming kernel's stage tables carry the segment boundaries
    h->plans.clear();
    h->last_plan = nullptr;
  } else {
    return fail("dcscn_set_option: unknown option '%s'", key);
  }
  return 0;
}

int dcscn_get_timings(dcscn_handle* h, float* ms, int capacity, int* count, char* names, int names_len) {
  if (!h || !count) return fail("dcscn_get_timings: null argument");
  *count = 0;
  if (h->ev_used < 2) return 0;
  CUDA_TRY(cudaEventSynchronize(h->ev[h->ev_used - 1]));
  const int n = h->ev_used - 1;
  for (int i = 0; i < n && i < capacity; ++i) CUDA_TRY(cudaEventElapsedTime(&ms[i], h->ev[i], h->ev[i + 1]));
  *count = n;
  if (names && names_len > 0) {
    std::string s = "CNN1";
    if (h->cfg.depthwise_separable) {
      s = "";
      for (const LayerDef& l : h->layers) {
        std::string nm = l.scope.substr(0, l.scope.find('/'));
        if (h->ds_impl == 0 && nm == "B1") continue;          // the tile kernels run A1 | B1 as one launch
        if (h->ds_impl == 0 && nm == "A1") nm = "A1+B1";
        s += (s.empty() ? "" : ",") + nm;
      }
    } else {
      for (const TcLayer& t : h->tcl) s += "," + t.name;
      s += ",R-CNN1";
    }
    snprintf(names, names_len, "%s", s.c_str());
  }
  return 0;
}

int dcscn_train_step(dcscn_handle* h, const float* x_dev, const float* x2_dev, const float* y_dev, int n, int height, int width,
                     float lr, uint32_t seed, int apply_update, float* out_loss, float* out_mse, void* stream) {
  if (!h || !x_dev || !x2_dev || !y_dev) return fail("dcscn_train_step: null argument");
  return train_step_impl(h, x_dev, x2_dev, y_dev, n, height, width, lr, seed, apply_update, out_loss, out_mse, (cudaStream_t)stream);
}

int dcscn_train_step_host(dcscn_handle* h, const float* x, const float* x2, const float* y, int n, int height, int width, float lr,
                          uint32_t seed, int apply_update, float* out_loss, float* out_mse) {
  if (!h || !x || !x2 || !y) return fail("dcscn_train_step_host: null argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  const size_t lr_px = (size_t)n * height * width;
  const size_t hr_px = lr_px * h->cfg.scale * h->cfg.scale;
  if (hr_px > h->io_cap) {
    cudaFree(h->io_x); cudaFree(h->io_x2); cudaFree(h->io_y);
    h->io_x = h->io_x2 = h->io_y = nullptr;
    CUDA_TRY(cudaMalloc((void**)&h->io_x, lr_px * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->io_x2, hr_px * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->io_y, hr_px * sizeof(float)));
    h->io_cap = hr_px;
  }
  cudaStream_t st = 0;
  CUDA_TRY(cudaMemcpyAsync(h->io_x, x, lr_px * sizeof(float), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(h->io_x2, x2, hr_px * sizeof(float), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(h->io_y, y, hr_px * sizeof(float), cudaMemcpyHostToDevice, st));
  return train_step_impl(h, h->io_x, h->io_x2, h->io_y, n, height, width, lr, seed, apply_update, out_loss, out_mse, st);
}

int dcscn_patch_store_set(dcscn_handle* h, const uint8_t* lr, const uint8_t* bicubic, const uint8_t* truth, int64_t count,
                          int patch_height, int patch_width) {
  if (!h || !lr || !bicubic || !truth) return fail("dcscn_patch_store_set: null argument");
  if (count <= 0 || count > 0x7FFFFFFF || patch_height <= 0 || patch_width <= 0) return fail("dcscn_patch_store_set: bad size");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  for (auto& pt : h->pil_tables) { cudaFree(pt.k); cudaFree(pt.bounds); }
  cudaFree(h->pil_tmp);
  cudaFree(h->ps_lr); cudaFree(h->ps_bic); cudaFree(h->ps_true);
  h->ps_lr = h->ps_bic = h->ps_true = nullptr;
  h->ps_count = 0;
  const size_t s2 = (size_t)h->cfg.scale * h->cfg.scale;
  const size_t lr_b = (size_t)count * patch_height * patch_width, hr_b = lr_b * s2;
  CUDA_TRY(cudaMalloc((void**)&h->ps_lr, lr_b));
  CUDA_TRY(cudaMalloc((void**)&h->ps_bic, hr_b));
  CUDA_TRY(cudaMalloc((void**)&h->ps_true, hr_b));
  CUDA_TRY(cudaMemcpy(h->ps_lr, lr, lr_b, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(h->ps_bic, bicubic, hr_b, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(h->ps_true, truth, hr_b, cudaMemcpyHostToDevice));
  h->ps_count = count;
  h->ps_h = patch_height;
  h->ps_w = patch_width;
  return 0;
}

// Gathers the indexed patches into the fp32 staging tensors io_x / io_x2 / io_y (shared with the host-buffer calls).
static int patch_gather(dcscn_handle* h, const int32_t* indices, int n, float max_value, cudaStream_t st) {
  if (h->ps_count == 0) return fail("train_step_indexed: no patch store (call dcscn_patch_store_set first)");
  if (n <= 0) return fail("train_step_indexed: empty mini-batch");
  for (int i = 0; i < n; ++i) {
    const int64_t k = indices[i] & 0x7FFFFFFF;
    if (k >= h->ps_count) return fail("train_step_indexed: patch index %lld out of range (%lld patches)", (long long)k, (long long)h->ps_count);
  }
  const int s = h->cfg.scale;
  const size_t lr_px = (size_t)n * h->ps_h * h->ps_w, hr_px = lr_px * s * s;
  if (hr_px > h->io_cap) {
    cudaFree(h->io_x); cudaFree(h->io_x2); cudaFree(h->io_y);
    h->io_x = h->io_x2 = h->io_y = nullptr;
    h->io_cap = 0;
    CUDA_TRY(cudaMalloc((void**)&h->io_x, lr_px * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->io_x2, hr_px * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->io_y, hr_px * sizeof(float)));
    h->io_cap = hr_px;
  }
  if (n > h->ps_idx_cap) {
    cudaFree(h->ps_idx);
    h->ps_idx = nullptr;
    CUDA_TRY(cudaMalloc((void**)&h->ps_idx, (size_t)n * sizeof(int)));
    h->ps_idx_cap = n;
  }
  CUDA_TRY(cudaMemcpyAsync(h->ps_idx, indices, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, st));
  const double scale = (double)max_value / 255.0;
  const int grid_lr = (int)std::min<size_t>((lr_px + 255) / 256, (size_t)h->sm_count * 8);
  const int grid_hr = (int)std::min<size_t>((hr_px + 255) / 256, (size_t)h->sm_count * 8);
  patch_gather_kernel<<<grid_lr, 256, 0, st>>>(h->ps_lr, h->ps_idx, h->io_x, n, h->ps_h, h->ps_w, scale);
  patch_gather_kernel<<<grid_hr, 256, 0, st>>>(h->ps_bic, h->ps_idx, h->io_x2, n, s * h->ps_h, s * h->ps_w, scale);
  patch_gather_kernel<<<grid_hr, 256, 0, st>>>(h->ps_true, h->ps_idx, h->io_y, n, s * h->ps_h, s * h->ps_w, scale);
  CUDA_TRY(cudaGetLastError());
  h->launches += 3;
  return 0;
}

int dcscn_train_step_indexed(dcscn_handle* h, const int32_t* indices, int n, float max_value, float lr, uint32_t seed,
                             int apply_update, float* out_loss, float* out_mse) {
  if (!h || !indices) return fail("dcscn_train_step_indexed: null argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  cudaStream_t st = 0;
  if (patch_gather(h, indices, n, max_value, st)) return 1;
  return train_step_impl(h, h->io_x, h->io_x2, h->io_y, n, h->ps_h, h->ps_w, lr, seed, apply_update, out_loss, out_mse, st);
}

int dcscn_patch_gather(dcscn_handle* h, const int32_t* indices, int n, float max_value, float* x, float* x2, float* y) {
  if (!h || !indices || !x || !x2 || !y) return fail("dcscn_patch_gather: null argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  cudaStream_t st = 0;
  if (patch_gather(h, indices, n, max_value, st)) return 1;
  const int s = h->cfg.scale;
  const size_t lr_px = (size_t)n * h->ps_h * h->ps_w, hr_px = lr_px * s * s;
  CUDA_TRY(cudaMemcpyAsync(x, h->io_x, lr_px * sizeof(float), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(x2, h->io_x2, hr_px * sizeof(float), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(y, h->io_y, hr_px * sizeof(float), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

int dcscn_get_grad(dcscn_handle* h, const char* name, float* host_data, int64_t numel) {
  if (!h || !name || !host_data) return fail("dcscn_get_grad: null argument");
  if (!h->train || h->train->total == 0) return fail("dcscn_get_grad: no train step has run yet");
  auto it = h->param_index.find(name);
  if (it == h->param_index.end()) return fail("dcscn_get_grad: unknown variable '%s'", name);
  const ParamDef& p = h->params[it->second];
  if (numel != p.numel()) return fail("dcscn_get_grad: '%s' has %lld elements, got %lld", name, (long long)p.numel(), (long long)numel);
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  CUDA_TRY(cudaMemcpy(host_data, h->train->d_g + h->train->off[it->second], (size_t)numel * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int dcscn_get_adam_slot(dcscn_handle* h, const char* name, int slot, float* host_data, int64_t numel) {
  if (!h || !name || !host_data) return fail("dcscn_get_adam_slot: null argument");
  if (!h->train || h->train->total == 0) return fail("dcscn_get_adam_slot: no train step has run yet");
  auto it = h->param_index.find(name);
  if (it == h->param_index.end()) return fail("dcscn_get_adam_slot: unknown variable '%s'", name);
  const ParamDef& p = h->params[it->second];
  if (numel != p.numel() || (slot != 0 && slot != 1)) return fail("dcscn_get_adam_slot: bad size or slot");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  const float* src = (slot == 0 ? h->train->d_m : h->train->d_v) + h->train->off[it->second];
  CUDA_TRY(cudaMemcpy(host_data, src, (size_t)numel * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int dcscn_set_adam_slot(dcscn_handle* h, const char* name, int slot, const float* host_data, int64_t numel) {
  if (!h || !name || !host_data) return fail("dcscn_set_adam_slot: null argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  if (train_init(h)) return 1;
  auto it = h->param_index.find(name);
  if (it == h->param_index.end()) return fail("dcscn_set_adam_slot: unknown variable '%s'", name);
  const ParamDef& p = h->params[it->second];
  if (numel != p.numel() || (slot != 0 && slot != 1)) return fail("dcscn_set_adam_slot: bad size or slot");
  float* dst = (slot == 0 ? h->train->d_m : h->train->d_v) + h->train->off[it->second];
  CUDA_TRY(cudaMemcpy(dst, host_data, (size_t)numel * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

int dcscn_get_adam_step(dcscn_handle* h, int64_t* step) {
  if (!h || !step) return fail("dcscn_get_adam_step: null argument");
  *step = h->train ? h->train->step : 0;
  return 0;
}

int dcscn_set_adam_step(dcscn_handle* h, int64_t step) {
  if (!h || step < 0) return fail("dcscn_set_adam_step: bad argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  if (train_init(h)) return 1;
  h->train->step = step;
  return 0;
}

int dcscn_reset_optimizer(dcscn_handle* h) {
  if (!h) return fail("dcscn_reset_optimizer: null argument");
  if (!h->train || h->train->total == 0) return 0;   // no optimizer state exists yet: slots start at zero anyway
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  CUDA_TRY(cudaMemset(h->train->d_m, 0, h->train->total * sizeof(float)));
  CUDA_TRY(cudaMemset(h->train->d_v, 0, h->train->total * sizeof(float)));
  h->train->step = 0;
  return 0;
}

int dcscn_grad_buffer(dcscn_handle* h, float** dev_ptr, int64_t* count) {
  if (!h || !dev_ptr || !count) return fail("dcscn_grad_buffer: null argument");
  if (!h->train || h->train->total == 0) return fail("dcscn_grad_buffer: no train step has run yet");
  *dev_ptr = h->train->d_g;
  *count = (int64_t)h->train->total + 2;   // gradients of every trainable, then {image_loss, mse} of the last step
  return 0;
}

int dcscn_apply_gradients(dcscn_handle* h, float lr, void* stream) {
  if (!h) return fail("dcscn_apply_gradients: null argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  return apply_gradients_impl(h, lr, true, (cudaStream_t)stream);
}

int dcscn_apply_gradients_avg(dcscn_handle* h, float lr, float grad_scale, float* out_loss, float* out_mse, void* stream) {
  if (!h) return fail("dcscn_apply_gradients_avg: null argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device_id));
  return apply_gradients_impl(h, lr, true, (cudaStream_t)stream, grad_scale, out_loss, out_mse);
}

float dcscn_last_grad_norm(dcscn_handle* h) { return (h && h->train) ? h->train->last_norm : 0.f; }

int dcscn_dropout_mask(dcscn_handle* h, const char* tensor, uint32_t seed, int n, int height, int width, uint8_t* mask, int64_t numel) {
  if (!h || !tensor || !mask) return fail("dcscn_dropout_mask: null argument");
  const dcscn_config& c = h->cfg;
  const std::string t(tensor);
  const int L = c.layers;
  int C = 0, n_total = 0, col0 = 0;
  uint32_t layer = 0;
  if (t.rfind("CNN", 0) == 0) {
    const int i = atoi(t.c_str() + 3) - 1;
    if (i < 0 || i >= L) return fail("dcscn_dropout_mask: no tensor '%s'", tensor);
    C = h->filters[i]; n_total = h->feat_w[i]; col0 = 0; layer = (uint32_t)(i + 1);
  } else if (t == "A1") { C = c.nin_filters; n_total = h->a1_w + h->b1_w; col0 = 0; layer = (uint32_t)(L + 1);
  } else if (t == "B1") { C = c.nin_filters2; n_total = h->a1_w + h->b1_w; col0 = h->a1_w; layer = (uint32_t)(L + 1);
  } else if (t == "B2") { C = c.nin_filters2; n_total = h->b1_w; col0 = 0; layer = (uint32_t)(L + 2);
  } else return fail("dcscn_dropout_mask: tensor '%s' has no dropout", tensor);
  if (c.depthwise_separable) {   // train_ds.inc: dense [pixel][channel] indexing, A1 / B2 / B1 are layers L+1 / L+2 / L+3
    n_total = C; col0 = 0;
    if (t == "B1") layer = (uint32_t)(L + 3);
  }
  const size_t px = (size_t)n * height * width;
  if (numel != (int64_t)(px * C)) return fail("dcscn_dropout_mask: expected %lld elements", (long long)(px * C));
  for (size_t q = 0; q < px; ++q)
    for (int k = 0; k < C; ++k)
      mask[q * C + k] = dropout_keep(seed, layer, (uint64_t)q * (uint64_t)n_total + col0 + k, c.dropout_keep) ? 1 : 0;
  return 0;
}

// Measurement entry (csrc/umma_probe.cuh): kind::f16 UMMA throughput with operands resident in shared memory.
// group = 1 | 2 (cta_group), n = accumulator width of one product, mode 0 = three products per K slice (the scheme
// of the conv kernels), 1 = stacked 2n + n (group 1 only), 2 = one product.  Returns the launch's duration and the
// longest issuing-thread span in cycles.
int dcscn_umma_probe(int device_id, int group, int n, int mode, int iters, float* out_ms, double* out_cycles) {
  if ((group != 1 && group != 2) || n < 16 || n > 256 || (n & 15) || mode < 0 || mode > 2 || iters < 1)
    return fail("dcscn_umma_probe: bad argument");
  if (mode == 1 && (group != 1 || n > 128)) return fail("dcscn_umma_probe: the stacked form needs group 1 and n <= 128");
  CUDA_TRY(cudaSetDevice(device_id));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device_id));
  if (prop.major != 10) return fail("dcscn_umma_probe: device %d is not sm_100", device_id);
  const int grid = (prop.multiProcessorCount / 2) * 2;
  const int b_rows = group == 2 ? n / 2 : n;
  const size_t smem = 2 * (size_t)(2 * 128 * 128 + 2 * b_rows * 128) + 1024 + 64;
  CUDA_TRY(cudaFuncSetAttribute(umma_probe_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  CUDA_TRY(cudaFuncSetAttribute(umma_probe_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  unsigned long long* d_cyc = nullptr;
  CUDA_TRY(cudaMalloc(&d_cyc, sizeof(unsigned long long) * grid));
  CUDA_TRY(cudaMemset(d_cyc, 0, sizeof(unsigned long long) * grid));
  UmmaProbeParams p{n, mode, iters, d_cyc};
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(128);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = group;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 3; ++rep) {          // first pass warms up; report the faster of the other two
    CUDA_TRY(cudaEventRecord(e0, 0));
    if (group == 2) CUDA_TRY(cudaLaunchKernelEx(&cfg, umma_probe_kernel<2>, p));
    else CUDA_TRY(cudaLaunchKernelEx(&cfg, umma_probe_kernel<1>, p));
    CUDA_TRY(cudaEventRecord(e1, 0));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    if (rep > 0 && ms < best) best = ms;
  }
  std::vector<unsigned long long> cyc(grid);
  CUDA_TRY(cudaMemcpy(cyc.data(), d_cyc, sizeof(unsigned long long) * grid, cudaMemcpyDeviceToHost));
  unsigned long long mx = 0;
  for (auto c : cyc) mx = std::max(mx, c);
  cudaFree(d_cyc);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (out_ms) *out_ms = best;
  if (out_cycles) *out_cycles = (double)mx;
  return 0;
}

int64_t dcscn_launch_count(dcscn_handle* h) { return h ? h->launches : 0; }
int64_t dcscn_device_bytes(dcscn_handle* h) { return h ? h->device_bytes : 0; }
int64_t dcscn_graph_replays(dcscn_handle* h) { return h ? h->graph_replays : 0; }

}  // extern "C"
