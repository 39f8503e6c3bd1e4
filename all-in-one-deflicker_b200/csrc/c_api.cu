// extern "C" entry points of libb200deflicker.so (include/b200_deflicker.h).
#include <stdarg.h>
#include <string.h>

#include "atlas_internal.cuh"
#include "loss_math.h"
#include "tc_api.cuh"

namespace b200 {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static long long g_launches = 0;
void count_launch() { ++g_launches; }

// one optional (start, stop) event pair per tagged launch site
static cudaEvent_t g_t0[8] = {}, g_t1[8] = {};

static void record_timer(cudaEvent_t ev, cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cs);
  if (cs == cudaStreamCaptureStatusActive) cudaEventRecordWithFlags(ev, st, cudaEventRecordExternal);
  else cudaEventRecord(ev, st);
}
void timer_begin(int tag, cudaStream_t st) { if (tag > 0 && tag < 8 && g_t0[tag]) record_timer(g_t0[tag], st); }
void timer_end(int tag, cudaStream_t st) { if (tag > 0 && tag < 8 && g_t1[tag]) record_timer(g_t1[tag], st); }

int resolve_mlp(const B200MlpDesc* d, MlpShape* s) {
  if (!d || !s) { set_error("null descriptor"); return B200_ERR_INVALID; }
  if (d->num_layers < 2 || d->num_layers > B200_MAX_LAYERS || d->input_dim < 1 || d->output_dim < 1 ||
      d->hidden_dim < 1 || d->pe_freqs < 0 || d->pe_freqs > 30) {
    set_error("invalid IMLP descriptor (layers=%d in=%d out=%d hidden=%d pe=%d)", d->num_layers, d->input_dim,
              d->output_dim, d->hidden_dim, d->pe_freqs);
    return B200_ERR_INVALID;
  }
  s->L = d->num_layers; s->in_dim = d->input_dim; s->out_dim = d->output_dim; s->hidden = d->hidden_dim;
  s->pe = d->pe_freqs; s->tanh_out = d->use_tanh != 0;
  s->enc = d->pe_freqs > 0 ? 2 * d->input_dim * d->pe_freqs : d->input_dim;   // implicit_neural_networks.py:32-36
  int64_t off = 0;
  for (int i = 0; i < s->L; ++i) {
    s->skip[i] = i > 0 && ((d->skip_mask >> i) & 1u);
    s->K[i] = i == 0 ? s->enc : (s->skip[i] ? s->hidden + s->enc : s->hidden);   // :40-45
    s->N[i] = i == s->L - 1 ? s->out_dim : s->hidden;
    s->w_off[i] = off; off = round_up(off + (int64_t)s->K[i] * s->N[i], 4);
    s->b_off[i] = off; off = round_up(off + s->N[i], 4);
  }
  s->total = off;
  return B200_OK;
}

const B200MlpDesc& mapping_desc() {   // src/stage1_neural_atlas.py:112-119 with config_flow_100.json
  static const B200MlpDesc d = {3, 2, 256, 6, 0, 0u, 1, 0};
  return d;
}
const B200MlpDesc& atlas_desc() {     // src/stage1_neural_atlas.py:121-128
  static const B200MlpDesc d = {2, 3, 256, 8, 10, (1u << 4) | (1u << 7), 1, 0};
  return d;
}

static char* carve(char*& p, int64_t bytes) {
  char* r = p;
  p += round_up(bytes, 256);
  return r;
}

int64_t plan_mlp_scratch(const MlpShape& s, int64_t rows, bool training, char* base, MlpScratch* out) {
  (void)training;
  char* p = base;
  MlpScratch sc{};
  for (int l = 0; l < s.L; ++l) {
    if (l == 0 && s.pe == 0) { sc.act[l] = nullptr; continue; }
    sc.act[l] = reinterpret_cast<float*>(carve(p, rows * s.K[l] * 4));
  }
  sc.y = reinterpret_cast<float*>(carve(p, rows * s.out_dim * 4));
  const int64_t wz = s.hidden > s.enc ? s.hidden : s.enc;
  sc.dz[0] = reinterpret_cast<float*>(carve(p, rows * wz * 4));
  sc.dz[1] = reinterpret_cast<float*>(carve(p, rows * wz * 4));
  sc.bytes = p - base;
  if (out) *out = sc;
  return sc.bytes;
}

// Workspace of one loop trip.
struct AtlasPlan {
  int cap = 0, n_groups = 0;
  int* counters = nullptr;     // [0] n_local [1] n_fwd [2] n_bwd
  int* list = nullptr;         // [cap]
  float* x_map = nullptr;      // [9*cap][4]
  float* targets = nullptr;    // [cap][TARGET_FLOATS]
  float* d_uv = nullptr;       // [9*cap][2]
  float* d_y = nullptr;        // [3*cap][3]
  float* d_pe = nullptr;       // [3*cap][enc]
  MlpScratch map, atlas;
  MlpShape ms, as;
  TcPlan tc;                   // tcgen05 operand buffers (precision == B200_PREC_TC)
  int64_t bytes = 0;
};

static int plan_atlas(const B200AtlasConfig* cfg, char* base, AtlasPlan* pl) {
  B200_REQUIRE(cfg && cfg->batch > 0 && cfg->batch <= 16384, "samples_batch must be in [1, 16384]");
  B200_PROPAGATE(resolve_mlp(&mapping_desc(), &pl->ms));
  B200_PROPAGATE(resolve_mlp(&atlas_desc(), &pl->as));
  pl->cap = (int)round_up(cfg->batch, kTileRows);
  pl->n_groups = G_COUNT;      // buffers always sized for the 9-group regime
  char* p = base;
  const int64_t cap = pl->cap;
  pl->counters = reinterpret_cast<int*>(carve(p, 64));
  pl->list = reinterpret_cast<int*>(carve(p, cap * 4));
  pl->x_map = reinterpret_cast<float*>(carve(p, G_COUNT * cap * 16));
  pl->targets = reinterpret_cast<float*>(carve(p, cap * TARGET_FLOATS * 4));
  pl->d_uv = reinterpret_cast<float*>(carve(p, G_COUNT * cap * 8));
  pl->d_y = reinterpret_cast<float*>(carve(p, 3 * cap * 12));
  pl->d_pe = reinterpret_cast<float*>(carve(p, 3 * cap * pl->as.enc * 4));
  if (cfg->precision == B200_PREC_FP32) {
    p += plan_mlp_scratch(pl->ms, G_COUNT * cap, true, p, &pl->map);
    p += plan_mlp_scratch(pl->as, 3 * cap, true, p, &pl->atlas);
  } else {
    // the tensor-core path keeps only the network outputs in fp32
    pl->map.y = reinterpret_cast<float*>(carve(p, G_COUNT * cap * 2 * 4));
    pl->atlas.y = reinterpret_cast<float*>(carve(p, 3 * cap * 3 * 4));
    p += tc_plan(pl->ms, pl->as, G_COUNT * cap, 3 * cap, p, &pl->tc);
  }
  pl->bytes = p - base;
  return B200_OK;
}

static inline float half_of(int v) { return (float)((double)v / 2.0); }

}  // namespace b200

using namespace b200;

extern "C" {

const char* b200_last_error(void) { return g_err; }
int b200_version(void) { return 100; }

long long b200_launch_count(void) { return g_launches; }

int b200_set_kernel_timer(void* ev_start, void* ev_stop, int tag) {
  if (tag == 0 && !ev_start && !ev_stop) {               // switch every site off
    for (int i = 0; i < 8; ++i) g_t0[i] = g_t1[i] = nullptr;
    return B200_OK;
  }
  B200_REQUIRE(tag > 0 && tag < 8, "unknown kernel tag %d", tag);
  g_t0[tag] = (ev_start && ev_stop) ? reinterpret_cast<cudaEvent_t>(ev_start) : nullptr;
  g_t1[tag] = (ev_start && ev_stop) ? reinterpret_cast<cudaEvent_t>(ev_stop) : nullptr;
  return B200_OK;
}

int b200_device_supports_tc(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}

int64_t b200_mlp_layout(const B200MlpDesc* d, int64_t* w_off, int64_t* b_off) {
  MlpShape s;
  if (resolve_mlp(d, &s) != B200_OK) return -1;
  for (int i = 0; i < s.L; ++i) {
    if (w_off) w_off[i] = s.w_off[i];
    if (b_off) b_off[i] = s.b_off[i];
  }
  return s.total;
}

// the tensor-core family of a descriptor as its ABI code: 1 mapping (6 or 4 layers), 2 atlas, 3 alpha, 0 none
int b200_mlp_tc_architecture(const B200MlpDesc* d) {
  MlpShape s;
  if (resolve_mlp(d, &s) != B200_OK) return -1;
  switch (tc_classify(s)) {
    case TcNet::Mapping6: case TcNet::Mapping4: return 1;
    case TcNet::Atlas: return 2;
    case TcNet::Alpha: return 3;
    default: return 0;
  }
}

// buffers of a stand-alone tensor-core call, carved from the caller's workspace
struct TcCallPlan { int* gmax2; float* x; float* y; float* dy; float* d_in; char* tc; int64_t bytes; };
static void plan_tc_call(const MlpShape& s, TcNet net, int64_t rows_pad, char* base, TcCallPlan* pl) {
  char* p = base;
  pl->gmax2 = reinterpret_cast<int*>(carve(p, 64));
  pl->x = reinterpret_cast<float*>(carve(p, rows_pad * 16));
  pl->y = reinterpret_cast<float*>(carve(p, rows_pad * s.out_dim * 4));
  pl->dy = reinterpret_cast<float*>(carve(p, rows_pad * s.out_dim * 4));
  pl->d_in = reinterpret_cast<float*>(carve(p, rows_pad * 8));
  pl->tc = p;
  pl->bytes = (p - base) + tc_single_workspace_bytes(s, net, rows_pad);
}

int64_t b200_mlp_workspace_bytes(const B200MlpDesc* d, int64_t rows, int training) {
  MlpShape s;
  if (resolve_mlp(d, &s) != B200_OK || rows < 0) return -1;
  const int64_t rows_pad = round_up(rows, kTileRows);
  int64_t need = plan_mlp_scratch(s, rows_pad, training != 0, nullptr, nullptr) + 256;
  const TcNet net = tc_classify(s);
  if (net != TcNet::None) {          // enough for either precision
    TcCallPlan pl;
    plan_tc_call(s, net, rows_pad, nullptr, &pl);
    if (pl.bytes + 2048 > need) need = pl.bytes + 2048;
  }
  return need;
}

static int tc_call_prepare(const B200MlpDesc* d, int64_t rows, void* ws, int64_t ws_bytes, MlpShape* s, TcNet* net,
                           int64_t* rows_pad, TcCallPlan* pl) {
  B200_PROPAGATE(resolve_mlp(d, s));
  *net = tc_classify(*s);
  B200_REQUIRE(*net != TcNet::None, "B200_PREC_TC serves the stage-1 architectures (mapping: 3-256x{2,4}-2 without encoding; alpha: 3-PE5-256x6-1; "
               "atlas: 2-PE10-256x6-3 with skips 4, 7); use B200_PREC_FP32 for other shapes");
  if (!b200_device_supports_tc()) { set_error("B200_PREC_TC needs a compute-capability 10.x device"); return B200_ERR_UNSUPPORTED; }
  B200_REQUIRE(rows > 0 && rows < (1ll << 26), "rows out of range: %lld", (long long)rows);
  B200_REQUIRE(ws != nullptr, "null workspace");
  *rows_pad = round_up(rows, kTileRows);
  char* base = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 1024));
  plan_tc_call(*s, *net, *rows_pad, base, pl);
  if (base + pl->bytes > reinterpret_cast<char*>(ws) + ws_bytes) {
    set_error("workspace too small: need %lld bytes", (long long)(pl->bytes + 2048));
    return B200_ERR_WORKSPACE;
  }
  return B200_OK;
}

static int mlp_prepare(const B200MlpDesc* d, int64_t rows, void* ws, int64_t ws_bytes, MlpShape* s,
                       MlpScratch* sc, RowSpan* span) {
  B200_PROPAGATE(resolve_mlp(d, s));
  B200_REQUIRE(rows > 0 && rows < (1ll << 31) / 512, "rows out of range: %lld", (long long)rows);
  B200_REQUIRE(ws != nullptr, "null workspace");
  char* base = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 256));
  const int64_t need = plan_mlp_scratch(*s, round_up(rows, kTileRows), true, base, sc);
  if (base + need > reinterpret_cast<char*>(ws) + ws_bytes) {
    set_error("workspace too small: need %lld bytes", (long long)(need + 256));
    return B200_ERR_WORKSPACE;
  }
  span->rows = rows; span->cap = 0; span->n_valid = nullptr;
  return B200_OK;
}

}  // extern "C"

namespace b200 {

int mlp_precision(const B200MlpDesc* d, int precision) {
  return (precision == B200_PREC_TC && b200_mlp_tc_architecture(d) > 0) ? B200_PREC_TC : B200_PREC_FP32;
}

int mlp_forward(const B200MlpDesc* d, const float* params, const float* x, float* y, int64_t rows, int training,
                int precision, void* ws, int64_t ws_bytes, void* stream, bool persistent) {
  MlpShape s; MlpScratch sc; RowSpan span;
  B200_REQUIRE(params && x && y, "null pointer");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (precision == B200_PREC_TC) {
    TcNet net; int64_t rows_pad; TcCallPlan pl;
    B200_PROPAGATE(tc_call_prepare(d, rows, ws, ws_bytes, &s, &net, &rows_pad, &pl));
    B200_PROPAGATE(launch_pack_rows(x, s.in_dim, s.in_dim, pl.x, net == TcNet::Atlas ? 2 : 4, rows, rows_pad, st));
    B200_PROPAGATE(tc_single_forward(s, net, params, pl.x, pl.y, rows_pad, training != 0, pl.tc, persistent, st));
    B200_CHECK_CUDA(cudaMemcpyAsync(y, pl.y, (size_t)rows * s.out_dim * 4, cudaMemcpyDeviceToDevice, st));
    return B200_OK;
  }
  B200_REQUIRE(precision == B200_PREC_FP32, "unknown precision %d", precision);
  B200_PROPAGATE(mlp_prepare(d, rows, ws, ws_bytes, &s, &sc, &span));
  if (s.pe > 0) {
    float* skips[B200_MAX_LAYERS]; int lds[B200_MAX_LAYERS]; int ns = 0;
    for (int l = 1; l < s.L; ++l) if (s.skip[l]) { skips[ns] = sc.act[l]; lds[ns] = s.K[l]; ++ns; }
    B200_PROPAGATE(launch_pe_forward(x, s.in_dim, 1.f, 0.f, s.in_dim, s.pe, sc.act[0], s.K[0], skips, lds, ns,
                                     s.hidden, span, st));
  } else {
    // skip layers concatenate the raw input
    for (int l = 1; l < s.L; ++l)
      if (s.skip[l])
        B200_CHECK_CUDA(cudaMemcpy2DAsync(sc.act[l] + s.hidden, (size_t)s.K[l] * 4, x, (size_t)s.in_dim * 4,
                                          (size_t)s.in_dim * 4, (size_t)rows, cudaMemcpyDeviceToDevice, st));
  }
  B200_PROPAGATE(simt_mlp_forward(s, params, x, s.in_dim, span, sc, sc.y, st));
  B200_CHECK_CUDA(cudaMemcpyAsync(y, sc.y, (size_t)rows * s.out_dim * 4, cudaMemcpyDeviceToDevice, st));
  return B200_OK;
}

int mlp_backward(const B200MlpDesc* d, const float* params, const float* x, const float* dy, float* dparams, float* dx,
                 int64_t rows, int precision, void* ws, int64_t ws_bytes, void* stream, bool persistent) {
  MlpShape s; MlpScratch sc; RowSpan span;
  B200_REQUIRE(params && dy && dparams && x, "null pointer");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (precision == B200_PREC_TC) {
    // the workspace still holds the padded input, the outputs and the activation images of the forward call
    TcNet net; int64_t rows_pad; TcCallPlan pl;
    B200_PROPAGATE(tc_call_prepare(d, rows, ws, ws_bytes, &s, &net, &rows_pad, &pl));
    const bool atlas = net == TcNet::Atlas;
    B200_REQUIRE(atlas || dx == nullptr, "the tensor-core mapping / alpha networks have no input gradient (their inputs "
                 "are pixel coordinates); use B200_PREC_FP32 when x requires grad");
    B200_PROPAGATE(launch_pack_rows(dy, s.out_dim, s.out_dim, pl.dy, s.out_dim, rows, rows_pad, st));
    B200_CHECK_CUDA(cudaMemsetAsync(pl.gmax2, 0, 8, st));
    B200_PROPAGATE(launch_absmax(pl.dy, rows_pad * s.out_dim, pl.gmax2 + (tc_pe_kernels(net) ? 0 : 1), st));
    B200_PROPAGATE(tc_single_backward(s, net, params, dparams, pl.x, pl.y, pl.dy, (atlas && dx) ? pl.d_in : nullptr,
                                      pl.gmax2, rows_pad, pl.tc, persistent, st));
    if (atlas && dx) B200_CHECK_CUDA(cudaMemcpyAsync(dx, pl.d_in, (size_t)rows * 8, cudaMemcpyDeviceToDevice, st));
    return B200_OK;
  }
  B200_REQUIRE(precision == B200_PREC_FP32, "unknown precision %d", precision);
  B200_PROPAGATE(mlp_prepare(d, rows, ws, ws_bytes, &s, &sc, &span));
  if (s.pe > 0) {
    // the encoded-input gradient is staged in a slice carved after the scratch
    float* d_enc = nullptr;
    char* extra = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 256)) + sc.bytes;
    if (dx) {
      const int64_t need = rows * s.enc * 4;
      if (extra + need > reinterpret_cast<char*>(ws) + ws_bytes) {
        set_error("workspace too small for the input gradient: need %lld more bytes", (long long)need);
        return B200_ERR_WORKSPACE;
      }
      d_enc = reinterpret_cast<float*>(extra);
    }
    B200_PROPAGATE(simt_mlp_backward(s, params, x, s.in_dim, span, sc, dy, dparams, d_enc, s.enc, st));
    if (dx) B200_PROPAGATE(launch_pe_backward(sc.act[0], s.K[0], d_enc, s.enc, s.in_dim, s.pe, 1.f, dx, s.in_dim,
                                              0, span, st));
  } else {
    B200_PROPAGATE(simt_mlp_backward(s, params, x, s.in_dim, span, sc, dy, dparams, dx, s.in_dim, st));
  }
  return B200_OK;
}

}  // namespace b200

extern "C" {

int b200_mlp_forward(const B200MlpDesc* d, const float* params, const float* x, float* y, int64_t rows,
                     int training, int precision, void* ws, int64_t ws_bytes, void* stream) {
  return mlp_forward(d, params, x, y, rows, training, precision, ws, ws_bytes, stream, false);
}

int b200_mlp_backward(const B200MlpDesc* d, const float* params, const float* x, const float* dy,
                      float* dparams, float* dx, int64_t rows, int precision, void* ws, int64_t ws_bytes,
                      void* stream) {
  return mlp_backward(d, params, x, dy, dparams, dx, rows, precision, ws, ws_bytes, stream, false);
}

int b200_video_pack(const float* frames, const float* frames_dx, const float* frames_dy, const float* flow_fwd,
                    const float* flow_bwd, const float* mask_fwd, const float* mask_bwd, int32_t H, int32_t W,
                    int32_t T, int32_t t_begin, int32_t t_end, float* records, uint32_t* mask_fwd_bits,
                    uint32_t* mask_bwd_bits, void* stream) {
  B200_REQUIRE(frames && frames_dx && frames_dy && flow_fwd && flow_bwd && mask_fwd && mask_bwd && records &&
               mask_fwd_bits && mask_bwd_bits, "null pointer");
  B200_REQUIRE(H > 0 && W > 0 && T > 0 && t_begin >= 0 && t_end <= T && t_begin <= t_end, "bad video extents");
  return launch_video_pack(frames, frames_dx, frames_dy, flow_fwd, flow_bwd, mask_fwd, mask_bwd, H, W, T, t_begin,
                           t_end, records, mask_fwd_bits, mask_bwd_bits, reinterpret_cast<cudaStream_t>(stream));
}

int64_t b200_atlas_param_floats(void) {
  MlpShape m, a;
  resolve_mlp(&mapping_desc(), &m);
  resolve_mlp(&atlas_desc(), &a);
  return m.total + a.total;
}

int64_t b200_atlas_workspace_bytes(const B200AtlasConfig* cfg) {
  AtlasPlan pl;
  if (plan_atlas(cfg, nullptr, &pl) != B200_OK) return -1;
  return pl.bytes + 256 + 2048;      // slack for the 256 / 1024-byte alignment of the real base address
}

int b200_atlas_workspace_offsets(const B200AtlasConfig* cfg, const void* ws, int64_t* offsets) {
  B200_REQUIRE(cfg && ws && offsets, "null pointer");
  AtlasPlan pl;
  char* base = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 256));
  B200_PROPAGATE(plan_atlas(cfg, base, &pl));
  const char* w = reinterpret_cast<const char*>(ws);
  offsets[0] = reinterpret_cast<char*>(pl.counters) - w;
  offsets[1] = reinterpret_cast<char*>(pl.list) - w;
  offsets[2] = reinterpret_cast<char*>(pl.x_map) - w;
  offsets[3] = reinterpret_cast<char*>(pl.targets) - w;
  offsets[4] = reinterpret_cast<char*>(pl.d_uv) - w;
  offsets[5] = reinterpret_cast<char*>(pl.d_y) - w;
  offsets[6] = reinterpret_cast<char*>(pl.map.y) - w;
  offsets[7] = reinterpret_cast<char*>(pl.atlas.y) - w;
  return B200_OK;
}

static int atlas_prepare(const B200AtlasConfig* cfg, void* ws, int64_t ws_bytes, AtlasPlan* pl) {
  B200_REQUIRE(ws != nullptr, "null workspace");
  char* base = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 256));
  B200_PROPAGATE(plan_atlas(cfg, base, pl));
  if (base + pl->bytes > reinterpret_cast<char*>(ws) + ws_bytes) {
    set_error("workspace too small: need %lld bytes", (long long)(pl->bytes + 256));
    return B200_ERR_WORKSPACE;
  }
  if (cfg->precision == B200_PREC_TC && !b200_device_supports_tc()) {
    set_error("B200_PREC_TC needs a compute-capability 10.x device");
    return B200_ERR_UNSUPPORTED;
  }
  B200_REQUIRE(cfg->precision == B200_PREC_FP32 || cfg->precision == B200_PREC_TC, "unknown precision %d",
               cfg->precision);
  return B200_OK;
}

int b200_atlas_loss_grad(const B200AtlasConfig* cfg, const B200Video* video, const int64_t* indices,
                         const float* params, float* grads, float* losses, void* ws, int64_t ws_bytes,
                         void* stream) {
  B200_REQUIRE(cfg && video && indices && params && grads && losses, "null pointer");
  B200_REQUIRE(video->records && video->mask_fwd_bits && video->mask_bwd_bits, "video not packed");
  B200_REQUIRE(video->H > 0 && video->W > 0 && video->T > 0 && video->t_begin >= 0 && video->t_end <= video->T,
               "bad video extents");
  AtlasPlan pl;
  B200_PROPAGATE(atlas_prepare(cfg, ws, ws_bytes, &pl));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int cap = pl.cap;
  const int ng = cfg->with_global ? G_COUNT : G_YMG;        // 9 or 7 row groups
  const int64_t n_params = pl.ms.total + pl.as.total;
  TcStep ts{};
  if (cfg->precision == B200_PREC_TC) {
    ts.ms = &pl.ms; ts.as = &pl.as; ts.plan = &pl.tc;
    ts.params = params; ts.grads = grads;
    ts.x_map = pl.x_map; ts.uv = pl.map.y; ts.y_atlas = pl.atlas.y;
    ts.d_uv = pl.d_uv; ts.d_y = pl.d_y;
    ts.cap = cap; ts.n_groups = ng; ts.counters = pl.counters; ts.flow_groups = 1;
    B200_PROPAGATE(tc_begin_step(ts, st));          // weight images on a side stream, under the sampling kernels
  }
  B200_CHECK_CUDA(cudaMemsetAsync(grads, 0, (size_t)n_params * 4, st));
  B200_CHECK_CUDA(cudaMemsetAsync(losses, 0, B200_LOSS_FLOATS * 4, st));

  const int larger = video->W > video->H ? video->W : video->H;
  SampleGeom geo;
  geo.half_larger = half_of(larger);
  geo.half_resx = half_of(cfg->resx > 0 ? cfg->resx : video->W);
  geo.half_frames = (float)((double)video->T / 2.0);
  geo.d_local = cfg->derivative_amount;
  geo.d_global = cfg->global_derivative_amount;
  B200_PROPAGATE(launch_select_sample(indices, cfg->batch, *video, geo, cap, ng, pl.counters, pl.list, pl.x_map,
                                      pl.targets, st));

  LossConfig lc{};
  lc.larger_dim = (float)larger;
  lc.uv_scale = cfg->uv_mapping_scale;
  lc.d_local = cfg->derivative_amount;
  lc.d_global = cfg->global_derivative_amount;
  lc.c_rgb = cfg->rgb_coeff; lc.c_grad = cfg->gradient_coeff; lc.c_rig = cfg->rigidity_coeff;
  lc.c_rig_global = cfg->with_global ? cfg->global_rigidity_coeff : 0.f;
  lc.c_flow = cfg->flow_coeff;
  lc.with_global = cfg->with_global;
  lc.inv_batch = 1.0f / (float)cfg->batch;

  RowSpan span_map{(int64_t)ng * cap, cap, pl.counters};
  RowSpan span_atl{(int64_t)3 * cap, cap, pl.counters};
  const float* p_map = params;
  const float* p_atl = params + pl.ms.total;
  float* g_map = grads;
  float* g_atl = grads + pl.ms.total;

  if (cfg->precision == B200_PREC_FP32) {
    B200_PROPAGATE(simt_mlp_forward(pl.ms, p_map, pl.x_map, 4, span_map, pl.map, pl.map.y, st));
    float* skips[2] = {pl.atlas.act[4], pl.atlas.act[7]};
    int lds[2] = {pl.as.K[4], pl.as.K[7]};
    B200_PROPAGATE(launch_pe_forward(pl.map.y, 2, 0.5f, 0.5f, 2, pl.as.pe, pl.atlas.act[0], pl.as.K[0], skips, lds,
                                     2, pl.as.hidden, span_atl, st));
    B200_PROPAGATE(simt_mlp_forward(pl.as, p_atl, nullptr, 0, span_atl, pl.atlas, pl.atlas.y, st));
    B200_PROPAGATE(launch_loss(pl.map.y, pl.atlas.y, pl.targets, pl.counters, cap, ng, lc, pl.d_uv, pl.d_y, losses,
                               st));
    B200_PROPAGATE(simt_mlp_backward(pl.as, p_atl, nullptr, 0, span_atl, pl.atlas, pl.d_y, g_atl, pl.d_pe,
                                     pl.as.enc, st));
    B200_PROPAGATE(launch_pe_backward(pl.atlas.act[0], pl.as.K[0], pl.d_pe, pl.as.enc, 2, pl.as.pe, 0.5f, pl.d_uv,
                                      2, 1, span_atl, st));
    B200_PROPAGATE(simt_mlp_backward(pl.ms, p_map, pl.x_map, 4, span_map, pl.map, pl.d_uv, g_map, nullptr, 0, st));
  } else {
    B200_PROPAGATE(tc_atlas_forward(ts, st));
    B200_PROPAGATE(launch_loss(pl.map.y, pl.atlas.y, pl.targets, pl.counters, cap, ng, lc, pl.d_uv, pl.d_y, losses,
                               st));
    B200_PROPAGATE(tc_atlas_backward(ts, st));
  }
  return B200_OK;
}

int b200_pretrain_loss_grad(const B200AtlasConfig* cfg, int32_t larger_dim, int32_t T, int32_t frame,
                            const int64_t* ys, const int64_t* xs, const float* params, float* grads,
                            float* losses, void* ws, int64_t ws_bytes, void* stream) {
  B200_REQUIRE(cfg && ys && xs && params && grads && losses, "null pointer");
  B200_REQUIRE(larger_dim > 0 && T > 0 && frame >= 0, "bad geometry");
  AtlasPlan pl;
  B200_PROPAGATE(atlas_prepare(cfg, ws, ws_bytes, &pl));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int cap = pl.cap;
  B200_CHECK_CUDA(cudaMemsetAsync(grads, 0, (size_t)pl.ms.total * 4, st));
  B200_CHECK_CUDA(cudaMemsetAsync(losses, 0, B200_LOSS_FLOATS * 4, st));
  // (f / (frames_num / 2.0) - 1) is a Python double, cast to fp32 by ones_like (unwrap_utils.py:189)
  const float t_norm = (float)((double)frame / ((double)T / 2.0) - 1.0);
  B200_PROPAGATE(launch_pretrain_sample(ys, xs, cfg->batch, cap, half_of(larger_dim), t_norm, pl.x_map,
                                        pl.counters, st));
  RowSpan span{(int64_t)cap, cap, pl.counters};
  if (cfg->precision == B200_PREC_FP32) {
    B200_PROPAGATE(simt_mlp_forward(pl.ms, params, pl.x_map, 4, span, pl.map, pl.map.y, st));
    B200_PROPAGATE(launch_pretrain_loss(pl.x_map, pl.map.y, cfg->batch, cap, cfg->uv_mapping_scale, pl.d_uv,
                                        losses, pl.counters, st));
    B200_PROPAGATE(simt_mlp_backward(pl.ms, params, pl.x_map, 4, span, pl.map, pl.d_uv, grads, nullptr, 0, st));
  } else {
    TcStep ts{};
    ts.ms = &pl.ms; ts.as = &pl.as; ts.plan = &pl.tc;
    ts.params = params; ts.grads = grads;
    ts.x_map = pl.x_map; ts.uv = pl.map.y; ts.d_uv = pl.d_uv;
    ts.cap = cap; ts.n_groups = 1; ts.counters = pl.counters;
    B200_PROPAGATE(tc_mapping_forward(ts, st));
    B200_PROPAGATE(launch_pretrain_loss(pl.x_map, pl.map.y, cfg->batch, cap, cfg->uv_mapping_scale, pl.d_uv,
                                        losses, pl.counters, st));
    B200_PROPAGATE(tc_mapping_backward(ts, st));
  }
  return B200_OK;
}

int b200_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, double lr,
                   double beta1, double beta2, double eps, float grad_scale, int64_t* step, void* stream) {
  B200_REQUIRE(params && grads && exp_avg && exp_avg_sq && step && n > 0, "null pointer / empty");
  B200_REQUIRE((reinterpret_cast<uintptr_t>(params) & 15) == 0 && (reinterpret_cast<uintptr_t>(grads) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(exp_avg) & 15) == 0 && (reinterpret_cast<uintptr_t>(exp_avg_sq) & 15) == 0,
               "buffers must be 16-byte aligned");
  return launch_adam(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, grad_scale, step,
                     reinterpret_cast<cudaStream_t>(stream));
}

int b200_debug_wgrad(long long* cycles_host, int32_t* shapes_host, int32_t max_ctas) {
  return tc_debug_wgrad(cycles_host, shapes_host, max_ctas);
}

int b200_dp_slice(int32_t world, int32_t rank, int64_t n_total, int64_t* begin, int64_t* count) {
  B200_REQUIRE(world >= 1 && world <= B200_MAX_RANKS && rank >= 0 && rank < world && n_total > 0 && begin && count,
               "bad slice request");
  const int64_t total4 = (n_total + 3) / 4, per = (total4 + world - 1) / world;
  const int64_t b4 = per * rank, e4 = per * (rank + 1) < total4 ? per * (rank + 1) : total4;
  *begin = b4 * 4 < n_total ? b4 * 4 : n_total;
  *count = e4 > b4 ? ((e4 * 4 < n_total ? e4 * 4 : n_total) - *begin) : 0;
  return B200_OK;
}

int b200_dp_adam_step(const B200DpComm* comm, float* exp_avg, float* exp_avg_sq, int64_t n_params, int64_t n_total,
                      double lr, double beta1, double beta2, double eps, int64_t* step, unsigned long long* epoch,
                      void* stream) {
  B200_REQUIRE(comm && exp_avg && exp_avg_sq && step && epoch, "null pointer");
  B200_REQUIRE(comm->world >= 1 && comm->world <= B200_MAX_RANKS && comm->rank >= 0 && comm->rank < comm->world,
               "bad communicator (world %d rank %d)", comm->world, comm->rank);
  B200_REQUIRE(n_params > 0 && n_params % 4 == 0 && n_total >= n_params, "n_params must be a positive multiple of 4");
  for (int j = 0; j < comm->world; ++j)
    B200_REQUIRE(comm->partials[j] && comm->params[j] && comm->flags[j] &&
                 (reinterpret_cast<uintptr_t>(comm->partials[j]) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(comm->params[j]) & 15) == 0, "peer buffer %d missing or misaligned", j);
  return launch_dp_adam(*comm, exp_avg, exp_avg_sq, n_params, n_total, lr, beta1, beta2, eps, step, epoch,
                        reinterpret_cast<cudaStream_t>(stream));
}

int64_t b200_render_workspace_bytes(int64_t pixels) {
  if (pixels <= 0) return -1;
  MlpShape m, a;
  resolve_mlp(&mapping_desc(), &m);
  resolve_mlp(&atlas_desc(), &a);
  const int64_t rows = round_up(pixels, kTileRows);
  const int64_t fp32_path = round_up(rows * 16, 256) + plan_mlp_scratch(m, rows, false, nullptr, nullptr) +
                            plan_mlp_scratch(a, rows, false, nullptr, nullptr) + 512;
  const int64_t tc_path = round_up(rows * 16, 256) + round_up(rows * 8, 256) + round_up(rows * 12, 256) +
                          tc_infer_workspace_bytes(m, a) + 1024;
  return fp32_path > tc_path ? fp32_path : tc_path;
}

int b200_render(const float* params, int32_t H, int32_t W, int32_t T, int32_t frame, int64_t pix_begin,
                int64_t pix_end, float* rgb, uint8_t* rgb_u8, int precision, void* ws, int64_t ws_bytes,
                void* stream) {
  B200_REQUIRE(params && ws && (rgb || rgb_u8), "null pointer");
  B200_REQUIRE(H > 0 && W > 0 && T > 0 && frame >= 0 && frame < T && pix_begin >= 0 && pix_end <= (int64_t)H * W &&
               pix_begin < pix_end, "bad render range");
  const int64_t count = pix_end - pix_begin;
  if (ws_bytes < b200_render_workspace_bytes(count)) {
    set_error("workspace too small: need %lld bytes", (long long)b200_render_workspace_bytes(count));
    return B200_ERR_WORKSPACE;
  }
  B200_REQUIRE(precision == B200_PREC_FP32 || precision == B200_PREC_TC, "unknown precision %d", precision);
  if (precision == B200_PREC_TC && !b200_device_supports_tc()) {
    set_error("B200_PREC_TC needs a compute-capability 10.x device");
    return B200_ERR_UNSUPPORTED;
  }
  MlpShape m, a;
  B200_PROPAGATE(resolve_mlp(&mapping_desc(), &m));
  B200_PROPAGATE(resolve_mlp(&atlas_desc(), &a));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t rows = round_up(count, kTileRows);
  char* p = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 256));
  float* x_map = reinterpret_cast<float*>(carve(p, rows * 16));
  const int larger = W > H ? W : H;
  const float t_norm = (float)((double)frame / ((double)T / 2.0) - 1.0);   // evaluate.py:657
  B200_PROPAGATE(launch_render_rows(W, half_of(larger), t_norm, pix_begin, count, rows, x_map, st));
  if (precision == B200_PREC_TC) {
    // the two fused tcgen05 forward kernels without their activation-image stores
    float* uv = reinterpret_cast<float*>(carve(p, rows * 8));
    float* y = reinterpret_cast<float*>(carve(p, rows * 12));
    B200_PROPAGATE(tc_infer_forward(m, a, params, x_map, uv, y, rows, p, st));
    B200_PROPAGATE(launch_render_out(y, count, rgb, rgb_u8, st));
    return B200_OK;
  }
  MlpScratch sm, sa;
  p += plan_mlp_scratch(m, rows, false, p, &sm);
  p += plan_mlp_scratch(a, rows, false, p, &sa);
  RowSpan span{rows, 0, nullptr};
  B200_PROPAGATE(simt_mlp_forward(m, params, x_map, 4, span, sm, sm.y, st));
  float* skips[2] = {sa.act[4], sa.act[7]};
  int lds[2] = {a.K[4], a.K[7]};
  B200_PROPAGATE(launch_pe_forward(sm.y, 2, 0.5f, 0.5f, 2, a.pe, sa.act[0], a.K[0], skips, lds, 2, a.hidden, span, st));
  B200_PROPAGATE(simt_mlp_forward(a, params + m.total, nullptr, 0, span, sa, sa.y, st));
  B200_PROPAGATE(launch_render_out(sa.y, count, rgb, rgb_u8, st));
  return B200_OK;
}

}  // extern "C"
