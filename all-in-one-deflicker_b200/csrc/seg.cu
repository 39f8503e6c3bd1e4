// Segmentation variant of the stage-1 loop (src/stage1_neural_atlas_seg.py:207-315 of the reference): entry points
// b200_seg_* and the generic mapping pre-training step.  The iteration is a fixed sequence of stream-ordered launches:
//
//   sample (9 coordinate-row groups per pixel, flow-match groups compacted)            atlas_kernels.cu
//   -> mapping1, mapping2 on all 9 groups, alpha on 5 groups                           b200_mlp_forward
//   -> atlas on 6 groups (layer 1: uv1*0.5+0.5, layer 2: uv2*0.5-0.5)                  b200_mlp_forward
//   -> fused loss head: every loss term and d/d(network outputs)                       seg_loss_kernel
//   -> atlas backward (+ input gradient chained into d uv1 / d uv2), alpha, mapping2, mapping1 backward
//
// Networks whose shape has tensor-core kernels run on them when the configuration asks for B200_PREC_TC.
#include "atlas_internal.cuh"
#include "seg_loss_math.h"
#include "tc_api.cuh"

namespace b200 {

static inline float half_of_i(int v) { return (float)((double)v / 2.0); }

static char* carve_seg(char*& p, int64_t bytes) {
  char* r = p;
  p += round_up(bytes, 256);
  return r;
}

struct SegNet {
  MlpShape s;
  int prec = B200_PREC_FP32;
  int64_t p_off = 0;          // float offset of this network in the flat parameter buffer
  char* ws = nullptr;         // its b200_mlp_forward / backward workspace
  int64_t ws_bytes = 0;
};

struct SegPlan {
  int cap = 0;
  int* counters = nullptr;
  float* x_map = nullptr;     // [9*cap][4]
  float* targets = nullptr;   // [cap][12]
  float* x3 = nullptr;        // [9*cap][3]   mapping inputs
  float* xa = nullptr;        // [5*cap][3]   alpha inputs
  float* xat = nullptr;       // [6*cap][2]   atlas inputs
  float* uv1 = nullptr, *uv2 = nullptr;       // [9*cap][2]
  float* ar = nullptr;        // [5*cap]
  float* yat = nullptr;       // [6*cap][3]
  float* d_uv1 = nullptr, *d_uv2 = nullptr, *d_ar = nullptr, *d_yat = nullptr, *d_xat = nullptr;
  SegNet net[4];              // mapping1, mapping2, alpha, atlas
  int64_t total_params = 0;
  int64_t bytes = 0;
};

static const int kNetRows[4] = {G_COUNT, G_COUNT, A_COUNT, SEG_ATLAS_ROWS};   // row groups each network evaluates

static int plan_seg(const B200SegConfig* cfg, char* base, SegPlan* pl) {
  B200_REQUIRE(cfg && cfg->batch > 0 && cfg->batch <= 16384, "samples_batch must be in [1, 16384]");
  B200_REQUIRE(cfg->precision == B200_PREC_FP32 || cfg->precision == B200_PREC_TC, "unknown precision %d", cfg->precision);
  B200_REQUIRE(cfg->uv_mapping_scale != 0.f && cfg->derivative_amount != 0.f && cfg->global_derivative_amount != 0.f,
               "uv_mapping_scale and the derivative amounts must be non-zero");
  const B200MlpDesc* descs[4] = {&cfg->mapping1, &cfg->mapping2, &cfg->alpha, &cfg->atlas};
  int64_t off = 0;
  for (int k = 0; k < 4; ++k) {
    B200_PROPAGATE(resolve_mlp(descs[k], &pl->net[k].s));
    pl->net[k].p_off = off;
    off += pl->net[k].s.total;
    pl->net[k].prec = mlp_precision(descs[k], cfg->precision);
  }
  pl->total_params = off;
  const MlpShape& m1 = pl->net[0].s; const MlpShape& m2 = pl->net[1].s;
  const MlpShape& al = pl->net[2].s; const MlpShape& at = pl->net[3].s;
  B200_REQUIRE(m1.in_dim == 3 && m1.out_dim == 2 && m2.in_dim == 3 && m2.out_dim == 2, "mapping networks are 3 -> 2");
  B200_REQUIRE(al.in_dim == 3 && al.out_dim == 1, "the alpha network is 3 -> 1");
  B200_REQUIRE(at.in_dim == 2 && at.out_dim == 3, "the atlas network is 2 -> 3");
  pl->cap = (int)round_up(cfg->batch, kTileRows);
  const int64_t cap = pl->cap;
  char* p = base;
  pl->counters = reinterpret_cast<int*>(carve_seg(p, 64));
  pl->x_map = reinterpret_cast<float*>(carve_seg(p, G_COUNT * cap * 16));
  pl->targets = reinterpret_cast<float*>(carve_seg(p, cap * TARGET_FLOATS * 4));
  pl->x3 = reinterpret_cast<float*>(carve_seg(p, G_COUNT * cap * 12));
  pl->xa = reinterpret_cast<float*>(carve_seg(p, A_COUNT * cap * 12));
  pl->xat = reinterpret_cast<float*>(carve_seg(p, SEG_ATLAS_ROWS * cap * 8));
  pl->uv1 = reinterpret_cast<float*>(carve_seg(p, G_COUNT * cap * 8));
  pl->uv2 = reinterpret_cast<float*>(carve_seg(p, G_COUNT * cap * 8));
  pl->ar = reinterpret_cast<float*>(carve_seg(p, A_COUNT * cap * 4));
  pl->yat = reinterpret_cast<float*>(carve_seg(p, SEG_ATLAS_ROWS * cap * 12));
  pl->d_uv1 = reinterpret_cast<float*>(carve_seg(p, G_COUNT * cap * 8));
  pl->d_uv2 = reinterpret_cast<float*>(carve_seg(p, G_COUNT * cap * 8));
  pl->d_ar = reinterpret_cast<float*>(carve_seg(p, A_COUNT * cap * 4));
  pl->d_yat = reinterpret_cast<float*>(carve_seg(p, SEG_ATLAS_ROWS * cap * 12));
  pl->d_xat = reinterpret_cast<float*>(carve_seg(p, SEG_ATLAS_ROWS * cap * 8));
  for (int k = 0; k < 4; ++k) {
    const int64_t rows = kNetRows[k] * cap;
    int64_t need = b200_mlp_workspace_bytes(descs[k], rows, 1);
    if (k == 3) need += rows * pl->net[k].s.enc * 4 + 512;       // input gradient of the atlas network
    pl->net[k].ws_bytes = round_up(need, 1024) + 1024;
    pl->net[k].ws = carve_seg(p, pl->net[k].ws_bytes);
  }
  pl->bytes = p - base;
  return B200_OK;
}

static int seg_prepare(const B200SegConfig* cfg, void* ws, int64_t ws_bytes, SegPlan* pl) {
  B200_REQUIRE(ws != nullptr, "null workspace");
  char* base = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 1024));
  B200_PROPAGATE(plan_seg(cfg, base, pl));
  if (base + pl->bytes > reinterpret_cast<char*>(ws) + ws_bytes) {
    set_error("workspace too small: need %lld bytes", (long long)(pl->bytes + 1024));
    return B200_ERR_WORKSPACE;
  }
  return B200_OK;
}

// x_map (float4 rows, 9 groups) -> packed 3-column inputs of the mapping networks (all groups) and of the alpha
// network (groups BASE, XP1, YP1, FWD, BWD)
__global__ void seg_pack_kernel(const float4* __restrict__ x_map, int cap, int64_t rows, float* __restrict__ x3,
                                float* __restrict__ xa) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float4 v = x_map[r];
  x3[r * 3 + 0] = v.x; x3[r * 3 + 1] = v.y; x3[r * 3 + 2] = v.z;
  if (xa) {
    const int g = (int)(r / cap);
    const int k = g < 3 ? g : (g == G_FWD ? A_FWD : (g == G_BWD ? A_BWD : -1));
    if (k >= 0) {
      float* d = xa + ((int64_t)k * cap + (r % cap)) * 3;
      d[0] = v.x; d[1] = v.y; d[2] = v.z;
    }
  }
}

// atlas inputs: rows [0, 3 cap) = uv1 * 0.5 + 0.5 (foreground quadrant), rows [3 cap, 6 cap) = uv2 * 0.5 - 0.5
__global__ void seg_atlas_in_kernel(const float* __restrict__ uv1, const float* __restrict__ uv2, int64_t rows_per_layer,
                                    float* __restrict__ xat) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * rows_per_layer) return;
  const bool second = i >= rows_per_layer;
  const float2 v = reinterpret_cast<const float2*>(second ? uv2 : uv1)[second ? i - rows_per_layer : i];
  const float sh = second ? -0.5f : 0.5f;
  reinterpret_cast<float2*>(xat)[i] = make_float2(__fadd_rn(v.x * 0.5f, sh), __fadd_rn(v.y * 0.5f, sh));
}

// d uv += 0.5 * d(atlas input) for the three colour groups of both layers
__global__ void seg_chain_kernel(const float* __restrict__ d_xat, int64_t rows_per_layer, float* __restrict__ d_uv1,
                                 float* __restrict__ d_uv2) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * rows_per_layer) return;
  const bool second = i >= rows_per_layer;
  const float2 g = reinterpret_cast<const float2*>(d_xat)[i];
  float2* d = reinterpret_cast<float2*>(second ? d_uv2 : d_uv1) + (second ? i - rows_per_layer : i);
  float2 v = *d;
  v.x += 0.5f * g.x; v.y += 0.5f * g.y;
  *d = v;
}

__global__ void seg_loss_kernel(const float* __restrict__ uv1, const float* __restrict__ uv2, const float* __restrict__ ar,
                                const float* __restrict__ yat, const float* __restrict__ targets,
                                const float* __restrict__ mask, const int64_t* __restrict__ indices,
                                const int* __restrict__ counters, int cap, int batch, SegLossConfig cfg,
                                float* __restrict__ d_uv1, float* __restrict__ d_uv2, float* __restrict__ d_ar,
                                float* __restrict__ d_yat, float* __restrict__ losses) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  const int n_f = counters[1], n_b = counters[2], n_lf = counters[5], n_lb = counters[6];
  cfg.inv_nf = n_f > 0 ? 1.0f / (float)n_f : 0.f;
  cfg.inv_nb = n_b > 0 ? 1.0f / (float)n_b : 0.f;
  float part[SV_COUNT];
#pragma unroll
  for (int k = 0; k < SV_COUNT; ++k) part[k] = 0.f;
  if (s < cap) {
    SegSampleOut out;
    int pf = -1, pb = -1;
    if (s < batch) {
      SegSampleIn in;
      const float* tg = targets + (int64_t)s * TARGET_FLOATS;
      pf = (int)tg[9] - 1; pb = (int)tg[10] - 1;
#pragma unroll
      for (int g = 0; g < G_COUNT; ++g) {
        const int r = g == G_FWD ? pf : (g == G_BWD ? pb : s);
        if (r >= 0) {
          const float2 a = *reinterpret_cast<const float2*>(uv1 + ((int64_t)g * cap + r) * 2);
          const float2 b = *reinterpret_cast<const float2*>(uv2 + ((int64_t)g * cap + r) * 2);
          in.uv1[g][0] = a.x; in.uv1[g][1] = a.y; in.uv2[g][0] = b.x; in.uv2[g][1] = b.y;
        } else { in.uv1[g][0] = in.uv1[g][1] = in.uv2[g][0] = in.uv2[g][1] = 0.f; }
      }
#pragma unroll
      for (int k = 0; k < A_COUNT; ++k) {
        const int r = k == A_FWD ? pf : (k == A_BWD ? pb : s);
        in.ar[k] = r >= 0 ? ar[(int64_t)k * cap + r] : 0.f;
      }
#pragma unroll
      for (int k = 0; k < SEG_ATLAS_ROWS; ++k)
#pragma unroll
        for (int c = 0; c < 3; ++c) in.y[k][c] = yat[((int64_t)k * cap + s) * 3 + c];
#pragma unroll
      for (int c = 0; c < 3; ++c) { in.rgb[c] = tg[c]; in.dx[c] = tg[3 + c]; in.dy[c] = tg[6 + c]; }
      in.a_gt = mask[indices[s]];
      in.wf = pf >= 0 ? 1.f : 0.f; in.wb = pb >= 0 ? 1.f : 0.f;
      seg_sample_loss(in, cfg, out);
#pragma unroll
      for (int k = 0; k < SV_COUNT; ++k) part[k] = out.val[k];
    } else {
#pragma unroll
      for (int g = 0; g < G_COUNT; ++g) out.duv1[g][0] = out.duv1[g][1] = out.duv2[g][0] = out.duv2[g][1] = 0.f;
#pragma unroll
      for (int k = 0; k < A_COUNT; ++k) out.dar[k] = 0.f;
#pragma unroll
      for (int k = 0; k < SEG_ATLAS_ROWS; ++k)
#pragma unroll
        for (int c = 0; c < 3; ++c) out.dy[k][c] = 0.f;
    }
#pragma unroll
    for (int g = 0; g < G_COUNT; ++g) {
      if (g == G_FWD || g == G_BWD) {
        // this sample's compacted row; as slot owner, zero for the rows past the group's count
        const int r = g == G_FWD ? pf : pb, n_rows = g == G_FWD ? n_lf : n_lb;
        if (r >= 0) {
          *reinterpret_cast<float2*>(d_uv1 + ((int64_t)g * cap + r) * 2) = make_float2(out.duv1[g][0], out.duv1[g][1]);
          *reinterpret_cast<float2*>(d_uv2 + ((int64_t)g * cap + r) * 2) = make_float2(out.duv2[g][0], out.duv2[g][1]);
        }
        if (s >= n_rows) {
          *reinterpret_cast<float2*>(d_uv1 + ((int64_t)g * cap + s) * 2) = make_float2(0.f, 0.f);
          *reinterpret_cast<float2*>(d_uv2 + ((int64_t)g * cap + s) * 2) = make_float2(0.f, 0.f);
        }
      } else {
        *reinterpret_cast<float2*>(d_uv1 + ((int64_t)g * cap + s) * 2) = make_float2(out.duv1[g][0], out.duv1[g][1]);
        *reinterpret_cast<float2*>(d_uv2 + ((int64_t)g * cap + s) * 2) = make_float2(out.duv2[g][0], out.duv2[g][1]);
      }
    }
#pragma unroll
    for (int k = 0; k < A_COUNT; ++k) {
      if (k == A_FWD || k == A_BWD) {
        const int r = k == A_FWD ? pf : pb, n_rows = k == A_FWD ? n_lf : n_lb;
        if (r >= 0) d_ar[(int64_t)k * cap + r] = out.dar[k];
        if (s >= n_rows) d_ar[(int64_t)k * cap + s] = 0.f;
      } else {
        d_ar[(int64_t)k * cap + s] = out.dar[k];
      }
    }
#pragma unroll
    for (int k = 0; k < SEG_ATLAS_ROWS; ++k)
#pragma unroll
      for (int c = 0; c < 3; ++c) d_yat[((int64_t)k * cap + s) * 3 + c] = out.dy[k][c];
  }
  // block reduction of the partial sums -> atomics on the loss vector
  __shared__ float red[SV_COUNT][4];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < SV_COUNT; ++q) {
    float v = part[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[q][wid] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float t[SV_COUNT];
    for (int q = 0; q < SV_COUNT; ++q) {
      float v = 0.f;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += red[q][w];
      t[q] = v;
    }
    const float ib = cfg.inv_batch;
    const float l_rgb = t[SV_RGB] * ib, l_grad = t[SV_GRAD] * ib, l_sp = t[SV_SPARSITY] * ib;
    const float l_r1 = t[SV_RIG1] * ib, l_r2 = t[SV_RIG2] * ib, l_g1 = t[SV_RIGG1] * ib, l_g2 = t[SV_RIGG2] * ib;
    float l_f1 = 0.5f * (t[SV_FLOW1_F] * cfg.inv_nf + t[SV_FLOW1_B] * cfg.inv_nb);
    float l_f2 = 0.5f * (t[SV_FLOW2_F] * cfg.inv_nf + t[SV_FLOW2_B] * cfg.inv_nb);
    float l_fa = 0.5f * (t[SV_AFLOW_F] * cfg.inv_nf + t[SV_AFLOW_B] * cfg.inv_nb);
    const float l_bce = t[SV_BCE] * ib;
    // the mean over an empty set is NaN in the reference (loss value only; gradients stay finite)
    if (blockIdx.x == 0 && (n_f == 0 || n_b == 0)) l_f1 = l_f2 = l_fa = nanf("");
    atomicAdd(losses + 1, l_rgb); atomicAdd(losses + 2, l_grad); atomicAdd(losses + 3, l_sp);
    atomicAdd(losses + 4, l_r1); atomicAdd(losses + 5, l_r2); atomicAdd(losses + 6, l_g1); atomicAdd(losses + 7, l_g2);
    atomicAdd(losses + 8, l_f1); atomicAdd(losses + 9, l_f2); atomicAdd(losses + 10, l_fa); atomicAdd(losses + 11, l_bce);
    atomicAdd(losses + 0, cfg.c_rig * (l_r1 + l_r2) + cfg.c_rig_global1 * l_g1 + cfg.c_rig_global2 * l_g2 +
                              cfg.c_rgb * l_rgb + cfg.c_flow * (l_f1 + l_f2) + cfg.c_boot * l_bce +
                              cfg.c_alpha_flow * l_fa + cfg.c_sparsity * l_sp + cfg.c_grad * l_grad);
    if (blockIdx.x == 0) { losses[12] = (float)n_f; losses[13] = (float)n_b; }
  }
}

// composite of the reconstruction (evaluate.py:320-335): rows [0, count) of layer 1, [rows_pad, rows_pad + count) of layer 2
__global__ void seg_compose_kernel(const float* __restrict__ yat, const float* __restrict__ ar, int64_t count,
                                   int64_t rows_pad, float* __restrict__ rgb, uint8_t* __restrict__ u8,
                                   float* __restrict__ alpha) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const float a = seg_alpha(ar[i]);
  if (alpha) alpha[i] = a;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float c1 = (yat[i * 3 + c] + 1.0f) * 0.5f, c2 = (yat[(rows_pad + i) * 3 + c] + 1.0f) * 0.5f;
    const float o = __fadd_rn(__fmul_rn(c1, a), __fmul_rn(c2, __fsub_rn(1.0f, a)));
    if (rgb) rgb[i * 3 + c] = o;
    if (u8) u8[i * 3 + c] = (uint8_t)(int)((double)o * 255.0);
  }
}

}  // namespace b200

using namespace b200;

extern "C" {

int64_t b200_seg_param_floats(const B200SegConfig* cfg, int64_t* offsets) {
  if (!cfg) return -1;
  const B200MlpDesc* descs[4] = {&cfg->mapping1, &cfg->mapping2, &cfg->alpha, &cfg->atlas};
  int64_t off = 0;
  for (int k = 0; k < 4; ++k) {
    const int64_t n = b200_mlp_layout(descs[k], nullptr, nullptr);
    if (n < 0) return -1;
    if (offsets) offsets[k] = off;
    off += n;
  }
  return off;
}

int64_t b200_seg_workspace_bytes(const B200SegConfig* cfg) {
  SegPlan pl;
  if (plan_seg(cfg, nullptr, &pl) != B200_OK) return -1;
  return pl.bytes + 2048;
}

int b200_seg_loss_grad(const B200SegConfig* cfg, const B200Video* video, const float* mask, const int64_t* indices,
                       const float* params, float* grads, float* losses, void* ws, int64_t ws_bytes, void* stream) {
  B200_REQUIRE(cfg && video && mask && indices && params && grads && losses, "null pointer");
  B200_REQUIRE(video->records && video->H > 0 && video->W > 0 && video->T > 0, "empty video");
  B200_REQUIRE(video->t_begin == 0 && video->t_end == video->T, "the segmentation variant needs the whole video resident");
  SegPlan pl;
  B200_PROPAGATE(seg_prepare(cfg, ws, ws_bytes, &pl));
  // the caller keeps `ws`, `params` and `grads` across trips: the networks' job tables are cached after the first
  // (eager) trip, which also makes the whole trip graph-capturable
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int cap = pl.cap, B = cfg->batch;
  const B200MlpDesc* descs[4] = {&cfg->mapping1, &cfg->mapping2, &cfg->alpha, &cfg->atlas};
  B200_CHECK_CUDA(cudaMemsetAsync(grads, 0, (size_t)pl.total_params * 4, st));
  B200_CHECK_CUDA(cudaMemsetAsync(losses, 0, B200_SEG_LOSS_FLOATS * 4, st));
  B200_CHECK_CUDA(cudaMemsetAsync(pl.x_map, 0, (size_t)G_COUNT * cap * 16, st));   // rows past the flow counts stay finite
  const int larger = video->W > video->H ? video->W : video->H;
  SampleGeom geo;
  geo.half_larger = half_of_i(larger);
  geo.half_resx = half_of_i(cfg->resx);
  geo.half_frames = (float)((double)video->T / 2.0);
  geo.d_local = cfg->derivative_amount;
  geo.d_global = cfg->global_derivative_amount;
  // without the global rigidity term the two D-offset groups are neither produced nor evaluated
  const int n_groups = cfg->with_global ? G_COUNT : G_YMG;
  B200_PROPAGATE(launch_select_sample(indices, B, *video, geo, cap, n_groups, pl.counters, nullptr, pl.x_map, pl.targets, st));
  const int64_t map_rows = (int64_t)n_groups * cap;
  seg_pack_kernel<<<(unsigned)((map_rows + 255) / 256), 256, 0, st>>>(reinterpret_cast<const float4*>(pl.x_map), cap,
                                                                     map_rows, pl.x3, pl.xa);
  B200_CHECK_LAUNCH();
  float* const ins[4] = {pl.x3, pl.x3, pl.xa, pl.xat};
  float* const outs[4] = {pl.uv1, pl.uv2, pl.ar, pl.yat};
  float* const douts[4] = {pl.d_uv1, pl.d_uv2, pl.d_ar, pl.d_yat};
  const int64_t net_rows[4] = {map_rows, map_rows, (int64_t)A_COUNT * cap, (int64_t)SEG_ATLAS_ROWS * cap};
  for (int k = 0; k < 3; ++k)
    B200_PROPAGATE(mlp_forward(descs[k], params + pl.net[k].p_off, ins[k], outs[k], net_rows[k], 1, pl.net[k].prec,
                               pl.net[k].ws, pl.net[k].ws_bytes, stream, true));
  const int64_t layer_rows = 3ll * cap;
  seg_atlas_in_kernel<<<(unsigned)((2 * layer_rows + 255) / 256), 256, 0, st>>>(pl.uv1, pl.uv2, layer_rows, pl.xat);
  B200_CHECK_LAUNCH();
  B200_PROPAGATE(mlp_forward(descs[3], params + pl.net[3].p_off, pl.xat, pl.yat, (int64_t)SEG_ATLAS_ROWS * cap, 1,
                             pl.net[3].prec, pl.net[3].ws, pl.net[3].ws_bytes, stream, true));
  SegLossConfig lc;
  lc.larger_dim = (float)larger; lc.uv_scale = cfg->uv_mapping_scale;
  lc.d_local = cfg->derivative_amount; lc.d_global = cfg->global_derivative_amount;
  lc.c_rgb = cfg->rgb_coeff; lc.c_grad = cfg->gradient_coeff; lc.c_rig = cfg->rigidity_coeff;
  lc.c_rig_global1 = cfg->global_rigidity_coeff_fg; lc.c_rig_global2 = cfg->global_rigidity_coeff_bg;
  lc.c_flow = cfg->flow_coeff; lc.c_alpha_flow = cfg->alpha_flow_factor; lc.c_sparsity = cfg->sparsity_coeff;
  lc.c_boot = cfg->bootstrapping_factor; lc.with_global = cfg->with_global != 0;
  lc.inv_batch = 1.0f / (float)B; lc.inv_nf = lc.inv_nb = 0.f;
  seg_loss_kernel<<<(cap + 127) / 128, 128, 0, st>>>(pl.uv1, pl.uv2, pl.ar, pl.yat, pl.targets, mask, indices, pl.counters,
                                                      cap, B, lc, pl.d_uv1, pl.d_uv2, pl.d_ar, pl.d_yat, losses);
  B200_CHECK_LAUNCH();
  // backward: atlas first (its input gradient feeds both mappings), then the other three networks
  B200_PROPAGATE(mlp_backward(descs[3], params + pl.net[3].p_off, pl.xat, pl.d_yat, grads + pl.net[3].p_off, pl.d_xat,
                              (int64_t)SEG_ATLAS_ROWS * cap, pl.net[3].prec, pl.net[3].ws, pl.net[3].ws_bytes, stream, true));
  seg_chain_kernel<<<(unsigned)((2 * layer_rows + 255) / 256), 256, 0, st>>>(pl.d_xat, layer_rows, pl.d_uv1, pl.d_uv2);
  B200_CHECK_LAUNCH();
  for (int k = 2; k >= 0; --k)
    B200_PROPAGATE(mlp_backward(descs[k], params + pl.net[k].p_off, ins[k], douts[k], grads + pl.net[k].p_off, nullptr,
                                net_rows[k], pl.net[k].prec, pl.net[k].ws, pl.net[k].ws_bytes, stream, true));
  return B200_OK;
}

// ---- generic pre-training step of a mapping-shaped IMLP ---------------------------------------------------------
struct PretrainPlan { int cap; int* counters; float* x_map; float* x3; float* uv; float* d_uv; char* ws; int64_t ws_bytes; int64_t bytes; };

static int plan_pretrain(const B200MlpDesc* d, int batch, char* base, PretrainPlan* pl) {
  MlpShape s;
  B200_PROPAGATE(resolve_mlp(d, &s));
  B200_REQUIRE(s.in_dim == 3 && s.out_dim == 2, "pre-training is defined for mapping networks (3 -> 2)");
  B200_REQUIRE(batch > 0 && batch <= 16384, "batch must be in [1, 16384]");
  pl->cap = (int)round_up(batch, kTileRows);
  const int64_t cap = pl->cap;
  char* p = base;
  pl->counters = reinterpret_cast<int*>(carve_seg(p, 64));
  pl->x_map = reinterpret_cast<float*>(carve_seg(p, cap * 16));
  pl->x3 = reinterpret_cast<float*>(carve_seg(p, cap * 12));
  pl->uv = reinterpret_cast<float*>(carve_seg(p, cap * 8));
  pl->d_uv = reinterpret_cast<float*>(carve_seg(p, cap * 8));
  pl->ws_bytes = round_up(b200_mlp_workspace_bytes(d, cap, 1), 1024) + 1024;
  pl->ws = carve_seg(p, pl->ws_bytes);
  pl->bytes = p - base;
  return B200_OK;
}

int64_t b200_mlp_pretrain_workspace_bytes(const B200MlpDesc* d, int32_t batch) {
  PretrainPlan pl;
  if (plan_pretrain(d, batch, nullptr, &pl) != B200_OK) return -1;
  return pl.bytes + 2048;
}

int b200_mlp_pretrain_loss_grad(const B200MlpDesc* d, int32_t batch, float uv_mapping_scale, int32_t larger_dim, int32_t T,
                                int32_t frame, const int64_t* ys, const int64_t* xs, const float* params, float* grads,
                                float* losses, int precision, void* ws, int64_t ws_bytes, void* stream) {
  B200_REQUIRE(d && ys && xs && params && grads && losses && ws, "null pointer");
  B200_REQUIRE(larger_dim > 0 && T > 0 && frame >= 0, "bad geometry");
  PretrainPlan pl;
  char* base = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 1024));
  B200_PROPAGATE(plan_pretrain(d, batch, base, &pl));
  if (base + pl.bytes > reinterpret_cast<char*>(ws) + ws_bytes) {
    set_error("workspace too small: need %lld bytes", (long long)(pl.bytes + 1024));
    return B200_ERR_WORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t total = b200_mlp_layout(d, nullptr, nullptr);
  const int prec = mlp_precision(d, precision);
  B200_CHECK_CUDA(cudaMemsetAsync(grads, 0, (size_t)total * 4, st));
  B200_CHECK_CUDA(cudaMemsetAsync(losses, 0, 4, st));
  const float t_norm = (float)((double)frame / ((double)T / 2.0) - 1.0);     // unwrap_utils.py:189
  B200_PROPAGATE(launch_pretrain_sample(ys, xs, batch, pl.cap, half_of_i(larger_dim), t_norm, pl.x_map, pl.counters, st));
  seg_pack_kernel<<<(unsigned)((pl.cap + 255) / 256), 256, 0, st>>>(reinterpret_cast<const float4*>(pl.x_map), pl.cap,
                                                                    pl.cap, pl.x3, nullptr);
  B200_CHECK_LAUNCH();
  B200_PROPAGATE(mlp_forward(d, params, pl.x3, pl.uv, pl.cap, 1, prec, pl.ws, pl.ws_bytes, stream, true));
  B200_PROPAGATE(launch_pretrain_loss(pl.x_map, pl.uv, batch, pl.cap, uv_mapping_scale, pl.d_uv, losses, pl.counters, st));
  B200_PROPAGATE(mlp_backward(d, params, pl.x3, pl.d_uv, grads, nullptr, pl.cap, prec, pl.ws, pl.ws_bytes, stream, true));
  return B200_OK;
}

// ---- reconstruction ----------------------------------------------------------------------------------------------
struct SegRenderPlan { int64_t rows_pad; float* x_map; float* x3; float* uv1; float* uv2; float* ar; float* xat; float* yat;
                       char* ws; int64_t ws_bytes; int64_t bytes; };

static int plan_seg_render(const B200SegConfig* cfg, int64_t pixels, char* base, SegRenderPlan* pl) {
  B200_REQUIRE(cfg && pixels > 0 && pixels <= (1ll << 24), "pixel count out of range");
  const B200MlpDesc* descs[4] = {&cfg->mapping1, &cfg->mapping2, &cfg->alpha, &cfg->atlas};
  const int64_t rp = round_up(pixels, kTileRows);
  pl->rows_pad = rp;
  char* p = base;
  pl->x_map = reinterpret_cast<float*>(carve_seg(p, rp * 16));
  pl->x3 = reinterpret_cast<float*>(carve_seg(p, rp * 12));
  pl->uv1 = reinterpret_cast<float*>(carve_seg(p, rp * 8));
  pl->uv2 = reinterpret_cast<float*>(carve_seg(p, rp * 8));
  pl->ar = reinterpret_cast<float*>(carve_seg(p, rp * 4));
  pl->xat = reinterpret_cast<float*>(carve_seg(p, 2 * rp * 8));
  pl->yat = reinterpret_cast<float*>(carve_seg(p, 2 * rp * 12));
  int64_t need = 0;
  for (int k = 0; k < 4; ++k) {
    const int64_t n = b200_mlp_workspace_bytes(descs[k], k == 3 ? 2 * rp : rp, 0);
    B200_REQUIRE(n > 0, "invalid network descriptor");
    if (n > need) need = n;
  }
  pl->ws_bytes = round_up(need, 1024) + 1024;
  pl->ws = carve_seg(p, pl->ws_bytes);
  pl->bytes = p - base;
  return B200_OK;
}

int64_t b200_seg_render_workspace_bytes(const B200SegConfig* cfg, int64_t pixels) {
  SegRenderPlan pl;
  if (plan_seg_render(cfg, pixels, nullptr, &pl) != B200_OK) return -1;
  return pl.bytes + 2048;
}

int b200_seg_render(const B200SegConfig* cfg, const float* params, int32_t H, int32_t W, int32_t T, int32_t frame,
                    int64_t pix_begin, int64_t pix_end, float* rgb, uint8_t* rgb_u8, float* alpha, void* ws,
                    int64_t ws_bytes, void* stream) {
  B200_REQUIRE(cfg && params && ws && (rgb || rgb_u8 || alpha), "null pointer");
  B200_REQUIRE(H > 0 && W > 0 && T > 0 && frame >= 0 && pix_begin >= 0 && pix_end > pix_begin && pix_end <= (int64_t)H * W,
               "bad geometry");
  const int64_t count = pix_end - pix_begin;
  SegRenderPlan pl;
  char* base = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 1024));
  B200_PROPAGATE(plan_seg_render(cfg, count, base, &pl));
  if (base + pl.bytes > reinterpret_cast<char*>(ws) + ws_bytes) {
    set_error("workspace too small: need %lld bytes", (long long)(pl.bytes + 1024));
    return B200_ERR_WORKSPACE;
  }
  int64_t offs[4];
  B200_REQUIRE(b200_seg_param_floats(cfg, offs) > 0, "invalid network descriptor");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const B200MlpDesc* descs[4] = {&cfg->mapping1, &cfg->mapping2, &cfg->alpha, &cfg->atlas};
  int prec[4];
  for (int k = 0; k < 4; ++k) prec[k] = mlp_precision(descs[k], cfg->precision);
  const int larger = W > H ? W : H;
  const float t_norm = (float)((double)frame / ((double)T / 2.0) - 1.0);      // evaluate.py:311
  const int64_t rp = pl.rows_pad;
  B200_PROPAGATE(launch_render_rows(W, half_of_i(larger), t_norm, pix_begin, count, rp, pl.x_map, st));
  seg_pack_kernel<<<(unsigned)((rp + 255) / 256), 256, 0, st>>>(reinterpret_cast<const float4*>(pl.x_map), (int)rp, rp,
                                                                 pl.x3, nullptr);
  B200_CHECK_LAUNCH();
  float* const outs[3] = {pl.uv1, pl.uv2, pl.ar};
  for (int k = 0; k < 3; ++k)
    B200_PROPAGATE(mlp_forward(descs[k], params + offs[k], pl.x3, outs[k], rp, 0, prec[k], pl.ws, pl.ws_bytes, stream, true));
  seg_atlas_in_kernel<<<(unsigned)((2 * rp + 255) / 256), 256, 0, st>>>(pl.uv1, pl.uv2, rp, pl.xat);
  B200_CHECK_LAUNCH();
  B200_PROPAGATE(mlp_forward(descs[3], params + offs[3], pl.xat, pl.yat, 2 * rp, 0, prec[3], pl.ws, pl.ws_bytes, stream, true));
  seg_compose_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(pl.yat, pl.ar, count, rp, rgb, rgb_u8, alpha);
  B200_CHECK_LAUNCH();
  return B200_OK;
}

}  // extern "C"
