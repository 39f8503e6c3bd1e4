// Per-pixel evaluation maps of one frame — the quantities the reference's evaluation dashboards show
// (src/models/stage_1/evaluate.py:640-708): the mapping's uv, the rigidity loss of every pixel
// (`get_rigidity_loss(..., return_all=True)`, loss_utils.py:227-278) and its forward optical-flow error
// (`get_optical_flow_loss_all`, loss_utils.py:283-295 with get_corresponding_flow_matches_all :360-382).
// Four mapping evaluations per pixel — (x, y, t), (x, y-d, t), (x-d, y, t), (x+fx, y+fy, t+1) — as four row groups of
// ONE b200_mlp_forward call, then one head kernel.
#include "atlas_internal.cuh"
#include "loss_math.h"
#include "tc_api.cuh"

namespace b200 {

static char* carve_ev(char*& p, int64_t bytes) { char* r = p; p += round_up(bytes, 256); return r; }

__global__ void eval_rows_kernel(B200Video vid, int frame, int64_t pix_begin, int64_t count, int64_t rows_pad, float hL,
                                 float hT, float d, float* __restrict__ x3, float* __restrict__ valid) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= rows_pad) return;
  float r[4][3];
#pragma unroll
  for (int g = 0; g < 4; ++g) r[g][0] = r[g][1] = r[g][2] = 0.f;
  float ok = 0.f;
  if (s < count) {
    const int64_t p = pix_begin + s;
    const int x = (int)(p % vid.W), y = (int)(p / vid.W);
    const float fx = (float)x, fy = (float)y, ft = (float)frame;
    const float tn = norm_coord(ft, hT);
    const float* rec = vid.records + (((int64_t)(frame - vid.t_begin) * vid.H + y) * vid.W + x) * B200_RECORD_FLOATS;
    r[0][0] = norm_coord(fx, hL); r[0][1] = norm_coord(fy, hL); r[0][2] = tn;
    r[1][0] = norm_coord(fx, hL); r[1][1] = norm_coord(fy - d, hL); r[1][2] = tn;
    r[2][0] = norm_coord(fx - d, hL); r[2][1] = norm_coord(fy, hL); r[2][2] = tn;
    r[3][0] = norm_coord(__fadd_rn(fx, rec[9]), hL); r[3][1] = norm_coord(__fadd_rn(fy, rec[10]), hL);
    r[3][2] = norm_coord(ft + 1.f, hT);
    ok = rec[13] > 0.f ? 1.f : 0.f;
  }
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float* dst = x3 + ((int64_t)g * rows_pad + s) * 3;
    dst[0] = r[g][0]; dst[1] = r[g][1]; dst[2] = r[g][2];
  }
  valid[s] = ok;
}

__global__ void eval_head_kernel(const float* __restrict__ uv, const float* __restrict__ valid, int64_t count,
                                 int64_t rows_pad, float L, float uv_scale, float d, int last_frame,
                                 float* __restrict__ out_uv, float* __restrict__ out_rig, float* __restrict__ out_flow) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= count) return;
  float u[4][2];
#pragma unroll
  for (int g = 0; g < 4; ++g) { u[g][0] = uv[((int64_t)g * rows_pad + s) * 2]; u[g][1] = uv[((int64_t)g * rows_pad + s) * 2 + 1]; }
  if (out_uv) { out_uv[s * 2] = u[0][0]; out_uv[s * 2 + 1] = u[0][1]; }
  if (out_rig) {
    float g0[2] = {0.f, 0.f}, ga[2] = {0.f, 0.f}, gb[2] = {0.f, 0.f};
    out_rig[s] = rigidity_term(u[0], u[1], u[2], L, uv_scale, d, 0.f, g0, ga, gb);
  }
  if (out_flow) {
    // evaluate.py:689-695: zero for the last frame (no next frame); loss_utils.py:292: zero where the flow is invalid
    float v = 0.f;
    if (!last_frame && valid[s] != 0.f) {
      float g0[2] = {0.f, 0.f}, gm[2] = {0.f, 0.f};
      v = flow_term(u[0], u[3], L, uv_scale, 0.f, g0, gm);
    }
    out_flow[s] = v;
  }
}

struct EvalPlan { int64_t rows_pad; float* x3; float* valid; float* uv; char* ws; int64_t ws_bytes; int64_t bytes; };

static int plan_eval(const B200MlpDesc* d, int64_t pixels, char* base, EvalPlan* pl) {
  B200_REQUIRE(d && pixels > 0 && pixels <= (1ll << 24), "pixel count out of range");
  const int64_t rp = round_up(pixels, kTileRows);
  pl->rows_pad = rp;
  char* p = base;
  pl->x3 = reinterpret_cast<float*>(carve_ev(p, 4 * rp * 12));
  pl->valid = reinterpret_cast<float*>(carve_ev(p, rp * 4));
  pl->uv = reinterpret_cast<float*>(carve_ev(p, 4 * rp * 8));
  const int64_t need = b200_mlp_workspace_bytes(d, 4 * rp, 0);
  B200_REQUIRE(need > 0, "invalid mapping descriptor");
  pl->ws_bytes = round_up(need, 1024) + 1024;
  pl->ws = carve_ev(p, pl->ws_bytes);
  pl->bytes = p - base;
  return B200_OK;
}

}  // namespace b200

using namespace b200;

extern "C" {

int64_t b200_eval_maps_workspace_bytes(const B200MlpDesc* mapping, int64_t pixels) {
  EvalPlan pl;
  if (plan_eval(mapping, pixels, nullptr, &pl) != B200_OK) return -1;
  return pl.bytes + 2048;
}

int b200_eval_maps(const B200MlpDesc* mapping, const float* mapping_params, const B200Video* video, int32_t frame,
                   int64_t pix_begin, int64_t pix_end, float derivative_amount, float uv_mapping_scale, int precision,
                   float* uv, float* rigidity, float* flow_error, void* ws, int64_t ws_bytes, void* stream) {
  B200_REQUIRE(mapping && mapping_params && video && video->records && ws && (uv || rigidity || flow_error), "null pointer");
  B200_REQUIRE(frame >= video->t_begin && frame < video->t_end, "frame %d is not resident", frame);
  B200_REQUIRE(pix_begin >= 0 && pix_end > pix_begin && pix_end <= (int64_t)video->H * video->W, "bad pixel range");
  B200_REQUIRE(derivative_amount != 0.f && uv_mapping_scale != 0.f, "bad geometry");
  MlpShape s;
  B200_PROPAGATE(resolve_mlp(mapping, &s));
  B200_REQUIRE(s.in_dim == 3 && s.out_dim == 2, "mapping networks are 3 -> 2");
  const int64_t count = pix_end - pix_begin;
  EvalPlan pl;
  char* base = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(ws), 1024));
  B200_PROPAGATE(plan_eval(mapping, count, base, &pl));
  if (base + pl.bytes > reinterpret_cast<char*>(ws) + ws_bytes) {
    set_error("workspace too small: need %lld bytes", (long long)(pl.bytes + 1024));
    return B200_ERR_WORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int larger = video->W > video->H ? video->W : video->H;
  const float hL = (float)((double)larger / 2.0), hT = (float)((double)video->T / 2.0);
  const int64_t rp = pl.rows_pad;
  eval_rows_kernel<<<(unsigned)((rp + 255) / 256), 256, 0, st>>>(*video, frame, pix_begin, count, rp, hL, hT,
                                                                  derivative_amount, pl.x3, pl.valid);
  B200_CHECK_LAUNCH();
  const int prec = mlp_precision(mapping, precision);
  B200_PROPAGATE(b200_mlp_forward(mapping, mapping_params, pl.x3, pl.uv, 4 * rp, 0, prec, pl.ws, pl.ws_bytes, stream));
  eval_head_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(pl.uv, pl.valid, count, rp, (float)larger,
                                                                    uv_mapping_scale, derivative_amount,
                                                                    frame >= video->T - 1 ? 1 : 0, uv, rigidity, flow_error);
  B200_CHECK_LAUNCH();
  return B200_OK;
}

}  // extern "C"
