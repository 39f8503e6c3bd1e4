// Interface of the tcgen05 path (mlp_tc.cu) and of the network calls that choose between it and the fp32 path
// (c_api.cu), used by c_api.cu, seg.cu and eval_maps.cu.
#pragma once
#include "common.cuh"

namespace b200 {

// The network shapes the tensor-core kernels are specialised to (hidden width 256 each); every other shape runs on the
// fp32 kernels.  Mapping6 is the stage-1 scripts' mapping (3 -> 256 x 4 -> 2, no encoding, no skips), Mapping4 the
// background mapping of the segmentation variant (same kernels, two hidden 256x256 layers), Atlas the atlas network
// (2 -> PE 10 -> 256 x 6 -> 3, skips 4 and 7) and Alpha the alpha network of the segmentation variant (3 -> PE 5 ->
// 256 x 6 -> 1, no skips).  Atlas and Alpha run the kernel variants with a positional-encoding input layer.
enum class TcNet { None, Mapping6, Mapping4, Atlas, Alpha };
TcNet tc_classify(const MlpShape& s);    // None: no tensor-core kernels for this shape
inline bool tc_pe_kernels(TcNet n) { return n == TcNet::Atlas || n == TcNet::Alpha; }

// Buffers of the tensor-core path, carved from the caller's workspace (see mlp_tc.cu).
struct TcPlan {
  char* base = nullptr;
  int64_t bytes = 0;
  int64_t rows_map = 0, rows_atlas = 0;
};

struct TcStep {
  const MlpShape* ms; const MlpShape* as;
  const TcPlan* plan;
  const float* params; float* grads;
  const float* x_map;        // [n_groups*cap][4]
  float* uv;                 // [n_groups*cap][2]  mapping output
  float* y_atlas;            // [3*cap][3]         atlas output
  const float* d_uv;         // [n_groups*cap][2]  direct gradient of the loss head
  const float* d_y;          // [3*cap][3]
  int cap, n_groups;
  const int* counters;
  int flow_groups;           // 1: groups 5 / 6 of the mapping batch hold counters[5] / counters[6] compacted rows
};

int64_t tc_plan(const MlpShape& ms, const MlpShape& as, int64_t rows_map, int64_t rows_atlas, char* base,
                TcPlan* out);
int tc_begin_step(const TcStep& s, cudaStream_t st);       // optional: start the weight-image preparation early (side stream)
int tc_atlas_forward(const TcStep& s, cudaStream_t st);    // mapping on all groups, atlas on groups 0..2
int tc_atlas_backward(const TcStep& s, cudaStream_t st);   // all parameter gradients
int tc_mapping_forward(const TcStep& s, cudaStream_t st);  // pre-training: mapping only
int tc_mapping_backward(const TcStep& s, cudaStream_t st);

// inference (render): x_map [rows][4] -> uv [rows][2] -> y [rows][3]; rows a multiple of 128; ws >= tc_infer_workspace_bytes
int64_t tc_infer_workspace_bytes(const MlpShape& ms, const MlpShape& as);
int tc_infer_forward(const MlpShape& ms, const MlpShape& as, const float* params, const float* x_map, float* uv,
                     float* y, int64_t rows, char* ws, cudaStream_t st);

// stand-alone IMLP (one network of family `net`, autograd): see mlp_tc.cu
int64_t tc_single_workspace_bytes(const MlpShape& sh, TcNet net, int64_t rows);
// persistent: the caller keeps this workspace and these parameter / gradient buffers across calls -> job tables are
// cached in their own device allocations and the calls become graph-capturable after one eager call; otherwise they
// are uploaded into the workspace on every call
int tc_single_forward(const MlpShape& sh, TcNet net, const float* params, const float* x, float* y, int64_t rows,
                      bool training, char* ws, bool persistent, cudaStream_t st);
int tc_single_backward(const MlpShape& sh, TcNet net, const float* params, float* grads, const float* x,
                       const float* y, const float* dy, float* d_in, int* gmax2, int64_t rows, char* ws, bool persistent,
                       cudaStream_t st);

// b200_mlp_forward / b200_mlp_backward with the persistence of the tensor-core job tables chosen by the caller: true
// only for callers that keep `ws`, `params` and the gradient buffer alive across calls (the entry points of seg.cu)
int mlp_forward(const B200MlpDesc* d, const float* params, const float* x, float* y, int64_t rows, int training,
                int precision, void* ws, int64_t ws_bytes, void* stream, bool persistent);
int mlp_backward(const B200MlpDesc* d, const float* params, const float* x, const float* dy, float* dparams, float* dx,
                 int64_t rows, int precision, void* ws, int64_t ws_bytes, void* stream, bool persistent);
// B200_PREC_TC when `precision` asks for it and the network has tensor-core kernels, else B200_PREC_FP32: for callers
// that run each of several networks at the best precision it has
int mlp_precision(const B200MlpDesc* d, int precision);

int tc_debug_wgrad(long long* cycles, int* shapes, int max_ctas);

}  // namespace b200
