// tcgen05 path of the two IMLPs (B200_PREC_TC).
//
// Every 256-wide Linear layer is a UMMA (tcgen05.mma kind::f16, M=128 rows per CTA tile, fp32
// accumulators in TMEM).  fp32 fidelity comes from a 2-term fp16 split of BOTH operands,
//     v * S = hi + lo,   hi = rn_f16(v*S),  lo = rn_f16(v*S - hi)          (22-bit significand)
// and three MMAs per product  hi*hi + hi*lo + lo*hi  (the dropped lo*lo term is 2^-22 relative).
// S is a power of two per operand class (activations 2^4, weights 2^8, gradients chosen per
// iteration from max|dL/dy|), undone exactly in the epilogues.
//
// Kernels
//   tc_prep_kernel   fp32 parameters -> split fp16 "stage images" (the exact 128B-swizzled smem
//                    layout a UMMA descriptor reads), W for the forward and W^T for the dgrad
//   tc_fwd_kernel    persistent; one 128-row tile walks through ALL layers on chip: activations live
//                    in TMEM (A operand, TS-mode MMA), weights stream L2->smem through the TMA engine
//                    (cp.async.bulk + mbarrier ring), epilogue (8 warps) = bias + ReLU + split ->
//                    TMEM store (next layer's A) and, via a swizzled smem staging tile + bulk store,
//                    the activation image the weight-gradient kernel consumes; first/last (K=3 / N=2,3)
//                    layers and the positional encoding run on CUDA cores inside the same kernel
//   tc_bwd_kernel    same structure for dL/dz: tanh', last layer on CUDA cores, hidden layers as
//                    dZ * W (B = W^T images), ReLU mask from 1-bit flags, bias gradients by an
//                    in-register butterfly column sum
//   tc_wgrad_kernel  dW = dZ^T * H as UMMA with both operands MN-major straight from the images
//                    the two kernels above left in HBM; split over rows, fp32 vector reductions
//
// Restates nn.Linear/ReLU/tanh/skip-concat forward+autograd of
//   src/models/stage_1/implicit_neural_networks.py:62-81 for the two networks of
//   src/stage1_neural_atlas.py:112-128.
#include <mutex>
#include <vector>

#include "tc_api.cuh"
#include "tc_ptx.cuh"
#include "loss_math.h"

namespace b200 {
using namespace ptx;

constexpr int TM = 128;                 // rows per tile (UMMA M)
constexpr int HID = 256;
constexpr int STAGE_BYTES = 32768;      // one weight image: 256 rows x 64 k (fp16), 128B swizzle
constexpr float S_ACT = 16.0f;          // activation scale before the fp16 split
constexpr float S_W = 256.0f;           // weight scale
constexpr int ATOM_BYTES = TM * 128;    // one 64-column block of a tile image, one term: 16 KB
constexpr int TILE_IMG_BYTES = 4 * ATOM_BYTES;   // one term of one [128 x 256] activation tile image: 64 KB
constexpr int PE_COLS = 40;

constexpr int EPI_WARPS = 16;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int TC_THREADS = 64 + EPI_THREADS;   // warp 0: TMA producer, warp 1: MMA issuer, warps 2..17: epilogue
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t TM_D = 0, TM_AHI = 256, TM_ALO = 384;

// Tile image = 4 atom blocks (64 columns each); an atom block is [16 groups of 8 rows][8 rows x 128 B]
// with the 16-byte chunks of a row XOR-swizzled by (row & 7).  The same bytes are a K-major SW128 UMMA
// operand (M/N = rows, K = the 64 columns) and an MN-major SW128 operand (MN = columns, K = rows).
__host__ __device__ __forceinline__ int atom_off(int m, int k) {          // k in [0, 64)
  const int r = m & 7;
  return (m >> 3) * 1024 + r * 128 + (((k >> 3) ^ r) << 4) + ((k & 7) << 1);
}

// ---------------------------------------------------------------------------------------------
// layout of the tensor-core workspace
// ---------------------------------------------------------------------------------------------
struct NetImages {
  // forward weight images, consumption order: per TC layer, per 64-wide k chunk: hi image, lo image
  char* w_fwd; int64_t w_fwd_layer[B200_MAX_LAYERS]; int n_chunks_fwd[B200_MAX_LAYERS];
  // dgrad weight images (W^T): per layer, per 64-wide chunk of the reduction (out) index: hi, lo
  char* w_bwd; int64_t w_bwd_layer[B200_MAX_LAYERS];
  // activation images h_0..h_{L-2} and dZ images: [slot][term][tile][4 atoms][16 KB]
  char* act; char* dz;
  int64_t slot_stride, term_stride;       // bytes
  // 64-wide images: [term][tile][16 KB]: positional encoding (atlas) and the output-layer dZ
  char* pe; char* dzl; int64_t w64_term_stride;
  uint32_t* bits;                         // ReLU flags [slot][rows][8]
  int64_t rows;
};

struct TcLayout { NetImages map, atl; };

static char* carve_tc(char*& p, int64_t bytes) { char* r = p; p += round_up(bytes, 1024); return r; }

// forward weight images: per layer on tensor cores, its 64-wide k chunks (the positional-encoding part is one more)
static void plan_fwd_images(const MlpShape& s, TcNet net, char*& p, NetImages* n) {
  const bool is_atlas = tc_pe_kernels(net);
  int64_t off = 0;
  for (int l = 0; l < s.L; ++l) {
    int chunks = 0;
    const bool tc_layer = is_atlas ? (l <= s.L - 2) : (l >= 1 && l <= s.L - 2);
    if (tc_layer) chunks = (l == 0 ? 0 : HID / 64) + ((l == 0 || s.skip[l]) && is_atlas ? 1 : 0);
    n->n_chunks_fwd[l] = chunks;
    n->w_fwd_layer[l] = off;
    off += (int64_t)chunks * 2 * STAGE_BYTES;
  }
  n->w_fwd = carve_tc(p, off);
}

static void plan_net(const MlpShape& s, int64_t rows, TcNet net, char*& p, NetImages* n) {
  const bool is_atlas = tc_pe_kernels(net);
  const int64_t tiles = rows / TM;
  n->rows = rows;
  plan_fwd_images(s, net, p, n);
  int64_t off = 0;
  for (int l = 0; l < s.L; ++l) {
    n->w_bwd_layer[l] = off;
    const bool used = l <= s.L - 2 && (is_atlas || l >= 1);
    if (used) off += (int64_t)(HID / 64) * 2 * STAGE_BYTES;
  }
  n->w_bwd = carve_tc(p, off);
  n->term_stride = tiles * TILE_IMG_BYTES;
  n->slot_stride = 2 * n->term_stride;
  n->act = carve_tc(p, (int64_t)(s.L - 1) * n->slot_stride);
  n->dz = carve_tc(p, (int64_t)(s.L - 1) * n->slot_stride);
  n->w64_term_stride = tiles * ATOM_BYTES;
  n->pe = is_atlas ? carve_tc(p, 2 * n->w64_term_stride) : nullptr;
  n->dzl = carve_tc(p, 2 * n->w64_term_stride);
  n->bits = reinterpret_cast<uint32_t*>(carve_tc(p, (int64_t)(s.L - 1) * rows * 32));
}

int64_t tc_plan(const MlpShape& ms, const MlpShape& as, int64_t rows_map, int64_t rows_atlas, char* base,
                TcPlan* out) {
  char* p = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(base), 1024));
  TcLayout lay{};
  plan_net(ms, rows_map, TcNet::Mapping6, p, &lay.map);
  plan_net(as, rows_atlas, TcNet::Atlas, p, &lay.atl);
  if (out) { out->base = base; out->bytes = p - base; out->rows_map = rows_map; out->rows_atlas = rows_atlas; }
  return p - base;
}

static TcLayout layout_of(const TcStep& s) {
  char* p = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(s.plan->base), 1024));
  TcLayout lay{};
  plan_net(*s.ms, s.plan->rows_map, TcNet::Mapping6, p, &lay.map);
  plan_net(*s.as, s.plan->rows_atlas, TcNet::Atlas, p, &lay.atl);
  return lay;
}

// ---------------------------------------------------------------------------------------------
// weight preparation
// ---------------------------------------------------------------------------------------------
struct PrepJob {
  const float* W; int ldw;          // fp32 weight [N][ldw]
  int n_rows, k0, k_cnt;            // valid image rows and the window [k0, k0+k_cnt) of the other index
  int transpose;                    // 0: image(row=n, col=k-k0) = W[n][k];  1: image(row=k, col=n-k0) = W[n][k]
  char* hi; char* lo;               // destination images (32 KB each, zero padded)
};
constexpr int MAX_PREP_JOBS = 96;
struct PrepJobs { PrepJob j[MAX_PREP_JOBS]; int n; };

__global__ void tc_prep_kernel(const PrepJobs* __restrict__ jobs_ptr) {
  const PrepJob jb = jobs_ptr->j[blockIdx.x >> 2];
  // one image = 256 rows x 64 cols; this block does 64 rows; thread handles one 16-byte chunk at a time
  for (int e = threadIdx.x; e < 64 * 8; e += blockDim.x) {
    const int row = (blockIdx.x & 3) * 64 + (e >> 3), c8 = (e & 7) * 8;
    float v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int col = c8 + q;
      v[q] = 0.f;
      if (row < jb.n_rows && col < jb.k_cnt)
        v[q] = jb.transpose ? jb.W[(int64_t)(jb.k0 + col) * jb.ldw + row] : jb.W[(int64_t)row * jb.ldw + jb.k0 + col];
    }
    uint32_t h[4], l[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) split2_f16(v[2 * q] * S_W, v[2 * q + 1] * S_W, h[q], l[q]);
    const int off = atom_off(row, c8);
    *reinterpret_cast<uint4*>(jb.hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(jb.lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// ---------------------------------------------------------------------------------------------
// shared pieces of the fused kernels
// ---------------------------------------------------------------------------------------------
template <int NST>
struct Pipe {                        // weight-image ring shared by producer and MMA warp
  uint64_t* full; uint64_t* empty; char* stage;
  uint32_t it;                       // running item counter
  __device__ __forceinline__ int slot() const { return it % NST; }
  __device__ __forceinline__ uint32_t parity() const { return (it / NST) & 1; }
};

struct TileIter {                    // static round-robin over the live tiles of a group-major batch
  int t0, tf, tb, total, cap_tiles, n_groups, flow;
  // counters: [0] rows of an ordinary group, [5] / [6] rows of the compacted flow-match groups (G_FWD = 5, G_BWD = 6
  // of the mapping batch when `flow_groups` is set); nullptr: every row of every group is live
  __device__ __forceinline__ void init(int cap, int groups, const int* counters, int flow_groups) {
    cap_tiles = cap / TM;
    n_groups = groups;
    flow = (flow_groups && groups > 6) ? 1 : 0;
    t0 = counters ? min(cap_tiles, (counters[0] + TM - 1) / TM) : cap_tiles;
    tf = flow ? min(cap_tiles, (counters[5] + TM - 1) / TM) : t0;
    tb = flow ? min(cap_tiles, (counters[6] + TM - 1) / TM) : t0;
    total = t0 * (groups - (flow ? 2 : 0)) + (flow ? tf + tb : 0);
  }
  __device__ __forceinline__ int group_tiles(int g) const { return (flow && g == 5) ? tf : ((flow && g == 6) ? tb : t0); }
  __device__ __forceinline__ int global_tile(int t) const {
    for (int g = 0; g < n_groups; ++g) {
      const int n = group_tiles(g);
      if (t < n) return g * cap_tiles + t;
      t -= n;
    }
    return 0;
  }
};

// MMAs of one 64-wide k chunk whose A operand is in TMEM (hi at TM_AHI, lo at TM_ALO):
//   D += A_hi*B_hi + A_lo*B_hi   (B_hi image)    then   D += A_hi*B_lo   (B_lo image)
template <int NST>
__device__ __forceinline__ void mma_chunk_ts(Pipe<NST>& pp, uint32_t tmem, int kchunk, uint32_t idesc, bool& first) {
  {
    mbar_wait(&pp.full[pp.slot()], pp.parity());
    tc_fence_after();
    const uint32_t sb = smem_u32(pp.stage + pp.slot() * STAGE_BYTES);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint64_t bd = make_desc(sb + ks * 32, 16, 1024);
      mma_ts(tmem + TM_D, tmem + TM_AHI + kchunk * 32 + ks * 8, bd, idesc, first ? 0u : 1u);
      first = false;
      mma_ts(tmem + TM_D, tmem + TM_ALO + kchunk * 32 + ks * 8, bd, idesc, 1u);
    }
    mma_commit(&pp.empty[pp.slot()]);
    ++pp.it;
  }
  {
    mbar_wait(&pp.full[pp.slot()], pp.parity());
    tc_fence_after();
    const uint32_t sb = smem_u32(pp.stage + pp.slot() * STAGE_BYTES);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
      mma_ts(tmem + TM_D, tmem + TM_AHI + kchunk * 32 + ks * 8, make_desc(sb + ks * 32, 16, 1024), idesc, 1u);
    mma_commit(&pp.empty[pp.slot()]);
    ++pp.it;
  }
}
// same with the A operand in shared memory (64-wide K-major SW128 tile: hi image, lo image)
template <int NST>
__device__ __forceinline__ void mma_chunk_ss(Pipe<NST>& pp, uint32_t tmem, const char* a_hi, const char* a_lo,
                                             uint32_t idesc, bool& first) {
  const uint32_t ah = smem_u32(a_hi), al = smem_u32(a_lo);
  {
    mbar_wait(&pp.full[pp.slot()], pp.parity());
    tc_fence_after();
    const uint32_t sb = smem_u32(pp.stage + pp.slot() * STAGE_BYTES);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint64_t bd = make_desc(sb + ks * 32, 16, 1024);
      mma_ss(tmem + TM_D, make_desc(ah + ks * 32, 16, 1024), bd, idesc, first ? 0u : 1u);
      first = false;
      mma_ss(tmem + TM_D, make_desc(al + ks * 32, 16, 1024), bd, idesc, 1u);
    }
    mma_commit(&pp.empty[pp.slot()]);
    ++pp.it;
  }
  {
    mbar_wait(&pp.full[pp.slot()], pp.parity());
    tc_fence_after();
    const uint32_t sb = smem_u32(pp.stage + pp.slot() * STAGE_BYTES);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
      mma_ss(tmem + TM_D, make_desc(ah + ks * 32, 16, 1024), make_desc(sb + ks * 32, 16, 1024), idesc, 1u);
    mma_commit(&pp.empty[pp.slot()]);
    ++pp.it;
  }
}

template <int NST>
__device__ __forceinline__ void produce_items(Pipe<NST>& pp, const char* src, int n_items) {
  for (int i = 0; i < n_items; ++i) {
    mbar_wait(&pp.empty[pp.slot()], pp.parity() ^ 1);
    mbar_expect_tx(&pp.full[pp.slot()], STAGE_BYTES);
    bulk_g2s(pp.stage + pp.slot() * STAGE_BYTES, src + (int64_t)i * STAGE_BYTES, STAGE_BYTES, &pp.full[pp.slot()]);
    ++pp.it;
  }
}

// dynamic shared memory map: [weight stages][staging 2 x (hi 16K | lo 16K)][aux tile 32 KB (atlas)][consts][barriers]
constexpr int SMEM_STAGING = 2 * 2 * ATOM_BYTES;             // 64 KB
constexpr int SMEM_AUX = 2 * ATOM_BYTES;                     // 32 KB
constexpr int SMEM_CONST_FLOATS = 4608;                      // 18 KB
constexpr int SMEM_BARS = 256;
// Both kernels stream the weights through a 4-stage ring (128 KB: a 64 KB k chunk is consumed in ~1.8 k cycles, the
// bulk copies take 2-4 k cycles to arrive, so three stages starved the atlas kernels' MMA warp).  The atlas kernels
// pay for the fourth stage and their positional-encoding tile with single-buffered image staging.
template <bool ATLAS> struct KCfg {
  static constexpr int NST = 4;
  static constexpr int STAGING_BUFS = ATLAS ? 1 : 2;
  static constexpr int STAGING = STAGING_BUFS * 4 * 8192;
  static constexpr int SMEM = NST * STAGE_BYTES + STAGING + (ATLAS ? SMEM_AUX : 0) + SMEM_CONST_FLOATS * 4 + SMEM_BARS;
};

template <int NST, bool ATLAS>
struct SmemMap {
  char* stage; char* staging; char* aux; float* cst;
  uint64_t* full; uint64_t* empty; uint64_t* a_ready; uint64_t* x_ready; uint64_t* d_ready; uint64_t* d_free;
  uint64_t* misc; uint32_t* tmem_slot;
  __device__ __forceinline__ void init(char* raw) {
    char* p = raw;                                   // 1024-aligned (checked in setup_cta): keeps the
    stage = p; p += NST * STAGE_BYTES;               // shared address space visible to the compiler (LDS/STS)
    staging = p; p += KCfg<ATLAS>::STAGING;
    aux = p; if (ATLAS) p += SMEM_AUX;
    cst = reinterpret_cast<float*>(p); p += SMEM_CONST_FLOATS * 4;
    full = reinterpret_cast<uint64_t*>(p);
    empty = full + NST;
    a_ready = empty + NST;          // [4]: one per 64-column k chunk of the next layer's A operand
    x_ready = a_ready + 4;          // layer-0 input of a tile is in place (atlas: positional-encoding tile)
    d_ready = x_ready + 1;          // accumulator of the current layer pass is complete
    d_free = d_ready + 1;           // ... and has been drained into registers by every epilogue thread
    misc = d_free + 1;
    tmem_slot = reinterpret_cast<uint32_t*>(misc + 2);
  }
};

template <int NST, bool ATLAS>
__device__ __forceinline__ uint32_t setup_cta(SmemMap<NST, ATLAS>& sm, int warp) {
  if (threadIdx.x == 0) {
    if (smem_u32(sm.stage) & 1023u) { printf("b200: dynamic shared memory is not 1024-byte aligned\n"); __trap(); }
    for (int i = 0; i < NST; ++i) { mbar_init(&sm.full[i], 1); mbar_init(&sm.empty[i], 1); }
    for (int i = 0; i < 4; ++i) mbar_init(&sm.a_ready[i], EPI_THREADS);       // every epilogue thread owns a piece of every chunk
    mbar_init(sm.x_ready, EPI_THREADS);
    mbar_init(sm.d_ready, 1);
    mbar_init(sm.d_free, EPI_THREADS);
    mbar_init(&sm.misc[0], 1);
    mbar_init(&sm.misc[1], EPI_THREADS);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(sm.tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return *sm.tmem_slot;
}

// Epilogue thread geometry: 16 warps.  A warp may only touch the TMEM lanes of quadrant (warp_id & 3); the four
// warps of a quadrant are the column slices j = 0..3, and every warp owns a 16-column piece of EACH of the four
// 64-column k chunks: columns [64c + 16j, 64c + 16j + 16), c = 0..3.  All 16 warps therefore finish k chunk 0 a quarter
// of the way through the epilogue, chunk 1 at half, ...: the next layer's A operand is released chunk by chunk in
// exactly the order the MMA warp consumes it.
struct EpiThread {
  int e, q, j, lane, m, tid;        // epilogue warp, TMEM quadrant, column slice, lane, tile row, 0..511
  uint32_t tlane;
  __device__ __forceinline__ void init(uint32_t tmem) {
    const int warp = threadIdx.x >> 5;
    lane = threadIdx.x & 31;
    e = warp - 2; q = warp & 3; j = e >> 2;
    m = q * 32 + lane;
    tid = threadIdx.x - 64;
    tlane = tmem + ((uint32_t)(q * 32) << 16);
  }
  __device__ __forceinline__ int col0(int c) const { return c * 64 + j * 16; }      // first column of the piece in chunk c
};

// Pushes one finished 16-column piece (packed hi/lo words of this thread's row) to the HBM image.  The four warps of
// a quadrant fill one 32-row x 64-column part of an atom block = 4 KB contiguous bytes of the image per term, staged
// in the quadrant's buffer `buf` (two alternate) and written with one bulk store per term.  Called by all four warps.
template <int BUFS>
__device__ __forceinline__ void stage_quad(const EpiThread& t, char* staging, int piece, const uint32_t (&ph)[8],
                                           const uint32_t (&pl)[8], char* g_hi_atom, char* g_lo_atom) {
  char* sh = staging + ((BUFS == 2 ? (piece & 1) : 0) * 4 + t.q) * 8192;
  char* sl = sh + 4096;
  const bool issuer = (t.j == 0) && t.lane == 0;
  if (issuer) {                                          // the previous store out of this buffer has read it
    if (BUFS == 2) bulk_wait_read1(); else bulk_wait_read0();
  }
  named_bar(1 + t.q, 128);
  const int r = t.m & 7;
  const int base = ((t.m & 31) >> 3) * 1024 + r * 128;
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int off = base + (((t.j * 2 + u) ^ r) << 4);
    *reinterpret_cast<uint4*>(sh + off) = make_uint4(ph[4 * u], ph[4 * u + 1], ph[4 * u + 2], ph[4 * u + 3]);
    *reinterpret_cast<uint4*>(sl + off) = make_uint4(pl[4 * u], pl[4 * u + 1], pl[4 * u + 2], pl[4 * u + 3]);
  }
  fence_proxy_async_smem();
  named_bar(1 + t.q, 128);
  if (issuer) {
    bulk_s2g(g_hi_atom + t.q * 4096, sh, 4096);
    bulk_s2g(g_lo_atom + t.q * 4096, sl, 4096);
    bulk_commit();
  }
}
constexpr int BAR_EPI = 9;                               // named barrier of all epilogue threads

struct FwdParams {
  const float* x;            // mapping: [rows][4] (x, y, t, 0);  atlas: uv [rows][2]
  float* y;                  // mapping: uv [rows][2];  atlas: y [rows][3]
  const float* params;       // fp32 parameters of this network
  int64_t w_off[B200_MAX_LAYERS], b_off[B200_MAX_LAYERS];
  NetImages img;
  int cap, n_groups; const int* n_valid;
  int flow_groups;           // mapping batch of the loop: groups 5 / 6 are compacted to counters[5] / counters[6] rows
  float in_scale, in_shift;  // atlas: network input = x * in_scale + in_shift (0.5, 0.5 inside the loop: uv -> [0,1])
  int store_images;          // 0: inference (render / IMLP.forward without grad): no activation images, no flags
  int tanh_out;
};

// =============================================================================================
// forward
// =============================================================================================
// Schedule of one layer pass (both fused kernels).  The accumulator D of pass n is drained into registers by the
// 16 epilogue warps as soon as it is complete (d_ready -> 2 tcgen05.ld per thread -> d_free), which frees TMEM for
// pass n+1 while the epilogue arithmetic of pass n is still running: the epilogue releases the next A operand one
// 64-column k chunk at a time (a_ready[kc]: chunks 0, 1 after the block-0 half of the epilogue, 2, 3 after the
// block-1 half) and the MMA warp consumes them in that order, so the tensor pipe works on layer l+1 underneath the
// epilogue of layer l.
// VAR (with ATLAS = true): 0 = the atlas network (2 inputs, 10 frequencies, skips at 4 and 7, 3 outputs), 1 = the alpha
// network of the segmentation variant (3 inputs, 5 frequencies, no skips, 1 output, no input gradient)
template <bool ATLAS, int NL = (ATLAS ? 8 : 6), int VAR = 0>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_fwd_kernel(const __grid_constant__ FwdParams P) {
  extern __shared__ __align__(1024) char smem_raw[];
  constexpr int NST = KCfg<ATLAS>::NST;
  SmemMap<NST, ATLAS> sm; sm.init(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int L = NL;                                   // mapping-shaped networks: 6 (stage-1 script) or 4 layers
  constexpr int FIRST_TC = ATLAS ? 0 : 1;
  constexpr int LAST_TC = L - 2;
  constexpr bool ALPHA = ATLAS && VAR == 1;
  constexpr bool SKIPS = ATLAS && !ALPHA;                 // PE chunk concatenated at layers 4 and L-1
  constexpr int OUT = ATLAS ? (ALPHA ? 1 : 3) : 2;
  constexpr int KLAST = SKIPS ? 296 : 256;
  // constants in shared memory: biases of layers 0..L-2 (pre-multiplied by S_ACT) at [l*256], last-layer
  // weights (pre-divided by S_ACT) + bias, (mapping) W0, and an exchange area for the output layer
  float* s_bias = sm.cst;
  float* s_wlast = sm.cst + (L - 1) * 256;
  float* s_blast = s_wlast + OUT * KLAST;
  float* s_w0 = s_blast + 4;                              // mapping only: 768 floats
  float* s_xch = sm.cst + SMEM_CONST_FLOATS - 3 * TM * 4; // [3][128][4] partial outputs of column slices 1..3
  for (int i = threadIdx.x; i < (L - 1) * 256; i += blockDim.x)
    s_bias[i] = P.params[P.b_off[i >> 8] + (i & 255)] * S_ACT;
  for (int i = threadIdx.x; i < OUT * KLAST; i += blockDim.x) s_wlast[i] = P.params[P.w_off[L - 1] + i] * (1.0f / S_ACT);
  if (threadIdx.x < OUT) s_blast[threadIdx.x] = P.params[P.b_off[L - 1] + threadIdx.x];
  if (!ATLAS)      // W0 (256 x 3) transposed to [3][256] so that column pairs are adjacent (FFMA2)
    for (int i = threadIdx.x; i < 768; i += blockDim.x) s_w0[(i % 3) * 256 + i / 3] = P.params[P.w_off[0] + i] * S_ACT;
  const uint32_t tmem = setup_cta(sm, warp);
  TileIter ti; ti.init(P.cap, P.n_groups, P.n_valid, P.flow_groups);
  constexpr uint32_t IDESC = make_idesc(128, 256, 0, 0);

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (consumption order)
    if (lane == 0) {
      Pipe<NST> pp{sm.full, sm.empty, sm.stage, 0};
      for (int t = blockIdx.x; t < ti.total; t += gridDim.x)
        for (int l = FIRST_TC; l <= LAST_TC; ++l) {
          const char* base = P.img.w_fwd + P.img.w_fwd_layer[l];
          if (ATLAS && l == 0) { produce_items(pp, base, 2); continue; }
          if (SKIPS && l == 4) produce_items(pp, base + (int64_t)4 * 2 * STAGE_BYTES, 2);      // skip (PE) chunk first
          produce_items(pp, base, 8);
        }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      Pipe<NST> pp{sm.full, sm.empty, sm.stage, 0};
      uint32_t pass = 0, ts_pass = 0, x_par = 0;
      for (int t = blockIdx.x; t < ti.total; t += gridDim.x) {
        for (int l = FIRST_TC; l <= LAST_TC; ++l) {
          if (pass > 0) mbar_wait(sm.d_free, (pass - 1) & 1);      // D of the previous pass is in registers
          bool first = true;
          if (ATLAS && l == 0) { mbar_wait(sm.x_ready, x_par); x_par ^= 1; }
          tc_fence_after();
          if (ATLAS && (l == 0 || (SKIPS && l == 4))) mma_chunk_ss(pp, tmem, sm.aux, sm.aux + ATOM_BYTES, IDESC, first);
          if (l > 0) {
            for (int kc = 0; kc < 4; ++kc) {
              mbar_wait(&sm.a_ready[kc], ts_pass & 1);
              tc_fence_after();
              mma_chunk_ts(pp, tmem, kc, IDESC, first);
            }
            ++ts_pass;
          }
          mma_commit(sm.d_ready);
          ++pass;
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (512 threads)
    EpiThread et; et.init(tmem);
    const int m = et.m, j = et.j;
    uint32_t d_par = 0;
    const float inv_scale = 1.0f / S_W;                 // D / (S_a S_w) * S_a : activations stay scaled by S_ACT
    uint16_t* bits16 = reinterpret_cast<uint16_t*>(P.img.bits);
    for (int t = blockIdx.x; t < ti.total; t += gridDim.x) {
      const int gt = ti.global_tile(t);
      const int64_t row = (int64_t)gt * TM + m;
      // ---------------- prologue: layer-0 input
      if (ATLAS) {
        // positional encoding of in = x*in_scale+in_shift (implicit_neural_networks.py:9-13) into the aux tile
        // (K-major SW128, columns k*4 + {sin x0, sin x1, cos x0, cos x1}); slice j does the 8-column chunks 2j, 2j+1
        float in[3] = {0.f, 0.f, 0.f};
        if (ALPHA) {                                     // rows padded to 4 floats, like the mapping's
          const float4 xv = *reinterpret_cast<const float4*>(P.x + row * 4);
          in[0] = xv.x * P.in_scale + P.in_shift; in[1] = xv.y * P.in_scale + P.in_shift; in[2] = xv.z * P.in_scale + P.in_shift;
        } else {
          const float2 uv = *reinterpret_cast<const float2*>(P.x + row * 2);
          in[0] = uv.x * P.in_scale + P.in_shift; in[1] = uv.y * P.in_scale + P.in_shift;
        }
        char* a_hi = sm.aux;
        char* a_lo = sm.aux + ATOM_BYTES;
        char* g_hi = P.img.pe + (int64_t)gt * ATOM_BYTES;
        char* g_lo = g_hi + P.img.w64_term_stride;
        for (int c8 = 2 * j; c8 < 2 * j + 2; ++c8) {     // chunks of 8 columns (atlas: 2 frequencies)
          float vals[8];
          if (ALPHA) {
            // column c = k*6 + r: r < 3 -> sin(x_r b_k), else cos(x_{r-3} b_k); 30 real columns
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int c = c8 * 8 + i;
              float v = 0.f;
              if (c < 30) {
                const int k = c / 6, r = c - k * 6;
                const float a = in[r < 3 ? r : r - 3] * pe_freq(k);
                v = r < 3 ? sinf(a) : cosf(a);
              }
              vals[i] = v * S_ACT;
            }
          } else {
#pragma unroll
          for (int half_k = 0; half_k < 2; ++half_k) {
            const int k = c8 * 2 + half_k;
            float s0 = 0.f, s1 = 0.f, c0 = 0.f, c1 = 0.f;
            if (k < 10) {
              const float bk = pe_freq(k);
              const float a0 = in[0] * bk, a1 = in[1] * bk;
              s0 = sinf(a0); s1 = sinf(a1); c0 = cosf(a0); c1 = cosf(a1);
            }
            vals[half_k * 4 + 0] = s0 * S_ACT; vals[half_k * 4 + 1] = s1 * S_ACT;
            vals[half_k * 4 + 2] = c0 * S_ACT; vals[half_k * 4 + 3] = c1 * S_ACT;
          }
          }
          uint32_t h[4], lo[4];
#pragma unroll
          for (int q2 = 0; q2 < 4; ++q2) split2_f16(vals[2 * q2], vals[2 * q2 + 1], h[q2], lo[q2]);
          const int off = atom_off(m, c8 * 8);
          const uint4 vh = make_uint4(h[0], h[1], h[2], h[3]), vl = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          *reinterpret_cast<uint4*>(a_hi + off) = vh;
          *reinterpret_cast<uint4*>(a_lo + off) = vl;
          if (P.store_images) {
            *reinterpret_cast<uint4*>(g_hi + off) = vh;
            *reinterpret_cast<uint4*>(g_lo + off) = vl;
          }
        }
        fence_proxy_async_smem();                      // generic-proxy smem writes -> visible to the MMA
        tc_fence_before();
        mbar_arrive(sm.x_ready);
      } else {
        // layer 0 (3 -> 256) on CUDA cores: h0 = relu(W0 x + b0), this thread's four 16-column pieces
        const float4 xv = *reinterpret_cast<const float4*>(P.x + row * 4);
        char* img = P.img.act + (int64_t)gt * TILE_IMG_BYTES;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int c0 = et.col0(c);
          uint32_t ph[8], pl[8];
          uint32_t bw = 0;
          const uint64_t x0 = pack2f(xv.x, xv.x), x1 = pack2f(xv.y, xv.y), x2 = pack2f(xv.z, xv.z);
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            const int n = c0 + i;
            uint64_t a = *reinterpret_cast<const uint64_t*>(s_bias + n);
            a = fma2(x0, *reinterpret_cast<const uint64_t*>(s_w0 + n), a);
            a = fma2(x1, *reinterpret_cast<const uint64_t*>(s_w0 + 256 + n), a);
            a = fma2(x2, *reinterpret_cast<const uint64_t*>(s_w0 + 512 + n), a);
            float z0, z1;
            unpack2f(a, z0, z1);
            const float v0 = fmaxf(z0, 0.f), v1 = fmaxf(z1, 0.f);
            bw = push_flag(push_flag(bw, v0), v1);
            split2_packed(v0, v1, ph[i / 2], pl[i / 2]);
          }
          tmem_st8(et.tlane + TM_AHI + c0 / 2, ph);
          tmem_st8(et.tlane + TM_ALO + c0 / 2, pl);
          tmem_st_wait();
          tc_fence_before();
          mbar_arrive(&sm.a_ready[c]);                 // this thread's share of k chunk c of A_1 is in TMEM
          if (P.store_images) {
            char* g = img + c * ATOM_BYTES;
            stage_quad<KCfg<ATLAS>::STAGING_BUFS>(et, sm.staging, c, ph, pl, g, g + P.img.term_stride);
            bits16[((int64_t)0 * P.img.rows + row) * 16 + (c0 >> 4)] = (uint16_t)bw;
          }
        }
      }
      // ---------------- tensor-core layers
      float outacc[OUT];
#pragma unroll
      for (int jj = 0; jj < OUT; ++jj) outacc[jj] = 0.f;
#pragma unroll 1
      for (int l = FIRST_TC; l <= LAST_TC; ++l) {
        mbar_wait(sm.d_ready, d_par); d_par ^= 1;
        tc_fence_after();
        // drain this thread's 64 accumulator columns, then hand D back to the MMA warp
        uint32_t raw[4][16];
#pragma unroll
        for (int c = 0; c < 4; ++c) tmem_ld16(et.tlane + TM_D + et.col0(c), raw[c]);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(sm.d_free);
        const bool last = (l == LAST_TC);
        char* img = P.img.act + (int64_t)l * P.img.slot_stride + (int64_t)gt * TILE_IMG_BYTES;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int c0 = et.col0(c);
          const float* bias = s_bias + l * 256 + c0;
          uint32_t ph[8], pl[8];
          uint32_t bw = 0;
          const uint64_t inv2 = pack2f(inv_scale, inv_scale);
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            float z0, z1;
            unpack2f(fma2(pack2u(raw[c][i], raw[c][i + 1]), inv2, *reinterpret_cast<const uint64_t*>(bias + i)), z0, z1);
            const float v0 = fmaxf(z0, 0.f), v1 = fmaxf(z1, 0.f);
            bw = push_flag(push_flag(bw, v0), v1);      // flag of column i is bit 15 - i
            if (last) {
#pragma unroll
              for (int jj = 0; jj < OUT; ++jj) {
                outacc[jj] = fmaf(v0, s_wlast[jj * KLAST + c0 + i], outacc[jj]);
                outacc[jj] = fmaf(v1, s_wlast[jj * KLAST + c0 + i + 1], outacc[jj]);
              }
            }
            split2_packed(v0, v1, ph[i / 2], pl[i / 2]);
          }
          if (!last) {
            tmem_st8(et.tlane + TM_AHI + c0 / 2, ph);
            tmem_st8(et.tlane + TM_ALO + c0 / 2, pl);
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(&sm.a_ready[c]);                // next layer's MMAs on k chunk c may start
          }
          if (P.store_images) {
            char* g = img + c * ATOM_BYTES;
            stage_quad<KCfg<ATLAS>::STAGING_BUFS>(et, sm.staging, c, ph, pl, g, g + P.img.term_stride);
            bits16[((int64_t)l * P.img.rows + row) * 16 + (c0 >> 4)] = (uint16_t)bw;
          }
        }
      }
      // ---------------- output layer (+ skip part for the atlas) and tanh; the four column slices of a row
      // combine through shared memory
      if (SKIPS) {
        const char* a_hi = sm.aux;
        const char* a_lo = sm.aux + ATOM_BYTES;
        for (int k = j * 10; k < j * 10 + 10; ++k) {
          const int off = atom_off(m, k);
          const float pv = __half2float(*reinterpret_cast<const __half*>(a_hi + off)) +
                           __half2float(*reinterpret_cast<const __half*>(a_lo + off));     // S_ACT * pe
#pragma unroll
          for (int jj = 0; jj < OUT; ++jj) outacc[jj] = fmaf(pv, s_wlast[jj * KLAST + 256 + k], outacc[jj]);
        }
      }
      if (j > 0) {
#pragma unroll
        for (int jj = 0; jj < OUT; ++jj) s_xch[((j - 1) * TM + m) * 4 + jj] = outacc[jj];
      }
      named_bar(BAR_EPI, EPI_THREADS);
      if (j == 0) {
#pragma unroll
        for (int jj = 0; jj < OUT; ++jj) {
          const float o = ((outacc[jj] + s_xch[(0 * TM + m) * 4 + jj]) + s_xch[(1 * TM + m) * 4 + jj]) +
                          s_xch[(2 * TM + m) * 4 + jj] + s_blast[jj];
          P.y[row * OUT + jj] = P.tanh_out ? tanhf(o) : o;
        }
      }
      named_bar(BAR_EPI, EPI_THREADS);                   // s_xch / aux tile reuse by the next tile
    }
    if (j == 0 && lane == 0) bulk_wait_all0();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, TMEM_COLS);
}

// =============================================================================================
// backward (dgrad chain + first-layer / bias gradients; the 64-wide output-layer dZ image)
// =============================================================================================
struct BwdParams {
  const float* dy;           // mapping: d_uv [rows][2];  atlas: d_y [rows][3]
  const float* y;            // network output (tanh applied)
  const float* x;            // mapping: x_map [rows][4]
  float* d_in;               // atlas: d_uv [rows][2] (accumulated: += 0.5 * dPE/din)
  const float* params;       // fp32 parameters of this network
  float* grads;              // fp32 gradient block of this network
  int64_t w_off[B200_MAX_LAYERS], b_off[B200_MAX_LAYERS];
  NetImages img;
  int cap, n_groups; const int* n_valid;
  int* gmax_bits;            // [0] max |dL/dy| from the loss head, [1] max |dL/duv| after the atlas backward
  int flow_groups;
  float in_scale;            // atlas: d(network input)/d(x) (0.5 inside the loop)
  int d_in_accumulate;       // atlas: 1 = d_in already holds the direct loss-head gradient (the loop), 0 = overwrite
  int tanh_out;
};

// column sums over the 32 rows of a warp: lane j ends with sum_rows v[j]
__device__ __forceinline__ float warp_colsum32(const float (&v)[32], int lane) {
  float a[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float send = (lane & 16) ? v[i] : v[i + 16];
    const float keep = (lane & 16) ? v[i + 16] : v[i];
    a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
  float b[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float send = (lane & 8) ? a[i] : a[i + 8];
    const float keep = (lane & 8) ? a[i + 8] : a[i];
    b[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  float c[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float send = (lane & 4) ? b[i] : b[i + 4];
    const float keep = (lane & 4) ? b[i + 4] : b[i];
    c[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  float d[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float send = (lane & 2) ? c[i] : c[i + 2];
    const float keep = (lane & 2) ? c[i + 2] : c[i];
    d[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  const float send = (lane & 1) ? d[0] : d[1];
  const float keep = (lane & 1) ? d[1] : d[0];
  return keep + __shfl_xor_sync(0xffffffffu, send, 1);
}

// column sums of 16 values over the 32 rows of a warp: lanes 2k and 2k+1 end with sum_rows v[k]
__device__ __forceinline__ float warp_colsum16(const float (&v)[16], int lane) {
  float a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float send = (lane & 16) ? v[i] : v[i + 8];
    const float keep = (lane & 16) ? v[i + 8] : v[i];
    a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
  float b[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float send = (lane & 8) ? a[i] : a[i + 4];
    const float keep = (lane & 8) ? a[i + 4] : a[i];
    b[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  float c[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float send = (lane & 4) ? b[i] : b[i + 2];
    const float keep = (lane & 4) ? b[i + 2] : b[i];
    c[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  const float send = (lane & 2) ? c[0] : c[1];
  const float keep = (lane & 2) ? c[1] : c[0];
  const float d = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  return d + __shfl_xor_sync(0xffffffffu, d, 1);
}

// gmax_bits[0]: max |dL/drgb| (atlas network);  gmax_bits[1]: max |dL/duv| (mapping network: loss head,
// then raised by the atlas backward, whose positional encoding multiplies gradients by up to 2^9*pi).
__device__ __forceinline__ void grad_scales(const int* gmax_bits, bool mapping, float& s_g, float& inv_sg) {
  const float mx = __int_as_float(gmax_bits[mapping ? 1 : 0]);
  int e = 0;
  if (mx > 0.f && mx < 3.0e38f) frexpf(mx, &e);        // mx < 2^e
  e = max(-60, min(60, e));
  s_g = ldexpf(1.0f, 13 - e);                           // mx * s_g < 8192: 8x headroom below the fp16 range
  inv_sg = ldexpf(1.0f, e - 13);                        // (conversions saturate), small entries keep their lo term
}

template <bool ATLAS, int NL = (ATLAS ? 8 : 6), int VAR = 0>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_bwd_kernel(const __grid_constant__ BwdParams P) {
  extern __shared__ __align__(1024) char smem_raw[];
  constexpr int NST = KCfg<ATLAS>::NST;
  SmemMap<NST, ATLAS> sm; sm.init(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int L = NL;                                   // mapping-shaped networks: 6 (stage-1 script) or 4 layers
  constexpr bool ALPHA = ATLAS && VAR == 1;
  constexpr bool SKIPS = ATLAS && !ALPHA;                 // PE chunk concatenated at layers 4 and L-1
  constexpr int OUT = ATLAS ? (ALPHA ? 1 : 3) : 2;
  constexpr int KLAST = SKIPS ? 296 : 256;
  constexpr int LOW = 1;                                  // dgrad layers L-2 .. 1 (atlas: + the dPE product)
  constexpr int N_DGRAD = L - 2 - LOW + 1;
  constexpr bool HAS_DPE = ATLAS && !ALPHA;               // input gradient through the positional encoding
  // shared constants: last-layer weights; bias-gradient accumulators for layers 0..L-2; (mapping) dW0; (atlas) the
  // exchange area of the dPE partial sums
  float* s_wlast = sm.cst;                               // OUT*KLAST (<= 888)
  float* s_bacc = sm.cst + 896;                          // (L-1)*256 (<= 1792)
  float* s_w0acc = s_bacc + (L - 1) * 256;               // mapping: 768   (896+1280+768 = 2944)
  float* s_xch = sm.cst + SMEM_CONST_FLOATS - 3 * TM * 2; // atlas: [3][128][2] partial dPE sums of slices 1..3
  for (int i = threadIdx.x; i < OUT * KLAST; i += blockDim.x) s_wlast[i] = P.params[P.w_off[L - 1] + i];
  for (int i = threadIdx.x; i < (L - 1) * 256 + (ATLAS ? 0 : 768); i += blockDim.x) s_bacc[i] = 0.f;
  const uint32_t tmem = setup_cta(sm, warp);
  TileIter ti; ti.init(P.cap, P.n_groups, P.n_valid, P.flow_groups);
  constexpr uint32_t IDESC = make_idesc(128, 256, 0, 0);
  constexpr uint32_t IDESC64 = make_idesc(128, 64, 0, 0);
  float s_g, inv_sg;
  grad_scales(P.gmax_bits, !ATLAS, s_g, inv_sg);

  if (warp == 0) {
    if (lane == 0) {
      Pipe<NST> pp{sm.full, sm.empty, sm.stage, 0};
      uint32_t h_par = 0;
      for (int t = blockIdx.x; t < ti.total; t += gridDim.x) {
        const int gt = ti.global_tile(t);
        if (HAS_DPE) {
          // aux tile <- positional-encoding image of this tile (hi, lo), completion on misc[0]
          mbar_wait(&sm.misc[1], h_par ^ 1);             // previous tile's readers are done with aux
          mbar_expect_tx(&sm.misc[0], 2 * ATOM_BYTES);
          bulk_g2s(sm.aux, P.img.pe + (int64_t)gt * ATOM_BYTES, ATOM_BYTES, &sm.misc[0]);
          bulk_g2s(sm.aux + ATOM_BYTES, P.img.pe + P.img.w64_term_stride + (int64_t)gt * ATOM_BYTES, ATOM_BYTES,
                   &sm.misc[0]);
          h_par ^= 1;
        }
        for (int l = L - 2; l >= (HAS_DPE ? 0 : LOW); --l) produce_items(pp, P.img.w_bwd + P.img.w_bwd_layer[l], 8);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      Pipe<NST> pp{sm.full, sm.empty, sm.stage, 0};
      uint32_t pass = 0;
      for (int t = blockIdx.x; t < ti.total; t += gridDim.x) {
        for (int l = 0; l < N_DGRAD + (HAS_DPE ? 1 : 0); ++l) {
          if (pass > 0) mbar_wait(sm.d_free, (pass - 1) & 1);
          tc_fence_after();
          bool first = true;
          const uint32_t idesc = (HAS_DPE && l == N_DGRAD) ? IDESC64 : IDESC;
          for (int kc = 0; kc < 4; ++kc) {
            mbar_wait(&sm.a_ready[kc], pass & 1);        // every pass of this kernel is a TMEM-operand pass
            tc_fence_after();
            mma_chunk_ts(pp, tmem, kc, idesc, first);
          }
          mma_commit(sm.d_ready);
          ++pass;
        }
      }
    }
  } else {
    EpiThread et; et.init(tmem);
    const int m = et.m, j = et.j;
    uint32_t d_par = 0, aux_par = 0;
    const float inv_dgrad = inv_sg * (1.0f / S_W);        // D = (S_g dZ)(S_w W)
    const uint16_t* bits16 = reinterpret_cast<const uint16_t*>(P.img.bits);
    const int col_lane = lane >> 1;                        // warp_colsum16: lanes 2k, 2k+1 hold column k
    for (int t = blockIdx.x; t < ti.total; t += gridDim.x) {
      const int gt = ti.global_tile(t);
      const int64_t row = (int64_t)gt * TM + m;
      // ---------------- output layer: tanh', bias gradient, the 64-wide dZ_L image, dA_{L-1}
      float dzl[OUT];
#pragma unroll
      for (int jj = 0; jj < OUT; ++jj) {
        const float yv = P.y[row * OUT + jj];
        dzl[jj] = P.dy[row * OUT + jj] * (P.tanh_out ? (1.0f - yv * yv) : 1.0f);
      }
      if (j == 0) {
#pragma unroll
        for (int jj = 0; jj < OUT; ++jj) {
          float sj = dzl[jj];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) sj += __shfl_xor_sync(0xffffffffu, sj, o);
          if (lane == 0 && sj != 0.f) atomicAdd(P.grads + P.b_off[L - 1] + jj, sj);
        }
        // image row: columns 0..OUT-1 = S_g * dz, rest zero
        uint32_t h0, l0, h1 = 0, l1 = 0;
        split2_f16(dzl[0] * s_g, OUT > 1 ? dzl[OUT > 1 ? 1 : 0] * s_g : 0.f, h0, l0);
        if (OUT == 3) split2_f16(dzl[OUT - 1] * s_g, 0.f, h1, l1);
        char* g_hi = P.img.dzl + (int64_t)gt * ATOM_BYTES;
        char* g_lo = g_hi + P.img.w64_term_stride;
        const int r = m & 7;
        const int base = (m >> 3) * 1024 + r * 128;
#pragma unroll
        for (int c16 = 0; c16 < 8; ++c16) {
          const int off = base + ((c16 ^ r) << 4);
          *reinterpret_cast<uint4*>(g_hi + off) = c16 == 0 ? make_uint4(h0, h1, 0, 0) : make_uint4(0, 0, 0, 0);
          *reinterpret_cast<uint4*>(g_lo + off) = c16 == 0 ? make_uint4(l0, l1, 0, 0) : make_uint4(0, 0, 0, 0);
        }
      }
      // dA_{L-1}[k] = sum_j dz[j] W_last[j][k], masked by relu'(h_{L-2}) -> dZ_{L-2}
      {
        char* img = P.img.dz + (int64_t)(L - 2) * P.img.slot_stride + (int64_t)gt * TILE_IMG_BYTES;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int c0 = et.col0(c);
          const uint32_t bits = bits16[((int64_t)(L - 2) * P.img.rows + row) * 16 + (c0 >> 4)];
          float v[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float a = 0.f;
#pragma unroll
            for (int jj = 0; jj < OUT; ++jj) a = fmaf(dzl[jj], s_wlast[jj * KLAST + c0 + i], a);
            v[i] = ((bits >> (15 - i)) & 1u) ? a : 0.f;
          }
          {
            const float cs = warp_colsum16(v, lane);
            if (!(lane & 1)) atomicAdd(&s_bacc[(L - 2) * 256 + c0 + col_lane], cs);
          }
          uint32_t ph[8], pl[8];
          const uint64_t sg2 = pack2f(s_g, s_g);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float w0, w1;
            unpack2f(mul2(pack2f(v[2 * i], v[2 * i + 1]), sg2), w0, w1);
            split2_packed(w0, w1, ph[i], pl[i]);
          }
          tmem_st8(et.tlane + TM_AHI + c0 / 2, ph);
          tmem_st8(et.tlane + TM_ALO + c0 / 2, pl);
          tmem_st_wait();
          tc_fence_before();
          mbar_arrive(&sm.a_ready[c]);
          char* g = img + c * ATOM_BYTES;
          stage_quad<KCfg<ATLAS>::STAGING_BUFS>(et, sm.staging, c, ph, pl, g, g + P.img.term_stride);
        }
      }
      // ---------------- hidden layers: dA_l = dZ_l W_l  ->  dZ_{l-1}
#pragma unroll 1
      for (int l = L - 2; l >= LOW; --l) {
        mbar_wait(sm.d_ready, d_par); d_par ^= 1;
        tc_fence_after();
        uint32_t raw[4][16];
#pragma unroll
        for (int c = 0; c < 4; ++c) tmem_ld16(et.tlane + TM_D + et.col0(c), raw[c]);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(sm.d_free);
        const int slot = l - 1;                           // produces dZ_{l-1}
        const bool need_img = ATLAS || slot >= 1;         // mapping dZ_0 feeds only the CUDA-core layer-0 gradient
        const bool need_tmem = HAS_DPE ? true : (slot >= 1);   // dZ_0 is an MMA operand only for the dPE product
        char* img = P.img.dz + (int64_t)slot * P.img.slot_stride + (int64_t)gt * TILE_IMG_BYTES;
        float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!ATLAS && slot == 0) xv = *reinterpret_cast<const float4*>(P.x + row * 4);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int c0 = et.col0(c);
          const uint32_t bits = bits16[((int64_t)slot * P.img.rows + row) * 16 + (c0 >> 4)];
          float v[16];
          const uint64_t invd2 = pack2f(inv_dgrad, inv_dgrad);
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            float a0, a1;
            unpack2f(mul2(pack2u(raw[c][i], raw[c][i + 1]), invd2), a0, a1);
            v[i] = ((bits >> (15 - i)) & 1u) ? a0 : 0.f;
            v[i + 1] = ((bits >> (14 - i)) & 1u) ? a1 : 0.f;
          }
          {
            const float cs = warp_colsum16(v, lane);
            if (!(lane & 1)) atomicAdd(&s_bacc[slot * 256 + c0 + col_lane], cs);
          }
          if (!ATLAS && slot == 0) {
            // layer-0 weight gradient dW0[n][d] = sum_m dZ0[m][n] * x[m][d]
            const int n = c0 + col_lane;
            float w[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) w[i] = v[i] * xv.x;
            float cs = warp_colsum16(w, lane);
            if (!(lane & 1)) atomicAdd(&s_w0acc[n * 3 + 0], cs);
#pragma unroll
            for (int i = 0; i < 16; ++i) w[i] = v[i] * xv.y;
            cs = warp_colsum16(w, lane);
            if (!(lane & 1)) atomicAdd(&s_w0acc[n * 3 + 1], cs);
#pragma unroll
            for (int i = 0; i < 16; ++i) w[i] = v[i] * xv.z;
            cs = warp_colsum16(w, lane);
            if (!(lane & 1)) atomicAdd(&s_w0acc[n * 3 + 2], cs);
          }
          if (need_img || need_tmem) {
            uint32_t ph[8], pl[8];
            const uint64_t sg2 = pack2f(s_g, s_g);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float w0, w1;
              unpack2f(mul2(pack2f(v[2 * i], v[2 * i + 1]), sg2), w0, w1);
              split2_packed(w0, w1, ph[i], pl[i]);
            }
            if (need_tmem) {
              tmem_st8(et.tlane + TM_AHI + c0 / 2, ph);
              tmem_st8(et.tlane + TM_ALO + c0 / 2, pl);
              tmem_st_wait();
              tc_fence_before();
              mbar_arrive(&sm.a_ready[c]);
            }
            if (need_img) {
              char* g = img + c * ATOM_BYTES;
              stage_quad<KCfg<ATLAS>::STAGING_BUFS>(et, sm.staging, c, ph, pl, g, g + P.img.term_stride);
            }
          }
        }
      }
      if (HAS_DPE) {
        // ---------------- dPE = dZ_0 W_0 (64 columns, 40 real) -> d(in) -> d_in += in_scale * d(in)
        mbar_wait(sm.d_ready, d_par); d_par ^= 1;
        tc_fence_after();
        mbar_wait(&sm.misc[0], aux_par);                  // PE tile of this row block
        uint32_t raw[16];                                 // slice j holds accumulator columns [16j, 16j + 16)
        tmem_ld16(et.tlane + TM_D + j * 16, raw);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(sm.d_free);
        float din[2] = {0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int col = j * 16 + i;
          if (col < PE_COLS) {
            const int k = col >> 2, e = col & 3;           // e: 0,1 = sin(x0),sin(x1); 2,3 = cos(x0),cos(x1)
            const float g = __uint_as_float(raw[i]) * inv_dgrad;
            const int pcol = (e < 2) ? col + 2 : col - 2;       // d sin = cos * b,  d cos = -sin * b
            const int off = atom_off(m, pcol);
            const float partner = (__half2float(*reinterpret_cast<const __half*>(sm.aux + off)) +
                                   __half2float(*reinterpret_cast<const __half*>(sm.aux + ATOM_BYTES + off))) *
                                  (1.0f / S_ACT);
            const float bk = pe_freq(k);
            din[e & 1] += (e < 2) ? g * partner * bk : -g * partner * bk;
          }
        }
        if (j > 0) { s_xch[((j - 1) * TM + m) * 2] = din[0]; s_xch[((j - 1) * TM + m) * 2 + 1] = din[1]; }
        named_bar(BAR_EPI, EPI_THREADS);
        if (j == 0 && P.d_in) {
          float2* dst = reinterpret_cast<float2*>(P.d_in + row * 2);
          float2 cur = P.d_in_accumulate ? *dst : make_float2(0.f, 0.f);
          cur.x += P.in_scale * (((din[0] + s_xch[m * 2]) + s_xch[(TM + m) * 2]) + s_xch[(2 * TM + m) * 2]);
          cur.y += P.in_scale * (((din[1] + s_xch[m * 2 + 1]) + s_xch[(TM + m) * 2 + 1]) + s_xch[(2 * TM + m) * 2 + 1]);
          *dst = cur;
          float mx = fmaxf(fabsf(cur.x), fabsf(cur.y));
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
          if (lane == 0 && mx > 0.f) atomicMax(P.gmax_bits + 1, __float_as_int(mx));
        }
        named_bar(BAR_EPI, EPI_THREADS);                  // s_xch reuse
        tc_fence_before();
        mbar_arrive(&sm.misc[1]);                         // aux tile may be overwritten
        aux_par ^= 1;
      }
    }
    if (j == 0 && lane == 0) bulk_wait_all0();
    // flush the per-CTA accumulators
    named_bar(BAR_EPI, EPI_THREADS);
    for (int i = et.tid; i < (L - 1) * 256; i += EPI_THREADS) {
      const float v = s_bacc[i];
      if (v != 0.f) atomicAdd(P.grads + P.b_off[i >> 8] + (i & 255), v);
    }
    if (!ATLAS)
      for (int i = et.tid; i < 768; i += EPI_THREADS) {
        const float v = s_w0acc[i];
        if (v != 0.f) atomicAdd(P.grads + P.w_off[0] + i, v);
      }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, TMEM_COLS);
}

// =============================================================================================
// weight gradients:  dW[n][k] += sum_rows dZ[row][n] * H[row][k]
// =============================================================================================
struct WgradItem {
  const char* a_img;      // dZ image, hi (lo at +a_term): 256 wide [tile][4 atoms][16 KB] or 64 wide [tile][16 KB]
  const char* b_img;      // input image, hi (lo at +b_term): same two shapes
  int64_t a_term, b_term;
  float* out; int ld_out; // fp32 dW block [a_cols rows][ld_out], columns [0, n_cols)
  int a_cols;             // 256: two M=128 MMAs;  64: one M=64 MMA (output-layer gradient, n_rows real rows)
  int b_cols;             // 256 or 64
  int n_rows, n_cols;     // real rows / columns to write
  int cap, n_groups;      // row geometry of the network this item belongs to
  int split, n_split;     // this CTA's share of the live tiles
  int mapping;            // 1: gradients of the mapping network (second gradient scale)
  int flow_groups;        // row geometry: compacted flow-match groups (mapping batch of the loop)
};
constexpr int MAX_WGRAD_ITEMS = 768;
struct WgradItems { WgradItem it[MAX_WGRAD_ITEMS]; int n; long long cycles[256]; };   // cycles: per-CTA duration (diagnostics)

constexpr int WG_STAGE = 65536;          // 32 rows: A hi 16K | A lo 16K | B hi 16K | B lo 16K, each [atom][4 groups][1 KB]
constexpr int WG_NSTAGE = 3;
constexpr int WG_SMEM = WG_NSTAGE * WG_STAGE + 256;
constexpr int WG_THREADS = 192;

// Work units ("items" = one dW GEMM restricted to a share of the rows) are dealt round-robin: CTA b processes items b,
// b + grid, b + 2 grid, ... (WG_UNITS_PER_CTA of them; the host builds the list).  The operand ring runs across units; the
// accumulator is flushed (vector atomics) after every unit.
__global__ void __launch_bounds__(WG_THREADS, 1)
tc_wgrad_kernel(const WgradItems* __restrict__ items, const int* __restrict__ n_valid, const int* __restrict__ gmax_bits) {
  extern __shared__ __align__(1024) char smem_raw[];
  char* p = smem_raw;
  char* stage = p;
  uint64_t* full = reinterpret_cast<uint64_t*>(p + WG_NSTAGE * WG_STAGE);
  uint64_t* empty = full + WG_NSTAGE;
  uint64_t* d_ready = empty + WG_NSTAGE;
  uint64_t* d_free = d_ready + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d_free + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    if (smem_u32(stage) & 1023u) { printf("b200: dynamic shared memory is not 1024-byte aligned\n"); __trap(); }
    for (int i = 0; i < WG_NSTAGE; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(d_ready, 1);
    mbar_init(d_free, WG_THREADS - 64);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int n_items = items->n;
  const long long t_start = clock64();

  if (warp == 0) {
    if (lane == 0) {
      uint32_t gs = 0;                                  // running stage counter across units
      for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
        const WgradItem W = items->it[it];
        TileIter ti; ti.init(W.cap, W.n_groups, n_valid, W.flow_groups);
        const int t_begin = (int)((int64_t)ti.total * W.split / W.n_split);
        const int t_end = (int)((int64_t)ti.total * (W.split + 1) / W.n_split);
        const int a_atoms = W.a_cols / 64, b_atoms = W.b_cols / 64;
        const int n_steps = (t_end - t_begin) * 4;     // 32-row steps
        for (int s = 0; s < n_steps; ++s, ++gs) {
          const int slot = gs % WG_NSTAGE;
          mbar_wait(&empty[slot], ((gs / WG_NSTAGE) & 1) ^ 1);
          const int gt = ti.global_tile(t_begin + (s >> 2));
          const int ch = s & 3;                        // 32-row chunk = groups 4ch .. 4ch+3 of every atom block
          char* dst = stage + slot * WG_STAGE;
          mbar_expect_tx(&full[slot], 2 * 4096 * (a_atoms + b_atoms));
          const char* a = W.a_img + (int64_t)gt * a_atoms * ATOM_BYTES + ch * 4096;
          for (int j = 0; j < a_atoms; ++j) {
            bulk_g2s(dst + j * 4096, a + (int64_t)j * ATOM_BYTES, 4096, &full[slot]);
            bulk_g2s(dst + 16384 + j * 4096, a + W.a_term + (int64_t)j * ATOM_BYTES, 4096, &full[slot]);
          }
          const char* b = W.b_img + (int64_t)gt * b_atoms * ATOM_BYTES + ch * 4096;
          for (int j = 0; j < b_atoms; ++j) {
            bulk_g2s(dst + 32768 + j * 4096, b + (int64_t)j * ATOM_BYTES, 4096, &full[slot]);
            bulk_g2s(dst + 49152 + j * 4096, b + W.b_term + (int64_t)j * ATOM_BYTES, 4096, &full[slot]);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t gs = 0, unit = 0;
      for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
        const WgradItem W = items->it[it];
        TileIter ti; ti.init(W.cap, W.n_groups, n_valid, W.flow_groups);
        const int t_begin = (int)((int64_t)ti.total * W.split / W.n_split);
        const int t_end = (int)((int64_t)ti.total * (W.split + 1) / W.n_split);
        const int n_steps = (t_end - t_begin) * 4;
        if (n_steps == 0) continue;
        // smem operand: [atom][4 groups][1 KB] -> MN-major SW128: LBO (atom stride) 4096, SBO (8-row group) 1024
        const int m_inst = W.a_cols == 256 ? 128 : 64;
        const uint32_t idesc = make_idesc(m_inst, W.b_cols, 1, 1);
        const int m_halves = W.a_cols == 256 ? 2 : 1;
        if (unit > 0) { mbar_wait(d_free, (unit - 1) & 1); tc_fence_after(); }   // previous accumulator flushed
        for (int s = 0; s < n_steps; ++s, ++gs) {
          const int slot = gs % WG_NSTAGE;
          mbar_wait(&full[slot], (gs / WG_NSTAGE) & 1);
          tc_fence_after();
          const uint32_t sb = smem_u32(stage + slot * WG_STAGE);
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {             // 16 rows = 2 groups per MMA
            for (int mh = 0; mh < m_halves; ++mh) {
              const uint32_t acc = (s | ks) ? 1u : 0u;
              const uint32_t d = tmem + mh * W.b_cols;
              const uint64_t a_hi = make_desc(sb + ks * 2048 + mh * 8192, 4096, 1024);
              const uint64_t a_lo = make_desc(sb + 16384 + ks * 2048 + mh * 8192, 4096, 1024);
              const uint64_t b_hi = make_desc(sb + 32768 + ks * 2048, 4096, 1024);
              const uint64_t b_lo = make_desc(sb + 49152 + ks * 2048, 4096, 1024);
              mma_ss(d, a_hi, b_hi, idesc, acc);
              mma_ss(d, a_hi, b_lo, idesc, 1u);
              mma_ss(d, a_lo, b_hi, idesc, 1u);
            }
          }
          mma_commit(&empty[slot]);
        }
        mma_commit(d_ready);
        ++unit;
      }
    }
  } else {
    float s_gm, inv_gm, s_ga, inv_ga;
    grad_scales(gmax_bits, true, s_gm, inv_gm);
    grad_scales(gmax_bits, false, s_ga, inv_ga);
    const int q = warp & 3;
    const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
    uint32_t unit = 0;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
      const WgradItem W = items->it[it];
      TileIter ti; ti.init(W.cap, W.n_groups, n_valid, W.flow_groups);
      const int t_begin = (int)((int64_t)ti.total * W.split / W.n_split);
      const int t_end = (int)((int64_t)ti.total * (W.split + 1) / W.n_split);
      if (t_end == t_begin) continue;
      const float inv = (W.mapping ? inv_gm : inv_ga) * (1.0f / S_ACT);
      mbar_wait(d_ready, unit & 1);
      tc_fence_after();
      const int m_halves = W.a_cols == 256 ? 2 : 1;
      for (int mh = 0; mh < m_halves; ++mh) {
        // M=128: accumulator row i of half mh lives in TMEM lane i.  M=64: rows 0..15 in lanes 0..15 of quadrant 0.
        const int n = mh * 128 + q * 32 + lane;              // layer output index of this thread's accumulator row
        const bool live = W.a_cols == 256 ? true : (q == 0 && lane < W.n_rows);
        float* orow = W.out + (int64_t)n * W.ld_out;
        for (int c = 0; c < W.b_cols / 32; ++c) {
          uint32_t raw[32];
          tmem_ld32(tlane + mh * W.b_cols + c * 32, raw);
          tmem_ld_wait();
          if (!live) continue;
          if (((W.ld_out & 3) == 0) && c * 32 + 32 <= W.n_cols) {
#pragma unroll
            for (int i = 0; i < 32; i += 4)
              atomicAdd(reinterpret_cast<float4*>(orow + c * 32 + i),
                        make_float4(__uint_as_float(raw[i]) * inv, __uint_as_float(raw[i + 1]) * inv,
                                    __uint_as_float(raw[i + 2]) * inv, __uint_as_float(raw[i + 3]) * inv));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c * 32 + i < W.n_cols) atomicAdd(orow + c * 32 + i, __uint_as_float(raw[i]) * inv);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(d_free);                                   // the MMA warp may overwrite the accumulator
      ++unit;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0 && blockIdx.x < 256) const_cast<WgradItems*>(items)->cycles[blockIdx.x] = clock64() - t_start;
  if (warp == 1) tmem_dealloc(tmem, TMEM_COLS);
}

// =============================================================================================
// host side
// =============================================================================================
static int g_sm_count = 0;
static int sm_count() {
  if (!g_sm_count) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev);
    if (g_sm_count <= 0) g_sm_count = 148;
  }
  return g_sm_count;
}

TcNet tc_classify(const MlpShape& s) {
  if (s.hidden != HID) return TcNet::None;
  uint32_t skips = 0;
  for (int l = 1; l < s.L; ++l)
    if (s.skip[l]) skips |= 1u << l;
  if ((s.L == 6 || s.L == 4) && s.pe == 0 && s.in_dim == 3 && s.out_dim == 2 && !skips)
    return s.L == 6 ? TcNet::Mapping6 : TcNet::Mapping4;
  if (s.L == 8 && s.pe == 10 && s.in_dim == 2 && s.out_dim == 3 && skips == ((1u << 4) | (1u << 7))) return TcNet::Atlas;
  if (s.L == 8 && s.pe == 5 && s.in_dim == 3 && s.out_dim == 1 && !skips) return TcNet::Alpha;
  return TcNet::None;
}

// the fused forward / backward kernels of a network family and their dynamic shared memory
struct TcKernels { void (*fwd)(FwdParams); void (*bwd)(BwdParams); int smem; };
static TcKernels kernels_of(TcNet net) {
  switch (net) {
    case TcNet::Mapping6: return {tc_fwd_kernel<false>, tc_bwd_kernel<false>, KCfg<false>::SMEM};
    case TcNet::Mapping4: return {tc_fwd_kernel<false, 4>, tc_bwd_kernel<false, 4>, KCfg<false>::SMEM};
    case TcNet::Atlas: return {tc_fwd_kernel<true>, tc_bwd_kernel<true>, KCfg<true>::SMEM};
    case TcNet::Alpha: return {tc_fwd_kernel<true, 8, 1>, tc_bwd_kernel<true, 8, 1>, KCfg<true>::SMEM};
    default: return {nullptr, nullptr, 0};
  }
}

// the fused kernels are persistent: at most one CTA per SM walks over the `tiles` 128-row tiles
static void launch_fwd(TcNet net, int tiles, const FwdParams& P, cudaStream_t st) {
  const TcKernels k = kernels_of(net);
  k.fwd<<<min(sm_count(), tiles), TC_THREADS, k.smem, st>>>(P);
}
static void launch_bwd(TcNet net, int tiles, const BwdParams& P, cudaStream_t st) {
  const TcKernels k = kernels_of(net);
  k.bwd<<<min(sm_count(), tiles), TC_THREADS, k.smem, st>>>(P);
}

static int ensure_attrs() {
  // cudaFuncSetAttribute is per device: remember which devices of this process have been configured
  static bool done_dev[64] = {};
  int dev = 0;
  B200_CHECK_CUDA(cudaGetDevice(&dev));
  B200_REQUIRE(dev >= 0 && dev < 64, "device ordinal %d out of range", dev);
  bool& done = done_dev[dev];
  if (done) return B200_OK;
  for (TcNet net : {TcNet::Mapping6, TcNet::Mapping4, TcNet::Atlas, TcNet::Alpha}) {
    const TcKernels k = kernels_of(net);
    B200_CHECK_CUDA(cudaFuncSetAttribute(k.fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, k.smem));
    B200_CHECK_CUDA(cudaFuncSetAttribute(k.bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, k.smem));
  }
  B200_CHECK_CUDA(cudaFuncSetAttribute(tc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM));
  done = true;
  return B200_OK;
}

static void add_prep(PrepJobs& pj, const float* W, int ldw, int n_rows, int k0, int k_cnt, int transpose, char* dst) {
  PrepJob& j = pj.j[pj.n++];
  j.W = W; j.ldw = ldw; j.n_rows = n_rows; j.k0 = k0; j.k_cnt = k_cnt; j.transpose = transpose;
  j.hi = dst; j.lo = dst + STAGE_BYTES;
}


// ---- table builders shared by the cached (training loop) and the ephemeral (stand-alone IMLP) paths
static void prep_jobs_for_net(PrepJobs& pj, const MlpShape& sh, const NetImages& im, const float* pp, TcNet net,
                              bool with_bwd) {
  const bool is_atlas = tc_pe_kernels(net);
  for (int l = 0; l < sh.L; ++l) {
    char* dst = im.w_fwd + im.w_fwd_layer[l];
    if (im.n_chunks_fwd[l] == 0) continue;
    const float* W = pp + sh.w_off[l];
    int item = 0;
    if (l > 0) for (int kc = 0; kc < 4; ++kc) add_prep(pj, W, sh.K[l], 256, kc * 64, 64, 0, dst + (int64_t)(item++) * 2 * STAGE_BYTES);
    if (is_atlas && (l == 0 || sh.skip[l]))
      add_prep(pj, W, sh.K[l], 256, l == 0 ? 0 : 256, sh.enc, 0, dst + (int64_t)(item++) * 2 * STAGE_BYTES);
  }
  if (!with_bwd) return;
  for (int l = 0; l < sh.L - 1; ++l) {
    // the atlas network back-propagates to its input (uv) through the positional encoding; the alpha network's inputs
    // are pixel coordinates
    if (l < 1 && net != TcNet::Atlas) continue;
    char* dst = im.w_bwd + im.w_bwd_layer[l];
    const float* W = pp + sh.w_off[l];
    // image rows = input index k of layer l (256, or 40 for atlas layer 0), chunk over the output index n
    const int rows = (is_atlas && l == 0) ? sh.enc : 256;
    for (int kc = 0; kc < 4; ++kc) add_prep(pj, W, sh.K[l], rows, kc * 64, 64, 1, dst + (int64_t)kc * 2 * STAGE_BYTES);
  }
}

// wgrad work list.  The kernel is HBM-bound: CTAs are balanced by bytes read per tile
// (A + B, both terms) corrected by the measured cost of narrow steps (step_cost): with plain byte counts the CTAs of
// the narrow GEMMs ran 1.3 - 1.6x longer than everyone else and the average SM idled 43 % of the kernel
// measured per-CTA busy time of the kernel at the benchmark shape (tests/perf/wgrad_balance.py), per 32-row step, in units
// of "image columns loaded": a 256x256 step (512 columns, 64 KB) is HBM-bound; a 320-column step costs 0.81 of it
// rather than 0.625, a 128-column step 0.66 rather than 0.25 (barrier round trips and M=64 / N=64 MMAs do not shrink)
static double step_cost(int cols) { return cols >= 512 ? 512.0 : (cols >= 320 ? 416.0 : 340.0); }

struct WgProto { const char* a; int64_t a_term; int a_cols; const char* b; int64_t b_term; int b_cols;
                 float* out; int ld; int n_rows, n_cols, groups; double bytes; int mapping; };

static void protos_for_net(WgProto* protos, int& np, const MlpShape& sh, const NetImages& im, float* g, TcNet net,
                           int groups) {
  const bool is_atlas = tc_pe_kernels(net);
  auto add = [&](const char* a, int64_t a_term, int a_cols, const char* b, int64_t b_term, int b_cols, float* out, int ld,
                 int n_rows, int n_cols) {
    protos[np++] = WgProto{a, a_term, a_cols, b, b_term, b_cols, out, ld, n_rows, n_cols, groups,
                           (double)groups * step_cost(a_cols + b_cols), is_atlas ? 0 : 1};
  };
  for (int l = 1; l <= sh.L - 2; ++l)
    add(im.dz + (int64_t)l * im.slot_stride, im.term_stride, 256, im.act + (int64_t)(l - 1) * im.slot_stride,
        im.term_stride, 256, g + sh.w_off[l], sh.K[l], 256, 256);
  add(im.dzl, im.w64_term_stride, 64, im.act + (int64_t)(sh.L - 2) * im.slot_stride, im.term_stride, 256,
      g + sh.w_off[sh.L - 1], sh.K[sh.L - 1], sh.out_dim, 256);
  if (is_atlas) {
    // positional-encoding parts: layer 0 and the skip layers; output layer's skip part
    add(im.dz, im.term_stride, 256, im.pe, im.w64_term_stride, 64, g + sh.w_off[0], sh.K[0], 256, sh.enc);
    for (int l = 1; l <= sh.L - 2; ++l)
      if (sh.skip[l])
        add(im.dz + (int64_t)l * im.slot_stride, im.term_stride, 256, im.pe, im.w64_term_stride, 64, g + sh.w_off[l] + 256,
            sh.K[l], 256, sh.enc);
    if (sh.skip[sh.L - 1])
      add(im.dzl, im.w64_term_stride, 64, im.pe, im.w64_term_stride, 64, g + sh.w_off[sh.L - 1] + 256, sh.K[sh.L - 1],
          sh.out_dim, sh.enc);
  }
}

// One CTA per SM (each CTA owns all 512 TMEM columns); the GEMMs are cut into WG_UNITS_PER_CTA x SMs units of equal
// cost (largest-remainder apportionment) that the CTAs take round-robin (see tc_wgrad_kernel).  More than one unit
// per CTA balances any cost-model error but multiplies the accumulator flushes (64 K fp32 vector atomics each): 4 units
// per CTA cost as much in L2 atomics as they gained in balance (measured), so the default is 1.
constexpr int WG_UNITS_PER_CTA = 1;
static void apportion_items(WgradItems& wi, const WgProto* protos, int np, int cap, int flow_groups) {
  double total_bytes = 0;
  for (int i = 0; i < np; ++i) total_bytes += protos[i].bytes;
  const int sms = sm_count() * WG_UNITS_PER_CTA;
  int n_split[32], used = 0;
  double frac[32];
  for (int i = 0; i < np; ++i) {
    const double want = protos[i].bytes / total_bytes * sms;
    n_split[i] = (int)want < 1 ? 1 : (int)want;
    frac[i] = want - (int)want;
    used += n_split[i];
  }
  while (used < sms) {
    int best = 0;
    for (int i = 1; i < np; ++i) if (frac[i] > frac[best]) best = i;
    ++n_split[best]; frac[best] = -1.0; ++used;
  }
  while (used > sms) {
    int best = -1;
    for (int i = 0; i < np; ++i) if (n_split[i] > 1 && (best < 0 || n_split[i] > n_split[best])) best = i;
    if (best < 0) break;
    --n_split[best]; --used;
  }
  for (int i = 0; i < np; ++i) {
    for (int sp = 0; sp < n_split[i] && wi.n < MAX_WGRAD_ITEMS; ++sp) {
      WgradItem& it = wi.it[wi.n++];
      const WgProto& pr = protos[i];
      it.a_img = pr.a; it.a_term = pr.a_term; it.a_cols = pr.a_cols;
      it.b_img = pr.b; it.b_term = pr.b_term; it.b_cols = pr.b_cols;
      it.out = pr.out; it.ld_out = pr.ld; it.n_rows = pr.n_rows; it.n_cols = pr.n_cols;
      it.cap = cap; it.n_groups = pr.groups; it.split = sp; it.n_split = n_split[i]; it.mapping = pr.mapping;
      it.flow_groups = (pr.mapping && flow_groups) ? 1 : 0;
    }
  }
}

// ---- job tables: PrepJobs (weight-image preparation) and WgradItems (weight-gradient work list).  They depend only on
// pointers and geometry.  Callers that keep their workspace and parameter / gradient buffers alive across calls (the
// fused loop, persistent stand-alone calls) have them built by one eager call into device allocations of their own and
// reuse them afterwards, inside captured graphs too; ephemeral callers get them uploaded into their workspace on every
// call.
enum TableKind { TABLE_PREP, TABLE_WGRAD };
// TableKey::nets of the fused loop (the mapping network alone in pre-training, with the atlas network in the loop); a
// stand-alone call uses its TcNet.  It also fixes the workspace layout the table points into.
constexpr int NETS_LOOP_MAPPING = 16, NETS_LOOP_ATLAS = 17;

struct TableKey {
  int dev; const void* ws; TableKind kind; int nets;
  int64_t rows; int groups;      // rows per group, groups
  const void* ptr;               // parameters (TABLE_PREP) or gradients (TABLE_WGRAD)
  int flow_groups; bool training;
  bool operator==(const TableKey& o) const {
    return dev == o.dev && ws == o.ws && kind == o.kind && nets == o.nets && rows == o.rows && groups == o.groups &&
           ptr == o.ptr && flow_groups == o.flow_groups && training == o.training;
  }
};
struct TableEntry { TableKey key; void* d; int n; };
// Captured graphs bake an entry's device pointer in, so an entry is NEVER recycled: the store only grows (up to ~60 KB
// of device memory per entry; one entry per table kind and (device, workspace, row geometry, parameter or gradient
// buffer)).
constexpr int MAX_TABLES = 4096;
static std::vector<TableEntry> g_tables;
static std::mutex g_tables_mutex;

static int current_device() { int d = 0; cudaGetDevice(&d); return d; }

static bool stream_is_capturing(cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cs);
  return cs == cudaStreamCaptureStatusActive;
}

static bool find_table(const TableKey& key, void** d, int* n) {
  std::lock_guard<std::mutex> lock(g_tables_mutex);
  for (const TableEntry& e : g_tables)
    if (e.key == key) { *d = e.d; *n = e.n; return true; }
  return false;
}

static int table_capacity(const PrepJobs&) { return MAX_PREP_JOBS; }
static int table_capacity(const WgradItems&) { return MAX_WGRAD_ITEMS; }

// The table of `key` (nullptr: an ephemeral caller) in *d_out / *n_out: found in the store, or built on the host by
// fill(table) and then kept in the store, or uploaded into `slot` in the caller's workspace when the caller is ephemeral
// or the store is full.  Building takes an eager call (a pageable copy).
template <class T, class Fill>
static int get_table(const TableKey* key, T* slot, cudaStream_t st, Fill fill, const T** d_out, int* n_out) {
  void* d = nullptr;
  if (key && find_table(*key, &d, n_out)) { *d_out = static_cast<const T*>(d); return B200_OK; }
  B200_REQUIRE(!stream_is_capturing(st), "tensor-core job tables are built by eager calls: run the same call once "
               "without stream capture first (only a persistent workspace keeps them for capture)");
  static thread_local T host;
  host = T{};
  fill(host);
  B200_REQUIRE(host.n <= table_capacity(host), "table overflow");
  *n_out = host.n;
  bool keep = key != nullptr;
  if (keep) {
    std::lock_guard<std::mutex> lock(g_tables_mutex);
    if ((int)g_tables.size() >= MAX_TABLES) {
      B200_REQUIRE(slot, "too many distinct tensor-core workspaces in one process (%d)", MAX_TABLES);
      keep = false;
    }
  }
  if (!keep) {
    B200_CHECK_CUDA(cudaMemcpyAsync(slot, &host, sizeof(T), cudaMemcpyHostToDevice, st));
    *d_out = slot;
    return B200_OK;
  }
  B200_CHECK_CUDA(cudaMalloc(&d, sizeof(T)));
  B200_CHECK_CUDA(cudaMemcpyAsync(d, &host, sizeof(T), cudaMemcpyHostToDevice, st));
  B200_CHECK_CUDA(cudaStreamSynchronize(st));
  std::lock_guard<std::mutex> lock(g_tables_mutex);
  g_tables.push_back(TableEntry{*key, d, host.n});
  *d_out = static_cast<const T*>(d);
  return B200_OK;
}

// Kernel parameters with the settings of the fused loop (network input x * 0.5 + 0.5, activation images stored, input
// gradient accumulated onto the loss head's); stand-alone calls override them.
static void fill_fwd(FwdParams& P, const MlpShape& sh, const NetImages& im, const float* x, float* y,
                     const float* params, int cap, int groups, const int* n_valid) {
  P.x = x; P.y = y; P.params = params; P.img = im; P.cap = cap; P.n_groups = groups; P.n_valid = n_valid;
  P.in_scale = 0.5f; P.in_shift = 0.5f; P.store_images = 1; P.tanh_out = sh.tanh_out ? 1 : 0; P.flow_groups = 0;
  for (int l = 0; l < sh.L; ++l) { P.w_off[l] = sh.w_off[l]; P.b_off[l] = sh.b_off[l]; }
}

static void fill_bwd(BwdParams& P, const MlpShape& sh, const NetImages& im, const float* dy, const float* y,
                     const float* x, float* d_in, const float* params, float* grads, int cap, int groups,
                     const int* n_valid, int* gmax_bits) {
  P.dy = dy; P.y = y; P.x = x; P.d_in = d_in; P.params = params; P.grads = grads; P.img = im;
  P.cap = cap; P.n_groups = groups; P.n_valid = n_valid; P.gmax_bits = gmax_bits;
  P.in_scale = 0.5f; P.d_in_accumulate = 1; P.tanh_out = sh.tanh_out ? 1 : 0; P.flow_groups = 0;
  for (int l = 0; l < sh.L; ++l) { P.w_off[l] = sh.w_off[l]; P.b_off[l] = sh.b_off[l]; }
}

// tables of the fused loop: the prep table depends on the parameters, the wgrad table on the gradients
static TableKey loop_key(const TcStep& s, TableKind kind) {
  return TableKey{current_device(), s.plan->base, kind, s.y_atlas ? NETS_LOOP_ATLAS : NETS_LOOP_MAPPING, s.cap,
                  s.n_groups, kind == TABLE_PREP ? static_cast<const void*>(s.params) : s.grads, s.flow_groups, true};
}

// The weight images depend only on the parameters, so their preparation runs on a side stream, forked from the
// caller's stream before the sampling kernels and joined before the first fused kernel (also under capture: the
// fork / join become parallel branches of the graph).
struct SideStream { cudaStream_t stream = nullptr; cudaEvent_t fork = nullptr, join = nullptr; bool pending = false; };
static SideStream g_side[64];

int tc_begin_step(const TcStep& s, cudaStream_t st) {
  B200_PROPAGATE(ensure_attrs());
  B200_REQUIRE(tc_classify(*s.ms) == TcNet::Mapping6 && tc_classify(*s.as) == TcNet::Atlas,
               "tensor-core path is specialised to the two stage-1 networks");
  const TcLayout lay = layout_of(s);
  const bool atlas = s.y_atlas != nullptr;
  const TableKey kp = loop_key(s, TABLE_PREP), kw = loop_key(s, TABLE_WGRAD);
  const PrepJobs* d_prep; int n_prep;
  const WgradItems* d_wg; int n_wg;
  // forward / dgrad weight images (the atlas network only where it is evaluated: not in pre-training)
  B200_PROPAGATE(get_table<PrepJobs>(&kp, nullptr, st, [&](PrepJobs& pj) {
    prep_jobs_for_net(pj, *s.ms, lay.map, s.params, TcNet::Mapping6, true);
    if (atlas) prep_jobs_for_net(pj, *s.as, lay.atl, s.params + s.ms->total, TcNet::Atlas, true);
  }, &d_prep, &n_prep));
  // wgrad items, for run_backward
  B200_PROPAGATE(get_table<WgradItems>(&kw, nullptr, st, [&](WgradItems& wi) {
    WgProto protos[32]; int np = 0;
    protos_for_net(protos, np, *s.ms, lay.map, s.grads, TcNet::Mapping6, s.n_groups);
    if (atlas) protos_for_net(protos, np, *s.as, lay.atl, s.grads + s.ms->total, TcNet::Atlas, 3);
    apportion_items(wi, protos, np, s.cap, s.flow_groups);
  }, &d_wg, &n_wg));
  SideStream& sd = g_side[current_device()];
  if (!sd.stream) {
    B200_CHECK_CUDA(cudaStreamCreateWithFlags(&sd.stream, cudaStreamNonBlocking));
    B200_CHECK_CUDA(cudaEventCreateWithFlags(&sd.fork, cudaEventDisableTiming));
    B200_CHECK_CUDA(cudaEventCreateWithFlags(&sd.join, cudaEventDisableTiming));
  }
  B200_CHECK_CUDA(cudaEventRecord(sd.fork, st));
  B200_CHECK_CUDA(cudaStreamWaitEvent(sd.stream, sd.fork, 0));
  // weight images of both networks — every step, since Adam changed the parameters
  tc_prep_kernel<<<n_prep * 4, 128, 0, sd.stream>>>(d_prep);
  B200_CHECK_LAUNCH();
  B200_CHECK_CUDA(cudaEventRecord(sd.join, sd.stream));
  sd.pending = true;
  return B200_OK;
}

static int run_forward(const TcStep& s, bool with_atlas, cudaStream_t st) {
  const TcLayout lay = layout_of(s);
  SideStream& sd = g_side[current_device()];
  if (!sd.pending) B200_PROPAGATE(tc_begin_step(s, st));     // callers that did not fork earlier
  B200_CHECK_CUDA(cudaStreamWaitEvent(st, sd.join, 0));
  sd.pending = false;
  FwdParams pm{};
  fill_fwd(pm, *s.ms, lay.map, s.x_map, s.uv, s.params, s.cap, s.n_groups, s.counters);
  pm.flow_groups = s.flow_groups;
  timer_begin(TAG_MAP_FWD, st);
  launch_fwd(TcNet::Mapping6, s.n_groups * (s.cap / TM), pm, st);
  timer_end(TAG_MAP_FWD, st);
  B200_CHECK_LAUNCH();
  if (with_atlas) {
    FwdParams pa{};
    fill_fwd(pa, *s.as, lay.atl, s.uv, s.y_atlas, s.params + s.ms->total, s.cap, 3, s.counters);
    timer_begin(TAG_ATLAS_FWD, st);
    launch_fwd(TcNet::Atlas, 3 * (s.cap / TM), pa, st);
    timer_end(TAG_ATLAS_FWD, st);
    B200_CHECK_LAUNCH();
  }
  return B200_OK;
}

static const WgradItems* g_last_wg = nullptr;
static int g_last_wg_n = 0;

// diagnostics: per-CTA cycle counts and (a_cols, b_cols, n_split) of the item each CTA ran in the last weight-gradient launch
int tc_debug_wgrad(long long* cycles, int* shapes, int max_ctas) {
  if (!g_last_wg) { set_error("no weight-gradient launch yet"); return -1; }
  static WgradItems host;
  if (cudaMemcpy(&host, g_last_wg, sizeof(WgradItems), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  const int n = g_last_wg_n < max_ctas ? g_last_wg_n : max_ctas;
  for (int i = 0; i < n; ++i) {
    cycles[i] = host.cycles[i];
    shapes[3 * i] = host.it[i].a_cols; shapes[3 * i + 1] = host.it[i].b_cols; shapes[3 * i + 2] = host.it[i].n_split;
  }
  return n;
}

static int run_backward(const TcStep& s, bool with_atlas, cudaStream_t st) {
  const TcLayout lay = layout_of(s);
  void* tab; int n_wg;
  if (!find_table(loop_key(s, TABLE_WGRAD), &tab, &n_wg)) {
    set_error("tensor-core backward called before forward");
    return B200_ERR_INVALID;
  }
  const WgradItems* d_wg = static_cast<const WgradItems*>(tab);
  int* gmax = const_cast<int*>(s.counters) + 3;
  if (with_atlas) {
    BwdParams pa{};
    fill_bwd(pa, *s.as, lay.atl, s.d_y, s.y_atlas, nullptr, const_cast<float*>(s.d_uv), s.params + s.ms->total,
             s.grads + s.ms->total, s.cap, 3, s.counters, gmax);
    timer_begin(TAG_ATLAS_BWD, st);
    launch_bwd(TcNet::Atlas, 3 * (s.cap / TM), pa, st);
    timer_end(TAG_ATLAS_BWD, st);
    B200_CHECK_LAUNCH();
  }
  BwdParams pm{};
  fill_bwd(pm, *s.ms, lay.map, s.d_uv, s.uv, s.x_map, nullptr, s.params, s.grads, s.cap, s.n_groups, s.counters, gmax);
  pm.flow_groups = s.flow_groups;
  timer_begin(TAG_MAP_BWD, st);
  launch_bwd(TcNet::Mapping6, s.n_groups * (s.cap / TM), pm, st);
  timer_end(TAG_MAP_BWD, st);
  B200_CHECK_LAUNCH();
  timer_begin(TAG_WGRAD, st);
  g_last_wg = d_wg; g_last_wg_n = min(n_wg, sm_count());
  tc_wgrad_kernel<<<min(n_wg, sm_count()), WG_THREADS, WG_SMEM, st>>>(d_wg, s.counters, gmax);
  timer_end(TAG_WGRAD, st);
  B200_CHECK_LAUNCH();
  return B200_OK;
}


// ---------------------------------------------------------------------------------------------
// inference: mapping -> atlas on `rows` coordinate rows, no activation images (full-video render,
// evaluate.py:640-708).  Workspace: [PrepJobs table][forward weight images of both networks].
// ---------------------------------------------------------------------------------------------

static void plan_infer(const MlpShape& ms, const MlpShape& as, char* base, NetImages* im_map, NetImages* im_atl,
                       PrepJobs** d_prep, int64_t* bytes) {
  char* p = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(base), 1024));
  *d_prep = reinterpret_cast<PrepJobs*>(carve_tc(p, sizeof(PrepJobs)));
  *im_map = NetImages{};
  plan_fwd_images(ms, TcNet::Mapping6, p, im_map);
  *im_atl = NetImages{};
  plan_fwd_images(as, TcNet::Atlas, p, im_atl);
  *bytes = p - base;
}

int64_t tc_infer_workspace_bytes(const MlpShape& ms, const MlpShape& as) {
  NetImages a, b; PrepJobs* d; int64_t bytes = 0;
  plan_infer(ms, as, nullptr, &a, &b, &d, &bytes);
  return bytes + 2048;
}

int tc_infer_forward(const MlpShape& ms, const MlpShape& as, const float* params, const float* x_map, float* uv,
                     float* y, int64_t rows, char* ws, cudaStream_t st) {
  B200_PROPAGATE(ensure_attrs());
  B200_REQUIRE(tc_classify(ms) == TcNet::Mapping6 && tc_classify(as) == TcNet::Atlas,
               "tensor-core path is specialised to the two stage-1 networks");
  B200_REQUIRE(rows > 0 && rows % TM == 0 && rows / TM < (1 << 24), "rows must be a positive multiple of %d", TM);
  NetImages im_map, im_atl; PrepJobs* slot; int64_t bytes;
  plan_infer(ms, as, ws, &im_map, &im_atl, &slot, &bytes);
  // The job table lives in the caller's workspace and is rebuilt on every call (4 KB, pageable copy: the call is
  // not graph-capturable, which a render does not need) — nothing is cached, so a recycled workspace is harmless.
  B200_REQUIRE(!stream_is_capturing(st), "the tensor-core render is not graph-capturable");
  const PrepJobs* d_prep; int n_prep;
  B200_PROPAGATE(get_table(nullptr, slot, st, [&](PrepJobs& pj) {
    prep_jobs_for_net(pj, ms, im_map, params, TcNet::Mapping6, false);
    prep_jobs_for_net(pj, as, im_atl, params + ms.total, TcNet::Atlas, false);
  }, &d_prep, &n_prep));
  tc_prep_kernel<<<n_prep * 4, 128, 0, st>>>(d_prep);
  B200_CHECK_LAUNCH();
  const int tiles = (int)(rows / TM);
  FwdParams pm{};
  fill_fwd(pm, ms, im_map, x_map, uv, params, (int)rows, 1, nullptr);
  pm.store_images = 0;
  launch_fwd(TcNet::Mapping6, tiles, pm, st);
  B200_CHECK_LAUNCH();
  FwdParams pa{};
  fill_fwd(pa, as, im_atl, uv, y, params + ms.total, (int)rows, 1, nullptr);
  pa.store_images = 0;
  launch_fwd(TcNet::Atlas, tiles, pa, st);
  B200_CHECK_LAUNCH();
  return B200_OK;
}

// ---------------------------------------------------------------------------------------------
// stand-alone evaluation of ONE network with autograd support: what the `IMLP` class needs
// (implicit_neural_networks.py:62-81 forward + the autograd of its Linear/ReLU/tanh/skip stack).  Job tables are
// cached for persistent callers and uploaded into the workspace on every call otherwise (see get_table).
// Workspace: [PrepJobs][WgradItems][images of the network].
// ---------------------------------------------------------------------------------------------
struct SinglePlan { PrepJobs* d_prep; WgradItems* d_wg; NetImages im; int64_t bytes; };

static void plan_single(const MlpShape& sh, TcNet net, int64_t rows, char* base, SinglePlan* out) {
  char* p = reinterpret_cast<char*>(round_up(reinterpret_cast<int64_t>(base), 1024));
  out->d_prep = reinterpret_cast<PrepJobs*>(carve_tc(p, sizeof(PrepJobs)));
  out->d_wg = reinterpret_cast<WgradItems*>(carve_tc(p, sizeof(WgradItems)));
  plan_net(sh, rows, net, p, &out->im);
  out->bytes = p - base;
}

int64_t tc_single_workspace_bytes(const MlpShape& sh, TcNet net, int64_t rows) {
  SinglePlan pl;
  plan_single(sh, net, rows, nullptr, &pl);
  return pl.bytes + 2048;
}

static int check_single(const MlpShape& sh, TcNet net, int64_t rows) {
  B200_PROPAGATE(ensure_attrs());
  B200_REQUIRE(net != TcNet::None && tc_classify(sh) == net, "tensor-core IMLP: not one of the stage-1 architectures "
               "(mapping 3-256x{2,4}-2, atlas 2-PE10-256x6-3 with skips 4,7, alpha 3-PE5-256x6-1)");
  B200_REQUIRE(rows > 0 && rows % TM == 0 && rows / TM < (1 << 20), "rows must be a positive multiple of %d", TM);
  return B200_OK;
}

// x: mapping [rows][4], atlas [rows][2] (network input itself).  y: [rows][out_dim].
int tc_single_forward(const MlpShape& sh, TcNet net, const float* params, const float* x, float* y, int64_t rows,
                      bool training, char* ws, bool persistent, cudaStream_t st) {
  B200_PROPAGATE(check_single(sh, net, rows));
  SinglePlan pl;
  plan_single(sh, net, rows, ws, &pl);
  const TableKey key{current_device(), ws, TABLE_PREP, (int)net, rows, 1, params, 0, training};
  const PrepJobs* d_prep; int n_prep;
  B200_PROPAGATE(get_table(persistent ? &key : nullptr, pl.d_prep, st, [&](PrepJobs& pj) {
    prep_jobs_for_net(pj, sh, pl.im, params, net, training);
  }, &d_prep, &n_prep));
  tc_prep_kernel<<<n_prep * 4, 128, 0, st>>>(d_prep);
  B200_CHECK_LAUNCH();
  FwdParams P{};
  fill_fwd(P, sh, pl.im, x, y, params, (int)rows, 1, nullptr);
  P.in_scale = 1.0f; P.in_shift = 0.0f; P.store_images = training ? 1 : 0;
  launch_fwd(net, (int)(rows / TM), P, st);
  B200_CHECK_LAUNCH();
  return B200_OK;
}

// after tc_single_forward(training) on the same workspace.  y: the saved outputs, dy [rows][out_dim] (zero in padding
// rows), gmax: device int holding the bits of max|dy| (>= 0), d_in: atlas only, [rows][2] or null.
int tc_single_backward(const MlpShape& sh, TcNet net, const float* params, float* grads, const float* x,
                       const float* y, const float* dy, float* d_in, int* gmax2, int64_t rows, char* ws,
                       bool persistent, cudaStream_t st) {
  B200_PROPAGATE(check_single(sh, net, rows));
  SinglePlan pl;
  plan_single(sh, net, rows, ws, &pl);
  const TableKey key{current_device(), ws, TABLE_WGRAD, (int)net, rows, 1, grads, 0, true};
  const WgradItems* d_wg; int n_wg;
  B200_PROPAGATE(get_table(persistent ? &key : nullptr, pl.d_wg, st, [&](WgradItems& wi) {
    WgProto protos[16]; int np = 0;
    protos_for_net(protos, np, sh, pl.im, grads, net, 1);
    apportion_items(wi, protos, np, (int)rows, 0);
  }, &d_wg, &n_wg));
  BwdParams P{};
  fill_bwd(P, sh, pl.im, dy, y, x, d_in, params, grads, (int)rows, 1, nullptr, gmax2);   // [0] atlas scale, [1] mapping scale
  P.in_scale = 1.0f; P.d_in_accumulate = 0;
  launch_bwd(net, (int)(rows / TM), P, st);
  B200_CHECK_LAUNCH();
  tc_wgrad_kernel<<<min(n_wg, sm_count()), WG_THREADS, WG_SMEM, st>>>(d_wg, nullptr, gmax2);
  B200_CHECK_LAUNCH();
  return B200_OK;
}

int tc_atlas_forward(const TcStep& s, cudaStream_t st) { return run_forward(s, true, st); }
int tc_atlas_backward(const TcStep& s, cudaStream_t st) { return run_backward(s, true, st); }
int tc_mapping_forward(const TcStep& s, cudaStream_t st) { return run_forward(s, false, st); }
int tc_mapping_backward(const TcStep& s, cudaStream_t st) { return run_backward(s, false, st); }

}  // namespace b200
