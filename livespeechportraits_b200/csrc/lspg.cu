// C-ABI implementation of the B200-native Feature2Face generator (see include/lspg.h).
//
// Host side: network structure (mirrors models/networks.py:554-675 of the reference), weight packing with
// eval-BatchNorm folding, activation-tensor planning, TMA descriptor construction, launch sequencing.
// Device side: conv_umma.cuh (tcgen05/TMA implicit-GEMM conv) and aux_kernels.cuh (input packer).
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "../../include/lspg.h"
#include "aux_kernels.cuh"
#include "raster.cuh"
#include "conv_umma.cuh"

namespace {

using namespace lspg;

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) return fail(LSPG_ECUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

enum Kind { K_HEAD = 0, K_S1 = 1, K_S2 = 2, K_UP = 3, K_TAIL = 4 };

uint16_t f32_to_bf16(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return static_cast<uint16_t>(u >> 16);   // inf / nan: truncate
  u += 0x7FFFu + ((u >> 16) & 1u);                                                // round to nearest even
  return static_cast<uint16_t>(u >> 16);
}
float bf16_to_f32(uint16_t h) {
  uint32_t u = static_cast<uint32_t>(h) << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
uint16_t f32_to_f16(float f) { return __half_as_ushort(__float2half_rn(f)); }     // round to nearest even, subnormals kept
float f16_to_f32(uint16_t h) { return __half2float(__ushort_as_half(h)); }

// PARITY packs weights as fp16 hi + lo limbs of (w * 2^kParityWeightShift): with the reference's N(0, 0.02) weights the lo
// limb of an unscaled weight sits in fp16's subnormal range; pre-scaling by a power of two (exact) moves it into the normal
// range, and the epilogue's folded BatchNorm scale carries the inverse factor (exact as well).
constexpr int kParityWeightShift = 8;

struct TensorInfo {
  int channels;
  int shift;       // per-image spatial extent = (H >> shift, W >> shift)
};

struct Layer {
  int kind = K_S1;
  int n_src = 1;
  int src[2] = {-1, -1};
  int cin[2] = {0, 0};
  int out = -1, res = -1;
  int cout = 0, cout_pad = 0;
  int n_phases = 1, n_taps = 9, k_total = 0;
  int relu = 0, has_bn = 0;
  int grid_shift = 0;            // sampling grid = (H >> grid_shift, W >> grid_shift)
  int8_t tap_map[4][kMaxTaps] = {}, tap_dx[4][kMaxTaps] = {}, tap_dy[4][kMaxTaps] = {};
  std::string conv_key, bn_key;
  // parameters (host, fp32, as loaded) and their packed forms
  std::vector<float> w;                      // OIHW
  std::vector<float> bn_w, bn_b, bn_m, bn_v;
  std::vector<uint16_t> packed[3];           // [phase][cout_pad][k_total] each: 0/1 = PARITY fp16 hi/lo limbs of w * 2^8, 2 = FAST bf16
  std::vector<float> scale, shift;           // [cout_pad]
  std::vector<float> scale_par;              // scale * 2^-8 (PARITY weights are pre-scaled)
  bool dirty = true;
  bool has_w = false;                        // the conv weight has been supplied at least once (forward refuses otherwise)
  // device copies
  uint16_t* d_w = nullptr;                   // PARITY: [limb][phase][cout_pad][k_total] fp16
  uint16_t* d_w_fast = nullptr;              // FAST:   [phase][cout_pad][k_total] bf16
  float* d_scale_par = nullptr;
  float* d_scale = nullptr;
  float* d_shift = nullptr;
};

struct PlanLayer {
  ConvParams prm;
  int bn = 64;
  int grid = 1;
  bool patch = false;     // conv_patch_kernel (halo patch per chunk) instead of conv_umma_kernel (one box per tap)
  bool pair = false;      // conv_pair_kernel (cta_group::2)
  int cluster = 1;        // CTAs per cluster sharing B stages by TMA multicast (patch mode only)
  bool split = false;     // split-K: conv kernel writes fp32 partials, splitk_reduce_kernel finishes
  int csplit = 0;         // split-K inside a cluster of this many CTAs (no finisher)
  int red_blocks = 0;     // grid of splitk_reduce_kernel
};

struct IoKey {
  const float* fm; int64_t fm_bstride; const float* cand; int64_t cand_bstride; void* out; int u8;
  bool operator==(const IoKey& o) const {
    return fm == o.fm && fm_bstride == o.fm_bstride && cand == o.cand && cand_bstride == o.cand_bstride && out == o.out && u8 == o.u8;
  }
};

struct Plan {
  // ONE instantiated CUDA graph per plan.  The caller's pointers (feature maps, candidates, output) are parameters of
  // two nodes only - the input packer and the tail conv - and are patched with cudaGraphExecKernelNodeSetParams when a
  // call brings different ones, so a caller that holds its outputs never re-captures (see forward_impl).
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  cudaGraphNode_t pack_node = nullptr, tail_node = nullptr;
  cudaKernelNodeParams pack_np{}, tail_np{};   // func / grid / block / smem of the two nodes as captured
  IoKey io{};                                  // pointers currently baked into `exec`
  unsigned long long last_use = 0;             // LRU stamp (lspg_ctx::use_clock)
  int batch = 0, height = 0, width = 0, mode = 0;
  void* workspace = nullptr;
  std::vector<size_t> tensor_off;            // byte offset of limb 0 of each activation tensor
  std::vector<size_t> tensor_limb_stride;    // bytes between limbs
  std::vector<PlanLayer> layers;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

struct lspg_ctx {
  int variant = 0, ngf = 64, num_downs = 8, in_nc = 13, out_nc = 3, device = -1;
  int num_sms = 0;
  std::vector<TensorInfo> tensors;
  std::vector<Layer> layers;
  bool weights_loaded = false;
  EncodeTiledFn encode = nullptr;
  std::map<std::tuple<int, int, int, int, void*>, std::unique_ptr<Plan>> plans;
  Plan* last_plan = nullptr;
  int num_sms_or_default() const { return num_sms > 0 ? num_sms : 148; }
  cudaStream_t capture_stream = nullptr;
  long long n_captures = 0, n_io_updates = 0, n_recaptures = 0;   // graph bookkeeping (lspg_graph_stats)
  const void* tail_func = nullptr;           // host stub of the tail kernel the last enqueue launched
  unsigned long long use_clock = 0;
  unsigned long long* trace_buf = nullptr;   // debug (LSPG_TRACE_LAYER): clock64 stamps of one layer's CTAs
  bool profiling = false;
  std::vector<std::vector<cudaEvent_t>> prof_events;   // one event set per recorded forward
  size_t prof_used = 0;
};

namespace {

// ------------------------------------------------------------------------------------------------
// Network structure.  Mirrors ResUnetSkipConnectionBlock[_small].__init__ (models/networks.py:585-640 /
// 489-544): nn.Sequential positions give the state-dict keys; execution order gives the layer list.
// ------------------------------------------------------------------------------------------------
struct BlockKeys {
  std::string down, down_bn, up, up_bn, sub;
  std::vector<std::string> res_down, res_up;
};

BlockKeys block_keys(const std::string& prefix, bool outer, bool inner, int nres) {
  BlockKeys b;
  int i = 0;
  auto at = [&](int k) { return prefix + "." + std::to_string(k); };
  b.down = at(i++);
  if (!outer && !inner) b.down_bn = at(i++);
  i++;  // ReLU
  for (int r = 0; r < nres; ++r) b.res_down.push_back(at(i++));
  if (!inner) b.sub = at(i++) + ".model";
  i++;  // Upsample
  b.up = at(i++);
  if (!outer) {
    b.up_bn = at(i++);
    i++;  // ReLU
    for (int r = 0; r < nres; ++r) b.res_up.push_back(at(i++));
  }
  return b;
}

void set_taps_s1(Layer& L) {
  L.n_phases = 1;
  L.n_taps = 9;
  for (int r = 0; r < 3; ++r)
    for (int s = 0; s < 3; ++s) {
      L.tap_map[0][r * 3 + s] = 0;
      L.tap_dx[0][r * 3 + s] = static_cast<int8_t>(s - 1);
      L.tap_dy[0][r * 3 + s] = static_cast<int8_t>(r - 1);
    }
}

// stride-2, pad-1: input row 2*oy + r - 1 = 2*(oy + d) + parity
void s2_row(int r, int* parity, int* d) {
  if (r == 0) { *parity = 1; *d = -1; }
  else if (r == 1) { *parity = 0; *d = 0; }
  else { *parity = 1; *d = 0; }
}

void set_taps_s2(Layer& L) {
  L.n_phases = 1;
  L.n_taps = 9;
  for (int r = 0; r < 3; ++r)
    for (int s = 0; s < 3; ++s) {
      int py, dy, px, dx;
      s2_row(r, &py, &dy);
      s2_row(s, &px, &dx);
      L.tap_map[0][r * 3 + s] = static_cast<int8_t>(py * 2 + px);
      L.tap_dx[0][r * 3 + s] = static_cast<int8_t>(dx);
      L.tap_dy[0][r * 3 + s] = static_cast<int8_t>(dy);
    }
}

// nearest-x2 upsample followed by 3x3 pad-1: output row 2*i + parity reads upsampled rows
// 2*i + parity + r - 1, i.e. source rows i + d.  Returns d for (parity, r).
int up_row(int parity, int r) {
  if (parity == 0) return r == 0 ? -1 : 0;
  return r == 2 ? 1 : 0;
}

void set_taps_up(Layer& L) {
  L.n_phases = 4;
  L.n_taps = 4;
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px)
      for (int ty = 0; ty < 2; ++ty)
        for (int tx = 0; tx < 2; ++tx) {
          const int z = py * 2 + px, t = ty * 2 + tx;
          L.tap_map[z][t] = 0;
          L.tap_dy[z][t] = static_cast<int8_t>(py == 0 ? ty - 1 : ty);
          L.tap_dx[z][t] = static_cast<int8_t>(px == 0 ? tx - 1 : tx);
        }
}

void set_taps_head(Layer& L) {
  L.n_phases = 1;
  L.n_taps = 4;
  for (int ty = 0; ty < 2; ++ty)
    for (int tx = 0; tx < 2; ++tx) {
      L.tap_map[0][ty * 2 + tx] = 0;
      L.tap_dy[0][ty * 2 + tx] = static_cast<int8_t>(ty - 1);
      L.tap_dx[0][ty * 2 + tx] = static_cast<int8_t>(tx - 1);
    }
}

void set_taps_tail(Layer& L) {
  L.n_phases = 1;
  L.n_taps = 9;
  for (int ty = 0; ty < 3; ++ty)
    for (int tx = 0; tx < 3; ++tx) {
      L.tap_map[0][ty * 3 + tx] = 0;
      L.tap_dy[0][ty * 3 + tx] = static_cast<int8_t>(ty - 1);
      L.tap_dx[0][ty * 3 + tx] = static_cast<int8_t>(tx - 1);
    }
}

int build_network(lspg_ctx* h) {
  const int D = h->num_downs, ngf = h->ngf;
  const int nres = h->variant == LSPG_VARIANT_LARGE ? 2 : 1;
  std::vector<std::pair<int, int>> levels;   // (outer_nc, inner_nc), outermost first; networks.py:558-571
  levels.push_back({h->out_nc, ngf});
  levels.push_back({ngf, ngf * 2});
  levels.push_back({ngf * 2, ngf * 4});
  levels.push_back({ngf * 4, ngf * 8});
  for (int i = 0; i < D - 5; ++i) levels.push_back({ngf * 8, ngf * 8});
  levels.push_back({ngf * 8, ngf * 8});

  auto new_tensor = [&](int c, int shift) {
    h->tensors.push_back({c, shift});
    return static_cast<int>(h->tensors.size()) - 1;
  };
  auto add_res = [&](const std::string& key, int x, int c, int shift) {
    // ResidualBlock (networks.py:662-674): conv-BN-ReLU, conv-BN, += x, ReLU
    Layer a;
    a.kind = K_S1; a.n_src = 1; a.src[0] = x; a.cin[0] = c; a.cout = a.cout_pad = c;
    a.relu = 1; a.has_bn = 1; a.grid_shift = shift;
    a.conv_key = key + ".block.0"; a.bn_key = key + ".block.1";
    set_taps_s1(a); a.k_total = 9 * c; a.out = new_tensor(c, shift);
    h->layers.push_back(a);
    Layer b = a;
    b.src[0] = a.out; b.res = x; b.conv_key = key + ".block.3"; b.bn_key = key + ".block.4";
    b.out = new_tensor(c, shift);
    h->layers.push_back(b);
    return b.out;
  };

  const int s_in = new_tensor(64, 1);        // tensor 0: space-to-depth packed input (aux_kernels.cuh)

  // recursive emission in execution order; returns the id of d_l (the block's up-path result)
  std::function<int(int, int, const std::string&)> emit = [&](int l, int x, const std::string& prefix) -> int {
    const bool outer = (l == 0), inner = (l == D - 1);
    const int outer_nc = levels[l].first, inner_nc = levels[l].second;
    const BlockKeys k = block_keys(prefix, outer, inner, nres);
    Layer dn;
    dn.cout = dn.cout_pad = inner_nc; dn.relu = 1; dn.grid_shift = l + 1;
    dn.conv_key = k.down; dn.bn_key = k.down_bn; dn.has_bn = k.down_bn.empty() ? 0 : 1;
    if (outer) {
      dn.kind = K_HEAD; dn.n_src = 1; dn.src[0] = s_in; dn.cin[0] = 64; set_taps_head(dn); dn.k_total = 4 * 64;
    } else {
      dn.kind = K_S2; dn.n_src = 1; dn.src[0] = x; dn.cin[0] = outer_nc; set_taps_s2(dn); dn.k_total = 9 * outer_nc;
    }
    dn.out = new_tensor(inner_nc, l + 1);
    h->layers.push_back(dn);
    int e = dn.out;
    for (const auto& rk : k.res_down) e = add_res(rk, e, inner_nc, l + 1);
    int d = -1;
    if (!inner) d = emit(l + 1, e, k.sub);
    Layer up;
    up.n_src = inner ? 1 : 2; up.src[0] = e; up.cin[0] = inner_nc;
    if (!inner) { up.src[1] = d; up.cin[1] = inner_nc; }
    up.grid_shift = l + 1;                    // sampling grid = source grid
    up.conv_key = k.up; up.bn_key = k.up_bn; up.has_bn = k.up_bn.empty() ? 0 : 1;
    if (outer) {
      up.kind = K_TAIL; up.cout = outer_nc; up.cout_pad = 16; up.relu = 0; set_taps_tail(up);
      up.k_total = 9 * up.n_src * inner_nc; up.out = -1;
      h->layers.push_back(up);
      return -1;
    }
    up.kind = K_UP; up.cout = up.cout_pad = outer_nc; up.relu = 1; set_taps_up(up);
    up.k_total = 4 * up.n_src * inner_nc; up.out = new_tensor(outer_nc, l);
    h->layers.push_back(up);
    int dd = up.out;
    for (const auto& rk : k.res_up) dd = add_res(rk, dd, outer_nc, l);
    return dd;
  };
  emit(0, -1, "netG.model.model");
  return LSPG_OK;
}

// ------------------------------------------------------------------------------------------------
// Weight packing: OIHW fp32 -> [phase][cout_pad][K] (K = tap-major, then concat source, then channel),
// BatchNorm folded into fp32 scale/shift that the epilogue applies (the weights themselves are NOT scaled,
// so operand rounding matches "conv then BN").
// ------------------------------------------------------------------------------------------------
void pack_layer(lspg_ctx* h, Layer& L) {
  const int cin_total = (L.kind == K_HEAD) ? h->in_nc : (L.cin[0] + (L.n_src == 2 ? L.cin[1] : 0));
  const size_t per_phase = static_cast<size_t>(L.cout_pad) * L.k_total;
  std::vector<float> P(per_phase * L.n_phases, 0.0f);
  auto W = [&](int o, int c, int r, int s) -> float {
    return L.w[((static_cast<size_t>(o) * cin_total + c) * 3 + r) * 3 + s];
  };
  const int kb_per_tap = (L.cin[0] + (L.n_src == 2 ? L.cin[1] : 0));   // K elements per tap
  auto kidx = [&](int tap, int c_concat) { return tap * kb_per_tap + c_concat; };

  if (L.kind == K_S1 || L.kind == K_S2) {
    for (int o = 0; o < L.cout; ++o)
      for (int r = 0; r < 3; ++r)
        for (int s = 0; s < 3; ++s)
          for (int c = 0; c < cin_total; ++c)
            P[static_cast<size_t>(o) * L.k_total + kidx(r * 3 + s, c)] = W(o, c, r, s);
  } else if (L.kind == K_UP) {
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        float* Pz = P.data() + per_phase * (py * 2 + px);
        for (int o = 0; o < L.cout; ++o)
          for (int r = 0; r < 3; ++r)
            for (int s = 0; s < 3; ++s) {
              const int ty = up_row(py, r) - (py == 0 ? -1 : 0);   // dy -> tap row index (see set_taps_up)
              const int tx = up_row(px, s) - (px == 0 ? -1 : 0);
              for (int c = 0; c < cin_total; ++c)
                Pz[static_cast<size_t>(o) * L.k_total + kidx(ty * 2 + tx, c)] += W(o, c, r, s);
            }
      }
  } else if (L.kind == K_HEAD) {
    // source channel (py*2+px)*16 + c of the space-to-depth input, taps (dy,dx) in {-1,0}^2
    for (int o = 0; o < L.cout; ++o)
      for (int r = 0; r < 3; ++r)
        for (int s = 0; s < 3; ++s) {
          int py, dy, px, dx;
          s2_row(r, &py, &dy);
          s2_row(s, &px, &dx);
          const int tap = (dy + 1) * 2 + (dx + 1);
          for (int c = 0; c < cin_total; ++c)
            P[static_cast<size_t>(o) * L.k_total + kidx(tap, (py * 2 + px) * 16 + c)] = W(o, c, r, s);
        }
  } else {  // K_TAIL: row n = (py*2+px)*out_nc + c, taps (dy,dx) in {-1,0,1}^2 on the source grid
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px)
        for (int o = 0; o < L.cout; ++o) {
          const int n = (py * 2 + px) * L.cout + o;
          for (int r = 0; r < 3; ++r)
            for (int s = 0; s < 3; ++s) {
              const int tap = (up_row(py, r) + 1) * 3 + (up_row(px, s) + 1);
              for (int c = 0; c < cin_total; ++c)
                P[static_cast<size_t>(n) * L.k_total + kidx(tap, c)] += W(o, c, r, s);
            }
        }
  }
  for (int l = 0; l < 3; ++l) L.packed[l].assign(P.size(), 0);
  const float up = static_cast<float>(1 << kParityWeightShift);
  for (size_t i = 0; i < P.size(); ++i) {
    const float ws = P[i] * up;                           // exact (power of two)
    const uint16_t hi = f32_to_f16(ws);
    L.packed[0][i] = hi;
    L.packed[1][i] = f32_to_f16(ws - f16_to_f32(hi));
    L.packed[2][i] = f32_to_bf16(P[i]);
  }
  L.scale.assign(L.cout_pad, 1.0f);
  L.shift.assign(L.cout_pad, 0.0f);
  if (L.has_bn) {
    for (int o = 0; o < L.cout; ++o) {
      const float inv = 1.0f / sqrtf(L.bn_v[o] + 1e-5f);   // eval-mode BatchNorm2d, eps = torch default
      L.scale[o] = L.bn_w[o] * inv;
      L.shift[o] = L.bn_b[o] - L.bn_m[o] * L.scale[o];
    }
  }
  L.scale_par.resize(L.cout_pad);
  for (int o = 0; o < L.cout_pad; ++o) L.scale_par[o] = L.scale[o] / up;      // exact
}

int upload_layer(lspg_ctx* h, Layer& L) {
  if (h->device < 0) return LSPG_OK;
  const size_t n = L.packed[0].size();
  if (!L.d_w) {
    CUDA_TRY(cudaMalloc(&L.d_w, 2 * n * sizeof(uint16_t)));
    CUDA_TRY(cudaMalloc(&L.d_w_fast, n * sizeof(uint16_t)));
    CUDA_TRY(cudaMalloc(&L.d_scale, L.cout_pad * sizeof(float)));
    CUDA_TRY(cudaMalloc(&L.d_scale_par, L.cout_pad * sizeof(float)));
    CUDA_TRY(cudaMalloc(&L.d_shift, L.cout_pad * sizeof(float)));
  }
  CUDA_TRY(cudaMemcpy(L.d_w, L.packed[0].data(), n * 2, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(L.d_w + n, L.packed[1].data(), n * 2, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(L.d_w_fast, L.packed[2].data(), n * 2, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(L.d_scale, L.scale.data(), L.cout_pad * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(L.d_scale_par, L.scale_par.data(), L.cout_pad * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(L.d_shift, L.shift.data(), L.cout_pad * 4, cudaMemcpyHostToDevice));
  return LSPG_OK;
}

// ------------------------------------------------------------------------------------------------
// Planning
// ------------------------------------------------------------------------------------------------
size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int nl_of(int mode) { return mode == LSPG_MODE_PARITY ? 2 : 1; }

size_t tensor_bytes_one_limb(const TensorInfo& t, int B, int H, int W) {
  return static_cast<size_t>(B) * (H >> t.shift) * (W >> t.shift) * t.channels * 2;
}

int ilog2(int v) {
  int l = 0;
  while ((1 << (l + 1)) <= v) ++l;
  return l;
}

// Tiling / kernel-variant decisions of one layer for a problem size (shared by planning and workspace sizing).
struct Geo {
  int hs, ws;                  // sampling grid
  int tw, th, nb;              // output tile = tw x th pixels x nb images (= 128 rows)
  bool patch;                  // conv_patch_kernel (halo patch) vs conv_umma_kernel (one box per tap)
  int bn, m_tiles, n_tiles, tiles_per_split;
  int k_items;                 // K-loop length: K blocks (v1) or (source, chunk) items (patch)
  int n_split, split_len;
  size_t partial_bytes;
  bool pair;                   // conv_pair_kernel: cta_group::2 UMMA over a 2-CTA cluster (wide layers)
  int csplit;                  // > 0: split-K inside a thread-block cluster of this many CTAs (DSMEM reduction, no finisher)
  int cluster;                 // CTAs per cluster of the launch: 2 = pair / weight multicast, csplit, else 1
};

Geo layer_geo(const lspg_ctx* h, const Layer& L, int B, int H, int W) {
  static const bool no_patch = getenv("LSPG_NO_PATCH") != nullptr;
  static const bool no_split = getenv("LSPG_NO_SPLITK") != nullptr;
  Geo g;
  g.hs = H >> L.grid_shift; g.ws = W >> L.grid_shift;
  g.tw = g.ws < 16 ? g.ws : 16;
  g.th = 128 / g.tw;
  if (g.th > g.hs) g.th = g.hs;
  g.nb = 128 / (g.tw * g.th);
  // patch mode needs 8-pixel-wide tiles (one UMMA 8-row group = one image row of the halo patch)
  g.patch = !no_patch && L.kind != K_S2 && g.ws >= 8 && g.hs >= 16;
  if (g.patch) { g.tw = 8; g.th = 16; g.nb = 1; }
  g.m_tiles = (g.ws / g.tw) * (g.hs / g.th) * ((B + g.nb - 1) / g.nb);
  const int chunks = L.cin[0] / 64 + (L.n_src == 2 ? L.cin[1] / 64 : 0);
  g.k_items = g.patch ? chunks : chunks * L.n_taps;
  if (L.kind == K_TAIL) g.bn = 16;
  else g.bn = (L.cout_pad % 128 == 0 && g.m_tiles * (L.cout_pad / 128) * L.n_phases >= h->num_sms_or_default()) ? 128 : 64;
  // per-tap kernel below 16^2: the N=128 tile halves the A traffic per MAC (the kernel is shared-memory bound) and split-K
  // restores the CTA count
  if (!g.patch && L.kind != K_TAIL && L.cout_pad % 128 == 0 && g.m_tiles >= 8) g.bn = 128;
  // CTA-pair kernel for the wide layers: N tile 256 (or 128), two neighbouring M tiles per cluster
  static const bool no_pair = getenv("LSPG_NO_PAIR") != nullptr;
  g.pair = false;
  if (!no_pair && g.patch && (L.kind == K_S1 || L.kind == K_UP) && L.cout_pad % 64 == 0 && g.m_tiles % 2 == 0) {
    const int sms = h->num_sms_or_default();
    int bnp = 0;
    // a pair tile runs the tensor pipe at full rate while the N=64 single-CTA tile is shared-memory bound at ~60 %,
    // so the pair kernel already wins when its tiles fill about two thirds of the SMs
    const int enough = sms * 2 / 3;
    // Tiles are equal-sized and statically strided over sms/2 clusters, so a launch costs ceil(pairs / clusters) waves of
    // one tile each: 256 pairs of N=256 tiles on 74 clusters are 4 waves (3.46 needed), the same work as 512 pairs of N=128
    // tiles is 7 half-sized waves (-12.5 %).  Take the N tile with the lower wave cost; ties go to the wider tile (fewer
    // A operand reads).
    auto wave_cost = [&](int bn) {
      const long long pairs = static_cast<long long>(g.m_tiles) * (L.cout_pad / bn) * L.n_phases / 2;
      const long long clusters = sms / 2;
      return (pairs + clusters - 1) / clusters * bn;
    };
    if (L.cout_pad % 256 == 0 && g.m_tiles * (L.cout_pad / 256) * L.n_phases >= sms)
      bnp = wave_cost(128) < wave_cost(256) ? 128 : 256;
    else if (L.cout_pad % 128 == 0 && g.m_tiles * (L.cout_pad / 128) * L.n_phases >= enough) bnp = 128;
    else if (L.cout_pad == 64 && g.m_tiles * L.n_phases >= enough) bnp = 64;
    if (bnp) { g.pair = true; g.bn = bnp; }
  }
  g.n_tiles = L.cout_pad / g.bn;
  g.tiles_per_split = g.m_tiles * g.n_tiles * L.n_phases;
  g.n_split = 1; g.split_len = g.k_items; g.partial_bytes = 0; g.csplit = 0;
  const int sms = h->num_sms_or_default();
  if (!no_split && !g.pair && L.kind != K_TAIL && g.tiles_per_split * 2 <= sms) {
    const int min_len = g.patch ? 1 : 4;                       // at least 4 K blocks (v1) / 1 chunk of all taps per split
    int want = sms / g.tiles_per_split;                        // floor: tiles x splits stay within one wave
    int max_split = g.k_items / min_len;
    if (max_split < 1) max_split = 1;
    if (want > max_split) want = max_split;
    // Cluster split-K: the 2 / 4 / 8 CTAs of a tile form a cluster, exchange their partial rows through distributed shared
    // memory and finish the tile themselves - no partials in global memory, no finisher launch.  Needs exactly `cs`
    // non-empty K ranges and tiles x cs CTAs in one wave.
    // Measured on one B200 (profiles/r02_t3_ab_cluster_split.txt, alternating runs): 32 frames per step 15.57-15.67 ms with
    // the cluster reduction vs 15.77-15.82 ms with finisher kernels (-1 %); one frame per call 1.283 vs 1.262 ms (+1.7 %: at
    // batch 1 a cluster of 8 leaves 64 CTAs streaming the layer's weights where 18 finisher-splits keep 144 busy, and under
    // PDL the finisher launches were almost free).  So clusters from 8 frames up, finishers below; LSPG_CLUSTER_SPLIT=0/1
    // forces either for A/B runs.
    static const int csplit_env = [] { const char* e = getenv("LSPG_CLUSTER_SPLIT"); return e ? atoi(e) : -1; }();
    const bool use_csplit = csplit_env >= 0 ? csplit_env != 0 : B >= 8;
    if (use_csplit && want > 1) {
      for (int cs : {8, 4, 2}) {
        if (cs > want) continue;
        const int len = (g.k_items + cs - 1) / cs;
        if ((g.k_items + len - 1) / len != cs) continue;
        g.csplit = cs; g.n_split = cs; g.split_len = len;
        break;
      }
    }
    if (!g.csplit && want > 1) {
      g.split_len = (g.k_items + want - 1) / want;
      g.n_split = (g.k_items + g.split_len - 1) / g.split_len;
      if (g.n_split > 1) g.partial_bytes = static_cast<size_t>(g.n_split) * g.tiles_per_split * kTileM * g.bn * sizeof(float);
      else g.split_len = g.k_items;
    }
  }
  // A patch-kernel layer that fills at least one wave without split-K runs its CTAs in pairs that share each weight stage
  // by TMA multicast.
  static const bool no_cluster = getenv("LSPG_NO_CLUSTER") != nullptr;
  if (g.pair) g.cluster = 2;
  else if (g.csplit) g.cluster = g.csplit;
  else g.cluster = (g.patch && !no_cluster && g.n_split == 1 && g.m_tiles % 2 == 0 && g.tiles_per_split >= sms) ? 2 : 1;
  return g;
}

size_t scratch_bytes(const lspg_ctx* h, int B, int H, int W) {
  size_t m = 0;
  for (const auto& L : h->layers) m = std::max(m, layer_geo(h, L, B, H, W).partial_bytes);
  return align_up(m, 1024);
}

size_t workspace_bytes(const lspg_ctx* h, int B, int H, int W, int mode) {
  size_t total = 0;
  for (const auto& t : h->tensors) total += align_up(tensor_bytes_one_limb(t, B, H, W), 1024) * nl_of(mode);
  return total + scratch_bytes(h, B, H, W) + 1024;
}

// Activation layout inside the workspace, from its first 1024-aligned byte: every tensor's limbs back to back, each limb
// padded to 1 KB.  Returns the end of the last tensor (where the split-K scratch begins).
size_t tensor_layout(const lspg_ctx* h, int B, int H, int W, int NL, std::vector<size_t>* off, std::vector<size_t>* limb_stride) {
  size_t o = 0;
  for (const auto& t : h->tensors) {
    const size_t one = align_up(tensor_bytes_one_limb(t, B, H, W), 1024);
    off->push_back(o);
    limb_stride->push_back(one);
    o += one * NL;
  }
  return o;
}

int check_shape(const lspg_ctx* h, int B, int H, int W, int mode) {
  if (B < 1 || B > 4096) return fail(LSPG_EINVAL, "batch %d out of range", B);
  const int m = 1 << h->num_downs;
  if (H < m || W < m || H % m || W % m)
    return fail(LSPG_EINVAL, "height/width must be positive multiples of %d (got %dx%d)", m, H, W);
  if (mode != LSPG_MODE_FAST && mode != LSPG_MODE_PARITY) return fail(LSPG_EINVAL, "unknown precision mode %d", mode);
  // Every level of the U-Net must be covered exactly by its power-of-two tiles (tile decode uses shifts, tiles_x/tiles_y
  // are exact quotients, there are no edge tiles).  A grid like 768 = 3*256 gives 24x24 / 12x12 / 6x6 / 3x3 levels that the
  // 16x8 boxes do not tile: reject it here instead of rendering garbage (the reference accepts any multiple of 256).
  for (const auto& L : h->layers) {
    const Geo g = layer_geo(h, L, B, H, W);
    const bool pow2 = (g.tw & (g.tw - 1)) == 0 && (g.th & (g.th - 1)) == 0 && (g.nb & (g.nb - 1)) == 0;
    if (!pow2 || g.tw * g.th * g.nb != kTileM || g.hs % g.th || g.ws % g.tw)
      return fail(LSPG_EINVAL, "%dx%d is not supported: the %dx%d level does not tile into %dx%d boxes (height and width "
                  "must be powers of two >= %d)", H, W, g.hs, g.ws, g.tw, g.th, m);
  }
  return LSPG_OK;
}

// 5-D activation view {C, X, Y, N, limb}; parity/phase views start at (py, px) and step 2 in X and Y.
int make_act_map(lspg_ctx* h, CUtensorMap* m, void* base, size_t limb_stride, int NL, int C, int B, int Ht, int Wt,
                 bool strided2, int py, int px, int tw, int th, int nb) {
  const size_t es = 2;
  uint8_t* p = static_cast<uint8_t*>(base);
  cuuint64_t dims[5];
  cuuint64_t strides[4];
  if (!strided2) {
    dims[0] = C; dims[1] = Wt; dims[2] = Ht; dims[3] = B; dims[4] = NL;
    strides[0] = static_cast<cuuint64_t>(C) * es;
    strides[1] = static_cast<cuuint64_t>(Wt) * C * es;
  } else {
    p += (static_cast<size_t>(py) * Wt + px) * C * es;
    dims[0] = C; dims[1] = Wt / 2; dims[2] = Ht / 2; dims[3] = B; dims[4] = NL;
    strides[0] = static_cast<cuuint64_t>(2) * C * es;
    strides[1] = static_cast<cuuint64_t>(2) * Wt * C * es;
  }
  strides[2] = static_cast<cuuint64_t>(Ht) * Wt * C * es;
  strides[3] = NL > 1 ? limb_stride : strides[2] * B;
  cuuint32_t box[5] = {64u, static_cast<cuuint32_t>(tw), static_cast<cuuint32_t>(th), static_cast<cuuint32_t>(nb), 1u};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = h->encode(m, NL > 1 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, p, dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(LSPG_ECUDA, "cuTensorMapEncodeTiled(activation C=%d %dx%d B=%d box %dx%dx%d) failed: %d", C, Wt, Ht, B,
                tw, th, nb, static_cast<int>(r));
  return LSPG_OK;
}

int make_weight_map(lspg_ctx* h, CUtensorMap* m, const Layer& L, int bn, int NL) {
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(L.k_total), static_cast<cuuint64_t>(L.cout_pad),
                        static_cast<cuuint64_t>(NL * L.n_phases)};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(L.k_total) * 2,
                           static_cast<cuuint64_t>(L.k_total) * L.cout_pad * 2};
  cuuint32_t box[3] = {64u, static_cast<cuuint32_t>(bn), 1u};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = h->encode(m, NL > 1 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, NL > 1 ? L.d_w : L.d_w_fast, dims,
                         strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LSPG_ECUDA, "cuTensorMapEncodeTiled(weights K=%d) failed: %d", L.k_total, static_cast<int>(r));
  return LSPG_OK;
}

// Patch-mode weight view {kc, Cout, tap, limb*phase}: K of the packed weights is tap-major, so the tap index is a
// dimension of its own and one TMA box {64, BN, taps_per_stage, 1} fetches the tiles of several taps at once.
int make_weight_map_taps(lspg_ctx* h, CUtensorMap* m, const Layer& L, int bn, int tps, int NL) {   // bn = box rows, tps = box taps
  const int kt = L.k_total / L.n_taps;       // K elements per tap
  cuuint64_t dims[4] = {static_cast<cuuint64_t>(kt), static_cast<cuuint64_t>(L.cout_pad), static_cast<cuuint64_t>(L.n_taps),
                        static_cast<cuuint64_t>(NL * L.n_phases)};
  cuuint64_t strides[3] = {static_cast<cuuint64_t>(L.k_total) * 2, static_cast<cuuint64_t>(kt) * 2,
                           static_cast<cuuint64_t>(L.k_total) * L.cout_pad * 2};
  cuuint32_t box[4] = {64u, static_cast<cuuint32_t>(bn), static_cast<cuuint32_t>(tps), 1u};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = h->encode(m, NL > 1 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, NL > 1 ? L.d_w : L.d_w_fast, dims,
                         strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LSPG_ECUDA, "cuTensorMapEncodeTiled(weights by tap, K=%d) failed: %d", L.k_total, static_cast<int>(r));
  return LSPG_OK;
}

uint32_t make_idesc(int bn, int m, bool f16) {
  // cute::UMMA::InstrDescriptor bit layout: c_format[4,6)=1 (F32), a_format[7,10) and b_format[10,13): 0 = F16, 1 = BF16,
  // a/b major [15],[16] = 0 (K-major), n_dim[17,23) = N>>3, m_dim[24,29) = M>>4
  uint32_t d = 0;
  d |= 1u << 4;
  if (!f16) {
    d |= 1u << 7;
    d |= 1u << 10;
  }
  d |= static_cast<uint32_t>(bn >> 3) << 17;
  d |= static_cast<uint32_t>(m >> 4) << 24;
  return d;
}

int build_plan(lspg_ctx* h, Plan* P, int B, int H, int W, int mode, void* workspace) {
  const int NL = nl_of(mode);
  P->batch = B; P->height = H; P->width = W; P->mode = mode; P->workspace = workspace;
  const size_t base = align_up(reinterpret_cast<size_t>(workspace), 1024) - reinterpret_cast<size_t>(workspace);
  const size_t off = base + tensor_layout(h, B, H, W, NL, &P->tensor_off, &P->tensor_limb_stride);
  for (auto& o : P->tensor_off) o += base;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  uint8_t* ws_scratch = ws + align_up(off, 1024);
  for (const Layer& L : h->layers) {
    PlanLayer pl;
    ConvParams& p = pl.prm;
    memset(&p, 0, sizeof(p));
    const Geo g = layer_geo(h, L, B, H, W);
    const int Hs = g.hs, Ws = g.ws;
    const int tw = g.tw, th = g.th, nb = g.nb;
    pl.patch = g.patch;
    int abox_w = tw, abox_h = th, abox_n = nb;
    if (pl.patch) {
      int pw = 0, ph = 0;
      for (int z = 0; z < L.n_phases; ++z) {
        int dx0 = 127, dx1 = -127, dy0 = 127, dy1 = -127;
        for (int t = 0; t < L.n_taps; ++t) {
          dx0 = std::min<int>(dx0, L.tap_dx[z][t]); dx1 = std::max<int>(dx1, L.tap_dx[z][t]);
          dy0 = std::min<int>(dy0, L.tap_dy[z][t]); dy1 = std::max<int>(dy1, L.tap_dy[z][t]);
        }
        p.patch_dx0[z] = static_cast<int8_t>(dx0); p.patch_dy0[z] = static_cast<int8_t>(dy0);
        pw = std::max(pw, tw + dx1 - dx0); ph = std::max(ph, th + dy1 - dy0);
      }
      p.patch_w = pw; p.patch_h = ph;
      for (int z = 0; z < L.n_phases; ++z)
        for (int t = 0; t < L.n_taps; ++t)
          p.tap_row[z][t] = static_cast<int16_t>((L.tap_dy[z][t] - p.patch_dy0[z]) * pw + (L.tap_dx[z][t] - p.patch_dx0[z]));
      if (pw * ph * 128 > kPatchSlot) return fail(LSPG_EINVAL, "patch %dx%d does not fit its smem slot", pw, ph);
      abox_w = pw; abox_h = ph; abox_n = 1;
    }
    pl.bn = g.bn;
    p.tw_log2 = ilog2(tw); p.th_log2 = ilog2(th);
    p.tiles_x = Ws / tw; p.tiles_y = Hs / th; p.tiles_n = (B + nb - 1) / nb;
    p.n_tiles = L.cout_pad / pl.bn;
    p.n_phases = L.n_phases;
    p.tiles_per_split = g.tiles_per_split;
    p.fd_tps = make_fast_div(g.tiles_per_split);
    p.fd_m_tiles = make_fast_div(p.tiles_x * p.tiles_y * p.tiles_n);
    p.fd_n_tiles = make_fast_div(p.n_tiles);
    p.fd_tiles_x = make_fast_div(p.tiles_x);
    p.fd_tiles_y = make_fast_div(p.tiles_y);
    p.n_split = g.n_split; p.split_len = g.split_len;
    p.total_tiles = g.tiles_per_split * g.n_split;
    if (g.pair) {
      const int n_items = g.k_items * L.n_taps;                           // weight tiles per output tile
      p.b_resident = (L.n_phases == 1 && g.n_tiles == 1 && n_items <= pair_b_stages(g.bn, NL)) ? 1 : 0;
    }
    p.partial = reinterpret_cast<float*>(ws_scratch);
    // Split-K is two-pass: raw fp32 partials, then splitk_reduce_kernel.  (Measured on B200 in round 1: letting the
    // last-arriving CTA sum the partials in-kernel was slower - one CTA's epilogue threads reduce a tile far more slowly
    // than a grid of them - so that variant was removed.)
    pl.split = g.n_split > 1 && g.csplit == 0;
    pl.csplit = g.csplit;
    p.cluster_split = g.csplit ? 1 : 0;
    p.n_taps = L.n_taps; p.n_src = L.n_src;
    p.chunks[0] = L.cin[0] / 64; p.chunks[1] = L.n_src == 2 ? L.cin[1] / 64 : 0;
    p.relu = L.relu; p.has_res = L.res >= 0 ? 1 : 0;
    p.batch = B; p.hs = Hs; p.ws = Ws;
    const bool f16 = NL > 1;                  // PARITY operands are fp16 limbs, FAST operands bf16
    p.idesc = make_idesc(pl.bn, g.pair ? 256 : kTileM, f16);
    p.idesc2 = make_idesc(2 * pl.bn > 256 ? 256 : 2 * pl.bn, g.pair ? 256 : kTileM, f16);
    p.scale = f16 ? L.d_scale_par : L.d_scale; p.shift = L.d_shift; p.out_f32 = nullptr;
    memcpy(p.tap_map, L.tap_map, sizeof(p.tap_map));
    memcpy(p.tap_dx, L.tap_dx, sizeof(p.tap_dx));
    memcpy(p.tap_dy, L.tap_dy, sizeof(p.tap_dy));
    int rc;
    // ---- source views
    for (int s = 0; s < L.n_src; ++s) {
      const TensorInfo& t = h->tensors[L.src[s]];
      const int Ht = H >> t.shift, Wt = W >> t.shift;
      void* tb = ws + P->tensor_off[L.src[s]];
      const size_t ls = P->tensor_limb_stride[L.src[s]];
      if (L.kind == K_S2) {
        for (int q = 0; q < 4; ++q)
          if ((rc = make_act_map(h, &p.a[q], tb, ls, NL, t.channels, B, Ht, Wt, true, q >> 1, q & 1, tw, th, nb))) return rc;
      } else {
        if ((rc = make_act_map(h, &p.a[s], tb, ls, NL, t.channels, B, Ht, Wt, false, 0, 0, abox_w, abox_h, abox_n))) return rc;
      }
    }
    // unused slots still need valid descriptors for prefetch.tensormap
    const int used = (L.kind == K_S2) ? 4 : L.n_src;
    for (int q = used; q < 4; ++q) p.a[q] = p.a[0];
    if (pl.patch) {
      pl.pair = g.pair;
      pl.cluster = g.csplit ? 1 : g.cluster;     // a cluster split launches CL = 1 code in clusters of csplit CTAs
      if (pl.cluster == 1 && NL == 1 && !pl.pair) rc = make_weight_map_taps(h, &p.w, L, pl.bn, patch_taps_per_stage(pl.bn, NL, L.kind == K_TAIL), NL);
      else rc = make_weight_map_taps(h, &p.w, L, pl.bn / pl.cluster, 1, NL);      // per-tap boxes (row slice per CTA when multicasting)
      if (rc) return rc;
    } else {
      if ((rc = make_weight_map(h, &p.w, L, pl.bn, NL))) return rc;
    }
    // ---- output / residual (the epilogue addresses both through plain pointers)
    if (L.kind != K_TAIL) {
      p.out_ptr = reinterpret_cast<__nv_bfloat16*>(ws + P->tensor_off[L.out]);
      p.out_limb_stride = static_cast<long long>(P->tensor_limb_stride[L.out] / 2);
      p.out_channels = h->tensors[L.out].channels;
      p.out_up = (L.kind == K_UP) ? 1 : 0;
      if (L.res >= 0) {
        p.res_ptr = reinterpret_cast<const __nv_bfloat16*>(ws + P->tensor_off[L.res]);
        p.res_limb_stride = static_cast<long long>(P->tensor_limb_stride[L.res] / 2);
        p.res_channels = h->tensors[L.res].channels;
      }
    }
    // A split layer's output holds exactly its cout_pad channels, and its residual (only ever on stride-1 layers) has the
    // output's grid and channel count: the split-K finishers rely on both, and build_network guarantees them.
    if (g.n_split > 1 && (p.out_channels != L.cout_pad || (L.res >= 0 && (p.out_up || p.res_channels != p.out_channels))))
      return fail(LSPG_EINVAL, "split-K layer %s: output/residual layout the split-K finishers do not support", L.conv_key.c_str());
    pl.grid = p.total_tiles < h->num_sms ? p.total_tiles : h->num_sms;
    if (pl.cluster > 1) pl.grid -= pl.grid % pl.cluster;
    {
      const char* tl = getenv("LSPG_TRACE_LAYER");
      if (tl && atoi(tl) == static_cast<int>(P->layers.size())) {
        if (!h->trace_buf) CUDA_TRY(cudaMalloc(&h->trace_buf, sizeof(unsigned long long) * 256 * kTraceSlots));
        CUDA_TRY(cudaMemset(h->trace_buf, 0, sizeof(unsigned long long) * 256 * kTraceSlots));
        p.trace = h->trace_buf;
        const char* ts = getenv("LSPG_TRACE_SKIP");
        p.trace_skip = ts ? atoi(ts) : 0;
      }
    }
    if (pl.split) {
      const long long work = static_cast<long long>(g.tiles_per_split) * kTileM * (g.bn / 4);   // one thread per pixel x 4 channels
      pl.red_blocks = static_cast<int>(std::min<long long>((work + 127) / 128, 8LL * h->num_sms));
    }
    P->layers.push_back(pl);
  }
  return LSPG_OK;
}

// Every kernel of the forward is launched with programmatic stream serialization (PDL): the next kernel's CTAs may
// be scheduled while this one drains; each kernel calls griddepcontrol.wait before it touches dependent memory.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster,
                               Args&&... args) {
  static const bool no_pdl = getenv("LSPG_NO_PDL") != nullptr;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (!no_pdl) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = static_cast<unsigned>(cluster);
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr; cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  return launch_pdl_cluster(kernel, grid, block, smem, st, 1, std::forward<Args>(args)...);
}

// Opt-in to > 48 KB of dynamic shared memory.  The attribute is per (function, device): a process that renders on
// several GPUs (two modules, or a module moved with .to('cuda:1')) must set it on each of them, so the "done" flag is a
// bit per device ordinal, not a process-wide bool.
template <typename K>
int ensure_smem(K kernel, int bytes, int device, unsigned long long* done_mask) {
  const unsigned long long bit = 1ull << (device & 63);
  if (!(*done_mask & bit)) {
    CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    *done_mask |= bit;
  }
  return LSPG_OK;
}

const void* g_last_func = nullptr;     // host stub of the most recent conv launch (identifies graph nodes after capture)

template <int BN, int NL, bool TAIL, bool CSP = false>
int launch_conv(const ConvParams& p, int grid, int device, cudaStream_t st, int cluster = 1) {
  using Cfg = ConvCfg<BN, NL, TAIL, CSP>;
  static unsigned long long done = 0;
  int rc = ensure_smem(conv_umma_kernel<BN, NL, TAIL, CSP>, Cfg::kSmemBytes, device, &done);
  if (rc) return rc;
  g_last_func = reinterpret_cast<const void*>(conv_umma_kernel<BN, NL, TAIL, CSP>);
  CUDA_TRY(launch_pdl_cluster(conv_umma_kernel<BN, NL, TAIL, CSP>, dim3(grid), dim3(kThreads), Cfg::kSmemBytes, st, cluster, p));
  return LSPG_OK;
}

// Epilogue warps: 4 for the tail (one fp32 / uint8 scatter per pixel), 8 for every other patch / pair kernel.
template <int BN, int NL, bool TAIL, int CL, bool CSP = false>
int launch_patch(const ConvParams& p, int grid, int device, cudaStream_t st, int cluster = CL) {
  using Cfg = PatchCfg<BN, NL, TAIL, CSP>;
  constexpr int EW = TAIL ? 4 : 8;
  static unsigned long long done = 0;
  int rc = ensure_smem(conv_patch_kernel<BN, NL, TAIL, CL, EW, CSP>, Cfg::kSmemBytes, device, &done);
  if (rc) return rc;
  g_last_func = reinterpret_cast<const void*>(conv_patch_kernel<BN, NL, TAIL, CL, EW, CSP>);
  CUDA_TRY(launch_pdl_cluster(conv_patch_kernel<BN, NL, TAIL, CL, EW, CSP>, dim3(grid), dim3(64 + EW * 32), Cfg::kSmemBytes, st, cluster, p));
  return LSPG_OK;
}

template <int BN, int NL, bool TAIL>
int launch_patch_cl(const ConvParams& p, int grid, int cluster, int device, cudaStream_t st) {
  return cluster == 2 ? launch_patch<BN, NL, TAIL, 2>(p, grid, device, st) : launch_patch<BN, NL, TAIL, 1>(p, grid, device, st);
}

template <int BN, int NL>
int launch_pair(const ConvParams& p, int grid, int device, cudaStream_t st) {
  constexpr bool STK = pair_stacked(BN, NL);
  using Cfg = PairCfg<BN, NL, STK>;
  static unsigned long long done = 0;
  int rc = ensure_smem(conv_pair_kernel<BN, NL, 8, STK>, Cfg::kSmemBytes, device, &done);
  if (rc) return rc;
  g_last_func = reinterpret_cast<const void*>(conv_pair_kernel<BN, NL, 8, STK>);
  CUDA_TRY(launch_pdl_cluster(conv_pair_kernel<BN, NL, 8, STK>, dim3(grid), dim3(64 + 8 * 32), Cfg::kSmemBytes, st, 2, p));
  return LSPG_OK;
}

int launch_layer(const PlanLayer& pl, int kind, int NL, int device, cudaStream_t st) {
  if (pl.pair) {
    if (pl.bn == 256) return NL == 1 ? launch_pair<256, 1>(pl.prm, pl.grid, device, st) : launch_pair<256, 2>(pl.prm, pl.grid, device, st);
    if (pl.bn == 64) return NL == 1 ? launch_pair<64, 1>(pl.prm, pl.grid, device, st) : launch_pair<64, 2>(pl.prm, pl.grid, device, st);
    return NL == 1 ? launch_pair<128, 1>(pl.prm, pl.grid, device, st) : launch_pair<128, 2>(pl.prm, pl.grid, device, st);
  }
  if (pl.csplit) {          // split-K inside a cluster of pl.csplit CTAs (one tile per CTA, grid = tiles x csplit)
    const int cs = pl.csplit;
    if (pl.patch) return NL == 1 ? launch_patch<64, 1, false, 1, true>(pl.prm, pl.grid, device, st, cs) : launch_patch<64, 2, false, 1, true>(pl.prm, pl.grid, device, st, cs);
    if (pl.bn == 128) return NL == 1 ? launch_conv<128, 1, false, true>(pl.prm, pl.grid, device, st, cs) : launch_conv<128, 2, false, true>(pl.prm, pl.grid, device, st, cs);
    return NL == 1 ? launch_conv<64, 1, false, true>(pl.prm, pl.grid, device, st, cs) : launch_conv<64, 2, false, true>(pl.prm, pl.grid, device, st, cs);
  }
  if (pl.patch) {
    const int c = pl.cluster;
    if (kind == K_TAIL) return NL == 1 ? launch_patch_cl<16, 1, true>(pl.prm, pl.grid, c, device, st) : launch_patch_cl<16, 2, true>(pl.prm, pl.grid, c, device, st);
    if (pl.bn == 128) return NL == 1 ? launch_patch_cl<128, 1, false>(pl.prm, pl.grid, c, device, st) : launch_patch_cl<128, 2, false>(pl.prm, pl.grid, c, device, st);
    return NL == 1 ? launch_patch_cl<64, 1, false>(pl.prm, pl.grid, c, device, st) : launch_patch_cl<64, 2, false>(pl.prm, pl.grid, c, device, st);
  }
  if (kind == K_TAIL) return NL == 1 ? launch_conv<16, 1, true>(pl.prm, pl.grid, device, st) : launch_conv<16, 2, true>(pl.prm, pl.grid, device, st);
  if (pl.bn == 128) return NL == 1 ? launch_conv<128, 1, false>(pl.prm, pl.grid, device, st) : launch_conv<128, 2, false>(pl.prm, pl.grid, device, st);
  return NL == 1 ? launch_conv<64, 1, false>(pl.prm, pl.grid, device, st) : launch_conv<64, 2, false>(pl.prm, pl.grid, device, st);
}

// The caller-dependent arguments of the two I/O nodes of a forward (input packer, tail conv).
struct PackArgs {
  const float* fm; long long fs; const float* cand; long long cs; int in_nc;
  __nv_bfloat16* dst; long long limb_stride; int batch, height, width;
  int blocks;
};

PackArgs make_pack_args(const lspg_ctx* h, const Plan* P, const IoKey& io) {
  PackArgs a;
  a.fm = io.fm; a.fs = io.fm_bstride; a.cand = io.cand; a.cs = io.cand_bstride; a.in_nc = h->in_nc;
  a.dst = reinterpret_cast<__nv_bfloat16*>(static_cast<uint8_t*>(P->workspace) + P->tensor_off[0]);
  a.limb_stride = static_cast<long long>(P->tensor_limb_stride[0] / 2);
  a.batch = P->batch; a.height = P->height; a.width = P->width;
  const long long total = static_cast<long long>(P->batch) * (P->height / 2) * (P->width / 2);
  a.blocks = static_cast<int>((total + 127) / 128);
  if (a.blocks > h->num_sms * 16) a.blocks = h->num_sms * 16;
  return a;
}

void set_tail_io(ConvParams* prm, const IoKey& io) {
  prm->out_f32 = io.u8 ? nullptr : static_cast<float*>(io.out);
  prm->out_u8 = io.u8 ? static_cast<uint8_t*>(io.out) : nullptr;
}

// Enqueue every kernel of one forward on `st` (plain stream launches; also the body of the graph capture).
int enqueue_forward(lspg_ctx* h, Plan* P, const IoKey& io, cudaStream_t st, bool debug_sync, bool profile) {
  const int NL = nl_of(P->mode);
  int rc;
  std::vector<cudaEvent_t>* evs = nullptr;
  if (profile && h->prof_used < 256) {
    if (h->prof_used == h->prof_events.size()) {
      std::vector<cudaEvent_t> set(h->layers.size() + 2);
      for (auto& e : set) CUDA_TRY(cudaEventCreate(&e));
      h->prof_events.push_back(set);
    }
    evs = &h->prof_events[h->prof_used++];
    CUDA_TRY(cudaEventRecord((*evs)[0], st));
  }
  // 1. input packer (cat + NCHW->NHWC + bf16 + space-to-depth)
  {
    const PackArgs a = make_pack_args(h, P, io);
    if (NL == 1)
      CUDA_TRY(launch_pdl(pack_input_s2d_kernel<1>, dim3(a.blocks), dim3(128), 0, st, a.fm, a.fs, a.cand, a.cs, a.in_nc, a.dst, a.limb_stride, a.batch, a.height, a.width));
    else
      CUDA_TRY(launch_pdl(pack_input_s2d_kernel<2>, dim3(a.blocks), dim3(128), 0, st, a.fm, a.fs, a.cand, a.cs, a.in_nc, a.dst, a.limb_stride, a.batch, a.height, a.width));
    if (debug_sync) CUDA_TRY(cudaStreamSynchronize(st));
    if (evs) CUDA_TRY(cudaEventRecord((*evs)[1], st));
  }
  // 2. conv stack
  for (size_t i = 0; i < h->layers.size(); ++i) {
    PlanLayer& pl = P->layers[i];
    if (h->layers[i].kind == K_TAIL) set_tail_io(&pl.prm, io);
    if ((rc = launch_layer(pl, h->layers[i].kind, NL, h->device, st))) return rc;
    if (h->layers[i].kind == K_TAIL) h->tail_func = g_last_func;
    if (pl.split) {
      if (NL == 1) CUDA_TRY(launch_pdl(splitk_reduce_kernel<1>, dim3(pl.red_blocks), dim3(128), 0, st, pl.prm, pl.bn));
      else CUDA_TRY(launch_pdl(splitk_reduce_kernel<2>, dim3(pl.red_blocks), dim3(128), 0, st, pl.prm, pl.bn));
    }
    if (evs) CUDA_TRY(cudaEventRecord((*evs)[i + 2], st));
    if (debug_sync) {
      cudaError_t e = cudaStreamSynchronize(st);
      if (e != cudaSuccess)
        return fail(LSPG_ECUDA, "layer %zu (kind %d, %s, bn %d, grid %d, tiles %d) failed: %s", i, h->layers[i].kind,
                    h->layers[i].conv_key.c_str(), pl.bn, pl.grid, pl.prm.total_tiles, cudaGetErrorString(e));
    }
  }
  return LSPG_OK;
}

void free_plan_graph(Plan* P) {
  if (P->exec) cudaGraphExecDestroy(P->exec);
  if (P->graph) cudaGraphDestroy(P->graph);
  P->exec = nullptr; P->graph = nullptr; P->pack_node = P->tail_node = nullptr;
}

// Capture one forward with `io` baked in, instantiate it, and find the two nodes that carry the caller's pointers.
int capture_plan_graph(lspg_ctx* h, Plan* P, const IoKey& io) {
  const int NL = nl_of(P->mode);
  if (!h->capture_stream) CUDA_TRY(cudaStreamCreateWithFlags(&h->capture_stream, cudaStreamNonBlocking));
  cudaGraph_t graph = nullptr;
  CUDA_TRY(cudaStreamBeginCapture(h->capture_stream, cudaStreamCaptureModeThreadLocal));
  int rc = enqueue_forward(h, P, io, h->capture_stream, false, false);
  cudaError_t ce = cudaStreamEndCapture(h->capture_stream, &graph);
  if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
  if (ce != cudaSuccess) return fail(LSPG_ECUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
  cudaGraphExec_t exec = nullptr;
  ce = cudaGraphInstantiate(&exec, graph, 0);
  if (ce != cudaSuccess) { cudaGraphDestroy(graph); return fail(LSPG_ECUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); }
  P->graph = graph; P->exec = exec; P->io = io;
  P->pack_node = P->tail_node = nullptr;
  // identify the packer and tail nodes by their kernel function (each occurs exactly once per forward)
  const void* pack_func = NL == 1 ? reinterpret_cast<const void*>(pack_input_s2d_kernel<1>)
                                  : reinterpret_cast<const void*>(pack_input_s2d_kernel<2>);
  size_t n = 0;
  if (cudaGraphGetNodes(graph, nullptr, &n) == cudaSuccess && n > 0) {
    std::vector<cudaGraphNode_t> nodes(n);
    if (cudaGraphGetNodes(graph, nodes.data(), &n) == cudaSuccess) {
      for (size_t i = 0; i < n; ++i) {
        cudaGraphNodeType ty;
        if (cudaGraphNodeGetType(nodes[i], &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
        cudaKernelNodeParams np{};
        if (cudaGraphKernelNodeGetParams(nodes[i], &np) != cudaSuccess) continue;
        if (np.func == pack_func) { P->pack_node = nodes[i]; P->pack_np = np; }
        else if (np.func == h->tail_func) { P->tail_node = nodes[i]; P->tail_np = np; }
      }
    }
  }
  cudaGetLastError();      // a failed query above only disables in-place updates (the next pointer change re-captures)
  ++h->n_captures;
  return LSPG_OK;
}

// Patch the caller's pointers into the instantiated graph (input packer arguments, tail ConvParams).
int update_graph_io(lspg_ctx* h, Plan* P, const IoKey& io) {
  if (!P->pack_node || !P->tail_node) return fail(LSPG_ECUDA, "graph nodes of the packer / tail conv were not identified");
  PackArgs a = make_pack_args(h, P, io);
  void* pargs[10] = {&a.fm, &a.fs, &a.cand, &a.cs, &a.in_nc, &a.dst, &a.limb_stride, &a.batch, &a.height, &a.width};
  cudaKernelNodeParams np = P->pack_np;
  np.kernelParams = pargs; np.extra = nullptr;
  CUDA_TRY(cudaGraphExecKernelNodeSetParams(P->exec, P->pack_node, &np));
  ConvParams prm = P->layers.back().prm;
  set_tail_io(&prm, io);
  void* targs[1] = {&prm};
  np = P->tail_np;
  np.kernelParams = targs; np.extra = nullptr;
  CUDA_TRY(cudaGraphExecKernelNodeSetParams(P->exec, P->tail_node, &np));
  P->layers.back().prm = prm;
  P->io = io;
  ++h->n_io_updates;
  return LSPG_OK;
}

}  // namespace

// ====================================================================================================
// C ABI
// ====================================================================================================
extern "C" {

const char* lspg_last_error(void) { return g_err.c_str(); }

int lspg_create(lspg_handle* out, int variant, int ngf, int num_downs, int in_nc, int out_nc, int device) {
  if (!out) return fail(LSPG_EINVAL, "out is NULL");
  *out = nullptr;
  if (variant != LSPG_VARIANT_NORMAL && variant != LSPG_VARIANT_LARGE)
    return fail(LSPG_EINVAL, "variant %d not supported (opt.size 'normal' or 'large')", variant);
  if (ngf < 64 || ngf % 64) return fail(LSPG_EINVAL, "ngf must be a multiple of 64 (got %d)", ngf);
  if (num_downs < 5 || num_downs > 10) return fail(LSPG_EINVAL, "num_downs %d out of range [5,10]", num_downs);
  if (in_nc < 1 || in_nc > 16) return fail(LSPG_EINVAL, "in_nc %d out of range [1,16]", in_nc);
  if (out_nc != 3) return fail(LSPG_EINVAL, "out_nc must be 3 (got %d)", out_nc);
  std::unique_ptr<lspg_ctx> h(new lspg_ctx);
  h->variant = variant; h->ngf = ngf; h->num_downs = num_downs; h->in_nc = in_nc; h->out_nc = out_nc; h->device = device;
  if (device >= 0) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) return fail(LSPG_ENODEV, "no CUDA device: %s", cudaGetErrorString(e));
    if (device >= count) return fail(LSPG_ENODEV, "device %d out of range (%d devices)", device, count);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
      return fail(LSPG_ENODEV, "device %d is sm_%d%d; this library contains sm_100a code only (no fallback)", device,
                  prop.major, prop.minor);
    h->num_sms = prop.multiProcessorCount;
    CUDA_TRY(cudaSetDevice(device));
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CUDA_TRY(cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &fn, 12000, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) return fail(LSPG_ECUDA, "cuTensorMapEncodeTiled not available");
    h->encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  int rc = build_network(h.get());
  if (rc) return rc;
  *out = h.release();
  return LSPG_OK;
}

int lspg_destroy(lspg_handle h) {
  if (!h) return LSPG_OK;
  if (h->device >= 0) {
    cudaSetDevice(h->device);
    for (auto& L : h->layers) {
      if (L.d_w) cudaFree(L.d_w);
      if (L.d_w_fast) cudaFree(L.d_w_fast);
      if (L.d_scale_par) cudaFree(L.d_scale_par);
      if (L.d_scale) cudaFree(L.d_scale);
      if (L.d_shift) cudaFree(L.d_shift);
    }
    for (auto& set : h->prof_events)
      for (auto& e : set) cudaEventDestroy(e);
    for (auto& kv : h->plans) free_plan_graph(kv.second.get());
    if (h->capture_stream) cudaStreamDestroy(h->capture_stream);
    if (h->trace_buf) cudaFree(h->trace_buf);
  }
  delete h;
  return LSPG_OK;
}

int lspg_load_weights(lspg_handle h, const lspg_tensor* tensors, int n) {
  if (!h || (!tensors && n > 0)) return fail(LSPG_EINVAL, "null argument");
  if (h->device >= 0) CUDA_TRY(cudaSetDevice(h->device));
  std::map<std::string, const lspg_tensor*> by_name;
  for (int i = 0; i < n; ++i) {
    if (!tensors[i].name || !tensors[i].data) return fail(LSPG_EINVAL, "tensor %d has a null name or data pointer", i);
    std::string nm = tensors[i].name;
    if (nm.rfind("module.", 0) == 0) nm = nm.substr(7);   // DataParallel prefix (base_model.py:213-215)
    by_name[nm] = &tensors[i];
  }
  auto take = [&](const std::string& key, std::vector<float>& dst, size_t expect, bool* changed) -> int {
    auto it = by_name.find(key);
    if (it == by_name.end()) return LSPG_OK;   // strict=False
    if (static_cast<size_t>(it->second->numel) != expect)
      return fail(LSPG_EINVAL, "%s has %lld elements, expected %zu", key.c_str(), static_cast<long long>(it->second->numel), expect);
    if (dst.size() == expect && memcmp(dst.data(), it->second->data, expect * sizeof(float)) == 0) return LSPG_OK;
    dst.assign(it->second->data, it->second->data + expect);
    *changed = true;
    return LSPG_OK;
  };
  bool synced = false;
  for (auto& L : h->layers) {
    const int cin_total = (L.kind == K_HEAD) ? h->in_nc : (L.cin[0] + (L.n_src == 2 ? L.cin[1] : 0));
    const size_t wn = static_cast<size_t>(L.cout) * cin_total * 9;
    bool changed = false;
    int rc;
    if (L.w.empty()) { L.w.assign(wn, 0.0f); changed = true; }
    if (by_name.count(L.conv_key + ".weight")) L.has_w = true;
    if ((rc = take(L.conv_key + ".weight", L.w, wn, &changed))) return rc;
    if (L.has_bn) {
      if (L.bn_w.empty()) { L.bn_w.assign(L.cout, 1.f); L.bn_b.assign(L.cout, 0.f); L.bn_m.assign(L.cout, 0.f); L.bn_v.assign(L.cout, 1.f); }
      if ((rc = take(L.bn_key + ".weight", L.bn_w, L.cout, &changed))) return rc;
      if ((rc = take(L.bn_key + ".bias", L.bn_b, L.cout, &changed))) return rc;
      if ((rc = take(L.bn_key + ".running_mean", L.bn_m, L.cout, &changed))) return rc;
      if ((rc = take(L.bn_key + ".running_var", L.bn_v, L.cout, &changed))) return rc;
    }
    if (changed || L.dirty) {
      pack_layer(h, L);
      // Packed weights are updated in place (cached plans and graphs keep pointing at them): a forward that is still
      // running on any stream must not see half-written tiles.  Loading weights is rare; one device-wide sync is cheap.
      if (h->device >= 0 && !synced) { CUDA_TRY(cudaDeviceSynchronize()); synced = true; }
      if ((rc = upload_layer(h, L))) return rc;
      L.dirty = false;
    }
  }
  h->weights_loaded = true;
  return LSPG_OK;
}

int lspg_workspace_bytes(lspg_handle h, int batch, int height, int width, int mode, size_t* out) {
  if (!h || !out) return fail(LSPG_EINVAL, "null argument");
  int rc = check_shape(h, batch, height, width, mode);
  if (rc) return rc;
  *out = workspace_bytes(h, batch, height, width, mode);
  return LSPG_OK;
}

static int forward_impl(lspg_handle h, const float* feature_map, int64_t fm_bstride, const float* cand, int64_t cand_bstride,
                        void* out, int out_is_u8, int batch, int height, int width, void* workspace, size_t workspace_bytes_in,
                        int mode, void* stream) {
  if (!h) return fail(LSPG_EINVAL, "null handle");
  if (h->device < 0) return fail(LSPG_ENODEV, "host-only handle: lspg_forward needs an sm_100 device (no CPU path exists)");
  if (!h->weights_loaded) return fail(LSPG_ESTATE, "lspg_load_weights has not been called");
  for (const auto& L : h->layers)
    if (!L.has_w)
      return fail(LSPG_ESTATE, "weights incomplete: %s.weight was never loaded (a forward with zero-filled convs would render "
                  "black frames; nn.DataParallel replicas do not carry parameters - use parallel.ShardedRenderer)", L.conv_key.c_str());
  if (!feature_map || !out || !workspace || (h->in_nc > 1 && !cand)) return fail(LSPG_EINVAL, "null buffer");
  int rc = check_shape(h, batch, height, width, mode);
  if (rc) return rc;
  const size_t need = workspace_bytes(h, batch, height, width, mode);
  if (workspace_bytes_in < need) return fail(LSPG_ESTATE, "workspace too small: %zu < %zu", workspace_bytes_in, need);
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const auto key = std::make_tuple(batch, height, width, mode, workspace);
  auto it = h->plans.find(key);
  if (it == h->plans.end()) {
    std::unique_ptr<Plan> P(new Plan);
    if ((rc = build_plan(h, P.get(), batch, height, width, mode, workspace))) return rc;
    if (h->plans.size() >= 16) {           // bounded: drop the least recently used plan (and its graph)
      auto victim = h->plans.begin();
      for (auto jt = h->plans.begin(); jt != h->plans.end(); ++jt)
        if (jt->second->last_use < victim->second->last_use) victim = jt;
      if (h->last_plan == victim->second.get()) h->last_plan = nullptr;
      free_plan_graph(victim->second.get());
      h->plans.erase(victim);
    }
    it = h->plans.emplace(key, std::move(P)).first;
  }
  Plan* P = it->second.get();
  P->last_use = ++h->use_clock;
  h->last_plan = P;
  IoKey io{feature_map, fm_bstride, cand, cand_bstride, out, out_is_u8};
  static const bool no_graph = getenv("LSPG_NO_GRAPH") != nullptr;
  static const bool debug_sync = getenv("LSPG_DEBUG_SYNC") != nullptr;   // per-layer sync + error attribution (bring-up)
  if (no_graph || debug_sync || h->profiling) return enqueue_forward(h, P, io, st, debug_sync, h->profiling);

  // CUDA-graph replay: the ~80-120 launches of one forward are captured ONCE per plan on a private stream (the caller's
  // stream may be the legacy default stream, which cannot be captured) and replayed with a single cudaGraphLaunch on the
  // caller's stream.  When a call brings other I/O pointers than the ones baked into the instantiated graph, only the
  // two nodes that hold them (input packer, tail conv) are patched - no re-capture, no re-instantiation.
  if (P->exec && !(P->io == io)) {
    if (update_graph_io(h, P, io) != LSPG_OK) {       // should not happen; keep the call correct by re-capturing
      ++h->n_recaptures;
      free_plan_graph(P);
    }
  }
  if (!P->exec) {
    if ((rc = capture_plan_graph(h, P, io))) return rc;
  }
  CUDA_TRY(cudaGraphLaunch(P->exec, st));
  return LSPG_OK;
}

int lspg_forward(lspg_handle h, const float* feature_map, int64_t fm_bstride, const float* cand, int64_t cand_bstride,
                 float* out, int batch, int height, int width, void* workspace, size_t workspace_bytes_in, int mode,
                 void* stream) {
  return forward_impl(h, feature_map, fm_bstride, cand, cand_bstride, out, 0, batch, height, width, workspace,
                      workspace_bytes_in, mode, stream);
}

int lspg_forward_image(lspg_handle h, const float* feature_map, int64_t fm_bstride, const float* cand, int64_t cand_bstride,
                       uint8_t* out_hwc, int batch, int height, int width, void* workspace, size_t workspace_bytes_in,
                       int mode, void* stream) {
  return forward_impl(h, feature_map, fm_bstride, cand, cand_bstride, out_hwc, 1, batch, height, width, workspace,
                      workspace_bytes_in, mode, stream);
}

int lspg_draw_feature_maps(lspg_handle h, const float* landmarks, const float* shoulders, int n_shoulder_points, float* out_fm,
                           int batch, int height, int width, void* stream) {
  if (!h || !landmarks || !out_fm) return fail(LSPG_EINVAL, "null argument");
  if (batch <= 0 || height <= 0 || width <= 0) return fail(LSPG_EINVAL, "bad shape %d x %d x %d", batch, height, width);
  if (shoulders != nullptr && (n_shoulder_points < 0 || n_shoulder_points % 2 != 0))
    return fail(LSPG_EINVAL, "n_shoulder_points must be even (two polylines), got %d", n_shoulder_points);
  if (h->device < 0) return fail(LSPG_ENODEV, "host-only handle: lspg_draw_feature_maps needs an sm_100 device (no CPU path exists)");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaMemsetAsync(out_fm, 0, sizeof(float) * static_cast<size_t>(batch) * height * width, st));
  const int n_sh = shoulders ? n_shoulder_points : 0;
  const int segs = kFaceSegments + (n_sh / 2 > 1 ? 2 * (n_sh / 2 - 1) : 0);
  const int threads = 32;                       // one warp per block: the segments of a frame spread over several SMs
  raster_feature_maps_kernel<<<dim3((segs + threads - 1) / threads, batch), threads, 0, st>>>(landmarks, shoulders, n_sh, out_fm,
                                                                                            height, width);
  CUDA_TRY(cudaGetLastError());
  return LSPG_OK;
}

// ---------------------------------------------------------------------------------------- introspection
int lspg_num_layers(lspg_handle h, int* out) {
  if (!h || !out) return fail(LSPG_EINVAL, "null argument");
  *out = static_cast<int>(h->layers.size());
  return LSPG_OK;
}

int lspg_layer_info_get(lspg_handle h, int layer, lspg_layer_info* o) {
  if (!h || !o) return fail(LSPG_EINVAL, "null argument");
  if (layer < 0 || layer >= static_cast<int>(h->layers.size())) return fail(LSPG_EINVAL, "layer %d out of range", layer);
  const Layer& L = h->layers[layer];
  memset(o, 0, sizeof(*o));
  o->kind = L.kind; o->n_src = L.n_src;
  for (int s = 0; s < 2; ++s) { o->src[s] = L.src[s]; o->cin[s] = L.cin[s]; }
  o->out = L.out; o->res = L.res; o->cout = L.cout; o->cout_pad = L.cout_pad;
  o->n_phases = L.n_phases; o->n_taps = L.n_taps; o->k_total = L.k_total; o->relu = L.relu; o->has_bn = L.has_bn;
  memcpy(o->tap_map, L.tap_map, sizeof(o->tap_map));
  memcpy(o->tap_dx, L.tap_dx, sizeof(o->tap_dx));
  memcpy(o->tap_dy, L.tap_dy, sizeof(o->tap_dy));
  snprintf(o->conv_key, sizeof(o->conv_key), "%s", L.conv_key.c_str());
  snprintf(o->bn_key, sizeof(o->bn_key), "%s", L.bn_key.c_str());
  return LSPG_OK;
}

int lspg_layer_packed(lspg_handle h, int layer, int limb, uint16_t* dst, int64_t count) {
  if (!h || !dst) return fail(LSPG_EINVAL, "null argument");
  if (layer < 0 || layer >= static_cast<int>(h->layers.size()) || limb < 0 || limb > 2) return fail(LSPG_EINVAL, "bad layer/limb");
  const Layer& L = h->layers[layer];
  if (L.packed[limb].empty()) return fail(LSPG_ESTATE, "weights not loaded");
  if (static_cast<size_t>(count) != L.packed[limb].size()) return fail(LSPG_EINVAL, "count %lld != %zu", static_cast<long long>(count), L.packed[limb].size());
  memcpy(dst, L.packed[limb].data(), L.packed[limb].size() * 2);
  return LSPG_OK;
}

int lspg_layer_affine(lspg_handle h, int layer, float* scale, float* shift, int64_t count) {
  if (!h || !scale || !shift) return fail(LSPG_EINVAL, "null argument");
  if (layer < 0 || layer >= static_cast<int>(h->layers.size())) return fail(LSPG_EINVAL, "bad layer");
  const Layer& L = h->layers[layer];
  if (L.scale.empty()) return fail(LSPG_ESTATE, "weights not loaded");
  if (count != L.cout_pad) return fail(LSPG_EINVAL, "count %lld != %d", static_cast<long long>(count), L.cout_pad);
  memcpy(scale, L.scale.data(), L.cout_pad * 4);
  memcpy(shift, L.shift.data(), L.cout_pad * 4);
  return LSPG_OK;
}

int lspg_num_tensors(lspg_handle h, int* out) {
  if (!h || !out) return fail(LSPG_EINVAL, "null argument");
  *out = static_cast<int>(h->tensors.size());
  return LSPG_OK;
}

int lspg_tensor_shape(lspg_handle h, int id, int height, int width, int* c, int* th, int* tw) {
  if (!h || !c || !th || !tw) return fail(LSPG_EINVAL, "null argument");
  if (id < 0 || id >= static_cast<int>(h->tensors.size())) return fail(LSPG_EINVAL, "tensor %d out of range", id);
  *c = h->tensors[id].channels; *th = height >> h->tensors[id].shift; *tw = width >> h->tensors[id].shift;
  return LSPG_OK;
}

int lspg_debug_read_tensor(lspg_handle h, int id, int limb, uint16_t* dst, int64_t count) {
  if (!h || !dst) return fail(LSPG_EINVAL, "null argument");
  if (h->device < 0 || !h->last_plan) return fail(LSPG_ESTATE, "no forward has run on this handle");
  Plan* P = h->last_plan;
  if (id < 0 || id >= static_cast<int>(h->tensors.size())) return fail(LSPG_EINVAL, "tensor %d out of range", id);
  if (limb < 0 || limb >= nl_of(P->mode)) return fail(LSPG_EINVAL, "limb %d not present in this mode", limb);
  const size_t bytes = tensor_bytes_one_limb(h->tensors[id], P->batch, P->height, P->width);
  if (static_cast<size_t>(count) * 2 != bytes) return fail(LSPG_EINVAL, "count %lld != %zu", static_cast<long long>(count), bytes / 2);
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(dst, static_cast<uint8_t*>(P->workspace) + P->tensor_off[id] + limb * P->tensor_limb_stride[id], bytes,
                      cudaMemcpyDeviceToHost));
  return LSPG_OK;
}

int lspg_debug_layer_geo(lspg_handle h, int layer, int batch, int height, int width, lspg_layer_geo* o) {
  if (!h || !o) return fail(LSPG_EINVAL, "null argument");
  if (layer < 0 || layer >= static_cast<int>(h->layers.size())) return fail(LSPG_EINVAL, "layer %d out of range", layer);
  int rc = check_shape(h, batch, height, width, LSPG_MODE_PARITY);
  if (rc) return rc;
  const Layer& L = h->layers[layer];
  const Geo g = layer_geo(h, L, batch, height, width);
  memset(o, 0, sizeof(*o));
  o->kernel = g.pair ? 2 : (g.patch ? 1 : 0);
  o->bn = g.bn;
  o->tile_w = g.tw; o->tile_h = g.th; o->tile_n = g.nb;
  o->m_tiles = g.m_tiles; o->n_tiles = g.n_tiles; o->n_phases = L.n_phases;
  o->n_split = g.n_split; o->split_len = g.split_len; o->k_items = g.k_items;
  const int sms = h->num_sms_or_default();
  int ctas = std::min(g.tiles_per_split * g.n_split, sms);
  if (g.pair) ctas -= ctas % 2;
  o->ctas = ctas;
  o->partial_bytes = static_cast<int64_t>(g.partial_bytes);
  o->cluster_split = g.csplit;
  o->cta_cluster = g.cluster;
  return LSPG_OK;
}

int lspg_debug_tensor_offset(lspg_handle h, int id, int limb, int batch, int height, int width, int mode, size_t* offset) {
  if (!h || !offset) return fail(LSPG_EINVAL, "null argument");
  int rc = check_shape(h, batch, height, width, mode);
  if (rc) return rc;
  if (id < 0 || id >= static_cast<int>(h->tensors.size())) return fail(LSPG_EINVAL, "tensor %d out of range", id);
  if (limb < 0 || limb >= nl_of(mode)) return fail(LSPG_EINVAL, "limb %d not present in this mode", limb);
  std::vector<size_t> off, limb_stride;
  tensor_layout(h, batch, height, width, nl_of(mode), &off, &limb_stride);
  *offset = off[id] + static_cast<size_t>(limb) * limb_stride[id];
  return LSPG_OK;
}

int lspg_debug_fast_div(uint32_t n, uint32_t d, uint32_t* q) {
  if (!q || d == 0 || n >= (1u << 31)) return fail(LSPG_EINVAL, "fast_div: need q, d >= 1 and n < 2^31");
  const FastDiv f = make_fast_div(d);
  // host form of the device's __umulhi(n, mul) >> shr
  *q = (f.d == 1) ? n : static_cast<uint32_t>((static_cast<uint64_t>(n) * f.mul) >> 32) >> f.shr;
  return LSPG_OK;
}

int lspg_debug_read_trace(lspg_handle h, uint64_t* dst, int64_t count) {
  if (!h || !dst) return fail(LSPG_EINVAL, "null argument");
  if (!h->trace_buf) return fail(LSPG_ESTATE, "no trace recorded (set LSPG_TRACE_LAYER=<layer index> before the first forward)");
  if (count != 256 * kTraceSlots) return fail(LSPG_EINVAL, "count must be %d", 256 * kTraceSlots);
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(dst, h->trace_buf, sizeof(uint64_t) * count, cudaMemcpyDeviceToHost));
  return LSPG_OK;
}

int lspg_graph_stats(lspg_handle h, int64_t* captures, int64_t* io_updates, int64_t* recaptures) {
  if (!h || !captures || !io_updates || !recaptures) return fail(LSPG_EINVAL, "null argument");
  *captures = h->n_captures; *io_updates = h->n_io_updates; *recaptures = h->n_recaptures;
  return LSPG_OK;
}

int lspg_release_workspace(lspg_handle h, void* workspace) {
  if (!h) return fail(LSPG_EINVAL, "null handle");
  if (h->device >= 0) {
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaDeviceSynchronize());            // forwards that still use the workspace finish before their plan goes
  }
  for (auto it = h->plans.begin(); it != h->plans.end();) {
    if (workspace == nullptr || std::get<4>(it->first) == workspace) {
      if (h->last_plan == it->second.get()) h->last_plan = nullptr;
      free_plan_graph(it->second.get());
      it = h->plans.erase(it);
    } else {
      ++it;
    }
  }
  return LSPG_OK;
}

int lspg_launches_per_forward(lspg_handle h, int* out) {
  if (!h || !out) return fail(LSPG_EINVAL, "null argument");
  int n = 1 + static_cast<int>(h->layers.size());
  if (h->last_plan)
    for (const auto& pl : h->last_plan->layers) n += pl.split ? 1 : 0;   // + split-K finishers of the last plan
  *out = n;
  return LSPG_OK;
}

int lspg_profile_enable(lspg_handle h, int enabled) {
  if (!h) return fail(LSPG_EINVAL, "null handle");
  if (h->device < 0) return fail(LSPG_ENODEV, "host-only handle");
  h->profiling = enabled != 0;
  h->prof_used = 0;
  return LSPG_OK;
}

int lspg_profile_read(lspg_handle h, float* avg_ms, int count, int* n_forwards) {
  if (!h || !avg_ms || !n_forwards) return fail(LSPG_EINVAL, "null argument");
  const int n = 1 + static_cast<int>(h->layers.size());
  if (count != n) return fail(LSPG_EINVAL, "count %d != launches per forward %d", count, n);
  CUDA_TRY(cudaSetDevice(h->device));
  for (int i = 0; i < n; ++i) avg_ms[i] = 0.f;
  for (size_t f = 0; f < h->prof_used; ++f) {
    auto& set = h->prof_events[f];
    CUDA_TRY(cudaEventSynchronize(set[n]));
    for (int i = 0; i < n; ++i) {
      float ms = 0.f;
      CUDA_TRY(cudaEventElapsedTime(&ms, set[i], set[i + 1]));
      avg_ms[i] += ms;
    }
  }
  *n_forwards = static_cast<int>(h->prof_used);
  if (h->prof_used)
    for (int i = 0; i < n; ++i) avg_ms[i] /= static_cast<float>(h->prof_used);
  h->prof_used = 0;
  return LSPG_OK;
}

int lspg_flops_per_frame(lspg_handle h, int height, int width, double* out) {
  if (!h || !out) return fail(LSPG_EINVAL, "null argument");
  double total = 0;
  for (const auto& L : h->layers) {
    // algorithmic work of the REFERENCE conv this layer implements: 2 * Ho*Wo*Cout*Cin*9
    const int cin_total = (L.kind == K_HEAD) ? h->in_nc : (L.cin[0] + (L.n_src == 2 ? L.cin[1] : 0));
    int oshift = L.grid_shift;                                   // output grid
    if (L.kind == K_UP || L.kind == K_TAIL) oshift = L.grid_shift - 1;   // upsampled output
    total += 2.0 * (height >> oshift) * (width >> oshift) * static_cast<double>(L.cout) * cin_total * 9.0;
  }
  *out = total;
  return LSPG_OK;
}

}  // extern "C"
