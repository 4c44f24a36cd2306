// Fused 3x3 convolution as an implicit GEMM on tcgen05 tensor cores (sm_100a).
//
// One kernel family serves every conv of the Res-UNet generator
// (reference: models/networks.py:585-675; SURVEY.md section 2a K1..K5):
//
//   D[128 pixels x BN channels] (+)= A[128 pixels x 64 ch] * B[BN x 64 ch]^T      per K block
//
//   * A K block = (tap, concat source, 64-channel chunk).  The A tile of a tap is the output tile's pixel
//     patch shifted by (dx, dy): ONE 5-D TMA box {64 ch, TW, TH, NB, 1 limb} out of the NHWC activation
//     tensor; out-of-range coordinates are zero-filled by TMA, which is the conv's zero padding.
//   * stride-2 convs read through four parity views of the input (base offset + doubled strides), the
//     nearest-x2 upsample is folded into four output phases with 2x2 pre-summed taps whose results are
//     stored through four phase views of the output, and torch.cat([skip, deeper]) is two K ranges fed from
//     two tensor maps - so upsample, concat, padding and stride never touch HBM as separate passes.
//   * B tiles come from a packed weight tensor [phase*limb][Cout][K] (K-major), same 128B-swizzled layout.
//   * Accumulators live in a TMEM ring (2-4 buffers); the epilogue warps read them with tcgen05.ld, apply the folded
//     eval-BatchNorm scale/shift in fp32, add the residual (256-bit ld.global.nc straight from the NHWC tensor, requested
//     one piece ahead), ReLU, convert to bf16 (hi, lo) and write the NHWC output with 256-bit global stores (no smem
//     staging, no TMA store).  The tail variant applies tanh and scatters fp32 NCHW or uint8 HWC directly.
//   * NL = 2 ("parity" precision): activations and weights are split into fp16 hi + lo limbs; each K step issues
//     hi*hi + hi*lo + lo*hi (22 mantissa bits per operand, fp32 accumulate) and the epilogue writes both limbs.
//     NL = 1 ("fast"): one bf16 limb, one MMA per K step.
//
// Three kernels share the epilogue: conv_umma_kernel (one TMA box per tap; stride-2 convs and everything below 16x16;
// 192 threads = producer warp + MMA warp + 4 epilogue warps), conv_patch_kernel (one halo patch per chunk; head and tail)
// and conv_pair_kernel (cta_group::2 over a 2-CTA cluster; the wide layers; 320 threads = 2 role warps + 8 epilogue
// warps).  All are persistent: each CTA walks tiles blockIdx.x, +gridDim.x, ...
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "ptx.cuh"

namespace lspg {

constexpr int kTileM = 128;                 // output pixels per tile (UMMA M)
constexpr int kChunk = 64;                  // channels per K block = 128 bytes of bf16 = one swizzle row
constexpr int kATile = kTileM * 128;        // bytes of one A (or staging) tile
constexpr int kMaxTaps = 9;
constexpr int kThreads = 192;            // 2 role warps + 4 epilogue warps
constexpr int kSmemBudget = 227 * 1024;

// Division by a launch-time constant as multiply-high + shift (dividend < 2^31): decode_tile runs between two tiles of
// the persistent loops, where ~9 hardware integer divisions cost more than a thousand cycles.
struct FastDiv {
  uint32_t mul, shr, d;
};
inline FastDiv make_fast_div(uint32_t d) {
  FastDiv f;
  f.d = d; f.mul = 0; f.shr = 0;
  if (d > 1) {
    uint32_t l = 0;
    while ((1u << l) < d) ++l;
    const uint64_t pw = 31 + l;
    f.mul = static_cast<uint32_t>(((1ull << pw) + d - 1) / d);
    f.shr = static_cast<uint32_t>(pw - 32);
  }
  return f;
}
__device__ __forceinline__ int fast_div(int n, const FastDiv& f) {
  return f.d == 1 ? n : static_cast<int>(__umulhi(static_cast<uint32_t>(n), f.mul) >> f.shr);
}

struct alignas(64) ConvParams {
  // Field order matters: kernel parameters live in constant bank 0 and are fetched through a small per-SM constant cache
  // that the three warp roles share.  An ncu source view of the 64-channel layers showed the epilogue's first touch of
  // each parameter line missing once per tile (6 % of all stall samples on one LDC), so everything the epilogue and the
  // tile decode read every tile sits in the first two 128-byte lines, the issue/producer scalars and tap tables follow,
  // and the tensor maps (read by the TMA unit through their generic address, not through the constant cache) come last.
  // ---- epilogue + tile decode (hot)
  const float* scale;        // folded BatchNorm (or 1/0), [Cout_pad]
  const float* shift;
  __nv_bfloat16* out_ptr;         // output tensor (NHWC), limb 0; written directly by the epilogue
  const __nv_bfloat16* res_ptr;   // residual tensor (NHWC, same grid as the output), limb 0; read directly by the epilogue
  long long out_limb_stride;      // elements between limbs
  long long res_limb_stride;      // elements between limbs
  float* out_f32;            // tail only: fp32 NCHW [B, 3, 2*hs, 2*ws]
  uint8_t* out_u8;           // tail only, optional: uint8 HWC image [B, 2*hs, 2*ws, 3] = util.tensor2im fused (then out_f32 is unused)
  float* partial;            // split-K partial tiles (see n_split)
  unsigned long long* trace; // debug: per-CTA clock64 stamps (null in production), see kTraceSlots
  int32_t out_channels, res_channels;
  int32_t out_up;            // the sampling grid is the source of a folded x2 upsample (phase tc.z -> (2y+py, 2x+px))
  int32_t relu, has_res;
  int32_t batch, hs, ws;     // sampling-grid extent (tail epilogue addressing)
  int32_t tw_log2, th_log2;  // tile = TW x TH pixels x NB images, TW*TH*NB = 128
  int32_t total_tiles;       // tiles_x*tiles_y*tiles_n * n_tiles * n_phases * n_split
  // split-K: the K loop (v1: K blocks; patch mode: (source, chunk) items) is cut into n_split ranges of split_len;
  // tile index = split * tiles_per_split + tile.  Each CTA writes its raw fp32 accumulator tile to
  // partial[tile_index][128][BN]; splitk_reduce_kernel (given these same parameters) sums the splits and finishes the tile.
  int32_t n_split, tiles_per_split;
  int32_t cluster_split;     // 1: the n_split CTAs of a tile form a thread-block cluster and reduce their partials through
                             // distributed shared memory (CSP kernel variants); 0: partials go to `partial` + finisher kernel
  int32_t n_tiles;           // Cout_pad / BN
  int32_t tiles_x, tiles_y, tiles_n;
  int32_t n_phases;
  int32_t trace_skip;        // debug: the trace records local tiles [trace_skip, trace_skip + kTraceTiles)
  FastDiv fd_tps, fd_m_tiles, fd_n_tiles, fd_tiles_x, fd_tiles_y;   // divisions of decode_tile (tiles_per_split, ...)
  // ---- MMA issue + TMA producer
  uint32_t idesc;            // UMMA instruction descriptor (M=128 or 256, N=BN, bf16 x bf16 -> f32, K-major)
  uint32_t idesc2;           // same with N=2*BN (parity: stacked [B_hi;B_lo] operand)
  int32_t n_taps, n_src;
  int32_t chunks[2];         // 64-channel chunks per concat source
  int32_t split_len;
  int32_t b_resident;        // pair kernel: every weight tile of the layer fits the B ring -> load once per CTA, no streaming
  // patch mode: one halo patch {64 ch, patch_w, patch_h} per (tile, source, chunk) whose origin is the tile origin +
  // (patch_dx0, patch_dy0)[phase]; every tap is a row offset inside the patch.
  int32_t patch_w, patch_h;
  int8_t patch_dx0[4], patch_dy0[4];
  int16_t tap_row[4][kMaxTaps];  // [phase][tap] -> first patch row of the tap's shifted A tile
  int8_t tap_map[4][kMaxTaps];   // [phase][tap] -> index into a[] (added to the concat source index)
  int8_t tap_dx[4][kMaxTaps];
  int8_t tap_dy[4][kMaxTaps];
  // ---- tensor maps
  CUtensorMap a[4];          // activation views: [parity or concat source], dims {C, X, Y, N, limb}
  CUtensorMap w;             // packed weights, dims {K, Cout_pad, limb*n_phases + phase}
};

// CSP ("cluster split"): split-K inside a thread-block cluster.  The n_split (2, 4 or 8) CTAs that share an output tile are
// one cluster; every CTA owns 128 / n_split rows of the tile and receives those rows of every CTA's fp32 partial in a
// staging buffer of its own shared memory (128 x BN floats in total), sums them in split order and applies the epilogue.
// No partials in global memory and no finisher launch (at batch 1 the finishers were 46 of 123 launches).
template <int BN, int NL, bool TAIL, bool CSP = false>
struct ConvCfg {
  static constexpr int kBTile = BN * 128;
  static constexpr int kStage = NL * (kATile + kBTile);
  static constexpr int kStgBytes = CSP ? kTileM * BN * 4 : 0;        // cluster split-K: partial rows from the cluster's CTAs
  static constexpr int kAux = 3072;                                  // 2 x (scale, shift) + barriers + tmem ptr
  static constexpr int kAvail = kSmemBudget - 1024 /*alignment slack*/ - kStgBytes - kAux;
  static constexpr int kStagesRaw = kAvail / kStage;
  static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
  static constexpr int kSmemBytes = 1024 + kStages * kStage + kStgBytes + kAux;
  static constexpr int kTmemCols = (2 * BN < 32) ? 32 : 2 * BN;
  static_assert(kStages >= 2, "pipeline needs at least two stages");
  static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "invalid UMMA N");
  // scale/shift, full/empty per stage, tfull/tempty per accumulator buffer, TMEM address
  static_assert(4 * BN * 4 + (2 * kStages + 2 * 2 + 1) * 8 <= kAux, "aux region too small");
};

// Debug trace layout per CTA: [0] kernel entry, [1] prologue done, then per local tile i (up to kTraceTiles):
//   base = 4 + 8*i: +0 MMA got TMEM buffer, +1 MMA first B stage landed, +2 MMA last commit issued,
//                   +3 EPI waiting for accumulator, +4 EPI accumulator ready, +5 EPI tile done,
//                   +6 PROD first B load of the tile issued, +7 PROD last B load issued
constexpr int kTraceTiles = 12;
constexpr int kTraceSlots = 4 + 8 * kTraceTiles + 4;   // tail: [+0] clock64 at kernel exit; slots 2/3: globaltimer (ns) at entry/exit
__device__ __forceinline__ void trace_stamp(const ConvParams& p, int slot);

struct TileCoord {
  int z, nt, x0, y0, n0, split;
};

__device__ __forceinline__ void trace_stamp(const ConvParams& p, int slot) {
  if (p.trace != nullptr && slot < kTraceSlots) p.trace[static_cast<size_t>(blockIdx.x) * kTraceSlots + slot] = clock64();
}

__device__ __forceinline__ void trace_time(const ConvParams& p, bool at_exit) {
  if (p.trace != nullptr) {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(ns));
    unsigned long long* t = p.trace + static_cast<size_t>(blockIdx.x) * kTraceSlots;
    t[at_exit ? 3 : 2] = ns;
    if (at_exit) t[4 + 8 * kTraceTiles] = clock64();
  }
}
__device__ __forceinline__ void trace_tile(const ConvParams& p, int lt, int k) {
  if (p.trace != nullptr) {
    const int i = lt - p.trace_skip;
    if (i >= 0 && i < kTraceTiles) p.trace[static_cast<size_t>(blockIdx.x) * kTraceSlots + 4 + 8 * i + k] = clock64();
  }
}

// The MMA-issuing warp only needs the phase and split index of a tile; for the common single-phase, unsplit layer that
// is (0, 0) without any integer division (the full decode costs several hundred cycles between two tiles).
__device__ __forceinline__ void decode_tile_zs(const ConvParams& p, int t, int& z, int& split) {
  if (p.n_phases == 1 && p.n_split == 1) { z = 0; split = 0; return; }
  split = fast_div(t, p.fd_tps);
  t -= split * p.tiles_per_split;
  z = fast_div(fast_div(t, p.fd_m_tiles), p.fd_n_tiles);
}

__device__ __forceinline__ TileCoord decode_tile(const ConvParams& p, int t) {
  TileCoord c;
  c.split = fast_div(t, p.fd_tps);
  t -= c.split * p.tiles_per_split;
  const int r = fast_div(t, p.fd_m_tiles);
  const int mt = t - r * static_cast<int>(p.fd_m_tiles.d);
  c.z = fast_div(r, p.fd_n_tiles);
  c.nt = r - c.z * p.n_tiles;
  const int r2 = fast_div(mt, p.fd_tiles_x);
  const int tx = mt - r2 * p.tiles_x;
  const int tn = fast_div(r2, p.fd_tiles_y);
  const int ty = r2 - tn * p.tiles_y;
  c.x0 = tx << p.tw_log2;
  c.y0 = ty << p.th_log2;
  c.n0 = tn << (7 - p.tw_log2 - p.th_log2);
  return c;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);   // .x = lo (low 16 bits), .y = hi
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

// 16-bit operand formats.  FAST (one limb) keeps bf16 (north_star's "bf16 in / fp32 accum").  PARITY (two limbs) uses fp16:
// hi = fp16(v), lo = fp16(v - hi) carry 22 mantissa bits where two bf16 limbs carry 16, at the same tensor cost
// (kind::f16 takes either format) - oracle/precision_study.py: 4.3e-5 instead of 2.2e-4 on the hard case.  The range is
// fp16's: conversions saturate at +-65504 instead of producing infinities (activations of this network are O(1..100)).
// F16 = (NL == 2) everywhere.
template <bool F16>
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  if constexpr (F16) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));     // upper half <- first source
    return r;
  } else {
    return pack_bf16x2(lo, hi);
  }
}
template <bool F16>
__device__ __forceinline__ float unpack_lo(uint32_t u) {
  if constexpr (F16) return __half2float(__ushort_as_half(static_cast<unsigned short>(u & 0xFFFFu)));
  else return bf16_lo(u);
}
template <bool F16>
__device__ __forceinline__ float unpack_hi(uint32_t u) {
  if constexpr (F16) return __half2float(__ushort_as_half(static_cast<unsigned short>(u >> 16)));
  else return bf16_hi(u);
}

// Output pixel of row `row` of tile `tc`: image n and sampling-grid position (y, x), whether it lies inside the image, and the
// element offset of its channel 0 in the NHWC output (limb 0).  A folded x2 upsample stores phase z at (2y + z/2, 2x + z%2).
struct OutPixel {
  int n, y, x;
  bool ok;
  size_t out;
};
__device__ __forceinline__ OutPixel out_pixel(const ConvParams& p, const TileCoord& tc, int row) {
  OutPixel o;
  o.n = tc.n0 + (row >> (p.tw_log2 + p.th_log2));
  o.y = tc.y0 + ((row >> p.tw_log2) & ((1 << p.th_log2) - 1));
  o.x = tc.x0 + (row & ((1 << p.tw_log2) - 1));
  o.ok = o.n < p.batch && o.y < p.hs && o.x < p.ws;
  const int oh = p.out_up ? 2 * p.hs : p.hs, ow = p.out_up ? 2 * p.ws : p.ws;
  const int oy = p.out_up ? 2 * o.y + (tc.z >> 1) : o.y, ox = p.out_up ? 2 * o.x + (tc.z & 1) : o.x;
  o.out = ((static_cast<size_t>(o.n) * oh + oy) * ow + ox) * p.out_channels;
  return o;
}
// the residual has the output's sampling grid (residual layers are never upsampling ones)
__device__ __forceinline__ size_t res_offset(const ConvParams& p, const OutPixel& o) {
  return ((static_cast<size_t>(o.n) * p.hs + o.y) * p.ws + o.x) * p.res_channels;
}

// The last steps of every conv output, shared by the epilogue and both split-K finishers so that they round alike.  y holds
// C channels of one pixel that already went through the folded BatchNorm (fmaf(acc, scale, shift)); res[l] holds the C / 2
// packed residual words of limb l (read only with has_res).  Adds the residual limbs in limb order, applies ReLU and rounds to
// the 16-bit hi limb (hi: C / 2 packed words); for NL == 2 also to the lo limb y - hi.
template <int NL, int C>
__device__ __forceinline__ void finish_channels(float (&y)[C], const uint32_t (&res)[NL][C / 2], bool has_res, bool relu,
                                                uint32_t (&hi)[C / 2], uint32_t (&lo)[C / 2]) {
  constexpr bool F16 = NL == 2;
  if (has_res) {
#pragma unroll
    for (int l = 0; l < NL; ++l)
#pragma unroll
      for (int e = 0; e < C / 2; ++e) {
        y[2 * e] += unpack_lo<F16>(res[l][e]);
        y[2 * e + 1] += unpack_hi<F16>(res[l][e]);
      }
  }
  if (relu) {
#pragma unroll
    for (int e = 0; e < C; ++e) y[e] = fmaxf(y[e], 0.0f);
  }
#pragma unroll
  for (int e = 0; e < C / 2; ++e) hi[e] = pack2<F16>(y[2 * e], y[2 * e + 1]);
  if constexpr (F16) {
#pragma unroll
    for (int e = 0; e < C / 2; ++e) lo[e] = pack2<true>(y[2 * e] - unpack_lo<true>(hi[e]), y[2 * e + 1] - unpack_hi<true>(hi[e]));
  }
}

// Split-K finishers: channels [ch, ch + 4) of pixel o from their summed fp32 accumulator, with scale, shift and residual
// read from global memory.  One thread = one pixel x 4 channels.
template <int NL>
__device__ __forceinline__ void finish4(const ConvParams& p, const OutPixel& o, int ch, float4 acc) {
  const float4 sc = *reinterpret_cast<const float4*>(p.scale + ch), sh = *reinterpret_cast<const float4*>(p.shift + ch);
  float y[4] = {fmaf(acc.x, sc.x, sh.x), fmaf(acc.y, sc.y, sh.y), fmaf(acc.z, sc.z, sh.z), fmaf(acc.w, sc.w, sh.w)};
  uint32_t r[NL][2];
  if (p.has_res) {
    const __nv_bfloat16* rr = p.res_ptr + res_offset(p, o) + ch;
#pragma unroll
    for (int l = 0; l < NL; ++l) {
      const uint2 v = *reinterpret_cast<const uint2*>(rr + l * p.res_limb_stride);
      r[l][0] = v.x; r[l][1] = v.y;
    }
  }
  uint32_t hi[2], lo[2];
  finish_channels<NL, 4>(y, r, p.has_res, p.relu, hi, lo);
  __nv_bfloat16* out = p.out_ptr + o.out + ch;
  *reinterpret_cast<uint2*>(out) = make_uint2(hi[0], hi[1]);
  if constexpr (NL == 2) *reinterpret_cast<uint2*>(out + p.out_limb_stride) = make_uint2(lo[0], lo[1]);
}

// Epilogue role (warps 2..2+EW-1): drains the TMEM accumulators of every tile this CTA owns.  Per tile it either
//   * tail: applies scale/shift and tanh and scatters fp32 NCHW or uint8 HWC,
//   * split-K: dumps the raw fp32 rows (to the owner CTA's staging buffer under CSP, else to `partial`), or
//   * regular: applies scale/shift from shared memory and finish_channels, and stores NHWC with 256-bit stores.
// STACK (parity mode of the patch kernel): the accumulator of a tile is 2*BN columns wide - columns [0,BN) hold
// A_hi*B_hi + A_lo*B_hi, columns [BN,2BN) hold A_hi*B_lo (one N=2BN MMA over the stacked [B_hi;B_lo] tile) - and the
// epilogue adds the two halves.
// EW = number of epilogue warps (4 or 8).  A warp may read TMEM lane quarter (warp % 4); with EW = 8 two warps share a
// quarter and split the columns in interleaved 32-column pieces, which doubles the loads/stores in flight and the issue
// slots of the epilogue (the 64-channel layers were epilogue-bound with 4 warps: 6.2k cycles vs 3.5k of MMAs per tile).
// stg_base: the cluster split-K staging buffer (CSP only).
template <int BN, int NL, bool TAIL, bool STACK, bool PAIR = false, int EW = 4, int NACC = 2, bool CSP = false>
__device__ __forceinline__ void epilogue_warps(const ConvParams& p, uint8_t* stg_base, float* s_scale0, uint64_t* tfull_bar,
                                               uint64_t* tempty_bar, uint32_t tmem_base, int warp, int lane, int t0, int tstep) {
  static_assert(EW == 4 || EW == 8, "4 or 8 epilogue warps");
  static_assert(!(TAIL && EW != 4), "the tail epilogue uses 4 warps");
  constexpr int kEpi = EW * 32;
  constexpr int kGroups = EW / 4;
  ptx::pdl_wait();   // residual reads, output / split-K partial writes must not overtake the previous kernel
  const int q = warp & 3;                     // TMEM lane quarter this warp may read
  const int grp = (warp - 2) >> 2;            // which interleaved share of the 32-column pieces this warp takes
  const int row = q * 32 + lane;              // tile row = pixel index inside the tile
  const int etid = threadIdx.x - 64;          // 0..kEpi-1
  const bool leader = (etid == 0);
  int acc = 0;
  uint32_t acc_phase = 0;
  auto release_tmem = [&]() {
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if constexpr (PAIR) ptx::mbar_arrive_cluster(&tempty_bar[acc], 0);
      else ptx::mbar_arrive(&tempty_bar[acc]);
    }
  };

  // Folded BatchNorm parameters of the current N tile, in shared memory.  Tiles are ordered M-fastest, so a CTA's N tile
  // changes a handful of times per launch (never when Cout = BN): the parameters are re-fetched only then, between two
  // barriers of the epilogue warps.  No per-tile barrier: TMEM double buffering bounds the skew between the warps.
  static_assert(BN / 2 <= kEpi, "one 16-byte piece of scale/shift per thread");
  float* const s_scale = s_scale0;
  float* const s_shift = s_scale0 + BN;
  int cur_nt = -1;
  auto fetch_affine = [&](int nt) {
    ptx::named_bar_sync(1, kEpi);        // every warp is done with the previous N tile's parameters
    if (etid < BN / 2) {
      const bool sh = etid >= BN / 4;
      const int i = (sh ? etid - BN / 4 : etid) * 4;
      ptx::cp_async16(s_scale0 + (sh ? BN : 0) + i, (sh ? p.shift : p.scale) + nt * BN + i);
    }
    ptx::cp_async_wait_all();
    ptx::named_bar_sync(1, kEpi);
    cur_nt = nt;
  };
  // Residual of this thread's pixel: 32 channels x NL limbs per 32-column piece, always requested one piece ahead - the
  // first piece of a tile while the previous tile is being finished - so that its L2/HBM latency never sits between the
  // accumulator becoming ready and the TMEM buffer being handed back to the MMA warp.
  const bool use_res = !TAIL && p.has_res && p.n_split == 1;
  uint4 rs[NL][4];
  auto load_res = [&](const TileCoord& c, int c32) {
    const OutPixel o = out_pixel(p, c, row);
    // rows outside the image read pixel 0 instead (their result is never stored): no branch around the loads, so the
    // destination registers stay plain in-flight load targets until the math consumes them
    const __nv_bfloat16* rr = p.res_ptr + (o.ok ? res_offset(p, o) : 0) + c.nt * BN + c32 * 32;
#pragma unroll
    for (int l = 0; l < NL; ++l)
#pragma unroll
      for (int h2 = 0; h2 < 2; ++h2)
        ptx::ldg256_nc(rr + l * p.res_limb_stride + h2 * 16, rs[l][2 * h2], rs[l][2 * h2 + 1]);
  };
  int lt = 0;
  TileCoord tc_next = decode_tile(p, t0);
  if (t0 < p.total_tiles) {
    if (use_res) load_res(tc_next, grp);
  }
  for (int t = t0; t < p.total_tiles; t += tstep, ++lt) {
    const TileCoord tc = tc_next;
    if (leader) trace_tile(p, lt, 3);
    const bool split_mode = !TAIL && p.n_split > 1;
    if (tc.nt != cur_nt) fetch_affine(tc.nt);
    const int t_next = t + tstep;
    if (t_next < p.total_tiles) tc_next = decode_tile(p, t_next);

    constexpr int kAccCols = STACK ? 2 * BN : BN;
    const uint32_t t_acc = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kAccCols;

    ptx::mbar_wait(&tfull_bar[acc], acc_phase);
    ptx::tc_fence_after();
    if (leader) trace_tile(p, lt, 4);

    if constexpr (TAIL) {
      // ---- tail: 16 columns = 4 phases x 3 channels (+4 pad); tanh; fp32 NCHW scatter or fused tensor2im
      uint32_t v[16];
      ptx::tmem_ld_32x16(t_acc, v);
      if constexpr (STACK) {
        uint32_t v2[16];
        ptx::tmem_ld_32x16(t_acc + BN, v2);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(v2[i]));
      }
      ptx::tmem_ld_wait();
      release_tmem();
      const OutPixel pix = out_pixel(p, tc, row);
      const int oh = 2 * p.hs, ow = 2 * p.ws;
      if (pix.ok && p.out_u8 != nullptr) {
        // fused util/util.py:tensor2im (reference lines 33-42): (x + 1) / 2 * 255 in fp32, clip to [0,255], truncate to
        // uint8, CHW -> HWC.  This thread owns output pixels (2y+py, 2x+px): per py, 2 pixels x 3 channels = 6 bytes.
#pragma unroll
        for (int py = 0; py < 2; ++py) {
          uint8_t b[6];
#pragma unroll
          for (int px = 0; px < 2; ++px)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              const int col = (py * 2 + px) * 3 + c;
              const float vf = tanhf(__uint_as_float(v[col]) * s_scale[col] + s_shift[col]);
              float u = __fmul_rn(__fmul_rn(__fadd_rn(vf, 1.0f), 0.5f), 255.0f);
              u = fminf(fmaxf(u, 0.0f), 255.0f);
              b[px * 3 + c] = static_cast<uint8_t>(static_cast<int>(u));
            }
          uint8_t* dst = p.out_u8 + ((static_cast<size_t>(pix.n) * oh + (2 * pix.y + py)) * ow + 2 * pix.x) * 3;
          uint16_t* d16 = reinterpret_cast<uint16_t*>(dst);          // 6-byte aligned: 2x * 3 is even
          d16[0] = static_cast<uint16_t>(b[0] | (b[1] << 8));
          d16[1] = static_cast<uint16_t>(b[2] | (b[3] << 8));
          d16[2] = static_cast<uint16_t>(b[4] | (b[5] << 8));
        }
      } else if (pix.ok) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
#pragma unroll
          for (int py = 0; py < 2; ++py) {
            float2 o;
            o.x = tanhf(__uint_as_float(v[(py * 2 + 0) * 3 + c]) * s_scale[(py * 2 + 0) * 3 + c] + s_shift[(py * 2 + 0) * 3 + c]);
            o.y = tanhf(__uint_as_float(v[(py * 2 + 1) * 3 + c]) * s_scale[(py * 2 + 1) * 3 + c] + s_shift[(py * 2 + 1) * 3 + c]);
            float* dst = p.out_f32 + ((static_cast<size_t>(pix.n) * 3 + c) * oh + (2 * pix.y + py)) * ow + 2 * pix.x;
            *reinterpret_cast<float2*>(dst) = o;
          }
        }
      }
    } else {
      constexpr int kPieces = BN / 32;             // 32-column pieces of the tile; this warp takes grp, grp+kGroups, ...
      if (split_mode) {
        // ---- split-K: this thread's raw fp32 accumulator row.  CSP: into the slot of this CTA's rank in the staging buffer
        // of the CTA that owns the row (distributed shared memory); cluster_split_finish() sums the slots after the cluster
        // barrier.  Otherwise: to partial[t][row][BN] in global memory, summed by splitk_reduce_kernel.
        uint32_t dst_cl = 0;
        float* dst = p.partial + (static_cast<size_t>(t) * kTileM + row) * BN;
        if constexpr (CSP) {
          const int rpo = kTileM / p.n_split;                      // rows per owner
          const uint32_t owner = static_cast<uint32_t>(row / rpo);
          const int lr = row - static_cast<int>(owner) * rpo;
          const uint32_t my_rank = ptx::cluster_ctarank();
          dst_cl = ptx::mapa_u32(ptx::smem_u32(stg_base) + ((my_rank * rpo + lr) * BN) * 4u, owner);
        }
#pragma unroll 1
        for (int c32 = grp; c32 < kPieces; c32 += kGroups) {
          uint32_t v[32];
          ptx::tmem_ld_32x32(t_acc + c32 * 32, v);
          if constexpr (STACK) {
            uint32_t v2[32];
            ptx::tmem_ld_32x32(t_acc + BN + c32 * 32, v2);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(v2[i]));
          }
          ptx::tmem_ld_wait();
          if (c32 + kGroups >= kPieces) release_tmem();
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            if constexpr (CSP)
              ptx::st_cluster_v4(dst_cl + (c32 * 32 + e * 4) * 4u, v[4 * e], v[4 * e + 1], v[4 * e + 2], v[4 * e + 3]);
            else
              *reinterpret_cast<uint4*>(dst + c32 * 32 + e * 4) = make_uint4(v[4 * e], v[4 * e + 1], v[4 * e + 2], v[4 * e + 3]);
          }
        }
      } else {
        // ---- regular: scale/shift (+ residual) + ReLU, 16-bit (hi, lo), written straight to the NHWC output.
        // Each thread owns one pixel row; per 32-column piece it reads its residual (64 B per limb) and writes its output
        // with 256-bit (one 32-byte sector) global accesses.  No smem staging and no TMA store: a TMA store queues behind
        // the producer's outstanding TMA loads in the SM's TMA pipe (measured ~3 us per chunk), and global stores are
        // fire-and-forget.
        const OutPixel pix = out_pixel(p, tc, row);
        __nv_bfloat16* out_row = p.out_ptr + pix.out + tc.nt * BN;
#pragma unroll 1
        for (int c32 = grp; c32 < kPieces; c32 += kGroups) {
          uint32_t vv[32];
          ptx::tmem_ld_32x32(t_acc + c32 * 32, vv);
          if constexpr (STACK) {
            // second half of the stacked accumulator 16 columns at a time (register pressure: 168 per thread at 10 warps;
            // even a force-inlined helper shared with the split-K branch above costs patch<128, NL=2> 20 more spill bytes)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              uint32_t v2[16];
              ptx::tmem_ld_32x16(t_acc + BN + c32 * 32 + hh * 16, v2);
              ptx::tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 16; ++i) vv[hh * 16 + i] = __float_as_uint(__uint_as_float(vv[hh * 16 + i]) + __uint_as_float(v2[i]));
            }
          }
          ptx::tmem_ld_wait();
          if (c32 + kGroups >= kPieces) release_tmem();   // this warp's share of the accumulator is in registers
          // this piece's residual was requested one piece ahead.  A warp with several pieces per tile keeps two register
          // sets (the next request is issued before the math); with one piece per tile the next request - the next TILE's
          // residual, a whole tile period ahead of its use - is issued after the math into the same registers.
          constexpr bool kDoubleRes = (kPieces / kGroups) > 1;
          uint4 rc[NL][4];
          if (use_res) {
#pragma unroll
            for (int l = 0; l < NL; ++l)
#pragma unroll
              for (int e = 0; e < 4; ++e) rc[l][e] = rs[l][e];
            if constexpr (kDoubleRes) {
              if (c32 + kGroups < kPieces) load_res(tc, c32 + kGroups);
              else if (t_next < p.total_tiles) load_res(tc_next, grp);
            }
          }
          uint4 o_prev = make_uint4(0u, 0u, 0u, 0u), ol_prev = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
          for (int piece = 0; piece < 4; ++piece) {          // 16-byte pieces: 8 channels each
            float y[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int ch = c32 * 32 + piece * 8 + e;
              y[e] = fmaf(__uint_as_float(vv[piece * 8 + e]), s_scale[ch], s_shift[ch]);
            }
            uint32_t r[NL][4], hi[4], lo[4];
#pragma unroll
            for (int l = 0; l < NL; ++l) {
              r[l][0] = rc[l][piece].x; r[l][1] = rc[l][piece].y; r[l][2] = rc[l][piece].z; r[l][3] = rc[l][piece].w;
            }
            finish_channels<NL, 8>(y, r, p.has_res, p.relu, hi, lo);
            const uint4 o = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            const uint4 ol = NL == 2 ? make_uint4(lo[0], lo[1], lo[2], lo[3]) : make_uint4(0u, 0u, 0u, 0u);
            if (piece & 1) {               // two 16-byte pieces = one 32-byte sector per store
              if (pix.ok) {
                ptx::stg256(out_row + c32 * 32 + (piece - 1) * 8, o_prev, o);
                if (NL == 2) ptx::stg256(out_row + p.out_limb_stride + c32 * 32 + (piece - 1) * 8, ol_prev, ol);
              }
            } else {
              o_prev = o;
              ol_prev = ol;
            }
          }
          if constexpr (!kDoubleRes) {
            if (use_res && t_next < p.total_tiles) load_res(tc_next, grp);
          }
        }
      }
    }
    if (leader) trace_tile(p, lt, 5);
    if (++acc == NACC) { acc = 0; acc_phase ^= 1; }
  }
}

// Cluster split-K, second half (after the cluster barrier): the epilogue warps of every CTA sum the n_split partial slots of
// the 128 / n_split tile rows this CTA owns (in split order: deterministic) and finish them (finish4), writing the NHWC output
// directly.  One thread = one pixel x 4 channels per trip.
template <int BN, int NL, int EW>
__device__ __forceinline__ void cluster_split_finish(const ConvParams& p, const uint8_t* stg_base, int t) {
  constexpr int kEpi = EW * 32;
  const int etid = threadIdx.x - 64;
  const TileCoord tc = decode_tile(p, t);
  const int cs = p.n_split, rpo = kTileM / cs;
  const int rank = static_cast<int>(ptx::cluster_ctarank());
  const float* stg = reinterpret_cast<const float*>(stg_base);
  constexpr int kGroups4 = BN / 4;
  for (int e = etid; e < rpo * kGroups4; e += kEpi) {
    const int g = e % kGroups4, lr = e / kGroups4;
    const OutPixel pix = out_pixel(p, tc, rank * rpo + lr);
    if (!pix.ok) continue;
    float4 acc = *reinterpret_cast<const float4*>(stg + (static_cast<size_t>(lr) * BN + g * 4));
    for (int sp = 1; sp < cs; ++sp) {
      const float4 a = *reinterpret_cast<const float4*>(stg + (static_cast<size_t>(sp * rpo + lr) * BN + g * 4));
      acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
    }
    finish4<NL>(p, pix, tc.nt * BN + g * 4, acc);
  }
}

// Tile walk of a CTA: persistent (blockIdx.x, +gridDim.x, ...) or, in a cluster split-K launch, exactly one tile whose
// split index is the CTA's rank in its cluster (grid = tiles x n_split, clusters of n_split consecutive CTAs).
template <bool CSP>
__device__ __forceinline__ void tile_walk(const ConvParams& p, int& t0, int& tstep) {
  if constexpr (CSP) {
    const int cs = p.n_split;
    const int tile = static_cast<int>(blockIdx.x) / cs, split = static_cast<int>(blockIdx.x) - tile * cs;
    t0 = split * p.tiles_per_split + tile;
    tstep = p.total_tiles;                  // one tile per CTA
  } else {
    t0 = static_cast<int>(blockIdx.x);
    tstep = static_cast<int>(gridDim.x);
  }
}

template <int BN, int NL, bool TAIL, bool CSP = false>
__global__ void __launch_bounds__(kThreads, 1) conv_umma_kernel(const __grid_constant__ ConvParams p) {
  using Cfg = ConvCfg<BN, NL, TAIL, CSP>;
  static_assert(!(CSP && TAIL), "the tail conv never splits K");
  int t0, tstep;
  tile_walk<CSP>(p, t0, tstep);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stg_base = smem + Cfg::kStages * Cfg::kStage;
  uint8_t* aux = stg_base + Cfg::kStgBytes;
  float* s_scale = reinterpret_cast<float*>(aux);
  uint64_t* bars = reinterpret_cast<uint64_t*>(aux + 4 * BN * 4);
  uint64_t* full_bar = bars;                       // [kStages]
  uint64_t* empty_bar = bars + Cfg::kStages;       // [kStages]
  uint64_t* tfull_bar = bars + 2 * Cfg::kStages;   // [2]
  uint64_t* tempty_bar = tfull_bar + 2;            // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // provably warp-uniform
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) ptx::prefetch_tmap(&p.a[i]);
    ptx::prefetch_tmap(&p.w);
    for (int i = 0; i < Cfg::kStages; ++i) {
      ptx::mbar_init(&full_bar[i], 1);
      ptx::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tfull_bar[i], 1);
      ptx::mbar_init(&tempty_bar[i], 4);   // one arrive per epilogue warp
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (CSP) ptx::cluster_sync();   // every CTA of the cluster is running before anyone writes into its shared memory
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  ptx::pdl_launch_dependents();   // the next kernel may start its prologue; it waits (pdl_wait) before touching our output

  int kb_per_tap = 0;
  for (int s = 0; s < p.n_src; ++s) kb_per_tap += p.chunks[s];
  const int num_kb = p.n_taps * kb_per_tap;

  if (warp == 0) {
    // ===================================================================== TMA producer
    // Weights are never written by a kernel, so the weight tiles of this CTA's first K blocks (a whole ring of them) are
    // requested BEFORE the programmatic-dependency wait: they stream from HBM/L2 while the previous layer is still
    // finishing.  At batch 1 the layers below 16x16 are one tile of 4-9 K blocks per CTA - their whole weight share.
    int pre = 0;
    if (t0 < p.total_tiles) {
      const TileCoord tc = decode_tile(p, t0);
      const int kb0 = tc.split * p.split_len;
      const int kb1 = (kb0 + p.split_len < num_kb) ? kb0 + p.split_len : num_kb;
      pre = (kb1 - kb0 < Cfg::kStages) ? kb1 - kb0 : Cfg::kStages;
      if (ptx::elect_one()) {
        for (int i = 0; i < pre; ++i) {          // first use of stages 0..pre-1: no empty-barrier wait needed
          uint8_t* st = smem + i * Cfg::kStage;
          ptx::mbar_expect_tx(&full_bar[i], Cfg::kStage);
#pragma unroll
          for (int l = 0; l < NL; ++l)
            ptx::tma_load_3d(&p.w, &full_bar[i], st + NL * kATile + l * Cfg::kBTile, (kb0 + i) * kChunk, tc.nt * BN,
                             l * p.n_phases + tc.z);
        }
      }
      __syncwarp();
    }
    ptx::pdl_wait();                // activations are written by the previous kernel
    int stage = 0;
    uint32_t phase = 0;
    int issued = 0;                 // K blocks issued so far by this CTA (the first `pre` already have their weight tiles)
    for (int t = t0; t < p.total_tiles; t += tstep) {
      const TileCoord tc = decode_tile(p, t);
      const int kb0 = tc.split * p.split_len;
      const int kb1 = (kb0 + p.split_len < num_kb) ? kb0 + p.split_len : num_kb;
      for (int kb = kb0; kb < kb1; ++kb, ++issued) {
        const int tap = kb / kb_per_tap;
        const int rem = kb - tap * kb_per_tap;
        const int s = (rem < p.chunks[0]) ? 0 : 1;
        const int c = s ? rem - p.chunks[0] : rem;
        const int amap = p.tap_map[tc.z][tap];
        const int xx = tc.x0 + p.tap_dx[tc.z][tap];
        const int yy = tc.y0 + p.tap_dy[tc.z][tap];
        const bool early = issued < pre;
        if (!early) ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
        if (ptx::elect_one()) {
          uint8_t* st = smem + stage * Cfg::kStage;
          if (!early) ptx::mbar_expect_tx(&full_bar[stage], Cfg::kStage);
#pragma unroll
          for (int l = 0; l < NL; ++l) {
            ptx::tma_load_5d(&p.a[amap + s], &full_bar[stage], st + l * kATile, c * kChunk, xx, yy, tc.n0, l);
            if (!early)
              ptx::tma_load_3d(&p.w, &full_bar[stage], st + NL * kATile + l * Cfg::kBTile, kb * kChunk, tc.nt * BN,
                               l * p.n_phases + tc.z);
          }
        }
        __syncwarp();
        if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = t0; t < p.total_tiles; t += tstep) {
      ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BN;
      const TileCoord tc = decode_tile(p, t);
      const int kb0 = tc.split * p.split_len;
      const int kb1 = (kb0 + p.split_len < num_kb) ? kb0 + p.split_len : num_kb;
      for (int kb = kb0; kb < kb1; ++kb) {
        ptx::mbar_wait(&full_bar[stage], phase);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          const uint32_t a0 = ptx::smem_u32(smem + stage * Cfg::kStage);
          const uint32_t b0 = a0 + NL * kATile;
          const uint64_t a_hi = ptx::umma_desc_sw128(a0);
          const uint64_t b_hi = ptx::umma_desc_sw128(b0);
#pragma unroll
          for (int k = 0; k < kChunk / 16; ++k) {
            const uint32_t accum = (kb > kb0 || k > 0) ? 1u : 0u;
            // +32 bytes along K inside the 128-byte swizzle row = +2 in descriptor address units
            ptx::umma_f16(d_tmem, a_hi + 2 * k, b_hi + 2 * k, p.idesc, accum);
            if (NL == 2) {
              const uint64_t a_lo = ptx::umma_desc_sw128(a0 + kATile);
              const uint64_t b_lo = ptx::umma_desc_sw128(b0 + Cfg::kBTile);
              ptx::umma_f16(d_tmem, a_hi + 2 * k, b_lo + 2 * k, p.idesc, 1u);
              ptx::umma_f16(d_tmem, a_lo + 2 * k, b_hi + 2 * k, p.idesc, 1u);
            }
          }
          ptx::umma_commit(&empty_bar[stage]);                 // smem slot reusable once these MMAs retire
          if (kb == kb1 - 1) ptx::umma_commit(&tfull_bar[acc]);   // accumulator complete
        }
        __syncwarp();
        if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else {
    epilogue_warps<BN, NL, TAIL, false, false, 4, 2, CSP>(p, stg_base, s_scale, tfull_bar, tempty_bar, tmem_base, warp, lane,
                                                           t0, tstep);
  }
  if constexpr (CSP) {
    // every CTA of the cluster has written its partial rows into the owners' staging buffers
    ptx::cluster_sync();
    if (warp >= 2) cluster_split_finish<BN, NL, 4>(p, stg_base, t0);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}


// ====================================================================================================
// Patch mode.  The v1 kernel above re-loads a 16 KB A tile for every tap, i.e. reads the layer input 9x from
// L2; ncu shows it pinned at the ~10.6 TB/s L2->SM limit with the tensor pipe 35-65 % busy
// (profiles/r01_v1_ncu_full_first14_convs.md).  Here ONE halo patch {64 ch, TW+halo, TH+halo} is loaded per
// (tile, source, 64-channel chunk) and all taps are addressed inside it: with TW = 8 an 8-row UMMA group is
// one image row of the patch, so the shifted A tile of tap (dx,dy) is the same swizzled buffer described by
//   start = patch + ((dy-dy0)*PW + (dx-dx0)) * 128 B,   stride between 8-row groups (SBO) = PW * 128 B.
// The swizzle phase of a row is a function of its absolute smem address for both TMA and UMMA, so rows that
// TMA wrote are read back consistently at any 128-byte-aligned start with a descriptor base offset of 0 (measured on
// B200: setting it to (start>>7)&7 corrupts the result).
// A and B move through separate mbarrier rings: an A patch is consumed by n_taps B tiles.
// ====================================================================================================
constexpr int kPatchSlot = 23 * 1024;           // >= 10*18*128 = 23040 bytes
constexpr int kPatchStride = 23 * 1024;         // distance between patch buffers (1024-byte aligned)

// Taps per B stage of conv_patch_kernel (build_plan encodes the FAST single-CTA weight view with boxes of this many taps):
// one mbarrier round trip per stage costs the MMA-issuing thread a few hundred cycles, so a stage must carry enough tensor
// work (>= ~500 cycles): 2 taps for N=128 bf16, 2-3 for N=64, all 9 for the tail.
constexpr int patch_taps_per_stage(int bn, int nl, bool tail) {
  return tail ? 9 : (bn >= 128 ? (nl == 1 ? 2 : 1) : (nl == 1 ? 3 : 2));
}

template <int BN, int NL, bool TAIL, bool CSP = false>
struct PatchCfg {
  static constexpr int kBTile = BN * 128;
  static constexpr int kTPS = patch_taps_per_stage(BN, NL, TAIL);
  static constexpr int kAStage = NL * kPatchStride;
  static constexpr int kBStage = NL * kTPS * kBTile;
  // In-kernel clock64 traces (tests/gpu_trace.py) showed the MMA warp stalling ~350 cycles per B stage: a stage is
  // refilled only after the MMAs that read it retire, and the refill (barrier -> TMA issue -> L2 -> smem) takes
  // ~2.3-2.7k cycles, so the B ring must hold more than that much tensor work.  Two A patches are enough (the next
  // one is requested a full chunk ahead); everything else goes to B stages.
  static constexpr int kAStages = 2;
  static constexpr int kStgBytes = CSP ? kTileM * BN * 4 : 0;        // cluster split-K staging (see ConvCfg)
  static constexpr int kAux = 3072;
  static constexpr int kAvail = kSmemBudget - 1024 - kStgBytes - kAux - kAStages * kAStage;
  static constexpr int kBStagesRaw = kAvail / kBStage;
  static constexpr int kBStages = kBStagesRaw > 12 ? 12 : kBStagesRaw;
  static constexpr int kSmemBytes = 1024 + kAStages * kAStage + kBStages * kBStage + kStgBytes + kAux;
  static constexpr int kAccCols = (NL == 2) ? 2 * BN : BN;                   // parity: stacked [hi*hi+lo*hi | hi*lo] accumulator
  static constexpr int kTmemCols = (2 * kAccCols < 32) ? 32 : 2 * kAccCols;
  static_assert(kTmemCols <= 512, "TMEM has 512 columns");
  static_assert(kBStages >= 2, "B ring needs at least two stages");
  static_assert(4 * BN * 4 + (2 * kBStages + 2 * kAStages + 2 * 2 + 1) * 8 <= kAux, "aux region too small");
};

__device__ __forceinline__ uint64_t umma_desc_sw128_strided(uint32_t smem_addr, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(sbo_bytes >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// CL = cluster size (1 or 2).  With CL = 2 the two CTAs of a cluster work on neighbouring M tiles of the same N tile and
// phase, so they consume identical B stages: each CTA fetches half the rows of every weight tile and multicasts them
// to both (cp.async.bulk.tensor ... .multicast::cluster), halving the L2->SM weight traffic that clock64 traces showed
// to be the limiter (~30-36 B/clk/SM of weight tiles, every SM asking L2 for the same lines).  A stage is refilled
// only after BOTH CTAs' MMAs released it (tcgen05.commit ... .multicast::cluster onto both bempty barriers).
template <int BN, int NL, bool TAIL, int CL, int EW, bool CSP = false>
__global__ void __launch_bounds__(64 + EW * 32, 1) conv_patch_kernel(const __grid_constant__ ConvParams p) {
  using Cfg = PatchCfg<BN, NL, TAIL, CSP>;
  static_assert(!(CSP && (TAIL || CL != 1)), "cluster split-K: no tail, no B multicast cluster");
  int t0, tstep;
  tile_walk<CSP>(p, t0, tstep);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_ring = smem;
  uint8_t* b_ring = a_ring + Cfg::kAStages * Cfg::kAStage;
  uint8_t* stg_base = b_ring + Cfg::kBStages * Cfg::kBStage;
  uint8_t* aux = stg_base + Cfg::kStgBytes;
  float* s_scale = reinterpret_cast<float*>(aux);
  uint64_t* bars = reinterpret_cast<uint64_t*>(aux + 4 * BN * 4);
  uint64_t* afull_bar = bars;                               // [kAStages]
  uint64_t* aempty_bar = afull_bar + Cfg::kAStages;         // [kAStages]
  uint64_t* bfull_bar = aempty_bar + Cfg::kAStages;         // [kBStages]
  uint64_t* bempty_bar = bfull_bar + Cfg::kBStages;         // [kBStages]
  uint64_t* tfull_bar = bempty_bar + Cfg::kBStages;         // [2]
  uint64_t* tempty_bar = tfull_bar + 2;                     // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // provably warp-uniform
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) trace_stamp(p, 0);

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) ptx::prefetch_tmap(&p.a[i]);
    ptx::prefetch_tmap(&p.w);
    for (int i = 0; i < Cfg::kAStages; ++i) { ptx::mbar_init(&afull_bar[i], 1); ptx::mbar_init(&aempty_bar[i], 1); }
    for (int i = 0; i < Cfg::kBStages; ++i) { ptx::mbar_init(&bfull_bar[i], 1); ptx::mbar_init(&bempty_bar[i], CL); }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tfull_bar[i], 1);
      ptx::mbar_init(&tempty_bar[i], EW);   // one arrive per epilogue warp
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (CL > 1 || CSP) ptx::cluster_sync();     // peers' barriers are initialised / peers are running before remote smem is touched
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t crank = (CL > 1) ? ptx::cluster_ctarank() : 0u;
  constexpr uint16_t kMask = static_cast<uint16_t>((1u << CL) - 1u);
  ptx::pdl_launch_dependents();   // the next kernel may start its prologue; it waits (pdl_wait) before touching our output
  if (threadIdx.x == 0) trace_stamp(p, 1);

  int kb_per_tap = 0;
  for (int s = 0; s < p.n_src; ++s) kb_per_tap += p.chunks[s];   // = (source, chunk) items per tile
  const int patch_bytes = p.patch_w * p.patch_h * 128;

  if (warp == 0) {
    // ===================================================================== TMA producer
    // Flat sequence of items (tile, concat-chunk ci).  The A patch of item j+1 is issued in the middle of item
    // j's B tiles so that it is in flight while the MMA warp still works on item j.
    ptx::pdl_wait();                // activations are written by the previous kernel
    int ia = 0, ib = 0;
    uint32_t pha = 0, phb = 0;
    int a_tile = t0, a_ci = -1;            // cursor of the next A patch to issue (-1: take the tile's first item)
    auto issue_a = [&]() {
      if (a_tile >= p.total_tiles) return;
      const TileCoord tc = decode_tile(p, a_tile);
      const int ci0 = tc.split * p.split_len;
      const int ci1 = (ci0 + p.split_len < kb_per_tap) ? ci0 + p.split_len : kb_per_tap;
      if (a_ci < 0) a_ci = ci0;
      const int s = (a_ci < p.chunks[0]) ? 0 : 1;
      const int c = (s == 0) ? a_ci : a_ci - p.chunks[0];
      ptx::mbar_wait(&aempty_bar[ia], pha ^ 1);
      if (ptx::elect_one()) {
        ptx::mbar_expect_tx(&afull_bar[ia], NL * patch_bytes);
#pragma unroll
        for (int l = 0; l < NL; ++l)
          ptx::tma_load_5d(&p.a[s], &afull_bar[ia], a_ring + ia * Cfg::kAStage + l * kPatchStride, c * kChunk,
                           tc.x0 + p.patch_dx0[tc.z], tc.y0 + p.patch_dy0[tc.z], tc.n0, l);
      }
      __syncwarp();
      if (++ia == Cfg::kAStages) { ia = 0; pha ^= 1; }
      if (++a_ci == ci1) { a_ci = -1; a_tile += tstep; }
    };
    issue_a();
    const int n_groups = (p.n_taps + Cfg::kTPS - 1) / Cfg::kTPS;
    const int a_after_group = (n_groups > 1) ? 1 : 0;
    int lt = 0;
    for (int t = t0; t < p.total_tiles; t += tstep, ++lt) {
      const TileCoord tc = decode_tile(p, t);
      const int ci0 = tc.split * p.split_len;
      const int ci1 = (ci0 + p.split_len < kb_per_tap) ? ci0 + p.split_len : kb_per_tap;
      if (lane == 0) trace_tile(p, lt, 6);
      for (int ci = ci0; ci < ci1; ++ci) {
        for (int g = 0; g < n_groups; ++g) {
          ptx::mbar_wait(&bempty_bar[ib], phb ^ 1);
          if (ptx::elect_one()) {
            uint8_t* st = b_ring + ib * Cfg::kBStage;
            if constexpr (CL == 1 && NL == 1) {
              ptx::mbar_expect_tx(&bfull_bar[ib], Cfg::kBStage);
              // one box = kTPS taps x BN rows x 64 channels (taps beyond n_taps are zero-filled)
              ptx::tma_load_4d(&p.w, &bfull_bar[ib], st, ci * kChunk, tc.nt * BN, g * Cfg::kTPS, tc.z);
            } else {
              // per-tap boxes of BN/CL rows.  Stage layout [tap][limb][BN rows]: B_lo follows B_hi so that one N=2*BN
              // descriptor covers the stacked pair.  With CL = 2 this CTA fetches rows [crank*BN/CL, +BN/CL) of every
              // tile and multicasts them to the whole cluster.
              const int tap0 = g * Cfg::kTPS;
              const int ntap = (tap0 + Cfg::kTPS < p.n_taps) ? Cfg::kTPS : p.n_taps - tap0;
              ptx::mbar_expect_tx(&bfull_bar[ib], NL * ntap * Cfg::kBTile);
              constexpr int kRows = BN / CL;
              for (int ti = 0; ti < ntap; ++ti)
#pragma unroll
                for (int l = 0; l < NL; ++l) {
                  uint8_t* dst = st + (ti * NL + l) * Cfg::kBTile + crank * kRows * 128;
                  if constexpr (CL == 1)
                    ptx::tma_load_4d(&p.w, &bfull_bar[ib], dst, ci * kChunk, tc.nt * BN, tap0 + ti, l * p.n_phases + tc.z);
                  else
                    ptx::tma_load_4d_mc(&p.w, &bfull_bar[ib], dst, ci * kChunk, tc.nt * BN + crank * kRows, tap0 + ti,
                                        l * p.n_phases + tc.z, kMask);
                }
            }
          }
          __syncwarp();
          if (++ib == Cfg::kBStages) { ib = 0; phb ^= 1; }
          if (g == a_after_group) issue_a();
        }
      }
      if (lane == 0) trace_tile(p, lt, 7);
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    int ia = 0, ib = 0;
    uint32_t pha = 0, phb = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    const uint32_t sbo = static_cast<uint32_t>(p.patch_w) * 128u;
    const int n_groups = (p.n_taps + Cfg::kTPS - 1) / Cfg::kTPS;
    bool b_ready = false;
    int lt = 0;
    for (int t = t0; t < p.total_tiles; t += tstep, ++lt) {
      TileCoord tc;
      decode_tile_zs(p, t, tc.z, tc.split);
      ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      ptx::tc_fence_after();
      if (lane == 0) trace_tile(p, lt, 0);
      const uint32_t d_tmem = tmem_base + acc * Cfg::kAccCols;
      const int ci0 = tc.split * p.split_len;
      const int ci1 = (ci0 + p.split_len < kb_per_tap) ? ci0 + p.split_len : kb_per_tap;
      for (int ci = ci0; ci < ci1; ++ci) {
        ptx::mbar_wait(&afull_bar[ia], pha);
        const uint32_t a0 = ptx::smem_u32(a_ring + ia * Cfg::kAStage);
        for (int g = 0; g < n_groups; ++g) {
          if (!b_ready) ptx::mbar_wait(&bfull_bar[ib], phb);
          ptx::tc_fence_after();
          if (lane == 0 && ci == ci0 && g == 0) trace_tile(p, lt, 1);
          const int tap0 = g * Cfg::kTPS;
          const int tap1 = (tap0 + Cfg::kTPS < p.n_taps) ? tap0 + Cfg::kTPS : p.n_taps;
          if (ptx::elect_one()) {
            const uint32_t b0 = ptx::smem_u32(b_ring + ib * Cfg::kBStage);
            for (int tap = tap0; tap < tap1; ++tap) {
              const uint32_t a_hi_addr = a0 + static_cast<uint32_t>(p.tap_row[tc.z][tap]) * 128u;
              const uint32_t b_hi_addr = b0 + static_cast<uint32_t>(tap - tap0) * (NL * Cfg::kBTile);
              const uint64_t a_hi = umma_desc_sw128_strided(a_hi_addr, sbo);
              const uint64_t b_hi = ptx::umma_desc_sw128(b_hi_addr);
#pragma unroll
              for (int k = 0; k < kChunk / 16; ++k) {
                const uint32_t accum = (ci > ci0 || tap > 0 || k > 0) ? 1u : 0u;
                if constexpr (NL == 1) {
                  ptx::umma_f16(d_tmem, a_hi + 2 * k, b_hi + 2 * k, p.idesc, accum);
                } else {
                  // [hi*hi | hi*lo] in one N=2*BN MMA (B_lo is stored right behind B_hi), then lo*hi into the first half
                  const uint64_t a_lo = umma_desc_sw128_strided(a_hi_addr + kPatchStride, sbo);
                  ptx::umma_f16(d_tmem, a_hi + 2 * k, b_hi + 2 * k, p.idesc2, accum);
                  ptx::umma_f16(d_tmem, a_lo + 2 * k, b_hi + 2 * k, p.idesc, 1u);
                }
              }
            }
            if constexpr (CL == 1) ptx::umma_commit(&bempty_bar[ib]);
            else ptx::umma_commit_mc(&bempty_bar[ib], kMask);     // the stage is shared: release it in every CTA
            if (g == n_groups - 1) {
              ptx::umma_commit(&aempty_bar[ia]);
              if (ci == ci1 - 1) ptx::umma_commit(&tfull_bar[acc]);
            }
          }
          __syncwarp();
          if (++ib == Cfg::kBStages) { ib = 0; phb ^= 1; }
          b_ready = ptx::mbar_try_wait(&bfull_bar[ib], phb);   // peek: overlaps the barrier round trip with the MMAs in flight
        }
        if (++ia == Cfg::kAStages) { ia = 0; pha ^= 1; }
      }
      if (lane == 0) trace_tile(p, lt, 2);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else {
    epilogue_warps<BN, NL, TAIL, (NL == 2), false, EW, 2, CSP>(p, stg_base, s_scale, tfull_bar, tempty_bar, tmem_base, warp, lane,
                                                                t0, tstep);
  }
  if constexpr (CSP) {
    ptx::cluster_sync();                 // every CTA's partial rows are in their owners' staging buffers
    if (warp >= 2) cluster_split_finish<BN, NL, EW>(p, stg_base, t0);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (CL > 1) ptx::cluster_sync();     // no CTA leaves while a peer may still signal its barriers / write its smem
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}


// ====================================================================================================
// CTA-pair variant (cta_group::2) of the patch kernel for the wide layers (N tile 128 or 256).
// The two CTAs of a cluster own neighbouring M tiles of the same N tile.  One tcgen05.mma.cta_group::2 (M = 256,
// issued by the leader only) multiplies both CTAs' A patches with a B tile of which each CTA stores - and fetches -
// only half the rows; each CTA's 128 accumulator lanes live in its own TMEM and are drained by its own epilogue warps.
// Per SM this halves the B operand reads and the B fill traffic of shared memory, which is what bounds the
// single-CTA kernel (DESIGN.md section 5.1), halves the L2->SM weight traffic and doubles the ring depth per byte.
// PARITY (NL = 2) issues hi*hi, hi*lo, lo*hi as three N = BN MMAs (B_hi and B_lo are each split across the pair).
// ====================================================================================================
// STK (parity, N tile 64): the stage of CTA r holds X = limb r of the whole 64-row tile (so that the pair's X tiles form the
// stacked [B_hi; B_lo] operand of one N = 128 MMA: A_hi*B_hi | A_hi*B_lo) and Y = rows [32r, 32r+32) of B_hi (the pair's
// Y tiles form B_hi for the N = 64 MMA A_lo*B_hi).  Two MMAs instead of three per K step and 11 KB instead of 15 KB of
// operand reads per SM: the N = 64 layers are bound by shared-memory bandwidth (A is re-read for every 64 columns).
constexpr bool pair_stacked(int bn, int nl) { return bn == 64 && nl == 2; }

// Shared memory of the pair kernel: two A patches, the aux region and a B ring of one tap per stage (this CTA's half of the
// B tile of every limb; three halves when stacked) that takes the rest, at most 16 stages.  build_plan keeps a layer's
// weights resident when all of its weight tiles fit that ring.
constexpr int kPairAStages = 2;
constexpr int kPairAux = 5120;
constexpr int pair_b_stage_bytes(int bn, int nl) { return (pair_stacked(bn, nl) ? 3 : nl) * (bn / 2) * 128; }
constexpr int pair_b_stages(int bn, int nl) {
  const int n = (kSmemBudget - 1024 - kPairAux - kPairAStages * nl * kPatchStride) / pair_b_stage_bytes(bn, nl);
  return n > 16 ? 16 : n;
}

template <int BN, int NL, bool STK>
struct PairCfg {
  static_assert(STK == pair_stacked(BN, NL), "stacked operands exactly in parity mode with N tile 64");
  static constexpr int kBHalf = (BN / 2) * 128;                   // bytes of this CTA's half of one B tile
  static constexpr int kAStage = NL * kPatchStride;
  static constexpr int kBStage = pair_b_stage_bytes(BN, NL);
  static constexpr int kAccCols = STK ? 2 * BN : BN;
  static constexpr int kAStages = kPairAStages;
  static constexpr int kAux = kPairAux;
  static constexpr int kBStages = pair_b_stages(BN, NL);
  static constexpr int kSmemBytes = 1024 + kAStages * kAStage + kBStages * kBStage + kAux;
  // TMEM accumulator ring: as many buffers as the 512 columns hold (4 for N tiles up to 128 columns wide, 2 for 256).
  // With two buffers the MMA warp idled ~15 % of a 64-channel tile waiting for the epilogue to hand one back (clock64
  // traces); a deeper ring absorbs the epilogue's latency jitter.
  static constexpr int kAccBufs = (4 * kAccCols <= 512) ? 4 : 2;
  static constexpr int kTmemCols = kAccBufs * kAccCols;
  static_assert(BN == 64 || BN == 128 || BN == 256, "pair kernel: N tile 64, 128 or 256");
  static_assert(kTmemCols <= 512, "TMEM has 512 columns");
  static_assert(kBStages >= 3, "B ring too shallow");
  static_assert(4 * BN * 4 + (2 * kBStages + 2 * kAStages + 2 * kAccBufs + 1) * 8 <= kAux, "aux region too small");
};

template <int BN, int NL, int EW, bool STK>
__global__ void __launch_bounds__(64 + EW * 32, 1) conv_pair_kernel(const __grid_constant__ ConvParams p) {
  using Cfg = PairCfg<BN, NL, STK>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_ring = smem;
  uint8_t* b_ring = a_ring + Cfg::kAStages * Cfg::kAStage;
  uint8_t* aux = b_ring + Cfg::kBStages * Cfg::kBStage;
  float* s_scale = reinterpret_cast<float*>(aux);
  uint64_t* bars = reinterpret_cast<uint64_t*>(aux + 4 * BN * 4);
  uint64_t* afull_bar = bars;                               // [kAStages]  (used in the leader)
  uint64_t* aempty_bar = afull_bar + Cfg::kAStages;         // [kAStages]
  uint64_t* bfull_bar = aempty_bar + Cfg::kAStages;         // [kBStages]  (used in the leader)
  uint64_t* bempty_bar = bfull_bar + Cfg::kBStages;         // [kBStages]
  constexpr int NACC = Cfg::kAccBufs;
  uint64_t* tfull_bar = bempty_bar + Cfg::kBStages;         // [NACC]
  uint64_t* tempty_bar = tfull_bar + NACC;                  // [NACC]     (used in the leader: 2*EW arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + NACC);

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const uint32_t crank = ptx::cluster_ctarank();
  const bool leader_cta = (crank == 0);
  if (threadIdx.x == 0) { trace_stamp(p, 0); trace_time(p, false); }

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) ptx::prefetch_tmap(&p.a[i]);
    ptx::prefetch_tmap(&p.w);
    for (int i = 0; i < Cfg::kAStages; ++i) { ptx::mbar_init(&afull_bar[i], 1); ptx::mbar_init(&aempty_bar[i], 1); }
    for (int i = 0; i < Cfg::kBStages; ++i) { ptx::mbar_init(&bfull_bar[i], 1); ptx::mbar_init(&bempty_bar[i], 1); }
    for (int i = 0; i < NACC; ++i) {
      ptx::mbar_init(&tfull_bar[i], 1);
      ptx::mbar_init(&tempty_bar[i], 2 * EW);  // the epilogue warps of both CTAs of the pair
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc_pair(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish_pair();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  ptx::pdl_launch_dependents();
  if (threadIdx.x == 0) trace_stamp(p, 1);

  int kb_per_tap = 0;
  for (int s = 0; s < p.n_src; ++s) kb_per_tap += p.chunks[s];
  const int patch_bytes = p.patch_w * p.patch_h * 128;
  constexpr uint16_t kMask = 0x3;

  if (warp == 0) {
    // ===================================================================== TMA producer (both CTAs)
    // (the dependency wait comes after the first weight requests: weights are never written by a kernel)
    int ia = 0, ib = 0;
    uint32_t pha = 0, phb = 0;
    int a_tile = blockIdx.x, a_ci = 0, a_lt = 0;
    auto issue_a = [&]() {
      if (a_tile >= p.total_tiles) return;
      const TileCoord tc = decode_tile(p, a_tile);
      const int s = (a_ci < p.chunks[0]) ? 0 : 1;
      const int c = (s == 0) ? a_ci : a_ci - p.chunks[0];
      ptx::mbar_wait(&aempty_bar[ia], pha ^ 1);
      if (lane == 0 && a_ci == 0) trace_tile(p, a_lt, 6);
      if (ptx::elect_one()) {
        if (leader_cta) ptx::mbar_expect_tx(&afull_bar[ia], 2 * NL * patch_bytes);     // both CTAs' patches
#pragma unroll
        for (int l = 0; l < NL; ++l)
          ptx::tma_load_5d_pair(&p.a[s], &afull_bar[ia], a_ring + ia * Cfg::kAStage + l * kPatchStride, c * kChunk,
                                tc.x0 + p.patch_dx0[tc.z], tc.y0 + p.patch_dy0[tc.z], tc.n0, l);
      }
      __syncwarp();
      if (++ia == Cfg::kAStages) { ia = 0; pha ^= 1; }
      if (++a_ci == kb_per_tap) {
        if (lane == 0) trace_tile(p, a_lt, 7);
        a_ci = 0; a_tile += gridDim.x; ++a_lt;
      }
    };
    // this CTA's share of one weight tile (K chunk ci, tap, phase z, N tile nt) -> dst, completing on the leader's `bar`
    auto load_b = [&](uint8_t* dst, uint64_t* bar, int ci, int nt, int tap, int z) {
      if constexpr (STK) {
#pragma unroll
        for (int h = 0; h < 2; ++h)      // X: limb `crank` of the whole tile, as two boxes of BN/2 rows
          ptx::tma_load_4d_pair(&p.w, bar, dst + h * Cfg::kBHalf, ci * kChunk, nt * BN + h * (BN / 2), tap,
                                static_cast<int>(crank) * p.n_phases + z);
        ptx::tma_load_4d_pair(&p.w, bar, dst + 2 * Cfg::kBHalf, ci * kChunk, nt * BN + static_cast<int>(crank) * (BN / 2), tap, z);
      } else {
#pragma unroll
        for (int l = 0; l < NL; ++l)     // rows [crank*BN/2, +BN/2) of every limb
          ptx::tma_load_4d_pair(&p.w, bar, dst + l * Cfg::kBHalf, ci * kChunk, nt * BN + static_cast<int>(crank) * (BN / 2), tap,
                                l * p.n_phases + z);
      }
    };
    if (p.b_resident) {
      // all weight tiles of the layer (this CTA's half of each) are loaded once; one barrier covers them
      if (blockIdx.x < p.total_tiles) {
        const TileCoord tc = decode_tile(p, blockIdx.x);      // nt and phase are the same for every tile of a resident layer
        if (ptx::elect_one()) {
          const int n_items = kb_per_tap * p.n_taps;
          if (leader_cta) ptx::mbar_expect_tx(&bfull_bar[0], 2 * n_items * Cfg::kBStage);
          for (int ci = 0; ci < kb_per_tap; ++ci)
            for (int tap = 0; tap < p.n_taps; ++tap)
              load_b(b_ring + (ci * p.n_taps + tap) * Cfg::kBStage, &bfull_bar[0], ci, tc.nt, tap, tc.z);
        }
        __syncwarp();
      }
    }
    // streaming layers: the first ring of weight tiles (first use of every stage: no empty-barrier wait) goes out early too
    int pre = 0, b_items = 0;
    if (!p.b_resident && static_cast<int>(blockIdx.x) < p.total_tiles) {
      const TileCoord tc = decode_tile(p, blockIdx.x);
      const int n_items = kb_per_tap * p.n_taps;
      pre = n_items < Cfg::kBStages ? n_items : Cfg::kBStages;
      if (ptx::elect_one()) {
        for (int i = 0; i < pre; ++i) {
          const int ci = i / p.n_taps, tap = i - ci * p.n_taps;
          if (leader_cta) ptx::mbar_expect_tx(&bfull_bar[i], 2 * Cfg::kBStage);
          load_b(b_ring + i * Cfg::kBStage, &bfull_bar[i], ci, tc.nt, tap, tc.z);
        }
      }
      __syncwarp();
    }
    ptx::pdl_wait();                // activations are written by the previous kernel
    issue_a();
    const int a_after = (p.n_taps > 2) ? 2 : p.n_taps - 1;
    for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
      const TileCoord tc = decode_tile(p, t);
      for (int ci = 0; ci < kb_per_tap; ++ci) {
        for (int tap = 0; tap < p.n_taps; ++tap) {
          if (p.b_resident) {
            if (tap == a_after) issue_a();
            continue;
          }
          const bool early = b_items < pre;
          ++b_items;
          if (!early) {
            ptx::mbar_wait(&bempty_bar[ib], phb ^ 1);
            if (ptx::elect_one()) {
              uint8_t* st = b_ring + ib * Cfg::kBStage;
              if (leader_cta) ptx::mbar_expect_tx(&bfull_bar[ib], 2 * Cfg::kBStage);    // both CTAs' shares
              load_b(st, &bfull_bar[ib], ci, tc.nt, tap, tc.z);
            }
          }
          __syncwarp();
          if (++ib == Cfg::kBStages) { ib = 0; phb ^= 1; }
          if (tap == a_after) issue_a();
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer (leader CTA only)
    if (leader_cta) {
      int ia = 0, ib = 0;
      uint32_t pha = 0, phb = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const uint32_t sbo = static_cast<uint32_t>(p.patch_w) * 128u;
      bool b_ready = false;
      const bool resident = p.b_resident != 0;
      if (resident && blockIdx.x < p.total_tiles) { ptx::mbar_wait(&bfull_bar[0], 0); b_ready = true; }
      int lt = 0;
      for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x, ++lt) {
        int z, split;
        decode_tile_zs(p, t, z, split);
        ptx::mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        if (lane == 0) trace_tile(p, lt, 0);
        const uint32_t d_tmem = tmem_base + acc * Cfg::kAccCols;
        for (int ci = 0; ci < kb_per_tap; ++ci) {
          ptx::mbar_wait(&afull_bar[ia], pha);
          if (lane == 0 && ci == 0) trace_tile(p, lt, 1);
          const uint32_t a0 = ptx::smem_u32(a_ring + ia * Cfg::kAStage);
          for (int tap = 0; tap < p.n_taps; ++tap) {
            if (!b_ready) ptx::mbar_wait(&bfull_bar[ib], phb);
            ptx::tc_fence_after();
            if (ptx::elect_one()) {
              const uint32_t b0 = ptx::smem_u32(b_ring + (resident ? ci * p.n_taps + tap : ib) * Cfg::kBStage);
              const uint32_t a_hi_addr = a0 + static_cast<uint32_t>(p.tap_row[z][tap]) * 128u;
              const uint64_t a_hi = umma_desc_sw128_strided(a_hi_addr, sbo);
              const uint64_t b_hi = ptx::umma_desc_sw128(b0);
#pragma unroll
              for (int k = 0; k < kChunk / 16; ++k) {
                const uint32_t accum = (ci > 0 || tap > 0 || k > 0) ? 1u : 0u;
                if constexpr (STK) {
                  const uint64_t a_lo = umma_desc_sw128_strided(a_hi_addr + kPatchStride, sbo);
                  const uint64_t b_y = ptx::umma_desc_sw128(b0 + 2 * Cfg::kBHalf);
                  ptx::umma_f16_pair(d_tmem, a_hi + 2 * k, b_hi + 2 * k, p.idesc2, accum);   // N = 2*BN: A_hi*[B_hi | B_lo]
                  ptx::umma_f16_pair(d_tmem, a_lo + 2 * k, b_y + 2 * k, p.idesc, 1u);        // N = BN:   A_lo*B_hi
                } else {
                ptx::umma_f16_pair(d_tmem, a_hi + 2 * k, b_hi + 2 * k, p.idesc, accum);
                if (NL == 2) {
                  const uint64_t a_lo = umma_desc_sw128_strided(a_hi_addr + kPatchStride, sbo);
                  const uint64_t b_lo = ptx::umma_desc_sw128(b0 + Cfg::kBHalf);
                  ptx::umma_f16_pair(d_tmem, a_hi + 2 * k, b_lo + 2 * k, p.idesc, 1u);
                  ptx::umma_f16_pair(d_tmem, a_lo + 2 * k, b_hi + 2 * k, p.idesc, 1u);
                }
                }
              }
              if (!resident) ptx::umma_commit_pair(&bempty_bar[ib], kMask);
              if (tap == p.n_taps - 1) {
                ptx::umma_commit_pair(&aempty_bar[ia], kMask);
                if (ci == kb_per_tap - 1) ptx::umma_commit_pair(&tfull_bar[acc], kMask);
              }
            }
            __syncwarp();
            if (!resident) {
              if (++ib == Cfg::kBStages) { ib = 0; phb ^= 1; }
              b_ready = ptx::mbar_try_wait(&bfull_bar[ib], phb);
            }
          }
          if (++ia == Cfg::kAStages) { ia = 0; pha ^= 1; }
        }
        if (lane == 0) trace_tile(p, lt, 2);
        if (++acc == NACC) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    epilogue_warps<BN, NL, false, STK, true, EW, NACC>(p, nullptr, s_scale, tfull_bar, tempty_bar, tmem_base, warp, lane,
                                                       static_cast<int>(blockIdx.x), static_cast<int>(gridDim.x));
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) trace_time(p, true);
  ptx::cluster_sync();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
  }
}

// ====================================================================================================
// Split-K finisher: out = epilogue( sum_s partial[s] ), for the layer's ConvParams and N tile `bn`.
// Memory-bound and tiny (the layers that use split-K have at most a few hundred output pixels per image).
// ====================================================================================================
// One thread = one pixel x 4 channels of a split-0 tile t (0 <= t < tiles_per_split).  The layers that use split-K are
// latency bound (a few hundred output pixels, 8-36 splits): what matters is how many dependent trips to L2 the sum takes, so
// up to 16 splits are in flight per trip (round 1 summed 4 per trip over 8-channel groups: 6 dependent trips for 18 splits,
// as long as the conv itself at batch 1).
template <int NL>
__global__ void __launch_bounds__(128) splitk_reduce_kernel(const __grid_constant__ ConvParams p, int bn) {
  ptx::pdl_wait();
  ptx::pdl_launch_dependents();
  const int groups = bn >> 2;
  const long long total = static_cast<long long>(p.tiles_per_split) * kTileM * groups;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(e % groups);
    const long long r0 = e / groups;
    const int row = static_cast<int>(r0 % kTileM);
    const int tile = static_cast<int>(r0 / kTileM);
    const TileCoord tc = decode_tile(p, tile);
    const OutPixel pix = out_pixel(p, tc, row);
    if (!pix.ok) continue;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const size_t split_stride = static_cast<size_t>(p.tiles_per_split) * kTileM * bn;      // floats between splits
    const float* src0 = p.partial + (static_cast<size_t>(tile) * kTileM + row) * bn + g * 4;
    int s = 0;
    for (; s + 16 <= p.n_split; s += 16) {     // sixteen independent 16-byte loads in flight
      float4 v[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) v[u] = *reinterpret_cast<const float4*>(src0 + (s + u) * split_stride);
#pragma unroll
      for (int u = 0; u < 16; ++u) {           // summation order stays s = 0, 1, 2, ... (deterministic)
        acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
      }
    }
    for (; s + 4 <= p.n_split; s += 4) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const float4*>(src0 + (s + u) * split_stride);
#pragma unroll
      for (int u = 0; u < 4; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
    }
    for (; s < p.n_split; ++s) {
      const float4 a = *reinterpret_cast<const float4*>(src0 + s * split_stride);
      acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
    }
    finish4<NL>(p, pix, tc.nt * bn + g * 4, acc);
  }
}

}  // namespace lspg
