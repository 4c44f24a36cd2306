/*
 * lspg.h - C ABI of the B200-native Feature2Face generator (LiveSpeechPortraits render hot path).
 *
 * The reference has no native code and no FFI: its "plugin boundary" for this path is the Python class
 * models/feature2face_G.py:Feature2Face_G (ctor(opt) :8-21, forward(input) :27-34) held by
 * models/feature2face_model.py:Feature2FaceModel (ctor :22-27, inference() :225-237) and fed by
 * models/base_model.py:load_networks (:193-223, state_dict in) / eval() (:108-113).
 * Each entry point below names the reference call it stands in for.  A Python `nn.Module` shim
 * (livespeechportraits_b200/generator.py) binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative LSPG_E* code and
 * records a message retrievable with lspg_last_error() (thread-local).  No CPU compute path exists:
 * forward needs an sm_100 device and fails loudly otherwise.  One handle per device; calls on one handle
 * must be serialised by the caller.  All device work is enqueued on the caller's stream; nothing
 * synchronises or allocates inside lspg_forward once the (B,H,W,mode,workspace) plan is cached.
 */
#ifndef LSPG_H_
#define LSPG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSPG_OK 0
#define LSPG_EINVAL (-1)     /* bad argument / unsupported shape */
#define LSPG_ENODEV (-2)     /* no sm_100 device / host-only handle */
#define LSPG_ECUDA (-3)      /* CUDA runtime or driver error */
#define LSPG_ESTATE (-4)     /* weights not loaded, workspace too small, ... */
#define LSPG_ENOMEM (-5)

/* opt.size values that reach this path (models/feature2face_G.py:16-21; 'small' is out of scope) */
#define LSPG_VARIANT_NORMAL 0
#define LSPG_VARIANT_LARGE 1

/* Precision modes.  FAST: bf16 operands, fp32 accumulate (1 MMA / K step).
 * PARITY: fp16 hi+lo split operands (22 mantissa bits), hi*hi + hi*lo + lo*hi, fp32 accumulate (3 MMAs / K step);
 * this is the mode that meets the 1e-3 max-abs contract against the fp32 reference.  Activations are stored as fp16
 * limbs: values beyond +-65504 saturate (the network's activations are O(1..100)). */
#define LSPG_MODE_FAST 0
#define LSPG_MODE_PARITY 1

typedef struct lspg_ctx* lspg_handle;

/* One state_dict entry (models/base_model.py:208-219 hands exactly these to load_state_dict).
 * `name` uses the reference key grammar without the DataParallel "module." prefix, e.g.
 * "netG.model.model.0.weight"; data is host memory, fp32, contiguous (conv weights OIHW). */
typedef struct lspg_tensor {
  const char* name;
  const float* data;
  int64_t numel;
} lspg_tensor;

/* Replaces Feature2Face_G.__init__ (models/feature2face_G.py:8-21) + networks.init_net's device move
 * (models/networks.py:392-394).  device >= 0: CUDA ordinal, must be compute capability 10.x.
 * device == -1: host-only handle for plan/packing introspection (lspg_forward returns LSPG_ENODEV). */
int lspg_create(lspg_handle* out, int variant, int ngf, int num_downs, int in_nc, int out_nc, int device);

/* Replaces net.load_state_dict(state_dict, strict=False) (models/base_model.py:219) and the eval-mode
 * BatchNorm semantics of BaseModel.eval() (:108-113): folds running stats into per-channel scale/shift
 * (eps 1e-5), packs conv weights into the K-major tap/phase layout the kernels read, uploads them.
 * Keys that are absent keep their previous value (strict=False); unknown keys are ignored;
 * a known key with the wrong element count is LSPG_EINVAL. */
int lspg_load_weights(lspg_handle h, const lspg_tensor* tensors, int n);

/* Bytes of caller-owned device workspace lspg_forward needs for this problem size and mode. */
int lspg_workspace_bytes(lspg_handle h, int batch, int height, int width, int mode, size_t* out);

/* Replaces Feature2FaceModel.inference's cat + G call (models/feature2face_model.py:231-233) and
 * Feature2Face_G.forward (models/feature2face_G.py:27-34), eval mode, opt.fp16 == 0.
 *   feature_map: device fp32 [B,1,H,W], batch stride fm_bstride elements
 *   cand:        device fp32 [B,12,H,W], batch stride cand_bstride elements (0 = one candidate set for
 *                every frame, as demo.py:266 does)
 *   out:         device fp32 [B,3,H,W] contiguous, values in (-1,1)
 * A single [B,13,H,W] tensor x is passed as feature_map=x, cand=x+H*W, both strides 13*H*W.
 * H and W must be powers of two >= 256 (8 stride-2 stages; every level must tile into the kernels' power-of-two boxes -
 * the reference accepts any multiple of 256, e.g. 768, which this library rejects with LSPG_EINVAL rather than
 * mis-render).  Asynchronous on `stream` (a cudaStream_t).  The launches of one (B,H,W,mode,workspace) plan are captured
 * once as a CUDA graph; a call with different feature_map / cand / out pointers patches two kernel nodes in place
 * (cudaGraphExecKernelNodeSetParams), it does not re-capture.  Returns LSPG_ESTATE if any conv weight was never loaded. */
int lspg_forward(lspg_handle h, const float* feature_map, int64_t fm_bstride, const float* cand,
                 int64_t cand_bstride, float* out, int batch, int height, int width, void* workspace,
                 size_t workspace_bytes, int mode, void* stream);

/* Same as lspg_forward with the reference's post-processing fused into the last kernel: replaces
 * util.tensor2im(pred_fake[i]) (util/util.py:19-42, called at demo.py:268) = (x+1)/2*255 in fp32, clip to [0,255],
 * truncate to uint8, CHW -> HWC.  out_hwc: device uint8 [B,H,W,3].  A quarter of the bytes of the fp32 frame, so the
 * device->host copy and the multi-GPU all-gather of frames shrink 4x. */
int lspg_forward_image(lspg_handle h, const float* feature_map, int64_t fm_bstride, const float* cand,
                       int64_t cand_bstride, uint8_t* out_hwc, int batch, int height, int width, void* workspace,
                       size_t workspace_bytes, int mode, void* stream);

/* Feature-map rasteriser for a batch of frames ("next" row N2): replaces FaceDataset.get_data_test_mode ->
 * get_feature_image -> draw_face_feature_maps + draw_shoulder_points (datasets/face_dataset.py:276-323; 72 + 16
 * cv2.line(img, int(p1), int(p2), 255, 2) calls per frame, then uint8 -> float32 / 255) and the per-frame 1 MB
 * host->device copy at demo.py:262-265.  Bit-exact with cv2.line (OpenCV 4.13 semantics, see oracle/raster_oracle.py).
 *   landmarks:  device fp32 [B,73,2] (x,y) in pixels; truncated toward zero like Python int()
 *   shoulders:  device fp32 [B,n_shoulder_points,2] or NULL (n_shoulder_points even; two polylines of n/2 points)
 *   out_fm:     device fp32 [B,1,H,W], every element written (0 or 1): ready to be lspg_forward's feature_map
 * Asynchronous on `stream`. */
int lspg_draw_feature_maps(lspg_handle h, const float* landmarks, const float* shoulders, int n_shoulder_points,
                           float* out_fm, int batch, int height, int width, void* stream);

/* Tell the library that the caller is about to free (or reuse) `workspace`: waits for the device, then drops every cached
 * plan / CUDA graph that points into it.  workspace == NULL drops all plans.  Replaces nothing in the reference. */
int lspg_release_workspace(lspg_handle h, void* workspace);

/* Replaces nothing in the reference (module garbage collection). */
int lspg_destroy(lspg_handle h);

const char* lspg_last_error(void);

/* ---- introspection (tests, bench accounting; no compute) ------------------------------------------ */

typedef struct lspg_layer_info {
  int kind;                 /* 0 head, 1 stride-1, 2 stride-2, 3 upsample-phase, 4 tail */
  int n_src, src[2], cin[2];/* activation tensor ids and channels of the concat sources */
  int out, res;             /* output / residual tensor ids (-1 = none; tail writes the user buffer) */
  int cout, cout_pad;
  int n_phases, n_taps, k_total; /* packed weights: [n_phases][cout_pad][k_total] */
  int relu, has_bn;
  int8_t tap_map[4][9], tap_dx[4][9], tap_dy[4][9];
  char conv_key[96];        /* state-dict key prefix of the conv (".weight" appended) */
  char bn_key[96];          /* "" when the conv has no BatchNorm */
} lspg_layer_info;

/* Tiling / kernel choice of one layer for a problem size, as the launch plan will make it (host logic only; works on a
 * host-only handle, where the SM count defaults to 148).  Lets the CPU tests pin the planner. */
typedef struct lspg_layer_geo {
  int kernel;            /* 0 conv_umma_kernel (one box per tap), 1 conv_patch_kernel, 2 conv_pair_kernel (cta_group::2) */
  int bn;                /* N tile */
  int tile_w, tile_h, tile_n;   /* output tile = tile_w x tile_h pixels x tile_n images = 128 rows */
  int m_tiles, n_tiles, n_phases;
  int n_split, split_len, k_items;   /* split-K: K loop of k_items cut into n_split ranges of split_len */
  int ctas;              /* CTAs launched = min(tiles * n_split, SMs), even for the pair kernel */
  int64_t partial_bytes; /* fp32 split-K partials this layer needs in the scratch region (0 for a cluster split) */
  int cluster_split;     /* > 0: the n_split CTAs of a tile are one thread-block cluster and reduce through distributed shared
                            memory (no finisher launch); then n_split == cluster_split in {2, 4, 8} */
  int cta_cluster;       /* CTAs per thread-block cluster of the launch: 2 for the pair kernel and for a patch kernel that
                            multicasts its weights, cluster_split for a cluster split, 1 otherwise */
} lspg_layer_geo;
int lspg_debug_layer_geo(lspg_handle h, int layer, int batch, int height, int width, lspg_layer_geo* out);

/* Byte offset of limb `limb` of activation tensor `id` in the workspace of a (batch,height,width,mode) forward, counted from
 * the first 1024-byte-aligned address of the workspace (where the launch plan places tensor 0).  Host logic only; works on
 * a host-only handle.  Lets a caller view the stored activations in place. */
int lspg_debug_tensor_offset(lspg_handle h, int id, int limb, int batch, int height, int width, int mode, size_t* offset);

/* Test hook (host only, no device): q = n / d computed exactly as the kernels' tile decode does it (multiply-high by a
 * launch-time constant, csrc/conv_umma.cuh make_fast_div / fast_div); valid for n < 2^31, d >= 1. */
int lspg_debug_fast_div(uint32_t n, uint32_t d, uint32_t* q);

int lspg_num_layers(lspg_handle h, int* out);
int lspg_layer_info_get(lspg_handle h, int layer, lspg_layer_info* out);
/* Packed weights as the kernels see them, 16-bit patterns: limb 0 / 1 = PARITY operands, fp16 hi and lo (v - hi) limbs of
 * v = w * LSPG_PARITY_WEIGHT_SCALE (the epilogue scale carries the inverse); limb 2 = FAST operand, bf16(w).
 * `count` must be n_phases*cout_pad*k_total.  scale/shift: cout_pad floats each (the unscaled BatchNorm fold). */
#define LSPG_PARITY_WEIGHT_SCALE 256.0f
int lspg_layer_packed(lspg_handle h, int layer, int limb, uint16_t* dst, int64_t count);
int lspg_layer_affine(lspg_handle h, int layer, float* scale, float* shift, int64_t count);
/* Activation tensor table for (batch,height,width): per-image channels/height/width of tensor `id`. */
int lspg_num_tensors(lspg_handle h, int* out);
int lspg_tensor_shape(lspg_handle h, int id, int height, int width, int* c, int* th, int* tw);
/* Copy activation tensor `id` (16-bit NHWC: bf16 after a FAST forward, fp16 limb 0 or 1 after a PARITY forward) of the most
 * recent forward to host memory. */
int lspg_debug_read_tensor(lspg_handle h, int id, int limb, uint16_t* dst, int64_t count);
/* Debug: with LSPG_TRACE_LAYER=<i> in the environment the conv kernel of layer i stamps clock64() at its pipeline
 * milestones (conv_umma.cuh: kTraceSlots values per CTA, 256 CTAs); this copies them out. */
int lspg_debug_read_trace(lspg_handle h, uint64_t* dst, int64_t count);
/* CUDA-graph bookkeeping since lspg_create: graphs captured + instantiated, in-place I/O pointer updates, and re-captures
 * forced by a failed update (expected 0). */
int lspg_graph_stats(lspg_handle h, int64_t* captures, int64_t* io_updates, int64_t* recaptures);
/* Kernels one lspg_forward call launches (for bench.py's gpu_launches accounting). */
int lspg_launches_per_forward(lspg_handle h, int* out);
/* Per-launch timing: when enabled, every lspg_forward records a CUDA event on `stream` before its first
 * kernel and after each kernel (no host synchronisation).  lspg_profile_read synchronises on the recorded
 * events, returns the average duration in milliseconds of each of the launches_per_forward launches over the
 * forwards recorded since the previous read (at most 256 are kept), and resets the record. */
int lspg_profile_enable(lspg_handle h, int enabled);
int lspg_profile_read(lspg_handle h, float* avg_ms, int count, int* n_forwards);
/* Algorithmic conv FLOPs per frame (2*MAC of the reference convs) at height x width. */
int lspg_flops_per_frame(lspg_handle h, int height, int width, double* out);

#ifdef __cplusplus
}
#endif
#endif /* LSPG_H_ */
