/*
 * mewzoom_b200.h -- C ABI of the B200-native MewZoom.upscale hot path.
 *
 * The reference (andrewdalpino/UltraZoom) has NO native interface: its hot path
 * is the Python method MewZoom.upscale (src/ultrazoom/model.py:166-179) which
 * dispatches torch.nn modules.  Every entry point below therefore cites the
 * reference *Python* symbol it replaces; the Python binding a maintainer would
 * add is shown in INTEGRATION.md (ctypes, as ultrazoom_b200/_native.py does).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - every function returns 0 on success, a negative mz_status otherwise;
 *     mz_last_error() returns a thread-local message for the last failure.
 *   - all `*_dev` pointers are DEVICE pointers on the model's GPU unless a
 *     function name ends in _host.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *     Nothing here synchronises the device or allocates on the hot call
 *     (mz_upscale), except the *_host convenience entry points.
 *   - threads: an mz_model is not re-entrant -- calls on ONE model are serialised by the caller (its
 *     prepared-launch cache and host lanes are unsynchronised); different models (one per GPU, or several
 *     per GPU) may be driven from different host threads concurrently.
 *   - streams: the kernels of one mz_upscale share the caller's workspace and run in order on `stream`; two calls
 *     on ONE model (or on one workspace) must not overlap on the device -- before enqueueing on another stream,
 *     make it wait for the previous call (an event).  The Python mirror does so.
 *   - there is no CPU fallback: without an sm_100 device every compute entry
 *     point fails with MZ_ERR_CUDA / MZ_ERR_UNSUPPORTED.
 */
#ifndef MEWZOOM_B200_H_
#define MEWZOOM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MZ_ABI_VERSION 4

typedef enum mz_status {
  MZ_OK = 0,
  MZ_ERR_INVALID = -1,     /* bad argument (the reference raises AssertionError) */
  MZ_ERR_CUDA = -2,        /* CUDA runtime / driver error                        */
  MZ_ERR_UNSUPPORTED = -3, /* shape or device not supported by the kernels       */
  MZ_ERR_WORKSPACE = -4,   /* workspace too small                                */
  MZ_ERR_STATE = -5        /* weights not (fully) set                            */
} mz_status;

/* flags for mz_upscale / mz_forward */
#define MZ_FLAG_CLAMP01 1u        /* torch.clamp(z, 0, 1), model.py:177              */
#define MZ_FLAG_SIMT_CONV 2u      /* diagnostic: SIMT direct conv instead of tcgen05  */
#define MZ_FLAG_IO_U8 8u          /* x and y are 8-bit images (B,3,H,W) / (B,3,rH,rW): x = x8 / 255 (ToDtype(float32,   */
                                  /* scale=True), test_compare.py:53-57), y8 = floor(255 clamp(y) + 0.5) (save_image,   */
                                  /* test_compare.py:89).  Needs MZ_FLAG_CLAMP01.  4x less image traffic on PCIe / HBM.  */
#define MZ_FLAG_U8_TRUNC 16u      /* with MZ_FLAG_IO_U8: y8 = floor(255 clamp(y)) (ToPILImage, README.md:81)             */
#define MZ_FLAG_SKIP_FROM_BUFFER 4u /* head reads a precomputed bicubic image (mz_bicubic_f32 output in y) instead of recomputing it in its epilogue */
/* Interleaved (channels-last) images, for callers that hold pixels as numpy / PIL / OpenCV arrays or rgb24 video frames:
 * the stem reads and the head writes them directly, so neither side needs a transpose.  The two flags are independent, fp32
 * or 8-bit (MZ_FLAG_IO_U8) alike, and apply to mz_upscale, mz_upscale_window, mz_upscale_stage, mz_upscale_host and
 * mz_upscale_host_async.  Images stay 3HW (3 rH rW) elements apart, so byte counts and per-image chunking are unchanged.
 * Neither combines with MZ_FLAG_SKIP_FROM_BUFFER (MZ_ERR_INVALID); an interleaved image must be below 2^31 elements. */
#define MZ_FLAG_X_NHWC 32u        /* x is (B,H,W,3): colour c of LR pixel (y, x) at ((b H + y) W + x) 3 + c             */
#define MZ_FLAG_Y_NHWC 64u        /* y is (B,rH,rW,3); windowed output: see mz_upscale_window                          */
/* 16-bit images, for 16-bit PNG / TIFF stills and 10/12-bit video decoded to rgb48le: x and y are uint16 in either
 * layout, 6 bytes per pixel instead of fp32's 12, without 8-bit's loss of precision.  x = x16 / 65535 (the IEEE quotient:
 * ToDtype(float32, scale=True)), y16 = floor(65535 clamp(y) + 0.5) -- the result equals the fp32 call on x16 / 65535,
 * quantised so.  Needs MZ_FLAG_CLAMP01; MZ_FLAG_IO_U8, MZ_FLAG_U8_TRUNC and MZ_FLAG_SKIP_FROM_BUFFER are refused
 * (MZ_ERR_INVALID).  Applies to mz_upscale, mz_upscale_window, mz_upscale_stage, mz_upscale_host and
 * mz_upscale_host_async. */
#define MZ_FLAG_IO_U16 128u

/* Constructor kwargs of the 0.2.x-style MewZoom (README.md:254-258, model.py:52-69). */
typedef struct mz_config {
  int32_t upscale_ratio;      /* 2, 3 or 4   (SubpixelConv2d, model.py:894-898)      */
  int32_t num_channels;       /* C <= 512    (README.md:37-42); C * hidden_ratio <= 1024 */
  int32_t hidden_ratio;       /* 1, 2 or 4   (InvertedBottleneck, model.py:738)      */
  int32_t num_encoder_layers; /* L                                                   */
  int32_t control_features;   /* 0 or 3      (ControlVector, README.md:118-122)      */
  int32_t device;             /* CUDA device ordinal                                 */
  int32_t operand_dtype;      /* MZ_DTYPE_F16 (default) or MZ_DTYPE_BF16: element type of  */
                              /* the tensor-core operands (activations + weights).  Both run */
                              /* at the same tcgen05 rate; accumulation is fp32 either way.  */
                              /* fp16's 10-bit mantissa keeps max|err| vs the fp32 reference */
                              /* ~8x smaller (DESIGN.md).                                    */
  int32_t residual_stream;    /* MZ_STREAM_AUTO (0) or MZ_STREAM_FP32 (1): the residual stream */
                              /* lives in HBM as fp32 z + a 16-bit shadow (the next block's  */
                              /* tensor-core operand).  (A third form, two 16-bit planes hi +  */
                              /* lo, was measured no faster in round 1 and removed in round 2.) */
} mz_config;

#define MZ_STREAM_AUTO 0
#define MZ_STREAM_FP32 1

#define MZ_DTYPE_F16 0
#define MZ_DTYPE_BF16 1

typedef struct mz_model mz_model; /* opaque */

/* weight identifiers for mz_model_set_weight (state_dict keys of the Python module) */
typedef enum mz_weight_kind {
  MZ_W_STEM_WEIGHT = 0,  /* stem.conv.weight            (C,3,1,1)      model.py:224     */
  MZ_W_STEM_BIAS = 1,    /* stem.conv.bias              (C,)           model.py:224     */
  MZ_W_CONV1 = 2,        /* encoder.{l}.convnet.conv1.weight (hC,C,3,3) model.py:742-744 */
  MZ_W_CONV2 = 3,        /* encoder.{l}.convnet.conv2.weight (C,hC,3,3) model.py:746-748 */
  MZ_W_CTRL_WEIGHT = 4,  /* encoder.{l}.control.linear.weight (2hC,F)  (control.py, absent) */
  MZ_W_CTRL_BIAS = 5,    /* encoder.{l}.control.linear.bias   (2hC,)                     */
  MZ_W_HEAD = 6          /* head.conv.weight            (3r^2,C,3,3)   model.py:902-909 */
} mz_weight_kind;

const char* mz_last_error(void);
int mz_abi_version(void);

/* Number of visible CUDA devices with compute capability 10.x (0 if none / no driver). */
int mz_device_count(void);

/* ---- model lifetime: replaces MewZoom.__init__ / load_state_dict (model.py:52-92) ---- */
int mz_model_create(const mz_config* cfg, mz_model** out);
void mz_model_destroy(mz_model* m);

/* Upload one fp32 HOST tensor in PyTorch layout (OIHW for convs); it is repacked to the
 * 16-bit K-major per-tap layout the tcgen05 kernels read.  `layer` is ignored for
 * stem/head kinds.  `numel` must match the shape implied by the config. */
int mz_model_set_weight(mz_model* m, int32_t kind, int32_t layer, const float* host_data, size_t numel);

/* The same from a DEVICE tensor (fp32, PyTorch layout) on `stream`: the repack runs as a kernel, so a model whose
 * parameters already live on the GPU (MewZoom.to("cuda"), model.py:47 of test_compare.py) is packed without a round
 * trip through host memory.  An fp16-operand weight beyond +-65504 cannot be reported synchronously here: it raises
 * the flag mz_model_saturated reads. */
int mz_model_set_weight_dev(mz_model* m, int32_t kind, int32_t layer, const float* dev_data, size_t numel, void* stream);

/* fp16 range guard.  With MZ_DTYPE_F16 operands every 16-bit rounding in the path saturates (cvt.rn.satfinite) instead
 * of producing inf; a kernel that rounds a magnitude above 65504 -- an activation of the stem, of a hidden tensor or
 * of the residual stream, or a device-packed weight -- also sets a host-mapped flag.  *saturated = 1 if any kernel
 * that has COMPLETED so far did (the call does not synchronise; synchronise the stream first for a definite answer
 * about a particular mz_upscale).  reset != 0 clears the flag.  A saturated result is wrong: re-run the frame on a
 * model created with MZ_DTYPE_BF16 (same range as fp32).  mz_model_set_weight rejects out-of-range weights at once.
 * No entry point of this ABI checks the flag itself (mz_upscale_host included): callers read it.  The Python mirror
 * (MewZoom) checks it at every entry point: upscale_host, host_wait and capture raise in the call, the others on the
 * next call; operand_dtype="auto" re-runs forward / upscale / upscale_into / upscale_host with bf16 operands.  The U-Net
 * operators (mz_adaptive_mix, mz_pixel_crush, ...) and the per-kernel entry points do not track the range. */
int mz_model_saturated(mz_model* m, int32_t reset, int32_t* saturated);

/* Bytes of device scratch mz_upscale needs for a (B,3,H,W) input. */
int mz_workspace_bytes(const mz_model* m, int32_t B, int32_t H, int32_t W, size_t* bytes);

/* ---- the hot path: replaces MewZoom.forward / MewZoom.upscale (model.py:149-179) ----
 * x_dev : (B,3,H,W) fp32 NCHW in [0,1]   (uint8 / uint16 with MZ_FLAG_IO_U8 / _U16; (B,H,W,3) with MZ_FLAG_X_NHWC)
 * c_dev : NULL for non-control models, else (B, control_features) fp32 (c_rows == B)
 *         or (1, control_features) (c_rows == 1, broadcast) -- validate.py:73-94
 * y_dev : (B,3,rH,rW) fp32 NCHW          (uint8 / uint16 with MZ_FLAG_IO_U8 / _U16; (B,rH,rW,3) with MZ_FLAG_Y_NHWC)
 * flags : MZ_FLAG_CLAMP01 => upscale(), 0 => forward()
 */
int mz_upscale(mz_model* m, const void* x_dev, const float* c_dev, int32_t c_rows, void* y_dev,
               int32_t B, int32_t H, int32_t W, void* workspace_dev, size_t workspace_bytes,
               uint32_t flags, void* stream);

/* The same call with a WINDOWED output, for halo-tiled inference (SURVEY.md 8(e), partitioning 2): of the (H, W) input
 * tile only the LR pixels win_y0 <= y < win_y1, win_x0 <= x < win_x1 (the tile's core) are written, and they go
 * straight into an assembled frame: y_dev is where HR pixel (win_y0 * r, win_x0 * r) of plane 0 of image 0 lands,
 * HR rows are y_row_pitch elements apart and the three colour planes (and then the images) y_plane_pitch elements.
 * y_dev may be another GPU's memory with peer access enabled (mz_enable_peer_access): the head kernel's stores then ARE
 * the transfer over NVLink -- no tile output buffer, no copy, no collective.  The bicubic skip is always recomputed.
 * With MZ_FLAG_Y_NHWC (interleaved output): y_dev is where colour 0 of HR pixel (win_y0 * r, win_x0 * r) of image 0
 * lands, y_row_pitch is the number of elements between HR rows (at least 3 * r * (win_x1 - win_x0)) and y_plane_pitch the
 * number between images.
 * y_dev and both pitches must be aligned to the head's vector stores: fp32 8 / 16 / 4 bytes at r = 2 / 4 / 3, 8-bit
 * 2 / 4 / 1 bytes, 16-bit 4 / 8 / 2 bytes -- in either layout. */
int mz_upscale_window(mz_model* m, const void* x_dev, const float* c_dev, int32_t c_rows, void* y_dev,
                      int64_t y_row_pitch, int64_t y_plane_pitch, int32_t B, int32_t H, int32_t W, int32_t win_y0,
                      int32_t win_y1, int32_t win_x0, int32_t win_x1, void* workspace_dev, size_t workspace_bytes,
                      uint32_t flags, void* stream);

/* The same call cut into STAGES along the depth of the network, for halo-tiled inference with a periodic halo refresh
 * (SURVEY.md 8(e), "per-layer halo exchange" made coarse): this call runs the encoder blocks [layer_begin, layer_end)
 * on the state in the workspace; the FiLM table and the stem run first when layer_begin == 0, the head (into y_dev,
 * windowed as in mz_upscale_window, or dense when win_y1 <= 0) runs last when layer_end == num_encoder_layers.  Between
 * two stages the caller may overwrite halo pixels of the residual stream with a neighbour tile's values: the workspace
 * holds zf (B,H,W,Cp) fp32 and its 16-bit shadow zb (B,H,W,zb_pitch) at the offsets mz_workspace_layout returns (from
 * the 1024-byte-aligned workspace pointer).  Models that run fused blocks keep the 16-bit stream in the HIDDEN buffer
 * (offset hidden_offset, pitch Cp) after an odd number of blocks (mz_model_fused_block). */
int mz_upscale_stage(mz_model* m, const void* x_dev, const float* c_dev, int32_t c_rows, void* y_dev, int64_t y_row_pitch,
                     int64_t y_plane_pitch, int32_t B, int32_t H, int32_t W, int32_t win_y0, int32_t win_y1, int32_t win_x0,
                     int32_t win_x1, void* workspace_dev, size_t workspace_bytes, uint32_t flags, void* stream,
                     int32_t layer_begin, int32_t layer_end);
/* channels_padded / zb_pitch: channels per pixel of zf / zb IN MEMORY.  They may be smaller than the GEMM width of the
 * convolutions (a 54-channel model keeps its fp32 stream at 56 channels per pixel, its GEMMs run 64 wide: the zero
 * padding is made by TMA in shared memory) -- always take them from this call. */
int mz_workspace_layout(const mz_model* m, int32_t B, int32_t H, int32_t W, size_t* zf_offset, size_t* zb_offset,
                        size_t* hidden_offset, int32_t* channels_padded, int32_t* zb_pitch);

/* Enable peer access between two visible devices in this process, both directions (idempotent).  Needed before kernels
 * or copies of device `a` touch memory of device `b` that was mapped from a CUDA IPC handle. */
int mz_enable_peer_access(int32_t a, int32_t b);

/* Same call with HOST buffers: H2D copy of x (and c), the kernels, D2H copy of y, stream
 * synchronise.  Workspace and staging buffers are owned (and cached) by the model.  This is
 * the end-to-end entry point bench.py times as `e2e`. */
int mz_upscale_host(mz_model* m, const void* x_host, const float* c_host, int32_t c_rows,
                    void* y_host, int32_t B, int32_t H, int32_t W, uint32_t flags);

/* Frame-stream form of the same call: enqueue one batch on lane 0 or 1 (each lane has its own stream, staging
 * buffers and workspace) and return at once; mz_upscale_host_wait(lane) blocks until everything enqueued on that
 * lane (-1: both lanes) has finished and y_host is valid.  Alternating lanes double-buffers a stream of frames: the
 * copies of frame i+1 and i-1 run under the kernels of frame i.  Host buffers should be pinned (cudaHostAlloc /
 * torch pin_memory) -- pageable memory makes the copies synchronous -- and must stay untouched until the wait. */
int mz_upscale_host_async(mz_model* m, int32_t lane, const void* x_host, const float* c_host, int32_t c_rows,
                          void* y_host, int32_t B, int32_t H, int32_t W, uint32_t flags);
int mz_upscale_host_wait(mz_model* m, int32_t lane);

/* Optional timing of the encoder's convolution stack (the 2L launches of the dominant kernel):
 * when enabled, mz_upscale records one CUDA event on `stream` before the first and one after the
 * last encoder convolution.  mz_model_conv_stack_ms waits for those events and returns the mean
 * elapsed milliseconds over the (up to 64 most recent) calls made since timing was enabled. */
int mz_model_enable_timing(mz_model* m, int32_t enable);
int mz_model_conv_stack_ms(mz_model* m, float* ms);

/* ---- per-kernel entry points (unit tests, benches, partial pipelines) ---- */

/* Tunables of the tcgen05 convolution kernel; every field 0 = let the library choose. */
typedef struct mz_conv_tune {
  int32_t rows;       /* image rows (accumulators) per patch, 1..4                                   */
  int32_t acc_stages; /* TMEM accumulator stages, 1 or 2                                             */
  int32_t kc;         /* channels per pipeline stage: 16, 32 or 64                                   */
  int32_t halo_mode;  /* 0 one shared halo tile per K chunk + row-shifted UMMA descriptors (default);  */
                      /* 1 three aligned TMA loads per chunk, one per horizontal tap shift (diagnostic) */
  int32_t b_stages;   /* weight ring depth                                                           */
  int32_t a_stages;   /* activation ring depth                                                       */
  int32_t max_ctas;   /* cap on the persistent grid                                                  */
  int32_t cluster;    /* CTAs per cluster sharing the weight stream via TMA multicast: 1, 2 or 4       */
  int32_t dbg;        /* timing experiments ONLY (results are wrong): 1 skip weight loads, 2 skip        */
                      /* activation loads, 4 skip the epilogue body, 8 skip the MMAs, 32 / 64 every UMMA */
                      /* reads the same rows / k-step; 16 (results stay right) prints per-role clock64   */
                      /* timers to stderr after a synchronising launch                                   */
  int32_t pair;       /* CTA pairs issue M = 256 UMMAs (cta_group::2), weights split between the two:    */
                      /* 0 only when that makes the filter bank resident, 1 always, 2 never              */
  int32_t resident;   /* filter bank resident in shared memory: 0 when it fits, 1 require, 2 never       */
  int32_t epi_warps;  /* epilogue warps per CTA: 0 auto (8), 4 or 8                                      */
  int32_t fuse;       /* vertical taps stacked along N, one UMMA per input row: 0 auto, 1 force, 2 off */
  int32_t block;      /* (which = 0 only) the whole encoder block as ONE kernel -- conv1 -> control -> SiLU -> conv2 ->    */
                      /* residual with the hidden tensor kept in shared memory: 0 when the model qualifies (48 channels,  */
                      /* hidden 96, fp32 stream), 1 require, 2 never (two kernels per block)                             */
  int32_t seg_rows;   /* fused block: output rows per segment, 0 auto                                                    */
} mz_conv_tune;

/* which = 0 conv1, 1 conv2, 2 head, -1 all.  Takes effect on the next mz_upscale. */
int mz_model_set_tune(mz_model* m, int32_t which, const mz_conv_tune* tune);

/* 1 if mz_upscale runs this model's encoder blocks as ONE kernel each (hidden tensor never written to HBM), else 0. */
int mz_model_fused_block(const mz_model* m);

/* One encoder block as one kernel (EncoderBlock.forward, model.py:507-511 = InvertedBottleneck :773-778 + skip :789-792,
 * with the control module between conv1 and SiLU), for 48 channels / hidden 96:
 *   zf += conv2(SiLU(scale * conv1(zb_in) + shift)) ; zb_out = round16(zf)
 * zb_in / zb_out: (B,H,W,48) 16-bit NHWC, DIFFERENT buffers (the input is read with a halo); zf: (B,H,W,48) fp32, in
 * place; w1_packed [9][96][48] and w2_packed [9][48][96] from mz_pack_conv_weight; film_dev (B,2,96) or NULL.
 * seg_rows / max_ctas: 0 = auto (tests use them to force several segments / rounds on small images).
 * This entry point synchronises `stream` (it stacks conv2's bank into a temporary); mz_upscale keeps stacked banks. */
int mz_block_fused(const void* zb_in_dev, void* zb_out_dev, float* zf_dev, const void* w1_packed_dev,
                   const void* w2_packed_dev, const float* film_dev, int32_t B, int32_t H, int32_t W,
                   int32_t operand_dtype, int32_t seg_rows, int32_t max_ctas, void* stream);

/* Upsample(scale_factor=r, mode="bicubic") -- model.py:71,156.  NCHW fp32, `planes` = B*3 planes. */
int mz_bicubic_f32(const float* x_dev, float* y_dev, int32_t planes, int32_t H, int32_t W, int32_t r,
                   void* stream);

/* FanOutProjection (model.py:212-242) fused with the NCHW->NHWC layout change:
 * zf (B,H,W,Cp) fp32 residual stream and zb (B,H,W,zb_pitch) 16-bit MMA operand (operand_dtype);
 * zb_pitch = 0 means Cp, a larger pitch is zero-filled (mz_zb_pitch gives the pitch mz_upscale uses).
 * w_dev is (Cp,3) fp32 and bias_dev (Cp,) fp32, zero-padded beyond the logical channel count. */
int mz_stem_pack(const float* x_dev, const float* w_dev, const float* bias_dev, float* zf_dev, void* zb_dev,
                 int32_t B, int32_t H, int32_t W, int32_t Cp, int32_t zb_pitch, int32_t operand_dtype, void* stream);

/* 3x3 / pad 1 / stride 1 / bias-free convolution on NHWC 16-bit activations (model.py:742-748) with
 * the fused epilogues of one encoder block.  `wpacked_dev` comes from mz_pack_conv_weight; input, weights
 * and the 16-bit output all have element type operand_dtype.
 *   mode 0: out16 = SiLU(scale[b,n]*acc + shift[b,n])   (conv1 + control + SiLU); film_dev is
 *           (B,2,cout_p) fp32 -- scale row then shift row per image -- or NULL for scale 1, shift 0
 *   mode 1: zf += acc ; out16 = round16(zf)              (conv2 + ResidualConnection, model.py:789-792)
 * in_pitch: channel pitch of the input in elements (0 = cin_p; larger: the first cin_p channels of a wider tensor).
 * out_pitch: channel pitch of out16 in elements (0 = cout_p); channels beyond cout_p are left untouched.
 * zf_pitch: channel pitch of zf in elements (0 = cout_p).  With both pitches a convolution wider than one launch (more than
 *   256 output channels in mode 0, 128 in mode 1) runs as one launch per slice of output channels, each with its own packed
 *   bank (and FiLM rows) and its out16 / zf pointers advanced to the slice's first channel.
 * use_tc = 1: tcgen05/TMEM/TMA kernel; 0: SIMT diagnostic kernel.  tune may be NULL. */
int mz_conv3x3(const void* in_dev, const void* wpacked_dev, int32_t mode, const float* film_dev,
               void* out16_dev, float* zf_dev, int32_t B, int32_t H, int32_t W, int32_t cin_p, int32_t in_pitch,
               int32_t cout_p, int32_t out_pitch, int32_t zf_pitch, int32_t operand_dtype, int32_t use_tc,
               const mz_conv_tune* tune, void* stream);

/* SubpixelConv2d (model.py:885-930) + global skip (model.py:162) + optional clamp (:177):
 * y = [clamp](skip + PixelShuffle_r(conv3x3(z))).  skip_mode 0: none, 1: read y_dev in place
 * (precomputed bicubic), 2: recompute the bicubic from x_dev inside the epilogue.
 * wpacked_dev has cout_p = mz_padded_channels(3*r*r) rows per tap. */
int mz_head_shuffle_add(const void* zb_dev, const void* wpacked_dev, const float* x_dev, float* y_dev,
                        int32_t B, int32_t H, int32_t W, int32_t cin_p, int32_t in_pitch, int32_t r,
                        int32_t skip_mode, int32_t clamp01, int32_t operand_dtype, int32_t use_tc,
                        const mz_conv_tune* tune, void* stream);

/* Repack OIHW fp32 (host) -> device fp16|bf16 [tap = ky*3+kx][cout_p][cin_p] (K-major rows; the TMA
 * applies the shared-memory swizzle).  With dst_dev == NULL only *bytes is written. */
int mz_pack_conv_weight(const float* w_host, int32_t cout, int32_t cin, int32_t cout_p, int32_t cin_p,
                        int32_t operand_dtype, void* dst_dev, size_t* bytes);

/* FiLM coefficients for every layer: film[l][b][0][n] = 1 + gamma, film[l][b][1][n] = beta,
 * from c (B or 1 rows) and the per-layer Linear(F, 2hC) weights (control module; README.md:11,88). */
int mz_control_film(const float* c_dev, int32_t c_rows, const float* w_dev /*L,2hC,F*/,
                    const float* b_dev /*L,2hC*/, float* film_dev /*L,B,2,hCp*/, int32_t L, int32_t B,
                    int32_t F, int32_t hC, int32_t hCp, void* stream);

/* Spatial sharding (SURVEY.md 8(e), partitioning 2): put a tile's HR core -- `height` rows of `width_bytes` bytes at
 * pitch `spitch` -- into the assembled frame at pitch `dpitch`, asynchronously on `stream`.  `dst` may live on another
 * GPU (a peer mapping opened from the owner's IPC handle) or in pinned host memory: a one-sided cudaMemcpy2DAsync, no
 * collective.  One call per colour plane of the tile. */
int mz_put_plane_async(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width_bytes, size_t height,
                       void* stream);

/* The assembled frame of a multi-process (one process per GPU) tiled run.  The owner allocates it and gets a 64-byte
 * CUDA IPC handle to hand to the other processes of the node (control plane: any byte transport); each of them opens
 * it WITH ITS OWN GPU CURRENT, which maps the owner's memory for that GPU's kernels and copy engines over NVLink
 * (cudaIpcMemLazyEnablePeerAccess) -- a mapping opened under another device is reachable by copies only.
 * close: owner != 0 frees the allocation, otherwise the mapping is released. */
int mz_ipc_frame_create(size_t bytes, void** dev_ptr, void* handle64);
int mz_ipc_frame_open(const void* handle64, void** dev_ptr);
int mz_ipc_frame_close(void* dev_ptr, int32_t owner);

/* ---- operators of the reference's 0.3.0 U-Net (SURVEY.md 8(f) rank 3) on NHWC fp32 feature maps ----------------------
 * Feature maps are (B,H,W,pitch) fp32 with the logical channels first; every operator can also write the 16-bit shadow
 * (operand_dtype) the tcgen05 convolutions read as their A operand (out16_dev, same pitch; NULL = none).  The 3x3
 * convolutions of these blocks (InvertedBottleneck model.py:731-778, SubpixelConv2d.conv :902-909) are mz_conv3x3 /
 * mz_head_shuffle_add; what follows is everything else.  Weights are passed as [N][K] fp32 device matrices, K-contiguous
 * (N = output channels), i.e. the reference's conv.weight with the kernel taps moved in front of the input channels:
 *   mix:    wt[n][k] = conv.weight[n][k][0][0]                 (K = 2C: x channels then z channels; a plain reshape)
 *   crush:  wt[n][(i*f + j)*Cin + c] = conv.weight[n][c][i][j]  (K = f*f*Cin)
 *   assess: wt[n][(ky*3 + kx)*C + c] = conv.weight[n][c][ky][kx] (K = 9C)
 * (the Python mirror, ultrazoom_b200/unet.py, builds them from the reference's state_dict tensors).
 * math: MZ_MATH_TF32 (default) runs the mix / crush GEMM on tcgen05 tensor cores straight from the fp32 feature maps
 * (operands truncated to tf32, fp32 accumulation; pointers 16-byte aligned, C and pitches multiples of 4);
 * MZ_MATH_FP32 is the exact fp32 SIMT twin of the same operator. */
#define MZ_MATH_TF32 0
#define MZ_MATH_FP32 1

/* AdaptiveResidualMix.forward (model.py:826-839): beta = sigmoid(conv1x1(cat[x, z])); w = sigmoid(alpha) * beta;
 * out = (1 - w) * x + w * z.  x, z, out: (npix, pitch) fp32. */
int mz_adaptive_mix(const float* x_dev, const float* z_dev, const float* wt_dev, float alpha_logit, float* out_dev,
                    void* out16_dev, int64_t npix, int32_t C, int32_t pitch, int32_t operand_dtype, int32_t math, void* stream);

/* PixelCrush.forward (model.py:881-882): Conv2d(Cin, Cout, kernel_size=f, stride=f, bias=False), f in {2, 3, 4};
 * (B,H,W,pitch_in) -> (B, H/f, W/f, pitch_out) (floor, as the convolution does). */
int mz_pixel_crush(const float* in_dev, const float* wt_dev, float* out_dev, void* out16_dev, int32_t B, int32_t H, int32_t W,
                   int32_t Cin, int32_t Cout, int32_t factor, int32_t pitch_in, int32_t pitch_out, int32_t operand_dtype,
                   int32_t math, void* stream);

/* QualityAssessor.forward (model.py:1024-1032): Conv2d(C, F, 3, padding=1) + bias -> AdaptiveAvgPool2d(1) -> (B, F). */
int mz_quality_assessor(const float* in_dev, const float* wt_dev, const float* bias_dev, float* out_dev, int32_t B, int32_t H,
                        int32_t W, int32_t C, int32_t F, int32_t pitch_in, void* stream);

/* PixelShuffle(r) on NHWC (mid-network SubpixelConv2d, model.py:911,928; Decoder :569-571):
 * out[b, h r + i, w r + j, c] = in[b, h, w, c r r + i r + j]; in (B,H,W,pitch_in >= C r r) -> out (B,rH,rW,pitch_out). */
int mz_pixel_shuffle_nhwc(const float* in_dev, float* out_dev, void* out16_dev, int32_t B, int32_t H, int32_t W, int32_t C,
                          int32_t r, int32_t pitch_in, int32_t pitch_out, int32_t operand_dtype, void* stream);

/* Decoder.crop_feature_maps (model.py:650-689): centre-crop or zero-pad (B,H,W,C) to (B,target_h,target_w,C). */
int mz_crop_feature_maps(const float* in_dev, float* out_dev, int32_t B, int32_t H, int32_t W, int32_t C, int32_t target_h,
                         int32_t target_w, int32_t pitch_in, int32_t pitch_out, void* stream);

/* Hardware probes used by tests and DESIGN.md (not on the hot path).
 * mz_probe_umma: one 128 x 64 x kc UMMA whose A descriptor starts `row_shift` rows into a
 * TMA-swizzled tile; base_offset_mode 0 leaves the descriptor's base_offset 0, 1 sets it to
 * (start >> 7) & 7.  Writes the max abs error against an exact host product.
 * mz_probe_mma_rate: `iters` back-to-back 128 x n x 16 UMMAs per CTA on `ctas` CTAs, cycling over
 * `distinct_a` A tiles and `distinct_d` TMEM accumulators, the A descriptor starting `a_row_shift` rows into its
 * tile (the shared-halo conv's shifted taps); writes SM cycles per UMMA (mean over CTAs). */
int mz_probe_umma(int32_t kc, int32_t row_shift, int32_t base_offset_mode, float* max_abs_err_out);
/* mz_probe_set_gap: subsequent mz_probe_mma_rate calls idle the issuing thread for `gap_cycles` (after a
 * tcgen05.commit when commit_in_gap != 0) between bursts of 8 * burst_iters UMMAs (0 = no gaps): measures how much
 * issuer-side bookkeeping the UMMA queue hides. */
int mz_probe_set_gap(int32_t burst_iters, int32_t gap_cycles, int32_t commit_in_gap);
int mz_probe_mma_rate(int32_t n, int32_t kc, int32_t iters, int32_t ctas, int32_t distinct_a,
                      int32_t distinct_d, int32_t a_row_shift, float* cycles_per_mma_out);

/* Padded channel counts the kernels use for a logical channel count. */
int mz_padded_channels(int32_t c);

/* Channel pitch of the 16-bit shadow `zb` of the residual stream for a padded channel count: 48 -> 64 (so that a
 * pixel is one 128-byte TMA row instead of three 32-byte ones), otherwise unchanged. */
int mz_zb_pitch(int32_t cp);

#ifdef __cplusplus
}
#endif
#endif /* MEWZOOM_B200_H_ */
