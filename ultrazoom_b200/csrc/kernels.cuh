// kernels.cuh -- internal launch interfaces and the fused epilogues shared by the tcgen05 and the
// SIMT (diagnostic) convolution kernels.  Everything here is device code for sm_100a or plain
// host structs; nothing is exported (the C ABI lives in api.cu / model.cu).
#pragma once

#include <string.h>

#include <type_traits>
#include <vector>

#include "common.cuh"

namespace mz {

// ----------------------------------------------------------------------------------------------
// Bicubic phase table -- Upsample(scale_factor=r, mode="bicubic"), reference model.py:71,156.
// For integer r an output coordinate o has phase p = o % r; its four taps start at
// (o / r) + off[p] - 1 and carry weights w[p][0..3] (Keys kernel, A = -0.75, half-pixel centres,
// align_corners=False).  Tap indices are clamped to the image (no renormalisation).
// ----------------------------------------------------------------------------------------------
struct BicubicTable {
  int r;
  int off[4];
  float w[4][4];
};
void make_bicubic_table(int r, BicubicTable* t);

// ----------------------------------------------------------------------------------------------
// The call's two images, as the stem reads x and the head reads x and writes y.
// ----------------------------------------------------------------------------------------------
// Element type of both images.  8 bits (MZ_FLAG_IO_U8): x holds round(255 * x), read back as x / 255 (ToDtype(float32,
// scale=True), reference test_compare.py:53-57); y = floor(255 * clamp(v, 0, 1) + 0.5) (torchvision save_image,
// test_compare.py:89) or floor(255 * clamp(v, 0, 1)) with u8_trunc (ToPILImage, README.md:81).  16 bits
// (MZ_FLAG_IO_U16): x is read as the IEEE quotient x / 65535; y = floor(65535 * clamp(v, 0, 1) + 0.5).
enum ImageType : int { kImgF32 = 0, kImgU8 = 1, kImgU16 = 2 };
struct ImageIo {
  const void* x;  // LR image (B,3,H,W)
  void* y;        // HR image (B,3,rH,rW)
  int type;       // ImageType
  // Interleaved images (MZ_FLAG_X_NHWC / MZ_FLAG_Y_NHWC): x is (B,H,W,3), y is (B,rH,rW,3) -- colour c of a pixel at
  // pixel * 3 + c, images 3HW (3 rH rW) elements apart as in the planar layout.
  int x_nhwc, y_nhwc;
  int u8_trunc;
  int skip_mode;  // 0 none, 1 y already holds the bicubic image (fp32 only), 2 recompute bicubic from x
  int clamp01;
  // Windowed output (mz_upscale_window; all zero = the whole image, densely): only LR pixels wy0 <= y < wy1,
  // wx0 <= x < wx1 are stored, pixel (wy0, wx0) of plane 0 of image 0 at y itself, HR rows y_row elements and colour
  // planes y_plane elements apart -- a tile's core written straight into an assembled (possibly remote) frame.  For an
  // interleaved output y points at colour 0 of HR pixel (wy0 r, wx0 r), y_row is the element pitch of HR rows and
  // y_plane that of images.
  int wy0, wy1, wx0, wx1;
  long long y_row, y_plane;
};

// ----------------------------------------------------------------------------------------------
// Epilogue parameters.
//   mode 0: hidden = SiLU(scale[b,n] * acc + shift[b,n])   -> bf16 NHWC      (conv1 + control + SiLU)
//   mode 1: zf += acc ; zb = bf16(zf)                                         (conv2 + ResidualConnection)
//   mode 2: y = [clamp](skip + PixelShuffle_r(acc))         -> the HR image   (SubpixelConv2d + skip)
// ----------------------------------------------------------------------------------------------
struct EpiParams {
  int mode;
  int B, H, W;
  int bf16;           // MMA-operand element type of every 16-bit tensor: 0 = fp16, 1 = bf16
  int n_pad;          // GEMM N (multiple of 16) == channel pitch of the 16-bit / fp32 NHWC outputs
  const float* film;  // mode 0: [B][2][n_pad] (scale row then shift row per image) or nullptr
  uint16_t* out_bf16;       // mode 0: hidden; mode 1: zb (fp16 or bf16 bits)
  int out_pitch;            // channel pitch of out_bf16 in elements (0 = n_pad); > n_pad when the consumer wants
                            // zero-padded channels (48-channel zb is kept at pitch 64: 128-byte TMA rows)
  int out_extent;           // channels of out_bf16 that exist in memory (0 = n_pad; a multiple of 8).  < n_pad = DENSE
                            // layout: the GEMM's zero padding lives in shared memory only -- the tensor maps end at the
                            // extent, so TMA neither writes the padding nor fetches it (out-of-bounds reads are zeros)
  float* zf;                // mode 1: fp32 residual stream, updated in place
  int zf_pitch;             // channel pitch of zf in elements (0 = n_pad); > n_pad when this launch owns a channel slice
  int zf_extent;            // channels of zf that exist in memory (0 = n_pad), as out_extent
  // mode 2: the images (a prepared launch takes them from each call: patch_conv_epi), the ratio and its bicubic table
  ImageIo img;
  int r;
  // fp16 range guard: a kernel that is about to round a value beyond +-65504 into a 16-bit fp16 operand (where
  // cvt.rn.satfinite would clip it silently) writes 1 here.  Points at a host-mapped word owned by the mz_model
  // (mz_model_saturated); nullptr = not tracked (per-kernel entry points).
  unsigned int* sat;
  BicubicTable bt;
};

// largest finite fp16: a pre-rounding magnitude above it saturates the operand
#define MZ_F16_MAX 65504.0f

// address of colour c of HR pixel (y r + i, x r + j) of image b in the output of mode 2, or -1 outside the window;
// YN: interleaved output (ImageIo::y_nhwc)
template <bool YN>
__host__ __device__ inline long long head_out_index_l(const EpiParams& p, int b, int c, int y, int x, int i, int j) {
  const ImageIo& io = p.img;
  const long long WR = static_cast<long long>(p.W) * p.r, HR = static_cast<long long>(p.H) * p.r;
  if (io.wy1 > 0 && (y < io.wy0 || y >= io.wy1 || x < io.wx0 || x >= io.wx1)) return -1;
  if (YN) {
    const long long row = io.y_row ? io.y_row : 3 * WR, img = io.y_plane ? io.y_plane : 3 * HR * WR;
    return static_cast<long long>(b) * img + (static_cast<long long>(y - io.wy0) * p.r + i) * row +
           (static_cast<long long>(x - io.wx0) * p.r + j) * 3 + c;
  }
  const long long row = io.y_row ? io.y_row : WR, plane = io.y_plane ? io.y_plane : HR * WR;
  return (static_cast<long long>(b) * 3 + c) * plane + (static_cast<long long>(y - io.wy0) * p.r + i) * row +
         static_cast<long long>(x - io.wx0) * p.r + j;
}
__host__ __device__ inline long long head_out_index(const EpiParams& p, int b, int c, int y, int x, int i, int j) {
  return p.img.y_nhwc ? head_out_index_l<true>(p, b, c, y, x, i, j) : head_out_index_l<false>(p, b, c, y, x, i, j);
}

// One 3x3 convolution launch (both kernels).
struct ConvArgs {
  const uint16_t* in;  // (B,H,W,cin_p) fp16 | bf16
  const uint16_t* w;   // [9][n_pad][cin_p] fp16 | bf16, tap = ky*3+kx
  int cin_p;
  int in_pitch;        // channel pitch of `in` in elements (0 = cin_p): a wider tensor's first cin_p channels are read
  int k_valid;         // channels of `in` that can be non-zero (0 = cin_p): whole 16-channel k-steps beyond them are zero
                       // padding and may be skipped by the kernel (results do not change: they would add zeros)
  int in_extent;       // channels of `in` that exist in memory (0 = cin_p; a multiple of 8): see EpiParams::out_extent
  EpiParams epi;
};

// Tunables of the tcgen05 kernel (0 = let the launcher choose).
struct ConvTcTune {
  int rows;        // image rows per patch (accumulators per TMEM stage), 1..4
  int acc_stages;  // 1 or 2 TMEM accumulator stages
  int kc;          // K chunk per pipeline stage: 16, 32 or 64 channels
  int halo_mode;   // 0: one shared halo tile per K chunk, row-shifted UMMA descriptors (default)
                   // 1: three TMA loads per chunk, one per horizontal tap shift (aligned descriptors; diagnostic)
  int b_stages;    // weight ring depth
  int a_stages;    // activation ring depth
  int max_ctas;    // cap on the persistent grid (0 = SM count)
  int cluster;     // CTAs per cluster sharing the weight stream through TMA multicast: 1, 2 or 4 (0 = auto)
  int pair;        // CTA pairs issue M = 256 UMMAs (cta_group::2), each CTA holding half of the weight rows:
                   // 0 = only when that makes the filter bank resident, 1 = always, 2 = never
  int resident;    // filter bank resident in shared memory: 0 = when it fits, 1 = require, 2 = never (stream per patch)
  int epi_warps;   // epilogue warps: 0 = auto (8), 4 or 8
  int fuse;        // filter rows fused along N (one UMMA per input row): 0 = when three taps stack (N <= 85), 1 = also with two, 2 = never
  int block;       // whole encoder block (conv1 -> FiLM -> SiLU -> conv2 -> residual) as ONE kernel (block_fused.cu):
                   // 0 = when the model qualifies (48 channels, hidden 96), 1 = require, 2 = never (two kernels per block)
  int seg_rows;    // fused block: output rows per segment (0 = auto)
  int dbg;         // timing experiments only (WRONG results): 1 skip weight loads, 2 skip activation loads,
                   // 4 skip the epilogue body, 8 skip the MMAs
};

int launch_conv_simt(const ConvArgs& a, cudaStream_t s);
int launch_conv_tc(const ConvArgs& a, const ConvTcTune& tune, int device, cudaStream_t s);
// The same in two steps: prepare (geometry search, tensor-map encoding, kernel selection -- host work only) and run.
struct alignas(64) ConvLaunch {
  unsigned char storage[2048];
  bool valid = false;
};
int prepare_conv_tc(const ConvArgs& a, const ConvTcTune& tune, int device, ConvLaunch* out);
int run_conv_tc(ConvLaunch& launch, cudaStream_t s);
// head (mode 2) only: replace the images (EpiParams::img) of a prepared launch (a new layout swaps the kernel
// instantiation)
int patch_conv_epi(ConvLaunch& launch, const EpiParams& e);
// ---- one encoder block as one kernel (block_fused.cu): zf += conv2(SiLU(FiLM(conv1(zb_in)))), zb_out = round16(zf) ----
struct FusedBlockArgs {
  const uint16_t* zb_in;  // (B,H,W,48) 16-bit: read with a halo, so the output goes to a second buffer
  uint16_t* zb_out;       // (B,H,W,48) 16-bit
  float* zf;              // (B,H,W,48) fp32 residual stream, updated in place
  const uint16_t* w1;     // conv1 bank [9][96][48]
  const uint16_t* w2s;    // conv2 bank, vertical taps stacked per filter column: [3 dx][144][96] (stack_conv2_bank)
  const float* film;      // [B][2][96] or nullptr
  unsigned int* sat;      // fp16 range guard (EpiParams::sat) or nullptr
  int B, H, W, bf16;
  int seg_rows;           // output rows per segment (0 = auto)
  int max_ctas;           // cap on the persistent grid (0 = SM count)
};
bool fused_block_applies(int Cp, int hCp, int zb_pitch);
int stack_conv2_bank(const uint16_t* packed, uint16_t* stacked, cudaStream_t s);
int prepare_block_fused(const FusedBlockArgs& a, int device, ConvLaunch* out);
int run_block_fused(ConvLaunch& launch, cudaStream_t s);

// ---- AdaptiveResidualMix / PixelCrush as one tcgen05 kind::tf32 GEMM on the fp32 feature maps (unet_tc.cu) ----
struct SgArgs {
  const float* a0;    // x | input feature map
  const float* a1;    // z | nullptr
  const float* wt;    // [N][K] fp32 (conv.weight as the reference stores it, K = taps x C)
  float* out;
  void* out16;        // optional 16-bit shadow
  int bf16;
  int mix;            // 1: gated mix of (a0, a1); 0: f x f / stride f crush of a0
  float gate;         // sigmoid(alpha)
  int C, N, f;
  long long rows;     // output rows (B * Ho | 1)
  long long wo;       // output pixels per row (Wo | npix)
  int H, Ho, W;       // crush: input rows per image, output rows per image, input width
  long long in_rows;  // crush: B * H
  int pitch_in, pitch_out;
};
bool seg_gemm_tc_applies(const float* a0, const float* a1, const float* wt, const float* out, const void* out16, int C, int N,
                         int K, int pitch_in, int pitch_out);
int launch_seg_gemm_tc(const SgArgs& a, cudaStream_t s);

int launch_bicubic(const float* x, float* y, int planes, int H, int W, int r, cudaStream_t s);
// image x (element type `type`, interleaved when x_nhwc: as ImageIo) -> fp32 stream zf + 16-bit shadow zb (pitch zb_pitch)
int launch_stem(const void* x, int type, int x_nhwc, const float* w, const float* bias, float* zf, uint16_t* zb, int bf16,
                int B, int H, int W, int Cp, int zb_pitch, cudaStream_t s, unsigned int* sat = nullptr);
// film: [L][hCp / ns][B][2][ns] -- one [B][2][ns] table (scale row, shift row) per conv1 launch; ns == hCp normally
int launch_film(const float* c, int c_rows, const float* w, const float* b, float* film, int L, int B, int F,
                int hC, int hCp, int ns, cudaStream_t s);

// 4:2:0 frames (yuv420.cu): colour matrix and code range of the MZ_FLAG_YUV* bits.  yuv_coef refuses (MZ_ERR_INVALID)
// flags without MZ_FLAG_YUV420, without exactly one of MZ_FLAG_IO_U8 / _U16, or with both matrix bits.
struct YuvCoef {
  float kr, kb, kg;             // Kr, Kb, Kg = 1 - Kr - Kb
  float yoff, yrange;           // Y = yoff + yrange Y'
  float coff, crange, maxcode;  // C = coff + crange C'; codes 0..maxcode
};
int yuv_coef(uint32_t flags, YuvCoef* k);
// yuv (B frames of 3HW/2 elements) <-> rgb16 (B,3,H,W); H and W even, the LR or HR luma size of the frame
int launch_yuv420_to_rgb16(const void* yuv, uint16_t* rgb, int B, int H, int W, uint32_t flags, cudaStream_t s);
int launch_rgb16_to_yuv420(const uint16_t* rgb, void* yuv, int B, int H, int W, uint32_t flags, cudaStream_t s);

ConvTcTune to_tune(const mz_conv_tune* t);
int current_device();
bool dtype_ok(int d);
// OIHW fp32 -> [tap = ky*3+kx][cout_p][cin_p] fp16 | bf16, zero padded (host).  Returns false when a weight does not
// fit the fp16 operand range (|w| > 65504 or not finite) -- it would be clipped silently.
bool pack_conv_weight_host(const float* w, int cout, int cin, int cout_p, int cin_p, int bf16,
                           std::vector<uint16_t>& out);
// The same on the device (w_dev fp32 OIHW -> out_dev); an out-of-range fp16 weight sets *sat (may be nullptr).
int launch_pack_conv_weight(const float* w_dev, uint16_t* out_dev, int cout, int cin, int cout_p, int cin_p, int bf16,
                            unsigned int* sat, cudaStream_t s);

#ifdef __CUDACC__
// ----------------------------------------------------------------------------------------------
// device-side epilogues
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_global_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// mode 1 with the residual row already in registers: zf += acc ; zb = round16(zf) for channels n0..n0+15.
__device__ __forceinline__ void epi_residual16(const EpiParams& p, int b, int y, int x, int n0, const float (&acc)[16],
                                               const float4* zin) {
  const size_t pix = (static_cast<size_t>(b) * p.H + y) * p.W + x;
  float4* zf = reinterpret_cast<float4*>(p.zf + pix * (p.zf_pitch ? p.zf_pitch : p.n_pad) + n0);
  uint32_t o[8];
  float amax = 0.f;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float4 z = zin[q];
    z.x += acc[4 * q + 0];
    z.y += acc[4 * q + 1];
    z.z += acc[4 * q + 2];
    z.w += acc[4 * q + 3];
    if (n0 + 4 * q < (p.zf_extent ? p.zf_extent : p.n_pad)) zf[q] = z;
    amax = fmaxf(fmaxf(amax, fmaxf(fabsf(z.x), fabsf(z.y))), fmaxf(fabsf(z.z), fabsf(z.w)));
    o[2 * q] = pack_op2(p.bf16, z.x, z.y);
    o[2 * q + 1] = pack_op2(p.bf16, z.z, z.w);
  }
  if (!p.bf16 && p.sat != nullptr && !(amax <= MZ_F16_MAX)) *p.sat = 1u;
  uint16_t* dst = p.out_bf16 + pix * (p.out_pitch ? p.out_pitch : p.n_pad) + n0;
  const int oe = p.out_extent ? p.out_extent : p.n_pad;
  if (n0 < oe) st_global_v4(dst, o[0], o[1], o[2], o[3]);
  if (n0 + 8 < oe) st_global_v4(dst + 8, o[4], o[5], o[6], o[7]);
}

// modes 0 and 1: sixteen consecutive output channels n0..n0+15 of pixel (b, y, x).  `film_rows` (mode 0) points at
// [scale row | shift row], each n_pad floats, of image b -- shared memory in the tcgen05 kernel, global otherwise;
// nullptr = identity.
template <int MODE>
__device__ __forceinline__ void epi_store16(const EpiParams& p, int b, int y, int x, int n0, float (&acc)[16],
                                            const float* film_rows) {
  const size_t pix = (static_cast<size_t>(b) * p.H + y) * p.W + x;
  if (MODE == 0) {
    if (film_rows != nullptr) {
      const float4* sc = reinterpret_cast<const float4*>(film_rows + n0);
      const float4* sh = reinterpret_cast<const float4*>(film_rows + p.n_pad + n0);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 a = sc[q], c = sh[q];
        acc[4 * q + 0] = fmaf(acc[4 * q + 0], a.x, c.x);
        acc[4 * q + 1] = fmaf(acc[4 * q + 1], a.y, c.y);
        acc[4 * q + 2] = fmaf(acc[4 * q + 2], a.z, c.z);
        acc[4 * q + 3] = fmaf(acc[4 * q + 3], a.w, c.w);
      }
    }
    uint32_t o[8];
    float amax = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float s0 = silu_f(acc[2 * q]), s1 = silu_f(acc[2 * q + 1]);
      amax = fmaxf(amax, fmaxf(fabsf(s0), fabsf(s1)));
      o[q] = pack_op2(p.bf16, s0, s1);
    }
    if (!p.bf16 && p.sat != nullptr && !(amax <= MZ_F16_MAX)) *p.sat = 1u;
    uint16_t* dst = p.out_bf16 + pix * (p.out_pitch ? p.out_pitch : p.n_pad) + n0;
    const int oe = p.out_extent ? p.out_extent : p.n_pad;
    if (n0 < oe) st_global_v4(dst, o[0], o[1], o[2], o[3]);
    if (n0 + 8 < oe) st_global_v4(dst + 8, o[4], o[5], o[6], o[7]);
  } else {
    const float4* zf = reinterpret_cast<const float4*>(p.zf + pix * (p.zf_pitch ? p.zf_pitch : p.n_pad) + n0);
    float4 zin[4];
#pragma unroll
    for (int q = 0; q < 4; ++q)
      zin[q] = n0 + 4 * q < (p.zf_extent ? p.zf_extent : p.n_pad) ? zf[q] : make_float4(0.f, 0.f, 0.f, 0.f);
    epi_residual16(p, b, y, x, n0, acc, zin);
  }
}

// LR pixel as float: fp32 planes as they are, 8-bit planes scaled by 1/255 (ToDtype(float32, scale=True))
__device__ __forceinline__ float lr_px(const float* p) { return __ldg(p); }
__device__ __forceinline__ float lr_px(const uint8_t* p) { return static_cast<float>(__ldg(p)) * (1.0f / 255.0f); }
// 16-bit planes: exactly the IEEE quotient x16 / 65535 -- what the stem computes with __fdiv_rn, so that a 16-bit call
// equals the fp32 call on x16.float() / 65535 bit for bit.  A reciprocal multiply and one FMA correction (the residual
// x - 65535 q is exact); checked against the quotient for all 65536 codes on the CPU (tests/test_gpu_u16_io.py).  The
// product alone is 1 ulp off for 512 codes.
__device__ __forceinline__ float lr_px(const uint16_t* p) {
  constexpr float kRcp = 1.0f / 65535.0f;
  const float x = static_cast<float>(__ldg(p)), q = __fmul_rn(x, kRcp);
  return fmaf(fmaf(-q, 65535.f, x), kRcp, q);
}
// [0,1] -> 8 bits: floor(255 v + 0.5) (save_image) or floor(255 v) (ToPILImage); v is clamped here in any case
__device__ __forceinline__ uint8_t to_u8(float v, int trunc) {
  v = fminf(fmaxf(v, 0.f), 1.f);
  return static_cast<uint8_t>(static_cast<int>(fmaf(v, 255.f, trunc ? 0.f : 0.5f)));
}
// [0,1] -> 16 bits: floor(65535 v + 0.5), one fmaf then truncation as to_u8; v is clamped here
__device__ __forceinline__ uint16_t to_u16(float v) {
  v = fminf(fmaxf(v, 0.f), 1.f);
  return static_cast<uint16_t>(static_cast<int>(fmaf(v, 65535.f, 0.5f)));
}
__device__ __forceinline__ uint32_t pack_u16x2(uint16_t lo, uint16_t hi) {
  return static_cast<uint32_t>(lo) | (static_cast<uint32_t>(hi) << 16);
}
// R contiguous values v of the HR image, quantised to T and stored at element d of y: fp32 clamped when clamp01 is set,
// 8 and 16 bits always (to_u8 / to_u16).  R = 2 or 4 leave in one vector store (fp32: float2 / float4; 8 bits:
// u16 / u32; 16 bits: u32 / 8 bytes), any other R element by element.
template <typename T, int R>
__device__ __forceinline__ void store_px(const ImageIo& io, size_t d, const float* v) {
  T* dst = static_cast<T*>(io.y) + d;
  if constexpr (std::is_same_v<T, float>) {
    float q[R];
#pragma unroll
    for (int j = 0; j < R; ++j) q[j] = io.clamp01 ? fminf(fmaxf(v[j], 0.f), 1.f) : v[j];
    if constexpr (R == 4) {
      *reinterpret_cast<float4*>(dst) = make_float4(q[0], q[1], q[2], q[3]);
    } else if constexpr (R == 2) {
      *reinterpret_cast<float2*>(dst) = make_float2(q[0], q[1]);
    } else {
#pragma unroll
      for (int j = 0; j < R; ++j) dst[j] = q[j];
    }
  } else if constexpr (std::is_same_v<T, uint8_t>) {
    uint32_t w = 0;
#pragma unroll
    for (int j = 0; j < R; ++j) w |= static_cast<uint32_t>(to_u8(v[j], io.u8_trunc)) << (8 * j);
    if constexpr (R == 4) {
      *reinterpret_cast<uint32_t*>(dst) = w;
    } else if constexpr (R == 2) {
      *reinterpret_cast<uint16_t*>(dst) = static_cast<uint16_t>(w);
    } else {
#pragma unroll
      for (int j = 0; j < R; ++j) dst[j] = static_cast<uint8_t>(w >> (8 * j));
    }
  } else {
    static_assert(std::is_same_v<T, uint16_t>, "HR images are fp32, 8 or 16 bits");
    uint16_t q[R];
#pragma unroll
    for (int j = 0; j < R; ++j) q[j] = to_u16(v[j]);
    if constexpr (R == 4) {
      *reinterpret_cast<uint2*>(dst) = make_uint2(pack_u16x2(q[0], q[1]), pack_u16x2(q[2], q[3]));
    } else if constexpr (R == 2) {
      *reinterpret_cast<uint32_t*>(dst) = pack_u16x2(q[0], q[1]);
    } else {
#pragma unroll
      for (int j = 0; j < R; ++j) dst[j] = q[j];
    }
  }
}
// store_px with the output type chosen by the caller's kernel: 16 bits when o16 (a compile-time constant in the tcgen05
// heads, whose LAY bit 2 selects 16-bit images), otherwise 8 bits or fp32 as io.type says (a runtime branch)
template <int R>
__device__ __forceinline__ void store_out(const ImageIo& io, size_t d, const float* v, bool o16) {
  if (o16)
    store_px<uint16_t, R>(io, d, v);
  else if (io.type == kImgU8)
    store_px<uint8_t, R>(io, d, v);
  else
    store_px<float, R>(io, d, v);
}

// Bicubic value of HR pixel (oy, ox) of one colour (H x W, fp32 | u8 | u16, pixels `ps` elements apart: 1 planar, 3
// interleaved): 16 clamped taps, rows first.
template <typename T>
__device__ __forceinline__ float bicubic_at(const T* __restrict__ plane, int H, int W, int ps, const BicubicTable& bt,
                                            int oy, int ox) {
  const int r = bt.r;
  const int py = oy % r, px = ox % r;
  const int by = oy / r + bt.off[py] - 1, bx = ox / r + bt.off[px] - 1;
  float acc = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int yy = min(max(by + k, 0), H - 1);
    const T* row = plane + static_cast<size_t>(yy) * W * ps;
    float h = 0.f;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const int xx = min(max(bx + m, 0), W - 1);
      h = fmaf(lr_px(row + static_cast<size_t>(xx) * ps), bt.w[px][m], h);
    }
    acc = fmaf(h, bt.w[py][k], acc);
  }
  return acc;
}

// mode 2: all head channels of LR pixel (b, y, x): acc[n], n = c*r*r + i*r + j  ->  y[b, c, y*r+i, x*r+j]
// (PixelShuffle index rule, reference model.py:911,928) plus the global skip (model.py:162) and the clamp
// of upscale() (model.py:177).
template <int NMAX>
__device__ __forceinline__ void epi_head(const EpiParams& p, int b, int y, int x, const float (&acc)[NMAX]) {
  const int r = p.r, rr = r * r;
#pragma unroll
  for (int n = 0; n < NMAX; ++n) {
    if (n < 3 * rr) {
      const int c = n / rr, i = (n % rr) / r, j = n % r;
      const int oy = y * r + i, ox = x * r + j;
      const long long di = head_out_index(p, b, c, y, x, i, j);
      if (di < 0) continue;
      float v = acc[n];
      if (p.img.skip_mode == 1) {
        v += static_cast<const float*>(p.img.y)[di];
      } else if (p.img.skip_mode == 2) {
        const size_t HW = static_cast<size_t>(p.H) * p.W;
        const size_t pl = p.img.x_nhwc ? static_cast<size_t>(b) * 3 * HW + c : (static_cast<size_t>(b) * 3 + c) * HW;
        const int ps = p.img.x_nhwc ? 3 : 1;
        v += p.img.type == kImgU16 ? bicubic_at(static_cast<const uint16_t*>(p.img.x) + pl, p.H, p.W, ps, p.bt, oy, ox)
             : p.img.type == kImgU8 ? bicubic_at(static_cast<const uint8_t*>(p.img.x) + pl, p.H, p.W, ps, p.bt, oy, ox)
                                    : bicubic_at(static_cast<const float*>(p.img.x) + pl, p.H, p.W, ps, p.bt, oy, ox);
      }
      store_out<1>(p.img, di, &v, p.img.type == kImgU16);
    }
  }
}
// One interleaved HR row segment of an LR pixel: v = R pixels x 3 colours at element d, as three stores of R values
template <int R, bool O16>
__device__ __forceinline__ void store_hr_row_nhwc(const ImageIo& io, size_t d, const float (&v)[3 * R]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) store_out<R>(io, d + k * R, v + k * R, O16);
}

// Same as epi_head with the ratio known at compile time: the 5x5 LR neighbourhood of the pixel is loaded once per
// colour, interpolated horizontally for the R phases (5 rows x R values) and then vertically (R x R values) --
// 25 loads + 20R + 4R^2 FMAs per colour instead of 16 loads + 20 FMAs per HR pixel -- and every HR row segment of
// the pixel (R contiguous floats) leaves in one vector store, so a warp writes 32*R contiguous floats.
// The epilogue warps are few (two per scheduler) and this code is latency-bound, so: the skip source's type is a
// template parameter (one load per tap instead of a predicated fp32 / 8-bit pair), the clamped row / column offsets
// are computed once for the three colours, and at R = 2 all 75 taps (R > 2: the 25 of a colour) are requested before
// the first FMA; skip-from-buffer reads all its row segments before the first store (a store to y orders every
// later load from y behind it).  Columns are only clamped in the first and last warp of an image row: the others
// (interior) read each neighbourhood row through one pointer with immediate offsets.
// XN / YN: interleaved input / output (ImageIo::x_nhwc / y_nhwc) -- compile-time, so that the planar instantiation is
// the code it was.  Interleaved, the taps of one colour are 3 elements apart (same FMA order per colour: bit-identical
// results) and each HR row of the pixel leaves as 3R contiguous values.
// T = uint16_t: 16-bit images on both sides (MZ_FLAG_IO_U16) -- the 16-bit heads are instantiations of their own.
template <int R, typename T, bool XN, bool YN>
__device__ __forceinline__ void epi_head_rt(const EpiParams& p, const T* __restrict__ lr, int b, int y, int x,
                                            const float (&acc)[48], bool interior) {
  constexpr bool O16 = std::is_same_v<T, uint16_t>;
  const int H = p.H, W = p.W;
  const long long first = head_out_index_l<YN>(p, b, 0, y, x, 0, 0);
  if (first < 0) return;  // outside the output window
  const size_t row_pitch = p.img.y_row ? static_cast<size_t>(p.img.y_row) : static_cast<size_t>(W) * R * (YN ? 3 : 1);
  const size_t plane_pitch = p.img.y_plane ? static_cast<size_t>(p.img.y_plane) : static_cast<size_t>(H) * R * W * R;
  constexpr int NC = (R == 2) ? 3 : 1;  // colours whose taps are in flight together
  constexpr int PS = XN ? 3 : 1;        // elements between horizontally adjacent LR pixels of one colour
  float out[3][R][R];
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
      for (int j = 0; j < R; ++j) out[c][i][j] = acc[c * R * R + i * R + j];

  if (p.img.skip_mode == 2) {
    const size_t HW = static_cast<size_t>(H) * W;
    const T* img = lr + static_cast<size_t>(b) * 3 * HW;
    int xo[5], ro[5];  // (a colour plane is below 2^31 pixels: prepare_conv_tc checks; an interleaved image is below
                       // 2^31 elements: upscale_impl checks)
#pragma unroll
    for (int m = 0; m < 5; ++m) xo[m] = min(max(x - 2 + m, 0), W - 1) * PS;
#pragma unroll
    for (int k = 0; k < 5; ++k) ro[k] = min(max(y - 2 + k, 0), H - 1) * W * PS;
#pragma unroll
    for (int c0 = 0; c0 < 3; c0 += NC) {
      float nb[NC][5][5];
#pragma unroll
      for (int cc = 0; cc < NC; ++cc) {
        const T* pl = img + (XN ? (c0 + cc) : (c0 + cc) * HW);
        if (interior) {  // warp-uniform: no column of the warp's neighbourhoods is clamped -> one pointer per row
#pragma unroll
          for (int k = 0; k < 5; ++k) {
            const T* rp = pl + (ro[k] + (x - 2) * PS);
#pragma unroll
            for (int m = 0; m < 5; ++m) nb[cc][k][m] = lr_px(rp + m * PS);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 5; ++k)
#pragma unroll
            for (int m = 0; m < 5; ++m) nb[cc][k][m] = lr_px(pl + (ro[k] + xo[m]));
        }
      }
#pragma unroll
      for (int cc = 0; cc < NC; ++cc) {
        float hz[5][R];
#pragma unroll
        for (int k = 0; k < 5; ++k)
#pragma unroll
          for (int j = 0; j < R; ++j) {
            const int s = (2 * j + 1 < R) ? 0 : 1;  // first tap relative to x-2 (phase offset -1 or 0)
            float a = 0.f;
#pragma unroll
            for (int m = 0; m < 4; ++m) a = fmaf(nb[cc][k][s + m], p.bt.w[j][m], a);
            hz[k][j] = a;
          }
#pragma unroll
        for (int i = 0; i < R; ++i) {
          const int s = (2 * i + 1 < R) ? 0 : 1;
#pragma unroll
          for (int j = 0; j < R; ++j) {
            float a = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) a = fmaf(hz[s + k][j], p.bt.w[i][k], a);
            out[c0 + cc][i][j] += a;
          }
        }
      }
    }
  }

  if constexpr (YN) {  // (no skip-from-buffer: the API refuses it with interleaved images)
#pragma unroll
    for (int i = 0; i < R; ++i) {
      float v[3 * R];
#pragma unroll
      for (int j = 0; j < R; ++j)
#pragma unroll
        for (int c = 0; c < 3; ++c) v[3 * j + c] = out[c][i][j];
      store_hr_row_nhwc<R, O16>(p.img, static_cast<size_t>(first) + static_cast<size_t>(i) * row_pitch, v);
    }
    return;
  }
  // y already holds the bicubic image (fp32: 8 and 16 bits recompute the skip): all of this pixel's segments first,
  // then the stores
  if (!O16 && p.img.skip_mode == 1) {
    const float* dst = static_cast<const float*>(p.img.y) + static_cast<size_t>(first);
    float sk[3][R][R];
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < R; ++i) {
        const float* rowp = dst + c * plane_pitch + static_cast<size_t>(i) * row_pitch;
        if (R == 4) {
          const float4 v = *reinterpret_cast<const float4*>(rowp);
          sk[c][i][0] = v.x, sk[c][i][1] = v.y, sk[c][i][R > 2 ? 2 : 0] = v.z, sk[c][i][R - 1] = v.w;
        } else if (R == 2) {
          const float2 v = *reinterpret_cast<const float2*>(rowp);
          sk[c][i][0] = v.x, sk[c][i][1] = v.y;
        } else {
#pragma unroll
          for (int j = 0; j < R; ++j) sk[c][i][j] = rowp[j];
        }
      }
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < R; ++j) out[c][i][j] += sk[c][i][j];
  }
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int i = 0; i < R; ++i)
      store_out<R>(p.img, static_cast<size_t>(first) + c * plane_pitch + static_cast<size_t>(i) * row_pitch, out[c][i], O16);
}
// interior: warp-uniform promise that x - 2 >= 0 and x + 2 < W for every lane of the calling warp
// (the layouts and the 16-bit image type, I16, are template parameters of the calling kernel: one runtime branch over
// four layouts in the same kernel raises the planar head's registers and makes it spill)
template <int R, bool XN, bool YN, bool I16>
__device__ __forceinline__ void epi_head_r(const EpiParams& p, int b, int y, int x, const float (&acc)[48], bool interior) {
  if constexpr (I16)
    epi_head_rt<R, uint16_t, XN, YN>(p, static_cast<const uint16_t*>(p.img.x), b, y, x, acc, interior);
  else if (p.img.type == kImgU8)
    epi_head_rt<R, uint8_t, XN, YN>(p, static_cast<const uint8_t*>(p.img.x), b, y, x, acc, interior);
  else
    epi_head_rt<R, float, XN, YN>(p, static_cast<const float*>(p.img.x), b, y, x, acc, interior);
}
// r = 2, TWO vertically adjacent LR pixels (y, x) and (y + 1, x) per thread: their 5x5 neighbourhoods share four of
// five rows, so the pair costs 6 x 5 loads and 6 x 2 horizontal interpolations per colour instead of 2 x (5 x 5) and
// 2 x (5 x 2), and -- what matters for the latency-bound epilogue warps -- ONE exposed load latency instead of two.
// Same FMA order per output as epi_head_rt<2>: the results are bit-identical.  v0 / v1: the twelve head channels of the
// two pixels as they come out of TMEM; second: row y + 1 exists (y + 1 < H).  XN / YN as in epi_head_rt.
template <typename T, bool XN, bool YN>
__device__ __forceinline__ void epi_head2_pair(const EpiParams& p, const T* __restrict__ lr, int b, int y, int x,
                                               const uint32_t (&v0)[16], const uint32_t (&v1)[16], bool interior,
                                               bool second) {
  constexpr bool O16 = std::is_same_v<T, uint16_t>;  // 16-bit images on both sides, as in epi_head_rt
  const int H = p.H, W = p.W;
  long long first[2];
  first[0] = head_out_index_l<YN>(p, b, 0, y, x, 0, 0);
  first[1] = second ? head_out_index_l<YN>(p, b, 0, y + 1, x, 0, 0) : -1;
  if (first[0] < 0 && first[1] < 0) return;  // both outside the output window
  const size_t row_pitch = p.img.y_row ? static_cast<size_t>(p.img.y_row) : static_cast<size_t>(W) * 2 * (YN ? 3 : 1);
  constexpr int PS = XN ? 3 : 1;  // elements between horizontally adjacent LR pixels of one colour
  const size_t plane_pitch = p.img.y_plane ? static_cast<size_t>(p.img.y_plane) : static_cast<size_t>(H) * 2 * W * 2;
  float out[2][3][2][2];
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        out[0][c][i][j] = __uint_as_float(v0[c * 4 + i * 2 + j]);
        out[1][c][i][j] = __uint_as_float(v1[c * 4 + i * 2 + j]);
      }
  if (p.img.skip_mode == 2) {
    const size_t HW = static_cast<size_t>(H) * W;
    const T* img = lr + static_cast<size_t>(b) * 3 * HW;
    int xo[5], ro[6];
#pragma unroll
    for (int m = 0; m < 5; ++m) xo[m] = min(max(x - 2 + m, 0), W - 1) * PS;
#pragma unroll
    for (int k = 0; k < 6; ++k) ro[k] = min(max(y - 2 + k, 0), H - 1) * W * PS;
    float nb[3][6][5];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const T* pl = img + (XN ? c : c * HW);
      if (interior) {
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          const T* rp = pl + (ro[k] + (x - 2) * PS);
#pragma unroll
          for (int m = 0; m < 5; ++m) nb[c][k][m] = lr_px(rp + m * PS);
        }
      } else {
#pragma unroll
        for (int k = 0; k < 6; ++k)
#pragma unroll
          for (int m = 0; m < 5; ++m) nb[c][k][m] = lr_px(pl + (ro[k] + xo[m]));
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float hz[6][2];
#pragma unroll
      for (int k = 0; k < 6; ++k)
#pragma unroll
        for (int j = 0; j < 2; ++j) {  // phase j: first tap at x - 2 + j
          float a = 0.f;
#pragma unroll
          for (int m = 0; m < 4; ++m) a = fmaf(nb[c][k][j + m], p.bt.w[j][m], a);
          hz[k][j] = a;
        }
#pragma unroll
      for (int rr = 0; rr < 2; ++rr)
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j) {  // pixel row y + rr, phase i: first tap at LR row y + rr - 2 + i
            float a = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) a = fmaf(hz[rr + i + k][j], p.bt.w[i][k], a);
            out[rr][c][i][j] += a;
          }
    }
  }
  if constexpr (YN) {  // (no skip-from-buffer: the API refuses it with interleaved images)
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      if (first[rr] < 0) continue;
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        float v[6];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int c = 0; c < 3; ++c) v[3 * j + c] = out[rr][c][i][j];
        store_hr_row_nhwc<2, O16>(p.img, static_cast<size_t>(first[rr]) + static_cast<size_t>(i) * row_pitch, v);
      }
    }
    return;
  }
  if (!O16 && p.img.skip_mode == 1) {  // y already holds the bicubic image (fp32): every segment is read before the first store
    const float* sy = static_cast<const float*>(p.img.y);
    float2 sk[2][3][2];
#pragma unroll
    for (int rr = 0; rr < 2; ++rr)
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < 2; ++i)
          sk[rr][c][i] = first[rr] < 0 ? make_float2(0.f, 0.f)
                                       : *reinterpret_cast<const float2*>(sy + static_cast<size_t>(first[rr]) + c * plane_pitch +
                                                                          static_cast<size_t>(i) * row_pitch);
#pragma unroll
    for (int rr = 0; rr < 2; ++rr)
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          out[rr][c][i][0] += sk[rr][c][i].x;
          out[rr][c][i][1] += sk[rr][c][i].y;
        }
  }
#pragma unroll
  for (int rr = 0; rr < 2; ++rr) {
    if (first[rr] < 0) continue;
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < 2; ++i)
        store_out<2>(p.img, static_cast<size_t>(first[rr]) + c * plane_pitch + static_cast<size_t>(i) * row_pitch,
                     out[rr][c][i], O16);
  }
}
template <bool XN, bool YN, bool I16>
__device__ __forceinline__ void epi_head2(const EpiParams& p, int b, int y, int x, const uint32_t (&v0)[16],
                                          const uint32_t (&v1)[16], bool interior, bool second) {
  if constexpr (I16)
    epi_head2_pair<uint16_t, XN, YN>(p, static_cast<const uint16_t*>(p.img.x), b, y, x, v0, v1, interior, second);
  else if (p.img.type == kImgU8)
    epi_head2_pair<uint8_t, XN, YN>(p, static_cast<const uint8_t*>(p.img.x), b, y, x, v0, v1, interior, second);
  else
    epi_head2_pair<float, XN, YN>(p, static_cast<const float*>(p.img.x), b, y, x, v0, v1, interior, second);
}
#endif  // __CUDACC__

}  // namespace mz
