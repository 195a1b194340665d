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
  const void* x;  // LR image (B,nc,H,W), nc = EpiParams::nc
  void* y;        // HR image (B,nc,rH,rW)
  int type;       // ImageType
  // Interleaved images (MZ_FLAG_X_NHWC / MZ_FLAG_Y_NHWC): x is (B,H,W,nc), y is (B,rH,rW,nc) -- channel c of a pixel at
  // pixel * nc + c, images nc HW (nc rH rW) elements apart as in the planar layout.
  int x_nhwc, y_nhwc;
  int u8_trunc;
  int skip_mode;  // 0 none, 1 y already holds the bicubic image (fp32 only), 2 recompute bicubic from x
  int clamp01;
  // Windowed output (mz_upscale_window; all zero = the whole image, densely): only LR pixels wy0 <= y < wy1,
  // wx0 <= x < wx1 are stored, pixel (wy0, wx0) of plane 0 of image 0 at y itself, HR rows y_row elements and colour
  // planes y_plane elements apart (images nc planes) -- a tile's core written straight into an assembled (possibly
  // remote) frame.  For an
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
  // mode 2: the images (a prepared launch takes them from each call: patch_conv_epi), the ratio, their channel count and
  // the bicubic table
  ImageIo img;
  int r;
  // Channels per pixel of both images: 3 (RGB) or 4 (RGBA, MZ_FLAG_RGBA: colour 0..2, then a straight alpha that the
  // network never reads; the head writes its bicubic resampling -- a colour skip's arithmetic started from 0 instead of
  // the accumulator).  Part of the images (patch_conv_epi replaces it with img), kept here, in what was padding after r,
  // so that every field the RGB kernels read stays where it was.
  int nc;
  // fp16 range guard: a kernel that is about to round a value beyond +-65504 into a 16-bit fp16 operand (where
  // cvt.rn.satfinite would clip it silently) writes 1 here.  Points at a host-mapped word owned by the mz_model
  // (mz_model_saturated); nullptr = not tracked (per-kernel entry points).
  unsigned int* sat;
  BicubicTable bt;
};

// largest finite fp16: a pre-rounding magnitude above it saturates the operand
#define MZ_F16_MAX 65504.0f

// address of channel c of HR pixel (y r + i, x r + j) of image b in the output of mode 2, or -1 outside the window;
// YN: interleaved output (ImageIo::y_nhwc); CH: channels per pixel (EpiParams::nc)
template <bool YN, int CH = 3>
__host__ __device__ inline long long head_out_index_l(const EpiParams& p, int b, int c, int y, int x, int i, int j) {
  const ImageIo& io = p.img;
  const long long WR = static_cast<long long>(p.W) * p.r, HR = static_cast<long long>(p.H) * p.r;
  if (io.wy1 > 0 && (y < io.wy0 || y >= io.wy1 || x < io.wx0 || x >= io.wx1)) return -1;
  if (YN) {
    const long long row = io.y_row ? io.y_row : CH * WR, img = io.y_plane ? io.y_plane : CH * HR * WR;
    return static_cast<long long>(b) * img + (static_cast<long long>(y - io.wy0) * p.r + i) * row +
           (static_cast<long long>(x - io.wx0) * p.r + j) * CH + c;
  }
  const long long row = io.y_row ? io.y_row : WR, plane = io.y_plane ? io.y_plane : HR * WR;
  return (static_cast<long long>(b) * CH + c) * plane + (static_cast<long long>(y - io.wy0) * p.r + i) * row +
         static_cast<long long>(x - io.wx0) * p.r + j;
}
__host__ __device__ inline long long head_out_index(const EpiParams& p, int b, int c, int y, int x, int i, int j) {
  if (p.nc == 4)
    return p.img.y_nhwc ? head_out_index_l<true, 4>(p, b, c, y, x, i, j) : head_out_index_l<false, 4>(p, b, c, y, x, i, j);
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
// head (mode 2) only: replace the images (EpiParams::img and nc) of a prepared launch (a new layout or channel count
// swaps the kernel instantiation)
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
// image x (element type `type`, interleaved when x_nhwc, nc = 3 or 4 channels: as ImageIo; colour 0..2 only is read)
// -> fp32 stream zf + 16-bit shadow zb (pitch zb_pitch)
int launch_stem(const void* x, int type, int x_nhwc, int nc, const float* w, const float* bias, float* zf, uint16_t* zb,
                int bf16, int B, int H, int W, int Cp, int zb_pitch, cudaStream_t s, unsigned int* sat = nullptr);
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
// u16 / u32; 16 bits: u32 / 8 bytes), any other R up to 4 element by element.  R = 8, 12, 16 (an interleaved RGBA row
// segment of a pixel at r = 2, 3, 4) are packed into 32-bit words and leave in the widest vectors that divide their
// R * sizeof(T) bytes, up to 16: fp32 in 16-byte stores; 16 bits in 16-byte stores at R = 8 and 16, 8-byte ones at
// R = 12; 8 bits in one 8-byte store at R = 8, three 4-byte ones at R = 12 and one 16-byte store at R = 16.
template <typename T, int R>
__device__ __forceinline__ void store_px(const ImageIo& io, size_t d, const float* v) {
  T* dst = static_cast<T*>(io.y) + d;
  if constexpr (R > 4) {
    static_assert(R % 4 == 0, "a wide run is whole RGBA pixels");
    constexpr int NW = R * static_cast<int>(sizeof(T)) / 4;  // 32-bit words of the run
    constexpr int VB = (NW % 4 == 0) ? 16 : ((NW % 2 == 0) ? 8 : 4);
    uint32_t w[NW];
#pragma unroll
    for (int k = 0; k < NW; ++k) {
      if constexpr (std::is_same_v<T, float>) {
        w[k] = __float_as_uint(io.clamp01 ? fminf(fmaxf(v[k], 0.f), 1.f) : v[k]);
      } else if constexpr (std::is_same_v<T, uint8_t>) {
        w[k] = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) w[k] |= static_cast<uint32_t>(to_u8(v[4 * k + q], io.u8_trunc)) << (8 * q);
      } else {
        static_assert(std::is_same_v<T, uint16_t>, "HR images are fp32, 8 or 16 bits");
        w[k] = pack_u16x2(to_u16(v[2 * k]), to_u16(v[2 * k + 1]));
      }
    }
    char* b = reinterpret_cast<char*>(dst);
#pragma unroll
    for (int k = 0; k < NW; k += VB / 4) {
      if constexpr (VB == 16)
        *reinterpret_cast<uint4*>(b + 4 * k) = make_uint4(w[k], w[k + 1], w[k + 2], w[k + 3]);
      else if constexpr (VB == 8)
        *reinterpret_cast<uint2*>(b + 4 * k) = make_uint2(w[k], w[k + 1]);
      else
        *reinterpret_cast<uint32_t*>(b + 4 * k) = w[k];
    }
  } else if constexpr (std::is_same_v<T, float>) {
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

// Bicubic value of HR pixel (oy, ox) of one channel (H x W, fp32 | u8 | u16, pixels `ps` elements apart: 1 planar, 3
// or 4 interleaved): 16 clamped taps, rows first.
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

// skip of channel c at HR pixel (oy, ox) of image b, read from x in its element type and layout (epi_head)
__device__ __forceinline__ float head_skip_at(const EpiParams& p, int b, int c, int oy, int ox) {
  const int nc = p.nc == 4 ? 4 : 3;
  const size_t HW = static_cast<size_t>(p.H) * p.W;
  const size_t pl = p.img.x_nhwc ? static_cast<size_t>(b) * nc * HW + c : (static_cast<size_t>(b) * nc + c) * HW;
  const int ps = p.img.x_nhwc ? nc : 1;
  return p.img.type == kImgU16 ? bicubic_at(static_cast<const uint16_t*>(p.img.x) + pl, p.H, p.W, ps, p.bt, oy, ox)
         : p.img.type == kImgU8 ? bicubic_at(static_cast<const uint8_t*>(p.img.x) + pl, p.H, p.W, ps, p.bt, oy, ox)
                                : bicubic_at(static_cast<const float*>(p.img.x) + pl, p.H, p.W, ps, p.bt, oy, ox);
}
// mode 2: all head channels of LR pixel (b, y, x): acc[n], n = c*r*r + i*r + j  ->  y[b, c, y*r+i, x*r+j]
// (PixelShuffle index rule, reference model.py:911,928) plus the global skip (model.py:162) and the clamp
// of upscale() (model.py:177).  An RGBA image's alpha (EpiParams::nc == 4) is the skip alone, channel 3's bicubic
// resampling with no accumulator (a loop over its r*r phases at run time).
template <int NMAX>
__device__ __forceinline__ void epi_head(const EpiParams& p, int b, int y, int x, const float (&acc)[NMAX]) {
  const int r = p.r, rr = r * r;
#pragma unroll
  for (int n = 0; n < NMAX; ++n) {
    if (n < 3 * rr) {
      const int c = n / rr, i = (n % rr) / r, j = n % r;
      const long long di = head_out_index(p, b, c, y, x, i, j);
      if (di < 0) continue;
      float v = acc[n];
      if (p.img.skip_mode == 1)
        v += static_cast<const float*>(p.img.y)[di];
      else if (p.img.skip_mode == 2)
        v += head_skip_at(p, b, c, y * r + i, x * r + j);
      store_out<1>(p.img, di, &v, p.img.type == kImgU16);
    }
  }
  if (p.nc == 4 && p.img.skip_mode == 2) {  // (RGBA recomputes the skip: check_image_flags)
    for (int n = 0; n < rr; ++n) {
      const int i = n / r, j = n % r;
      const long long di = head_out_index(p, b, 3, y, x, i, j);
      if (di < 0) continue;
      const float v = head_skip_at(p, b, 3, y * r + i, x * r + j);
      store_out<1>(p.img, di, &v, p.img.type == kImgU16);
    }
  }
}
// One interleaved HR row segment of an LR pixel: v = R pixels x CH channels at element d -- RGB as three stores of R
// values, RGBA (whole pixels, 4R values) as one run in the widest aligned vectors (store_px)
template <int R, bool O16, int CH = 3>
__device__ __forceinline__ void store_hr_row_nhwc(const ImageIo& io, size_t d, const float (&v)[CH * R]) {
  if constexpr (CH == 4) {
    store_out<4 * R>(io, d, v, O16);
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) store_out<R>(io, d + k * R, v + k * R, O16);
  }
}

// ---- the tcgen05 head's epilogue (mode 2) ----
// The epilogue warps are few (two per scheduler) and this code is latency-bound, so: the skip source's type is a
// template parameter (one load per tap instead of a predicated fp32 / 8-bit pair), the clamped row / column offsets are
// computed once per pixel for every colour, at r = 2 all 75 colour taps (pair: 90; r > 2: the 25 of a colour) are
// requested before the first FMA, and columns are only clamped in the first and last warp of an image row: the others
// (interior) read each neighbourhood row through one pointer with immediate offsets.

// Clamped offsets of the NR x 5 LR neighbourhood of pixel (y, x) -- rows y - 2 .. y + NR - 3, columns x - 2 .. x + 2 --
// in elements from the start of a channel plane whose pixels are PS elements apart (a colour plane is below 2^31 pixels:
// prepare_conv_tc checks; an interleaved image is below 2^31 elements: upscale_impl checks)
template <int NR, int PS>
struct NbOffsets {
  int ro[NR], xo[5];
  __device__ __forceinline__ NbOffsets(int y, int x, int H, int W) {
#pragma unroll
    for (int m = 0; m < 5; ++m) xo[m] = min(max(x - 2 + m, 0), W - 1) * PS;
#pragma unroll
    for (int k = 0; k < NR; ++k) ro[k] = min(max(y - 2 + k, 0), H - 1) * W * PS;
  }
};
// That neighbourhood of channel plane pl as float.  interior: warp-uniform promise that x - 2 >= 0 and x + 2 < W for
// every lane of the calling warp (no column of its neighbourhoods is clamped -> one pointer per row)
template <int NR, int PS, typename T>
__device__ __forceinline__ void load_nb(const T* __restrict__ pl, int x, const NbOffsets<NR, PS>& o, bool interior,
                                        float (&nb)[NR][5]) {
  if (interior) {
#pragma unroll
    for (int k = 0; k < NR; ++k) {
      const T* rp = pl + (o.ro[k] + (x - 2) * PS);
#pragma unroll
      for (int m = 0; m < 5; ++m) nb[k][m] = lr_px(rp + m * PS);
    }
  } else {
#pragma unroll
    for (int k = 0; k < NR; ++k)
#pragma unroll
      for (int m = 0; m < 5; ++m) nb[k][m] = lr_px(pl + (o.ro[k] + o.xo[m]));
  }
}
// Bicubic skip of one channel at ratio R for the P vertically adjacent LR pixels (y + rr, x) whose neighbourhoods are
// the rows of nb (rr + 0 .. rr + 4): the 4 + P rows interpolated horizontally for the R phases, then vertically --
// s[rr][i][j] for HR pixel ((y + rr) R + i, x R + j).  Phase i's first tap is at offset -2 + (2i + 1 < R ? 0 : 1) from
// the pixel, in both directions.  Each sum starts from 0 and takes its four taps in order, so a value is the same FMA
// chain whatever P: two pixels at r = 2 cost 6 x 5 loads and 6 x 2 horizontal interpolations per channel instead of
// 2 x (5 x 5) and 2 x (5 x 2), with one exposed load latency instead of two, and give bit-identical results.
template <int R, int P>
__device__ __forceinline__ void skip_interp(const BicubicTable& bt, const float (&nb)[4 + P][5], float (&s)[P][R][R]) {
  float hz[4 + P][R];
#pragma unroll
  for (int k = 0; k < 4 + P; ++k)
#pragma unroll
    for (int j = 0; j < R; ++j) {
      const int sh = (2 * j + 1 < R) ? 0 : 1;
      float a = 0.f;
#pragma unroll
      for (int m = 0; m < 4; ++m) a = fmaf(nb[k][sh + m], bt.w[j][m], a);
      hz[k][j] = a;
    }
#pragma unroll
  for (int rr = 0; rr < P; ++rr)
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int sh = (2 * i + 1 < R) ? 0 : 1;
#pragma unroll
      for (int j = 0; j < R; ++j) {
        float a = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) a = fmaf(hz[rr + sh + k][j], bt.w[i][k], a);
        s[rr][i][j] = a;
      }
    }
}
// R contiguous fp32 values of an HR image at src: the load counterpart of store_px<float, R> (one float4 / float2 at
// R = 4 / 2, element by element otherwise)
template <int R>
__device__ __forceinline__ void load_px(const float* src, float (&v)[R]) {
  if constexpr (R == 4) {
    const float4 q = *reinterpret_cast<const float4*>(src);
    v[0] = q.x, v[1] = q.y, v[2] = q.z, v[3] = q.w;
  } else if constexpr (R == 2) {
    const float2 q = *reinterpret_cast<const float2*>(src);
    v[0] = q.x, v[1] = q.y;
  } else {
#pragma unroll
    for (int j = 0; j < R; ++j) v[j] = src[j];
  }
}

// The alpha of an RGBA image (EpiParams::nc == 4): the skip of its channel plane pl alone -- a colour's loads and FMAs
// in the same order, each sum started from 0 instead of from the accumulator.  A function of its own, with its plane
// pointer formed at the call rather than by epi_head_t's plane(): written inline or given plane(3), the compiler folds
// the RGBA heads' address arithmetic worse (2-5 % more instructions; 10 % more head time with planar input and
// interleaved output).
template <int R, int P, int PS, typename T>
__device__ __forceinline__ void alpha_skip(const EpiParams& p, const T* __restrict__ pl, int y, int x, bool interior,
                                           float (&al)[P][R][R]) {
  const NbOffsets<4 + P, PS> o(y, x, p.H, p.W);
  float nb[4 + P][5];
  load_nb(pl, x, o, interior, nb);
  skip_interp<R, P>(p.bt, nb, al);
}
// epi_head with the ratio R known at compile time, for P = 1 LR pixel (y, x) (any ratio) or P = 2 vertically adjacent
// pixels (y, x) and (y + 1, x) (r = 2; second: row y + 1 exists).  acc[rr][n]: the head channels of pixel (y + rr, x) as
// they come out of TMEM, n = c R^2 + i R + j for HR pixel ((y + rr) R + i, x R + j) of colour c.  The 5 x 5 (pair:
// 6 x 5) LR neighbourhood is loaded once per colour and interpolated by skip_interp -- 25 loads + 20R + 4R^2 FMAs per
// colour of a pixel instead of 16 loads + 20 FMAs per HR pixel -- and every HR row segment of a pixel (R contiguous
// values) leaves in one vector store, so a warp writes 32R contiguous values.  Skip-from-buffer reads all of a pixel's
// row segments before the first store (a store to y orders every later load from y behind it).
// XN / YN: interleaved input / output (ImageIo::x_nhwc / y_nhwc) -- compile-time, so that the planar instantiation is
// the code it was.  Interleaved, the taps of one colour are CH elements apart (same FMA order per colour: bit-identical
// results) and each HR row of the pixel leaves as CH R contiguous values.
// T = uint16_t: 16-bit images on both sides (MZ_FLAG_IO_U16) -- the 16-bit heads are instantiations of their own.
// CH = 4: RGBA images (EpiParams::nc) -- pixels 4 elements apart when interleaved, images 4 planes apart when planar, and
// the alpha (channel 3's skip alone: skip_interp started from 0 instead of from the accumulator; RGBA always recomputes
// the skip, image_io refuses skip-from-buffer) written beside the colour: interleaved output computes it before the
// stores and leaves every HR row segment of the pixel as one run of 4R values (alpha live with the colour: 4R^2 more
// registers at the peak); planar output computes it after the colour stores, once out is dead, and stores it as a
// fourth plane.
template <int R, int P, typename T, bool XN, bool YN, int CH, int NA>
__device__ __forceinline__ void epi_head_t(const EpiParams& p, const T* __restrict__ lr, int b, int y, int x,
                                           const float (&acc)[P][NA], bool interior, bool second) {
  static_assert(P == 1 || R == 2, "pixel pairs at r = 2 only");
  static_assert(NA >= 3 * R * R, "every colour's R x R accumulators");
  constexpr bool O16 = std::is_same_v<T, uint16_t>;
  const int H = p.H, W = p.W;
  long long first[P];
  first[0] = head_out_index_l<YN, CH>(p, b, 0, y, x, 0, 0);
  if constexpr (P == 2) first[1] = second ? head_out_index_l<YN, CH>(p, b, 0, y + 1, x, 0, 0) : -1;
  if (first[0] < 0 && first[P - 1] < 0) return;  // outside the output window
  const size_t row_pitch = p.img.y_row ? static_cast<size_t>(p.img.y_row) : static_cast<size_t>(W) * R * (YN ? CH : 1);
  const size_t plane_pitch = p.img.y_plane ? static_cast<size_t>(p.img.y_plane) : static_cast<size_t>(H) * R * W * R;
  constexpr int NC = (R == 2) ? 3 : 1;  // colours whose taps are in flight together
  constexpr int PS = XN ? CH : 1;       // elements between horizontally adjacent LR pixels of one channel
  auto plane = [&](int c) {             // channel c of LR image b
    const size_t HW = static_cast<size_t>(H) * W;
    return lr + static_cast<size_t>(b) * CH * HW + (XN ? c : c * HW);
  };
  auto alpha = [&](float (&al)[P][R][R]) {  // (the plane formed here, not by plane(3): see alpha_skip)
    const size_t HW = static_cast<size_t>(H) * W;
    alpha_skip<R, P, PS>(p, lr + static_cast<size_t>(b) * CH * HW + (XN ? 3 : 3 * HW), y, x, interior, al);
  };
  float out[P][3][R][R];
#pragma unroll
  for (int rr = 0; rr < P; ++rr)
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < R; ++i)
#pragma unroll
        for (int j = 0; j < R; ++j) out[rr][c][i][j] = acc[rr][c * R * R + i * R + j];

  if (p.img.skip_mode == 2) {
    const NbOffsets<4 + P, PS> o(y, x, H, W);
#pragma unroll
    for (int c0 = 0; c0 < 3; c0 += NC) {
      float nb[NC][4 + P][5];
#pragma unroll
      for (int cc = 0; cc < NC; ++cc) load_nb(plane(c0 + cc), x, o, interior, nb[cc]);
#pragma unroll
      for (int cc = 0; cc < NC; ++cc) {
        float s[P][R][R];
        skip_interp<R, P>(p.bt, nb[cc], s);
#pragma unroll
        for (int rr = 0; rr < P; ++rr)
#pragma unroll
          for (int i = 0; i < R; ++i)
#pragma unroll
            for (int j = 0; j < R; ++j) out[rr][c0 + cc][i][j] += s[rr][i][j];
      }
    }
  }

  if constexpr (YN) {  // (no skip-from-buffer: the API refuses it with interleaved images)
    float al[P][R][R];
    if constexpr (CH == 4) alpha(al);
#pragma unroll
    for (int rr = 0; rr < P; ++rr) {
      if (first[rr] < 0) continue;
#pragma unroll
      for (int i = 0; i < R; ++i) {
        float v[CH * R];
#pragma unroll
        for (int j = 0; j < R; ++j) {
#pragma unroll
          for (int c = 0; c < 3; ++c) v[CH * j + c] = out[rr][c][i][j];
          if constexpr (CH == 4) v[CH * j + 3] = al[rr][i][j];
        }
        store_hr_row_nhwc<R, O16, CH>(p.img, static_cast<size_t>(first[rr]) + static_cast<size_t>(i) * row_pitch, v);
      }
    }
    return;
  }
  if (!O16 && p.img.skip_mode == 1) {  // y already holds the bicubic image (fp32: 8 and 16 bits recompute the skip)
    const float* sy = static_cast<const float*>(p.img.y);
    float sk[P][3][R][R];
#pragma unroll
    for (int rr = 0; rr < P; ++rr)
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < R; ++i) {
          if (first[rr] < 0) {
#pragma unroll
            for (int j = 0; j < R; ++j) sk[rr][c][i][j] = 0.f;
          } else {
            load_px<R>(sy + static_cast<size_t>(first[rr]) + c * plane_pitch + static_cast<size_t>(i) * row_pitch,
                       sk[rr][c][i]);
          }
        }
#pragma unroll
    for (int rr = 0; rr < P; ++rr)
#pragma unroll
      for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int i = 0; i < R; ++i)
#pragma unroll
          for (int j = 0; j < R; ++j) out[rr][c][i][j] += sk[rr][c][i][j];
  }
#pragma unroll
  for (int rr = 0; rr < P; ++rr) {
    if (first[rr] < 0) continue;
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
      for (int i = 0; i < R; ++i)
        store_out<R>(p.img, static_cast<size_t>(first[rr]) + c * plane_pitch + static_cast<size_t>(i) * row_pitch,
                     out[rr][c][i], O16);
  }
  if constexpr (CH == 4) {
    float al[P][R][R];
    alpha(al);
#pragma unroll
    for (int rr = 0; rr < P; ++rr) {
      if (first[rr] < 0) continue;
#pragma unroll
      for (int i = 0; i < R; ++i)
        store_out<R>(p.img, static_cast<size_t>(first[rr]) + 3 * plane_pitch + static_cast<size_t>(i) * row_pitch,
                     al[rr][i], O16);
    }
  }
}
// The layouts and the 16-bit image type (I16) are template parameters of the calling kernel: one runtime branch over four
// layouts in the same kernel raises the planar head's registers and makes it spill.  8 bits or fp32 is a runtime choice.
template <int R, int P, bool XN, bool YN, bool I16, int CH, int NA>
__device__ __forceinline__ void epi_head_tc(const EpiParams& p, int b, int y, int x, const float (&acc)[P][NA],
                                            bool interior, bool second = false) {
  if constexpr (I16)
    epi_head_t<R, P, uint16_t, XN, YN, CH>(p, static_cast<const uint16_t*>(p.img.x), b, y, x, acc, interior, second);
  else if (p.img.type == kImgU8)
    epi_head_t<R, P, uint8_t, XN, YN, CH>(p, static_cast<const uint8_t*>(p.img.x), b, y, x, acc, interior, second);
  else
    epi_head_t<R, P, float, XN, YN, CH>(p, static_cast<const float*>(p.img.x), b, y, x, acc, interior, second);
}
#endif  // __CUDACC__

}  // namespace mz
