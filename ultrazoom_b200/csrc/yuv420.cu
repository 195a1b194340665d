// yuv420.cu -- 4:2:0 video frames (NV12, P010) <-> 16-bit planar RGB, on either side of a 16-bit upscale.
//
// A frame is a luma plane of H x W elements, then an interleaved Cb,Cr plane of H/2 x W/2 pairs; frames are 3HW/2
// elements apart.  NV12 elements are bytes; P010 elements are uint16 words with the 10-bit code in the top bits
// (word = code << 6; the low 6 bits are ignored on input and zero on output).  Chroma siting is the H.264 / HEVC default:
// chroma sample (i, j) sits at luma row 2i + 1/2, luma column 2j.
//   decode: vertical [1/4, 3/4] / [3/4, 1/4] upsampling, then horizontal: even columns take C[j], odd columns the mean of
//           C[j] and C[j+1] (edges clamped); R = Y' + 2(1-Kr) Cr', B = Y' + 2(1-Kb) Cb', G = (Y' - Kr R - Kb B) / Kg;
//           clamp to [0, 1] and store floor(65535 v + 0.5).
//   encode: v = rgb16 / 65535; luma per pixel; chroma = the mean of rows 2i and 2i+1, then [1, 2, 1] / 4 over columns
//           2j-1, 2j, 2j+1 (column -1 clamped to 0); every code floor(offset + scale v + 0.5), clamped to the code range.
// Both kernels are bandwidth-bound streams.  A thread owns one 2 x 2 luma quad and its chroma sample; a block is 128
// consecutive quads of one chroma row, and the grid's y dimension walks (image, chroma row) pairs: one 32-bit division
// per row, none per element.
#include "kernels.cuh"

namespace mz {

// elements of T as codes: bytes as they are, P010 words shifted down by 6
template <typename T>
static __device__ __forceinline__ void ld_pair(const T* p, float& a, float& b) {
  if constexpr (sizeof(T) == 1) {
    const unsigned v = __ldg(reinterpret_cast<const unsigned short*>(p));
    a = static_cast<float>(v & 0xFFu);
    b = static_cast<float>(v >> 8);
  } else {
    const unsigned v = __ldg(reinterpret_cast<const unsigned int*>(p));
    a = static_cast<float>((v & 0xFFFFu) >> 6);
    b = static_cast<float>(v >> 22);
  }
}

template <typename T>
static __device__ __forceinline__ void st_pair(T* p, unsigned a, unsigned b) {
  if constexpr (sizeof(T) == 1)
    *reinterpret_cast<unsigned short*>(p) = static_cast<unsigned short>(a | (b << 8));
  else
    *reinterpret_cast<unsigned int*>(p) = (a << 6) | (b << 22);
}

static __device__ __forceinline__ unsigned q16(float v) {  // floor(65535 clamp(v) + 0.5)
  return __float2uint_rd(fmaf(fminf(fmaxf(v, 0.f), 1.f), 65535.f, 0.5f));
}

static __device__ __forceinline__ unsigned qcode(float v, float off, float scale, float maxcode) {
  return static_cast<unsigned>(fminf(fmaxf(floorf(fmaf(scale, v, off + 0.5f)), 0.f), maxcode));
}

template <typename T>
__global__ void __launch_bounds__(128) yuv420_to_rgb16_kernel(const T* __restrict__ x, uint16_t* __restrict__ rgb, int B,
                                                               int H, int W, YuvCoef k) {
  const int Hc = H >> 1, Wc = W >> 1;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= Wc) return;
  const int jn = min(j + 1, Wc - 1);
  const size_t plane = static_cast<size_t>(H) * W;
  const float yinv = 1.f / k.yrange, cinv = 1.f / k.crange;
  for (int row = blockIdx.y; row < B * Hc; row += gridDim.y) {
    const int b = row / Hc, i = row - b * Hc;
    const T* frame = x + static_cast<size_t>(b) * (plane + plane / 2);
    const T* chroma = frame + plane;
    const int rows[3] = {max(i - 1, 0), i, min(i + 1, Hc - 1)};
    float cb[3][2], cr[3][2];  // [row i-1, i, i+1][column j, j+1]
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const T* cp = chroma + static_cast<size_t>(rows[t]) * W;
      ld_pair(cp + 2 * j, cb[t][0], cr[t][0]);
      ld_pair(cp + 2 * jn, cb[t][1], cr[t][1]);
    }
    const T* luma = frame + static_cast<size_t>(2 * i) * W + 2 * j;
    float yv[2][2];
    ld_pair(luma, yv[0][0], yv[0][1]);
    ld_pair(luma + W, yv[1][0], yv[1][1]);
    uint16_t* dst = rgb + static_cast<size_t>(b) * 3 * plane + static_cast<size_t>(2 * i) * W + 2 * j;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int o = r == 0 ? 0 : 2;  // the outer chroma row: i-1 above luma row 2i, i+1 below row 2i+1
      unsigned px[3][2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        float vb[2], vr[2];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          vb[c] = fmaf(0.75f, cb[1][c], 0.25f * cb[o][c]);
          vr[c] = fmaf(0.75f, cr[1][c], 0.25f * cr[o][c]);
        }
        const float ub = q == 0 ? vb[0] : 0.5f * (vb[0] + vb[1]);
        const float ur = q == 0 ? vr[0] : 0.5f * (vr[0] + vr[1]);
        const float Y = (yv[r][q] - k.yoff) * yinv, Cb = (ub - k.coff) * cinv, Cr = (ur - k.coff) * cinv;
        const float R = fmaf(2.f * (1.f - k.kr), Cr, Y), Bl = fmaf(2.f * (1.f - k.kb), Cb, Y);
        const float G = (Y - k.kr * R - k.kb * Bl) / k.kg;
        px[0][q] = q16(R);
        px[1][q] = q16(G);
        px[2][q] = q16(Bl);
      }
#pragma unroll
      for (int c = 0; c < 3; ++c)
        *reinterpret_cast<unsigned int*>(dst + c * plane + static_cast<size_t>(r) * W) = px[c][0] | (px[c][1] << 16);
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(128) rgb16_to_yuv420_kernel(const uint16_t* __restrict__ rgb, T* __restrict__ y, int B,
                                                               int H, int W, YuvCoef k) {
  const int Hc = H >> 1, Wc = W >> 1;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= Wc) return;
  const int jl = max(2 * j - 1, 0);  // (column -1 is clamped to 0)
  const size_t plane = static_cast<size_t>(H) * W;
  const float inv = 1.f / 65535.f;
  const float kcb = 1.f / (2.f * (1.f - k.kb)), kcr = 1.f / (2.f * (1.f - k.kr));
  for (int row = blockIdx.y; row < B * Hc; row += gridDim.y) {
    const int b = row / Hc, i = row - b * Hc;
    const uint16_t* src = rgb + static_cast<size_t>(b) * 3 * plane + static_cast<size_t>(2 * i) * W;
    float v[2][3][3];  // [row][colour][column 2j-1, 2j, 2j+1]
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const uint16_t* p = src + c * plane + static_cast<size_t>(r) * W;
        const unsigned two = __ldg(reinterpret_cast<const unsigned int*>(p + 2 * j));
        v[r][c][0] = static_cast<float>(__ldg(p + jl)) * inv;
        v[r][c][1] = static_cast<float>(two & 0xFFFFu) * inv;
        v[r][c][2] = static_cast<float>(two >> 16) * inv;
      }
    float cbm[3], crm[3];  // chroma of the three columns, mean of the two rows
    T* frame = y + static_cast<size_t>(b) * (plane + plane / 2);
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      float sb = 0.f, sr = 0.f;
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const float R = v[r][0][q], G = v[r][1][q], Bl = v[r][2][q];
        const float Y = fmaf(k.kr, R, fmaf(k.kg, G, k.kb * Bl));
        sb += (Bl - Y) * kcb;
        sr += (R - Y) * kcr;
      }
      cbm[q] = 0.5f * sb;
      crm[q] = 0.5f * sr;
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      unsigned yc[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const float R = v[r][0][q + 1], G = v[r][1][q + 1], Bl = v[r][2][q + 1];
        yc[q] = qcode(fmaf(k.kr, R, fmaf(k.kg, G, k.kb * Bl)), k.yoff, k.yrange, k.maxcode);
      }
      st_pair(frame + static_cast<size_t>(2 * i + r) * W + 2 * j, yc[0], yc[1]);
    }
    const float cb = 0.25f * (cbm[0] + cbm[2]) + 0.5f * cbm[1], cr = 0.25f * (crm[0] + crm[2]) + 0.5f * crm[1];
    st_pair(frame + plane + static_cast<size_t>(i) * W + 2 * j, qcode(cb, k.coff, k.crange, k.maxcode),
            qcode(cr, k.coff, k.crange, k.maxcode));
  }
}

// grid: 128 quads of one chroma row per block; (image, chroma row) pairs along y, strided when there are more than 65535
static dim3 yuv_grid(int B, int H, int W) {
  const long long rows = static_cast<long long>(B) * (H / 2);
  return dim3(static_cast<unsigned>((W / 2 + 127) / 128), static_cast<unsigned>(rows < 65535 ? rows : 65535));
}

int yuv_coef(uint32_t flags, YuvCoef* k) {
  MZ_REQUIRE(flags & MZ_FLAG_YUV420, "yuv420: MZ_FLAG_YUV420 is not set");
  MZ_REQUIRE(((flags & MZ_FLAG_IO_U8) != 0) != ((flags & MZ_FLAG_IO_U16) != 0),
             "yuv420: a 4:2:0 frame is NV12 (MZ_FLAG_IO_U8) or P010 (MZ_FLAG_IO_U16): exactly one of them");
  MZ_REQUIRE(!((flags & MZ_FLAG_YUV_BT601) && (flags & MZ_FLAG_YUV_BT2020)),
             "yuv420: MZ_FLAG_YUV_BT601 and MZ_FLAG_YUV_BT2020 exclude each other");
  if (flags & MZ_FLAG_YUV_BT601) {
    k->kr = 0.299f, k->kb = 0.114f;
  } else if (flags & MZ_FLAG_YUV_BT2020) {
    k->kr = 0.2627f, k->kb = 0.0593f;
  } else {
    k->kr = 0.2126f, k->kb = 0.0722f;
  }
  k->kg = 1.f - k->kr - k->kb;
  const int bits = (flags & MZ_FLAG_IO_U16) ? 10 : 8;
  const float u = static_cast<float>(1 << (bits - 8));
  k->maxcode = static_cast<float>((1 << bits) - 1);
  k->coff = static_cast<float>(1 << (bits - 1));
  if (flags & MZ_FLAG_YUV_FULL_RANGE) {
    k->yoff = 0.f, k->yrange = k->maxcode, k->crange = k->maxcode;
  } else {
    k->yoff = 16.f * u, k->yrange = 219.f * u, k->crange = 224.f * u;
  }
  return MZ_OK;
}

static int check_yuv_call(const void* yuv, const void* rgb, int B, int H, int W, uint32_t flags, YuvCoef* k) {
  MZ_REQUIRE(yuv && rgb, "yuv420: null pointer");
  const int rc = yuv_coef(flags, k);
  if (rc != MZ_OK) return rc;
  MZ_REQUIRE(B > 0 && H > 0 && W > 0, "yuv420: empty frame (B %d, H %d, W %d)", B, H, W);
  MZ_REQUIRE(H % 2 == 0 && W % 2 == 0, "yuv420: a 4:2:0 frame has even dimensions, %d x %d given", H, W);
  MZ_REQUIRE(static_cast<long long>(B) * H < (1LL << 31), "yuv420: too many rows");
  const unsigned ea = (flags & MZ_FLAG_IO_U16) ? 4 : 2;  // (a luma or chroma pair is one load / store)
  MZ_REQUIRE(reinterpret_cast<uintptr_t>(yuv) % ea == 0 && reinterpret_cast<uintptr_t>(rgb) % 4 == 0,
             "yuv420: the frame must be aligned to %u bytes and the RGB image to 4", ea);
  return MZ_OK;
}

int launch_yuv420_to_rgb16(const void* yuv, uint16_t* rgb, int B, int H, int W, uint32_t flags, cudaStream_t s) {
  YuvCoef k;
  const int rc = check_yuv_call(yuv, rgb, B, H, W, flags, &k);
  if (rc != MZ_OK) return rc;
  const dim3 grid = yuv_grid(B, H, W);
  if (flags & MZ_FLAG_IO_U16)
    yuv420_to_rgb16_kernel<uint16_t><<<grid, 128, 0, s>>>(static_cast<const uint16_t*>(yuv), rgb, B, H, W, k);
  else
    yuv420_to_rgb16_kernel<uint8_t><<<grid, 128, 0, s>>>(static_cast<const uint8_t*>(yuv), rgb, B, H, W, k);
  MZ_CUDA(cudaGetLastError());
  return MZ_OK;
}

int launch_rgb16_to_yuv420(const uint16_t* rgb, void* yuv, int B, int H, int W, uint32_t flags, cudaStream_t s) {
  YuvCoef k;
  const int rc = check_yuv_call(yuv, rgb, B, H, W, flags, &k);
  if (rc != MZ_OK) return rc;
  const dim3 grid = yuv_grid(B, H, W);
  if (flags & MZ_FLAG_IO_U16)
    rgb16_to_yuv420_kernel<uint16_t><<<grid, 128, 0, s>>>(rgb, static_cast<uint16_t*>(yuv), B, H, W, k);
  else
    rgb16_to_yuv420_kernel<uint8_t><<<grid, 128, 0, s>>>(rgb, static_cast<uint8_t*>(yuv), B, H, W, k);
  MZ_CUDA(cudaGetLastError());
  return MZ_OK;
}

}  // namespace mz

using namespace mz;

extern "C" {

int mz_yuv420_to_rgb16(const void* yuv_dev, uint16_t* rgb_dev, int32_t B, int32_t H, int32_t W, uint32_t flags, void* stream) {
  return launch_yuv420_to_rgb16(yuv_dev, rgb_dev, B, H, W, flags, static_cast<cudaStream_t>(stream));
}

int mz_rgb16_to_yuv420(const uint16_t* rgb_dev, void* yuv_dev, int32_t B, int32_t H, int32_t W, uint32_t flags, void* stream) {
  return launch_rgb16_to_yuv420(rgb_dev, yuv_dev, B, H, W, flags, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
