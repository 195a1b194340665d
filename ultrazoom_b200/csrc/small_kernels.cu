// small_kernels.cu -- the bandwidth-bound kernels around the conv stack:
//   * bicubic zoom            (Upsample(mode="bicubic"),  reference model.py:71,156)
//   * stem + layout change    (FanOutProjection,          reference model.py:212-242)
//   * FiLM coefficient table  (control module, restated -- SURVEY.md Appendix C)
//   * SIMT direct 3x3 conv    (diagnostic twin of the tcgen05 kernel; same epilogues)
#include <math.h>

#include "kernels.cuh"

namespace mz {

// ----------------------------------------------------------------------------------------------
// bicubic phase table (host) -- follows ATen's upsample_bicubic2d arithmetic in fp32:
//   src = scale * (dst + 0.5) - 0.5 with scale = 1/r, idx = floor(src), t = src - idx,
//   w = {cc2(t+1), cc1(t), cc1(1-t), cc2(2-t)}, A = -0.75.
// ----------------------------------------------------------------------------------------------
static float cc1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
static float cc2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }

void make_bicubic_table(int r, BicubicTable* t) {
  const float A = -0.75f;
  const float scale = 1.0f / static_cast<float>(r);
  t->r = r;
  for (int p = 0; p < 4; ++p) {
    t->off[p] = 0;
    for (int k = 0; k < 4; ++k) t->w[p][k] = 0.f;
  }
  for (int p = 0; p < r && p < 4; ++p) {
    const float src = scale * (static_cast<float>(p) + 0.5f) - 0.5f;
    const float fl = floorf(src);
    const float tt = src - fl;
    t->off[p] = static_cast<int>(fl);
    t->w[p][0] = cc2(tt + 1.f, A);
    t->w[p][1] = cc1(tt, A);
    const float x2 = 1.f - tt;
    t->w[p][2] = cc1(x2, A);
    t->w[p][3] = cc2(x2 + 1.f, A);
  }
}

// ----------------------------------------------------------------------------------------------
// bicubic zoom.  One thread owns one LR column of a strip of STRIP LR rows and slides a 5-row window of horizontally
// interpolated values down it: each LR row costs five (coalesced, L1-resident) loads and R horizontal interpolations,
// then the R x R HR pixels of the LR pixel leave as R row segments of R contiguous floats (a warp writes 32 * R
// contiguous floats per HR row).  ~2 loads per HR pixel at r = 2 (0.5 at r = 4) instead of 10 (5).
// A store stream (12 / r^2 B read, 12 B written per HR pixel).  Every tap of the strip -- STRIP + 4 rows x 5 columns --
// is requested before the first FMA: each row is first touched by this very block, and with the loads of a row issued
// when the window reached it a thread exposed one L2 / HBM round trip per row.  The strip loop is fully unrolled (the
// window rotates through compile-time indices: no register moves) and blocks whose columns need no clamping read each
// row through one pointer with immediate offsets; that halved the instruction count and, alone, changed nothing.
// Arithmetic order follows ATen's upsample_bicubic2d: horizontal taps first, then vertical.
// ----------------------------------------------------------------------------------------------
template <int R, int STRIP>
__global__ void __launch_bounds__(128) bicubic_kernel(const float* __restrict__ x, float* __restrict__ y, int H, int W,
                                                      int n_strips, BicubicTable bt) {
  const int lx = blockIdx.x * 128 + threadIdx.x;
  if (lx >= W) return;
  const int pl = blockIdx.y / n_strips, strip = blockIdx.y - pl * n_strips;
  const int ly0 = strip * STRIP, ly1 = min(ly0 + STRIP, H);
  const float* plane = x + static_cast<size_t>(pl) * H * W;
  const size_t WR = static_cast<size_t>(W) * R;
  float* out = y + static_cast<size_t>(pl) * H * R * WR + static_cast<size_t>(lx) * R;
  const bool interior = blockIdx.x > 0 && static_cast<int>(blockIdx.x) * 128 + 129 < W;  // (block-uniform) no clamped column
  int xs[5];
#pragma unroll
  for (int m = 0; m < 5; ++m) xs[m] = min(max(lx - 2 + m, 0), W - 1);
  float raw[STRIP + 4][5];  // strip row n = LR row ly0 - 2 + n (clamped)
#pragma unroll
  for (int n = 0; n < STRIP + 4; ++n) {
    const float* row = plane + static_cast<size_t>(min(max(ly0 - 2 + n, 0), H - 1)) * W;
    if (interior) {
      const float* rp = row + (lx - 2);
#pragma unroll
      for (int m = 0; m < 5; ++m) raw[n][m] = __ldg(rp + m);
    } else {
#pragma unroll
      for (int m = 0; m < 5; ++m) raw[n][m] = __ldg(row + xs[m]);
    }
  }
  // horizontally interpolated values of strip row n at the R phases of this column
  auto hrow = [&](int n, float (&h)[R]) {
#pragma unroll
    for (int j = 0; j < R; ++j) {
      const int s = (2 * j + 1 < R) ? 0 : 1;  // first tap relative to lx-2 (phase offset -1 or 0)
      float a = 0.f;
#pragma unroll
      for (int m = 0; m < 4; ++m) a = fmaf(raw[n][s + m], bt.w[j][m], a);
      h[j] = a;
    }
  };
  float win[5][R];  // a ring: strip row n lives in win[n % 5]
#pragma unroll
  for (int k = 0; k < 4; ++k) hrow(k, win[k]);
#pragma unroll
  for (int t = 0; t < STRIP; ++t) {
    const int ly = ly0 + t;
    if (ly >= ly1) break;  // (block-uniform)
    hrow(t + 4, win[(t + 4) % 5]);
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int s = (2 * i + 1 < R) ? 0 : 1;
      float o[R];
#pragma unroll
      for (int j = 0; j < R; ++j) {
        float a = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) a = fmaf(win[(t + s + k) % 5][j], bt.w[i][k], a);
        o[j] = a;
      }
      float* dst = out + (static_cast<size_t>(ly) * R + i) * WR;
      if (R == 4) {
        *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[R > 2 ? 2 : 0], o[R - 1]);
      } else if (R == 2) {
        *reinterpret_cast<float2*>(dst) = make_float2(o[0], o[1]);
      } else {
#pragma unroll
        for (int j = 0; j < R; ++j) dst[j] = o[j];
      }
    }
  }
}

template <int STRIP>
static void launch_bicubic_strip(const float* x, float* y, int H, int W, int r, int n_strips, dim3 grid, const BicubicTable& bt,
                                 cudaStream_t s) {
  if (r == 2)
    bicubic_kernel<2, STRIP><<<grid, 128, 0, s>>>(x, y, H, W, n_strips, bt);
  else if (r == 3)
    bicubic_kernel<3, STRIP><<<grid, 128, 0, s>>>(x, y, H, W, n_strips, bt);
  else
    bicubic_kernel<4, STRIP><<<grid, 128, 0, s>>>(x, y, H, W, n_strips, bt);
}

int launch_bicubic(const float* x, float* y, int planes, int H, int W, int r, cudaStream_t s) {
  MZ_REQUIRE(r == 2 || r == 3 || r == 4, "Upscale ratio must be either 2, 3, or 4, %d given.", r);
  MZ_REQUIRE(planes > 0 && H > 0 && W > 0, "bicubic: empty input (planes %d, H %d, W %d)", planes, H, W);
  BicubicTable bt;
  make_bicubic_table(r, &bt);
  // strips of 8 LR rows (60 taps in flight per thread), of 4 while the grid would not fill the GPU four times over
  const long long bx = (W + 127) / 128;
  const int strip_rows = bx * planes * ((H + 7) / 8) < 148LL * 16 * 4 ? 4 : 8;
  const int n_strips = (H + strip_rows - 1) / strip_rows;
  const long long gy = static_cast<long long>(planes) * n_strips;
  MZ_REQUIRE(gy <= 65535, "bicubic: planes x row strips (%lld) exceeds the grid limit", gy);
  const dim3 grid(static_cast<unsigned>(bx), static_cast<unsigned>(gy));
  if (strip_rows == 8)
    launch_bicubic_strip<8>(x, y, H, W, r, n_strips, grid, bt, s);
  else
    launch_bicubic_strip<4>(x, y, H, W, r, n_strips, grid, bt, s);
  MZ_CUDA(cudaGetLastError());
  return MZ_OK;
}

// ----------------------------------------------------------------------------------------------
// stem: x (B,3,H,W) -> zf (B,H,W,Cp) fp32 and zb (B,H,W,Cz) 16-bit; z = W x + bias,
// channels >= C are written as zero (w/bias are zero-padded to Cp by the caller).
// A store-only stream (12 B read, 6 Cp B written per pixel).  One thread -> 4 channels of one pixel, threads of a
// block laid out channel-fastest over consecutive pixels: a warp's fp32 store is 512 contiguous bytes, its 16-bit
// store 256 (the first version's 8 channels per thread wrote every other 16 bytes of a 1 KB span per instruction:
// 1.67 x the L2 sectors, ncu l1tex 75 % busy at 62 % of the DRAM peak).  The block first stages the three colour
// planes of its pixel range in shared memory with coalesced loads, so the store loop never waits for a global load.
// x_nhwc: x is interleaved (B,H,W,3); images are 3HW elements apart in both layouts, so the block's pixel range is one
// contiguous run of 3n elements even across images, read with coalesced loads into the same planar staging.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_global_v2(void* p, uint32_t a, uint32_t b) {
  asm volatile("st.global.v2.b32 [%0], {%1, %2};" ::"l"(p), "r"(a), "r"(b) : "memory");
}

// element i of the image (ImageType `type`) as float: fp32 as it is; 8 / 16 bits as the exact quotient x / 255,
// x / 65535 (IEEE division, what ToDtype(float32, scale=True) computes): the network amplifies a 1-ulp difference of its
// input through 20..40 layers of 16-bit rounding to ~1e-3 at the output
__device__ __forceinline__ float stem_px(const void* __restrict__ x, int type, size_t i) {
  switch (type) {
    case kImgU8: return __fdiv_rn(static_cast<float>(static_cast<const uint8_t*>(x)[i]), 255.f);
    case kImgU16: return __fdiv_rn(static_cast<float>(static_cast<const uint16_t*>(x)[i]), 65535.f);
    default: return static_cast<const float*>(x)[i];
  }
}

__global__ void __launch_bounds__(256) stem_kernel(const void* __restrict__ x, int type, int x_nhwc,
                                                   const float* __restrict__ w, const float* __restrict__ bias,
                                                   float* __restrict__ zf, uint16_t* __restrict__ zb, int bf16, int B,
                                                   int H, int W, int Cp, int Cz, int ppb, unsigned int* sat) {
  extern __shared__ float xs[];  // [3][ppb]: the block's pixels, colour planes apart
  // blockDim = (channel groups of 4, pixels per pass): a thread keeps ITS four channels' weights and bias in registers
  const int g = threadIdx.x;
  const bool real = g * 4 < Cp;  // groups beyond Cp exist only in the 16-bit shadow (zero padding up to its pitch Cz)
  float wr[4][3], br[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = g * 4 + i;
    br[i] = real ? __ldg(bias + n) : 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) wr[i][c] = real ? __ldg(w + n * 3 + c) : 0.f;
  }
  const size_t plane = static_cast<size_t>(H) * W;
  const size_t npix = static_cast<size_t>(B) * plane;
  const size_t p0 = static_cast<size_t>(blockIdx.x) * ppb;
  const int n = static_cast<int>((p0 + ppb < npix ? p0 + ppb : npix) - p0);
  if (x_nhwc) {
    const int tid = threadIdx.y * blockDim.x + threadIdx.x, nt = blockDim.x * blockDim.y;
    const size_t e0 = p0 * 3;
    for (int e = tid; e < 3 * n; e += nt) {
      const int j = e / 3, c = e - 3 * j;
      xs[c * ppb + j] = stem_px(x, type, e0 + e);
    }
  } else {
    const size_t b0 = p0 / plane, rem0 = p0 - b0 * plane;  // (one division per block; the range may cross images)
    const int tid = threadIdx.y * blockDim.x + threadIdx.x, nt = blockDim.x * blockDim.y;
    for (int j = tid; j < n; j += nt) {
      size_t b = b0, rem = rem0 + j;
      while (rem >= plane) {
        rem -= plane;
        ++b;
      }
      const size_t xo = b * 3 * plane + rem;
#pragma unroll
      for (int c = 0; c < 3; ++c) xs[c * ppb + j] = stem_px(x, type, xo + c * plane);
    }
  }
  __syncthreads();
  float amax = 0.f;
  for (int j = threadIdx.y; j < n; j += blockDim.y) {
    const float r0 = xs[j], r1 = xs[ppb + j], r2 = xs[2 * ppb + j];
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      o[i] = fmaf(wr[i][2], r2, fmaf(wr[i][1], r1, fmaf(wr[i][0], r0, br[i])));
      amax = fmaxf(amax, fabsf(o[i]));
    }
    const size_t pix = p0 + j;
    if (real) *reinterpret_cast<float4*>(zf + pix * Cp + g * 4) = make_float4(o[0], o[1], o[2], o[3]);
    if (g * 4 < Cz) st_global_v2(zb + pix * Cz + g * 4, pack_op2(bf16, o[0], o[1]), pack_op2(bf16, o[2], o[3]));
  }
  if (!bf16 && sat != nullptr && !(amax <= MZ_F16_MAX)) *sat = 1u;  // fp16 range guard (see EpiParams::sat)
}

int launch_stem(const void* x, int type, int x_nhwc, const float* w, const float* bias, float* zf, uint16_t* zb, int bf16,
                int B, int H, int W, int Cp, int zb_pitch, cudaStream_t s, unsigned int* sat) {
  MZ_REQUIRE(Cp > 0 && Cp % 8 == 0, "stem: padded channel count must be a multiple of 8, %d given", Cp);
  MZ_REQUIRE(B > 0 && H > 0 && W > 0, "stem: empty input");
  MZ_REQUIRE(zf != nullptr, "stem: null fp32 stream");
  const int Cz = zb_pitch ? zb_pitch : Cp;
  // (the shadow may be wider than the fp32 stream -- zero padding up to its pitch -- or narrower: a dense shadow beside a
  // padded stream; padded channels are zeros either way)
  MZ_REQUIRE(Cz > 0 && Cz % 8 == 0, "stem: zb pitch %d must be a positive multiple of 8", Cz);
  const int groups = (Cz > Cp ? Cz : Cp) / 4;
  MZ_REQUIRE(groups <= 256, "stem: %d channels per pixel exceed 1024", groups * 4);
  const int py = 256 / groups > 0 ? 256 / groups : 1;  // pixels per pass of a block
  const long long npix = static_cast<long long>(B) * H * W;
  // ~16 passes per block, but at least ~8 blocks per SM so that a small frame still fills the GPU
  long long ppb = static_cast<long long>(py) * 16;
  while (ppb > py && (npix + ppb - 1) / ppb < 148LL * 8) ppb -= py;
  const long long blocks = (npix + ppb - 1) / ppb;
  MZ_REQUIRE(blocks < (1LL << 31), "stem: too many pixels");
  const size_t smem = static_cast<size_t>(3) * ppb * sizeof(float);
  stem_kernel<<<static_cast<unsigned>(blocks), dim3(groups, py), smem, s>>>(x, type, x_nhwc, w, bias, zf, zb, bf16, B, H, W,
                                                                         Cp, Cz, static_cast<int>(ppb), sat);
  MZ_CUDA(cudaGetLastError());
  return MZ_OK;
}

// ----------------------------------------------------------------------------------------------
// weight repack on the device: OIHW fp32 -> [tap][cout_p][cin_p] fp16 | bf16, zero padded (what
// pack_conv_weight_host does on the CPU; used by mz_model_set_weight_dev so that a model living on
// the GPU is packed without a round trip through host memory).
// ----------------------------------------------------------------------------------------------
__global__ void pack_conv_weight_kernel(const float* __restrict__ w, uint16_t* __restrict__ out, int cout, int cin,
                                        int cout_p, int cin_p, int bf16, unsigned int* sat) {
  const long long total = 9LL * cout_p * cin_p;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(idx % cin_p);
    const long long r = idx / cin_p;
    const int o = static_cast<int>(r % cout_p), t = static_cast<int>(r / cout_p);
    float v = 0.f;
    if (o < cout && i < cin) v = __ldg(w + (static_cast<size_t>(o) * cin + i) * 9 + t);
    if (!bf16 && sat != nullptr && !(fabsf(v) <= MZ_F16_MAX)) *sat = 1u;
    out[idx] = bf16 ? __bfloat16_as_ushort(__float2bfloat16_rn(v)) : __half_as_ushort(__float2half_rn(v));
  }
}

int launch_pack_conv_weight(const float* w_dev, uint16_t* out_dev, int cout, int cin, int cout_p, int cin_p, int bf16,
                            unsigned int* sat, cudaStream_t s) {
  MZ_REQUIRE(cout >= 0 && cin > 0 && cout_p >= cout && cin_p >= cin, "pack: bad shape (%d,%d)->(%d,%d)", cout, cin, cout_p, cin_p);
  const long long total = 9LL * cout_p * cin_p;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  pack_conv_weight_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(w_dev, out_dev, cout, cin, cout_p, cin_p, bf16, sat);
  MZ_CUDA(cudaGetLastError());
  return MZ_OK;
}

// ----------------------------------------------------------------------------------------------
// FiLM table: film[l][b][0][n] = 1 + gamma, film[l][b][1][n] = beta, g = Linear_l(c_b);
// gamma = g[n], beta = g[hC + n]; padded channels n >= hC get scale 1, shift 0.
// ----------------------------------------------------------------------------------------------
__global__ void film_kernel(const float* __restrict__ c, int c_rows, const float* __restrict__ w,
                            const float* __restrict__ bias, float* __restrict__ film, int L, int B, int F, int hC,
                            int hCp, int ns) {
  const long long total = static_cast<long long>(L) * B * hCp;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(idx % hCp);
    const long long t = idx / hCp;
    const int b = static_cast<int>(t % B);
    const int l = static_cast<int>(t / B);
    float scale = 1.f, shift = 0.f;
    if (n < hC) {
      const float* cb = c + static_cast<size_t>(c_rows == 1 ? 0 : b) * F;
      const float* wg = w + (static_cast<size_t>(l) * 2 * hC + n) * F;
      const float* wb = w + (static_cast<size_t>(l) * 2 * hC + hC + n) * F;
      float g = bias[static_cast<size_t>(l) * 2 * hC + n];
      float be = bias[static_cast<size_t>(l) * 2 * hC + hC + n];
      for (int f = 0; f < F; ++f) {
        g = fmaf(cb[f], wg[f], g);
        be = fmaf(cb[f], wb[f], be);
      }
      scale = 1.f + g;
      shift = be;
    }
    // [l][slice][b][scale row | shift row][ns]: one [B][2][ns] table per conv1 launch (ns == hCp: one slice)
    const int sl = n / ns, j = n - sl * ns;
    float* dst = film + ((static_cast<size_t>(l) * (hCp / ns) + sl) * B + b) * 2 * ns;
    dst[j] = scale;
    dst[ns + j] = shift;
  }
}

int launch_film(const float* c, int c_rows, const float* w, const float* b, float* film, int L, int B, int F, int hC,
                int hCp, int ns, cudaStream_t s) {
  MZ_REQUIRE(c_rows == 1 || c_rows == B, "Batch size of c (%d) must match x (%d).", c_rows, B);
  MZ_REQUIRE(L > 0 && B > 0 && F > 0 && hC > 0 && hCp >= hC, "film: bad shape");
  MZ_REQUIRE(ns > 0 && hCp % ns == 0, "film: slice width %d does not divide the padded width %d", ns, hCp);
  const long long total = static_cast<long long>(L) * B * hCp;
  long long blocks = (total + 255) / 256;
  if (blocks > 1024) blocks = 1024;
  film_kernel<<<static_cast<unsigned>(blocks), 256, 0, s>>>(c, c_rows, w, b, film, L, B, F, hC, hCp, ns);
  MZ_CUDA(cudaGetLastError());
  return MZ_OK;
}

// ----------------------------------------------------------------------------------------------
// SIMT direct convolution (diagnostic).  Same operands (16-bit NHWC activations, 16-bit [tap][n][k]
// weights), fp32 accumulation, same epilogues -- so that a tcgen05 result can be bisected against
// it on the GPU.  One thread -> 16 output channels of one pixel (modes 0/1) or the whole head.
// ----------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(128) conv_simt_kernel(ConvArgs a) {
  const EpiParams& p = a.epi;
  const int groups = MODE == 2 ? 1 : p.n_pad / 16;
  const long long total = static_cast<long long>(p.B) * p.H * p.W * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(idx % groups);
    long long t = idx / groups;
    const int x = static_cast<int>(t % p.W);
    t /= p.W;
    const int y = static_cast<int>(t % p.H);
    const int b = static_cast<int>(t / p.H);
    constexpr int NACC = MODE == 2 ? 48 : 16;
    float acc[NACC];
#pragma unroll
    for (int i = 0; i < NACC; ++i) acc[i] = 0.f;
    const int n0 = g * 16;
    const int nlim = MODE == 2 ? p.n_pad : 16;
    for (int ky = 0; ky < 3; ++ky) {
      const int yy = y + ky - 1;
      if (yy < 0 || yy >= p.H) continue;
      for (int kx = 0; kx < 3; ++kx) {
        const int xx = x + kx - 1;
        if (xx < 0 || xx >= p.W) continue;
        const uint16_t* src = a.in + ((static_cast<size_t>(b) * p.H + yy) * p.W + xx) * (a.in_pitch ? a.in_pitch : a.cin_p);
        const uint16_t* wt = a.w + (static_cast<size_t>(ky * 3 + kx) * p.n_pad + n0) * a.cin_p;
        const int kmax = a.in_extent ? a.in_extent : a.cin_p;  // (channels beyond the extent are zero padding)
        for (int k = 0; k < kmax; ++k) {
          const float v = op_to_float(p.bf16, src[k]);
#pragma unroll
          for (int i = 0; i < NACC; ++i)
            if (i < nlim) acc[i] = fmaf(v, op_to_float(p.bf16, wt[static_cast<size_t>(i) * a.cin_p + k]), acc[i]);
        }
      }
    }
    if (MODE == 2) {
      float h[48];
#pragma unroll
      for (int i = 0; i < 48; ++i) h[i] = i < NACC ? acc[i] : 0.f;
      epi_head<48>(p, b, y, x, h);
    } else {
      float h[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) h[i] = acc[i];
      constexpr int M01 = MODE == 2 ? 0 : MODE;  // (epilogue mode 0 or 1)
      epi_store16<M01>(p, b, y, x, n0, h,
                       p.film != nullptr ? p.film + static_cast<size_t>(b) * 2 * p.n_pad : nullptr);
    }
  }
}

int launch_conv_simt(const ConvArgs& a, cudaStream_t s) {
  const EpiParams& p = a.epi;
  MZ_REQUIRE(p.n_pad % 16 == 0 && p.n_pad > 0, "conv: n_pad must be a positive multiple of 16, %d given", p.n_pad);
  MZ_REQUIRE(p.mode != 2 || p.n_pad <= 48, "head conv: n_pad must be <= 48, %d given", p.n_pad);
  const long long total = static_cast<long long>(p.B) * p.H * p.W * (p.mode == 2 ? 1 : p.n_pad / 16);
  long long blocks = (total + 127) / 128;
  if (blocks > 148LL * 64) blocks = 148LL * 64;
  const unsigned gb = static_cast<unsigned>(blocks);
  if (p.mode == 0)
    conv_simt_kernel<0><<<gb, 128, 0, s>>>(a);
  else if (p.mode == 1)
    conv_simt_kernel<1><<<gb, 128, 0, s>>>(a);
  else
    conv_simt_kernel<2><<<gb, 128, 0, s>>>(a);
  MZ_CUDA(cudaGetLastError());
  return MZ_OK;
}

}  // namespace mz
