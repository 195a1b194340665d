// api.cu -- extern "C" per-kernel entry points declared in include/mewzoom_b200.h.
#include <mutex>
#include <vector>

#include <math.h>
#include <string.h>

#include "kernels.cuh"

namespace mz {

ConvTcTune to_tune(const mz_conv_tune* t) {
  ConvTcTune o;
  memset(&o, 0, sizeof(o));
  if (t) {
    o.rows = t->rows;
    o.acc_stages = t->acc_stages;
    o.kc = t->kc;
    o.halo_mode = t->halo_mode;
    o.b_stages = t->b_stages;
    o.a_stages = t->a_stages;
    o.max_ctas = t->max_ctas;
    o.cluster = t->cluster;
    o.dbg = t->dbg;
    o.pair = t->pair;
    o.resident = t->resident;
    o.epi_warps = t->epi_warps;
    o.fuse = t->fuse;
    o.block = t->block;
    o.seg_rows = t->seg_rows;
  }
  return o;
}

int current_device() {
  int d = 0;
  cudaGetDevice(&d);
  return d;
}

// OIHW fp32 -> [tap][cout_p][cin_p] fp16 | bf16 bits (zero padded), host side.
bool pack_conv_weight_host(const float* w, int cout, int cin, int cout_p, int cin_p, int bf16,
                           std::vector<uint16_t>& out) {
  out.assign(static_cast<size_t>(9) * cout_p * cin_p, 0);
  bool in_range = true;
  for (int o = 0; o < cout; ++o)
    for (int i = 0; i < cin; ++i)
      for (int t = 0; t < 9; ++t) {
        const float v = w[(static_cast<size_t>(o) * cin + i) * 9 + t];
        if (!bf16 && !(fabsf(v) <= MZ_F16_MAX)) in_range = false;
        uint16_t bits;
        if (bf16) {
          const __nv_bfloat16 h = __float2bfloat16_rn(v);
          memcpy(&bits, &h, 2);
        } else {
          const __half h = __float2half_rn(v);
          memcpy(&bits, &h, 2);
        }
        out[(static_cast<size_t>(t) * cout_p + o) * cin_p + i] = bits;
      }
  return in_range;
}

bool dtype_ok(int d) { return d == MZ_DTYPE_F16 || d == MZ_DTYPE_BF16; }

}  // namespace mz

using namespace mz;

extern "C" {

int mz_bicubic_f32(const float* x_dev, float* y_dev, int32_t planes, int32_t H, int32_t W, int32_t r, void* stream) {
  MZ_REQUIRE(x_dev && y_dev, "bicubic: null pointer");
  return launch_bicubic(x_dev, y_dev, planes, H, W, r, static_cast<cudaStream_t>(stream));
}

int mz_stem_pack(const float* x_dev, const float* w_dev, const float* bias_dev, float* zf_dev, void* zb_dev, int32_t B,
                 int32_t H, int32_t W, int32_t Cp, int32_t zb_pitch, int32_t operand_dtype, void* stream) {
  MZ_REQUIRE(x_dev && w_dev && bias_dev && zf_dev && zb_dev, "stem: null pointer");
  MZ_REQUIRE(dtype_ok(operand_dtype), "operand_dtype must be MZ_DTYPE_F16 or MZ_DTYPE_BF16, %d given", operand_dtype);
  return launch_stem(x_dev, kImgF32, 0, 3, w_dev, bias_dev, zf_dev, static_cast<uint16_t*>(zb_dev), operand_dtype, B, H, W, Cp,
                     zb_pitch, static_cast<cudaStream_t>(stream));
}

int mz_conv3x3(const void* in_dev, const void* wpacked_dev, int32_t mode, const float* film_dev, void* out_bf16_dev,
               float* zf_dev, int32_t B, int32_t H, int32_t W, int32_t cin_p, int32_t in_pitch, int32_t cout_p,
               int32_t out_pitch, int32_t zf_pitch, int32_t operand_dtype, int32_t use_tc, const mz_conv_tune* tune,
               void* stream) {
  MZ_REQUIRE(in_pitch == 0 || (in_pitch >= cin_p && in_pitch % 8 == 0), "conv: in_pitch %d must be 0 or a multiple of 8 >= cin_p", in_pitch);
  MZ_REQUIRE(out_pitch == 0 || (out_pitch >= cout_p && out_pitch % 8 == 0), "conv: out_pitch %d must be 0 or a multiple of 8 >= cout_p", out_pitch);
  MZ_REQUIRE(zf_pitch == 0 || (zf_pitch >= cout_p && zf_pitch % 4 == 0), "conv: zf_pitch %d must be 0 or a multiple of 4 >= cout_p", zf_pitch);
  MZ_REQUIRE(in_dev && wpacked_dev && out_bf16_dev, "conv: null pointer");
  MZ_REQUIRE(dtype_ok(operand_dtype), "operand_dtype must be MZ_DTYPE_F16 or MZ_DTYPE_BF16, %d given", operand_dtype);
  MZ_REQUIRE(mode == 0 || mode == 1, "conv: mode must be 0 or 1, %d given", mode);
  MZ_REQUIRE(mode != 1 || zf_dev, "conv: mode 1 needs the fp32 residual stream");
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.in = static_cast<const uint16_t*>(in_dev);
  a.w = static_cast<const uint16_t*>(wpacked_dev);
  a.cin_p = cin_p;
  a.in_pitch = in_pitch;
  a.epi.bf16 = operand_dtype == MZ_DTYPE_BF16;
  a.epi.mode = mode;
  a.epi.B = B;
  a.epi.H = H;
  a.epi.W = W;
  a.epi.n_pad = cout_p;
  a.epi.film = film_dev;
  a.epi.out_bf16 = static_cast<uint16_t*>(out_bf16_dev);
  a.epi.out_pitch = out_pitch;
  a.epi.zf = zf_dev;
  a.epi.zf_pitch = zf_pitch;
  if (use_tc) return launch_conv_tc(a, to_tune(tune), current_device(), static_cast<cudaStream_t>(stream));
  return launch_conv_simt(a, static_cast<cudaStream_t>(stream));
}

int mz_head_shuffle_add(const void* zb_dev, const void* wpacked_dev, const float* x_dev, float* y_dev, int32_t B,
                        int32_t H, int32_t W, int32_t cin_p, int32_t in_pitch, int32_t r, int32_t skip_mode,
                        int32_t clamp01, int32_t operand_dtype, int32_t use_tc, const mz_conv_tune* tune, void* stream) {
  MZ_REQUIRE(in_pitch == 0 || (in_pitch >= cin_p && in_pitch % 8 == 0), "head: in_pitch %d must be 0 or a multiple of 8 >= cin_p", in_pitch);
  MZ_REQUIRE(zb_dev && wpacked_dev && y_dev, "head: null pointer");
  MZ_REQUIRE(dtype_ok(operand_dtype), "operand_dtype must be MZ_DTYPE_F16 or MZ_DTYPE_BF16, %d given", operand_dtype);
  MZ_REQUIRE(r == 2 || r == 3 || r == 4, "Upscale ratio must be either 2, 3, or 4, %d given.", r);
  MZ_REQUIRE(skip_mode >= 0 && skip_mode <= 2, "head: skip_mode must be 0, 1 or 2, %d given", skip_mode);
  MZ_REQUIRE(skip_mode != 2 || x_dev, "head: skip_mode 2 needs the LR image");
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.in = static_cast<const uint16_t*>(zb_dev);
  a.w = static_cast<const uint16_t*>(wpacked_dev);
  a.cin_p = cin_p;
  a.in_pitch = in_pitch;
  a.epi.bf16 = operand_dtype == MZ_DTYPE_BF16;
  a.epi.mode = 2;
  a.epi.B = B;
  a.epi.H = H;
  a.epi.W = W;
  a.epi.n_pad = mz_padded_channels(3 * r * r);
  a.epi.img.x = x_dev;
  a.epi.img.y = y_dev;
  a.epi.img.type = kImgF32;
  a.epi.nc = 3;
  a.epi.img.skip_mode = skip_mode;
  a.epi.img.clamp01 = clamp01;
  a.epi.r = r;
  make_bicubic_table(r, &a.epi.bt);
  if (use_tc) return launch_conv_tc(a, to_tune(tune), current_device(), static_cast<cudaStream_t>(stream));
  return launch_conv_simt(a, static_cast<cudaStream_t>(stream));
}

int mz_block_fused(const void* zb_in_dev, void* zb_out_dev, float* zf_dev, const void* w1_packed_dev,
                   const void* w2_packed_dev, const float* film_dev, int32_t B, int32_t H, int32_t W, int32_t operand_dtype,
                   int32_t seg_rows, int32_t max_ctas, void* stream) {
  MZ_REQUIRE(zb_in_dev && zb_out_dev && zf_dev && w1_packed_dev && w2_packed_dev, "block_fused: null pointer");
  MZ_REQUIRE(dtype_ok(operand_dtype), "operand_dtype must be MZ_DTYPE_F16 or MZ_DTYPE_BF16, %d given", operand_dtype);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint16_t* stacked = nullptr;
  MZ_CUDA(cudaMalloc(&stacked, sizeof(uint16_t) * 9 * 48 * 96));
  int rc = stack_conv2_bank(static_cast<const uint16_t*>(w2_packed_dev), stacked, s);
  if (rc == MZ_OK) {
    FusedBlockArgs a;
    memset(&a, 0, sizeof(a));
    a.zb_in = static_cast<const uint16_t*>(zb_in_dev);
    a.zb_out = static_cast<uint16_t*>(zb_out_dev);
    a.zf = zf_dev;
    a.w1 = static_cast<const uint16_t*>(w1_packed_dev);
    a.w2s = stacked;
    a.film = film_dev;
    a.B = B;
    a.H = H;
    a.W = W;
    a.bf16 = operand_dtype == MZ_DTYPE_BF16;
    a.seg_rows = seg_rows;
    a.max_ctas = max_ctas;
    ConvLaunch L;
    rc = prepare_block_fused(a, current_device(), &L);
    if (rc == MZ_OK) rc = run_block_fused(L, s);
  }
  const cudaError_t e = cudaStreamSynchronize(s);
  cudaFree(stacked);
  if (rc == MZ_OK && e != cudaSuccess) return cuda_fail(e, "block_fused synchronize", __FILE__, __LINE__);
  return rc;
}

int mz_pack_conv_weight(const float* w_host, int32_t cout, int32_t cin, int32_t cout_p, int32_t cin_p,
                        int32_t operand_dtype, void* dst_dev, size_t* bytes) {
  MZ_REQUIRE(dtype_ok(operand_dtype), "operand_dtype must be MZ_DTYPE_F16 or MZ_DTYPE_BF16, %d given", operand_dtype);
  MZ_REQUIRE(cout > 0 && cin > 0 && cout_p >= cout && cin_p >= cin, "pack: bad shape (%d,%d)->(%d,%d)", cout, cin,
             cout_p, cin_p);
  MZ_REQUIRE(cout_p % 16 == 0 && cin_p % 16 == 0, "pack: padded sizes must be multiples of 16");
  const size_t n = static_cast<size_t>(9) * cout_p * cin_p * sizeof(uint16_t);
  if (bytes) *bytes = n;
  if (!dst_dev) return MZ_OK;
  MZ_REQUIRE(w_host, "pack: null weight pointer");
  std::vector<uint16_t> tmp;
  MZ_REQUIRE(pack_conv_weight_host(w_host, cout, cin, cout_p, cin_p, operand_dtype == MZ_DTYPE_BF16, tmp),
             "pack: a weight exceeds the fp16 operand range (|w| > 65504 or not finite); use MZ_DTYPE_BF16");
  MZ_CUDA(cudaMemcpy(dst_dev, tmp.data(), n, cudaMemcpyHostToDevice));
  return MZ_OK;
}

int mz_enable_peer_access(int32_t a, int32_t b) {
  static bool enabled[64][64];
  static std::mutex mu;
  MZ_REQUIRE(a >= 0 && a < 64 && b >= 0 && b < 64, "enable_peer_access: device index out of range (%d, %d)", a, b);
  if (a == b) return MZ_OK;
  std::lock_guard<std::mutex> lock(mu);
  if (enabled[a][b]) return MZ_OK;
  int prev = 0;
  MZ_CUDA(cudaGetDevice(&prev));
  const int pair[2][2] = {{a, b}, {b, a}};
  for (const auto& pr : pair) {
    int can = 0;
    MZ_CUDA(cudaDeviceCanAccessPeer(&can, pr[0], pr[1]));
    if (!can) {
      cudaSetDevice(prev);
      set_error("enable_peer_access: device %d cannot access device %d", pr[0], pr[1]);
      return MZ_ERR_UNSUPPORTED;
    }
    MZ_CUDA(cudaSetDevice(pr[0]));
    const cudaError_t e = cudaDeviceEnablePeerAccess(pr[1], 0);
    cudaGetLastError();  // (clears cudaErrorPeerAccessAlreadyEnabled)
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
      cudaSetDevice(prev);
      MZ_CUDA(e);
    }
  }
  MZ_CUDA(cudaSetDevice(prev));
  enabled[a][b] = enabled[b][a] = true;
  return MZ_OK;
}

int mz_put_plane_async(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width_bytes, size_t height,
                       void* stream) {
  MZ_REQUIRE(dst && src, "put_plane: null pointer");
  MZ_REQUIRE(width_bytes > 0 && height > 0 && dpitch >= width_bytes && spitch >= width_bytes,
             "put_plane: bad geometry (width %zu bytes, height %zu, pitches %zu / %zu)", width_bytes, height, dpitch, spitch);
  // a put into another GPU's memory goes over NVLink only with peer access enabled between the two devices in THIS
  // process (a mapping opened from an IPC handle does not imply it); without it the runtime stages through the host
  cudaPointerAttributes as, ad;
  if (cudaPointerGetAttributes(&as, src) == cudaSuccess && cudaPointerGetAttributes(&ad, dst) == cudaSuccess &&
      as.type == cudaMemoryTypeDevice && ad.type == cudaMemoryTypeDevice && as.device != ad.device) {
    (void)mz_enable_peer_access(as.device, ad.device);  // (without a peer path the copy still works, through the host)
  } else {
    cudaGetLastError();  // (an unregistered host pointer makes cudaPointerGetAttributes fail on old drivers)
  }
  MZ_CUDA(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width_bytes, height, cudaMemcpyDefault,
                            static_cast<cudaStream_t>(stream)));
  return MZ_OK;
}

int mz_ipc_frame_create(size_t bytes, void** dev_ptr, void* handle64) {
  MZ_REQUIRE(bytes > 0 && dev_ptr && handle64, "ipc_frame_create: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the C ABI passes IPC handles as 64 bytes");
  *dev_ptr = nullptr;
  void* p = nullptr;
  MZ_CUDA(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    MZ_CUDA(e);
  }
  memcpy(handle64, &h, 64);
  *dev_ptr = p;
  return MZ_OK;
}

int mz_ipc_frame_open(const void* handle64, void** dev_ptr) {
  MZ_REQUIRE(handle64 && dev_ptr, "ipc_frame_open: null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  *dev_ptr = nullptr;
  MZ_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return MZ_OK;
}

int mz_ipc_frame_close(void* dev_ptr, int32_t owner) {
  if (!dev_ptr) return MZ_OK;
  if (owner)
    MZ_CUDA(cudaFree(dev_ptr));
  else
    MZ_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return MZ_OK;
}

int mz_control_film(const float* c_dev, int32_t c_rows, const float* w_dev, const float* b_dev, float* film_dev,
                    int32_t L, int32_t B, int32_t F, int32_t hC, int32_t hCp, void* stream) {
  MZ_REQUIRE(c_dev && w_dev && b_dev && film_dev, "film: null pointer");
  return launch_film(c_dev, c_rows, w_dev, b_dev, film_dev, L, B, F, hC, hCp, hCp, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
