// model.cu -- mz_model: device-resident packed weights + the MewZoom forward schedule.
//
// Replaces MewZoom.__init__/load_state_dict (reference model.py:52-92) and MewZoom.forward/upscale
// (model.py:149-179) for the flat 0.2.x architecture BASELINE.json names (SURVEY.md Appendix C):
//   film  = FiLM table from c                      (control modules)
//   zf,zb = stem(x)                                (FanOutProjection + NCHW->NHWC)
//   L x { h = SiLU(film . conv1(zb)) ; zf += conv2(h) ; zb = bf16(zf) }
//   y     = [clamp](bicubic(x) + PixelShuffle(head(zb)))
// 2L + 3 kernel launches on the caller's stream, no host synchronisation, no allocation.
#include <stdlib.h>

#include <vector>

#include "kernels.cuh"

using namespace mz;

struct mz_model {
  mz_config cfg;
  int C, Cp, Cz, hC, hCp, L, r, F, headN, headNp, bf16;  // Cz: channel pitch of zb (>= Cp, zero padded)
  // Channels per pixel IN MEMORY of the fp32 stream, its 16-bit shadow and the hidden tensor.  Equal to the GEMM widths
  // (Cp, Cz, hCp) unless the layout is dense: channels rounded up to 8 only (54 -> 56, 108 -> 112 instead of 64 / 128) --
  // the GEMM's zero padding then exists in shared memory only (ConvArgs::in_extent, EpiParams::out_extent / zf_extent).
  int Cpm, Czm, hCm;
  // A hidden width above the 256 columns of one UMMA tile runs conv1 as S launches of ns output channels each
  // (hCp = S * ns): slice s has its own packed filter bank and FiLM rows and writes channels [s * ns, (s + 1) * ns) of
  // the hidden tensor.  Likewise conv2 above 128 output channels (its epilogue stages whole fp32 + 16-bit row tiles):
  // S2 launches of ns2 channels each (Cp = S2 * ns2), each adding into its channel slice of the residual stream.
  // S = S2 = 1 for every named model.
  int S = 1, ns = 0, S2 = 1, ns2 = 0;
  float* stem_w = nullptr;  // (Cp,3)
  float* stem_b = nullptr;  // (Cp)
  uint16_t* conv1 = nullptr;  // L x S x [9][ns][Cz]
  uint16_t* conv2 = nullptr;  // L x S2 x [9][ns2][hCp]
  uint16_t* head = nullptr;   // [9][headNp][Cp]
  // fused encoder block (block_fused.cu; 48-channel models): conv2's banks with the vertical taps stacked per filter
  // column, L x [3 dx][144][96]; the 16-bit stream then ping-pongs between zb and the (otherwise unused) hidden buffer
  uint16_t* conv2s = nullptr;
  bool fused_ok = false;
  struct FusedKey {
    FusedBlockArgs a;
  };
  std::vector<ConvLaunch> fprepared;  // kWays per layer, like `prepared`
  std::vector<FusedKey> fkeys;
  std::vector<uint8_t> fvictim;
  float* ctrl_w = nullptr;         // (L, 2hC, F)
  float* ctrl_b = nullptr;         // (L, 2hC)
  // fp16 range guard (EpiParams::sat): one host-mapped word the kernels set when a value beyond +-65504 is about to be
  // rounded into an fp16 operand; read without synchronising by mz_model_saturated
  unsigned int* sat_host = nullptr;
  unsigned int* sat_dev = nullptr;
  float* pack_tmp = nullptr;  // device staging for mz_model_set_weight_dev (largest fp32 tensor of the model)
  size_t pack_tmp_elems = 0;
  std::vector<uint8_t> have;       // per (kind, layer) upload flags
  ConvTcTune tune[3];
  // the *_host entry points: two lanes, each with its own stream, staging buffers and workspace, so that the
  // host-to-device copy of one chunk / frame overlaps the kernels of the previous one and the device-to-host copy
  // of the one before (the conv kernels fill the GPU on their own: two lanes never compute at the same time)
  struct HostLane {
    cudaStream_t stream = nullptr;
    void* ws = nullptr;
    size_t ws_bytes = 0;
    float* hx = nullptr;
    float* hy = nullptr;
    float* hc = nullptr;
    size_t hx_bytes = 0, hy_bytes = 0, hc_bytes = 0;
    cudaEvent_t kernels_done = nullptr;  // recorded after the lane's last kernel of a call
    bool has_work = false;
  };
  HostLane lane[2];
  // prepared launches, one per convolution of the model (layer l: conv1 slices at l (S + S2) + s, conv2 slices after
  // them; head -> L (S + S2)), reused while the
  // operands, shape and tunables of that convolution stay the same (`keys` holds what they were prepared for)
  struct ConvKey {
    ConvArgs a;
    ConvTcTune t;
  };
  std::vector<ConvLaunch> prepared;
  std::vector<ConvKey> keys;
  std::vector<uint8_t> victim;  // which of a convolution's two cache ways is replaced next
  // optional conv-stack timing
  bool timing = false;
  int timing_calls = 0;  // mz_upscale calls recorded since timing was enabled (ring of kTimingSlots)
  std::vector<cudaEvent_t> ev;  // 2 * kTimingSlots events
};

static constexpr int kTimingSlots = 64;
// Prepared launches per convolution: the two host lanes, the engine's own workspace and a captured graph's private one
// are four buffer sets that may alternate; the victim is chosen round-robin.
static constexpr int kWays = 4;

namespace {

struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
};

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct WsPlan {
  size_t zf, zb, hid, film, rgb_lr, rgb_hr, total;
};

constexpr uint32_t kYuvColourFlags = MZ_FLAG_YUV_BT601 | MZ_FLAG_YUV_BT2020 | MZ_FLAG_YUV_FULL_RANGE;

// With MZ_FLAG_YUV420 the two 16-bit RGB images of the call follow everything else, so that mz_workspace_layout's offsets
// are the same for every call.
WsPlan plan_ws(const mz_model* m, int B, int H, int W, uint32_t flags = 0) {
  const size_t npix = static_cast<size_t>(B) * H * W;
  WsPlan p;
  size_t off = 0;
  p.zf = off;
  off = align_up(off + npix * m->Cpm * sizeof(float), 1024);
  p.zb = off;
  off = align_up(off + npix * m->Czm * sizeof(uint16_t), 1024);
  p.hid = off;
  off = align_up(off + npix * m->hCm * sizeof(uint16_t), 1024);
  p.film = off;
  if (m->F > 0) off = align_up(off + static_cast<size_t>(m->L) * B * 2 * m->hCp * sizeof(float), 1024);
  p.rgb_lr = p.rgb_hr = off;
  if (flags & MZ_FLAG_YUV420) {
    const size_t lr = static_cast<size_t>(B) * 3 * H * W * sizeof(uint16_t);
    off = align_up(off + lr, 1024);
    p.rgb_hr = off;
    off = align_up(off + lr * m->r * m->r, 1024);
  }
  p.total = off;
  return p;
}

int flag_index(const mz_model* m, int kind, int layer) {
  switch (kind) {
    case MZ_W_STEM_WEIGHT: return 0;
    case MZ_W_STEM_BIAS: return 1;
    case MZ_W_HEAD: return 2;
    case MZ_W_CONV1: return 3 + layer;
    case MZ_W_CONV2: return 3 + m->L + layer;
    case MZ_W_CTRL_WEIGHT: return 3 + 2 * m->L + layer;
    case MZ_W_CTRL_BIAS: return 3 + 3 * m->L + layer;
  }
  return -1;
}

int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}

}  // namespace

// launch convolution `slot` of the model through its prepared-launch cache
static int run_conv(mz_model* m, int slot, const ConvArgs& a, const ConvTcTune& t, cudaStream_t s) {
  mz_model::ConvKey key;
  memset(&key, 0, sizeof(key));
  key.a = a;
  key.t = t;
  if (a.epi.mode == 2) {
    // The head reads the LR image and writes the HR image through plain pointers (no tensor map): the images are not
    // part of what was prepared -- a fresh output tensor per call must not cost a geometry search and two tensor-map
    // encodes.  They and their channel count are patched into the prepared launch below (RGB <-> RGBA swaps the head).
    key.a.epi.img = ImageIo{};
    key.a.epi.nc = 0;
  }
  // kWays prepared launches per convolution: the host lanes, the engine workspace and captured graphs alternate operands
  for (int way = 0; way < kWays; ++way) {
    const int i = kWays * slot + way;
    if (m->prepared[i].valid && memcmp(&key, &m->keys[i], sizeof(key)) == 0) {
      if (a.epi.mode == 2) {
        const int rc = patch_conv_epi(m->prepared[i], a.epi);
        if (rc != MZ_OK) return rc;
      }
      return run_conv_tc(m->prepared[i], s);
    }
  }
  const int i = kWays * slot + m->victim[slot];
  m->victim[slot] = static_cast<uint8_t>((m->victim[slot] + 1) % kWays);
  m->prepared[i].valid = false;
  const int rc = prepare_conv_tc(a, t, m->cfg.device, &m->prepared[i]);
  if (rc != MZ_OK) return rc;
  m->keys[i] = key;
  return run_conv_tc(m->prepared[i], s);
}

// launch fused block `layer` through its prepared-launch cache
static int run_fused(mz_model* m, int layer, const FusedBlockArgs& a, cudaStream_t s) {
  mz_model::FusedKey key;
  memset(&key, 0, sizeof(key));
  key.a = a;
  for (int way = 0; way < kWays; ++way) {
    const int i = kWays * layer + way;
    if (m->fprepared[i].valid && memcmp(&key, &m->fkeys[i], sizeof(key)) == 0) {
      return run_block_fused(m->fprepared[i], s);
    }
  }
  const int i = kWays * layer + m->fvictim[layer];
  m->fvictim[layer] = static_cast<uint8_t>((m->fvictim[layer] + 1) % kWays);
  m->fprepared[i].valid = false;
  const int rc = prepare_block_fused(a, m->cfg.device, &m->fprepared[i]);
  if (rc != MZ_OK) return rc;
  m->fkeys[i] = key;
  return run_block_fused(m->fprepared[i], s);
}

static bool fused_wanted(const mz_model* m) {
  static const bool env_off = getenv("MZ_NO_FUSED_BLOCK") != nullptr;
  return m->fused_ok && !env_off && m->tune[0].block != 2;
}

extern "C" {

int mz_model_fused_block(const mz_model* m) { return (m && fused_wanted(m)) ? 1 : 0; }

int mz_model_create(const mz_config* cfg, mz_model** out) {
  MZ_REQUIRE(cfg && out, "model_create: null pointer");
  *out = nullptr;
  MZ_REQUIRE(cfg->upscale_ratio == 2 || cfg->upscale_ratio == 3 || cfg->upscale_ratio == 4,
             "Upscale ratio must be one of {2, 3, 4}, but got %d.", cfg->upscale_ratio);
  MZ_REQUIRE(cfg->num_channels > 3, "Output channels must be greater than input channels (3), %d given.",
             cfg->num_channels);
  MZ_REQUIRE(cfg->hidden_ratio == 1 || cfg->hidden_ratio == 2 || cfg->hidden_ratio == 4,
             "Hidden ratio must be either 1, 2, or 4, %d given.", cfg->hidden_ratio);
  MZ_REQUIRE(cfg->num_encoder_layers > 0, "Number of encoder layers must be greater than 0, %d given.",
             cfg->num_encoder_layers);
  MZ_REQUIRE(cfg->control_features >= 0 && cfg->control_features <= 64,
             "control_features must be in [0, 64], %d given.", cfg->control_features);
  MZ_REQUIRE(cfg->operand_dtype == MZ_DTYPE_F16 || cfg->operand_dtype == MZ_DTYPE_BF16,
             "operand_dtype must be MZ_DTYPE_F16 or MZ_DTYPE_BF16, %d given.", cfg->operand_dtype);
  MZ_REQUIRE(cfg->residual_stream == MZ_STREAM_AUTO || cfg->residual_stream == MZ_STREAM_FP32,
             "residual_stream must be MZ_STREAM_AUTO or MZ_STREAM_FP32, %d given.", cfg->residual_stream);
  const int hC = cfg->num_channels * cfg->hidden_ratio;
  MZ_REQUIRE(cfg->num_channels <= 512 && hC <= 1024, "num_channels %d / hidden width %d exceed 512 / 1024 channels",
             cfg->num_channels, hC);

  int ndev = 0;
  MZ_CUDA(cudaGetDeviceCount(&ndev));
  MZ_REQUIRE(cfg->device >= 0 && cfg->device < ndev, "device %d out of range (%d visible)", cfg->device, ndev);
  int major = 0;
  MZ_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, cfg->device));
  if (major != 10) {
    set_error("device %d has compute capability %d.x; this library is sm_100a only (no fallback)", cfg->device, major);
    return MZ_ERR_UNSUPPORTED;
  }

  mz_model* m = new mz_model();
  m->cfg = *cfg;
  m->C = cfg->num_channels;
  m->Cp = mz_padded_channels(m->C);
  m->S2 = (m->Cp + 127) / 128;
  m->ns2 = (m->Cp + 16 * m->S2 - 1) / (16 * m->S2) * 16;
  m->Cp = m->S2 * m->ns2;
  m->Cz = mz_zb_pitch(m->Cp);
  m->hC = hC;
  m->hCp = mz_padded_channels(hC);
  m->S = (m->hCp + 255) / 256;
  m->ns = (m->hCp + 16 * m->S - 1) / (16 * m->S) * 16;
  m->hCp = m->S * m->ns;
  m->L = cfg->num_encoder_layers;
  m->r = cfg->upscale_ratio;
  m->F = cfg->control_features;
  m->headN = 3 * m->r * m->r;
  m->headNp = mz_padded_channels(m->headN);
  m->bf16 = cfg->operand_dtype == MZ_DTYPE_BF16;
  m->have.assign(3 + 4 * m->L, 0);
  const int n_convs = (m->S + m->S2) * m->L + 1;
  m->prepared.resize(kWays * n_convs);
  m->keys.resize(kWays * n_convs);
  m->victim.assign(n_convs, 0);
  for (auto& k : m->keys) memset(&k, 0xff, sizeof(k));
  memset(m->tune, 0, sizeof(m->tune));
  const int hm = env_int("MZ_HALO_MODE", 0);  // 1 = diagnostic per-dx loads
  for (int i = 0; i < 3; ++i) m->tune[i].halo_mode = hm;

  DeviceGuard g(cfg->device);
  const size_t c1 = static_cast<size_t>(9) * m->hCp * m->Cz, c2 = static_cast<size_t>(9) * m->Cp * m->hCp;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(p, bytes);
    if (e == cudaSuccess) e = cudaMemset(*p, 0, bytes);
  };
  alloc(reinterpret_cast<void**>(&m->stem_w), sizeof(float) * m->Cp * 3);
  alloc(reinterpret_cast<void**>(&m->stem_b), sizeof(float) * m->Cp);
  alloc(reinterpret_cast<void**>(&m->conv1), sizeof(uint16_t) * c1 * m->L);
  alloc(reinterpret_cast<void**>(&m->conv2), sizeof(uint16_t) * c2 * m->L);
  alloc(reinterpret_cast<void**>(&m->head), sizeof(uint16_t) * 9 * m->headNp * m->Cz);
  m->fused_ok = m->S == 1 && m->S2 == 1 && fused_block_applies(m->Cp, m->hCp, m->Cz);
  // dense layout (3X-Ctrl: 54 / 108 channels move as 56 / 112 instead of 64 / 128: -12.5 % of every block's bytes);
  // not with sliced convolutions (a slice's tensor map starts inside the pixel) -- MZ_NO_DENSE_LAYOUT=1 restores the
  // padded pitches (diagnostic)
  m->Cpm = m->Cp, m->Czm = m->Cz, m->hCm = m->hCp;
  if (m->S == 1 && m->S2 == 1 && !m->fused_ok && getenv("MZ_NO_DENSE_LAYOUT") == nullptr) {
    const int mask = env_int("MZ_DENSE_LAYOUT", 1);  // 1 = fp32 stream, 2 = 16-bit shadow, 4 = hidden tensor
    if (mask & 1) m->Cpm = (m->C + 7) / 8 * 8;
    if (mask & 2) m->Czm = (m->C + 7) / 8 * 8;
    if (mask & 4) m->hCm = (m->hC + 7) / 8 * 8;
  }
  if (m->fused_ok) {
    alloc(reinterpret_cast<void**>(&m->conv2s), sizeof(uint16_t) * c2 * m->L);
    m->fprepared.resize(kWays * m->L);
    m->fkeys.resize(kWays * m->L);
    m->fvictim.assign(m->L, 0);
    for (auto& k : m->fkeys) memset(&k, 0xff, sizeof(k));
  }
  if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&m->sat_host), sizeof(unsigned int), cudaHostAllocMapped);
  if (e == cudaSuccess) {
    *m->sat_host = 0u;
    e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&m->sat_dev), m->sat_host, 0);
  }
  if (m->F > 0) {
    alloc(reinterpret_cast<void**>(&m->ctrl_w), sizeof(float) * m->L * 2 * m->hC * m->F);
    alloc(reinterpret_cast<void**>(&m->ctrl_b), sizeof(float) * m->L * 2 * m->hC);
  }
  for (int i = 0; i < 2; ++i) {
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&m->lane[i].stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->lane[i].kernels_done, cudaEventDisableTiming);
  }
  if (e != cudaSuccess) {
    const int rc = cuda_fail(e, "model allocation", __FILE__, __LINE__);
    mz_model_destroy(m);
    return rc;
  }
  *out = m;
  return MZ_OK;
}

void mz_model_destroy(mz_model* m) {
  if (!m) return;
  DeviceGuard g(m->cfg.device);
  cudaFree(m->stem_w);
  cudaFree(m->stem_b);
  cudaFree(m->conv1);
  cudaFree(m->conv2);
  cudaFree(m->head);
  cudaFree(m->conv2s);
  cudaFree(m->ctrl_w);
  cudaFree(m->ctrl_b);
  cudaFree(m->pack_tmp);
  if (m->sat_host) cudaFreeHost(m->sat_host);
  for (int i = 0; i < 2; ++i) {
    cudaFree(m->lane[i].ws);
    cudaFree(m->lane[i].hx);
    cudaFree(m->lane[i].hy);
    cudaFree(m->lane[i].hc);
    if (m->lane[i].kernels_done) cudaEventDestroy(m->lane[i].kernels_done);
    if (m->lane[i].stream) cudaStreamDestroy(m->lane[i].stream);
  }
  for (cudaEvent_t e : m->ev) cudaEventDestroy(e);
  delete m;
}

static const char* const kRangeMsg =
    "set_weight: a %s weight of layer %d exceeds the fp16 operand range (|w| > 65504 or not finite): it would be clipped "
    "silently -- build the model with operand_dtype bfloat16";

int mz_model_set_weight(mz_model* m, int32_t kind, int32_t layer, const float* host_data, size_t numel) {
  MZ_REQUIRE(m && host_data, "set_weight: null pointer");
  const bool per_layer =
      kind == MZ_W_CONV1 || kind == MZ_W_CONV2 || kind == MZ_W_CTRL_WEIGHT || kind == MZ_W_CTRL_BIAS;
  MZ_REQUIRE(!per_layer || (layer >= 0 && layer < m->L), "set_weight: layer %d out of range [0, %d)", layer, m->L);
  MZ_REQUIRE((kind != MZ_W_CTRL_WEIGHT && kind != MZ_W_CTRL_BIAS) || m->F > 0,
             "set_weight: this model has no control modules");
  DeviceGuard g(m->cfg.device);
  std::vector<uint16_t> packed;
  switch (kind) {
    case MZ_W_STEM_WEIGHT: {
      MZ_REQUIRE(numel == static_cast<size_t>(m->C) * 3, "stem weight: expected %d elements, got %zu", m->C * 3,
                 numel);
      MZ_CUDA(cudaMemcpy(m->stem_w, host_data, sizeof(float) * numel, cudaMemcpyHostToDevice));
      break;
    }
    case MZ_W_STEM_BIAS: {
      MZ_REQUIRE(numel == static_cast<size_t>(m->C), "stem bias: expected %d elements, got %zu", m->C, numel);
      MZ_CUDA(cudaMemcpy(m->stem_b, host_data, sizeof(float) * numel, cudaMemcpyHostToDevice));
      break;
    }
    case MZ_W_CONV1: {
      MZ_REQUIRE(numel == static_cast<size_t>(m->hC) * m->C * 9, "conv1 weight: expected %d elements, got %zu",
                 m->hC * m->C * 9, numel);
      for (int sl = 0; sl < m->S; ++sl) {  // one packed bank per slice of ns output channels
        const int n0 = sl * m->ns, rows = n0 < m->hC ? (m->hC - n0 < m->ns ? m->hC - n0 : m->ns) : 0;
        MZ_REQUIRE(pack_conv_weight_host(host_data + static_cast<size_t>(n0 < m->hC ? n0 : 0) * m->C * 9, rows, m->C, m->ns,
                                         m->Cz, m->bf16, packed), kRangeMsg, "conv1", layer);
        MZ_CUDA(cudaMemcpy(m->conv1 + (static_cast<size_t>(layer) * m->S + sl) * packed.size(), packed.data(),
                           packed.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
      }
      break;
    }
    case MZ_W_CONV2: {
      MZ_REQUIRE(numel == static_cast<size_t>(m->hC) * m->C * 9, "conv2 weight: expected %d elements, got %zu",
                 m->hC * m->C * 9, numel);
      for (int sl = 0; sl < m->S2; ++sl) {  // one packed bank per slice of ns2 output channels
        const int n0 = sl * m->ns2, rows = n0 < m->C ? (m->C - n0 < m->ns2 ? m->C - n0 : m->ns2) : 0;
        MZ_REQUIRE(pack_conv_weight_host(host_data + static_cast<size_t>(n0 < m->C ? n0 : 0) * m->hC * 9, rows, m->hC, m->ns2,
                                         m->hCp, m->bf16, packed), kRangeMsg, "conv2", layer);
        MZ_CUDA(cudaMemcpy(m->conv2 + (static_cast<size_t>(layer) * m->S2 + sl) * packed.size(), packed.data(),
                           packed.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
      }
      if (m->fused_ok) {  // the fused block's view of the same bank
        const size_t bank = static_cast<size_t>(9) * m->Cp * m->hCp;
        const int rc = stack_conv2_bank(m->conv2 + layer * bank, m->conv2s + layer * bank, nullptr);
        if (rc != MZ_OK) return rc;
        MZ_CUDA(cudaStreamSynchronize(nullptr));  // (callers' streams need not be ordered with the legacy stream)
      }
      break;
    }
    case MZ_W_HEAD: {
      MZ_REQUIRE(numel == static_cast<size_t>(m->headN) * m->C * 9, "head weight: expected %d elements, got %zu",
                 m->headN * m->C * 9, numel);
      MZ_REQUIRE(pack_conv_weight_host(host_data, m->headN, m->C, m->headNp, m->Cz, m->bf16, packed), kRangeMsg, "head", 0);
      MZ_CUDA(cudaMemcpy(m->head, packed.data(), packed.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
      break;
    }
    case MZ_W_CTRL_WEIGHT: {
      const size_t n = static_cast<size_t>(2) * m->hC * m->F;
      MZ_REQUIRE(numel == n, "control weight: expected %zu elements, got %zu", n, numel);
      MZ_CUDA(cudaMemcpy(m->ctrl_w + layer * n, host_data, sizeof(float) * n, cudaMemcpyHostToDevice));
      break;
    }
    case MZ_W_CTRL_BIAS: {
      const size_t n = static_cast<size_t>(2) * m->hC;
      MZ_REQUIRE(numel == n, "control bias: expected %zu elements, got %zu", n, numel);
      MZ_CUDA(cudaMemcpy(m->ctrl_b + layer * n, host_data, sizeof(float) * n, cudaMemcpyHostToDevice));
      break;
    }
    default:
      set_error("set_weight: unknown weight kind %d", kind);
      return MZ_ERR_INVALID;
  }
  m->have[flag_index(m, kind, layer)] = 1;
  return MZ_OK;
}

int mz_model_set_weight_dev(mz_model* m, int32_t kind, int32_t layer, const float* dev_data, size_t numel, void* stream) {
  MZ_REQUIRE(m && dev_data, "set_weight_dev: null pointer");
  const bool per_layer =
      kind == MZ_W_CONV1 || kind == MZ_W_CONV2 || kind == MZ_W_CTRL_WEIGHT || kind == MZ_W_CTRL_BIAS;
  MZ_REQUIRE(!per_layer || (layer >= 0 && layer < m->L), "set_weight: layer %d out of range [0, %d)", layer, m->L);
  MZ_REQUIRE((kind != MZ_W_CTRL_WEIGHT && kind != MZ_W_CTRL_BIAS) || m->F > 0,
             "set_weight: this model has no control modules");
  DeviceGuard g(m->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int rc = MZ_OK;
  switch (kind) {
    case MZ_W_STEM_WEIGHT:
      MZ_REQUIRE(numel == static_cast<size_t>(m->C) * 3, "stem weight: expected %d elements, got %zu", m->C * 3, numel);
      MZ_CUDA(cudaMemcpyAsync(m->stem_w, dev_data, sizeof(float) * numel, cudaMemcpyDeviceToDevice, s));
      break;
    case MZ_W_STEM_BIAS:
      MZ_REQUIRE(numel == static_cast<size_t>(m->C), "stem bias: expected %d elements, got %zu", m->C, numel);
      MZ_CUDA(cudaMemcpyAsync(m->stem_b, dev_data, sizeof(float) * numel, cudaMemcpyDeviceToDevice, s));
      break;
    case MZ_W_CONV1: {
      MZ_REQUIRE(numel == static_cast<size_t>(m->hC) * m->C * 9, "conv1 weight: expected %d elements, got %zu",
                 m->hC * m->C * 9, numel);
      const size_t bank = static_cast<size_t>(9) * m->ns * m->Cz;
      for (int sl = 0; sl < m->S && rc == MZ_OK; ++sl) {
        const int n0 = sl * m->ns, rows = n0 < m->hC ? (m->hC - n0 < m->ns ? m->hC - n0 : m->ns) : 0;
        rc = launch_pack_conv_weight(dev_data + static_cast<size_t>(n0 < m->hC ? n0 : 0) * m->C * 9,
                                     m->conv1 + (static_cast<size_t>(layer) * m->S + sl) * bank, rows, m->C, m->ns, m->Cz,
                                     m->bf16, m->sat_dev, s);
      }
      break;
    }
    case MZ_W_CONV2: {
      MZ_REQUIRE(numel == static_cast<size_t>(m->hC) * m->C * 9, "conv2 weight: expected %d elements, got %zu",
                 m->hC * m->C * 9, numel);
      const size_t bank = static_cast<size_t>(9) * m->ns2 * m->hCp;
      for (int sl = 0; sl < m->S2 && rc == MZ_OK; ++sl) {
        const int n0 = sl * m->ns2, rows = n0 < m->C ? (m->C - n0 < m->ns2 ? m->C - n0 : m->ns2) : 0;
        rc = launch_pack_conv_weight(dev_data + static_cast<size_t>(n0 < m->C ? n0 : 0) * m->hC * 9,
                                     m->conv2 + (static_cast<size_t>(layer) * m->S2 + sl) * bank, rows, m->hC, m->ns2,
                                     m->hCp, m->bf16, m->sat_dev, s);
      }
      if (rc == MZ_OK && m->fused_ok) rc = stack_conv2_bank(m->conv2 + layer * bank, m->conv2s + layer * bank, s);
      break;
    }
    case MZ_W_HEAD:
      MZ_REQUIRE(numel == static_cast<size_t>(m->headN) * m->C * 9, "head weight: expected %d elements, got %zu",
                 m->headN * m->C * 9, numel);
      rc = launch_pack_conv_weight(dev_data, m->head, m->headN, m->C, m->headNp, m->Cz, m->bf16, m->sat_dev, s);
      break;
    case MZ_W_CTRL_WEIGHT: {
      const size_t n = static_cast<size_t>(2) * m->hC * m->F;
      MZ_REQUIRE(numel == n, "control weight: expected %zu elements, got %zu", n, numel);
      MZ_CUDA(cudaMemcpyAsync(m->ctrl_w + layer * n, dev_data, sizeof(float) * n, cudaMemcpyDeviceToDevice, s));
      break;
    }
    case MZ_W_CTRL_BIAS: {
      const size_t n = static_cast<size_t>(2) * m->hC;
      MZ_REQUIRE(numel == n, "control bias: expected %zu elements, got %zu", n, numel);
      MZ_CUDA(cudaMemcpyAsync(m->ctrl_b + layer * n, dev_data, sizeof(float) * n, cudaMemcpyDeviceToDevice, s));
      break;
    }
    default:
      set_error("set_weight: unknown weight kind %d", kind);
      return MZ_ERR_INVALID;
  }
  if (rc != MZ_OK) return rc;
  m->have[flag_index(m, kind, layer)] = 1;
  return MZ_OK;
}

int mz_model_saturated(mz_model* m, int32_t reset, int32_t* saturated) {
  MZ_REQUIRE(m && saturated, "saturated: null pointer");
  *saturated = (m->sat_host && *static_cast<volatile unsigned int*>(m->sat_host)) ? 1 : 0;
  if (reset && m->sat_host) *static_cast<volatile unsigned int*>(m->sat_host) = 0u;
  return MZ_OK;
}

int mz_model_set_tune(mz_model* m, int32_t which, const mz_conv_tune* tune) {
  MZ_REQUIRE(m, "set_tune: null model");
  MZ_REQUIRE(which >= -1 && which <= 2, "set_tune: which must be -1..2, %d given", which);
  const ConvTcTune t = to_tune(tune);
  for (int i = 0; i < 3; ++i)
    if (which < 0 || which == i) m->tune[i] = t;
  return MZ_OK;
}

int mz_model_enable_timing(mz_model* m, int32_t enable) {
  MZ_REQUIRE(m, "enable_timing: null model");
  DeviceGuard g(m->cfg.device);
  if (enable && m->ev.empty()) {
    m->ev.resize(2 * kTimingSlots, nullptr);
    for (auto& e : m->ev) MZ_CUDA(cudaEventCreate(&e));
  }
  m->timing = enable != 0;
  m->timing_calls = 0;
  return MZ_OK;
}

int mz_model_conv_stack_ms(mz_model* m, float* ms) {
  MZ_REQUIRE(m && ms, "conv_stack_ms: null pointer");
  if (!m->timing || m->timing_calls == 0) {
    set_error("conv_stack_ms: timing is not enabled or no mz_upscale call has been made since");
    return MZ_ERR_STATE;
  }
  DeviceGuard g(m->cfg.device);
  const int n = m->timing_calls < kTimingSlots ? m->timing_calls : kTimingSlots;
  double sum = 0.0;
  for (int i = 0; i < n; ++i) {
    float t = 0.f;
    MZ_CUDA(cudaEventSynchronize(m->ev[2 * i + 1]));
    MZ_CUDA(cudaEventElapsedTime(&t, m->ev[2 * i], m->ev[2 * i + 1]));
    sum += t;
  }
  *ms = static_cast<float>(sum / n);
  return MZ_OK;
}

int mz_workspace_bytes(const mz_model* m, int32_t B, int32_t H, int32_t W, size_t* bytes) {
  MZ_REQUIRE(m && bytes, "workspace_bytes: null pointer");
  MZ_REQUIRE(B > 0 && H > 0 && W > 0, "workspace_bytes: empty input (B %d, H %d, W %d)", B, H, W);
  *bytes = plan_ws(m, B, H, W).total;
  return MZ_OK;
}

int mz_workspace_bytes_flags(const mz_model* m, int32_t B, int32_t H, int32_t W, uint32_t flags, size_t* bytes) {
  MZ_REQUIRE(m && bytes, "workspace_bytes: null pointer");
  MZ_REQUIRE(B > 0 && H > 0 && W > 0, "workspace_bytes: empty input (B %d, H %d, W %d)", B, H, W);
  *bytes = plan_ws(m, B, H, W, flags).total;
  return MZ_OK;
}

}  // extern "C"

// output window of mz_upscale_window and mz_upscale_stage (nullptr: the whole image, densely)
struct OutWindow {
  int y0, y1, x0, x1;
  long long row_pitch, plane_pitch;
};

// element type of both images: fp32, 8 bits (MZ_FLAG_IO_U8) or 16 bits (MZ_FLAG_IO_U16), and its size in bytes
static int image_type(uint32_t flags) {
  return (flags & MZ_FLAG_IO_U8) ? kImgU8 : ((flags & MZ_FLAG_IO_U16) ? kImgU16 : kImgF32);
}
static int type_bytes(int type) { return type == kImgU8 ? 1 : (type == kImgU16 ? 2 : 4); }
// channels per pixel of an image: 4 with MZ_FLAG_RGBA, otherwise 3
static int image_channels(uint32_t flags) { return (flags & MZ_FLAG_RGBA) ? 4 : 3; }
// bytes of one image: 3HW (RGBA: 4HW) elements of fp32, 8 or 16 bits, or a 4:2:0 frame of 3HW/2
static size_t image_bytes(uint32_t flags, int H, int W) {
  const size_t es = type_bytes(image_type(flags));
  const size_t px = static_cast<size_t>(H) * W;
  return (flags & MZ_FLAG_YUV420) ? px * 3 / 2 * es : px * image_channels(flags) * es;
}

// The images of a call -- its flags, the H x W input x, the output y and its window (nullptr: the whole image, densely)
// -- as the stem and head read them (*img, *nc channels per pixel), or MZ_ERR_INVALID.  staged: a call of
// mz_upscale_stage.  Every entry point refuses here, before anything is enqueued.
static int image_io(const mz_model* m, const void* x, void* y, uint32_t flags, int H, int W, const OutWindow* win,
                    bool staged, ImageIo* img, int* nc) {
  // y holds the bicubic image of a planar fp32 RGB x, whole: every other image recomputes the skip
  MZ_REQUIRE(!(flags & MZ_FLAG_SKIP_FROM_BUFFER) ||
                 !(win || staged || (flags & (MZ_FLAG_IO_U8 | MZ_FLAG_IO_U16 | MZ_FLAG_YUV420 | MZ_FLAG_RGBA |
                                              MZ_FLAG_X_NHWC | MZ_FLAG_Y_NHWC))),
             "upscale: MZ_FLAG_SKIP_FROM_BUFFER takes a planar fp32 RGB image, neither windowed nor staged");
  MZ_REQUIRE(!(flags & (MZ_FLAG_IO_U8 | MZ_FLAG_IO_U16)) || (flags & MZ_FLAG_CLAMP01),
             "upscale: 8- and 16-bit image I/O needs MZ_FLAG_CLAMP01");
  MZ_REQUIRE(!(flags & MZ_FLAG_IO_U16) || !(flags & (MZ_FLAG_IO_U8 | MZ_FLAG_U8_TRUNC)),
             "upscale: 16-bit image I/O excludes MZ_FLAG_IO_U8 and MZ_FLAG_U8_TRUNC");
  MZ_REQUIRE((flags & MZ_FLAG_YUV420) || !(flags & kYuvColourFlags),
             "upscale: the colour bits MZ_FLAG_YUV_* apply to 4:2:0 frames only (MZ_FLAG_YUV420)");
  if (flags & MZ_FLAG_YUV420) {
    YuvCoef k;
    const int rc = yuv_coef(flags, &k);  // (NV12 or P010, one colour matrix)
    if (rc != MZ_OK) return rc;
    MZ_REQUIRE(!(flags & (MZ_FLAG_X_NHWC | MZ_FLAG_Y_NHWC | MZ_FLAG_U8_TRUNC | MZ_FLAG_RGBA)),
               "upscale: 4:2:0 frames exclude MZ_FLAG_X_NHWC, MZ_FLAG_Y_NHWC, MZ_FLAG_U8_TRUNC and MZ_FLAG_RGBA");
    MZ_REQUIRE(!win && !staged, "upscale: 4:2:0 frames are neither windowed nor staged");
    MZ_REQUIRE(H % 2 == 0 && W % 2 == 0, "upscale: a 4:2:0 frame has even dimensions, %d x %d given", H, W);
  }
  *img = ImageIo{};
  *nc = image_channels(flags);
  img->x = x;
  img->y = y;
  img->type = image_type(flags);
  img->x_nhwc = (flags & MZ_FLAG_X_NHWC) ? 1 : 0;
  img->y_nhwc = (flags & MZ_FLAG_Y_NHWC) ? 1 : 0;
  img->u8_trunc = (flags & MZ_FLAG_U8_TRUNC) ? 1 : 0;
  img->skip_mode = (flags & MZ_FLAG_SKIP_FROM_BUFFER) ? 1 : 2;
  img->clamp01 = (flags & MZ_FLAG_CLAMP01) ? 1 : 0;
  MZ_REQUIRE(!(img->x_nhwc || img->y_nhwc) || static_cast<long long>(H) * W * *nc < (1LL << 31),
             "upscale: an interleaved %d x %d x %d image exceeds 2^31 elements", H, W, *nc);
  if (!win) return MZ_OK;
  MZ_REQUIRE(0 <= win->y0 && win->y0 < win->y1 && win->y1 <= H && 0 <= win->x0 && win->x0 < win->x1 && win->x1 <= W,
             "upscale: window [%d, %d) x [%d, %d) is not inside the %d x %d input", win->y0, win->y1, win->x0, win->x1, H,
             W);
  const long long r = m->r, ch = img->y_nhwc ? *nc : 1;  // (elements per HR pixel in a row)
  MZ_REQUIRE(win->row_pitch >= (win->x1 - win->x0) * r * ch && win->plane_pitch >= win->row_pitch * (win->y1 - win->y0) * r,
             "upscale: pitches (%lld, %lld) are smaller than the window", win->row_pitch, win->plane_pitch);
  // bytes of one vector store: RGB the same in both layouts (an interleaved HR row segment of a pixel is three of them);
  // interleaved RGBA stores a pixel's row segment of 4r values in the widest vectors that divide its 4r es bytes, up to 16
  const int es = type_bytes(img->type), seg = 4 * m->r * es;
  const int vec = (*nc == 4 && img->y_nhwc) ? (seg % 16 == 0 ? 16 : (seg % 8 == 0 ? 8 : 4)) : m->r == 3 ? es : es * m->r;
  MZ_REQUIRE(reinterpret_cast<uintptr_t>(y) % vec == 0 && (win->row_pitch * es) % vec == 0 &&
                 (win->plane_pitch * es) % vec == 0,
             "upscale: y and its pitches must be aligned to %d bytes", vec);
  img->wy0 = win->y0;
  img->wy1 = win->y1;
  img->wx0 = win->x0;
  img->wx1 = win->x1;
  img->y_row = win->row_pitch;
  img->y_plane = win->plane_pitch;
  return MZ_OK;
}

// layer_begin / layer_end: the encoder blocks [layer_begin, layer_end) of this call (mz_upscale_stage).  The FiLM table and
// the stem run when layer_begin == 0, the head when layer_end == L; in between the state lives in the workspace.
static int upscale_impl(mz_model* m, const void* x_dev_v, const float* c_dev, int32_t c_rows, void* y_dev_v, int32_t B,
                        int32_t H, int32_t W, void* workspace_dev, size_t workspace_bytes, uint32_t flags, void* stream,
                        const OutWindow* win, bool staged = false, int layer_begin = 0, int layer_end = -1) {
  MZ_REQUIRE(m && x_dev_v && y_dev_v && workspace_dev, "upscale: null pointer");
  if (layer_end < 0) layer_end = m->L;
  MZ_REQUIRE(0 <= layer_begin && layer_begin <= layer_end && layer_end <= m->L, "upscale: bad layer range [%d, %d) of %d",
             layer_begin, layer_end, m->L);
  const bool front = layer_begin == 0, back = layer_end == m->L;
  ImageIo img;
  int nc;
  const int irc = image_io(m, x_dev_v, y_dev_v, flags, H, W, win, staged, &img, &nc);
  if (irc != MZ_OK) return irc;
  const bool yuv = (flags & MZ_FLAG_YUV420) != 0;
  MZ_REQUIRE(B > 0 && H > 0 && W > 0, "upscale: empty input (B %d, H %d, W %d)", B, H, W);
  if (m->F > 0) {
    MZ_REQUIRE(c_dev != nullptr, "Control vector c is required for control models.");
    MZ_REQUIRE(c_rows == 1 || c_rows == B, "Batch size of c (%d) must match x (%d).", c_rows, B);
  } else {
    MZ_REQUIRE(c_dev == nullptr, "This model has no control modules; c must be None.");
  }
  for (size_t i = 0; i < m->have.size(); ++i) {
    const bool ctrl = i >= static_cast<size_t>(3 + 2 * m->L);
    if (!m->have[i] && (!ctrl || m->F > 0)) {
      set_error("upscale: weights not fully set (missing slot %zu)", i);
      return MZ_ERR_STATE;
    }
  }
  const WsPlan wp = plan_ws(m, B, H, W, flags);
  if (workspace_bytes < wp.total) {
    set_error("upscale: workspace too small (%zu < %zu bytes)", workspace_bytes, wp.total);
    return MZ_ERR_WORKSPACE;
  }
  MZ_REQUIRE((reinterpret_cast<uintptr_t>(workspace_dev) & 1023) == 0, "upscale: workspace must be 1024-byte aligned");

  DeviceGuard g(m->cfg.device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
  float* zf = reinterpret_cast<float*>(ws + wp.zf);
  uint16_t* zb = reinterpret_cast<uint16_t*>(ws + wp.zb);
  uint16_t* hid = reinterpret_cast<uint16_t*>(ws + wp.hid);
  float* film = reinterpret_cast<float*>(ws + wp.film);
  const bool simt = (flags & MZ_FLAG_SIMT_CONV) != 0;
  int rc;
  if (yuv) {  // decode, the 16-bit planar upscale, encode (the intermediates follow its workspace)
    uint16_t* lr = reinterpret_cast<uint16_t*>(ws + wp.rgb_lr);
    uint16_t* hr = reinterpret_cast<uint16_t*>(ws + wp.rgb_hr);
    rc = launch_yuv420_to_rgb16(x_dev_v, lr, B, H, W, flags, s);
    if (rc != MZ_OK) return rc;
    const uint32_t f16 = (flags & ~(MZ_FLAG_YUV420 | kYuvColourFlags | MZ_FLAG_IO_U8)) | MZ_FLAG_IO_U16;
    rc = upscale_impl(m, lr, c_dev, c_rows, hr, B, H, W, workspace_dev, wp.rgb_lr, f16, stream, nullptr);
    if (rc != MZ_OK) return rc;
    return launch_rgb16_to_yuv420(hr, y_dev_v, B, H * m->r, W * m->r, flags, s);
  }

  if (front && m->F > 0) {
    rc = launch_film(c_dev, c_rows, m->ctrl_w, m->ctrl_b, film, m->L, B, m->F, m->hC, m->hCp, m->ns, s);
    if (rc != MZ_OK) return rc;
  }
  rc = MZ_OK;
  if (front)
    rc = launch_stem(img.x, img.type, img.x_nhwc, nc, m->stem_w, m->stem_b, zf, zb, m->bf16, B, H, W, m->Cpm, m->Czm, s,
                     m->sat_dev);
  if (rc != MZ_OK) return rc;

  const int slot = m->timing_calls % kTimingSlots;
  if (m->timing && front) MZ_CUDA(cudaEventRecord(m->ev[2 * slot], s));
  // one slice of conv1's / conv2's filter bank
  const size_t c1s = static_cast<size_t>(9) * m->ns * m->Cz, c2s = static_cast<size_t>(9) * m->ns2 * m->hCp;
  const int S = m->S, S2 = m->S2;
  // Fused blocks (48-channel models): one kernel per block, the hidden tensor stays on the SM; the 16-bit stream
  // ping-pongs between zb and the hidden buffer (a block reads its input with a halo, so it cannot write in place).
  const bool fused = !simt && fused_wanted(m);
  if (m->tune[0].block == 1 && !fused) {
    set_error("upscale: the fused encoder block was required (tune.block = 1) but does not apply to this model / call");
    return MZ_ERR_UNSUPPORTED;
  }
  // (after an odd number of fused blocks the 16-bit stream lives in the hidden buffer: mz_workspace_layout documents it)
  uint16_t* zcur = (fused && (layer_begin & 1)) ? hid : zb;
  uint16_t* znxt = (fused && (layer_begin & 1)) ? zb : hid;
  for (int l = layer_begin; l < layer_end && fused; ++l) {
    FusedBlockArgs fa;
    memset(&fa, 0, sizeof(fa));
    fa.zb_in = zcur;
    fa.zb_out = znxt;
    fa.zf = zf;
    fa.w1 = m->conv1 + static_cast<size_t>(l) * c1s;
    fa.w2s = m->conv2s + static_cast<size_t>(l) * c2s;
    fa.film = m->F > 0 ? film + static_cast<size_t>(l) * B * 2 * m->ns : nullptr;
    fa.sat = m->sat_dev;
    fa.B = B;
    fa.H = H;
    fa.W = W;
    fa.bf16 = m->bf16;
    fa.seg_rows = m->tune[0].seg_rows;
    fa.max_ctas = m->tune[0].max_ctas;
    rc = run_fused(m, l, fa, s);
    if (rc != MZ_OK) return rc;
    uint16_t* t = zcur;
    zcur = znxt;
    znxt = t;
  }
  for (int l = layer_begin; l < layer_end && !fused; ++l) {
    ConvArgs a;
    for (int sl = 0; sl < S; ++sl) {
      memset(&a, 0, sizeof(a));
      a.in = zb;
      a.w = m->conv1 + (static_cast<size_t>(l) * S + sl) * c1s;
      a.cin_p = m->Cz;
      a.in_pitch = m->Czm != m->Cz ? m->Czm : 0;
      a.in_extent = m->Czm != m->Cz ? m->Czm : 0;
      a.epi.mode = 0;
      a.epi.bf16 = m->bf16;
      a.epi.B = B;
      a.epi.H = H;
      a.epi.W = W;
      a.epi.n_pad = m->ns;
      a.epi.film = m->F > 0 ? film + (static_cast<size_t>(l) * S + sl) * B * 2 * m->ns : nullptr;
      a.epi.out_bf16 = hid + static_cast<size_t>(sl) * m->ns;
      a.epi.out_pitch = (S > 1 || m->hCm != m->hCp) ? m->hCm : 0;
      a.epi.out_extent = m->hCm != m->hCp ? m->hCm : 0;
      a.epi.sat = m->sat_dev;
      rc = simt ? launch_conv_simt(a, s) : run_conv(m, l * (S + S2) + sl, a, m->tune[0], s);
      if (rc != MZ_OK) return rc;
    }

    for (int sl = 0; sl < S2; ++sl) {
      memset(&a, 0, sizeof(a));
      a.in = hid;
      a.w = m->conv2 + (static_cast<size_t>(l) * S2 + sl) * c2s;
      a.cin_p = m->hCp;
      a.k_valid = S == 1 ? (m->hC + 15) / 16 * 16 : 0;  // (hidden channels >= hC are SiLU(0) = 0, written by conv1)
      a.in_pitch = m->hCm != m->hCp ? m->hCm : 0;
      a.in_extent = m->hCm != m->hCp ? m->hCm : 0;
      a.epi.mode = 1;
      a.epi.bf16 = m->bf16;
      a.epi.B = B;
      a.epi.H = H;
      a.epi.W = W;
      a.epi.n_pad = m->ns2;
      a.epi.out_bf16 = zb + static_cast<size_t>(sl) * m->ns2;
      a.epi.out_pitch = m->Czm;
      a.epi.out_extent = m->Czm < m->ns2 ? m->Czm : 0;
      a.epi.zf = zf + static_cast<size_t>(sl) * m->ns2;
      a.epi.zf_pitch = (S2 > 1 || m->Cpm != m->Cp) ? m->Cpm : 0;
      a.epi.zf_extent = m->Cpm != m->Cp ? m->Cpm : 0;
      a.epi.sat = m->sat_dev;
      rc = simt ? launch_conv_simt(a, s) : run_conv(m, l * (S + S2) + S + sl, a, m->tune[1], s);
      if (rc != MZ_OK) return rc;
    }
  }

  if (m->timing && back) {
    MZ_CUDA(cudaEventRecord(m->ev[2 * slot + 1], s));
    ++m->timing_calls;
  }
  if (!back) return MZ_OK;

  if (img.skip_mode == 1) {  // (planar fp32 RGB only: image_io)
    rc = launch_bicubic(static_cast<const float*>(img.x), static_cast<float*>(img.y), B * 3, H, W, m->r, s);
    if (rc != MZ_OK) return rc;
  }
  ConvArgs a;
  memset(&a, 0, sizeof(a));
  a.in = zcur;
  a.w = m->head;
  a.cin_p = m->Cz;
  a.in_pitch = m->Czm != m->Cz ? m->Czm : 0;
  a.in_extent = m->Czm != m->Cz ? m->Czm : 0;
  a.epi.mode = 2;
  a.epi.bf16 = m->bf16;
  a.epi.B = B;
  a.epi.H = H;
  a.epi.W = W;
  a.epi.n_pad = m->headNp;
  a.epi.img = img;
  a.epi.r = m->r;
  a.epi.nc = nc;
  make_bicubic_table(m->r, &a.epi.bt);
  return simt ? launch_conv_simt(a, s) : run_conv(m, m->L * (S + S2), a, m->tune[2], s);
}

extern "C" {

int mz_upscale(mz_model* m, const void* x_dev, const float* c_dev, int32_t c_rows, void* y_dev, int32_t B, int32_t H,
               int32_t W, void* workspace_dev, size_t workspace_bytes, uint32_t flags, void* stream) {
  return upscale_impl(m, x_dev, c_dev, c_rows, y_dev, B, H, W, workspace_dev, workspace_bytes, flags, stream, nullptr);
}

int mz_upscale_window(mz_model* m, const void* x_dev, const float* c_dev, int32_t c_rows, void* y_dev, int64_t y_row_pitch,
                      int64_t y_plane_pitch, int32_t B, int32_t H, int32_t W, int32_t win_y0, int32_t win_y1,
                      int32_t win_x0, int32_t win_x1, void* workspace_dev, size_t workspace_bytes, uint32_t flags,
                      void* stream) {
  const OutWindow w{win_y0, win_y1, win_x0, win_x1, y_row_pitch, y_plane_pitch};
  return upscale_impl(m, x_dev, c_dev, c_rows, y_dev, B, H, W, workspace_dev, workspace_bytes, flags, stream, &w);
}

int mz_upscale_stage(mz_model* m, const void* x_dev, const float* c_dev, int32_t c_rows, void* y_dev, int64_t y_row_pitch,
                     int64_t y_plane_pitch, int32_t B, int32_t H, int32_t W, int32_t win_y0, int32_t win_y1, int32_t win_x0,
                     int32_t win_x1, void* workspace_dev, size_t workspace_bytes, uint32_t flags, void* stream,
                     int32_t layer_begin, int32_t layer_end) {
  const OutWindow w{win_y0, win_y1, win_x0, win_x1, y_row_pitch, y_plane_pitch};
  return upscale_impl(m, x_dev, c_dev, c_rows, y_dev, B, H, W, workspace_dev, workspace_bytes, flags, stream,
                      win_y1 > 0 ? &w : nullptr, true, layer_begin, layer_end);  // (win_y1 <= 0: dense output)
}

int mz_workspace_layout(const mz_model* m, int32_t B, int32_t H, int32_t W, size_t* zf_offset, size_t* zb_offset,
                        size_t* hidden_offset, int32_t* channels_padded, int32_t* zb_pitch) {
  MZ_REQUIRE(m && zf_offset && zb_offset && hidden_offset && channels_padded && zb_pitch, "workspace_layout: null pointer");
  MZ_REQUIRE(B > 0 && H > 0 && W > 0, "workspace_layout: empty input");
  const WsPlan wp = plan_ws(m, B, H, W);
  *zf_offset = wp.zf;
  *zb_offset = wp.zb;
  *hidden_offset = wp.hid;
  *channels_padded = m->Cpm;
  *zb_pitch = m->Czm;
  return MZ_OK;
}

// one chunk (B images) on one lane: H2D, kernels, D2H -- all asynchronous on the lane's stream
static int host_enqueue(mz_model* m, int li, const void* x_host, const float* c_host, int32_t c_rows, void* y_host,
                        int32_t B, int32_t H, int32_t W, uint32_t flags) {
  mz_model::HostLane& L = m->lane[li];
  const size_t xb = image_bytes(flags, H, W) * B;
  const size_t yb = xb * m->r * m->r;
  const size_t cb = c_host ? sizeof(float) * c_rows * (m->F > 0 ? m->F : 1) : 0;
  size_t wsb = 0;
  int rc = mz_workspace_bytes_flags(m, B, H, W, flags, &wsb);
  if (rc != MZ_OK) return rc;
  auto ensure = [&](void** p, size_t* have, size_t need) -> int {
    if (*have >= need) return MZ_OK;
    MZ_CUDA(cudaStreamSynchronize(L.stream));  // nothing in flight may still use the old buffer
    if (*p) cudaFree(*p);
    *p = nullptr;
    *have = 0;
    MZ_CUDA(cudaMalloc(p, need));
    *have = need;
    return MZ_OK;
  };
  if ((rc = ensure(reinterpret_cast<void**>(&L.hx), &L.hx_bytes, xb)) != MZ_OK) return rc;
  if ((rc = ensure(reinterpret_cast<void**>(&L.hy), &L.hy_bytes, yb)) != MZ_OK) return rc;
  if (cb && (rc = ensure(reinterpret_cast<void**>(&L.hc), &L.hc_bytes, cb)) != MZ_OK) return rc;
  // (cudaMalloc only promises 256-byte alignment, and where a small block lands depends on what the process allocated
  // before; the workspace must start on a 1024-byte boundary)
  if ((rc = ensure(&L.ws, &L.ws_bytes, wsb + 1024)) != MZ_OK) return rc;
  uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(L.ws) + 1023) & ~static_cast<uintptr_t>(1023));
  const size_t ws_bytes = L.ws_bytes - static_cast<size_t>(ws - static_cast<uint8_t*>(L.ws));
  MZ_CUDA(cudaMemcpyAsync(L.hx, x_host, xb, cudaMemcpyHostToDevice, L.stream));
  if (cb) MZ_CUDA(cudaMemcpyAsync(L.hc, c_host, cb, cudaMemcpyHostToDevice, L.stream));
  // The two lanes take turns on the SMs: this lane's kernels start when the other lane's have finished, so that one
  // step's kernels run back to back (programmatic dependent launch, L2 prefetch) while the copies of its neighbours
  // proceed on the copy engines -- instead of the kernels of two steps interleaving and both finishing late.
  mz_model::HostLane& O = m->lane[li ^ 1];
  if (O.has_work) MZ_CUDA(cudaStreamWaitEvent(L.stream, O.kernels_done, 0));
  rc = mz_upscale(m, L.hx, cb ? L.hc : nullptr, c_rows, L.hy, B, H, W, ws, ws_bytes, flags, L.stream);
  if (rc != MZ_OK) return rc;
  MZ_CUDA(cudaEventRecord(L.kernels_done, L.stream));
  L.has_work = true;
  MZ_CUDA(cudaMemcpyAsync(y_host, L.hy, yb, cudaMemcpyDeviceToHost, L.stream));
  return MZ_OK;
}

int mz_upscale_host_async(mz_model* m, int32_t lane, const void* x_host, const float* c_host, int32_t c_rows,
                          void* y_host, int32_t B, int32_t H, int32_t W, uint32_t flags) {
  MZ_REQUIRE(m && x_host && y_host, "upscale_host_async: null pointer");
  MZ_REQUIRE(lane == 0 || lane == 1, "upscale_host_async: lane must be 0 or 1, %d given", lane);
  MZ_REQUIRE(B > 0 && H > 0 && W > 0, "upscale_host_async: empty input (B %d, H %d, W %d)", B, H, W);
  ImageIo img;
  int nc;
  const int irc = image_io(m, x_host, y_host, flags, H, W, nullptr, false, &img, &nc);  // (before the copies are enqueued)
  if (irc != MZ_OK) return irc;
  DeviceGuard g(m->cfg.device);
  return host_enqueue(m, lane, x_host, c_host, c_rows, y_host, B, H, W, flags);
}

int mz_upscale_host_wait(mz_model* m, int32_t lane) {
  MZ_REQUIRE(m, "upscale_host_wait: null model");
  MZ_REQUIRE(lane >= -1 && lane <= 1, "upscale_host_wait: lane must be -1 (both), 0 or 1, %d given", lane);
  DeviceGuard g(m->cfg.device);
  for (int i = 0; i < 2; ++i)
    if (lane < 0 || lane == i) MZ_CUDA(cudaStreamSynchronize(m->lane[i].stream));
  return MZ_OK;
}

int mz_upscale_host(mz_model* m, const void* x_host_v, const float* c_host, int32_t c_rows, void* y_host_v, int32_t B,
                    int32_t H, int32_t W, uint32_t flags) {
  const uint8_t* x_host = static_cast<const uint8_t*>(x_host_v);
  uint8_t* y_host = static_cast<uint8_t*>(y_host_v);
  MZ_REQUIRE(m && x_host && y_host, "upscale_host: null pointer");
  MZ_REQUIRE(B > 0 && H > 0 && W > 0, "upscale_host: empty input (B %d, H %d, W %d)", B, H, W);
  ImageIo img;
  int nc;
  const int irc = image_io(m, x_host, y_host, flags, H, W, nullptr, false, &img, &nc);  // (before the copies are enqueued)
  if (irc != MZ_OK) return irc;
  if (m->F > 0) {
    MZ_REQUIRE(c_host != nullptr, "Control vector c is required for control models.");
    MZ_REQUIRE(c_rows == 1 || c_rows == B, "Batch size of c (%d) must match x (%d).", c_rows, B);
  }
  DeviceGuard g(m->cfg.device);
  // A batch is cut into up to eight chunks that alternate between the two lanes: copies of chunk i+1 / i-1 run under
  // the kernels of chunk i.  (Images are independent: chunking does not change any result.)
  const int n_chunks = B >= 8 ? 8 : B;
  const size_t x_img = image_bytes(flags, H, W), y_img = x_img * m->r * m->r;  // bytes per image
  const int F = m->F > 0 ? m->F : 1;
  int b0 = 0, rc = MZ_OK;
  for (int i = 0; i < n_chunks && rc == MZ_OK; ++i) {
    const int nb = (B - b0 + (n_chunks - i) - 1) / (n_chunks - i);
    const float* cc = c_host ? (c_rows == B ? c_host + static_cast<size_t>(b0) * F : c_host) : nullptr;
    rc = host_enqueue(m, i & 1, x_host + b0 * x_img, cc, c_host ? (c_rows == B ? nb : 1) : 0, y_host + b0 * y_img, nb,
                      H, W, flags);
    b0 += nb;
  }
  for (int i = 0; i < 2; ++i) {
    const cudaError_t e = cudaStreamSynchronize(m->lane[i].stream);
    if (e != cudaSuccess && rc == MZ_OK) rc = cuda_fail(e, "upscale_host synchronize", __FILE__, __LINE__);
  }
  return rc;
}

}  // extern "C"
