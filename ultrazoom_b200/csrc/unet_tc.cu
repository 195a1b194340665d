// unet_tc.cu -- AdaptiveResidualMix (reference model.py:795-839) and PixelCrush (model.py:842-882) as ONE tcgen05 GEMM
// kernel that reads the fp32 NHWC feature maps as they lie in HBM (kind::tf32: fp32 containers, 10-bit mantissa operands,
// fp32 accumulation in TMEM) -- no 16-bit copy of the activations, no im2col:
//
//   D[128 output pixels][N] = sum over K segments ("taps")  A_tap[128 pixels][C] * W[N][tap*C .. tap*C + C)^T
//     mix:    two taps, the same pixel of x and of z (K = 2C);              epilogue  out = (1 - w) x + w z,  w = s(alpha) s(D)
//     crush:  f*f taps, input pixel (yo f + i, xo f + j) of output pixel (yo, xo) (K = f f Cin);   epilogue  out = D
//
// A tile of a tap is one TMA box of a 4-D view (channel, j, xo, input row) of the feature map -- 128 pixels x 32 channels
// = 128-byte rows, 128-byte swizzle, the K-major operand layout as it lands; channels past C arrive as zeros (TMA
// out-of-bounds fill), so C needs no padding and the weight matrix [N][K] is read as the reference stores it
// (conv.weight reshaped), one TMA box per 32-channel chunk.  On a dense map (pitch = C) the f pixels under one output
// pixel of the crush are f C consecutive floats, so a whole input row is one K segment.  The [ns][K] weight slice of the
// CTA stays in shared memory when it fits beside three ring stages (else N is sliced over CTAs, or -- deep K -- the weight
// chunks travel through the ring with their A chunks: whichever moves fewer bytes per tile through L2).
//
// Roles (192 | 320 threads, persistent over tiles): warp 0 TMA producer (a ring of 3-6 A chunks), warp 1 TMEM allocation
// + UMMA issue (4 x K = 8 per chunk, two accumulator stages), 4 (crush) or 8 (mix) epilogue warps: per 16-channel slice
// tcgen05.ld -> (mix: the x and z slices of the warp's 32 pixels, TMA-loaded two slices ahead into the warp's own slots --
// L2 hits, the producer fetched them for the GEMM a moment ago) -> fp32 slice (+ optional 16-bit shadow) written in
// place -> TMA store.  Everything a pixel needs is read from HBM once and written once: 12 C bytes per pixel for the mix,
// 4 (f f Cin + Cout) for the crush; tf32 tensor time is a fifth of the HBM time at C = 96, so the roofline is HBM.
// Measured (one B200, maps larger than L2; tools/unet_shapes.py): mix 4.2-5.9 TB/s over C = 32 .. 192, crush 5.2-5.9 TB/s
// (0.64-0.90 of the 6.55 TB/s copy peak) -- the fp32 SIMT twin of unet_ops.cu runs the same shapes at 0.4-0.5 TB/s.
// What it took beyond the first correct version (0.39 of peak): every role is ONE warp per scheduler with nothing to hide
// instruction latency behind, so the producer and the epilogue loops carry cursors instead of dividing (an integer
// division per chunk in the single producer thread alone held the crush at 2.9 TB/s), the mix epilogue runs on eight
// warps, and its shared-memory loads are issued before the math.
#include <vector>

#include "kernels.cuh"

namespace mz {

namespace sg {
constexpr int kMaxThreads = 320;                          // warp 0 TMA, warp 1 issuer, 4 or 8 epilogue warps
constexpr int kTileM = 128;
constexpr uint32_t kAStage = kTileM * 128;               // one A chunk: 128 pixels x 32 fp32
// epilogue slots per warp, 32 pixels x 16 channels each.  mix: [x fp32 -> out in place | z fp32 -> 16-bit shadow in place],
// six of them: the x / z slices are requested five slices ahead (an L2 round trip under load is several slices long).
// crush: [out fp32 | 16-bit shadow], three of them (two stores in flight).
constexpr int kSlotsMix = 6, kSlotsCrush = 3, kSlotsMax = 6;
constexpr uint32_t kSlotX = 32 * 64, kSlotO16 = 32 * 32;
constexpr uint32_t kSlotMix = 2 * kSlotX, kSlotCrush = kSlotX + kSlotO16;
constexpr uint32_t kSmemMax = 227 * 1024;
constexpr int kMaxStages = 6;
}  // namespace sg

struct SgParams {
  CUtensorMap tmA[2];  // GEMM operand boxes (32 ch, 1, 128 px, 1) of the input(s), 128-byte swizzle
  CUtensorMap tmW;     // (32 k, ns rows) of W[N][K]
  CUtensorMap tmE[2];  // mix epilogue: boxes (16 ch, 1, 32 px, 1) of x and z, 64-byte swizzle
  CUtensorMap tmO;     // fp32 output box (16 ch, 1, 32 px, 1)
  CUtensorMap tmO16;   // 16-bit shadow box (32-byte swizzle)
  int taps, f, fj, cpt;  // K segments, crush factor (1: mix), taps per input row (1: the f pixels of a dense row are one
                         // segment of f C channels), 32-channel chunks per tap
  int C, N, ns;        // channels per tap (f C for a merged crush), output channels, output channels per CTA (multiple of 16)
  int wo, H, Ho;       // output pixels per row; crush: input / output rows per image
  int tiles_x, n_tiles;
  int stages, wres;    // A ring depth; 1: the weight slice is resident, 0: its chunks travel with the A chunks
  uint32_t stage_bytes;
  int mix, has16, bf16;
  float gate;
  uint32_t idesc, tmem_cols, acc_stride;
  uint32_t oA, oEpi, oBars;  // shared-memory offsets (weights at 0)
  uint32_t slot_bytes;
  int n_slots, prefetch, n_epi;
};

__host__ __device__ constexpr uint32_t umma_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__global__ void __launch_bounds__(sg::kMaxThreads, 1) seg_gemm_tc_kernel(const __grid_constant__ SgParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chunks = p.taps * p.cpt;
  // barriers: w_full | a_full[stages] | a_empty[stages] | acc_full[2] | acc_empty[2] | slot[8][kSlotsMax] | tmem pointer
  const uint32_t bar_w = base + p.oBars;
  const uint32_t bar_a_full = bar_w + 8, bar_a_empty = bar_a_full + 8 * sg::kMaxStages;
  const uint32_t bar_acc_full = bar_a_empty + 8 * sg::kMaxStages, bar_acc_empty = bar_acc_full + 16;
  const uint32_t bar_slot = bar_acc_empty + 16;
  const uint32_t tmem_slot = bar_slot + 8 * 8 * sg::kSlotsMax;

  if (threadIdx.x == 0) {
    mbar_init(bar_w, 1);
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(bar_a_full + 8 * i, 1);
      mbar_init(bar_a_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_acc_full + 8 * i, 1);
      mbar_init(bar_acc_empty + 8 * i, p.n_epi);
    }
    for (int i = 0; i < 8 * sg::kSlotsMax; ++i) mbar_init(bar_slot + 8 * i, 1);
    fence_mbar_init();
    tma_prefetch_desc(&p.tmA[0]);
    tma_prefetch_desc(&p.tmW);
    tma_prefetch_desc(&p.tmO);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const int n0 = blockIdx.y * p.ns;
  const int my_tiles = p.n_tiles > static_cast<int>(blockIdx.x) ? (p.n_tiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;

  if (warp == 0) {
    if (lane == 0) {
      // ---- producer: the weight slice once, then the A chunks of every tile through the ring ----
      if (p.wres) {
        mbar_expect_tx(bar_w, static_cast<uint32_t>(chunks) * p.ns * 128u);
        for (int t = 0; t < p.taps; ++t)
          for (int q = 0; q < p.cpt; ++q)
            tma_load_2d(base + static_cast<uint32_t>(t * p.cpt + q) * p.ns * 128u, &p.tmW, bar_w, t * p.C + q * 32, n0);
      }
      const uint32_t w_chunk = p.wres ? 0u : static_cast<uint32_t>(p.ns) * 128u;
      // A cursor over this CTA's chunk sequence (tile, tap = (i, j), 32-channel chunk q) that advances without a
      // division: one thread issues every load, so whatever it computes per chunk is on the critical path.
      struct Cursor {
        int k, i, j, q, x0, yin;
      };
      auto tile_geom = [&](Cursor& c) {
        const int tile = blockIdx.x + c.k * gridDim.x;
        const int row = tile / p.tiles_x;
        c.x0 = (tile - row * p.tiles_x) * sg::kTileM;
        c.yin = p.mix ? 0 : (row / p.Ho) * p.H + (row % p.Ho) * p.f;
      };
      auto advance = [&](Cursor& c) {
        if (++c.q < p.cpt) return;
        c.q = 0;
        if (++c.j == p.fj) {  // (mix: one j and the two taps are i = 0, 1: x then z)
          c.j = 0;
          if (++c.i == (p.mix ? 2 : p.f)) {
            c.i = 0;
            if (++c.k < my_tiles) tile_geom(c);
          }
        }
      };
      Cursor ld = {0, 0, 0, 0, 0, 0}, pf;
      if (my_tiles > 0) tile_geom(ld);
      pf = ld;
      // (experiment, off by default: chunks requested into L2 `prefetch` chunks ahead of the ring)
      for (int n = 0; n < p.prefetch && pf.k < my_tiles; ++n, advance(pf))
        tma_prefetch_4d(&p.tmA[p.mix ? pf.i : 0], pf.q * 32, p.mix ? 0 : pf.j, pf.x0, p.mix ? 0 : pf.yin + pf.i);
      uint32_t s = 0, ph = 0;
      for (; ld.k < my_tiles; advance(ld)) {
        if (p.prefetch > 0 && pf.k < my_tiles) {
          tma_prefetch_4d(&p.tmA[p.mix ? pf.i : 0], pf.q * 32, p.mix ? 0 : pf.j, pf.x0, p.mix ? 0 : pf.yin + pf.i);
          advance(pf);
        }
        mbar_wait(bar_a_empty + 8 * s, ph ^ 1u);
        mbar_expect_tx(bar_a_full + 8 * s, sg::kAStage + w_chunk);
        const uint32_t stage = base + p.oA + s * p.stage_bytes;
        tma_load_4d(stage, &p.tmA[p.mix ? ld.i : 0], bar_a_full + 8 * s, ld.q * 32, p.mix ? 0 : ld.j, ld.x0, p.mix ? 0 : ld.yin + ld.i);
        if (!p.wres) tma_load_2d(stage + sg::kAStage, &p.tmW, bar_a_full + 8 * s, (ld.i * p.fj + ld.j) * p.C + ld.q * 32, n0);
        if (++s == static_cast<uint32_t>(p.stages)) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ---- UMMA issuer ----
      if (p.wres) {
        mbar_wait(bar_w, 0);
        tc_fence_after();
      }
      uint32_t s = 0, ph = 0;
      for (int k = 0; k < my_tiles; ++k) {
        const uint32_t as = k & 1, aph = (k >> 1) & 1u;
        mbar_wait(bar_acc_empty + 8 * as, aph ^ 1u);
        tc_fence_after();
        const uint32_t d = tmem_base + as * p.acc_stride;
        for (int kq = 0; kq < chunks; ++kq) {
          mbar_wait(bar_a_full + 8 * s, ph);
          tc_fence_after();
          const uint32_t a_base = base + p.oA + s * p.stage_bytes;
          const uint32_t b_base = p.wres ? base + static_cast<uint32_t>(kq) * p.ns * 128u : a_base + sg::kAStage;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)  // K = 8 tf32 (32 bytes) per instruction, four per 128-byte row
            umma_tf32(d, umma_smem_desc(a_base + kk * 32, 1024, 2), umma_smem_desc(b_base + kk * 32, 1024, 2), p.idesc,
                      (kq | kk) != 0);
          umma_commit(bar_a_empty + 8 * s);
          if (++s == static_cast<uint32_t>(p.stages)) {
            s = 0;
            ph ^= 1u;
          }
        }
        umma_commit(bar_acc_full + 8 * as);
      }
    }
  } else {
    // ---- epilogue: warp w reads TMEM lanes 32 (w % 4) .. +31 = pixels x0 + 32 (w % 4) .. of the tile; with eight
    // epilogue warps the two warps of a lane quarter take the even / the odd 16-channel slices.  One warp per scheduler
    // has nothing to hide its instruction latencies behind, so the loop keeps no division, no modulo and no address
    // arithmetic that the previous iteration has not already done. ----
    const int q = warp & 3, h = (warp - 2) >> 2, nh = p.n_epi >> 2;
    const int wi = h * 4 + q;
    const uint32_t n_slots = p.n_slots;
    const uint32_t my_slots = base + p.oEpi + wi * (n_slots * p.slot_bytes);
    const uint32_t my_bars = bar_slot + 8 * (wi * sg::kSlotsMax);
    const int n_hi = p.N - n0 < p.ns ? p.N - n0 : p.ns;  // output channels of this CTA
    const int slices = (n_hi + 15) / 16;
    const uint32_t lane_tmem = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    uint32_t swz[4];  // byte offset of 16-byte chunk kk of this lane's row in a 64-byte-swizzled slot
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) swz[kk] = lane * 64 + swz_chunk(lane, kk, 64) * 16;
    const uint32_t swz16_0 = lane * 32 + swz_chunk(lane, 0, 32) * 16, swz16_1 = lane * 32 + swz_chunk(lane, 1, 32) * 16;
    auto geom = [&](int k, int& row, int& xw) {
      const int tile = blockIdx.x + k * gridDim.x;
      row = tile / p.tiles_x;
      xw = (tile - row * p.tiles_x) * sg::kTileM + q * 32;
    };
    // request cursor (lane 0, mix): the x / z slices of this warp's iterations, n_slots - 1 iterations ahead.  Slots and
    // their barriers advance with LIVE iterations only (a warp whose 32 pixels lie past the end of the row neither
    // loads nor stores), so a slot is reused n_slots committed store groups after its store.
    int rk = 0, rsl = h, rrow = 0, rxw = 0;
    uint32_t rsi = 0;
    if (my_tiles > 0) geom(0, rrow, rxw);
    auto request = [&]() {  // issue the cursor's loads (if its pixels exist) and advance it
      if (rxw < p.wo) {
        const uint32_t slot = my_slots + rsi * p.slot_bytes, bar = my_bars + 8 * rsi;
        mbar_expect_tx(bar, 2 * sg::kSlotX);
        tma_load_4d(slot, &p.tmE[0], bar, n0 + rsl * 16, 0, rxw, rrow);
        tma_load_4d(slot + sg::kSlotX, &p.tmE[1], bar, n0 + rsl * 16, 0, rxw, rrow);
        if (++rsi == n_slots) rsi = 0;
      }
      rsl += nh;
      if (rsl >= slices) {
        rsl = h;
        if (++rk < my_tiles) geom(rk, rrow, rxw);
      }
    };
    const bool requester = p.mix && lane == 0 && h < slices;
    if (requester)
      for (uint32_t e = 0; e + 1 < n_slots && rk < my_tiles; ++e) request();
    uint32_t si = 0, sph = 0;
    for (int k = 0; k < my_tiles; ++k) {
      const uint32_t as = k & 1;
      int row, xw;
      geom(k, row, xw);
      const bool live = xw < p.wo;  // (warp-uniform)
      mbar_wait(bar_acc_full + 8 * as, (k >> 1) & 1u);
      tc_fence_after();
      const uint32_t acc = lane_tmem + as * p.acc_stride;
      if (h >= slices) {  // fewer slices than warps per lane quarter: nothing to read, but the stage needs every arrival
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_acc_empty + 8 * as);
      }
      for (int sl = h; sl < slices; sl += nh) {
        uint32_t v[16];
        tmem_ld16(acc + sl * 16, v);
        tmem_ld_wait();
        if (sl + nh >= slices) {  // this warp's last slice of the accumulator stage is in registers: hand it back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_acc_empty + 8 * as);
        }
        if (!live) continue;
        const uint32_t slot = my_slots + si * p.slot_bytes;
        float4 o[4];
        if (p.mix) {
          mbar_wait(my_bars + 8 * si, sph);
          float4 xv[4], zv[4];
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {  // (all loads first: the accessors are volatile, i.e. ordered)
            xv[kk] = lds128f(slot + swz[kk]);
            zv[kk] = lds128f(slot + sg::kSlotX + swz[kk]);
          }
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            const float w0 = p.gate * __fdividef(1.f, 1.f + __expf(-__uint_as_float(v[4 * kk + 0])));
            const float w1 = p.gate * __fdividef(1.f, 1.f + __expf(-__uint_as_float(v[4 * kk + 1])));
            const float w2 = p.gate * __fdividef(1.f, 1.f + __expf(-__uint_as_float(v[4 * kk + 2])));
            const float w3 = p.gate * __fdividef(1.f, 1.f + __expf(-__uint_as_float(v[4 * kk + 3])));
            o[kk].x = (1.f - w0) * xv[kk].x + w0 * zv[kk].x;  // (the reference's expression: model.py:837)
            o[kk].y = (1.f - w1) * xv[kk].y + w1 * zv[kk].y;
            o[kk].z = (1.f - w2) * xv[kk].z + w2 * zv[kk].z;
            o[kk].w = (1.f - w3) * xv[kk].w + w3 * zv[kk].w;
          }
        } else {
          if (lane == 0) bulk_wait_read<sg::kSlotsCrush - 1>();  // the slot's previous store has been read out
          __syncwarp();
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            o[kk] = make_float4(__uint_as_float(v[4 * kk]), __uint_as_float(v[4 * kk + 1]), __uint_as_float(v[4 * kk + 2]),
                                __uint_as_float(v[4 * kk + 3]));
        }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          sts128(slot + swz[kk], __float_as_uint(o[kk].x), __float_as_uint(o[kk].y), __float_as_uint(o[kk].z), __float_as_uint(o[kk].w));
        if (p.has16) {
          if (p.mix) __syncwarp();  // the shadow goes where z was: every lane has read its z row
          sts128(slot + sg::kSlotX + swz16_0, pack_shadow2(p.bf16, o[0].x, o[0].y), pack_shadow2(p.bf16, o[0].z, o[0].w),
                 pack_shadow2(p.bf16, o[1].x, o[1].y), pack_shadow2(p.bf16, o[1].z, o[1].w));
          sts128(slot + sg::kSlotX + swz16_1, pack_shadow2(p.bf16, o[2].x, o[2].y), pack_shadow2(p.bf16, o[2].z, o[2].w),
                 pack_shadow2(p.bf16, o[3].x, o[3].y), pack_shadow2(p.bf16, o[3].z, o[3].w));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_4d(&p.tmO, slot, n0 + sl * 16, 0, xw, row);
          if (p.has16) tma_store_4d(&p.tmO16, slot + sg::kSlotX, n0 + sl * 16, 0, xw, row);
          bulk_commit();
          if (requester && rk < my_tiles) {
            // the cursor's slot was last used n_slots live iterations before it, i.e. at least one store group back
            bulk_wait_read<1>();
            request();
          }
        }
        if (++si == n_slots) {
          si = 0;
          sph ^= 1u;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
bool seg_gemm_tc_applies(const float* a0, const float* a1, const float* wt, const float* out, const void* out16, int C, int N,
                         int K, int pitch_in, int pitch_out) {
  auto al16 = [](const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 15u) == 0; };
  return al16(a0) && al16(a1) && al16(wt) && al16(out) && al16(out16) && pitch_in % 4 == 0 && pitch_out % 4 == 0 && K % 4 == 0 &&
         (out16 == nullptr || pitch_out % 8 == 0) && C >= 1 && N >= 1;
}

int launch_seg_gemm_tc(const SgArgs& a, cudaStream_t s) {
  SgParams p;
  memset(&p, 0, sizeof(p));
  int device = 0;
  MZ_CUDA(cudaGetDevice(&device));
  int sms = sm_count(device);
  if (sms <= 0) sms = 148;
  p.mix = a.mix;
  // crush on a dense map (pitch = C): the f pixels under one output pixel are f C consecutive floats of an input row --
  // one K segment per input row instead of f (fewer, fuller 32-channel chunks; the weight's K order (i, j, c) is the same)
  const bool merged = !a.mix && a.pitch_in == a.C;
  p.f = a.mix ? 1 : a.f;
  p.fj = a.mix || merged ? 1 : a.f;
  p.taps = a.mix ? 2 : a.f * p.fj;
  p.C = merged ? a.f * a.C : a.C;
  p.cpt = ceil_div(p.C, 32);
  p.N = a.N;
  p.gate = a.gate;
  p.has16 = a.out16 != nullptr;
  p.bf16 = a.bf16;
  p.H = a.H;
  p.Ho = a.Ho > 0 ? a.Ho : 1;
  MZ_REQUIRE(a.wo < (1LL << 31) && a.rows < (1LL << 31), "segment GEMM: too many pixels");
  p.wo = static_cast<int>(a.wo);
  const int chunks = p.taps * p.cpt;
  // Epilogue warps: the mix epilogue is a long dependent chain per slice, so two warps per scheduler (eight), three slots
  // each; the crush epilogue only copies, four warps leave the shared memory to the weights.
  p.n_epi = a.mix ? 8 : 4;
  {
    const char* e = getenv("MZ_SG_EPI");  // 4 | 8 epilogue warps (experiments)
    if (e && (atoi(e) == 4 || atoi(e) == 8)) p.n_epi = atoi(e);
  }
  p.n_slots = a.mix ? sg::kSlotsMix * 4 / p.n_epi : sg::kSlotsCrush;
  {
    const char* e = getenv("MZ_SG_SLOTS");  // mix: slots per epilogue warp (experiments)
    if (e && a.mix && atoi(e) >= 2 && atoi(e) <= sg::kSlotsMax) p.n_slots = atoi(e);
  }
  p.slot_bytes = a.mix ? sg::kSlotMix : sg::kSlotCrush;
  const uint32_t epi_bytes = static_cast<uint32_t>(p.n_epi) * p.n_slots * p.slot_bytes;
  const uint32_t w_budget = sg::kSmemMax - 2048 - epi_bytes - 3 * sg::kAStage;  // at least three ring stages stay
  // Output channels per CTA.  Resident form: the [ns][K] weight slice stays in shared memory and the A tiles are read once
  // per slice; streamed form (deep K): ns = up to 256 and every 32-channel weight chunk travels with its A chunk (an L2
  // hit after the first tile).  Whichever moves fewer bytes per 128-pixel tile through L2.
  const int n16 = ceil_div(a.N, 16) * 16;
  const double a_tile = 128.0 * chunks * 128.0, w_all = static_cast<double>(n16) * chunks * 128.0;
  int ns_res = 0, slices_res = 0;
  for (int n = 1; n <= n16 / 16; ++n) {
    const int ns = ceil_div(ceil_div(n16, n), 16) * 16;
    if (ns <= 256 && static_cast<uint32_t>(chunks) * ns * 128u <= w_budget) {
      ns_res = ns;
      slices_res = ceil_div(n16, ns);
      break;
    }
  }
  const int slices_str = ceil_div(n16, 256), ns_str = ceil_div(ceil_div(n16, slices_str), 16) * 16;
  p.wres = ns_res > 0 && slices_res * a_tile <= slices_str * a_tile + w_all;
  {
    const char* force = getenv("MZ_SG_WEIGHTS");  // "stream" | "resident": tests / experiments
    if (force && force[0] == 's') p.wres = 0;
    if (force && force[0] == 'r' && ns_res > 0) p.wres = 1;
  }
  p.ns = p.wres ? ns_res : ns_str;
  const int n_slices = ceil_div(n16, p.ns);
  const uint32_t w_bytes = p.wres ? static_cast<uint32_t>(chunks) * p.ns * 128u : 0u;  // (a multiple of 2048)
  p.stage_bytes = sg::kAStage + (p.wres ? 0u : static_cast<uint32_t>(p.ns) * 128u);
  p.oA = w_bytes;
  int stages = static_cast<int>((sg::kSmemMax - 1024 - w_bytes - epi_bytes - 1024) / p.stage_bytes);
  if (stages > sg::kMaxStages) stages = sg::kMaxStages;
  MZ_REQUIRE(stages >= 2, "segment GEMM: no room for the activation ring");
  p.stages = stages;
  p.oEpi = p.oA + stages * p.stage_bytes;
  p.oBars = p.oEpi + epi_bytes;
  p.prefetch = 0;  // (measured: 12 chunks ahead costs 3-15 %, 32 ahead 20-40 % -- the ring's own loads keep HBM busy)
  {
    const char* e = getenv("MZ_SG_PREFETCH");
    if (e) p.prefetch = atoi(e);
  }
  const uint32_t smem = 1024 + p.oBars + 1024;
  p.acc_stride = static_cast<uint32_t>(p.ns);
  uint32_t cols = 32;
  while (cols < 2 * p.acc_stride) cols *= 2;
  p.tmem_cols = cols;
  p.idesc = umma_idesc_tf32(sg::kTileM, p.ns);
  p.tiles_x = ceil_div(p.wo, sg::kTileM);
  const long long n_tiles = a.rows * p.tiles_x;
  MZ_REQUIRE(n_tiles < (1LL << 31), "segment GEMM: too many tiles");
  p.n_tiles = static_cast<int>(n_tiles);
  int gx = sms / n_slices;
  if (gx < 1) gx = 1;
  if (gx > p.n_tiles) gx = p.n_tiles;

  int rc;
  const uint64_t pin = static_cast<uint64_t>(a.pitch_in) * 4, pout = static_cast<uint64_t>(a.pitch_out) * 4;
  if (a.mix) {
    const uint64_t dims[4] = {static_cast<uint64_t>(a.C), 1, static_cast<uint64_t>(a.wo), 1};
    const uint64_t st[3] = {pin, pin, pin * static_cast<uint64_t>(a.wo)};
    const uint32_t boxA[4] = {32u, 1u, 128u, 1u}, boxE[4] = {16u, 1u, 32u, 1u};
    const float* src[2] = {a.a0, a.a1};
    for (int i = 0; i < 2; ++i) {
      if ((rc = encode_tmap(&p.tmA[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(src[i]), dims, st, boxA,
                            CU_TENSOR_MAP_SWIZZLE_128B)) != MZ_OK) return rc;
      if ((rc = encode_tmap(&p.tmE[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(src[i]), dims, st, boxE,
                            CU_TENSOR_MAP_SWIZZLE_64B)) != MZ_OK) return rc;
    }
  } else {
    const uint64_t f = a.f;
    const uint64_t dims[4] = {static_cast<uint64_t>(p.C), static_cast<uint64_t>(p.fj), static_cast<uint64_t>(a.wo),
                              static_cast<uint64_t>(a.in_rows)};
    const uint64_t st[3] = {pin, f * pin, static_cast<uint64_t>(a.W) * pin};
    const uint32_t boxA[4] = {32u, 1u, 128u, 1u};
    if ((rc = encode_tmap(&p.tmA[0], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(a.a0), dims, st, boxA,
                          CU_TENSOR_MAP_SWIZZLE_128B)) != MZ_OK) return rc;
    p.tmA[1] = p.tmA[0];
    p.tmE[0] = p.tmE[1] = p.tmA[0];  // (unused)
  }
  {
    const uint64_t K = static_cast<uint64_t>(p.taps) * p.C;
    const uint64_t dims[2] = {K, static_cast<uint64_t>(a.N)};
    const uint64_t st[1] = {K * 4};
    const uint32_t box[2] = {32u, static_cast<uint32_t>(p.ns)};
    if ((rc = encode_tmap(&p.tmW, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(a.wt), dims, st, box,
                          CU_TENSOR_MAP_SWIZZLE_128B)) != MZ_OK) return rc;
  }
  {
    const uint64_t dims[4] = {static_cast<uint64_t>(a.N), 1, static_cast<uint64_t>(a.wo), static_cast<uint64_t>(a.rows)};
    const uint64_t st[3] = {pout, pout, pout * static_cast<uint64_t>(a.wo)};
    const uint32_t box[4] = {16u, 1u, 32u, 1u};
    if ((rc = encode_tmap(&p.tmO, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a.out, dims, st, box, CU_TENSOR_MAP_SWIZZLE_64B)) != MZ_OK)
      return rc;
    if (a.out16) {
      const uint64_t st16[3] = {pout / 2, pout / 2, pout / 2 * static_cast<uint64_t>(a.wo)};
      if ((rc = encode_tmap(&p.tmO16, a.bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, a.out16, dims,
                            st16, box, CU_TENSOR_MAP_SWIZZLE_32B)) != MZ_OK) return rc;
    } else {
      p.tmO16 = p.tmO;
    }
  }
  MZ_CUDA(cudaFuncSetAttribute(seg_gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  {
    static const bool verbose = getenv("MZ_VERBOSE") != nullptr;
    if (verbose)
      fprintf(stderr, "[mz seg gemm] %s C %d N %d taps %d | ns %d x %d slices (%s weights), %d chunks, stages %d, epilogue warps %d x %d slots, smem %u, tmem %u | tiles %d grid %d x %d\n",
              a.mix ? "mix" : "crush", a.C, a.N, p.taps, p.ns, n_slices, p.wres ? "resident" : "streamed", chunks, stages, p.n_epi, p.n_slots, smem,
              p.tmem_cols, p.n_tiles, gx, n_slices);
  }
  seg_gemm_tc_kernel<<<dim3(gx, n_slices), 64 + 32 * p.n_epi, smem, s>>>(p);
  MZ_CUDA(cudaGetLastError());
  return MZ_OK;
}

}  // namespace mz
