// conv_tc.cu -- 3x3 / pad 1 / stride 1 convolution as an implicit GEMM on the 5th-gen tensor cores.
//
//   D[128 pixels, N] += A[128 pixels, K = (tap, cin)] * W[N, K]^T        (fp16 | bf16 operands -> fp32 in TMEM)
//
// Replaces InvertedBottleneck.conv1/conv2 (reference model.py:742-748,773-778) and
// SubpixelConv2d.conv (model.py:902-909) with their elementwise successors fused in the epilogue.
//
// Work unit ("patch"): `rows` consecutive image rows x 128 pixels of one image; one fp32
// accumulator (128 TMEM lanes x N columns) per row.  Persistent CTAs walk the patches.
//
// Warp roles (256 threads):
//   warp 0 (one lane)  TMA producer: per K chunk ONE activation halo tile
//                      [(rows+2) image rows][130 pixels][kc channels] (TMA zero-fills the conv padding),
//                      then nine weight tiles [N][kc] -- one per filter tap.
//   warp 1 (one lane)  MMA issuer: for each tap the A operand is the SAME halo tile addressed through a
//                      shared-memory descriptor shifted by (dy*130 + dx) pixel rows, so activations are
//                      read from L2 once per chunk instead of nine times.
//   warp 2             TMEM allocator.
//   warps 4..7         epilogue: tcgen05.ld -> FiLM scale/shift + SiLU -> bf16 | residual add | pixel-shuffle.
//                      With two TMEM stages the epilogue of patch i overlaps the MMAs of patch i+1.
#include <stdlib.h>

#include "kernels.cuh"

namespace mz {

constexpr int kTileW = 128;
constexpr int kThreads = 384;  // 4 control warps (TMA, MMA, TMEM alloc, spare) + up to 8 epilogue warps
constexpr int kMaxSmem = 232448;  // 227 KB opt-in limit per CTA on sm_100

struct TcParams {
  CUtensorMap tmA;  // activations: (cin_p, W, H, B) bf16
  CUtensorMap tmB;  // weights:     (cin_p, n_pad, 9) bf16
  CUtensorMap tmO;  // 16-bit output (hidden | zb): (n_pad, W, H, B), box (e16, 32 px, 1, 1), swizzled
  CUtensorMap tmZ;  // fp32 residual stream (mode 1): (n_pad, W, H, B), box (e32, 32 px, 1, 1), swizzled
  int e16, e32;     // channels per output box: box rows are 128 / 64 / 32 bytes
  int stage_bytes;  // epilogue staging (all four warps)
  int o_ring;       // mode 0: warp-private ring of output boxes (2 or 4)
  int res_rows;     // mode 1: row buffers (fp32 residual tile + 16-bit tile) per epilogue warp: 1, or all its rows
  int sliced;       // mode 1, res_rows == 1: the row is finished box by box (e16 == e32), each box with its own residual barrier,
                    // and the NEXT row's boxes are requested as soon as this row's stores of them have been read
  int epi_warps;    // 4 or 8 epilogue warps; with 8, two warps share a TMEM lane quarter and split the rows / boxes
  int kt_last;      // k-steps issued for the LAST K chunk of a patch (resident banks): fewer than kc / 16 when the tail of
                    // the input channels is zero padding (108 -> 128: the eighth k-step would multiply zeros)
  EpiParams epi;
  int kc, n_chunks;  // channels per swizzled sub-tile; pipeline chunks per patch (each = subs sub-tiles)
  int subs;          // 16-channel sub-tiles fused into one stage (3 for Cin = 48), else 1
  int a_kp, b_kp;    // k-step pitch inside a stage in 16-byte units (A / B): 2 within a swizzled row, else the sub-tile pitch
  int b_tap;         // tap pitch inside a weight stage in 16-byte units
  int rows, acc_stages, acc_stride;
  int halo_mode;
  int a_stages, b_stages;
  int a_stage_bytes, b_stage_bytes;
  int a_tx_bytes, b_tx_bytes;
  int pw;  // pixel rows per image row inside an A stage
  int tiles_x, tiles_y, n_units, n_rounds;
  int cluster;       // CTAs per cluster sharing the weight stream by TMA multicast (1, 2 or 4)
  int pair;          // 1: CTA pairs issue M = 256 UMMAs (cta_group::2), weights split N/2 + N/2 between them
  int b_slice_rows;  // n_pad / cluster: weight rows each CTA loads and multicasts per stage
  int fuse_g;        // FUSE kernels: vertical taps per UMMA window (2 | 3); 0 otherwise
  uint32_t idesc_w[3];  // FUSE: instruction descriptors for windows of 1, 2, 3 stacked taps (N, 2N, 3N columns)
  int res_b;         // 1: the whole filter bank stays resident in shared memory (b_stages == 3 * n_chunks): it is
                     // loaded during the first patch and never again -- the persistent CTA then streams activations only
  long long* prof;   // optional per-CTA role timers (clock64 ticks), [grid][3 roles][8]; nullptr = off
  int dbg;           // timing experiments only (results are wrong): 1 skip weight loads, 2 skip activation loads,
                     // 4 skip the epilogue body, 8 skip the MMAs
  uint32_t idesc;
  uint32_t tmem_cols;
};

struct SmemPlan {
  uint32_t a, b, bars, tmem_ptr, film, stage, total;
};

__host__ __device__ inline SmemPlan plan_smem(const TcParams& p) {
  SmemPlan s;
  s.a = 0;
  s.b = s.a + p.a_stages * p.a_stage_bytes;
  s.bars = s.b + p.b_stages * p.b_stage_bytes;
  const uint32_t nbars = 2 * p.a_stages + 2 * p.b_stages + 4 + 64;  // + up to eight residual-load barriers per epilogue warp
  s.tmem_ptr = s.bars + nbars * 8;
  s.film = s.tmem_ptr + 16;  // [2][n_pad <= 256] fp32: FiLM scale / shift rows of the current image
  s.stage = (s.film + 2 * 256 * 4 + 1023u) & ~1023u;  // epilogue staging: swizzled boxes for TMA store / load
  s.total = s.stage + p.stage_bytes;
  return s;
}

// role timers: accumulate clock64 ticks spent in a statement when profiling is on (warp-uniform flag)
#define MZ_TIMED(slot, stmt)                         \
  do {                                               \
    if (prof_on) {                                   \
      const long long _t = clock64();                \
      stmt;                                          \
      tick[slot] += clock64() - _t;                  \
    } else {                                         \
      stmt;                                          \
    }                                                \
  } while (0)

// PAIR: the CTA pair of a cluster works as one 256-row UMMA (cta_group::2): the leader CTA issues M = 256 UMMAs whose
// A operand is each CTA's own 128-pixel tile and whose B operand is split -- each CTA holds N/2 weight rows -- so
// per CTA the weight stream (TMA writes AND tensor-core operand reads from shared memory) is halved.
// VAR 0: plain.  VAR 1 (PAIR): see above.  VAR 2 (FUSE, resident filter bank only): filter rows are fused along N --
// one UMMA multiplies an INPUT row's tile with the weights of up to three vertical taps stacked as [dy][N] rows and
// accumulates into the adjacent accumulators of the output rows those taps feed (output row r lives at TMEM block
// ROWS-1-r, so blocks of dy, dy+1, dy+2 are contiguous).  A patch of R rows then takes R+2 UMMAs per (dx, k-step)
// instead of 3R: the 128 x 16 activation tile -- 4 KB of shared-memory operand fetch per UMMA, what bounds the small-N
// shapes -- is fetched once per input row instead of once per (output row, tap).  Every UMMA accumulates; the epilogue
// zeroes each accumulator column group right after reading it.
// LAY (head only): bit 0 interleaved input image, bit 1 interleaved output image (ImageIo::x_nhwc / y_nhwc), bit 2
// 16-bit images (ImageIo::type kImgU16).
template <int MODE, int KT, int ROWS, int VAR, int LAY = 0>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_kernel(const __grid_constant__ TcParams p) {
  constexpr bool PAIR = VAR == 1, FUSE = VAR == 2;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* gen_base = smem_raw + (base - raw);
  const SmemPlan sp = plan_smem(p);

  const uint32_t a_base = base + sp.a;
  const uint32_t b_base = base + sp.b;
  const uint32_t bar_a_full = base + sp.bars;
  const uint32_t bar_a_empty = bar_a_full + 8 * p.a_stages;
  const uint32_t bar_b_full = bar_a_empty + 8 * p.a_stages;
  const uint32_t bar_b_empty = bar_b_full + 8 * p.b_stages;
  const uint32_t bar_acc_full = bar_b_empty + 8 * p.b_stages;
  const uint32_t bar_acc_empty = bar_acc_full + 16;
  const uint32_t bar_res = bar_acc_empty + 16;
  volatile uint32_t* tmem_ptr_gen = reinterpret_cast<volatile uint32_t*>(gen_base + sp.tmem_ptr);

  // (broadcast from lane 0 so that the compiler knows the warp index -- and everything derived from it: role, TMEM lane
  // quarter, staging addresses, TMA coordinates -- is warp-uniform and keeps it in uniform registers)
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA);
    tma_prefetch_desc(&p.tmB);
    if (MODE != 2) tma_prefetch_desc(&p.tmO);
    if (MODE == 1) tma_prefetch_desc(&p.tmZ);
    for (int i = 0; i < p.a_stages; ++i) {
      mbar_init(bar_a_full + 8 * i, 1);
      mbar_init(bar_a_empty + 8 * i, 1);
    }
    for (int i = 0; i < p.b_stages; ++i) {
      mbar_init(bar_b_full + 8 * i, 1);
      mbar_init(bar_b_empty + 8 * i, p.cluster);  // one tcgen05.commit arrive per CTA sharing the stage
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_acc_full + 8 * i, 1);
      mbar_init(bar_acc_empty + 8 * i, (PAIR ? 2 : 1) * p.epi_warps);  // one arrive per epilogue warp (of both CTAs of a pair)
    }
    for (int i = 0; i < 64; ++i) mbar_init(bar_res + 8 * i, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    if (PAIR) {
      tmem_alloc2(base + sp.tmem_ptr, p.tmem_cols);
      tmem_relinquish2();
    } else {
      tmem_alloc(base + sp.tmem_ptr, p.tmem_cols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR || p.cluster > 1) cluster_sync_all();  // peers' barriers must be initialised before anything is signalled to them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_gen;
  // Programmatic dependent launch: the next convolution of the stream may place its CTAs on SMs as this grid's CTAs
  // retire and run its prologue (barriers, TMEM, the resident filter bank) there; it touches activations only after
  // its own griddepcontrol.wait, i.e. once this grid has completed.
  griddep_launch_dependents();
  if (FUSE) {  // every UMMA accumulates: the accumulators start from zero (afterwards the epilogue re-zeroes them)
    if (warp >= 4 && warp < 8) {
      for (uint32_t col = 0; col < p.tmem_cols; col += 16)
        tmem_zero16(tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16) + col);
      tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  const uint32_t cta_rank = (PAIR || p.cluster > 1) ? cluster_ctarank() : 0u;
  const uint16_t cta_mask = static_cast<uint16_t>((1u << p.cluster) - 1u);

  const int row_bytes = p.kc * 2;
  const int units_per_img = p.tiles_x * p.tiles_y;
  const bool prof_on = p.prof != nullptr;
  long long tick[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long t_role0 = prof_on ? clock64() : 0;

  if (warp == 0) {
    // =============================== TMA producer ===============================
    // The whole warp walks the (uniform) loop so that addresses stay in uniform registers; lane 0 issues.
    // Ring positions advance incrementally (no integer division in the hot loops).
    uint32_t sa = 0, pa = 0, sb = 0, pb = 0;
    bool a_wrapped = false, b_wrapped = false;
    const uint32_t per_dx = (ROWS + 2) * kTileW * row_bytes;
    const uint32_t tap_bytes = p.epi.n_pad * row_bytes;  // one tap's [N][kc] tile inside a weight stage
    const uint32_t a_sub_bytes = static_cast<uint32_t>(p.a_kp) << 4;  // one 16-channel sub-tile of a fused stage
    // fill weight stage `sbi` with the taps of (chunk c, filter row dy) [FUSE: filter column dy]
    auto issue_b = [&](int c, int dy, uint32_t sbi) {
      const uint32_t full_b = bar_b_full + 8 * sbi;
      const uint32_t dstB = b_base + sbi * p.b_stage_bytes;
      if (FUSE) {
        if (lane == 0) {  // stage (c, dx): the three vertical taps of filter column dx, [sub][dy][N][kc]
          const int dx = dy;
          mbar_expect_tx(full_b, p.b_tx_bytes);
          for (int sub = 0; sub < p.subs; ++sub)
            for (int v = 0; v < 3; ++v)
              tma_load_3d(dstB + (sub * 3 + v) * tap_bytes, &p.tmB, full_b, (c * p.subs + sub) * p.kc, 0, v * 3 + dx);
        }
      } else if (PAIR) {
        if (lane == 0) {  // this CTA's half of the weight rows; stage layout [3 taps][N/2][kc]
          if (cta_rank == 0) mbar_expect_tx(full_b, 2 * p.b_tx_bytes);
          tma2_load_3d(dstB, &p.tmB, mapa_u32(full_b, 0), c * p.kc, cta_rank * p.b_slice_rows, dy * 3);
        }
      } else if (lane == 0 && (p.dbg & 1) && b_wrapped) {
        mbar_arrive(full_b);
      } else if (lane == 0) {
        mbar_expect_tx(full_b, p.b_tx_bytes);
        if (p.cluster > 1) {
          for (int dx = 0; dx < 3; ++dx)
            tma_load_3d_mcast(dstB + dx * tap_bytes + cta_rank * p.b_slice_rows * row_bytes, &p.tmB, full_b,
                              c * p.kc, cta_rank * p.b_slice_rows, dy * 3 + dx, cta_mask);
        } else {
          for (int sub = 0; sub < p.subs; ++sub)  // stage layout [sub][3 taps][N][kc]
            tma_load_3d(dstB + sub * 3 * tap_bytes, &p.tmB, full_b, (c * p.subs + sub) * p.kc, 0, dy * 3);
        }
      }
    };
    if (p.res_b) {
      // The resident filter bank does not depend on the previous kernel: request all of it BEFORE waiting for that
      // kernel to finish (programmatic dependent launch), so it is in shared memory when the first activations arrive.
      for (int c = 0; c < p.n_chunks; ++c)
        for (int dy = 0; dy < 3; ++dy) issue_b(c, dy, static_cast<uint32_t>(c * 3 + dy));
    }
    griddep_wait();  // activations (and everything else the previous kernels wrote) are valid from here on
    for (int round = 0; round < p.n_rounds; ++round) {
      // every CTA of a cluster walks the same number of rounds (the weight stream is shared); a CTA whose unit
      // index runs past the end recomputes the last unit and its epilogue stores nothing
      const int unit = min(round * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x), p.n_units - 1);
      const int b = unit / units_per_img;
      const int rem = unit - b * units_per_img;
      const int ty = rem / p.tiles_x, tx = rem - ty * p.tiles_x;
      const int x0 = tx * kTileW, y0 = ty * ROWS;
      for (int c = 0; c < p.n_chunks; ++c) {
        MZ_TIMED(0, mbar_wait(bar_a_empty + 8 * sa, pa ^ 1u));
        const uint32_t dstA = a_base + sa * p.a_stage_bytes;
        const uint32_t full_a = bar_a_full + 8 * sa;
        if (PAIR) {
          // both CTAs' bytes complete on the LEADER's barrier, which the leader arms for the pair
          if (lane == 0) {
            if (cta_rank == 0) mbar_expect_tx(full_a, 2 * p.a_tx_bytes);
            tma2_load_4d(dstA, &p.tmA, mapa_u32(full_a, 0), c * p.kc, x0 - 1, y0 - 1, b);
          }
        } else if (lane == 0 && (p.dbg & 2) && a_wrapped) {
          mbar_arrive(full_a);
        } else if (lane == 0) {
          mbar_expect_tx(full_a, p.a_tx_bytes);
          if (p.halo_mode == 1) {
            for (int dx = 0; dx < 3; ++dx)
              tma_load_4d(dstA + dx * per_dx, &p.tmA, full_a, c * p.kc, x0 + dx - 1, y0 - 1, b);
          } else {
            for (int sub = 0; sub < p.subs; ++sub)
              tma_load_4d(dstA + sub * a_sub_bytes, &p.tmA, full_a, (c * p.subs + sub) * p.kc, x0 - 1, y0 - 1, b);
          }
        }
        if (++sa == static_cast<uint32_t>(p.a_stages)) {
          sa = 0;
          pa ^= 1u;
          a_wrapped = true;
        }
        // (streamed weights are issued by warp 3: see below)
      }
    }
  } else if (warp == 3 && !p.res_b) {
    // =============================== weight producer (streamed filter banks) ===============================
    // Its own warp, so that the activation loads above never queue behind a full weight ring: with one producer loop
    // the next chunk's activation tile could only be requested after all three weight stages of the current chunk had
    // found a free slot, which limited the activation prefetch to about one chunk and left the tensor pipe waiting for
    // loads (96-channel conv2: 28 % of the kernel in wait_a_full).  Weights do not depend on the previous kernel: no
    // griddepcontrol.wait here.
    uint32_t sb = 0, pb = 0;
    bool b_wrapped = false;
    const uint32_t tap_bytes = p.epi.n_pad * row_bytes;
    auto issue_b = [&](int c, int dy, uint32_t sbi) {
      const uint32_t full_b = bar_b_full + 8 * sbi;
      const uint32_t dstB = b_base + sbi * p.b_stage_bytes;
      if (PAIR) {
        if (lane == 0) {  // this CTA's half of the weight rows; stage layout [3 taps][N/2][kc]
          if (cta_rank == 0) mbar_expect_tx(full_b, 2 * p.b_tx_bytes);
          tma2_load_3d(dstB, &p.tmB, mapa_u32(full_b, 0), c * p.kc, cta_rank * p.b_slice_rows, dy * 3);
        }
      } else if (lane == 0 && (p.dbg & 1) && b_wrapped) {
        mbar_arrive(full_b);
      } else if (lane == 0) {
        mbar_expect_tx(full_b, p.b_tx_bytes);
        if (p.cluster > 1) {
          for (int dx = 0; dx < 3; ++dx)
            tma_load_3d_mcast(dstB + dx * tap_bytes + cta_rank * p.b_slice_rows * row_bytes, &p.tmB, full_b,
                              c * p.kc, cta_rank * p.b_slice_rows, dy * 3 + dx, cta_mask);
        } else {
          for (int sub = 0; sub < p.subs; ++sub)  // stage layout [sub][3 taps][N][kc]
            tma_load_3d(dstB + sub * 3 * tap_bytes, &p.tmB, full_b, (c * p.subs + sub) * p.kc, 0, dy * 3);
        }
      }
    };
    for (int round = 0; round < p.n_rounds; ++round) {
      for (int c = 0; c < p.n_chunks; ++c) {
        // one weight stage = the three horizontal taps of filter row dy: [3][N][kc]
        for (int dy = 0; dy < 3; ++dy) {
          MZ_TIMED(1, mbar_wait(bar_b_empty + 8 * sb, pb ^ 1u));
          issue_b(c, dy, sb);
          if (++sb == static_cast<uint32_t>(p.b_stages)) {
            sb = 0;
            pb ^= 1u;
            b_wrapped = true;
          }
        }
      }
    }
  } else if (warp == 1 && (!PAIR || cta_rank == 0)) {
    // =============================== MMA issuer ===============================
    // Uniform loop over the whole warp; one elected lane issues tcgen05.mma / tcgen05.commit.  Per weight stage
    // (filter row dy) all 3 * KSTEPS * ROWS UMMAs are issued back to back from ONE predicated region: the
    // descriptor high word is constant, the low words are uniform 32-bit adds computed outside the region, so the
    // SASS is a run of UTCHMMA with ~2 uniform instructions each (an earlier version spent ~100 issue cycles per
    // UMMA on descriptor construction, integer division and R2UR/ELECT waterfalls -- more than the 48..96 cycles a
    // 128 x N x 16 UMMA takes).
    const uint32_t lt = umma_layout_type(p.kc);
    const uint32_t sbo = 8u * row_bytes;
    const uint32_t desc_hi = static_cast<uint32_t>(umma_smem_desc(0, sbo, lt, 0) >> 32);
    const uint32_t desc_lo0 = static_cast<uint32_t>(umma_smem_desc(0, sbo, lt, 0));
    // tap (dy, dx) and accumulator row r start at dy * DY + dx * DX + r * RP sixteen-byte units into the A stage
    uint32_t DY, DX, RP;
    if (p.halo_mode == 1) {
      DX = ((ROWS + 2) * kTileW * row_bytes) >> 4;
      DY = (kTileW * row_bytes) >> 4;
      RP = DY;
    } else {
      DX = row_bytes >> 4;
      DY = (p.pw * row_bytes) >> 4;
      RP = DY;
    }
    if (p.dbg & 32) DY = DX = RP = 0;  // timing experiment: every UMMA reads the same A rows
    const uint32_t TB = (p.dbg & 32) ? 0u : p.b_tap;  // tap pitch inside a weight stage
    const bool leader = elect_one();  // the same lane issues every tcgen05.mma and tcgen05.commit
    const bool issue = leader && !(p.dbg & 8);
    const uint32_t idesc = p.idesc;
    const uint32_t acc_stride = p.acc_stride;
    const uint32_t a_kp = (p.dbg & 64) ? 0u : p.a_kp, b_kp = (p.dbg & 64) ? 0u : p.b_kp;  // 64: same k-step
    // One tap (dx) of the current weight stage: KT k-steps x ROWS accumulators, all descriptor words uniform.
#define MZ_ISSUE_TAP(DXV)                                                                                         \
  if (issue) {                                                                                                    \
    _Pragma("unroll") for (int t = 0; t < KT; ++t) {                                                              \
      if (t >= static_cast<int>(cur_kt)) break; /* (uniform) k-steps over zero padding are not issued */           \
      const uint64_t bdesc = (static_cast<uint64_t>(desc_hi) << 32) | (b_lo_stage + (DXV) * TB + t * b_kp);        \
      _Pragma("unroll") for (int r = 0; r < ROWS; ++r) {                                                          \
        const uint64_t adesc = (static_cast<uint64_t>(desc_hi) << 32) | (a_lo_dy + (DXV) * DX + r * RP + t * a_kp); \
        if (PAIR) {                                                                                               \
          if ((DXV) == 0 && t == 0)                                                                               \
            umma2_bf16(d_base + r * acc_stride, adesc, bdesc, idesc, first);                                      \
          else                                                                                                    \
            umma2_acc(d_base + r * acc_stride, adesc, bdesc, idesc);                                              \
        } else if ((DXV) == 0 && t == 0) {                                                                        \
          umma_bf16(d_base + r * acc_stride, adesc, bdesc, idesc, first);                                         \
        } else {                                                                                                  \
          umma_acc(d_base + r * acc_stride, adesc, bdesc, idesc);                                                 \
        }                                                                                                         \
      }                                                                                                           \
    }                                                                                                             \
  }
    uint32_t sa = 0, pa = 0, sb = 0, pb = 0, as = 0, pacc = 0;
    uint32_t cur_kt = KT;  // k-steps of the current step's chunk (only the resident path ever lowers it)
    // Barrier state of the NEXT step is sampled (non-blocking mbarrier.test_wait) in the middle of the current
    // step, so in the common case -- the producer is ahead -- the blocking wait and its latency are skipped and
    // the tensor pipe never drains between stages.  The commit of the current stage is NOT delayed by this.
    auto test_uniform = [&](uint32_t bar, uint32_t parity) -> bool { return __all_sync(0xffffffffu, mbar_test(bar, parity)); };
    const bool la_acc = p.acc_stages > 1;
    MZ_TIMED(0, mbar_wait(bar_acc_empty + 8 * as, pacc ^ 1u));
    MZ_TIMED(1, mbar_wait(bar_a_full + 8 * sa, pa));
    MZ_TIMED(2, mbar_wait(bar_b_full + 8 * sb, pb));
    tc_fence_after();
    if (FUSE) {
      // ---- resident filter bank, filter rows fused along N (see the kernel comment) ----
      const uint32_t a_stage_u = static_cast<uint32_t>(p.a_stage_bytes) >> 4, b_stage_u = static_cast<uint32_t>(p.b_stage_bytes) >> 4;
      const uint32_t a_lo0 = desc_lo0 + (a_base >> 4), b_lo0 = desc_lo0 + (b_base >> 4);
      const uint32_t n_a_stages = static_cast<uint32_t>(p.a_stages), acc_cols = ROWS * acc_stride;
      const uint32_t idw1 = p.idesc_w[0], idw2 = p.idesc_w[1], idw3 = p.idesc_w[2];
      const bool g3 = p.fuse_g >= 3;
      const int n_chunks = p.n_chunks;
      const int total_steps = p.n_rounds * n_chunks;
      uint32_t cur_a_lo = a_lo0, cur_b_lo = b_lo0, cur_d = tmem_base;
      uint32_t cur_commit_a = bar_a_empty, cur_commit_acc = n_chunks == 1 ? bar_acc_full : 0u;
      int c = 0;
      bool first_round = true;
      for (int step = 0; step < total_steps; ++step) {
        const uint32_t d_base = cur_d;
        uint32_t n_a_lo = 0, n_b_lo = 0, n_d = 0, n_commit_a = 0, n_commit_acc = 0;
        uint32_t nsa = sa, npa = pa, nas = as, npacc = pacc;
        bool ready = true, next_new_patch = false;
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          const uint32_t b_lo_dx = cur_b_lo + dx * b_stage_u;
          if (first_round && step + dx > 0) {  // (stage 0 was waited for before the loop)
            MZ_TIMED(2, mbar_wait(bar_b_full + 8 * (c * 3 + dx), 0));
            tc_fence_after();
          }
          if (dx == 2) {
            // ---- bookkeeping of the NEXT step, one filter column of tensor work still to be issued after it ----
            const bool last_chunk = c == n_chunks - 1;
            if (++nsa == n_a_stages) {
              nsa = 0;
              npa ^= 1u;
            }
            n_a_lo = a_lo0 + nsa * a_stage_u;
            n_commit_a = bar_a_empty + 8 * nsa;
            if (last_chunk) {
              if (++nas == static_cast<uint32_t>(p.acc_stages)) {
                nas = 0;
                npacc ^= 1u;
              }
              n_b_lo = b_lo0;
              next_new_patch = true;
              c = 0;
              first_round = false;
            } else {
              n_b_lo = cur_b_lo + 3 * b_stage_u;
              ++c;
            }
            n_d = tmem_base + nas * acc_cols;
            n_commit_acc = c == n_chunks - 1 ? bar_acc_full + 8 * nas : 0u;  // (c is already the next step's chunk)
            if (step + 1 < total_steps) {
              ready = test_uniform(bar_a_full + 8 * nsa, npa);
              if (last_chunk) ready = test_uniform(bar_acc_empty + 8 * nas, npacc ^ 1u) && ready;
              tc_fence_after();
            }
          }
          if (issue) {
#pragma unroll
            for (int t = 0; t < KT; ++t) {
#pragma unroll
              for (int i = -1; i <= ROWS; ++i) {  // input row i feeds output rows i+1-dy, dy in [dy_lo, dy_hi]
                const int dy_lo = (i + 2 - ROWS) > 0 ? (i + 2 - ROWS) : 0, dy_hi = (i + 1) < 2 ? (i + 1) : 2;
                const int cnt = dy_hi - dy_lo + 1;
                const uint64_t adesc = (static_cast<uint64_t>(desc_hi) << 32) | (cur_a_lo + (i + 1) * RP + dx * DX + t * a_kp);
                const uint32_t b_lo = b_lo_dx + dy_lo * TB + t * b_kp;
                const uint32_t d_lo = d_base + (ROWS - 2 - i + dy_lo) * acc_stride;  // block of output row i+1-dy_lo
                if (cnt == 1) {
                  umma_acc(d_lo, adesc, (static_cast<uint64_t>(desc_hi) << 32) | b_lo, idw1);
                } else if (cnt == 2) {
                  umma_acc(d_lo, adesc, (static_cast<uint64_t>(desc_hi) << 32) | b_lo, idw2);
                } else if (g3) {
                  umma_acc(d_lo, adesc, (static_cast<uint64_t>(desc_hi) << 32) | b_lo, idw3);
                } else {  // three taps, windows of two: (dy0, dy1) then dy2
                  umma_acc(d_lo, adesc, (static_cast<uint64_t>(desc_hi) << 32) | b_lo, idw2);
                  umma_acc(d_lo + 2 * acc_stride, adesc, (static_cast<uint64_t>(desc_hi) << 32) | (b_lo + 2 * TB), idw1);
                }
              }
            }
          }
        }
        if (leader) {
          umma_commit(cur_commit_a);
          if (cur_commit_acc != 0u) umma_commit(cur_commit_acc);
        }
        if (!ready) {  // rare: the producer or the epilogue is behind
          if (next_new_patch) MZ_TIMED(0, mbar_wait(bar_acc_empty + 8 * nas, npacc ^ 1u));
          MZ_TIMED(1, mbar_wait(bar_a_full + 8 * nsa, npa));
          tc_fence_after();
        }
        sa = nsa;
        pa = npa;
        as = nas;
        pacc = npacc;
        cur_a_lo = n_a_lo;
        cur_b_lo = n_b_lo;
        cur_d = n_d;
        cur_commit_a = n_commit_a;
        cur_commit_acc = n_commit_acc;
      }
    } else if (p.res_b) {
      // ---- resident filter bank: one hand-off per K chunk, all nine taps issued back to back ----
      // Measured with mz_probe_set_gap (tools/gpu_diag.py gap): for the operand-fetch-bound UMMA shapes (N <= 128 at
      // M = 128) the tensor pipe has NO slack -- every cycle the issuing thread spends away from the next tcgen05.mma
      // beyond one UMMA time (44 / 56 cycles at N = 48 / 96) is a bubble.  So all bookkeeping of the next step (ring
      // positions, descriptor bases, commit addresses, barrier sampling, the after-sync fence) runs between the second
      // and the third filter row of the current step, and what follows the last UMMA of a step is two commits and one
      // normally-not-taken branch.  The weight stages are waited for once, during the first patch.
      const uint32_t a_stage_u = static_cast<uint32_t>(p.a_stage_bytes) >> 4, b_stage_u = static_cast<uint32_t>(p.b_stage_bytes) >> 4;
      const uint32_t a_lo0 = desc_lo0 + (a_base >> 4), b_lo0 = desc_lo0 + (b_base >> 4);
      const uint32_t n_a_stages = static_cast<uint32_t>(p.a_stages), acc_cols = ROWS * acc_stride;
      const int n_chunks = p.n_chunks;
      const int total_steps = p.n_rounds * n_chunks;
      uint32_t cur_a_lo = a_lo0, cur_b_lo = b_lo0, cur_d = tmem_base;
      uint32_t cur_commit_a = bar_a_empty, cur_commit_acc = n_chunks == 1 ? bar_acc_full : 0u;
      uint32_t cur_first = 0u;  // 0: the first UMMA of the step overwrites the accumulator (first chunk of a patch)
      int c = 0;
      bool first_round = true;
      const uint32_t kt_last = static_cast<uint32_t>(p.kt_last);
      cur_kt = n_chunks == 1 ? kt_last : KT;
      for (int step = 0; step < total_steps; ++step) {
        const uint32_t d_base = cur_d;
        uint32_t n_a_lo = 0, n_b_lo = 0, n_d = 0, n_commit_a = 0, n_commit_acc = 0, n_first = 0, n_kt = KT;
        uint32_t nsa = sa, npa = pa, nas = as, npacc = pacc;
        bool ready = true;
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
          const uint32_t b_lo_stage = cur_b_lo + dy * b_stage_u;
          if (first_round && step + dy > 0) {  // (stage 0 was waited for before the loop)
            MZ_TIMED(2, mbar_wait(bar_b_full + 8 * (c * 3 + dy), 0));
            tc_fence_after();
          }
          const uint32_t a_lo_dy = cur_a_lo + dy * DY;
          const uint32_t first = dy == 0 ? cur_first : 1u;
          if (dy == 2) {
            // ---- bookkeeping of the NEXT step, one filter row of tensor work still to be issued after it ----
            const bool last_chunk = c == n_chunks - 1;
            if (++nsa == n_a_stages) {
              nsa = 0;
              npa ^= 1u;
            }
            n_a_lo = a_lo0 + nsa * a_stage_u;
            n_commit_a = bar_a_empty + 8 * nsa;
            if (last_chunk) {
              if (++nas == static_cast<uint32_t>(p.acc_stages)) {
                nas = 0;
                npacc ^= 1u;
              }
              n_b_lo = b_lo0;
              n_first = 0u;
              c = 0;
              first_round = false;
            } else {
              n_b_lo = cur_b_lo + 3 * b_stage_u;
              n_first = 1u;
              ++c;
            }
            n_d = tmem_base + nas * acc_cols;
            n_commit_acc = c == n_chunks - 1 ? bar_acc_full + 8 * nas : 0u;  // (c is already the next step's chunk)
            n_kt = c == n_chunks - 1 ? kt_last : KT;
            if (step + 1 < total_steps) {
              ready = test_uniform(bar_a_full + 8 * nsa, npa);
              if (last_chunk) ready = test_uniform(bar_acc_empty + 8 * nas, npacc ^ 1u) && ready;
              tc_fence_after();
            }
          }
          MZ_ISSUE_TAP(0)
          MZ_ISSUE_TAP(1)
          MZ_ISSUE_TAP(2)
        }
        if (leader) {
          if (PAIR) {
            umma2_commit_mcast(cur_commit_a, 3);
            if (cur_commit_acc != 0u) umma2_commit_mcast(cur_commit_acc, 3);
          } else {
            umma_commit(cur_commit_a);
            if (cur_commit_acc != 0u) umma_commit(cur_commit_acc);
          }
        }
        if (!ready) {  // rare: the producer or the epilogue is behind
          if (n_first == 0u) MZ_TIMED(0, mbar_wait(bar_acc_empty + 8 * nas, npacc ^ 1u));
          MZ_TIMED(1, mbar_wait(bar_a_full + 8 * nsa, npa));
          tc_fence_after();
        }
        sa = nsa;
        pa = npa;
        as = nas;
        pacc = npacc;
        cur_a_lo = n_a_lo;
        cur_b_lo = n_b_lo;
        cur_d = n_d;
        cur_commit_a = n_commit_a;
        cur_commit_acc = n_commit_acc;
        cur_first = n_first;
        cur_kt = n_kt;
      }
    } else {
      // ---- streamed weights: one hand-off per filter row (weight stage), same minimal-gap structure ----
      const uint32_t a_stage_u = static_cast<uint32_t>(p.a_stage_bytes) >> 4, b_stage_u = static_cast<uint32_t>(p.b_stage_bytes) >> 4;
      const uint32_t a_lo0 = desc_lo0 + (a_base >> 4), b_lo0 = desc_lo0 + (b_base >> 4);
      const uint32_t n_a_stages = static_cast<uint32_t>(p.a_stages), n_b_stages = static_cast<uint32_t>(p.b_stages);
      const uint32_t n_acc_stages = static_cast<uint32_t>(p.acc_stages), acc_cols = ROWS * acc_stride;
      const int n_chunks = p.n_chunks;
      const int total_steps = p.n_rounds * n_chunks * 3;
      uint32_t cur_a_lo_dy = a_lo0, cur_b_lo = b_lo0, cur_d = tmem_base;
      uint32_t cur_commit_b = bar_b_empty, cur_commit_a = 0u, cur_commit_acc = 0u, cur_first = 0u;
      int c = 0, dy = 0;
      for (int step = 0; step < total_steps; ++step) {
        const uint32_t d_base = cur_d, a_lo_dy = cur_a_lo_dy, b_lo_stage = cur_b_lo, first = cur_first;
        MZ_ISSUE_TAP(0)
        MZ_ISSUE_TAP(1)
        // ---- bookkeeping of the NEXT step, one tap of tensor work still to be issued after it ----
        uint32_t nsb = sb + 1, npb = pb, nsa = sa, npa = pa, nas = as, npacc = pacc;
        if (nsb == n_b_stages) {
          nsb = 0;
          npb ^= 1u;
        }
        uint32_t n_a_lo_dy = cur_a_lo_dy + DY, n_d = cur_d, n_first = 1u;
        int ndy = dy + 1, nc = c;
        bool need_a = false, need_acc = false;
        if (dy == 2) {
          ndy = 0;
          need_a = true;
          if (++nsa == n_a_stages) {
            nsa = 0;
            npa ^= 1u;
          }
          n_a_lo_dy = a_lo0 + nsa * a_stage_u;
          if (c == n_chunks - 1) {
            nc = 0;
            need_acc = true;
            if (++nas == n_acc_stages) {
              nas = 0;
              npacc ^= 1u;
            }
            n_d = tmem_base + nas * acc_cols;
            n_first = 0u;
          } else {
            nc = c + 1;
          }
        }
        const uint32_t n_b_lo = b_lo0 + nsb * b_stage_u, n_commit_b = bar_b_empty + 8 * nsb;
        const uint32_t n_commit_a = ndy == 2 ? bar_a_empty + 8 * nsa : 0u;
        const uint32_t n_commit_acc = (ndy == 2 && nc == n_chunks - 1) ? bar_acc_full + 8 * nas : 0u;
        bool ready = true;
        if (step + 1 < total_steps) {
          ready = test_uniform(bar_b_full + 8 * nsb, npb);
          if (need_a) ready = test_uniform(bar_a_full + 8 * nsa, npa) && ready;
          // (a single TMEM stage is released by the epilogue of THIS patch: always the slow path)
          if (need_acc) ready = la_acc ? (test_uniform(bar_acc_empty + 8 * nas, npacc ^ 1u) && ready) : false;
          tc_fence_after();
        } else {
          need_a = need_acc = false;
        }
        MZ_ISSUE_TAP(2)
        if (leader) {
          if (PAIR) {  // release / signal in BOTH CTAs of the pair
            umma2_commit_mcast(cur_commit_b, 3);
            if (cur_commit_a != 0u) umma2_commit_mcast(cur_commit_a, 3);
            if (cur_commit_acc != 0u) umma2_commit_mcast(cur_commit_acc, 3);
          } else {
            if (p.cluster > 1)
              umma_commit_mcast(cur_commit_b, cta_mask);
            else
              umma_commit(cur_commit_b);
            if (cur_commit_a != 0u) umma_commit(cur_commit_a);
            if (cur_commit_acc != 0u) umma_commit(cur_commit_acc);
          }
        }
        if (!ready) {  // the producer or the epilogue is behind
          if (need_acc) MZ_TIMED(0, mbar_wait(bar_acc_empty + 8 * nas, npacc ^ 1u));
          if (need_a) MZ_TIMED(1, mbar_wait(bar_a_full + 8 * nsa, npa));
          MZ_TIMED(2, mbar_wait(bar_b_full + 8 * nsb, npb));
          tc_fence_after();
        }
        sb = nsb;
        pb = npb;
        sa = nsa;
        pa = npa;
        as = nas;
        pacc = npacc;
        dy = ndy;
        c = nc;
        cur_a_lo_dy = n_a_lo_dy;
        cur_b_lo = n_b_lo;
        cur_d = n_d;
        cur_commit_b = n_commit_b;
        cur_commit_a = n_commit_a;
        cur_commit_acc = n_commit_acc;
        cur_first = n_first;
      }
    }
#undef MZ_ISSUE_TAP
    __syncwarp();
  } else if (warp >= 4 && warp < 4 + p.epi_warps) {
    // =============================== epilogue ===============================
    // Warp w owns the 32 pixels of TMEM lane quarter w % 4.  With eight epilogue warps two warps share a quarter and
    // split the work of a patch -- (row, output box) items in mode 0, accumulator rows in modes 1 and 2 -- so each SM
    // sub-partition has two warps to hide tcgen05.ld / MUFU / fence latencies behind one another.
    // Nothing goes to or from global memory through the LSU: results are written as swizzled 16-byte chunks into
    // warp-private staging boxes and leave by TMA store (coalesced, asynchronous); the fp32 residual row-tile arrives
    // by TMA load before the accumulator is waited for, and the tiles of the NEXT patch are prefetched into L2 a whole
    // patch ahead.  (Per-thread 16-byte global accesses at a 384-byte lane stride cost 32 sectors per instruction
    // and made the epilogue, not the tensor pipe, the bottleneck.)
    griddep_wait();  // FiLM table, residual stream, LR image: written by earlier kernels of the stream
    const int q = warp & 3;          // TMEM lane quarter this warp may read (== warp % 4)
    const int ew = warp - 4;         // staging slot / residual barrier of this warp
    const int half = ew >> 2;        // 0 | 1: which share of a patch this warp takes
    const int nh = p.epi_warps >> 2;  // warps per lane quarter (1 | 2)
    float* film_s = reinterpret_cast<float*>(gen_base + sp.film);
    int film_b = -1;
    float amax = 0.f;  // fp16 range guard: largest magnitude this thread rounded into a 16-bit operand (EpiParams::sat)
    uint32_t as = 0, pacc = 0, rpar = 0, ring = 0;
    const uint32_t n_pad = p.epi.n_pad;
    const uint32_t row16 = p.e16 * 2, row32 = p.e32 * 4;  // staging row bytes (= TMA box inner extent): 16-bit / fp32 boxes
    const uint32_t box16 = 32 * row16, box32 = 32 * row32;        // one warp-box: 32 pixels
    const uint32_t nb16 = n_pad / p.e16, nb32 = n_pad / p.e32;
    const uint32_t sh16 = 31 - __clz(p.e16), sh32 = 31 - __clz(p.e32);  // box widths are powers of two
    // warp-private staging: mode 0 -> ring of 16-bit boxes; mode 1 -> res_rows x (fp32 row-tile + 16-bit row-tile)
    // one accumulator row of this warp: fp32 tile + 16-bit tile
    const uint32_t row_stage = 32 * n_pad * 6;
    const uint32_t st_base = base + sp.stage + ew * (MODE == 0 ? p.o_ring * box16 : p.res_rows * row_stage);
    const bool all_rows = p.res_rows > 1;
    const uint32_t my_res = bar_res + 64 * ew;  // (eight barriers per warp: one per residual box in the sliced form)
    const int n_epi_threads = p.epi_warps * 32;
    bool preloaded = false, pending_last = false;  // sliced form: what of the current row's residual was requested ahead
    for (int round = 0; round < p.n_rounds; ++round) {
      const int unit_raw = round * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
      const bool unit_ok = unit_raw < p.n_units;  // CTA-uniform
      const int unit = min(unit_raw, p.n_units - 1);
      const int b = unit / units_per_img;
      const int rem = unit - b * units_per_img;
      const int ty = rem / p.tiles_x, tx = rem - ty * p.tiles_x;
      const int xw = tx * kTileW + q * 32;  // first pixel of this warp
      const int x = xw + lane;
      const int y0 = ty * ROWS;
      const bool ok = x < p.epi.W;
      const bool live = unit_ok && !(p.dbg & 4);

      if (MODE == 0 && b != film_b) {  // CTA-uniform: all epilogue warps take it together
        named_bar_sync(1, n_epi_threads);  // nobody still reads the previous image's rows
        for (int i = threadIdx.x - 128; i < 2 * p.epi.n_pad; i += n_epi_threads) {
          float v = i < p.epi.n_pad ? 1.f : 0.f;
          if (p.epi.film != nullptr) v = __ldg(p.epi.film + static_cast<size_t>(b) * 2 * p.epi.n_pad + i);
          film_s[i] = 0.5f * v;  // SiLU's v/2 folded into scale and shift (exact): see silu_h
        }
        named_bar_sync(1, n_epi_threads);
        film_b = b;
      }

      if (MODE == 1 && p.sliced) {
        // ---- sliced residual epilogue (one row buffer per warp) ----
        // The fp32 row tile and its 16-bit shadow are handled box by box (e32 channels x 32 pixels; e16 == e32): box j is
        // waited for, updated and stored on its own, and box j of the NEXT row of this warp -- in this patch or the next
        // one -- is requested one box later, when the stores of box j have been read (bulk_wait_read<1>).  Residual loads
        // therefore run a row ahead, and neither their latency nor the store read-out sits between two rows.
        const uint32_t st_z = st_base, st_o = st_z + 32 * n_pad * 4;
        const uint32_t slice_bytes = 32 * p.e32 * 4;
        auto finish16s = [&](const uint32_t* v, uint32_t n0) {
          const uint32_t bz = n0 >> sh32, cz = (n0 - (bz << sh32)) >> 2;
          const uint32_t zrow = st_z + bz * box32 + lane * row32;
          uint32_t o[8], addr[4];
          float4 z[4];
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            addr[kk] = zrow + swz_chunk(lane, cz + kk, row32) * 16;
            z[kk] = lds128f(addr[kk]);
          }
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            z[kk].x += __uint_as_float(v[4 * kk + 0]);
            z[kk].y += __uint_as_float(v[4 * kk + 1]);
            z[kk].z += __uint_as_float(v[4 * kk + 2]);
            z[kk].w += __uint_as_float(v[4 * kk + 3]);
            sts128(addr[kk], __float_as_uint(z[kk].x), __float_as_uint(z[kk].y), __float_as_uint(z[kk].z), __float_as_uint(z[kk].w));
            amax = fmaxf(fmaxf(amax, fmaxf(fabsf(z[kk].x), fabsf(z[kk].y))), fmaxf(fabsf(z[kk].z), fabsf(z[kk].w)));
            o[2 * kk] = pack_op2(p.epi.bf16, z[kk].x, z[kk].y);
            o[2 * kk + 1] = pack_op2(p.epi.bf16, z[kk].z, z[kk].w);
          }
          const uint32_t bo = n0 >> sh16, co = (n0 - (bo << sh16)) >> 3;
          const uint32_t orow = st_o + bo * box16 + lane * row16;
          sts128(orow + swz_chunk(lane, co, row16) * 16, o[0], o[1], o[2], o[3]);
          sts128(orow + swz_chunk(lane, co + 1, row16) * 16, o[4], o[5], o[6], o[7]);
        };
        bool acc_waited = false;
        for (int r = half; r < ROWS; r += nh) {
          const int y = y0 + r;
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                                 (as * ROWS + (FUSE ? ROWS - 1 - r : r)) * p.acc_stride;
          const bool valid = live && y < p.epi.H;  // (warp-uniform)
          if (valid && lane == 0) {
            if (!preloaded) {  // nothing of this row was requested ahead (first row, or the previous one was skipped)
              bulk_wait_read<0>();
              for (uint32_t j = 0; j < nb32; ++j) {
                mbar_expect_tx(my_res + 8 * j, slice_bytes);
                tma_load_4d(st_z + j * box32, &p.tmZ, my_res + 8 * j, j * p.e32, xw, y, b);
              }
            } else if (pending_last) {
              bulk_wait_read<0>();
              mbar_expect_tx(my_res + 8 * (nb32 - 1), slice_bytes);
              tma_load_4d(st_z + (nb32 - 1) * box32, &p.tmZ, my_res + 8 * (nb32 - 1), (nb32 - 1) * p.e32, xw, y, b);
            }
          }
          if (!acc_waited) {
            MZ_TIMED(0, mbar_wait(bar_acc_full + 8 * as, pacc));
            __syncwarp();
            tc_fence_after();
            acc_waited = true;
          }
          if (!valid) {  // below the image / surplus patch: nothing to store (FUSE still re-zeroes its accumulators)
            if (FUSE)
              for (uint32_t n0 = 0; n0 < n_pad; n0 += 16) tmem_zero16(taddr + n0);
            preloaded = pending_last = false;
            continue;
          }
          // this warp's next row: in this patch, or the first one of its next patch
          int nb_ = b, ny = y + nh, nxw = xw;
          bool nvalid = r + nh < ROWS;
          if (!nvalid) {
            const int nunit = unit_raw + static_cast<int>(gridDim.x);
            if (round + 1 < p.n_rounds && nunit < p.n_units) {
              nb_ = nunit / units_per_img;
              const int nrem = nunit - nb_ * units_per_img;
              const int nty = nrem / p.tiles_x, ntx = nrem - nty * p.tiles_x;
              ny = nty * ROWS + half;
              nxw = ntx * kTileW + q * 32;
              nvalid = half < ROWS;
            }
          }
          nvalid = nvalid && ny < p.epi.H && !(p.dbg & 4);
          for (uint32_t j = 0; j < nb32; ++j) {
            mbar_wait(my_res + 8 * j, rpar);
            const uint32_t n0 = j * p.e32;
            if (p.e32 == 32) {
              uint32_t v[32];
              tmem_ld32(taddr + n0, v);
              tmem_ld_wait();
              if (FUSE) {
                tmem_zero16(taddr + n0);
                tmem_zero16(taddr + n0 + 16);
              }
              finish16s(v, n0);
              finish16s(v + 16, n0 + 16);
            } else {
              uint32_t v[16];
              tmem_ld16(taddr + n0, v);
              tmem_ld_wait();
              if (FUSE) tmem_zero16(taddr + n0);
              finish16s(v, n0);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              tma_store_4d(&p.tmZ, st_z + j * box32, j * p.e32, xw, y, b);
              tma_store_4d(&p.tmO, st_o + j * box16, j * p.e16, xw, y, b);
              bulk_commit();
              if (j >= 1 && nvalid) {  // box j-1: its stores (one group back) have been read -> the next row's box j-1
                bulk_wait_read<1>();
                mbar_expect_tx(my_res + 8 * (j - 1), slice_bytes);
                tma_load_4d(st_z + (j - 1) * box32, &p.tmZ, my_res + 8 * (j - 1), (j - 1) * p.e32, nxw, ny, nb_);
              }
            }
          }
          rpar ^= 1u;
          preloaded = nvalid && nb32 > 1;
          pending_last = preloaded;
        }
        if (!acc_waited) {  // (a warp without rows in this patch still takes part in the accumulator hand-off)
          MZ_TIMED(0, mbar_wait(bar_acc_full + 8 * as, pacc));
          __syncwarp();
          tc_fence_after();
        }
        if (FUSE) tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR)
            mbar_arrive_remote(mapa_u32(bar_acc_empty + 8 * as, 0));
          else
            mbar_arrive(bar_acc_empty + 8 * as);
        }
        if (++as == static_cast<uint32_t>(p.acc_stages)) {
          as = 0;
          pacc ^= 1u;
        }
        continue;
      }

      // residual row-tiles of this warp's rows (r = half, half + nh, ...): TMA load into the warp's staging once its
      // previous stores have finished reading it.  With a buffer per row (res_rows > 1) all of them are requested up
      // front on one barrier; otherwise row k+1 is requested when row k has been stored.
      auto load_residual = [&](int k_lo, int k_hi) {  // k indexes this warp's rows: r = half + k * nh
        if (MODE == 1 && live && lane == 0) {
          int nrows = 0;
          for (int k = k_lo; k < k_hi; ++k) nrows += (half + k * nh < ROWS && y0 + half + k * nh < p.epi.H) ? 1 : 0;
          if (nrows > 0) {
            bulk_wait_read<0>();
            mbar_expect_tx(my_res, nrows * 32 * n_pad * 4);
            for (int k = k_lo; k < k_hi; ++k) {
              const int r = half + k * nh;
              if (r >= ROWS || y0 + r >= p.epi.H) break;
              const uint32_t dst = st_base + (all_rows ? k : 0) * row_stage;
              for (uint32_t bx = 0; bx < nb32; ++bx) tma_load_4d(dst + bx * box32, &p.tmZ, my_res, bx * p.e32, xw, y0 + r, b);
            }
          }
        }
      };
      constexpr int kMyRowsMax = ROWS;  // upper bound of rows per warp
      load_residual(0, all_rows ? kMyRowsMax : 1);
      if (MODE == 1 && lane == 0 && !(p.dbg & 4)) {
        // L2 prefetch of the residual tiles this warp will need for the NEXT patch: by then they are an L2 hit
        // (~0.5 us) instead of an HBM round trip that a single row buffer cannot hide
        const int nunit = unit_raw + static_cast<int>(gridDim.x);
        if (nunit < p.n_units) {
          const int nb = nunit / units_per_img;
          const int nrem = nunit - nb * units_per_img;
          const int nty = nrem / p.tiles_x, ntx = nrem - nty * p.tiles_x;
          for (int r = half; r < ROWS; r += nh) {
            if (nty * ROWS + r >= p.epi.H) break;
            for (uint32_t bx = 0; bx < nb32; ++bx)
              tma_prefetch_4d(&p.tmZ, bx * p.e32, ntx * kTileW + q * 32, nty * ROWS + r, nb);
          }
        }
      }

      MZ_TIMED(0, mbar_wait(bar_acc_full + 8 * as, pacc));
      __syncwarp();
      tc_fence_after();
      bool rows_done = false;
      if constexpr (MODE == 2 && ROWS == 4) {
        // 2X head, eight epilogue warps: each warp finishes two ADJACENT rows of the patch in one pass (their bicubic
        // neighbourhoods share four of five LR rows, and one load latency is exposed instead of two: epi_head2_pair)
        if (nh == 2 && p.epi.r == 2 && !(p.dbg & 128)) {  // (warp-uniform; dbg 128: row-by-row form)
          rows_done = true;
          const int r0 = 2 * half, y = y0 + r0;
          const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
          const uint32_t t0 = lane_base + (as * ROWS + (FUSE ? ROWS - 1 - r0 : r0)) * p.acc_stride;
          const uint32_t t1 = lane_base + (as * ROWS + (FUSE ? ROWS - 2 - r0 : r0 + 1)) * p.acc_stride;
          if (y >= p.epi.H || !live) {  // (warp-uniform) neither row is stored
            if (FUSE) {
              tmem_zero16(t0);
              tmem_zero16(t1);
            }
          } else {
            uint32_t v0[16], v1[16];
            tmem_ld16(t0, v0);
            tmem_ld16(t1, v1);
            tmem_ld_wait();
            if (FUSE) {
              tmem_zero16(t0);
              tmem_zero16(t1);
            }
            if (ok) {
              const bool interior = xw >= 2 && xw + 33 < p.epi.W;  // (warp-uniform) no clamped column in this warp
              const bool second = y + 1 < p.epi.H;
              epi_head2<(LAY & 1) != 0, (LAY & 2) != 0, (LAY & 4) != 0>(p.epi, b, y, x, v0, v1, interior, second);
            }
          }
        }
      }
      for (int r = (MODE == 0 ? 0 : half), k = 0; r < ROWS && !rows_done; r += (MODE == 0 ? 1 : nh), ++k) {
        const int y = y0 + r;
        // (FUSE keeps output row r in TMEM block ROWS-1-r so that the blocks of stacked vertical taps are adjacent)
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                               (as * ROWS + (FUSE ? ROWS - 1 - r : r)) * p.acc_stride;
        if (y >= p.epi.H || !live) {  // warp-uniform: nothing to store for this row
          if constexpr (!FUSE) {
            break;
          } else {
            // the accumulators of a row that is not stored (below the image, surplus patch) still have to be re-zeroed
            for (uint32_t n0 = 0; n0 < n_pad; n0 += 16) {
              if (MODE == 0 && nh == 2 &&
                  ((static_cast<uint32_t>(r) * nb16 + n0 / static_cast<uint32_t>(p.e16)) & 1u) != static_cast<uint32_t>(half))
                continue;  // the other warp of this lane quarter owns that box
              tmem_zero16(taddr + n0);
            }
            continue;
          }
        }
        if (MODE == 2) {
          float acc[48];
          uint32_t v[16];
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            if (j * 16 < p.epi.n_pad) {  // warp-uniform
              tmem_ld16(taddr + j * 16, v);
              tmem_ld_wait();
              if (FUSE) tmem_zero16(taddr + j * 16);
#pragma unroll
              for (int i = 0; i < 16; ++i) acc[j * 16 + i] = __uint_as_float(v[i]);
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) acc[j * 16 + i] = 0.f;
            }
          }
          if (ok) {
            const bool interior = xw >= 2 && xw + 33 < p.epi.W;  // (warp-uniform) no clamped column in this warp
            constexpr bool XN = (LAY & 1) != 0, YN = (LAY & 2) != 0, I16 = (LAY & 4) != 0;
            if (p.epi.r == 4)
              epi_head_r<4, XN, YN, I16>(p.epi, b, y, x, acc, interior);
            else if (p.epi.r == 2)
              epi_head_r<2, XN, YN, I16>(p.epi, b, y, x, acc, interior);
            else
              epi_head_r<3, XN, YN, I16>(p.epi, b, y, x, acc, interior);
          }
        } else if (MODE == 1) {
          if (k > 0 && !all_rows) load_residual(k, k + 1);
          if (k == 0 || !all_rows) {
            mbar_wait(my_res, rpar);
            rpar ^= 1u;
          }
          const uint32_t st_z = st_base + (all_rows ? k : 0) * row_stage, st_o = st_z + 32 * n_pad * 4;
          // sixteen channels: z += acc in the fp32 staging tile (in place), 16-bit shadow into the output tile
          auto finish16 = [&](const uint32_t* v, uint32_t n0) {
            const uint32_t bz = n0 >> sh32, cz = (n0 - (bz << sh32)) >> 2;  // fp32 box, first 16-byte chunk in its row
            const uint32_t zrow = st_z + bz * box32 + lane * row32;
            uint32_t o[8], addr[4];
            float4 z[4];
            // all four loads first: the shared-memory accessors are volatile (ordered), so a load / add / store per chunk
            // would expose the full load latency four times per sixteen channels
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              addr[kk] = zrow + swz_chunk(lane, cz + kk, row32) * 16;
              z[kk] = lds128f(addr[kk]);
            }
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              z[kk].x += __uint_as_float(v[4 * kk + 0]);
              z[kk].y += __uint_as_float(v[4 * kk + 1]);
              z[kk].z += __uint_as_float(v[4 * kk + 2]);
              z[kk].w += __uint_as_float(v[4 * kk + 3]);
              sts128(addr[kk], __float_as_uint(z[kk].x), __float_as_uint(z[kk].y), __float_as_uint(z[kk].z), __float_as_uint(z[kk].w));
              amax = fmaxf(fmaxf(amax, fmaxf(fabsf(z[kk].x), fabsf(z[kk].y))), fmaxf(fabsf(z[kk].z), fabsf(z[kk].w)));
              o[2 * kk] = pack_op2(p.epi.bf16, z[kk].x, z[kk].y);
              o[2 * kk + 1] = pack_op2(p.epi.bf16, z[kk].z, z[kk].w);
            }
            const uint32_t bo = n0 >> sh16, co = (n0 - (bo << sh16)) >> 3;
            const uint32_t orow = st_o + bo * box16 + lane * row16;
            sts128(orow + swz_chunk(lane, co, row16) * 16, o[0], o[1], o[2], o[3]);
            sts128(orow + swz_chunk(lane, co + 1, row16) * 16, o[4], o[5], o[6], o[7]);
          };
          if ((n_pad & 31u) == 0) {  // one TMEM load + one wait per 32 columns
            for (uint32_t n0 = 0; n0 < n_pad; n0 += 32) {
              uint32_t v[32];
              tmem_ld32(taddr + n0, v);
              tmem_ld_wait();
              if (FUSE) {
                tmem_zero16(taddr + n0);
                tmem_zero16(taddr + n0 + 16);
              }
              finish16(v, n0);
              finish16(v + 16, n0 + 16);
            }
          } else {
            for (uint32_t n0 = 0; n0 < n_pad; n0 += 16) {
              uint32_t v[16];
              tmem_ld16(taddr + n0, v);
              tmem_ld_wait();
              if (FUSE) tmem_zero16(taddr + n0);
              finish16(v, n0);
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            for (uint32_t bx = 0; bx < nb32; ++bx) tma_store_4d(&p.tmZ, st_z + bx * box32, bx * p.e32, xw, y, b);
            for (uint32_t bx = 0; bx < nb16; ++bx) tma_store_4d(&p.tmO, st_o + bx * box16, bx * p.e16, xw, y, b);
            bulk_commit();
          }
        } else {
          for (uint32_t bx = 0; bx < nb16; ++bx) {
            if (nh == 2 && ((static_cast<uint32_t>(r) * nb16 + bx) & 1u) != static_cast<uint32_t>(half)) continue;
            const uint32_t buf = st_base + (ring & static_cast<uint32_t>(p.o_ring - 1)) * box16;
            ++ring;
            if (lane == 0) {  // the store issued o_ring boxes ago has finished reading this buffer
              if (p.o_ring == 4)
                bulk_wait_read<3>();
              else
                bulk_wait_read<1>();
            }
            __syncwarp();
            const uint32_t orow = buf + lane * row16;
            // sixteen output channels: FiLM (pre-halved rows) + SiLU + 16-bit pack -> two swizzled 16-byte chunks
            auto finish16 = [&](const uint32_t* v, uint32_t n0, uint32_t sub) {
              const float4* sc = reinterpret_cast<const float4*>(film_s + n0);
              const float4* sh = reinterpret_cast<const float4*>(film_s + n_pad + n0);
              uint32_t o[8];
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                const float4 g = sc[kk], h = sh[kk];
                const float a0 = silu_h(fmaf(__uint_as_float(v[4 * kk + 0]), g.x, h.x));
                const float a1 = silu_h(fmaf(__uint_as_float(v[4 * kk + 1]), g.y, h.y));
                const float a2 = silu_h(fmaf(__uint_as_float(v[4 * kk + 2]), g.z, h.z));
                const float a3 = silu_h(fmaf(__uint_as_float(v[4 * kk + 3]), g.w, h.w));
                amax = fmaxf(fmaxf(amax, fmaxf(fabsf(a0), fabsf(a1))), fmaxf(fabsf(a2), fabsf(a3)));
                o[2 * kk] = pack_op2(p.epi.bf16, a0, a1);
                o[2 * kk + 1] = pack_op2(p.epi.bf16, a2, a3);
              }
              const uint32_t co = sub >> 3;
              sts128(orow + swz_chunk(lane, co, row16) * 16, o[0], o[1], o[2], o[3]);
              sts128(orow + swz_chunk(lane, co + 1, row16) * 16, o[4], o[5], o[6], o[7]);
            };
            if (p.e16 >= 32) {  // one TMEM load + one wait per 32 columns
              for (uint32_t sub = 0; sub < static_cast<uint32_t>(p.e16); sub += 32) {
                const uint32_t n0 = bx * p.e16 + sub;
                uint32_t v[32];
                tmem_ld32(taddr + n0, v);
                tmem_ld_wait();
                if (FUSE) {
                  tmem_zero16(taddr + n0);
                  tmem_zero16(taddr + n0 + 16);
                }
                finish16(v, n0, sub);
                finish16(v + 16, n0 + 16, sub + 16);
              }
            } else {
              const uint32_t n0 = bx * p.e16;
              uint32_t v[16];
              tmem_ld16(taddr + n0, v);
              tmem_ld_wait();
              if (FUSE) tmem_zero16(taddr + n0);
              finish16(v, n0, 0);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              tma_store_4d(&p.tmO, buf, bx * p.e16, xw, y, b);
              bulk_commit();
            }
          }
        }
      }
      if (FUSE) tmem_st_wait();  // the zeroes are in TMEM before the issuer may accumulate into this stage again
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR)
          mbar_arrive_remote(mapa_u32(bar_acc_empty + 8 * as, 0));  // the leader's issuer waits for both CTAs
        else
          mbar_arrive(bar_acc_empty + 8 * as);
      }
      if (++as == static_cast<uint32_t>(p.acc_stages)) {
        as = 0;
        pacc ^= 1u;
      }
    }
    if (lane == 0) bulk_wait_all();  // every TMA store of this warp has landed before the CTA exits
    // (an infinite value is caught too; fmaxf drops NaNs, which the 16-bit conversion keeps as NaN anyway)
    if (MODE != 2 && !p.epi.bf16 && p.epi.sat != nullptr && !(amax <= MZ_F16_MAX)) *p.epi.sat = 1u;
  }

  if (prof_on && lane == 0 && (warp == 0 || warp == 1 || warp == 4)) {
    const int role = warp == 4 ? 2 : warp;
    long long* dst = p.prof + (static_cast<size_t>(blockIdx.x) * 3 + role) * 8;
    tick[7] = clock64() - t_role0;  // whole role
    for (int i = 0; i < 8; ++i) dst[i] = tick[i];
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR || p.cluster > 1) cluster_sync_all();  // no CTA may exit while a peer can still signal into it
  if (warp == 2) {
    tc_fence_after();
    if (PAIR)
      tmem_dealloc2(tmem_base, p.tmem_cols);
    else
      tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
// ---- kernel lookup -------------------------------------------------------------------------------------------------
// One lookup function per epilogue mode and head layout, so that the build can compile the instantiations of each in
// its own translation unit: build.py compiles this file with -DMZ_TC_PART=<mode> for the kernels of modes 0 and 1,
// -DMZ_TC_PART=4 for the host side, -DMZ_TC_PART=2 for the planar head (LAY 0) and -DMZ_TC_PART=5..11 for the heads of
// LAY 1..7.  Without the define (a plain `nvcc -c conv_tc.cu`) everything lands in one object.
//   var 0: one CTA per patch, 1: CTA pair (cta_group::2), 2: fused rows.  Returns nullptr for a shape that has no kernel.
const void* tc_kernel_mode0(int ks, int rows, int var);
const void* tc_kernel_mode1(int ks, int rows, int var);
template <int LAY>  // the head for image layouts LAY
const void* tc_kernel_head_lay(int ks, int rows, int var);

template <int M, int K, int LAY = 0>
static const void* tc_kernel_rows(int rows, int var) {
  if (var == 0) {
    if (rows == 1) return reinterpret_cast<const void*>(conv_tc_kernel<M, K, 1, 0, LAY>);
    if (rows == 2) return reinterpret_cast<const void*>(conv_tc_kernel<M, K, 2, 0, LAY>);
    if (rows == 4) return reinterpret_cast<const void*>(conv_tc_kernel<M, K, 4, 0, LAY>);
  }
  if constexpr (M != 2 && K != 3) {  // pairs: the shapes the 64/96/128-channel encoders use (the head has no pair form)
    if (var == 1 && rows == 1) return reinterpret_cast<const void*>(conv_tc_kernel<M, K, 1, 1>);
    if (var == 1 && rows == 2) return reinterpret_cast<const void*>(conv_tc_kernel<M, K, 2, 1>);
  }
  if constexpr (M != 2) {
    if (var == 2 && rows == 2) return reinterpret_cast<const void*>(conv_tc_kernel<M, K, 2, 2>);
  }
  if (var == 2 && rows == 4) return reinterpret_cast<const void*>(conv_tc_kernel<M, K, 4, 2, LAY>);  // (head: four-row patches only)
  return nullptr;
}

template <int M, int LAY = 0>
static const void* tc_kernel_lookup(int ks, int rows, int var) {
  switch (ks) {
    case 1: return tc_kernel_rows<M, 1, LAY>(rows, var);
    case 2: return tc_kernel_rows<M, 2, LAY>(rows, var);
    case 3: return tc_kernel_rows<M, 3, LAY>(rows, var);
    case 4: return tc_kernel_rows<M, 4, LAY>(rows, var);
    default: return nullptr;
  }
}

#if !defined(MZ_TC_PART) || MZ_TC_PART == 0
const void* tc_kernel_mode0(int ks, int rows, int var) { return tc_kernel_lookup<0>(ks, rows, var); }
#endif
#if !defined(MZ_TC_PART) || MZ_TC_PART == 1
const void* tc_kernel_mode1(int ks, int rows, int var) { return tc_kernel_lookup<1>(ks, rows, var); }
#endif
#if !defined(MZ_TC_PART) || MZ_TC_PART == 2 || MZ_TC_PART >= 5
template <int LAY>
const void* tc_kernel_head_lay(int ks, int rows, int var) { return tc_kernel_lookup<2, LAY>(ks, rows, var); }
#endif
#if defined(MZ_TC_PART) && MZ_TC_PART == 2
template const void* tc_kernel_head_lay<0>(int ks, int rows, int var);
#elif defined(MZ_TC_PART) && MZ_TC_PART >= 5
template const void* tc_kernel_head_lay<MZ_TC_PART - 4>(int ks, int rows, int var);
#endif

#if !defined(MZ_TC_PART) || MZ_TC_PART == 4  // ---- host side ----------------------------------------------------------

static int pick_kc(int cin_p) { return cin_p % 64 == 0 ? 64 : (cin_p % 32 == 0 ? 32 : 16); }

static uint32_t pow2_cols(uint32_t c) {
  uint32_t v = 32;
  while (v < c) v <<= 1;
  return v;
}

// staging: 2 = deep (four output boxes / every accumulator row's residual in flight per warp), 1 = two boxes / one row,
// 0 = slim (two boxes of at most 32 channels) -- what is left beside a resident filter bank, -1 = two boxes of 16
// channels (1 KB each: eight epilogue warps beside a 166 KB bank and three activation stages)
static void fill_geometry(TcParams& p, int cin_p, int kc, int rows, int acc_stages, int halo_mode, int a_stages,
                          int b_stages, int staging, bool res_b) {
  const int nh = p.epi_warps / 4;
  p.o_ring = staging == 2 ? 4 : 2;
  p.res_rows = staging == 2 ? (rows + nh - 1) / nh : 1;
  p.res_b = res_b ? 1 : 0;
  p.kc = kc;
  // 16-channel sub-tiles are fused into one pipeline stage when the whole K extent is small (Cin = 48): three times
  // the UMMAs per barrier round trip
  p.subs = (kc == 16 && halo_mode == 0 && cin_p / 16 <= 3 && p.cluster <= 1 && !p.pair) ? cin_p / 16 : 1;
  p.n_chunks = cin_p / (kc * p.subs);
  p.rows = rows;
  p.acc_stages = acc_stages;
  p.acc_stride = p.fuse_g ? p.epi.n_pad : ((p.epi.n_pad + 31) / 32) * 32;  // FUSE: adjacent blocks, no padding
  p.halo_mode = halo_mode;
  p.a_stages = a_stages;
  p.b_stages = res_b ? 3 * p.n_chunks : b_stages;
  p.pw = halo_mode == 1 ? kTileW : kTileW + 2;
  int a_sub = (rows + 2) * p.pw * kc * 2;
  if (p.subs > 1) a_sub = ((a_sub + 1023) / 1024) * 1024;  // each sub-tile is its own TMA destination / swizzle frame
  const int a_bytes = (halo_mode == 1 ? 3 : p.subs) * a_sub;
  p.a_tx_bytes = (halo_mode == 1 ? 3 : p.subs) * (rows + 2) * p.pw * kc * 2;
  p.a_stage_bytes = ((a_bytes + 1023) / 1024) * 1024;
  const int n_local = p.pair ? p.epi.n_pad / 2 : p.epi.n_pad;  // weight rows held by this CTA
  p.b_tx_bytes = p.subs * 3 * n_local * kc * 2;  // the three horizontal taps of one filter row
  p.b_stage_bytes = ((p.b_tx_bytes + 1023) / 1024) * 1024;
  p.b_tap = (n_local * kc * 2) >> 4;
  p.a_kp = p.subs > 1 ? a_sub >> 4 : 2;
  p.b_kp = p.subs > 1 ? (3 * n_local * kc * 2) >> 4 : 2;
  p.tmem_cols = pow2_cols(static_cast<uint32_t>(acc_stages * rows * p.acc_stride));
  const int n = p.epi.n_pad;
  p.e16 = (n % 64 == 0 && staging > 0) ? 64 : ((n % 32 == 0 && staging >= 0) ? 32 : 16);  // staging -1: 16-channel boxes
  p.e32 = n % 32 == 0 ? 32 : 16;
  static const bool no_sliced = getenv("MZ_NO_SLICED_EPILOGUE") != nullptr;
  p.sliced = (p.epi.mode == 1 && p.res_rows == 1 && !no_sliced) ? 1 : 0;
  if (p.sliced) p.e16 = p.e32;  // one 16-bit box per fp32 box
  p.stage_bytes = p.epi.mode == 0   ? p.epi_warps * p.o_ring * 32 * p.e16 * 2
                  : p.epi.mode == 1 ? p.epi_warps * p.res_rows * 32 * n * 6
                                    : 0;
}

static bool fits(const TcParams& p) {
  return p.acc_stages * p.rows * p.acc_stride <= 512 && plan_smem(p).total + 1024 <= static_cast<uint32_t>(kMaxSmem);
}

// Everything a launch needs, prepared once per (operands, shape, tunables): the chosen geometry, the encoded tensor
// maps and the kernel instantiation.  mz_upscale keeps one per convolution of the model, so a repeated call costs one
// cudaLaunchKernelEx per convolution on the host instead of a configuration search and four cuTensorMapEncodeTiled.
struct ConvLaunchImpl {
  TcParams p;
  const void* fn;
  int grid, k;
  uint32_t smem;
  int mode, n_pad;
  int ks, var, lay;  // what `fn` was looked up for (the head's image layouts are patched per call)
};

// the head kernel for image layouts `lay` (bit 0 interleaved input, bit 1 interleaved output, bit 2 16-bit images)
static const void* tc_kernel_head(int lay, int ks, int rows, int var) {
  static const void* (*const heads[8])(int, int, int) = {tc_kernel_head_lay<0>, tc_kernel_head_lay<1>, tc_kernel_head_lay<2>,
                                                         tc_kernel_head_lay<3>, tc_kernel_head_lay<4>, tc_kernel_head_lay<5>,
                                                         tc_kernel_head_lay<6>, tc_kernel_head_lay<7>};
  return heads[lay](ks, rows, var);
}
static int head_layout(const EpiParams& e) {
  return (e.img.x_nhwc ? 1 : 0) | (e.img.y_nhwc ? 2 : 0) | (e.img.type == kImgU16 ? 4 : 0);
}
static_assert(sizeof(ConvLaunchImpl) <= sizeof(ConvLaunch::storage), "ConvLaunch::storage too small");

static int run_prepared(ConvLaunchImpl& L, cudaStream_t s) {
  TcParams& p = L.p;
  static long long* g_prof = nullptr;
  const bool prof = (p.dbg & 16) != 0;
  if (prof) {
    if (!g_prof) MZ_CUDA(cudaMalloc(&g_prof, sizeof(long long) * 4096 * 24));
    MZ_CUDA(cudaMemsetAsync(g_prof, 0, sizeof(long long) * 4096 * 24, s));
  }
  TcParams q = p;  // what the kernel sees
  q.prof = prof ? g_prof : nullptr;
  q.dbg &= ~16;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(L.grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = L.smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (L.k > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = L.k;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  static const bool no_pdl = getenv("MZ_NO_PDL") != nullptr;
  if (!no_pdl && !prof) {  // this grid may start while the previous kernel of the stream drains (see the kernel)
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  void* args[1] = {&q};
  MZ_CUDA(cudaLaunchKernelExC(&cfg, L.fn, args));
  if (prof) {  // diagnostic: synchronise and print mean ticks per role (stderr)
    MZ_CUDA(cudaStreamSynchronize(s));
    std::vector<long long> h(static_cast<size_t>(L.grid) * 24);
    MZ_CUDA(cudaMemcpy(h.data(), g_prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    double m[24] = {0};
    for (int c = 0; c < L.grid; ++c)
      for (int i = 0; i < 24; ++i) m[i] += static_cast<double>(h[static_cast<size_t>(c) * 24 + i]) / L.grid;
    fprintf(stderr,
            "[mz prof] mode %d rows %d kc %d n %d rounds %d | producer: wait_a_empty %.0f wait_b_empty %.0f total %.0f | "
            "mma: wait_acc_empty %.0f wait_a_full %.0f wait_b_full %.0f total %.0f | epilogue: wait_acc_full %.0f total %.0f\n",
            L.mode, p.rows, p.kc, L.n_pad, p.n_rounds, m[0], m[1], m[7], m[8], m[9], m[10], m[15], m[16], m[23]);
  }
  return MZ_OK;
}

int run_conv_tc(ConvLaunch& launch, cudaStream_t s) {
  MZ_REQUIRE(launch.valid, "conv: launch was not prepared");
  return run_prepared(*reinterpret_cast<ConvLaunchImpl*>(launch.storage), s);
}

int patch_conv_epi(ConvLaunch& launch, const EpiParams& e) {
  ConvLaunchImpl& L = *reinterpret_cast<ConvLaunchImpl*>(launch.storage);
  const int lay = head_layout(e);
  if (lay != L.lay) {  // same geometry, the instantiation for the other layouts
    const void* fn = tc_kernel_head(lay, L.ks, L.p.rows, L.var);
    MZ_REQUIRE(fn != nullptr, "conv: no head kernel for image layouts %d", lay);
    MZ_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    L.fn = fn;
    L.lay = lay;
  }
  L.p.epi.img = e.img;
  return MZ_OK;
}

int launch_conv_tc(const ConvArgs& a, const ConvTcTune& tune, int device, cudaStream_t s) {
  ConvLaunch L;
  L.valid = false;
  const int rc = prepare_conv_tc(a, tune, device, &L);
  return rc != MZ_OK ? rc : run_conv_tc(L, s);
}

int prepare_conv_tc(const ConvArgs& a, const ConvTcTune& tune, int device, ConvLaunch* out) {
  out->valid = false;
  ConvLaunchImpl& L = *reinterpret_cast<ConvLaunchImpl*>(out->storage);
  const EpiParams& e = a.epi;
  MZ_REQUIRE(e.B > 0 && e.H > 0 && e.W > 0, "conv: empty input (B %d, H %d, W %d)", e.B, e.H, e.W);
  MZ_REQUIRE(a.cin_p > 0 && a.cin_p % 16 == 0, "conv: cin_p must be a positive multiple of 16, %d given", a.cin_p);
  MZ_REQUIRE(e.n_pad >= 16 && e.n_pad % 16 == 0 && e.n_pad <= 256,
             "conv: n_pad must be a multiple of 16 in [16, 256], %d given", e.n_pad);
  MZ_REQUIRE(e.mode >= 0 && e.mode <= 2, "conv: bad epilogue mode %d", e.mode);
  MZ_REQUIRE(e.mode != 2 || e.n_pad <= 48, "head conv: n_pad must be <= 48, %d given", e.n_pad);
  MZ_REQUIRE(static_cast<long long>(e.H) * e.W < (1LL << 31), "conv: an image plane of %d x %d pixels exceeds 2^31", e.H, e.W);
  {  // dense layouts: extents are whole 16-byte runs, inside the GEMM width, and not wider than the pitch
    const int ie = a.in_extent ? a.in_extent : a.cin_p, oe = e.out_extent ? e.out_extent : e.n_pad;
    const int ze = e.zf_extent ? e.zf_extent : e.n_pad;
    MZ_REQUIRE(ie > 0 && ie <= a.cin_p && ie % 8 == 0 && (a.in_pitch == 0 ? ie == a.cin_p : ie <= a.in_pitch),
               "conv: in_extent %d does not fit cin_p %d / in_pitch %d (multiple of 8)", ie, a.cin_p, a.in_pitch);
    MZ_REQUIRE(e.mode == 2 || (oe > 0 && oe <= e.n_pad && oe % 8 == 0 && (e.out_pitch == 0 ? oe == e.n_pad : oe <= e.out_pitch)),
               "conv: out_extent %d does not fit n_pad %d / out_pitch %d (multiple of 8)", oe, e.n_pad, e.out_pitch);
    MZ_REQUIRE(e.mode != 1 || (ze > 0 && ze <= e.n_pad && ze % 4 == 0 && (e.zf_pitch == 0 ? ze == e.n_pad : ze <= e.zf_pitch)),
               "conv: zf_extent %d does not fit n_pad %d / zf_pitch %d (multiple of 4)", ze, e.n_pad, e.zf_pitch);
  }
  MZ_REQUIRE(tune.halo_mode >= 0 && tune.halo_mode <= 1, "conv: bad halo_mode %d", tune.halo_mode);
  MZ_REQUIRE(tune.cluster == 0 || tune.cluster == 1 || tune.cluster == 2 || tune.cluster == 4,
             "conv: cluster must be 0 (auto), 1, 2 or 4, %d given", tune.cluster);
  MZ_REQUIRE(tune.rows == 0 || tune.rows == 1 || tune.rows == 2 || tune.rows == 4,
             "conv: rows must be 0 (auto), 1, 2 or 4, %d given", tune.rows);
  MZ_REQUIRE(tune.kc == 0 || ((tune.kc == 16 || tune.kc == 32 || tune.kc == 64) && a.cin_p % tune.kc == 0),
             "conv: kc %d does not divide cin_p %d (or is not 16/32/64)", tune.kc, a.cin_p);

  MZ_REQUIRE(tune.epi_warps == 0 || tune.epi_warps == 4 || tune.epi_warps == 8,
             "conv: epi_warps must be 0 (auto), 4 or 8, %d given", tune.epi_warps);

  TcParams& p = L.p;
  memset(&p, 0, sizeof(p));
  p.epi = e;
  p.epi_warps = tune.epi_warps ? tune.epi_warps : 8;

  // cluster size: share the weight stream between k CTAs when the slices keep whole 8-row swizzle atoms
  {
    int k = tune.cluster ? tune.cluster : 1;  // multicast is opt-in: L2 is not the limiter at these tile sizes
    while (k > 1 && (e.n_pad % k != 0 || (e.n_pad / k) % 8 != 0)) k >>= 1;
    p.cluster = k;
    p.b_slice_rows = e.n_pad / k;
    p.dbg = (tune.dbg & 1) && k > 1 ? (tune.dbg & ~1) : tune.dbg;  // skipping multicast loads would deadlock peers
  }
  // ---- choose the patch geometry ----
  // First choice: the whole filter bank resident in shared memory (the persistent CTA then streams activations only;
  // re-streaming 83..332 KB of weights per patch is what saturates the L2 -> SM path otherwise).  It needs two TMEM
  // stages, two-row patches (unless TMEM only holds one-row stages) and at least two activation stages beside the
  // bank.  A bank that does not fit one CTA is split between the two CTAs of a pair (cta_group::2, M = 256 UMMAs:
  // each CTA holds N/2 weight rows).  Otherwise the weights are streamed per patch.
  // tune.pair: 0 = pair only when that makes the bank resident, 1 = always pair, 2 = never.
  bool found = false;
  const int kc_first = tune.kc ? tune.kc : pick_kc(a.cin_p);
  const bool pair_ok = p.cluster == 1 && e.mode != 2 && tune.halo_mode == 0 && (e.n_pad / 2) % 8 == 0 &&
                       a.cin_p % 16 == 0 && tune.pair != 2;
  auto set_pair = [&](int on) {
    p.pair = on;
    p.b_slice_rows = on ? e.n_pad / 2 : e.n_pad / p.cluster;
  };
  int want_rows = tune.rows;  // (the head's fused-row attempt below asks for four-row patches)
  auto rows_cap = [&](int acc_stages) {
    const int acc_stride = p.fuse_g ? e.n_pad : ((e.n_pad + 31) / 32) * 32;
    int rmax = 512 / (acc_stages * acc_stride);
    if (rmax > 4) rmax = 4;
    if (rmax > e.H) rmax = e.H;
    if (p.pair && rmax > 2) rmax = 2;  // pair kernels are instantiated for one and two accumulator rows
    if (want_rows) rmax = want_rows;
    return rmax;
  };
  // epilogue warps: eight (two per TMEM lane quarter) unless their staging does not fit beside the operand rings
  const int ew_first = tune.epi_warps ? tune.epi_warps : 8, ew_last = tune.epi_warps ? tune.epi_warps : 4;
  auto try_resident = [&]() {
    if (tune.resident == 2 || p.cluster != 1 || tune.halo_mode != 0 || !(tune.acc_stages == 0 || tune.acc_stages == 2))
      return;
    const int rcap = rows_cap(2);
    const int rmin = (rcap >= 2 && !want_rows) ? 2 : 1;  // a one-row patch reads every activation row three times
    // ONE-ROW patches (the 96-channel conv1: TMEM holds one 192-column row per stage): a third activation stage beats
    // wider K chunks and a second set of epilogue warps -- one K chunk of a one-row patch is ~0.55 us of UMMAs against
    // ~1 us of TMA latency, so with two stages the tensor pipe waits for loads (15.23 -> 14.9 ms per 4X-Ctrl frame).  Pass
    // 0 of such a search only accepts the deepest activation ring, over every K chunk and warp count; pass 1 takes whatever
    // fits.  Patches of two rows have twice the work per chunk and prefer the eight epilogue warps (3X-Ctrl: 8.5 vs 9.4 ms).
    const bool stages_first = rcap == 1;
    for (int outer = 0; outer < (stages_first ? 2 : 1) && !found; ++outer) {
      for (int kc = kc_first; kc >= 16 && !found; kc >>= 1) {  // wide K chunks first: fewer hand-offs per patch
        const int as_first = tune.a_stages ? tune.a_stages : 3;
        for (int ew = ew_first; ew >= ew_last && !found; ew -= 4) {
          p.epi_warps = ew;
          for (int rows = rcap; rows >= rmin && !found; --rows) {
            if (rows == 3) continue;
            for (int as = as_first; as >= 2 && !found; --as) {
              if (stages_first && outer == 0 && as != as_first) break;
              for (int staging = 2; staging >= (stages_first && e.mode == 0 ? -1 : 0) && !found; --staging) {
                fill_geometry(p, a.cin_p, kc, rows, 2, 0, as, 0, staging, true);
                if (fits(p)) found = true;
              }
              if (tune.a_stages) break;
            }
            if (want_rows) break;
          }
        }
        if (tune.kc) break;
      }
    }
  };
  auto try_stream = [&]() {
    for (int acc_stages = tune.acc_stages ? tune.acc_stages : 2; acc_stages >= 1 && !found; --acc_stages) {
      const int rmax = rows_cap(acc_stages);
      for (int rows = rmax; rows >= 1 && !found; --rows) {
        if (rows == 3) continue;  // instantiated for 1, 2 and 4 accumulator rows
        for (int kc = kc_first; kc >= 16 && !found; kc >>= 1) {
          for (int ew = ew_first; ew >= ew_last && !found; ew -= 4) {
            p.epi_warps = ew;
            for (int bs = tune.b_stages ? tune.b_stages : 4; bs >= 2 && !found; --bs) {
              // deeper epilogue staging (more TMA stores / residual loads in flight) when shared memory allows
              // (measured on the 96-channel conv2: three activation stages beat deeper epilogue staging and a fifth
              // weight stage; the pair's halved weight stages make room for them)
              for (int as = tune.a_stages ? tune.a_stages : 3; as >= 2 && !found; --as) {
                for (int staging = 2; staging >= 1 && !found; --staging) {
                  fill_geometry(p, a.cin_p, kc, rows, acc_stages, tune.halo_mode, as, bs, staging, false);
                  if (fits(p)) found = true;
                }
                if (tune.a_stages) break;
              }
              if (tune.b_stages) break;
            }
          }
          if (tune.kc) break;
        }
        if (want_rows) break;
      }
      if (tune.acc_stages) break;
    }
  };
  // filter rows fused along N (VAR 2): resident, un-paired encoder convolutions whose stacked taps fit one UMMA
  const int fuse_g = (256 / e.n_pad) >= 3 ? 3 : (256 / e.n_pad);
  // Automatic with three stacked taps (N <= 85: the 48-channel conv2, -19 % tensor-only time, -3.5 % on the whole 2X-Ctrl
  // step); with two (N = 96 | 128) the 2N-wide windows measured slower than they save: opt-in (tune.fuse = 1) only.
  // The head (mode 2, N = 16 / 32 / 48: every UMMA re-fetches its 4 KB activation tile for a few output columns) stacks
  // its taps too, in four-row patches (six UMMAs per filter column and k-step instead of twelve).
  const bool head_fuse = e.mode == 2 && tune.fuse != 2 && e.H >= 4 && (tune.rows == 0 || tune.rows == 4);
  const bool fuse_ok = (e.mode != 2 || head_fuse) && tune.fuse != 2 && (fuse_g >= 3 || (tune.fuse == 1 && fuse_g >= 2)) &&
                       e.H >= 2 && (tune.rows == 0 || tune.rows >= 2) && tune.pair != 1;
  if (tune.pair == 1 && pair_ok) {
    set_pair(1);
    try_resident();
  } else {
    set_pair(0);
    if (fuse_ok) {
      p.fuse_g = fuse_g;
      if (e.mode == 2) want_rows = 4;
      try_resident();
      want_rows = tune.rows;
      if (found && p.rows < (e.mode == 2 ? 4 : 2)) found = false;
      if (!found) p.fuse_g = 0;
    }
    if (!found && tune.fuse == 1) {
      set_error("conv: the fused-row kernel does not apply (cin_p %d, n_pad %d)", a.cin_p, e.n_pad);
      return MZ_ERR_UNSUPPORTED;
    }
    if (!found) try_resident();
    if (!found && pair_ok && tune.pair == 0) {
      set_pair(1);
      try_resident();
      if (!found) set_pair(0);
    }
  }
  if (!found && tune.resident == 1) {
    set_error("conv: the filter bank (cin_p %d, n_pad %d) does not fit resident in shared memory", a.cin_p, e.n_pad);
    return MZ_ERR_UNSUPPORTED;
  }
  if (!found && pair_ok && tune.pair == 0 && e.mode != 0 && a.cin_p >= 128) {
    // streamed weights: the pair halves every CTA's weight stream and leaves room for a third activation stage
    // (96-channel conv2: 181 vs 199 us)
    set_pair(1);
    try_stream();
    if (found && (p.a_stages < 3 || p.kc < 32)) found = false;
    if (!found) set_pair(0);
  }
  if (!found) try_stream();
  if (!found) {
    set_error("conv: no tcgen05 configuration fits (cin_p %d, n_pad %d, rows %d, acc_stages %d, kc %d, halo_mode %d)",
              a.cin_p, e.n_pad, tune.rows, tune.acc_stages, tune.kc, tune.halo_mode);
    return MZ_ERR_UNSUPPORTED;
  }

  // k-steps over zero padding at the end of K (a.k_valid: the input channels that can be non-zero): not issued for the
  // last chunk of a resident, un-fused bank (what the 54-channel model's conv2 runs: K = 108 -> 128, seven of eight)
  p.kt_last = p.subs > 1 ? p.subs : p.kc / 16;  // (= the kernel's KT: every k-step)
  {
    const int kv = a.k_valid ? a.k_valid : a.cin_p;
    MZ_REQUIRE(kv > 0 && kv <= a.cin_p, "conv: k_valid %d outside (0, %d]", kv, a.cin_p);
    const bool no_kskip = getenv("MZ_NO_KSKIP") != nullptr;  // (diagnostic; read per prepared launch)
    const int dead = (a.cin_p - kv) / 16;  // whole k-steps of zeros
    if (!no_kskip && p.res_b && !p.fuse_g && p.subs == 1 && dead > 0 && dead < p.kc / 16) p.kt_last = p.kc / 16 - dead;
  }
  p.tiles_x = ceil_div(e.W, kTileW);
  p.tiles_y = ceil_div(e.H, p.rows);
  const long long n_units = static_cast<long long>(e.B) * p.tiles_x * p.tiles_y;
  MZ_REQUIRE(n_units < (1LL << 31), "conv: too many patches (%lld)", n_units);
  p.n_units = static_cast<int>(n_units);
  const int mma_m = p.pair ? 256 : 128;
  p.idesc = e.bf16 ? umma_idesc_bf16(mma_m, e.n_pad) : umma_idesc_f16(mma_m, e.n_pad);
  for (int k = 1; k <= 3; ++k) {
    const int nw = k * e.n_pad <= 256 ? k * e.n_pad : e.n_pad;
    p.idesc_w[k - 1] = e.bf16 ? umma_idesc_bf16(128, nw) : umma_idesc_f16(128, nw);
  }
  const CUtensorMapDataType tdt = e.bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;

  const CUtensorMapSwizzle swz =
      p.kc == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (p.kc == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  {
    const uint64_t dims[4] = {static_cast<uint64_t>(a.in_extent ? a.in_extent : a.cin_p), static_cast<uint64_t>(e.W),
                              static_cast<uint64_t>(e.H), static_cast<uint64_t>(e.B)};
    const uint64_t ip = a.in_pitch ? a.in_pitch : a.cin_p;  // pixel pitch in elements (a wider tensor's first cin_p channels)
    const uint64_t strides[3] = {ip * 2, static_cast<uint64_t>(e.W) * ip * 2, static_cast<uint64_t>(e.H) * e.W * ip * 2};
    const uint32_t box[4] = {static_cast<uint32_t>(p.kc), static_cast<uint32_t>(p.pw),
                             static_cast<uint32_t>(p.rows + 2), 1u};
    int rc = encode_tmap(&p.tmA, tdt, 4, const_cast<uint16_t*>(a.in), dims, strides, box, swz);
    if (rc != MZ_OK) return rc;
  }
  {
    const uint64_t dims[3] = {static_cast<uint64_t>(a.cin_p), static_cast<uint64_t>(e.n_pad), 9};
    const uint64_t strides[2] = {static_cast<uint64_t>(a.cin_p) * 2, static_cast<uint64_t>(e.n_pad) * a.cin_p * 2};
    const uint32_t box[3] = {static_cast<uint32_t>(p.kc), static_cast<uint32_t>(p.b_slice_rows),
                             (p.cluster > 1 || p.fuse_g) ? 1u : 3u};  // pair: this CTA's N/2 rows of all three taps
    int rc = encode_tmap(&p.tmB, tdt, 3, const_cast<uint16_t*>(a.w), dims, strides, box, swz);
    if (rc != MZ_OK) return rc;
  }

  auto swz_of = [](int row_bytes) {
    return row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                            : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  };
  if (e.mode != 2) {
    uint64_t dims[4] = {static_cast<uint64_t>(e.out_extent ? e.out_extent : e.n_pad), static_cast<uint64_t>(e.W),
                        static_cast<uint64_t>(e.H), static_cast<uint64_t>(e.B)};
    const uint64_t op = e.out_pitch ? e.out_pitch : e.n_pad;
    const uint64_t st16[3] = {op * 2, static_cast<uint64_t>(e.W) * op * 2, static_cast<uint64_t>(e.H) * e.W * op * 2};
    const uint32_t box16[4] = {static_cast<uint32_t>(p.e16), 32u, 1u, 1u};
    int rc = encode_tmap(&p.tmO, tdt, 4, e.out_bf16, dims, st16, box16, swz_of(p.e16 * 2));
    if (rc != MZ_OK) return rc;
    if (e.mode == 1) {
      const uint64_t zp = e.zf_pitch ? e.zf_pitch : e.n_pad;
      const uint64_t st32[3] = {zp * 4, static_cast<uint64_t>(e.W) * zp * 4, static_cast<uint64_t>(e.H) * e.W * zp * 4};
      const uint32_t box32[4] = {static_cast<uint32_t>(p.e32), 32u, 1u, 1u};
      dims[0] = static_cast<uint64_t>(e.zf_extent ? e.zf_extent : e.n_pad);
      rc = encode_tmap(&p.tmZ, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, e.zf, dims, st32, box32, swz_of(p.e32 * 4));
      if (rc != MZ_OK) return rc;
    }
  }

  const uint32_t smem = plan_smem(p).total + 1024;
  int sms = sm_count(device);
  if (sms <= 0) sms = 148;
  const int k = p.pair ? 2 : p.cluster;
  int grid = p.n_units < sms ? p.n_units : sms;
  if (tune.max_ctas > 0 && grid > tune.max_ctas) grid = tune.max_ctas;
  grid = ceil_div(grid, k) * k;  // whole clusters (surplus CTAs recompute the last patch without storing)
  if (grid > sms) grid = (sms / k) * k;
  p.n_rounds = ceil_div(p.n_units, grid);

  {
    static const bool verbose = getenv("MZ_VERBOSE") != nullptr;
    if (verbose)
      fprintf(stderr,
              "[mz conv] mode %d cin_p %d n %d | rows %d kc %d subs %d chunks %d a_stages %d b_stages %d resident %d pair %d "
              "fuse %d cluster %d epi_warps %d o_ring %d res_rows %d e16 %d e32 %d acc_stages %d smem %u grid %d rounds %d\n",
              e.mode, a.cin_p, e.n_pad, p.rows, p.kc, p.subs, p.n_chunks, p.a_stages, p.b_stages, p.res_b, p.pair,
              p.fuse_g, p.cluster, p.epi_warps, p.o_ring, p.res_rows, p.e16, p.e32, p.acc_stages, smem, grid, p.n_rounds);
  }
  const int ks = p.subs > 1 ? p.subs : p.kc / 16;  // k-steps per stage and tap
  MZ_REQUIRE(p.a_stages >= 2 && p.b_stages >= 2, "conv: the look-ahead issue loop needs at least two A and two B stages");
  const int var = p.fuse_g ? 2 : (p.pair ? 1 : 0);
  const void* fn = e.mode == 0   ? tc_kernel_mode0(ks, p.rows, var)
                   : e.mode == 1 ? tc_kernel_mode1(ks, p.rows, var)
                                 : tc_kernel_head(head_layout(e), ks, p.rows, var);
  if (!fn) {
    set_error("conv: no %s kernel for mode %d, %d k-steps, %d rows", var == 2 ? "fused-row" : (var == 1 ? "CTA-pair" : "tcgen05"),
              e.mode, ks, p.rows);
    return MZ_ERR_UNSUPPORTED;
  }
  // (records the instantiation; run_prepared launches it)
  MZ_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
  L.fn = fn;
  L.grid = grid;
  L.k = k;
  L.smem = smem;
  L.mode = e.mode;
  L.n_pad = e.n_pad;
  L.ks = ks;
  L.var = var;
  L.lay = e.mode == 2 ? head_layout(e) : 0;
  out->valid = true;
  return MZ_OK;
}

#endif  // host side

}  // namespace mz
