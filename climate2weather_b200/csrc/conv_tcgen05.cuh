// K1 — implicit-GEMM 3x3 convolution / plain GEMM on tcgen05 tensor cores (sm_100a).
//
// Computes every Conv2d of the reference UNet (model/nn.py:155,157,169,185,193,194) and the
// attention 1x1 Conv1d (model/nn.py:45,47) as  D[M, N] = A[M, K] * B[N, K]^T  with
//   M = pixels (n, h, w flattened, NHWC activations, bf16),
//   N = output channels, K = taps * Cin  (k index = (r*3 + s) * Cin + c).
//
// Feeding:   A is never materialised.  Generic path: for filter tap (r, s) the 128-pixel A tile (whole output rows,
//            or one 128-pixel segment of a row wider than 128) is a SHIFTED BOX of the NHWC input: one 4-D TMA load
//            {64 ch, W or 128, tile_h, tile_n} at (c0, w0+s-1, h0+r-1, n0); out-of-bounds rows/columns are zero-filled by the TMA unit, which is exactly
//            padding=1 / padding_mode=zeros (configs/sda_unet.yml:16).  Stride-2 convs use the same box with element
//            strides {1, 2, 2, 1}.  Activation-reuse path (AR; stride-1 convs with 64/128-wide N tiles): the M tile is
//            a 16 x 8 spatial block and ONE halo'd box [18 rows x 10 px][64 ch] per channel block serves all nine
//            taps: tap (r, s) is the sub-view r rows and s pixels into it, addressed by the MMA descriptor alone.
//            B (packed weights [Cout, 9*Cin], K-major) is a 2-D TMA load {64, BN} (AR: one box holds the three
//            filter rows' tiles of one filter column).
//            Both land in 128B-swizzled K-major tiles that tcgen05.mma consumes directly.
// Roles:     warp 0 = TMA producer, warp 1 = MMA issuer (single thread), warp 2 = TMEM allocator + TMA stores of the
//            finished tiles + residual prefetch, warps 4..11 = epilogue, warps 12..15 (fused-LayerNorm kernels only)
//            = LayerNorm pass; the register file is re-split per warpgroup with setmaxnreg in those kernels.
//            Persistent CTAs (grid = #SMs, static round-robin tiles), a ring of operand stages (full/empty
//            mbarriers; AR: a ring of activation units and a ring of weight stages), two TMEM accumulators
//            (tmem_full/tmem_empty; released as soon as the epilogue's tcgen05.ld have landed), staging tiles handed
//            between epilogue, LayerNorm and store warps by mbarriers only.
//            Two CTAs (a cluster) share one MMA (cta_group::2, 256 x BN tile) whenever there are two M tiles.
// Epilogue:  TMEM -> registers (tcgen05.ld 32x32b.x32) -> +bias [-> SiLU | + residual] -> bf16 -> 128B-swizzled
//            staging tile in shared memory -> TMA store (per-thread row stores cost 8x the L1 wavefronts of the
//            staged path, profiles/r01a_ncu_conv_G2.csv).  The residual tile is TMA-prefetched into the staging tile;
//            the fused channel LayerNorm re-reads the staged rows and writes a second tensor with coalesced stores.
//            The last conv of the UNet (64-wide tile) writes fp32 / the fused window compose
//            (src/thor/score.py:76-88,111-141) straight from registers.
// What bounds it (profiles/r01d_k1_role_cycles.log, r01e_ncu_conv_G2.csv): L2 -> SM TMA throughput with streamed
//            operands; with activation reuse the operand-ring depth (TMA latency) and the SM's L1/shared-memory
//            data pipe (tensor-core operand reads + TMA writes + epilogue traffic).
#pragma once
#include <cuda_bf16.h>
#include <stdio.h>

#include "c2w_ptx.cuh"

namespace c2w {

// Diagnostics (per-role cycle counters, load-skipping timing experiments) exist only in builds with -DC2W_DIAG
// (`python -m climate2weather_b200.build --diag` -> libc2w_b200_diag.so, used by tools/bringup_conv.py).  The shipped
// library carries none of it: no clock64() around the barrier waits, no dbg_* branches in the producer.
#ifdef C2W_DIAG
#define C2W_TIMED_WAIT(ACC, BAR, PARITY) \
  do {                                   \
    const long long t0_ = clock64();     \
    mbar_wait(BAR, PARITY);              \
    (ACC) += clock64() - t0_;            \
  } while (0)
#define C2W_DIAG_CLOCK() clock64()
#else
#define C2W_TIMED_WAIT(ACC, BAR, PARITY) mbar_wait(BAR, PARITY)
#define C2W_DIAG_CLOCK() 0ll
#endif

enum EpiMode : int {
  EPI_BIAS = 0,       // out = acc + bias                       -> bf16
  EPI_BIAS_SILU = 1,  // out = silu(acc + bias)                 -> bf16
  EPI_BIAS_RES = 2,   // out += acc + bias                      -> bf16   (in place)
  EPI_COMPOSE = 3,    // centre-pick / edge-fill compose        -> fp32 eps [L, H, W, 4]
  EPI_F32 = 4,        // out = acc + bias                       -> fp32 [M, ldc]
  EPI_MUL_DSILU = 5,  // out = (acc + bias) * silu'(out)        -> bf16   (in place: `out` holds the pre-activation)
  EPI_BIAS_SILU_DUAL = 6,  // out = acc + bias AND out2 = silu(acc + bias) -> two bf16 tensors (stashing forward: the
                           // backward needs the pre-activation, the next conv its SiLU; BN <= 128)
};

struct ConvParams {
  // main loop
  int taps;        // 9: 3x3 pad 1 (stride 1 or 2) on NHWC input; 1: A is a plain [M, K] matrix
  int stride;      // taps == 9: input pixel = stride * output pixel + tap - 1
  int cin_blocks;  // Cin / 64
  int num_m_tiles, num_n_tiles;
  int m_total;  // valid rows
  int tile_h, tile_n, tiles_per_img;
  int tiles_w;      // AR: 16 x 8 spatial tiles per image row (W / 8); tiles_per_img = (H / 16) * tiles_w
  int img_h, img_w; // AR: output image size
  // AR on 8-row images (ar2): the 16 x 8 M tile is two images stacked row-interleaved — tile row = (image row, image,
  // pixel) — so that tap (r, s) is still one strided sub-view of the halo'd unit ([10 rows][2 img][10 px][64 ch],
  // 25 KB): the tensor maps list the image dimension BEFORE the row dimension.  tiles_per_img = tiles per image pair.
  int ar2;
  int ar_row_step16;  // (bytes >> 4) from filter row r to r + 1 inside the unit: 80 (ar2: 160)
  int ar_tx_a;        // bytes one CTA's activation unit delivers
  int ar_tx_b;        // bytes one CTA's three weight tiles of a filter column deliver
  int num_stages;   // depth of the A/B ring (AR: of the weight ring)
  int num_staging;  // epilogue staging tiles (2: used alternately)
  // epilogue
  int mode;
  int ldc;  // output row pitch (elements)
  const float* bias;
  float* out_f32;
  // fused channel LayerNorm of the output row (model/nn.py:154,183; needs one N tile = all channels):
  //   ln_out[pixel] = (v - mean_C v) / sqrt(var_C v + eps),  v = bf16(out) + ln_mod, unbiased variance;
  //   ln_up: every pixel is written to its 2x2 nearest-neighbour block of a [n, 2H, 2W, C] tensor (model/nn.py:184)
  __nv_bfloat16* ln_out;
  float* ln_inv;  // optional: 1 / sqrt(var + eps) per row (stash for the LayerNorm backward)
  const float* ln_mod;
  int ln_mod_stride;  // 0: one modulation vector for the batch; else floats between consecutive IMAGES' vectors (one
                      // diffusion time per sample, training) — needs tiles that lie inside one image
  int ln_up, ln_H, ln_W;  // ln_H x ln_W: output image of this conv (for the upsampled addressing)
  float ln_eps;
  // EPI_COMPOSE
  float* eps;       // [local frames, H, W, 4] fp32
  int hw;           // H*W
  int order_k;      // Markov order k (window = 2k+1)
  int win_first;    // global index of the first window of this launch
  int win_last_global;  // global index of the last window of the trajectory (Nw - 1)
  int frame_base;   // global frame index of eps[0]
  const int* win_list;  // global window index per image of this launch (a selection), or null: win_first + image
  long long* dbg_timeline;  // diagnostics only (-DC2W_DIAG): [2] = {min over CTAs of the start, max of the end} in
                            // %globaltimer ns for THIS launch (tools/timeline.py: kernel-inside time vs gaps)
  long long* dbg_stats;  // diagnostics only: per-CTA wait cycles [grid][12] (see tools/bringup_conv.py --stats)
  int dbg_skip_loads;  // diagnostics only: after the ring is primed, signal `full` without issuing TMA loads
  // EPI_COMPOSE over an ensemble stored member-major (0: one trajectory): windows per member Nw.  Window G is window
  // G mod Nw of member G div Nw, whose frames start at frame G + 2k (G div Nw); head / tail tests are member-local.
  // Last, in the struct's tail padding, so that the fields above keep their offsets.
  int member_win;
  // Streamed 3x3 main loop: 128-pixel segments per output row (1: tiles of whole rows; Wo / 128 when Wo > 128)
  int row_segs;
};

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;
constexpr int kATileBytes = kBlockM * kBlockK * 2;  // 16 KB
constexpr int kEpiWarps = 8;                        // two warps per TMEM lane quarter, each half of the columns
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kConvThreads = 128 + kEpiThreads;  // + kLnThreads in kernels with the fused LayerNorm
constexpr int kLnWarps = 4;                      // LayerNorm warps (one warpgroup) of those kernels
constexpr int kLnThreads = kLnWarps * 32;
constexpr int kSmemLimit = 232448;  // 227 KB
constexpr int kARUnitW = 10;        // AR: pixel columns of a unit (8 + the halo on either side)

// BN   : N tile (output channels per tile).
// CG   : CTAs per MMA (tcgen05 cta_group).  CG == 2: a cluster of two CTAs computes a 256 x BN tile, each CTA
//        holding its own 128 A rows and HALF of the B rows in shared memory.
// Shared memory: [A ring][B ring][1 or 2 staging tiles][barriers]; the ring depth is a launch-time number (what is
// left after the staging tiles: residual convs double-buffer them so the residual prefetch runs a tile ahead).  AR:
// [kARUnits activation units][weight stages of three B tiles][staging][barriers], the weight ring taking what is left.
template <int BN, int CG>
struct ConvCfg {
  // A pipeline stage holds kSub K-sub-blocks of 64 (one 128 B swizzle row each).  With BN <= 128 a 64-wide
  // sub-block is only 256 tensor-pipe cycles of work, less than one barrier round trip of the issuing thread,
  // so two sub-blocks share one full/empty barrier pair (measured both ways, profiles/).
  static constexpr int kSub = (BN > 128) ? 1 : 2;
  static constexpr int kBRows = BN / CG;                 // B rows held by one CTA
  static constexpr int kBTileBytes = kBRows * kBlockK * 2;
  static constexpr int kSubBytes = kATileBytes + kBTileBytes;
  static constexpr int kStageBytes = kSub * kSubBytes;
  static constexpr int kStagingBytes = (BN / 64) * kATileBytes;  // bf16 [BN/64 boxes][128 rows][64 ch], swizzled
  static constexpr int kBarrierBytes = 512 + 4096;  // mbarriers, TMEM slot; LN row statistics float2[2 tiles][2][128]
  static constexpr int kMaxStages = 8;
  // AR (activation reuse, 3x3 stride 1): the M tile is a 16 x 8 spatial block.  One UNIT per channel block holds the
  // block's input with a one-pixel halo on every side ([18 rows][10 px][64 ch] = 22.5 KB), loaded by one TMA box.
  // Tap (r, s) is the sub-view starting r rows and s pixels into it: an MMA descriptor whose start address is
  // r * 1280 + s * 128 bytes into the unit and whose 8-row groups (one tile row of 8 pixels each) are 1280 B apart.
  // So the unit is loaded once and multiplied nine times: 2.5 KB of A per K block instead of 16 KB.  The units have
  // their own ring; the weight ring holds, per stage, the three B tiles (r = 0..2) of one filter column s, loaded by
  // one TMA box too.
  // (K1 with streamed operands is bound by the chip-wide L2 -> SM TMA throughput, ~12 TB/s: profiles/r01c_*.)
  static constexpr int kARTileH = 16, kARTileW = 8;
  // unit slot, 1024-aligned: 23 KB; 25 KB for 128-wide tiles, which also run the two-image form (ConvParams::ar2)
  static constexpr int kARUnitBytes = ((BN == 128 ? 20 : 18) * kARUnitW * kBlockK * 2 + 1023) / 1024 * 1024;
  // units in flight (the weight ring takes what is left; 64-wide tiles, whose weight ring is at kMaxStages, take three)
  static constexpr int kARUnits = BN == 64 ? 3 : 2;
  static constexpr int kARBStageBytes = 3 * kBTileBytes;
  static constexpr int ar_stages_for(int num_staging) {
    const int n = (kSmemLimit - 1024 - kBarrierBytes - num_staging * kStagingBytes - kARUnits * kARUnitBytes) /
                  kARBStageBytes;
    return n > kMaxStages ? kMaxStages : n;
  }
  static constexpr int ar_smem_bytes(int num_staging) {
    return kARUnits * kARUnitBytes + ar_stages_for(num_staging) * kARBStageBytes + num_staging * kStagingBytes +
           kBarrierBytes + 1024;
  }
  static constexpr int kTmemCols = (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  static constexpr int stages_for(int num_staging) {
    const int n = (kSmemLimit - 1024 - kBarrierBytes - num_staging * kStagingBytes) / kStageBytes;
    return n > kMaxStages ? kMaxStages : n;
  }
  static constexpr int smem_bytes(int num_staging) {
    return stages_for(num_staging) * kStageBytes + num_staging * kStagingBytes + kBarrierBytes + 1024;
  }
  static_assert(BN % 64 == 0 && BN >= 64 && BN <= 256, "BN must be 64..256, multiple of 64");
  static_assert(CG == 1 || CG == 2, "cta_group is 1 or 2");
  static_assert(stages_for(2) >= 1 && stages_for(1) >= 2, "pipeline too shallow");
  static_assert(2 * kMaxStages + 2 * kARUnits + 10 <= 512 / 8 - 1, "barrier block too small");
};

// SiLU = x * sigmoid(x) = h + h * tanh(h), h = x / 2: one MUFU op per element (tanh.approx, rel. error 2^-11, far
// below the bf16 output rounding) instead of ex2 + rcp — the epilogue's SFU budget is 16 ops/clk/SM.
__device__ __forceinline__ float silu_f(float x) {
  const float h = 0.5f * x;
  return fmaf(h, tanh_approx(h), h);
}

// Direct-to-global epilogue of one 32-column chunk of one accumulator row (final conv only: fp32 / compose).
__device__ __forceinline__ void epilogue_chunk_direct(const ConvParams& p, const uint32_t (&v)[32], int col0, int m,
                                                      bool valid) {
  float f[32];
  const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 b = __ldg(b4 + i);
    f[4 * i + 0] = __uint_as_float(v[4 * i + 0]) + b.x;
    f[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b.y;
    f[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b.z;
    f[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b.w;
  }
  if (!valid) return;
  if (p.mode == EPI_COMPOSE) {
    const int n_img = m / p.hw;
    const int pix = m - n_img * p.hw;
    const int win = p.win_list ? __ldg(p.win_list + n_img) : p.win_first + n_img;
    int j = win, last = p.win_last_global, f0 = win - p.frame_base;  // window within its member, its first frame
    if (p.member_win > 0) {
      const int m = win / p.member_win;
      j = win - m * p.member_win;
      last = p.member_win - 1;
      f0 += 2 * p.order_k * m;
    }
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const int tau = (col0 >> 2) + g;  // window slot of channels [4*tau, 4*tau+4)
      const bool take = (tau == p.order_k) || (j == 0 && tau < p.order_k) ||
                        (j == last && tau > p.order_k && tau <= 2 * p.order_k);
      if (take) {
        const long long fl = static_cast<long long>(f0 + tau);
        float4 o = make_float4(f[4 * g], f[4 * g + 1], f[4 * g + 2], f[4 * g + 3]);
        *reinterpret_cast<float4*>(p.eps + (fl * p.hw + pix) * 4) = o;
      }
    }
  } else {
    float4* o4 = reinterpret_cast<float4*>(p.out_f32 + static_cast<size_t>(m) * p.ldc + col0);
#pragma unroll
    for (int i = 0; i < 8; ++i) o4[i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
  }
}

// Staged epilogue of one 32-column chunk: bf16 result into the 128B-swizzled staging tile, in place over the
// TMA-prefetched residual tile in EPI_BIAS_RES.  `stg_row` = this row in box 0 of the tile.  LN: also accumulates the
// row's LayerNorm statistics (sums of v = out + mod and v^2 over this thread's columns).
// (Packed fp32 pairs — FADD2 / FFMA2 via __fadd2_rn / __ffma2_rn — were tried for this function: 5 % fewer SASS
// instructions, no measurable change: the epilogue is bound by latency, not by issue slots.)
template <bool LN>
__device__ __forceinline__ void epilogue_chunk_staged(const ConvParams& p, const uint32_t (&v)[32], int gcol, int col,
                                                      uint8_t* stg_row, int row, float& s1, float& s2,
                                                      const float* ln_mod, uint32_t dual_off = 0) {
  float f[32];
  const float4* b4 = reinterpret_cast<const float4*>(p.bias + gcol);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 b = __ldg(b4 + i);
    f[4 * i + 0] = __uint_as_float(v[4 * i + 0]) + b.x;
    f[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b.y;
    f[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b.z;
    f[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b.w;
  }
  const uint32_t boff = static_cast<uint32_t>(col >> 6) * kATileBytes;
  const int j0 = (col & 63) >> 3;  // first 16 B chunk of this 32-column group inside the 128 B row
  if (p.mode == EPI_BIAS_SILU) {
#pragma unroll
    for (int i = 0; i < 32; ++i) f[i] = silu_f(f[i]);
  } else if (p.mode == EPI_BIAS_SILU_DUAL) {
    // second staging tile (dual_off bytes further on): silu of the same values; the pre-activation goes out below
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        __nv_bfloat162 h = __floats2bfloat162_rn(silu_f(f[8 * i + 2 * j]), silu_f(f[8 * i + 2 * j + 1]));
        o[j] = *reinterpret_cast<uint32_t*>(&h);
      }
      st_shared_v4(stg_row, dual_off + boff + (static_cast<uint32_t>((j0 + i) ^ (row & 7)) << 4), o[0], o[1], o[2], o[3]);
    }
  } else if (p.mode == EPI_BIAS_RES) {
    // all residual loads of the chunk first: the in-place stores below alias them as far as the compiler can tell
    uint4 aux[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) aux[i] = ld_shared_v4(stg_row, boff + (static_cast<uint32_t>((j0 + i) ^ (row & 7)) << 4));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t w[4] = {aux[i].x, aux[i].y, aux[i].z, aux[i].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
        f[8 * i + 2 * j] += __low2float(h);
        f[8 * i + 2 * j + 1] += __high2float(h);
      }
    }
  } else if (p.mode == EPI_MUL_DSILU) {
    // input-gradient pass: the staging tile holds the forward pre-activation x; g *= silu'(x) with
    // silu'(x) = s (1 + x (1 - s)), s = sigmoid(x) = 1/2 + 1/2 tanh(x / 2)
    uint4 aux[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) aux[i] = ld_shared_v4(stg_row, boff + (static_cast<uint32_t>((j0 + i) ^ (row & 7)) << 4));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t w[4] = {aux[i].x, aux[i].y, aux[i].z, aux[i].w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
        const float x0 = __low2float(h), x1 = __high2float(h);
        const float s0 = fmaf(0.5f, tanh_approx(0.5f * x0), 0.5f), s1 = fmaf(0.5f, tanh_approx(0.5f * x1), 0.5f);
        f[8 * i + 2 * j] *= s0 * fmaf(x0, 1.0f - s0, 1.0f);
        f[8 * i + 2 * j + 1] *= s1 * fmaf(x1, 1.0f - s1, 1.0f);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      __nv_bfloat162 h = __floats2bfloat162_rn(f[8 * i + 2 * j], f[8 * i + 2 * j + 1]);
      o[j] = *reinterpret_cast<uint32_t*>(&h);
    }
    st_shared_v4(stg_row, boff + (static_cast<uint32_t>((j0 + i) ^ (row & 7)) << 4), o[0], o[1], o[2], o[3]);
  }
  if (LN) {
    float sa[4] = {0.f, 0.f, 0.f, 0.f}, sb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float4 mv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ln_mod) mv = __ldg(reinterpret_cast<const float4*>(ln_mod + gcol) + i);
      const float mm[4] = {mv.x, mv.y, mv.z, mv.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float vv = f[4 * i + e] + mm[e];
        sa[e] += vv;
        sb[e] = fmaf(vv, vv, sb[e]);
      }
    }
    s1 += (sa[0] + sa[1]) + (sa[2] + sa[3]);
    s2 += (sb[0] + sb[1]) + (sb[2] + sb[3]);
  }
}

// Phase form (PH) of the activation-reuse kernels: the conv3x3 of a nearest x2 upsampled input (the ascent tails,
// model/nn.py:184-185) computed at the LOW resolution.  Output pixel (2i + a, 2j + b) reads upsampled rows 2i + a - 1
// .. 2i + a + 1, i.e. low-res rows {i - 1, i} (a = 0) or {i, i + 1} (a = 1), and the same for columns: so each output
// phase (a, b) is an exact 2x2 conv of the low-res input with merged weights (conv_pack_phase_weights), 16 instead of
// 36 tap-MACs per low-res pixel, and the upsampled input is never written.  The M tile is a 16 x 8 block of low-res
// pixels and one phase; its taps (tr, ts) are the sub-views a + tr rows and b + ts pixels into the same halo'd unit.
// The two CTAs of a pair share the weights, hence the phase: M tile mt -> pair g = mt / 2, phase g % 4, low-res tile
// 2 (g / 4) + mt % 2 (the four phases of a low-res pair run back to back and find its input in L2).
__device__ __forceinline__ int ph_split(int mt, int& phase) {
  const int g = mt >> 1;
  phase = g & 3;
  return ((g >> 2) << 1) | (mt & 1);
}

template <int BN, int CG, bool LN, bool AR, bool PH = false>
__global__ void __launch_bounds__(kConvThreads + (LN ? kLnThreads : 0), 1)
conv_gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ CUtensorMap tmOut2,
                         const ConvParams p) {
  using Cfg = ConvCfg<BN, CG>;
  static_assert(!PH || (AR && CG == 2), "the phase form is an activation-reuse main loop of a CTA pair");
  constexpr int kCols = PH ? 2 : 3;  // filter columns (= rows) of the main loop: 2x2 phase taps or 3x3
  extern __shared__ uint8_t smem_raw[];
  // 1024 B alignment by POINTER arithmetic (an integer round trip hides the address space from the compiler and
  // every staging-tile access becomes a generic LD/ST with 64-bit address math instead of LDS/STS)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int num_stages = p.num_stages;
  constexpr int num_units = AR ? Cfg::kARUnits : 0;
  // AR: [A units][B stages of [r0][r1][r2]]; otherwise [A ring][B ring]
  uint8_t* smA = smem;
  uint8_t* smB = smem + (AR ? num_units * Cfg::kARUnitBytes : num_stages * Cfg::kSub * kATileBytes);
  uint8_t* stg0 = smB + num_stages * (AR ? Cfg::kARBStageBytes : Cfg::kSub * Cfg::kBTileBytes);  // staging tile(s)
  uint64_t* bars = reinterpret_cast<uint64_t*>(stg0 + p.num_staging * Cfg::kStagingBytes);
  uint64_t* full = bars;  // [kMaxStages] operand stage landed (AR: weight stage)
  uint64_t* empty = bars + Cfg::kMaxStages;
  uint64_t* tmem_full = bars + 2 * Cfg::kMaxStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* res_full = tmem_empty + 2;  // [2] auxiliary tile landed in staging[b]
  uint64_t* stg_full = res_full + 2;    // [2] staging[b] written by the epilogue warps
  uint64_t* stg_free = stg_full + 2;    // [2] staging[b] read by its store (and the LayerNorm pass)
  uint64_t* ln_done = stg_free + 2;     // [2] LayerNorm pass over staging[b] finished (all epilogue warps)
  uint64_t* a_full = ln_done + 2;       // [kARUnits] AR: activation unit landed
  uint64_t* a_empty = a_full + Cfg::kARUnits;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_empty + Cfg::kARUnits);
  float2* ln_stats = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(bars) + 512);  // [2][2][128]

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;  // 0 = leader: arms the full barriers, issues the MMAs
  const int group_id = blockIdx.x / CG;
  const int num_groups = gridDim.x / CG;
  const int num_tiles = ((p.num_m_tiles + CG - 1) / CG) * p.num_n_tiles;
  const int num_kb = p.taps * p.cin_blocks;
  // direct (fp32 / compose) epilogues exist for the 64-wide tile only: the last conv of the UNet
  const bool staged = BN != 64 || (p.mode != EPI_COMPOSE && p.mode != EPI_F32);
  // TMA-prefetched auxiliary tile (the residual / the pre-activation the gradient is multiplied with), overwritten in place
  const bool has_aux = p.mode == EPI_BIAS_RES || p.mode == EPI_MUL_DSILU;
  // two staging tiles used alternately (residual convs: the residual tile is prefetched two tiles ahead)
  // EPI_BIAS_SILU_DUAL fills BOTH staging tiles for every output tile (pre-activation and its SiLU) and stores them
  // through two tensor maps; the auxiliary-tile modes use the two tiles alternately
  const bool dual = p.mode == EPI_BIAS_SILU_DUAL;
  const bool two_bufs = p.num_staging == 2 && !dual;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (staged) tma_prefetch_desc(&tmOut);
    if (dual) tma_prefetch_desc(&tmOut2);
  }
  if (warp_idx == 1 && lane == 0) {
    for (int s = 0; s < num_stages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int u = 0; u < num_units; ++u) {
      mbar_init(&a_full[u], 1);
      mbar_init(&a_empty[u], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], kEpiWarps * CG);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&res_full[b], 1);
      mbar_init(&stg_full[b], kEpiWarps);
      mbar_init(&stg_free[b], 1);
      mbar_init(&ln_done[b], kLnWarps);
    }
    fence_mbar_init();
  }
  if (warp_idx == 2) {
    if (CG == 2) tmem_alloc_pair(tmem_slot, Cfg::kTmemCols);
    else tmem_alloc(tmem_slot, Cfg::kTmemCols);
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all();  // the peer's barriers must be initialised before remote arrives / TMA signals
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, tensor-map prefetch) touched only
  // this CTA's shared memory / TMEM and may run while the PREVIOUS kernel of the stream is still draining its last
  // tiles on other SMs.  launch_dependents lets the next kernel's CTAs be scheduled as SMs free up; wait blocks until
  // the previous grid has completed and its global writes are visible — every global read below comes after it.
  // (No-ops when the kernel was launched without the programmatic-serialization attribute.)
  griddep_launch_dependents();
  griddep_wait();
#ifdef C2W_DIAG
  if (p.dbg_timeline != nullptr && threadIdx.x == 0) {
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    atomicMin(reinterpret_cast<unsigned long long*>(p.dbg_timeline), now);
  }
#endif

  // Producer and MMA warps run CONVERGED (all 32 lanes wait on the barriers) and issue under elect_one():
  // operands stay warp-uniform, so ptxas keeps descriptors/coordinates in uniform registers instead of wrapping
  // every tcgen05/TMA instruction in an R2UR waterfall.
  // Roles by warpgroup.  Kernels with the fused LayerNorm run 16 warps (512 threads x 128 registers at launch) and
  // re-split the register file per warpgroup (setmaxnreg at the top of each warpgroup's code region): producer /
  // MMA / store warps 56, epilogue warps 168, LayerNorm warps 96.
  if (warp_idx < 4) {
    if constexpr (LN) asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (warp_idx == 0) {
      // ------------------------------------------------------------ TMA producer (every CTA loads its own rows)
      int stage = 0;
      uint32_t phase = 0;
      int issued = 0;
      int unit = 0;
      uint32_t a_phase = 0;
      int a_issued = 0;
      [[maybe_unused]] long long w_empty = 0;
      [[maybe_unused]] const long long t_begin = C2W_DIAG_CLOCK();
      for (int tile = group_id; AR && tile < num_tiles; tile += num_groups) {
        const int nt = tile % p.num_n_tiles;
        int mt = (tile / p.num_n_tiles) * CG + rank;
        int ph = 0;
        if (PH) mt = ph_split(mt, ph);
        const int img = mt / p.tiles_per_img, tt = mt % p.tiles_per_img;
        const int h0 = (tt / p.tiles_w) * Cfg::kARTileH, w0 = (tt % p.tiles_w) * Cfg::kARTileW;
        const int a2 = p.ar2 ? 2 * img : h0 - 1, a3 = p.ar2 ? -1 : img;
        for (int cb = 0; cb < p.cin_blocks; ++cb) {
          // ---- the channel block's halo'd unit
          C2W_TIMED_WAIT(w_empty, &a_empty[unit], a_phase ^ 1);
          if (elect_one()) {
            // timing experiments (diagnostics build): after the rings are primed, 4 and 1 signal the unit as landed
            // without loading it
#ifdef C2W_DIAG
            const bool skip_a = (p.dbg_skip_loads == 4 || p.dbg_skip_loads == 1) && a_issued >= num_units;
#else
            constexpr bool skip_a = false;
#endif
            if (rank == 0) mbar_arrive_expect_tx(&a_full[unit], skip_a ? 0 : CG * p.ar_tx_a);
            uint8_t* adst = smA + unit * Cfg::kARUnitBytes;
            if (skip_a) {
            } else if (CG == 2) {
              tma_load_4d_pair(&tmA, mapa_shared(smem_u32(&a_full[unit]), 0), adst, cb * kBlockK, w0 - 1, a2, a3);
            } else {
              tma_load_4d(&tmA, &a_full[unit], adst, cb * kBlockK, w0 - 1, a2, a3);
            }
          }
          __syncwarp();
          ++a_issued;
          if (++unit == num_units) {
            unit = 0;
            a_phase ^= 1;
          }
          // ---- the weights of filter columns s = 0..2 (PH: 0..1), one stage each
          for (int s3 = 0; s3 < kCols; ++s3) {
            C2W_TIMED_WAIT(w_empty, &empty[stage], phase ^ 1);
            if (elect_one()) {
#ifdef C2W_DIAG
              // 2: every other tile reuses stale weights — the operand traffic of a 256-row M tile sharing one B
              // load, without its data flow; 3 and 1: no weight loads at all
              const bool skip_b = ((p.dbg_skip_loads == 2 && ((tile / num_groups) & 1)) || p.dbg_skip_loads == 3 ||
                                   p.dbg_skip_loads == 1) &&
                                  issued >= num_stages;
#else
              constexpr bool skip_b = false;
#endif
              if (rank == 0) mbar_arrive_expect_tx(&full[stage], skip_b ? 0 : CG * p.ar_tx_b);
              // one box {64 ch, B rows, r = 0..2} at channel s * Cin + cb * 64 of the [Cout][r][s * Cin] weight view
              // (PH: {64 ch, B rows, r = 0..1, 1} of the [phase][Cout][r][s * Cin] view)
              uint8_t* bdst = smB + stage * Cfg::kARBStageBytes;
              const int kc = (s3 * p.cin_blocks + cb) * kBlockK;
              if (skip_b) {
              } else if (CG == 2) {
                tma_load_4d_pair(&tmB, mapa_shared(smem_u32(&full[stage]), 0), bdst, kc, nt * BN + rank * Cfg::kBRows,
                                 0, ph);
              } else {
                tma_load_4d(&tmB, &full[stage], bdst, kc, nt * BN, 0, 0);
              }
            }
            __syncwarp();
            ++issued;
            if (++stage == num_stages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
      for (int tile = group_id; !AR && tile < num_tiles; tile += num_groups) {
        const int nt = tile % p.num_n_tiles;
        const int mt = (tile / p.num_n_tiles) * CG + rank;
        int b1, b2, b3;
        if (p.taps == 9) {  // row segments (Wo > 128): tile = 128-pixel segment tt % row_segs of row tt / row_segs
          const int tt = mt % p.tiles_per_img;
          b1 = (tt % p.row_segs) * kBlockM * p.stride;
          b2 = (tt / p.row_segs) * p.tile_h * p.stride;
          b3 = (mt / p.tiles_per_img) * p.tile_n;
        } else {
          b1 = mt * kBlockM;
          b2 = 0;
          b3 = 0;
        }
        for (int kb = 0; kb < num_kb; kb += Cfg::kSub) {
          const int nsub = (num_kb - kb) < Cfg::kSub ? (num_kb - kb) : Cfg::kSub;
          C2W_TIMED_WAIT(w_empty, &empty[stage], phase ^ 1);
          if (elect_one()) {
            const uint32_t full_bar = (CG == 2) ? mapa_shared(smem_u32(&full[stage]), 0) : smem_u32(&full[stage]);
#ifdef C2W_DIAG
            if (p.dbg_skip_loads == 1 && issued >= num_stages) {
              if (rank == 0) mbar_arrive(&full[stage]);
            } else
#endif
            {
              if (rank == 0) mbar_arrive_expect_tx(&full[stage], CG * nsub * Cfg::kSubBytes);
              for (int sub = 0; sub < nsub; ++sub) {
                const int kk = kb + sub;
                const int tap = kk / p.cin_blocks;
                const int cb = kk - tap * p.cin_blocks;
                const int dr = (p.taps == 9) ? tap / 3 - 1 : 0;
                const int ds = (p.taps == 9) ? tap % 3 - 1 : 0;
                const int slot = stage * Cfg::kSub + sub;
                if (CG == 2) {
                  tma_load_4d_pair(&tmA, full_bar, smA + slot * kATileBytes, cb * kBlockK, b1 + ds, b2 + dr, b3);
                  tma_load_2d_pair(&tmB, full_bar, smB + slot * Cfg::kBTileBytes, kk * kBlockK,
                                   nt * BN + rank * Cfg::kBRows);
                } else {
                  tma_load_4d(&tmA, &full[stage], smA + slot * kATileBytes, cb * kBlockK, b1 + ds, b2 + dr, b3);
                  tma_load_2d(&tmB, &full[stage], smB + slot * Cfg::kBTileBytes, kk * kBlockK, nt * BN);
                }
              }
            }
          }
          __syncwarp();
          ++issued;
          if (++stage == num_stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
#ifdef C2W_DIAG
      if (p.dbg_stats && lane == 0) {
        p.dbg_stats[blockIdx.x * 12 + 0] = clock64() - t_begin;
        p.dbg_stats[blockIdx.x * 12 + 1] = w_empty;
      }
#endif
    } else if (warp_idx == 1 && rank == 0) {
      // ------------------------------------------------------------ MMA issuer (leader CTA, one elected lane issues)
      constexpr uint32_t idesc = umma_idesc_bf16(kBlockM * CG, BN);
      // AR: 8-row groups = tile rows of 8 pixels, one unit row (kARUnitW pixels) apart
      const uint64_t adesc0 = umma_desc_kmajor_sw128(smem_u32(smA), AR ? kARUnitW * 128 : 1024);
      const uint64_t bdesc0 = umma_desc_kmajor_sw128(smem_u32(smB));
      int stage = 0;
      uint32_t phase = 0;
      int unit = 0;
      uint32_t a_phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      [[maybe_unused]] long long w_full = 0, w_tmem = 0;
      [[maybe_unused]] const long long t_begin = C2W_DIAG_CLOCK();
      for (int tile = group_id; tile < num_tiles; tile += num_groups) {
        C2W_TIMED_WAIT(w_tmem, &tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        const uint32_t ar_row_step = static_cast<uint32_t>(p.ar_row_step16);
        // PH: output phase (a, b) = the unit from its a-th row and b-th pixel on (leader: rank 0 = even M tile)
        uint32_t ph_off = 0;
        if (PH) {
          int ph;
          ph_split((tile / p.num_n_tiles) * CG, ph);
          ph_off = (ph >> 1) * ar_row_step + (ph & 1) * 8;
        }
        // K order cb -> s -> r -> k: each filter column's weight stage is released as soon as its nine MMAs are issued
        for (int cb = 0; AR && cb < p.cin_blocks; ++cb) {
          C2W_TIMED_WAIT(w_full, &a_full[unit], a_phase);
          const uint64_t adesc_u = adesc0 + static_cast<uint64_t>(unit * (Cfg::kARUnitBytes >> 4)) + ph_off;
          for (int s3 = 0; s3 < kCols; ++s3) {
            C2W_TIMED_WAIT(w_full, &full[stage], phase);
            tc_fence_after();
            if (elect_one()) {
              const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(stage * (Cfg::kARBStageBytes >> 4));
  #pragma unroll
              for (int r = 0; r < kCols; ++r) {
                // tap (r, s) = the unit from its r-th pixel row and s-th pixel column on.  The 128B swizzle is a
                // function of the absolute shared-memory address for the MMA's reads as for TMA's writes, so a start
                // address s * 128 B into a swizzle atom with 1280 B between 8-row groups reads what TMA wrote; the
                // descriptor's base-offset field stays 0 (set to (start >> 7) & 7 it gives wrong results).
                const uint64_t adesc = adesc_u + r * ar_row_step + s3 * 8;
  #pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k) {
                  const uint64_t a = adesc + 2 * k;
                  const uint64_t b = bdesc + r * (Cfg::kBTileBytes >> 4) + 2 * k;
                  if (CG == 2) umma_bf16_pair(tmem_d, a, b, idesc, (cb | s3 | r | k) != 0);
                  else umma_bf16(tmem_d, a, b, idesc, (cb | s3 | r | k) != 0);
                }
              }
              const bool last = s3 == kCols - 1 && cb + 1 == p.cin_blocks;
              if (CG == 2) {
                umma_commit_pair(&empty[stage]);
                if (s3 == kCols - 1) umma_commit_pair(&a_empty[unit]);
                if (last) umma_commit_pair(&tmem_full[acc]);
              } else {
                umma_commit(&empty[stage]);
                if (s3 == kCols - 1) umma_commit(&a_empty[unit]);
                if (last) umma_commit(&tmem_full[acc]);
              }
            }
            __syncwarp();
            if (++stage == num_stages) {
              stage = 0;
              phase ^= 1;
            }
          }
          if (++unit == num_units) {
            unit = 0;
            a_phase ^= 1;
          }
        }
        for (int kb = 0; !AR && kb < num_kb; kb += Cfg::kSub) {
          const int nsub = (num_kb - kb) < Cfg::kSub ? (num_kb - kb) : Cfg::kSub;
          C2W_TIMED_WAIT(w_full, &full[stage], phase);
          tc_fence_after();
          if (elect_one()) {
            // descriptor start-address field is (addr >> 4): slot stride and the 32 B K-advance are plain adds
            const uint64_t adesc = adesc0 + static_cast<uint64_t>(stage * Cfg::kSub * (kATileBytes >> 4));
            const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(stage * Cfg::kSub * (Cfg::kBTileBytes >> 4));
  #pragma unroll
            for (int sub = 0; sub < Cfg::kSub; ++sub) {
              if (sub < nsub) {
  #pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k) {
                  const uint64_t a = adesc + sub * (kATileBytes >> 4) + 2 * k;
                  const uint64_t b = bdesc + sub * (Cfg::kBTileBytes >> 4) + 2 * k;
                  if (CG == 2) umma_bf16_pair(tmem_d, a, b, idesc, (kb | sub | k) != 0);
                  else umma_bf16(tmem_d, a, b, idesc, (kb | sub | k) != 0);
                }
              }
            }
            if (CG == 2) {
              umma_commit_pair(&empty[stage]);
              if (kb + Cfg::kSub >= num_kb) umma_commit_pair(&tmem_full[acc]);
            } else {
              umma_commit(&empty[stage]);
              if (kb + Cfg::kSub >= num_kb) umma_commit(&tmem_full[acc]);
            }
          }
          __syncwarp();
          if (++stage == num_stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
#ifdef C2W_DIAG
      if (p.dbg_stats && lane == 0) {
        p.dbg_stats[blockIdx.x * 12 + 2] = clock64() - t_begin;
        p.dbg_stats[blockIdx.x * 12 + 3] = w_full;
        p.dbg_stats[blockIdx.x * 12 + 4] = w_tmem;
      }
#endif
    } else if (staged && warp_idx == 2) {
      // ------------------------------------------------------------ warp 2: staging tile -> global
      // TMA store of the finished tile and the prefetch of the auxiliary tile of the staging tile's next user; the
      // epilogue warps never wait for a TMA transfer.
      const bool leader = lane == 0;                // owns every bulk async-group of this CTA
      // PH: the box {64 ch, b, 8 px, a, 16 rows} at (b, j0, a, n * H + i0) of the {C, b, j, a, n * H + i} view of the
      // [n, 2H, 2W, C] output (H x W the low-res image): c1 = b, c2 = j0, c3 = a, c4 = n * H + i0
      auto ph_coords = [&](int mt, int& c1, int& c2, int& c3, int& c4) {
        int ph;
        mt = ph_split(mt, ph);
        const int img = mt / p.tiles_per_img, tt = mt % p.tiles_per_img;
        c1 = ph & 1;
        c2 = (tt % p.tiles_w) * Cfg::kARTileW;
        c3 = ph >> 1;
        c4 = img * p.img_h + (tt / p.tiles_w) * Cfg::kARTileH;
      };
      auto box_coords = [&](int mt, int& c1, int& c2, int& c3) {
        const int img = mt / p.tiles_per_img, tt = mt % p.tiles_per_img;
        c1 = (tt % p.tiles_w) * Cfg::kARTileW;
        c2 = (tt / p.tiles_w) * Cfg::kARTileH;  // ar2: 0
        c3 = p.ar2 ? 2 * img : img;             // ar2: first of the tile's two images
      };
      auto prefetch_aux = [&](int tile, int buf) {  // leader only: staging[buf] <- aux[tile]
        const int nt = tile % p.num_n_tiles;
        const int mt = (tile / p.num_n_tiles) * CG + rank;
        uint8_t* dst = stg0 + buf * Cfg::kStagingBytes;
#ifdef C2W_DIAG
        if (p.dbg_skip_loads == 5) {  // timing experiment: no residual traffic (stale staging contents are used)
          mbar_arrive(&res_full[buf]);
          return;
        }
#endif
        mbar_arrive_expect_tx(&res_full[buf], Cfg::kStagingBytes);
  #pragma unroll
        for (int b = 0; b < BN / 64; ++b) {
          if (PH) {
            int c1, c2, c3, c4;
            ph_coords(mt, c1, c2, c3, c4);
            tma_load_5d(&tmOut, &res_full[buf], dst + b * kATileBytes, nt * BN + b * 64, c1, c2, c3, c4);
          } else if (AR) {
            int c1, c2, c3;
            box_coords(mt, c1, c2, c3);
            if (p.ar2) {
              tma_load_4d(&tmOut, &res_full[buf], dst + b * kATileBytes, nt * BN + b * 64, c1, c2, c3);
              tma_load_4d(&tmOut, &res_full[buf], dst + b * kATileBytes + kATileBytes / 2, nt * BN + b * 64, c1, c2, c3 + 1);
            } else {
              tma_load_4d(&tmOut, &res_full[buf], dst + b * kATileBytes, nt * BN + b * 64, c1, c2, c3);
            }
          } else {
            tma_load_2d(&tmOut, &res_full[buf], dst + b * kATileBytes, nt * BN + b * 64, mt * kBlockM);
          }
        }
      };
      if (has_aux && leader) {  // two staging tiles: the auxiliary tile is prefetched two tiles ahead
        if (group_id < num_tiles) prefetch_aux(group_id, 0);
        if (two_bufs && group_id + num_groups < num_tiles) prefetch_aux(group_id + num_groups, 1);
      }
      int it_local = 0;
      for (int tile = group_id; tile < num_tiles; tile += num_groups) {
        const int nt = tile % p.num_n_tiles;
        const int mt = (tile / p.num_n_tiles) * CG + rank;
        const int buf = two_bufs ? (it_local & 1) : 0;
        const int use = two_bufs ? (it_local >> 1) : it_local;
        uint8_t* stg = stg0 + buf * Cfg::kStagingBytes;
        mbar_wait(&stg_full[buf], use & 1);
        if (leader) {
  #pragma unroll
          for (int b = 0; b < BN / 64; ++b) {
            if (PH) {
              int c1, c2, c3, c4;
              ph_coords(mt, c1, c2, c3, c4);
              tma_store_5d(&tmOut, stg + b * kATileBytes, nt * BN + b * 64, c1, c2, c3, c4);
            } else if (AR) {
              int c1, c2, c3;
              box_coords(mt, c1, c2, c3);
              tma_store_4d(&tmOut, stg + b * kATileBytes, nt * BN + b * 64, c1, c2, c3);
              if (p.ar2) tma_store_4d(&tmOut, stg + b * kATileBytes + kATileBytes / 2, nt * BN + b * 64, c1, c2, c3 + 1);
              if (dual) {
                const uint8_t* s2 = stg + Cfg::kStagingBytes + b * kATileBytes;
                tma_store_4d(&tmOut2, s2, nt * BN + b * 64, c1, c2, c3);
                if (p.ar2) tma_store_4d(&tmOut2, s2 + kATileBytes / 2, nt * BN + b * 64, c1, c2, c3 + 1);
              }
            } else {
              tma_store_2d(&tmOut, stg + b * kATileBytes, nt * BN + b * 64, mt * kBlockM);
              if (dual) tma_store_2d(&tmOut2, stg + Cfg::kStagingBytes + b * kATileBytes, nt * BN + b * 64, mt * kBlockM);
            }
          }
          bulk_commit();
        }
        // ---- the staging tile is free once the store has read it and every epilogue warp is done with its LayerNorm rows
        if (LN) mbar_wait(&ln_done[buf], use & 1);
        if (leader) {
          bulk_wait_read_all();
          const int next = tile + (two_bufs ? 2 : 1) * num_groups;  // this staging tile's next user
          if (has_aux) {
            if (next < num_tiles) prefetch_aux(next, buf);
          } else {
            mbar_arrive(&stg_free[buf]);
          }
        }
        ++it_local;
      }
      if (leader) bulk_wait_all();  // global writes of the last stores are complete before the CTA retires
    }
  } else if (warp_idx < 4 + kEpiWarps) {
    if constexpr (LN) asm volatile("setmaxnreg.inc.sync.aligned.u32 168;");
    {
      // ------------------------------------------------------------ epilogue: 8 warps = 128 rows x 2 column halves
      // TMEM -> registers -> (accumulator released) -> bias / SiLU / residual -> bf16 -> staging tile -> stg_full.
      // The stores, the LayerNorm pass and the auxiliary-tile prefetch belong to warps 2-3 (below): these warps never
      // wait for a TMA transfer they issued.
      const int ew = warp_idx - 4;
      const int q = ew & 3;       // TMEM lane quarter this warp may access (warp_idx % 4)
      const int half = ew >> 2;   // column half
      const int row = q * 32 + lane;
      constexpr int kHalfCols = BN / 2;
      constexpr int kChunks = kHalfCols / 32;  // 32-column chunks per warp (BN = 64: 1 ... BN = 256: 4)
      const int col_base = half * kHalfCols;
      int acc = 0;
      uint32_t acc_phase = 0;
      int it_local = 0;  // tiles processed by this CTA: staging tile it_local % 2 when double-buffered
      [[maybe_unused]] long long w_tfull = 0, w_stg = 0, c_pass1 = 0;
      [[maybe_unused]] const long long t_epi_begin = C2W_DIAG_CLOCK();
      for (int tile = group_id; tile < num_tiles; tile += num_groups) {
        const int nt = tile % p.num_n_tiles;
        const int mt = (tile / p.num_n_tiles) * CG + rank;
        int m = mt * kBlockM + row;
        if (AR) {
          const int img = mt / p.tiles_per_img, tt = mt % p.tiles_per_img;
          m = (img * p.img_h + (tt / p.tiles_w) * Cfg::kARTileH + (row >> 3)) * p.img_w + (tt % p.tiles_w) * Cfg::kARTileW +
              (row & 7);
          if (p.ar2)
            m = ((2 * img + ((row >> 3) & 1)) * p.img_h + (row >> 4)) * p.img_w + tt * Cfg::kARTileW + (row & 7);
        }
        const bool valid = m < p.m_total;
        // modulation vector of this tile's image (per-sample diffusion times) or of the whole batch
        const float* ln_mod_t = nullptr;
        if (LN && p.ln_mod != nullptr) {
          int ph, mt_img = mt;
          if (PH) mt_img = ph_split(mt, ph);
          ln_mod_t = p.ln_mod + static_cast<size_t>(p.ln_mod_stride) * (mt_img / p.tiles_per_img);
        }
        C2W_TIMED_WAIT(w_tfull, &tmem_full[acc], acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN + col_base;
        const int buf = two_bufs ? (it_local & 1) : 0;
        const int use = two_bufs ? (it_local >> 1) : it_local;  // how often this staging tile has been used before
        uint8_t* stg = stg0 + buf * Cfg::kStagingBytes;
        // ar2: the staging tile is kept image-major ([img][row][px]) so that each image is one plain TMA box
        const int srow = (AR && p.ar2) ? (((row >> 3) & 1) << 6) + ((row >> 4) << 3) + (row & 7) : row;
        uint8_t* stg_row = stg + srow * 128;
        // The accumulator is handed back to the MMA warp as soon as its last tcgen05.ld has landed in registers, before
        // the epilogue math: the MMAs of the next tile but one only ever wait for TMEM reads.
        auto release_acc = [&]() {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (CG == 2 && rank != 0) mbar_arrive_remote(mapa_shared(smem_u32(&tmem_empty[acc]), 0));
            else mbar_arrive(&tmem_empty[acc]);
          }
        };
        // staging tile ready to be written: its auxiliary tile has landed, or its previous store has read it
        auto wait_staging = [&]() {
          if (!staged) return;
          if (has_aux) C2W_TIMED_WAIT(w_stg, &res_full[buf], use & 1);
          else C2W_TIMED_WAIT(w_stg, &stg_free[buf], (use & 1) ^ 1);
        };
        [[maybe_unused]] const long long t_p1 = C2W_DIAG_CLOCK();
        float s1 = 0.f, s2 = 0.f;
        uint32_t va[32], vb[32];
        if constexpr (kChunks <= 2) {
          tmem_ld_32x32(taddr, va);
          if (kChunks == 2) tmem_ld_32x32(taddr + 32, vb);
          tmem_ld_wait();
          release_acc();
          wait_staging();
          if (staged) epilogue_chunk_staged<LN>(p, va, nt * BN + col_base, col_base, stg_row, row, s1, s2, ln_mod_t, dual ? static_cast<uint32_t>(Cfg::kStagingBytes) : 0u);
          else if constexpr (BN == 64) epilogue_chunk_direct(p, va, nt * BN + col_base, m, valid);
          if (kChunks == 2) {
            if (staged) epilogue_chunk_staged<LN>(p, vb, nt * BN + col_base + 32, col_base + 32, stg_row, row, s1, s2, ln_mod_t, dual ? static_cast<uint32_t>(Cfg::kStagingBytes) : 0u);
            else if constexpr (BN == 64) epilogue_chunk_direct(p, vb, nt * BN + col_base + 32, m, valid);
          }
        } else {
          // two register buffers: the tcgen05.ld of chunk i+1 is in flight while chunk i is processed
          tmem_ld_32x32(taddr, va);
          wait_staging();
  #pragma unroll
          for (int c = 0; c < kChunks; ++c) {
            tmem_ld_wait();
            if (c + 1 < kChunks) tmem_ld_32x32(taddr + 32 * (c + 1), (c & 1) ? va : vb);
            else release_acc();
            const int col = col_base + 32 * c;
            if (staged) epilogue_chunk_staged<LN>(p, (c & 1) ? vb : va, nt * BN + col, col, stg_row, row, s1, s2, ln_mod_t, dual ? static_cast<uint32_t>(Cfg::kStagingBytes) : 0u);
          }
        }
        if (staged) {
          if (LN) ln_stats[(buf * 2 + half) * kBlockM + row] = make_float2(s1, s2);
          fence_proxy_async();  // generic-proxy writes of the tile -> visible to the TMA store
          __syncwarp();
          if (lane == 0) mbar_arrive(&stg_full[buf]);
        }
#ifdef C2W_DIAG
        c_pass1 += clock64() - t_p1;
#endif
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
        ++it_local;
      }
#ifdef C2W_DIAG
      if (p.dbg_stats && threadIdx.x == 128) {
        p.dbg_stats[blockIdx.x * 12 + 5] = clock64() - t_epi_begin;
        p.dbg_stats[blockIdx.x * 12 + 6] = w_tfull;
        p.dbg_stats[blockIdx.x * 12 + 7] = w_stg;
        p.dbg_stats[blockIdx.x * 12 + 8] = c_pass1;
      }
#endif
    }
  } else {
    if constexpr (LN) asm volatile("setmaxnreg.dec.sync.aligned.u32 96;");
    if (LN && staged) {
      // ------------------------------------------------------------ warps 12-15: fused channel LayerNorm
      // Warp lw normalises rows [32 lw, 32 lw + 32) of every staged tile with the row statistics the epilogue warps
      // summed, while those warps are already working on the next tile.
      const int lw = warp_idx - (4 + kEpiWarps);
      constexpr int kLPR = BN / 8;                  // lanes per row (8 channels = 16 B each)
      constexpr int kRPI = (kLPR >= 32) ? 1 : 32 / kLPR;  // rows per warp iteration
      static_assert(!LN || (kLPR == 8 || kLPR == 16 || kLPR == 32), "fused LayerNorm needs BN in {64, 128, 256}");
      const int ln_chunk = lane % kLPR;             // 16 B chunk of the row this lane owns (channels 8 ln_chunk .. +8)
      float ln_m[8];
  #pragma unroll
      for (int e = 0; e < 8; ++e) ln_m[e] = (LN && p.ln_mod) ? __ldg(p.ln_mod + (ln_chunk * 8 + e) % BN) : 0.f;
      const bool ln_per_img = LN && p.ln_mod != nullptr && p.ln_mod_stride != 0;


      [[maybe_unused]] long long w_lnfull = 0, c_ln = 0;
      int it_local = 0;
      for (int tile = group_id; tile < num_tiles; tile += num_groups) {
        int mt = (tile / p.num_n_tiles) * CG + rank;
        int ph = 0;  // PH: output phase of the tile; mt becomes its low-res tile
        if (PH) mt = ph_split(mt, ph);
        const int buf = two_bufs ? (it_local & 1) : 0;
        const int use = two_bufs ? (it_local >> 1) : it_local;
        uint8_t* stg = stg0 + buf * Cfg::kStagingBytes;
        if (ln_per_img) {  // one diffusion time per sample: this tile's image has its own modulation vector
          const float* mv = p.ln_mod + static_cast<size_t>(p.ln_mod_stride) * (mt / p.tiles_per_img);
  #pragma unroll
          for (int e = 0; e < 8; ++e) ln_m[e] = __ldg(mv + (ln_chunk * 8 + e) % BN);
        }
        [[maybe_unused]] const long long t_ln0 = C2W_DIAG_CLOCK();
        if (LN) {
          C2W_TIMED_WAIT(w_lnfull, &stg_full[buf], use & 1);  // every warp's columns of the tile and the row statistics are in place
          // ---- channel LayerNorm of the staged rows: y = (x + mod - mean) * inv with the row statistics the epilogue
          //      warps summed (unbiased variance, model/nn.py:154,183); kLPR lanes write a row's C channels as one
          //      contiguous segment (x4 when the output is 2x nearest-upsampled, model/nn.py:184)
          const float2* st0 = ln_stats + (buf * 2 + 0) * kBlockM;
          const float2* st1 = ln_stats + (buf * 2 + 1) * kBlockM;
          // Output addressing, strength-reduced (this warp shares an issue port with two epilogue warps: every
          // instruction here is taken from them).  Row r of the tile -> element offset from a per-tile base:
          //   AR    : 16 x 8 block: ((r >> 3) * W' + (r & 7) * px) * BN     (W', px doubled when upsampled)
          //   rows  : plain [M, C] rows: r * BN  (the upsampled form of these tiles keeps the general path below)
          const bool fast = AR || !p.ln_up;
          __nv_bfloat16* tile_out = p.ln_out + ln_chunk * 8;
          long long tile_pix = 0;   // pixel index of tile row 0 (ln_inv, validity)
          int row_pitch = 0, px_pitch = BN;  // elements per image row / per pixel inside the tile
          bool tile_valid = true;
          if (AR) {
            const int tt = mt % p.tiles_per_img, img = mt / p.tiles_per_img;
            const int th0 = (tt / p.tiles_w) * Cfg::kARTileH, tw0 = (tt % p.tiles_w) * Cfg::kARTileW;
            tile_pix = (static_cast<long long>(img) * p.ln_H + th0) * p.ln_W + tw0;
            if (PH)  // tile row (i, j) is output pixel (2 (th0 + i) + a, 2 (tw0 + j) + b) of the ln_H x ln_W image
              tile_pix = (static_cast<long long>(img) * p.ln_H + 2 * th0 + (ph >> 1)) * p.ln_W + 2 * tw0 + (ph & 1);
            tile_valid = tile_pix < p.m_total;
            if (PH) {
              tile_out += tile_pix * BN;
              row_pitch = 2 * p.ln_W * BN;
              px_pitch = 2 * BN;
            } else if (p.ln_up) {
              tile_out += ((static_cast<long long>(img) * 2 * p.ln_H + 2 * th0) * 2 * p.ln_W + 2 * tw0) * BN;
              row_pitch = 4 * p.ln_W * BN;
              px_pitch = 2 * BN;
            } else {
              tile_out += tile_pix * BN;
              row_pitch = p.ln_W * BN;
            }
          } else {
            tile_pix = static_cast<long long>(mt) * kBlockM;
            tile_out += tile_pix * BN;
          }
          const int up_row = 2 * p.ln_W * BN;  // upsampled output: one output row further down
          constexpr int kIters = 32 / kRPI;
          constexpr int kBatch = kIters < 4 ? kIters : 4;
          const int rlane = lw * 32 + lane / kLPR;
          const uint32_t cbox = static_cast<uint32_t>(ln_chunk >> 3) * kATileBytes;
  #pragma unroll 1
          for (int it0 = 0; it0 < kIters; it0 += kBatch) {
            // loads of the whole batch, then the math, then the stores: the global stores alias the shared-memory
            // loads as far as the compiler can tell and would otherwise serialise the rows
            uint4 xr[kBatch];
            float2 sa[kBatch], sb[kBatch];
  #pragma unroll
            for (int bb = 0; bb < kBatch; ++bb) {
              const int r = rlane + (it0 + bb) * kRPI;
              xr[bb] = ld_shared_v4(stg, cbox + static_cast<uint32_t>(r) * 128u +
                                             (static_cast<uint32_t>((ln_chunk ^ r) & 7) << 4));
              sa[bb] = st0[r];
              sb[bb] = st1[r];
            }
            uint4 yv[kBatch];
            float invv[kBatch];
  #pragma unroll
            for (int bb = 0; bb < kBatch; ++bb) {
              const float sum = sa[bb].x + sb[bb].x, sq = sa[bb].y + sb[bb].y;
              const float mean = sum * (1.0f / BN);
              const float var = fmaxf(sq - sum * mean, 0.f) * (1.0f / (BN - 1));
              const float inv = rsqrtf(var + p.ln_eps);
              const float nmi = -mean * inv;
              const uint32_t w[4] = {xr[bb].x, xr[bb].y, xr[bb].z, xr[bb].w};
              uint32_t o4[4];
  #pragma unroll
              for (int j = 0; j < 4; ++j) {
                // bf16 pair -> fp32: low half shifted up, high half masked
                const float x0 = __uint_as_float(w[j] << 16), x1 = __uint_as_float(w[j] & 0xffff0000u);
                const float y0 = fmaf(x0, inv, fmaf(ln_m[2 * j], inv, nmi));
                const float y1 = fmaf(x1, inv, fmaf(ln_m[2 * j + 1], inv, nmi));
                __nv_bfloat162 y = __floats2bfloat162_rn(y0, y1);
                o4[j] = *reinterpret_cast<uint32_t*>(&y);
              }
              yv[bb] = make_uint4(o4[0], o4[1], o4[2], o4[3]);
              invv[bb] = inv;
            }
            if (fast) {
  #pragma unroll
              for (int bb = 0; bb < kBatch; ++bb) {
                const int r = rlane + (it0 + bb) * kRPI;
                const int eo = AR ? (r >> 3) * row_pitch + (r & 7) * px_pitch : r * BN;
                const bool ok = AR ? tile_valid : (tile_pix + r < p.m_total);
                if (ok) {
                  if (p.ln_inv != nullptr && ln_chunk == 0)
                    p.ln_inv[tile_pix + (PH ? 2 * ((r >> 3) * p.ln_W + (r & 7)) : AR ? (r >> 3) * p.ln_W + (r & 7) : r)] =
                        invv[bb];
                  __nv_bfloat16* dst = tile_out + eo;
                  *reinterpret_cast<uint4*>(dst) = yv[bb];
                  if (AR && p.ln_up) {
                    *reinterpret_cast<uint4*>(dst + BN) = yv[bb];
                    *reinterpret_cast<uint4*>(dst + up_row) = yv[bb];
                    *reinterpret_cast<uint4*>(dst + up_row + BN) = yv[bb];
                  }
                }
              }
            } else {
  #pragma unroll
              for (int bb = 0; bb < kBatch; ++bb) {  // upsampled output of a row tile: pixel coordinates by division
                const int r = rlane + (it0 + bb) * kRPI;
                const int mr = mt * kBlockM + r;
                const int ww = mr % p.ln_W;
                const int t = mr / p.ln_W;
                const int hh = t % p.ln_H, nimg = t / p.ln_H;
                if (mr < p.m_total) {
                  if (p.ln_inv != nullptr && ln_chunk == 0) p.ln_inv[mr] = invv[bb];
                  const long long o00 = (static_cast<long long>(nimg) * 2 * p.ln_H + 2 * hh) * 2 * p.ln_W + 2 * ww;
                  __nv_bfloat16* dst = p.ln_out + o00 * BN + ln_chunk * 8;
                  *reinterpret_cast<uint4*>(dst) = yv[bb];
                  *reinterpret_cast<uint4*>(dst + BN) = yv[bb];
                  *reinterpret_cast<uint4*>(dst + up_row) = yv[bb];
                  *reinterpret_cast<uint4*>(dst + up_row + BN) = yv[bb];
                }
              }
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&ln_done[buf]);
#ifdef C2W_DIAG
          c_ln += clock64() - t_ln0;
#endif
        }
        ++it_local;
      }
#ifdef C2W_DIAG
      if (p.dbg_stats && lane == 0 && lw == 0) {
        p.dbg_stats[blockIdx.x * 12 + 9] = w_lnfull;
        p.dbg_stats[blockIdx.x * 12 + 10] = c_ln;
      }
#endif
    }
  }

  tc_fence_before();
  if (CG == 2) cluster_sync_all();  // the leader's MMAs read the peer's shared memory until the last commit
  else __syncthreads();
#ifdef C2W_DIAG
  if (p.dbg_timeline != nullptr && threadIdx.x == 0) {
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    atomicMax(reinterpret_cast<unsigned long long*>(p.dbg_timeline) + 1, now);
  }
#endif
  if (warp_idx == 2) {
    tc_fence_after();
    // AR: the TMEM base is read back from shared memory rather than kept live through the whole kernel, which would
    // take a register from the 56 of the producer / MMA warps of the LayerNorm kernels (ptxas spills it otherwise)
    if (CG == 2) tmem_dealloc_pair(AR ? *tmem_slot : tmem_base, Cfg::kTmemCols);
    else tmem_dealloc(AR ? *tmem_slot : tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
// Host side

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !ptr) return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  }
  return fn;
}

inline char* tmap_error_slot() {
  static thread_local char buf[256] = {0};
  return buf;
}

// bf16 tensor map with 128B swizzle and zero OOB fill.  dims/box/estride are innermost-first; with an element
// stride e > 1 in a dimension the box TRAVERSES box[i] elements and loads every e-th one (ceil(box/e) elements).
// strides_bytes (rank - 1 entries, for dims 1..rank-1) defaults to the packed layout.
inline bool make_tmap_bf16(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint32_t* box,
                           const uint32_t* estride = nullptr, const uint64_t* strides_bytes = nullptr) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  // The driver entry point needs the primary context current on THIS thread; a thread that has made no runtime call
  // yet (e.g. PyTorch's autograd worker) has none.  cudaFree(0) is the canonical no-op that binds it.
  static thread_local bool ctx_bound = false;
  if (!ctx_bound) {
    cudaFree(0);
    ctx_bound = true;
  }
  cuuint64_t gdim[5];
  cuuint64_t gstride[4];
  cuuint32_t bdim[5];
  cuuint32_t estr[5];
  uint64_t pitch = 2;
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = estride ? estride[i] : 1;
    pitch *= dims[i];
    if (i < rank - 1) gstride[i] = strides_bytes ? strides_bytes[i] : pitch;
  }
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), gdim, gstride, bdim, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char* e = tmap_error_slot();
    int o = snprintf(e, 256, "cuTensorMapEncodeTiled -> %d: base %p rank %d dims", (int)r, base, rank);
    for (int i = 0; i < rank && o < 230; ++i) o += snprintf(e + o, 256 - o, " %llu/%u", (unsigned long long)gdim[i], bdim[i]);
  }
  return r == CUDA_SUCCESS;
}

// One prepared launch of K1: tensor maps + parameters.  Built once per (layer, batch) and replayed.
struct ConvLaunch {
  CUtensorMap tmA, tmB, tmOut, tmOut2;
  ConvParams p;
  int bn;
  int cg;     // CTAs per MMA (1 or 2)
  int ln;     // fused LayerNorm output
  int ar;     // activation-reuse main loop (16 x 8 spatial tiles)
  int ph;     // phase form of the activation-reuse main loop (conv_launch_init_phase)
  int grid;   // CTAs (a multiple of cg)
  int n_img, Ho, Wo, cout_pad;
  const void* out_ptr;  // bf16 output bound by conv_launch_set_out (LayerNorm fusion matches on it)
};

// Kernel variant of a launch: a pair of CTAs per MMA whenever there are at least two M tiles.
inline int conv_pick_cg(int num_m_tiles) { return num_m_tiles >= 2 ? 2 : 1; }

inline void conv_set_grid(ConvLaunch* L, int num_sms) {
  const int groups = ((L->p.num_m_tiles + L->cg - 1) / L->cg) * L->p.num_n_tiles;
  const int max_groups = num_sms / L->cg;
  L->grid = (groups < max_groups ? groups : max_groups) * L->cg;
  if (L->grid < L->cg) L->grid = L->cg;
}

// Geometry of the activation operand.
//  conv3x3: x is NHWC [n_img, H, W, cin] bf16 (cin % 64 == 0); stride 1: output [n_img, H, W], stride 2: output
//           [n_img, H/2, W/2] (pad 1 either way)
//  gemm   : x is [m, k] bf16 row-major (k % 64 == 0) with m = n_img * H * W
// Images the activation-reuse main loop can tile: 16 x 8 pixel blocks.
inline bool conv_ar_geometry_ok(int H, int W) { return (H % 16 == 0 || H == 8) && W % 8 == 0; }

// variant: -1 = pick; else bit 0 = CTA pair (cta_group::2), bit 2 = activation-reuse main loop
inline bool conv_launch_init(ConvLaunch* L, bool is_conv3x3, const __nv_bfloat16* x, int n_img, int H, int W, int cin,
                             const __nv_bfloat16* w_packed, int cout_pad, int bn, int num_sms, int stride = 1,
                             int variant = -1) {
  ConvParams& p = L->p;
  memset(&p, 0, sizeof(p));
  memset(&L->tmOut, 0, sizeof(CUtensorMap));
  memset(&L->tmOut2, 0, sizeof(CUtensorMap));
  L->bn = bn;
  L->ln = 0;
  L->ph = 0;
  L->out_ptr = nullptr;
  if (cin % kBlockK != 0 || cout_pad % bn != 0) return false;
  if (stride != 1 && !(stride == 2 && is_conv3x3 && H % 2 == 0 && W % 2 == 0)) return false;
  p.cin_blocks = cin / kBlockK;
  p.num_n_tiles = cout_pad / bn;
  p.stride = stride;
  p.ln_eps = 1e-5f;
  const int Ho = H / stride, Wo = W / stride;
  L->n_img = n_img;
  L->Ho = Ho;
  L->Wo = Wo;
  L->cout_pad = cout_pad;
  const long long m_total = static_cast<long long>(n_img) * Ho * Wo;
  p.m_total = static_cast<int>(m_total);
  p.num_m_tiles = static_cast<int>((m_total + kBlockM - 1) / kBlockM);
  L->cg = variant < 0 ? conv_pick_cg(p.num_m_tiles) : ((variant & 1) ? 2 : 1);
  L->ar = 0;
  if (is_conv3x3) {
    // streamed M tile: whole output rows of 1..n images (Wo <= 128), or one 128-pixel segment of a row (Wo > 128)
    const bool segs = Wo > kBlockM;
    if (segs ? Wo % kBlockM != 0 : kBlockM % Wo != 0) return false;
    int th = segs ? 1 : kBlockM / Wo;
    if (th > Ho) th = Ho;
    if (Ho % th != 0) return false;
    const int tn = segs ? 1 : kBlockM / (Wo * th);
    p.taps = 9;
    p.tile_h = th;
    p.tile_n = tn;
    p.row_segs = segs ? Wo / kBlockM : 1;
    p.tiles_per_img = (Ho / th) * p.row_segs;
    // activation reuse: stride-1 convs with 64- or 128-wide N tiles per CTA pair on images that tile into 16 x 8 blocks
    static int ar_ok = -1;
    if (ar_ok < 0) {
      const char* e = getenv("C2W_NO_AR");
      ar_ok = (e && e[0] == '1') ? 0 : 1;
    }
    const bool want_ar = (variant < 0) ? ar_ok != 0 : (variant & 4) != 0;
    if (want_ar && stride == 1 && (bn == 128 || bn == 64) && L->cg == 2 && H % 16 == 0 && W % 8 == 0) {
      L->ar = 1;
      p.tiles_w = W / 8;
      p.tiles_per_img = (H / 16) * p.tiles_w;
      p.img_h = H;
      p.img_w = W;
      p.ar_row_step16 = (kARUnitW * 128) >> 4;
      p.ar_tx_a = 18 * kARUnitW * kBlockK * 2;
      p.ar_tx_b = 3 * (bn / L->cg) * kBlockK * 2;
      const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)W, (uint64_t)H, (uint64_t)n_img};
      const uint32_t box[4] = {(uint32_t)kBlockK, (uint32_t)kARUnitW, 18u, 1u};
      if (!make_tmap_bf16(&L->tmA, x, 4, dims, box)) return false;
    } else if (want_ar && stride == 1 && bn == 128 && L->cg == 2 && H == 8 && W % 8 == 0 && n_img >= 2) {
      // two 8-row images per M tile, image dimension inside the row dimension (see ConvParams::ar2)
      L->ar = 1;
      p.ar2 = 1;
      p.tiles_w = W / 8;
      p.tiles_per_img = p.tiles_w;
      p.num_m_tiles = ((n_img + 1) / 2) * p.tiles_w;
      p.img_h = H;
      p.img_w = W;
      p.ar_row_step16 = (2 * kARUnitW * 128) >> 4;
      p.ar_tx_a = 10 * 2 * kARUnitW * kBlockK * 2;
      p.ar_tx_b = 3 * (bn / L->cg) * kBlockK * 2;
      const uint64_t row_b = (uint64_t)W * cin * 2;
      const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)W, (uint64_t)n_img, (uint64_t)H};
      const uint64_t strides[3] = {(uint64_t)cin * 2, row_b * H, row_b};
      const uint32_t box[4] = {(uint32_t)kBlockK, (uint32_t)kARUnitW, 2u, 10u};
      if (!make_tmap_bf16(&L->tmA, x, 4, dims, box, nullptr, strides)) return false;
    } else {
      if (variant >= 0 && (variant & 4)) return false;  // AR was requested explicitly but does not apply
      const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)W, (uint64_t)H, (uint64_t)n_img};
      const uint32_t box[4] = {(uint32_t)kBlockK, (uint32_t)((Wo / p.row_segs) * stride), (uint32_t)(th * stride),
                               (uint32_t)tn};
      const uint32_t est[4] = {1u, (uint32_t)stride, (uint32_t)stride, 1u};
      if (!make_tmap_bf16(&L->tmA, x, 4, dims, box, est)) return false;
    }
  } else {
    p.taps = 1;
    p.tile_h = 1;
    p.tile_n = 1;
    p.tiles_per_img = 1;
    const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)m_total, 1, 1};
    const uint32_t box[4] = {(uint32_t)kBlockK, (uint32_t)kBlockM, 1, 1};
    if (!make_tmap_bf16(&L->tmA, x, 4, dims, box)) return false;
  }
  if (L->ar) {
    // the three B tiles (r = 0..2) of one (filter column s, channel block) in one box: the packed weights
    // [Cout][r][s][Cin] viewed as {s * Cin + c, Cout, r}, the r tiles landing one after the other in the stage
    const uint64_t dims[4] = {(uint64_t)3 * cin, (uint64_t)cout_pad, 3, 1};
    const uint64_t strides[3] = {(uint64_t)9 * cin * 2, (uint64_t)3 * cin * 2, (uint64_t)9 * cin * 2 * cout_pad};
    const uint32_t box[4] = {(uint32_t)kBlockK, (uint32_t)(bn / L->cg), 3u, 1u};
    if (!make_tmap_bf16(&L->tmB, w_packed, 4, dims, box, nullptr, strides)) return false;
  } else {
    const uint64_t dims[2] = {(uint64_t)p.taps * cin, (uint64_t)cout_pad};
    const uint32_t box[2] = {(uint32_t)kBlockK, (uint32_t)(bn / L->cg)};
    if (!make_tmap_bf16(&L->tmB, w_packed, 2, dims, box)) return false;
  }
  conv_set_grid(L, num_sms);
  p.ldc = cout_pad;
  return true;
}

// Phase weights of a 3x3 conv applied to a nearest x2 upsampled input (see ph_split): fp32 OIHW [cout, cin, 3, 3] ->
// bf16 [4 phases][cout_pad][4 taps * cin_pad], phase = 2a + b, tap = 2 tr + ts, k = tap * cin_pad + c (zero padding).
// Merged weight (a, b, tr, ts) = sum of w[r][s] over the filter rows r that read low-res row offset tr of phase a
// (a = 0: tr 0 <- r 0, tr 1 <- r 1, 2; a = 1: tr 0 <- r 0, 1, tr 1 <- r 2) and the same for columns, summed in fp32 in
// the order r -> s (ascending) and rounded to bf16 once.  refresh_weights_kernel repeats this sum in the same order.
__host__ __device__ inline float conv_phase_weight(const float* w9, int a, int b, int tr, int ts) {
  const int r0 = tr == 0 ? 0 : 1 + a, r1 = tr == 0 ? a : 2;
  const int s0 = ts == 0 ? 0 : 1 + b, s1 = ts == 0 ? b : 2;
  float acc = 0.f;
  for (int r = r0; r <= r1; ++r)
    for (int s = s0; s <= s1; ++s) acc += w9[r * 3 + s];
  return acc;
}
inline void conv_pack_phase_weights(const float* w, int cout, int cin, int cin_pad, int cout_pad, __nv_bfloat16* out) {
  const size_t K = static_cast<size_t>(4) * cin_pad;
  for (size_t i = 0; i < 4 * static_cast<size_t>(cout_pad) * K; ++i) out[i] = __float2bfloat16_rn(0.f);
  for (int ph = 0; ph < 4; ++ph)
    for (int o = 0; o < cout; ++o)
      for (int c = 0; c < cin; ++c)
        for (int t = 0; t < 4; ++t)
          out[(static_cast<size_t>(ph) * cout_pad + o) * K + static_cast<size_t>(t) * cin_pad + c] = __float2bfloat16_rn(
              conv_phase_weight(w + (static_cast<size_t>(o) * cin + c) * 9, ph >> 1, ph & 1, t >> 1, t & 1));
}

// The phase form of conv3x3(nearest x2 (x)) (see ph_split): x is the LOW-RES NHWC input [n_img, H, W, cin], w_phase
// the phase weights (conv_pack_phase_weights), the output [n_img, 2H, 2W, cout_pad].  Needs the activation-reuse
// geometry at the low resolution with an even number of 16 x 8 tiles per image (the two CTAs of a pair share a phase).
inline bool conv_phase_geometry_ok(int H, int W) { return H % 16 == 0 && W % 8 == 0 && (H / 16) * (W / 8) % 2 == 0; }
inline bool conv_launch_init_phase(ConvLaunch* L, const __nv_bfloat16* x, int n_img, int H, int W, int cin,
                                   const __nv_bfloat16* w_phase, int cout_pad, int bn, int num_sms) {
  ConvParams& p = L->p;
  memset(&p, 0, sizeof(p));
  memset(&L->tmOut, 0, sizeof(CUtensorMap));
  memset(&L->tmOut2, 0, sizeof(CUtensorMap));
  L->bn = bn;
  L->ln = 0;
  L->out_ptr = nullptr;
  if (cin % kBlockK != 0 || !(bn == 64 || bn == 128) || cout_pad % bn != 0 || n_img < 1 ||
      !conv_phase_geometry_ok(H, W))
    return false;
  L->cg = 2;
  L->ar = 1;
  L->ph = 1;
  L->n_img = n_img;
  L->Ho = 2 * H;
  L->Wo = 2 * W;
  L->cout_pad = cout_pad;
  p.taps = 4;
  p.stride = 1;
  p.cin_blocks = cin / kBlockK;
  p.num_n_tiles = cout_pad / bn;
  p.ln_eps = 1e-5f;
  p.m_total = 4 * n_img * H * W;
  p.tiles_w = W / 8;
  p.tiles_per_img = (H / 16) * p.tiles_w;
  p.num_m_tiles = 4 * n_img * p.tiles_per_img;
  p.img_h = H;
  p.img_w = W;
  p.ar_row_step16 = (kARUnitW * 128) >> 4;
  p.ar_tx_a = 18 * kARUnitW * kBlockK * 2;
  p.ar_tx_b = 2 * (bn / 2) * kBlockK * 2;
  {
    const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)W, (uint64_t)H, (uint64_t)n_img};
    const uint32_t box[4] = {(uint32_t)kBlockK, (uint32_t)kARUnitW, 18u, 1u};
    if (!make_tmap_bf16(&L->tmA, x, 4, dims, box)) return false;
  }
  {  // [phase][Cout][tr][ts * Cin + c] viewed as {ts * Cin + c, Cout, tr, phase}: the two tr tiles of one (ts, cb)
    const uint64_t dims[4] = {(uint64_t)2 * cin, (uint64_t)cout_pad, 2, 4};
    const uint64_t strides[3] = {(uint64_t)4 * cin * 2, (uint64_t)2 * cin * 2, (uint64_t)4 * cin * 2 * cout_pad};
    const uint32_t box[4] = {(uint32_t)kBlockK, (uint32_t)(bn / 2), 2u, 1u};
    if (!make_tmap_bf16(&L->tmB, w_phase, 4, dims, box, nullptr, strides)) return false;
  }
  conv_set_grid(L, num_sms);
  p.ldc = cout_pad;
  return true;
}

// Tensor map of a bf16 [M, cout_pad] epilogue tensor: rows of 128 pixels, or (AR) 16 x 8 spatial blocks of the
// [n, H, W, cout_pad] view of the same memory (PH: the {C, b, j, a, n * H + i} view of [n, 2H, 2W, C], see ph_coords).
inline bool conv_make_epi_map(const ConvLaunch* L, CUtensorMap* m, const void* ptr) {
  if (L->ph) {
    const uint64_t C = L->cout_pad, Wl = L->Wo / 2, Hl = L->Ho / 2;
    const uint64_t dims[5] = {C, 2, Wl, 2, (uint64_t)L->n_img * Hl};
    const uint64_t strides[4] = {C * 2, 2 * C * 2, 2 * Wl * C * 2, 4 * Wl * C * 2};
    const uint32_t box[5] = {64u, 1u, 8u, 1u, 16u};
    return make_tmap_bf16(m, ptr, 5, dims, box, nullptr, strides);
  }
  if (L->ar) {  // ar2: one 8 x 8 box per image (the staging tile is image-major)
    const uint64_t dims[4] = {(uint64_t)L->cout_pad, (uint64_t)L->Wo, (uint64_t)L->Ho, (uint64_t)L->n_img};
    const uint32_t box[4] = {64u, 8u, L->p.ar2 ? 8u : 16u, 1u};
    return make_tmap_bf16(m, ptr, 4, dims, box);
  }
  const uint64_t dims[2] = {(uint64_t)L->cout_pad, (uint64_t)L->p.m_total};
  const uint32_t box[2] = {64u, (uint32_t)kBlockM};
  return make_tmap_bf16(m, ptr, 2, dims, box);
}
// bf16 output [M, cout_pad] (modes 0..2).  Mode 2 accumulates in place: `out` is also the residual.
inline bool conv_launch_set_out(ConvLaunch* L, __nv_bfloat16* out) {
  L->out_ptr = out;
  return conv_make_epi_map(L, &L->tmOut, out);
}

// Second bf16 output of EPI_BIAS_SILU_DUAL (the SiLU of the first)
inline bool conv_launch_set_out2(ConvLaunch* L, __nv_bfloat16* out2) {
  if (L->bn > 128 || L->ph) return false;  // two staging tiles of a wider tile leave no operand ring
  return conv_make_epi_map(L, &L->tmOut2, out2);
}

// Whether this launch can also emit the channel LayerNorm of its output (one N tile = all channels of a pixel).
inline bool conv_launch_can_ln(const ConvLaunch* L, int upsample) {
  const ConvParams& p = L->p;
  if (L->ln || p.ar2 || p.num_n_tiles != 1 || !(L->bn == 64 || L->bn == 128 || L->bn == 256)) return false;
  if (!(p.mode == EPI_BIAS || p.mode == EPI_BIAS_RES)) return false;
  if (upsample && (p.taps != 9 || L->ph)) return false;
  return true;
}

// Fused LayerNorm output: ln_out is [M, C] or, upsampled, [n_img, 2Ho, 2Wo, C]
// ln_mod_stride != 0: one modulation vector per image (tiles must lie inside one image: 16 x 8 blocks, or 128-pixel row
// tiles of images with a multiple of 128 pixels)
inline bool conv_launch_set_ln(ConvLaunch* L, __nv_bfloat16* ln_out, const float* ln_mod, int upsample,
                               int ln_mod_stride = 0) {
  ConvParams& p = L->p;
  if (!conv_launch_can_ln(L, upsample)) return false;
  if (ln_mod_stride != 0 && !(L->ar || (p.taps == 9 && p.tile_n == 1))) return false;
  p.ln_out = ln_out;
  p.ln_mod = ln_mod;
  p.ln_mod_stride = ln_mod_stride;
  p.ln_up = upsample;
  p.ln_H = L->Ho;
  p.ln_W = L->Wo;
  L->ln = 1;
  return true;
}

// C2W_PDL=0 launches K1 fully stream-serialised (A/B runs); default: programmatic dependent launch.
inline bool conv_use_pdl() {
  static int pdl = -1;
  if (pdl < 0) {
    const char* e = getenv("C2W_PDL");
    pdl = (e && e[0] == '0') ? 0 : 1;
  }
  return pdl != 0;
}

template <int BN, int CG, bool LN, bool AR, bool PH = false>
inline cudaError_t conv_launch_variant(const ConvLaunch& L, cudaStream_t stream) {
  using Cfg = ConvCfg<BN, CG>;
  static_assert(!AR || Cfg::ar_stages_for(2) >= 3, "activation-reuse weight ring too shallow");
  // the attribute is per device: remember which devices of this process have it
  static unsigned long long attr_done = 0;
  int dev = 0;
  cudaGetDevice(&dev);
  if (!((attr_done >> (dev & 63)) & 1ull)) {
    cudaError_t e = cudaFuncSetAttribute(conv_gemm_tcgen05_kernel<BN, CG, LN, AR, PH>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
    if (e != cudaSuccess) return e;
    attr_done |= 1ull << (dev & 63);
  }
  ConvParams p = L.p;
  const bool staged = p.mode != EPI_COMPOSE && p.mode != EPI_F32;
  if (!staged && BN != 64) return cudaErrorInvalidValue;  // fp32 / compose epilogues: 64-wide tiles only
  // Two staging tiles only for residual convs with narrow tiles (the residual tile is prefetched two tiles ahead; wide
  // tiles take long enough to prefetch one ahead into the single tile); everywhere else the shared memory is worth
  // more as ring stages (G2: 1239 -> 1345 TFLOP/s with 4 instead of 3 activation-reuse stages).  Residual convs with
  // ONE staging tile and a 4-deep ring were measured too: residual 1215 -> 1187, residual + LayerNorm 1050 -> 860.
  p.num_staging = ((p.mode == EPI_BIAS_RES || p.mode == EPI_MUL_DSILU) && BN <= 128) ? 2 : 1;
  if (p.mode == EPI_BIAS_SILU_DUAL) {
    if (BN > 128) return cudaErrorInvalidValue;
    p.num_staging = 2;
  }
  p.num_stages = AR ? Cfg::ar_stages_for(p.num_staging) : Cfg::stages_for(p.num_staging);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(L.grid);
  cfg.blockDim = dim3(kConvThreads + (LN ? kLnThreads : 0));
  cfg.dynamicSmemBytes = AR ? Cfg::ar_smem_bytes(p.num_staging) : Cfg::smem_bytes(p.num_staging);
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (conv_use_pdl()) {  // overlap this kernel's prologue with the previous kernel's tail (griddepcontrol in the kernel)
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
  }
  return cudaLaunchKernelEx(&cfg, conv_gemm_tcgen05_kernel<BN, CG, LN, AR, PH>, L.tmA, L.tmB, L.tmOut, L.tmOut2, p);
}

template <int BN, bool LN>
inline cudaError_t conv_launch_bn_ln(const ConvLaunch& L, cudaStream_t stream) {
  if (L.cg == 2) {
    if constexpr (BN == 128 || BN == 64) {
      if (L.ph) return conv_launch_variant<BN, 2, LN, true, true>(L, stream);
      if (L.ar) return conv_launch_variant<BN, 2, LN, true>(L, stream);
    }
    return conv_launch_variant<BN, 2, LN, false>(L, stream);
  }
  return conv_launch_variant<BN, 1, LN, false>(L, stream);
}

template <int BN>
inline cudaError_t conv_launch_bn(const ConvLaunch& L, cudaStream_t stream) {
  if constexpr (BN != 192) {
    if (L.ln) return conv_launch_bn_ln<BN, true>(L, stream);
  }
  return conv_launch_bn_ln<BN, false>(L, stream);
}

inline cudaError_t conv_launch(const ConvLaunch& L, cudaStream_t stream) {
  switch (L.bn) {
    case 64: return conv_launch_bn<64>(L, stream);
    case 128: return conv_launch_bn<128>(L, stream);
    case 192: return conv_launch_bn<192>(L, stream);
    case 256: return conv_launch_bn<256>(L, stream);
    default: return cudaErrorInvalidValue;
  }
}

// N tile for a (padded) output-channel count.
inline int conv_pick_bn(int cout_pad) {
  if (cout_pad % 256 == 0) return 256;
  if (cout_pad % 192 == 0) return 192;
  if (cout_pad % 128 == 0) return 128;
  return 64;
}

// N-tile width for one conv of the UNet.  Below 256 output channels one tile holds a whole pixel.  From 256 up the
// choice is made on the number of WAVES the persistent grid needs — ceil(pair tiles / CTA pairs) * BN, weighted by
// the measured per-flop cost of each main loop with a full grid (tools/bringup_conv.py --tiles, 156 windows:
// activation reuse with 128-wide tiles ~1540 TFLOP/s, 256-wide streamed ~1470, 192-wide streamed ~1340, 128-wide
// streamed ~1110).  E.g. 16x16x384: 5 waves of 192 (94 us) -> 7 waves of 128 with activation reuse (69 us); 8x8x512:
// 2 waves of 256 (55 us) -> 3 waves of 128 in the two-image form (41 us).  A 256-channel conv whose output feeds a
// LayerNorm is rebuilt with one 256-wide tile by the engine (the fused normalisation needs the whole pixel).
inline int conv_pick_bn_tiled(int cout_pad, bool is_conv3x3, int n_img, int H, int W, int stride, int num_sms) {
  static int policy = -1;
  if (policy < 0) {
    const char* e = getenv("C2W_BN_POLICY");
    policy = e ? atoi(e) : 1;
  }
  if (policy == 0 || cout_pad < 256) return conv_pick_bn(cout_pad);
  const long long m_tiles = (static_cast<long long>(n_img) * (H / stride) * (W / stride) + kBlockM - 1) / kBlockM;
  if (m_tiles < 2) return conv_pick_bn(cout_pad);
  const bool ar = is_conv3x3 && stride == 1 && conv_ar_geometry_ok(H, W);
  const long long pairs = num_sms / 2 > 0 ? num_sms / 2 : 1;
  int best = 0;
  double best_cost = 0.0;
  const int cand[4] = {256, 192, 128, 64};
  for (int bn : cand) {
    if (cout_pad % bn != 0) continue;
    const bool bn_ar = ar && (bn == 128 || (bn == 64 && H != 8));
    const double per_flop = bn_ar ? (bn == 128 ? 1.0 : 1.35) : (bn == 256 ? 1.05 : bn == 192 ? 1.15 : bn == 128 ? 1.39 : 1.9);
    const long long groups = ((m_tiles + 1) / 2) * (cout_pad / bn);
    const long long waves = (groups + pairs - 1) / pairs;
    const double cost = static_cast<double>(waves) * bn * per_flop;
    if (best == 0 || cost < best_cost - 1e-9) {
      best = bn;
      best_cost = cost;
    }
  }
  return best ? best : conv_pick_bn(cout_pad);
}

}  // namespace c2w
