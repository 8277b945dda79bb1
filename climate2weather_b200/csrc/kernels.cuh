// Fused, coalesced, vectorised CUDA kernels around K1 (all HBM- or latency-bound; no tensor cores):
//   K0  gather_windows      src/thor/score.py:68-74,143-154   unfold -> bf16 NHWC window batch
//   K2  channel_layernorm   model/nn.py:154,183,44 (zuko LayerNorm over C) + modulation add (+ 2x nearest upsample)
//   K3  time embedding MLP + all modulation projections        model/score.py:14-34,61-67 ; model/nn.py:149
//   K4  attention core      model/nn.py:64-85
//   K6  guided eps + predictor update                          src/thor/score.py:44-60,24-35 ; pipelines.py:41-46
//   K7  corrector (guided eps, ||eps||^2, Langevin update)     src/thor/pipelines.py:81-88
//   layout converters between the reference's NCHW fp32 tensors and the device layouts
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace c2w {

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t w) {
  __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&w);
  return make_float2(__low2float(h), __high2float(h));
}

// ------------------------------------------------------------------------------------------------ K0
// traj: fp32 [frames, HW, C]; window i of this launch starts at local frame f0 + i.
// out : bf16 [n, HW, cin_pad], channel tau*C + c  <-  traj[f0 + i + tau, pix, c]; channels >= wC are zero.
// One thread writes 8 channels (16 B): writes are fully coalesced, reads are 16 B (C = 4) sectors.
// win_list (optional): GLOBAL window indices of the n windows (a selection, e.g. the windows whose output carries a
// non-zero cotangent); window i then starts at local frame win_list[i] - f0 (f0 = global index of local frame 0).
__global__ void gather_windows_kernel(const float* __restrict__ traj, bf16* __restrict__ out, int n, int hw, int C,
                                      int wC, int cin_pad, int f0, const int* __restrict__ win_list = nullptr) {
  const int groups = cin_pad >> 3;
  const long long total = static_cast<long long>(n) * hw * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(idx % groups);
    const long long pw = idx / groups;
    const int pix = static_cast<int>(pw % hw);
    const int i = static_cast<int>(pw / hw);
    const int fw = win_list ? (win_list[i] - f0) : (f0 + i);  // first local frame of window i
    float v[8];
    if (C == 4) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int tau = 2 * g + h;
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
        if (tau * 4 < wC)
          q = __ldg(reinterpret_cast<const float4*>(traj + (static_cast<long long>(fw + tau) * hw + pix) * 4));
        v[4 * h + 0] = q.x;
        v[4 * h + 1] = q.y;
        v[4 * h + 2] = q.z;
        v[4 * h + 3] = q.w;
      }
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int ch = 8 * g + e;
        const int tau = ch / C, c = ch - tau * C;
        v[e] = (ch < wC) ? __ldg(traj + (static_cast<long long>(fw + tau) * hw + pix) * C + c) : 0.f;
      }
    }
    uint4 o = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]),
                         pack_bf16x2(v[6], v[7]));
    *reinterpret_cast<uint4*>(out + (static_cast<long long>(i) * hw + pix) * cin_pad + 8 * g) = o;
  }
}

// Tiled form for C = 4 (the shipped 4-variable frames): a CTA owns 64 pixels x kGatherWin consecutive windows, reads the
// kGatherWin + w - 1 frames they span ONCE (coalesced float4 -> packed bf16x4 in shared memory) and writes every
// window's 128-byte pixel rows from there: each frame pixel leaves L2 1.75 times (w = 13) instead of 13 times.
constexpr int kGatherWin = 16, kGatherPix = 64;
__global__ void __launch_bounds__(256) gather_windows_tiled_kernel(const float* __restrict__ traj, bf16* __restrict__ out,
                                                                   int n, int hw, int w, int cin_pad, int f0) {
  extern __shared__ uint2 gtile[];  // [frames][kGatherPix] bf16x4
  const int pix0 = blockIdx.x * kGatherPix, i0 = blockIdx.y * kGatherWin;
  const int nwin = (n - i0) < kGatherWin ? (n - i0) : kGatherWin;
  const int nfr = nwin + w - 1;
  for (int idx = threadIdx.x; idx < nfr * kGatherPix; idx += blockDim.x) {
    const int fr = idx / kGatherPix, px = idx - fr * kGatherPix;
    const float4 q = __ldg(reinterpret_cast<const float4*>(traj + (static_cast<long long>(f0 + i0 + fr) * hw + pix0 + px) * 4));
    gtile[idx] = make_uint2(pack_bf16x2(q.x, q.y), pack_bf16x2(q.z, q.w));
  }
  __syncthreads();
  const int groups = cin_pad >> 3;
  for (int idx = threadIdx.x; idx < nwin * kGatherPix * groups; idx += blockDim.x) {
    const int g = idx % groups;
    const int t = idx / groups;
    const int px = t % kGatherPix, il = t / kGatherPix;
    const int tau = 2 * g;
    uint2 a = make_uint2(0u, 0u), b = make_uint2(0u, 0u);
    if (tau < w) a = gtile[(il + tau) * kGatherPix + px];
    if (tau + 1 < w) b = gtile[(il + tau + 1) * kGatherPix + px];
    *reinterpret_cast<uint4*>(out + (static_cast<long long>(i0 + il) * hw + pix0 + px) * cin_pad + 8 * g) =
        make_uint4(a.x, a.y, b.x, b.y);
  }
}

// ------------------------------------------------------------------------------------------------ K2
// y = (v - mean_C(v)) / sqrt(var_C(v) + eps), v = x + mod, unbiased variance (torch.var_mean default), no affine.
// One warp per pixel; lane owns NCH chunks of VEC channels: chunk j = channels [j*32*VEC + lane*VEC, +VEC)
// so every chunk is one coalesced warp access.  upsample != 0 writes each pixel to its 2x2 nearest-neighbour
// block of a [n, 2H, 2W, C] tensor (model/nn.py:183-184 fused).
template <int C>
__global__ void channel_layernorm_kernel(const bf16* __restrict__ x, const float* __restrict__ mod,
                                         bf16* __restrict__ out, float* __restrict__ inv_out, long long npix, int H,
                                         int W, int upsample, float eps, long long mod_img_stride) {
  constexpr int VEC = (C % 128 == 0) ? 4 : 2;
  constexpr int NCH = C / (32 * VEC);
  static_assert(C % 64 == 0 && NCH >= 1, "C must be a multiple of 64");
  const int lane = threadIdx.x & 31;
  const long long warp0 = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  float m[NCH * VEC];
#pragma unroll
  for (int j = 0; j < NCH; ++j)
#pragma unroll
    for (int e = 0; e < VEC; ++e) m[j * VEC + e] = mod ? __ldg(mod + j * 32 * VEC + lane * VEC + e) : 0.f;

  for (long long pix = warp0; pix < npix; pix += nwarps) {
    const bf16* px = x + pix * C;
    if (mod && mod_img_stride) {  // per-sample diffusion times: every image has its own modulation vector
      const float* mi = mod + (pix / (static_cast<long long>(H) * W)) * mod_img_stride;
#pragma unroll
      for (int j = 0; j < NCH; ++j)
#pragma unroll
        for (int e = 0; e < VEC; ++e) m[j * VEC + e] = __ldg(mi + j * 32 * VEC + lane * VEC + e);
    }
    float v[NCH * VEC];
#pragma unroll
    for (int j = 0; j < NCH; ++j) {
      const int c0 = j * 32 * VEC + lane * VEC;
      if (VEC == 4) {
        const uint2 r = *reinterpret_cast<const uint2*>(px + c0);
        const float2 a = unpack_bf16x2(r.x), b = unpack_bf16x2(r.y);
        v[j * 4 + 0] = a.x + m[j * 4 + 0];
        v[j * 4 + 1] = a.y + m[j * 4 + 1];
        v[j * 4 + 2] = b.x + m[j * 4 + 2];
        v[j * 4 + 3] = b.y + m[j * 4 + 3];
      } else {
        const float2 a = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(px + c0));
        v[j * 2 + 0] = a.x + m[j * 2 + 0];
        v[j * 2 + 1] = a.y + m[j * 2 + 1];
      }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NCH * VEC; ++i) s += v[i];
    const float mean = warp_sum(s) * (1.0f / C);
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < NCH * VEC; ++i) {
      v[i] -= mean;
      ss += v[i] * v[i];
    }
    const float var = warp_sum(ss) * (1.0f / (C - 1));
    const float inv = 1.0f / sqrtf(var + eps);
    if (inv_out != nullptr && lane == 0) inv_out[pix] = inv;
    long long obase[4];
    int nout = 1;
    if (upsample) {
      const int w = static_cast<int>(pix % W);
      const long long t = pix / W;
      const int h = static_cast<int>(t % H);
      const long long n = t / H;
      const long long o00 = ((n * 2 * H + 2 * h) * 2 * W + 2 * w);
      obase[0] = o00;
      obase[1] = o00 + 1;
      obase[2] = o00 + 2 * W;
      obase[3] = o00 + 2 * W + 1;
      nout = 4;
    } else {
      obase[0] = pix;
    }
#pragma unroll
    for (int j = 0; j < NCH; ++j) {
      const int c0 = j * 32 * VEC + lane * VEC;
      if (VEC == 4) {
        const uint2 o = make_uint2(pack_bf16x2(v[j * 4] * inv, v[j * 4 + 1] * inv),
                                   pack_bf16x2(v[j * 4 + 2] * inv, v[j * 4 + 3] * inv));
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (q < nout) *reinterpret_cast<uint2*>(out + obase[q] * C + c0) = o;
      } else {
        const uint32_t o = pack_bf16x2(v[j * 2] * inv, v[j * 2 + 1] * inv);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (q < nout) *reinterpret_cast<uint32_t*>(out + obase[q] * C + c0) = o;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ K3
// h0 = silu(W0 * [cos(t f), sin(t f)] + b0)      (model/score.py:14-34, :62-63)
// blockIdx.x = sample: t_dev != null reads the sample's own diffusion time (training / DSM loss,
// src/thor/pipelines.py:27-35), else every sample uses the scalar t (sampling).
__global__ void time_embed_kernel(float t_scalar, const float* __restrict__ t_dev, const float* __restrict__ W0,
                                  const float* __restrict__ b0, float* __restrict__ h0_all, int E, int nf) {
  extern __shared__ float e[];
  const float t = t_dev ? t_dev[blockIdx.x] : t_scalar;
  float* h0 = h0_all + static_cast<size_t>(blockIdx.x) * E;
  const int half = nf / 2;
  if (threadIdx.x < half) {
    const float f = expf(-9.210340371976184f * static_cast<float>(threadIdx.x) / static_cast<float>(half));
    const float a = t * f;
    e[threadIdx.x] = cosf(a);
    e[half + threadIdx.x] = sinf(a);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < E; i += blockDim.x) {
    float acc = b0[i];
    for (int j = 0; j < nf; ++j) acc += W0[i * nf + j] * e[j];
    h0[i] = acc / (1.0f + expf(-acc));
  }
}
// y[r] = act(b[r] + W[r, :] . x)   warp per row, float4 lanes.  act: 0 none, 1 SiLU
// blockIdx.y = sample: x and y advance by cols / rows per sample
// add_all (optional): a per-sample vector added before the activation (the forcing term, model/score.py:65-66)
__global__ void matvec_kernel(const float* __restrict__ W, const float* __restrict__ b, const float* __restrict__ x_all,
                              float* __restrict__ y_all, int rows, int cols, int act,
                              const float* __restrict__ add_all = nullptr) {
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= rows) return;
  const float* x = x_all + static_cast<size_t>(blockIdx.y) * cols;
  float* y = y_all + static_cast<size_t>(blockIdx.y) * rows;
  const float4* w4 = reinterpret_cast<const float4*>(W + static_cast<size_t>(row) * cols);
  const float4* x4 = reinterpret_cast<const float4*>(x);
  float acc = 0.f;
  for (int j = lane; j < cols / 4; j += 32) {
    const float4 a = __ldg(w4 + j), v = x4[j];
    acc += a.x * v.x + a.y * v.y + a.z * v.z + a.w * v.w;
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    acc += b[row];
    if (add_all) acc += add_all[static_cast<size_t>(blockIdx.y) * rows + row];
    y[row] = act ? acc / (1.0f + expf(-acc)) : acc;
  }
}
// rows of `cols` floats -> rows of `cols_pad` floats, zero-padded (matvec_kernel reads float4 lanes)
__global__ void pad_rows_kernel(const float* __restrict__ in, float* __restrict__ out, int n, int cols, int cols_pad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * cols_pad) return;
  const int r = i / cols_pad, c = i - r * cols_pad;
  out[i] = c < cols ? in[r * cols + c] : 0.f;
}

// ------------------------------------------------------------------------------------------------ K4
// qkv: bf16 [n*T, 3C] (q | k | v along channels, model/nn.py:74), out: bf16 [n*T, C].
// CTA = (query block of QB, window).  S^T = (K Q^T) / sqrt(C) in fp32 smem, fp32 softmax over keys, O = P V.
// QB = 64 when there are enough windows to fill the SMs, 16 otherwise (4x the CTAs; K and V are re-read from L2).
constexpr int kAttnThreads = 256;
inline size_t attention_smem_bytes(int T, int C, int QB = 64) {
  const size_t pitch = (C + 2) * 2;
  return (QB + 2 * static_cast<size_t>(T)) * pitch + static_cast<size_t>(T) * (QB + 4) * 4;
}
template <int QB>
__global__ void __launch_bounds__(kAttnThreads)
attention_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int T, int C, float scale2) {
  extern __shared__ __align__(128) uint8_t smraw[];
  const int pitch = C + 2;  // bf16 elements; +2 shifts consecutive rows by one bank
  bf16* sq = reinterpret_cast<bf16*>(smraw);
  bf16* sk = sq + QB * pitch;
  bf16* sv = sk + static_cast<size_t>(T) * pitch;
  const int sp = QB + 4;  // pitch of S^T rows (floats), keeps float4 alignment
  float* st = reinterpret_cast<float*>(sv + static_cast<size_t>(T) * pitch);
  const int q0 = blockIdx.x * QB;
  const int nq = min(QB, T - q0);
  const bf16* base = qkv + static_cast<size_t>(blockIdx.y) * T * 3 * C;
  const int tid = threadIdx.x;
  const int c8 = C / 8;
  // ---- load q block, k, v (16 B global reads, 4 B smem writes because of the padded pitch)
  for (int idx = tid; idx < (QB + 2 * T) * c8; idx += kAttnThreads) {
    const int row = idx / c8, g = idx - row * c8;
    const bf16* src;
    bf16* dst;
    bool ok = true;
    if (row < QB) {
      ok = row < nq;
      src = base + static_cast<size_t>(q0 + row) * 3 * C + g * 8;
      dst = sq + row * pitch + g * 8;
    } else if (row < QB + T) {
      const int r = row - QB;
      src = base + static_cast<size_t>(r) * 3 * C + C + g * 8;
      dst = sk + static_cast<size_t>(r) * pitch + g * 8;
    } else {
      const int r = row - QB - T;
      src = base + static_cast<size_t>(r) * 3 * C + 2 * C + g * 8;
      dst = sv + static_cast<size_t>(r) * pitch + g * 8;
    }
    uint4 v = make_uint4(0, 0, 0, 0);
    if (ok) v = *reinterpret_cast<const uint4*>(src);
    uint32_t* d = reinterpret_cast<uint32_t*>(dst);
    d[0] = v.x;
    d[1] = v.y;
    d[2] = v.z;
    d[3] = v.w;
  }
  __syncthreads();
  // ---- S^T[s][tq] = scale2 * q[tq] . k[s]   (MQ x 4 register micro-tiles; 16 query groups x T/4 key groups)
  constexpr int MQ = QB / 16;
  const int tiles = 16 * (T / 4);
  for (int mt = tid; mt < tiles; mt += kAttnThreads) {
    const int tqg = mt % 16, s4 = mt / 16;
    float acc[MQ][4];
#pragma unroll
    for (int i = 0; i < MQ; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const uint32_t* qp = reinterpret_cast<const uint32_t*>(sq + (tqg * MQ) * pitch);
    const uint32_t* kp = reinterpret_cast<const uint32_t*>(sk + static_cast<size_t>(s4 * 4) * pitch);
    const int pw = pitch / 2;
    for (int c = 0; c < C / 2; ++c) {
      float2 qv[MQ], kv[4];
#pragma unroll
      for (int i = 0; i < MQ; ++i) qv[i] = unpack_bf16x2(qp[i * pw + c]);
#pragma unroll
      for (int j = 0; j < 4; ++j) kv[j] = unpack_bf16x2(kp[j * pw + c]);
#pragma unroll
      for (int i = 0; i < MQ; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] += qv[i].x * kv[j].x + qv[i].y * kv[j].y;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int i = 0; i < MQ; ++i) st[(s4 * 4 + j) * sp + tqg * MQ + i] = acc[i][j] * scale2;
  }
  __syncthreads();
  // ---- softmax over keys s for each query column tq (fp32, model/nn.py:82)
  {
    const int warp = tid >> 5, lane = tid & 31;
    for (int tq = warp; tq < QB; tq += kAttnThreads / 32) {
      float mx = -INFINITY;
      for (int s = lane; s < T; s += 32) mx = fmaxf(mx, st[s * sp + tq]);
      mx = warp_max(mx);
      float sum = 0.f;
      for (int s = lane; s < T; s += 32) {
        const float e = expf(st[s * sp + tq] - mx);
        st[s * sp + tq] = e;
        sum += e;
      }
      sum = warp_sum(sum);
      const float inv = 1.0f / sum;
      for (int s = lane; s < T; s += 32) st[s * sp + tq] *= inv;
    }
  }
  __syncthreads();
  // ---- O[tq][c] = sum_s P[tq][s] v[s][c]; thread = (channel pair, 8 queries)
  const int pairs = C / 2;
  for (int item = tid; item < pairs * (QB / 8); item += kAttnThreads) {
    const int c2 = item % pairs, qb = item / pairs;
    float a0[8], a1[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a0[i] = a1[i] = 0.f;
    const uint32_t* vp = reinterpret_cast<const uint32_t*>(sv) + c2;
    const int pw = pitch / 2;
    for (int s = 0; s < T; ++s) {
      const float2 vv = unpack_bf16x2(vp[static_cast<size_t>(s) * pw]);
      const float4 p0 = *reinterpret_cast<const float4*>(st + s * sp + qb * 8);
      const float4 p1 = *reinterpret_cast<const float4*>(st + s * sp + qb * 8 + 4);
      const float pr[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        a0[i] += pr[i] * vv.x;
        a1[i] += pr[i] * vv.y;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int tq = qb * 8 + i;
      if (tq < nq)
        *reinterpret_cast<uint32_t*>(out + (static_cast<size_t>(blockIdx.y) * T + q0 + tq) * C + 2 * c2) =
            pack_bf16x2(a0[i], a1[i]);
    }
  }
}

// ------------------------------------------------------------------------------------------------ layout converters
// fp32 NCHW [F, C, HW]  ->  fp32 [F, HW, C]   (trajectory state layout; C = 4 -> one float4 per pixel)
__global__ void nchw_to_fhwc_kernel(const float* __restrict__ in, float* __restrict__ out, long long F, int C, int hw) {
  const long long total = F * hw;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long f = idx / hw;
    const int pix = static_cast<int>(idx - f * hw);
    for (int c = 0; c < C; ++c) out[idx * C + c] = in[(f * C + c) * hw + pix];
  }
}
__global__ void fhwc_to_nchw_kernel(const float* __restrict__ in, float* __restrict__ out, long long F, int C, int hw) {
  const long long total = F * hw;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long f = idx / hw;
    const int pix = static_cast<int>(idx - f * hw);
    for (int c = 0; c < C; ++c) out[(f * C + c) * hw + pix] = in[idx * C + c];
  }
}
// N4 (SURVEY 8(f)): the step either side of the path, data/pipeline.py:183-272 — per-variable normalisation
// (normalize_ds: (x - shift) / scale, the five modes differ only in which quantiles shift and scale are) fused with the
// layout change ds_to_sorted_np + trajectory packing: per-variable arrays [C][F][hw] (clhw != 0; what xarray holds,
// concatenated) or the sorted-numpy order [F][C][hw] -> device trajectory [F, hw, C].  shift / scale: [C], or [C][hw]
// per-grid-point fields (field != 0).  One thread per pixel: C strided coalesced reads, one contiguous C-vector write.
template <int CT>
__global__ void normalize_pack_kernel(const float* __restrict__ in, float* __restrict__ out, long long F, int C, int hw,
                                      int clhw, const float* __restrict__ shift, const float* __restrict__ scale,
                                      int field) {
  const long long total = F * hw;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long f = idx / hw;
    const int pix = static_cast<int>(idx - f * hw);
    float v[CT > 0 ? CT : 1];
    const int cc = CT > 0 ? CT : C;
#pragma unroll
    for (int c = 0; c < cc; ++c) {
      const float x = in[clhw ? (static_cast<long long>(c) * F + f) * hw + pix : (f * cc + c) * hw + pix];
      const int q = field ? c * hw + pix : c;
      const float y = (x - __ldg(shift + q)) / __ldg(scale + q);  // IEEE division, as the reference divides
      if (CT > 0) v[c] = y;
      else out[idx * cc + c] = y;
    }
    if (CT == 4) *reinterpret_cast<float4*>(out + idx * 4) = make_float4(v[0], v[1], v[2], v[3]);
  }
}
// C = 4, hw % 4 == 0: four pixels per thread — one 16 B load per variable, a register transpose, four 16 B stores
// (64 contiguous bytes per thread): enough bytes in flight to approach the HBM copy rate.
__global__ void normalize_pack4_kernel(const float* __restrict__ in, float* __restrict__ out, long long F, int hw,
                                       int clhw, const float* __restrict__ shift, const float* __restrict__ scale,
                                       int field) {
  const long long total4 = F * hw / 4;
  const int hw4 = hw / 4;
  for (long long i4 = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i4 < total4;
       i4 += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long f = i4 / hw4;
    const int pix = static_cast<int>(i4 - f * hw4) * 4;
    float v[4][4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float4 x = *reinterpret_cast<const float4*>(in + (clhw ? (static_cast<long long>(c) * F + f) * hw + pix
                                                                    : (f * 4 + c) * hw + pix));
      float4 sh, sc;
      if (field) {
        sh = __ldg(reinterpret_cast<const float4*>(shift + c * hw + pix));
        sc = __ldg(reinterpret_cast<const float4*>(scale + c * hw + pix));
      } else {
        const float a = __ldg(shift + c), b = __ldg(scale + c);
        sh = make_float4(a, a, a, a);
        sc = make_float4(b, b, b, b);
      }
      v[0][c] = (x.x - sh.x) / sc.x;
      v[1][c] = (x.y - sh.y) / sc.y;
      v[2][c] = (x.z - sh.z) / sc.z;
      v[3][c] = (x.w - sh.w) / sc.w;
    }
    float4* o = reinterpret_cast<float4*>(out + (f * hw + pix) * 4);
#pragma unroll
    for (int q = 0; q < 4; ++q) o[q] = make_float4(v[q][0], v[q][1], v[q][2], v[q][3]);
  }
}
__global__ void unpack_unnormalize4_kernel(const float* __restrict__ in, float* __restrict__ out, long long F, int hw,
                                           int clhw, const float* __restrict__ shift, const float* __restrict__ scale,
                                           int field) {
  const long long total4 = F * hw / 4;
  const int hw4 = hw / 4;
  for (long long i4 = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i4 < total4;
       i4 += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long f = i4 / hw4;
    const int pix = static_cast<int>(i4 - f * hw4) * 4;
    const float4* x = reinterpret_cast<const float4*>(in + (f * hw + pix) * 4);
    float v[4][4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 t = x[q];
      v[q][0] = t.x, v[q][1] = t.y, v[q][2] = t.z, v[q][3] = t.w;
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float4 sh, sc;
      if (field) {
        sh = __ldg(reinterpret_cast<const float4*>(shift + c * hw + pix));
        sc = __ldg(reinterpret_cast<const float4*>(scale + c * hw + pix));
      } else {
        const float a = __ldg(shift + c), b = __ldg(scale + c);
        sh = make_float4(a, a, a, a);
        sc = make_float4(b, b, b, b);
      }
      const float4 y = make_float4(__fadd_rn(__fmul_rn(v[0][c], sc.x), sh.x), __fadd_rn(__fmul_rn(v[1][c], sc.y), sh.y),
                                   __fadd_rn(__fmul_rn(v[2][c], sc.z), sh.z), __fadd_rn(__fmul_rn(v[3][c], sc.w), sh.w));
      *reinterpret_cast<float4*>(out + (clhw ? (static_cast<long long>(c) * F + f) * hw + pix : (f * 4 + c) * hw + pix)) = y;
    }
  }
}
// unnormalize_ds + np_to_ds: device trajectory [F, hw, C] -> x * scale + shift in per-variable / sorted-numpy order
template <int CT>
__global__ void unpack_unnormalize_kernel(const float* __restrict__ in, float* __restrict__ out, long long F, int C,
                                          int hw, int clhw, const float* __restrict__ shift,
                                          const float* __restrict__ scale, int field) {
  const long long total = F * hw;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long f = idx / hw;
    const int pix = static_cast<int>(idx - f * hw);
    const int cc = CT > 0 ? CT : C;
    float v[CT > 0 ? CT : 1];
    if (CT == 4) {
      const float4 t = *reinterpret_cast<const float4*>(in + idx * 4);
      v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
    }
#pragma unroll
    for (int c = 0; c < cc; ++c) {
      const float x = CT == 4 ? v[c] : in[idx * cc + c];
      const int q = field ? c * hw + pix : c;
      out[clhw ? (static_cast<long long>(c) * F + f) * hw + pix : (f * cc + c) * hw + pix] =
          __fadd_rn(__fmul_rn(x, __ldg(scale + q)), __ldg(shift + q));  // two roundings, as `ds * range + lo`
    }
  }
}
// fp32 NCHW [n, C, HW] -> bf16 [n, HW, cpad] (zero padded channels); smem transpose keeps both sides coalesced
__global__ void nchw_to_nhwc_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, int C, int hw, int cpad) {
  __shared__ float tile[32][33];
  const long long img = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, p = p0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && p < hw) ? in[(img * C + c) * hw + p] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int p = p0 + i, c = c0 + threadIdx.x;
    if (p < hw && c < cpad) out[(img * hw + p) * cpad + c] = __float2bfloat16_rn(tile[threadIdx.x][i]);
  }
}
// fp32 [n, HW, cpad] -> fp32 NCHW [n, C, HW]
__global__ void nhwc_f32_to_nchw_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int hw, int cpad) {
  __shared__ float tile[32][33];
  const long long img = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int p = p0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (p < hw && c < cpad) ? in[(img * hw + p) * cpad + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, p = p0 + threadIdx.x;
    if (c < C && p < hw) out[(img * C + c) * hw + p] = tile[threadIdx.x][i];
  }
}

// ------------------------------------------------------------------------------------------------ K4 (tensor cores)
// Attention core for T = 64 tokens (the reference's 8 x 8 attention level) on warp-level tensor-core MMAs
// (mma.sync m16n8k16, bf16 in, fp32 accumulate): 0.04 % of the UNet's FLOPs, so the legacy warp MMA is plenty — the
// point is to get it off the CUDA cores, where it cost 5 % of a step.  One CTA per window:
//   cp.async q, k, v [64, C] -> shared (16 B chunks XOR-swizzled by row for conflict-free ldmatrix)
//   warps 0-3: S = scale2 q k^T for 16 query rows each, fp32 softmax in registers, P -> shared (bf16)
//   warps 0-7: O = P v for 16 rows x C/2 channels each, bf16 -> global
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
inline size_t attention_mma_smem_bytes(int C) { return static_cast<size_t>(3) * 64 * C * 2 + 64 * 64 * 2; }
template <int C>
__global__ void __launch_bounds__(256) attention_mma_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out,
                                                            float scale2) {
  constexpr int T = 64, CH = C / 8, PITCH = C * 2;  // CH: 16 B chunks per row
  extern __shared__ __align__(128) uint8_t smraw[];
  const uint32_t sQ = static_cast<uint32_t>(__cvta_generic_to_shared(smraw));
  const uint32_t sK = sQ + T * PITCH, sV = sK + T * PITCH, sP = sV + T * PITCH;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bf16* src = qkv + static_cast<size_t>(blockIdx.x) * T * 3 * C;
  for (int idx = tid; idx < 3 * T * CH; idx += 256) {
    const int which = idx / (T * CH), rem = idx - which * (T * CH);
    const int r = rem / CH, cc = rem - r * CH;
    const uint32_t dst = sQ + which * (T * PITCH) + r * PITCH + ((cc ^ (r & 7)) << 4);
    const bf16* g = src + static_cast<size_t>(r) * 3 * C + which * C + cc * 8;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(g) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  const int mat = lane >> 3, rr = lane & 7;  // ldmatrix: lane -> (8x8 matrix, row)
  const int g = lane >> 2, tq = lane & 3;    // mma fragments: row group, column pair
  if (warp < 4) {
    const int r0 = 16 * warp;
    float acc[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] = 0.f;
    const int arow = r0 + rr + (mat & 1) * 8;
#pragma unroll 4
    for (int ks = 0; ks < C / 16; ++ks) {
      uint32_t a[4];
      ldmatrix_x4(a, sQ + arow * PITCH + (((2 * ks + (mat >> 1)) ^ (arow & 7)) << 4));
#pragma unroll
      for (int jp = 0; jp < 4; ++jp) {  // key tiles 2 jp, 2 jp + 1
        const int key = 16 * jp + rr + (mat >> 1) * 8;
        uint32_t b[4];
        ldmatrix_x4(b, sK + key * PITCH + (((2 * ks + (mat & 1)) ^ (key & 7)) << 4));
        mma_bf16_16816(acc[2 * jp], a, b[0], b[1]);
        mma_bf16_16816(acc[2 * jp + 1], a, b[2], b[3]);
      }
    }
    // fp32 softmax over the 64 keys of rows g and g + 8 (model/nn.py:82); a row lives in the 4 lanes of a quad
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] *= scale2;
      m0 = fmaxf(m0, fmaxf(acc[j][0], acc[j][1]));
      m1 = fmaxf(m1, fmaxf(acc[j][2], acc[j][3]));
    }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc[j][0] = expf(acc[j][0] - m0);
      acc[j][1] = expf(acc[j][1] - m0);
      acc[j][2] = expf(acc[j][2] - m1);
      acc[j][3] = expf(acc[j][3] - m1);
      s0 += acc[j][0] + acc[j][1];
      s1 += acc[j][2] + acc[j][3];
    }
    s0 += __shfl_xor_sync(0xffffffffu, s0, 1);
    s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
    s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
    s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
    const float i0 = 1.0f / s0, i1 = 1.0f / s1;
    const int row0 = r0 + g, row1 = r0 + g + 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) {  // P[row][8 j + 2 tq, +1] (bf16): chunk j of the 128 B row, swizzled
      const uint32_t p0 = pack_bf16x2(acc[j][0] * i0, acc[j][1] * i0), p1 = pack_bf16x2(acc[j][2] * i1, acc[j][3] * i1);
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sP + row0 * 128 + ((j ^ (row0 & 7)) << 4) + tq * 4), "r"(p0) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sP + row1 * 128 + ((j ^ (row1 & 7)) << 4) + tq * 4), "r"(p1) : "memory");
    }
  }
  __syncthreads();
  {
    const int r0 = 16 * (warp & 3), cbase = (warp >> 2) * (C / 2);
    const int arow = r0 + rr + (mat & 1) * 8;
    uint32_t pa[4][4];  // P fragments of the 4 k-steps over the 64 keys
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) ldmatrix_x4(pa[ks], sP + arow * 128 + (((2 * ks + (mat >> 1)) ^ (arow & 7)) << 4));
    bf16* orow0 = out + (static_cast<size_t>(blockIdx.x) * T + r0 + g) * C;
    bf16* orow1 = orow0 + static_cast<size_t>(8) * C;
#pragma unroll 1
    for (int grp = 0; grp < C / 128; ++grp) {  // 64 channels at a time
      const int c0 = cbase + 64 * grp;
      float acc[8][4];
#pragma unroll
      for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[j][e] = 0.f;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const int key = 16 * ks + rr + (mat & 1) * 8;
#pragma unroll
        for (int jp = 0; jp < 4; ++jp) {  // channel tiles 2 jp, 2 jp + 1
          const int chunk = (c0 >> 3) + 2 * jp + (mat >> 1);
          uint32_t b[4];
          ldmatrix_x4_trans(b, sV + key * PITCH + ((chunk ^ (key & 7)) << 4));
          mma_bf16_16816(acc[2 * jp], pa[ks], b[0], b[1]);
          mma_bf16_16816(acc[2 * jp + 1], pa[ks], b[2], b[3]);
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int col = c0 + 8 * j + 2 * tq;
        *reinterpret_cast<uint32_t*>(orow0 + col) = pack_bf16x2(acc[j][0], acc[j][1]);
        *reinterpret_cast<uint32_t*>(orow1 + col) = pack_bf16x2(acc[j][2], acc[j][3]);
      }
    }
  }
}

// ---- backward of the T = 64 attention core on the same warp MMAs (exact_grad / training: K8)
//   P = softmax(scale2 q k^T),  gP = go v^T,  gS = P o (gP - rowsum(gP o P)),
//   gq = scale2 gS k,  gk = scale2 gS^T q,  gv = P^T go            (model/nn.py:79-84 differentiated)
// One CTA (8 warps) per window, three [64, C] operand slots in shared memory (same XOR-swizzled 16 B chunks as the
// forward kernel) that q, k, v, go rotate through, P and scale2 gS as bf16 [64, 64] tiles for the three output GEMMs:
//   slots {q, k, v}:  warps 0-3: S, softmax -> P in registers
//   slots {go, k, v}: warps 0-3: gP -> gS; P, gS -> shared
//   slots {go, k, q}: all warps: gv = P^T go, gq = gS k, then gk = gS^T q (q reloaded under the first two)
template <int C>
__device__ __forceinline__ void attn_slot_load(uint32_t sdst, const bf16* src, int row_stride, int tid) {
  constexpr int CH = C / 8, PITCH = C * 2;
  for (int idx = tid; idx < 64 * CH; idx += 256) {
    const int r = idx / CH, cc = idx - r * CH;
    const uint32_t dst = sdst + r * PITCH + ((cc ^ (r & 7)) << 4);
    const bf16* g = src + static_cast<size_t>(r) * row_stride + cc * 8;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(g) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}
// acc[16 rows r0.. of A][64 rows of B] = A[.][:] . B[.][:] over the C channels (both [64, C] slots)
template <int C>
__device__ __forceinline__ void attn_rows_dot_rows(float (&acc)[8][4], uint32_t sA, uint32_t sB, int r0, int lane) {
  constexpr int PITCH = C * 2;
  const int mat = lane >> 3, rr = lane & 7;
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[j][e] = 0.f;
  const int arow = r0 + rr + (mat & 1) * 8;
#pragma unroll 4
  for (int ks = 0; ks < C / 16; ++ks) {
    uint32_t a[4];
    ldmatrix_x4(a, sA + arow * PITCH + (((2 * ks + (mat >> 1)) ^ (arow & 7)) << 4));
#pragma unroll
    for (int jp = 0; jp < 4; ++jp) {
      const int key = 16 * jp + rr + (mat >> 1) * 8;
      uint32_t b[4];
      ldmatrix_x4(b, sB + key * PITCH + (((2 * ks + (mat & 1)) ^ (key & 7)) << 4));
      mma_bf16_16816(acc[2 * jp], a, b[0], b[1]);
      mma_bf16_16816(acc[2 * jp + 1], a, b[2], b[3]);
    }
  }
}
// out[r0 + 16 rows][cbase + C/2 channels] = M' [64 x 64] . X [64, C]; M' = M (TRANS = false) or M^T (TRANS = true),
// M a bf16 [64][64] tile (128 B rows, swizzled chunks), X a [64, C] slot; rows of `out` are 3C apart (the qkv gradient).
template <int C, bool TRANS>
__device__ __forceinline__ void attn_tile_times_slot(bf16* out, uint32_t sM, uint32_t sX, int r0, int cbase, int lane) {
  constexpr int PITCH = C * 2;
  const int mat = lane >> 3, rr = lane & 7, g = lane >> 2, tq = lane & 3;
  uint32_t ma[4][4];  // A fragments of the 4 k-steps over the 64 summed rows
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    if (!TRANS) {
      const int arow = r0 + rr + (mat & 1) * 8;
      ldmatrix_x4(ma[ks], sM + arow * 128 + (((2 * ks + (mat >> 1)) ^ (arow & 7)) << 4));
    } else {  // A[m][k] = M[k][m]: 8 x 8 blocks of M read transposed
      const int krow = 16 * ks + rr + (mat >> 1) * 8;
      ldmatrix_x4_trans(ma[ks], sM + krow * 128 + ((((r0 >> 3) + (mat & 1)) ^ (krow & 7)) << 4));
    }
  }
  bf16* orow0 = out + static_cast<size_t>(r0 + g) * 3 * C;
  bf16* orow1 = orow0 + static_cast<size_t>(8) * 3 * C;
#pragma unroll 1
  for (int grp = 0; grp < C / 128; ++grp) {  // 64 channels at a time
    const int c0 = cbase + 64 * grp;
    float acc[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const int key = 16 * ks + rr + (mat & 1) * 8;
#pragma unroll
      for (int jp = 0; jp < 4; ++jp) {
        const int chunk = (c0 >> 3) + 2 * jp + (mat >> 1);
        uint32_t b[4];
        ldmatrix_x4_trans(b, sX + key * PITCH + ((chunk ^ (key & 7)) << 4));
        mma_bf16_16816(acc[2 * jp], ma[ks], b[0], b[1]);
        mma_bf16_16816(acc[2 * jp + 1], ma[ks], b[2], b[3]);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = c0 + 8 * j + 2 * tq;
      *reinterpret_cast<uint32_t*>(orow0 + col) = pack_bf16x2(acc[j][0], acc[j][1]);
      *reinterpret_cast<uint32_t*>(orow1 + col) = pack_bf16x2(acc[j][2], acc[j][3]);
    }
  }
}
inline size_t attention_bwd_mma_smem_bytes(int C) { return static_cast<size_t>(3) * 64 * C * 2 + 2 * 64 * 64 * 2; }
template <int C>
__global__ void __launch_bounds__(256) attention_bwd_mma_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ go,
                                                                bf16* __restrict__ gqkv, float scale2) {
  constexpr int T = 64, PITCH = C * 2;
  extern __shared__ __align__(128) uint8_t smraw[];
  const uint32_t s0 = static_cast<uint32_t>(__cvta_generic_to_shared(smraw));
  const uint32_t s1 = s0 + T * PITCH, s2 = s1 + T * PITCH, sP = s2 + T * PITCH, sG = sP + T * 128;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bf16* src = qkv + static_cast<size_t>(blockIdx.x) * T * 3 * C;
  const bf16* gsrc = go + static_cast<size_t>(blockIdx.x) * T * C;
  bf16* dst = gqkv + static_cast<size_t>(blockIdx.x) * T * 3 * C;
  attn_slot_load<C>(s0, src, 3 * C, tid);          // q
  attn_slot_load<C>(s1, src + C, 3 * C, tid);      // k
  attn_slot_load<C>(s2, src + 2 * C, 3 * C, tid);  // v
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  const int g = lane >> 2, tq = lane & 3;
  const int r0 = 16 * (warp & 3);
  float p[8][4];
  if (warp < 4) {
    attn_rows_dot_rows<C>(p, s0, s1, r0, lane);  // S
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
#pragma unroll
      for (int e = 0; e < 4; ++e) p[j][e] *= scale2;
      m0 = fmaxf(m0, fmaxf(p[j][0], p[j][1]));
      m1 = fmaxf(m1, fmaxf(p[j][2], p[j][3]));
    }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      p[j][0] = expf(p[j][0] - m0);
      p[j][1] = expf(p[j][1] - m0);
      p[j][2] = expf(p[j][2] - m1);
      p[j][3] = expf(p[j][3] - m1);
      sum0 += p[j][0] + p[j][1];
      sum1 += p[j][2] + p[j][3];
    }
    sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
    sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
    sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
    sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
    const float i0 = 1.0f / sum0, i1 = 1.0f / sum1;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      p[j][0] *= i0;
      p[j][1] *= i0;
      p[j][2] *= i1;
      p[j][3] *= i1;
    }
  }
  __syncthreads();                        // every warp is done with q
  attn_slot_load<C>(s0, gsrc, C, tid);    // go over q
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  if (warp < 4) {
    float gp[8][4];
    attn_rows_dot_rows<C>(gp, s0, s2, r0, lane);  // gP = go v^T
    float d0 = 0.f, d1 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      d0 += gp[j][0] * p[j][0] + gp[j][1] * p[j][1];
      d1 += gp[j][2] * p[j][2] + gp[j][3] * p[j][3];
    }
    d0 += __shfl_xor_sync(0xffffffffu, d0, 1);
    d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 1);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
    const int row0 = r0 + g, row1 = r0 + g + 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) {  // [row][8 j + 2 tq, +1] (bf16): chunk j of the 128 B row, swizzled
      const uint32_t o0 = (row0 * 128 + ((j ^ (row0 & 7)) << 4) + tq * 4), o1 = (row1 * 128 + ((j ^ (row1 & 7)) << 4) + tq * 4);
      const uint32_t p0 = pack_bf16x2(p[j][0], p[j][1]), p1 = pack_bf16x2(p[j][2], p[j][3]);
      const uint32_t g0 = pack_bf16x2(scale2 * p[j][0] * (gp[j][0] - d0), scale2 * p[j][1] * (gp[j][1] - d0));
      const uint32_t g1 = pack_bf16x2(scale2 * p[j][2] * (gp[j][2] - d1), scale2 * p[j][3] * (gp[j][3] - d1));
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sP + o0), "r"(p0) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sP + o1), "r"(p1) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sG + o0), "r"(g0) : "memory");
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(sG + o1), "r"(g1) : "memory");
    }
  }
  __syncthreads();                                 // P, gS visible; v is dead
  attn_slot_load<C>(s2, src, 3 * C, tid);          // q over v, under the next two products
  const int cbase = (warp >> 2) * (C / 2);
  attn_tile_times_slot<C, true>(dst + 2 * C, sP, s0, r0, cbase, lane);   // gv = P^T go
  attn_tile_times_slot<C, false>(dst, sG, s1, r0, cbase, lane);          // gq = scale2 gS k
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  attn_tile_times_slot<C, true>(dst + C, sG, s2, r0, cbase, lane);       // gk = scale2 gS^T q
}

// ------------------------------------------------------------------------------------------------ VJP kernels
// Backward of the channel LayerNorm (model/nn.py:154,183; zuko LayerNorm, unbiased variance):
//   g_v = inv * (g_y - mean_C(g_y) - y * sum_C(g_y y) / (C - 1)),   out = gres + g_v
// y is the stashed normalised output, inv the stashed 1/sqrt(var + eps).  down != 0: the LayerNorm output had been
// nearest-upsampled 2x (model/nn.py:184): g_y is the sum of the 2x2 block of gy [n, 2H, 2W, C] and y is read from
// the block's first pixel.  One warp per pixel, same lane -> channel mapping as the forward kernel.
// dmod != null (training): every CTA owns a contiguous chunk of `chunk` pixels of ONE image and also accumulates the
// per-image column sums of g_v — the gradient w.r.t. the block's modulation vector mod = Linear(emb) (model/nn.py:27,
// v = x + mod[:, :, None, None]) — in registers (the lane -> channel mapping is fixed), reduced over the CTA's warps in
// shared memory and added to dmod[image * dmod_stride + c] with one atomic per channel per CTA.
template <int C>
__global__ void channel_layernorm_bwd_kernel(const bf16* __restrict__ gy, const bf16* __restrict__ y,
                                             const float* __restrict__ inv, const bf16* gres, bf16* out,
                                             long long npix, int H, int W, int down, float* dmod = nullptr,
                                             int dmod_stride = 0, int pix_per_img = 1, int chunk = 0) {
  constexpr int VEC = (C % 128 == 0) ? 4 : 2;
  constexpr int NCH = C / (32 * VEC);
  const int lane = threadIdx.x & 31;
  long long warp0 = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  long long pix_end = npix;
  float macc[NCH * VEC];
#pragma unroll
  for (int i = 0; i < NCH * VEC; ++i) macc[i] = 0.f;
  if (dmod != nullptr) {
    warp0 = static_cast<long long>(blockIdx.x) * chunk + (threadIdx.x >> 5);
    nwarps = blockDim.x >> 5;
    pix_end = static_cast<long long>(blockIdx.x + 1) * chunk;
    if (pix_end > npix) pix_end = npix;
  }
  for (long long pix = warp0; pix < pix_end; pix += nwarps) {
    long long src[4];
    int nsrc = 1;
    if (down) {
      const int w = static_cast<int>(pix % W);
      const long long t = pix / W;
      const int h = static_cast<int>(t % H);
      const long long n = t / H;
      const long long o00 = ((n * 2 * H + 2 * h) * 2 * W + 2 * w);
      src[0] = o00;
      src[1] = o00 + 1;
      src[2] = o00 + 2 * W;
      src[3] = o00 + 2 * W + 1;
      nsrc = 4;
    } else {
      src[0] = pix;
    }
    float g[NCH * VEC], yv[NCH * VEC];
#pragma unroll
    for (int i = 0; i < NCH * VEC; ++i) g[i] = 0.f;
#pragma unroll
    for (int j = 0; j < NCH; ++j) {
      const int c0 = j * 32 * VEC + lane * VEC;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (q < nsrc) {
          if (VEC == 4) {
            const uint2 r = *reinterpret_cast<const uint2*>(gy + src[q] * C + c0);
            const float2 a = unpack_bf16x2(r.x), b = unpack_bf16x2(r.y);
            g[j * 4 + 0] += a.x;
            g[j * 4 + 1] += a.y;
            g[j * 4 + 2] += b.x;
            g[j * 4 + 3] += b.y;
          } else {
            const float2 a = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(gy + src[q] * C + c0));
            g[j * 2 + 0] += a.x;
            g[j * 2 + 1] += a.y;
          }
        }
      }
      const bf16* yp = y + src[0] * C + c0;
      if (VEC == 4) {
        const uint2 r = *reinterpret_cast<const uint2*>(yp);
        const float2 a = unpack_bf16x2(r.x), b = unpack_bf16x2(r.y);
        yv[j * 4 + 0] = a.x;
        yv[j * 4 + 1] = a.y;
        yv[j * 4 + 2] = b.x;
        yv[j * 4 + 3] = b.y;
      } else {
        const float2 a = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(yp));
        yv[j * 2 + 0] = a.x;
        yv[j * 2 + 1] = a.y;
      }
    }
    float s = 0.f, sy = 0.f;
#pragma unroll
    for (int i = 0; i < NCH * VEC; ++i) {
      s += g[i];
      sy += g[i] * yv[i];
    }
    s = warp_sum(s) * (1.0f / C);
    sy = warp_sum(sy) * (1.0f / (C - 1));
    const float iv = inv[pix];
#pragma unroll
    for (int j = 0; j < NCH; ++j) {
      const int c0 = j * 32 * VEC + lane * VEC;
      float o[VEC];
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        o[e] = iv * (g[j * VEC + e] - s - yv[j * VEC + e] * sy);
        macc[j * VEC + e] += o[e];
      }
      if (gres != nullptr) {
        if (VEC == 4) {
          const uint2 r = *reinterpret_cast<const uint2*>(gres + pix * C + c0);
          const float2 a = unpack_bf16x2(r.x), b = unpack_bf16x2(r.y);
          o[0] += a.x;
          o[1] += a.y;
          o[2] += b.x;
          o[3] += b.y;
        } else {
          const float2 a = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(gres + pix * C + c0));
          o[0] += a.x;
          o[1] += a.y;
        }
      }
      if (VEC == 4)
        *reinterpret_cast<uint2*>(out + pix * C + c0) = make_uint2(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]));
      else
        *reinterpret_cast<uint32_t*>(out + pix * C + c0) = pack_bf16x2(o[0], o[1]);
    }
  }
  if (dmod != nullptr) {
    __shared__ float red[8][C];
    const int w = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < NCH; ++j)
#pragma unroll
      for (int e = 0; e < VEC; ++e) red[w][j * 32 * VEC + lane * VEC + e] = macc[j * VEC + e];
    __syncthreads();
    const long long img = (static_cast<long long>(blockIdx.x) * chunk) / pix_per_img;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float v = 0.f;
      for (int q = 0; q < (blockDim.x >> 5); ++q) v += red[q][c];
      atomicAdd(dmod + img * dmod_stride + c, v);
    }
  }
}

// ------------------------------------------------------------------------------------------------ training: time MLP
// Small fp32 kernels of the modulation / time-embedding backward (model/score.py:59-67, model/nn.py:149): a few GFLOP
// per step against ~45 TFLOP of convolutions — one thread per output element, coalesced along the output's last axis.
//   C[m][n] (+)= sum_k A[k][m] * B[k][n]        (dW = dpre^T . input, summed over the batch)
__global__ void gemm_tn_f32_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb,
                                   float* __restrict__ Cm, int ldc, int K, int M, int N, int accumulate) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(M) * N) return;
  const int m = static_cast<int>(i / N), n = static_cast<int>(i - static_cast<long long>(m) * N);
  float acc = 0.f;
  for (int k = 0; k < K; ++k) acc = fmaf(A[static_cast<size_t>(k) * lda + m], B[static_cast<size_t>(k) * ldb + n], acc);
  float* d = Cm + static_cast<size_t>(m) * ldc + n;
  *d = accumulate ? *d + acc : acc;
}
//   C[m][n] (+)= sum_k A[m][k] * B[k][n]          (d input = dpre . W); gridDim.y > 1 splits K and adds atomically
//   into a ZEROED C (the long reduction over all modulation channels would otherwise run on 64 K threads only)
__global__ void gemm_nn_f32_kernel(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb,
                                   float* __restrict__ Cm, int ldc, int M, int K, int N) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(M) * N) return;
  const int m = static_cast<int>(i / N), n = static_cast<int>(i - static_cast<long long>(m) * N);
  const int kper = (K + gridDim.y - 1) / gridDim.y;
  const int k0 = blockIdx.y * kper, k1 = (k0 + kper < K) ? k0 + kper : K;
  float acc = 0.f;
  for (int k = k0; k < k1; ++k) acc = fmaf(A[static_cast<size_t>(m) * lda + k], B[static_cast<size_t>(k) * ldb + n], acc);
  float* d = Cm + static_cast<size_t>(m) * ldc + n;
  if (gridDim.y > 1) atomicAdd(d, acc);
  else *d = acc;
}
// All modulation projections at once (model/nn.py:149, 30 Linear layers): row m of dmods^T . emb is one output channel
// of one block's `project` weight and goes to its own place in the flat gradient buffer:
//   grad[row_w[m] + e] += sum_s dmods[s][m] * emb[s][e]      grad[row_b[m]] += sum_s dmods[s][m]
__global__ void proj_grad_kernel(const float* __restrict__ dmods, int TM, const float* __restrict__ emb, int E, int ns,
                                 float* __restrict__ grad, const long long* __restrict__ row_w,
                                 const long long* __restrict__ row_b) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(TM) * E) return;
  const int m = static_cast<int>(i / E), e = static_cast<int>(i - static_cast<long long>(m) * E);
  float acc = 0.f, bsum = 0.f;
  for (int sidx = 0; sidx < ns; ++sidx) {
    const float d = dmods[static_cast<size_t>(sidx) * TM + m];
    acc = fmaf(d, emb[static_cast<size_t>(sidx) * E + e], acc);
    bsum += d;
  }
  if (row_w[m] >= 0) grad[row_w[m] + e] += acc;
  if (e == 0 && row_b[m] >= 0) grad[row_b[m]] += bsum;
}
//   out[m] (+)= sum_k A[k][m]                    (bias gradients)
__global__ void colsum_f32_kernel(const float* __restrict__ A, int lda, float* __restrict__ out, int K, int M, int accumulate) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  float acc = 0.f;
  for (int k = 0; k < K; ++k) acc += A[static_cast<size_t>(k) * lda + m];
  out[m] = accumulate ? out[m] + acc : acc;
}
//   g <- g * silu'(pre)
__global__ void dsilu_f32_kernel(float* __restrict__ g, const float* __restrict__ pre, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = pre[i], sg = 1.0f / (1.0f + expf(-x));
  g[i] *= sg * (1.0f + x * (1.0f - sg));
}
// Sinusoidal features of the diffusion times (model/score.py:14-34): feat[s] = [cos(t f_j), sin(t f_j)], f_j as in
// time_embed_kernel (which fuses them with the first Linear and does not store them).
__global__ void time_features_kernel(const float* __restrict__ t_dev, float* __restrict__ feat, int nf) {
  const int half = nf / 2;
  const float t = t_dev[blockIdx.x];
  if (threadIdx.x < half) {
    const float f = expf(-9.210340371976184f * static_cast<float>(threadIdx.x) / static_cast<float>(half));
    feat[static_cast<size_t>(blockIdx.x) * nf + threadIdx.x] = cosf(t * f);
    feat[static_cast<size_t>(blockIdx.x) * nf + half + threadIdx.x] = sinf(t * f);
  }
}
// Denoising-score-matching objective and its cotangent in one pass (src/thor/pipelines.py:27-35 followed by the
// caller's `.mean()`, training_loop.py:377):  loss = mean((out - eps)^2) * loss_scale,
//   gout = 2 (out - eps) * loss_scale / n   (what autograd hands the network), per-CTA partial sums of (out - eps)^2.
__global__ void dsm_loss_grad_kernel(const float* __restrict__ out, const float* __restrict__ eps, float* __restrict__ gout,
                                     float* __restrict__ partials, long long n, float gscale) {
  float acc = 0.f;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float d = out[i] - eps[i];
    acc = fmaf(d, d, acc);
    gout[i] = d * gscale;
  }
  __shared__ float wsum[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = (threadIdx.x < (blockDim.x >> 5)) ? wsum[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) partials[blockIdx.x] = v;
  }
}

// Device-side re-pack of the weights after an optimiser step.  A conv: fp32 OIHW (torch layout, in the flat parameter
// buffer) -> the bf16 forward operand [cout_pad][taps * cin_pad] (k = tap * cin_pad + c) and the flipped / transposed
// input-gradient operand [cin_pad][taps * cout_pad] (k = (taps - 1 - tap) * cout_pad + o); padding entries stay zero.
// The whole re-pack as ONE launch: a table of jobs (every conv's weights, every bias / projection / MLP copy, the
// zero-padded forcing rows), 1024 elements per block step; `first_chunk[j]` = index of job j's first 1024-element chunk.
struct RefreshJob {
  long long src;   // offset in the flat fp32 parameter buffer
  long long n;     // copy: floats; padded rows: rows * cols_pad; conv: unused
  bf16* wp;        // conv: forward operand
  bf16* wd;        // conv: input-gradient operand
  float* fdst;     // copy / padded rows: destination
  int kind;        // 0 conv weights, 1 fp32 copy, 2 rows of `cin` floats padded to `cin_pad`
  int cout, cin, taps, cin_pad, cout_pad;
  int chunks;      // conv: ceil(cout / 32) * ceil(cin / 32) tiles; else ceil(n / 1024)
};
constexpr int kRefreshChunk = 1024;
constexpr int kRefreshTile = 32;  // conv jobs: [32 output x 32 input channels x taps] tiles through shared memory
__global__ void __launch_bounds__(256)
refresh_weights_kernel(const RefreshJob* __restrict__ jobs, const int* __restrict__ first_chunk, int n_jobs, int n_chunks,
                       const float* __restrict__ flat) {
  __shared__ float tile[kRefreshTile][kRefreshTile * 9 + 1];  // [o][c * taps + t], taps <= 9
  for (int ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
    int lo = 0, hi = n_jobs - 1;  // last job whose first chunk <= ch
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (first_chunk[mid] <= ch) lo = mid;
      else hi = mid - 1;
    }
    const RefreshJob jb = jobs[lo];
    const float* src = flat + jb.src;
    const int local = ch - first_chunk[lo];
    if (jb.kind == 0) {
      // tile (ob, cb): rows of 32 * taps contiguous floats in, 64-byte runs of c (forward operand) and o (gradient
      // operand) out — the element-wise version wrote 2-byte values 2 * K bytes apart
      const int c_tiles = (jb.cin + kRefreshTile - 1) / kRefreshTile;
      const int o0 = (local / c_tiles) * kRefreshTile, c0 = (local % c_tiles) * kRefreshTile;
      const int no = min(kRefreshTile, jb.cout - o0), nc = min(kRefreshTile, jb.cin - c0);
      const int run = nc * jb.taps;
      for (int k = threadIdx.x; k < no * run; k += blockDim.x) {
        const int o = k / run, r = k - o * run;
        tile[o][r] = src[(static_cast<long long>(o0 + o) * jb.cin + c0) * jb.taps + r];
      }
      __syncthreads();
      const size_t K = static_cast<size_t>(jb.taps) * jb.cin_pad, Kd = static_cast<size_t>(jb.taps) * jb.cout_pad;
      for (int k = threadIdx.x; k < no * jb.taps * nc; k += blockDim.x) {  // (o, t, c), c fastest
        const int c = k % nc, ot = k / nc, t = ot % jb.taps, o = ot / jb.taps;
        jb.wp[(o0 + o) * K + static_cast<size_t>(t) * jb.cin_pad + c0 + c] = __float2bfloat16_rn(tile[o][c * jb.taps + t]);
      }
      for (int k = threadIdx.x; k < nc * jb.taps * no; k += blockDim.x) {  // (c, t, o), o fastest
        const int o = k % no, ct = k / no, t = ct % jb.taps, c = ct / jb.taps;
        jb.wd[(c0 + c) * Kd + static_cast<size_t>(jb.taps - 1 - t) * jb.cout_pad + o0 + o] =
            __float2bfloat16_rn(tile[o][c * jb.taps + t]);
      }
      __syncthreads();
      continue;
    }
    const long long i0 = static_cast<long long>(local) * kRefreshChunk;
    for (int k = threadIdx.x; k < kRefreshChunk; k += blockDim.x) {
      const long long i = i0 + k;
      if (i >= jb.n) break;
      if (jb.kind == 1) {
        jb.fdst[i] = src[i];
      } else {
        const int r = static_cast<int>(i / jb.cin_pad), c = static_cast<int>(i - static_cast<long long>(r) * jb.cin_pad);
        jb.fdst[i] = c < jb.cin ? src[static_cast<long long>(r) * jb.cin + c] : 0.f;
      }
    }
  }
}

// Backward of the attention core (model/nn.py:74-85).  qkv: bf16 [n*T, 3C] (stash), go: bf16 [n*T, C] (gradient w.r.t.
// the attention output), gqkv: bf16 [n*T, 3C].
//   S = scale2 q k^T, P = softmax_s(S), o = P v
//   gv = P^T go ; gP = go v^T ; gS = P * (gP - rowsum(gP * P)) ; gq = scale2 gS k ; gk = scale2 gS^T q
// Two kernels: (1) per (query block, window): P and gS rows -> fp32 scratch [n, T, T];  (2) per (row block, window,
// {q, k, v}): the three products against k, q, go.
constexpr int kAttnBwdRows = 64;
inline size_t attention_bwd_scores_smem(int T, int C, int QB) {
  return (static_cast<size_t>(T) + QB) * (C + 2) * 2 + 2 * static_cast<size_t>(QB) * (T + 1) * 4;
}
inline size_t attention_bwd_grads_smem(int T, int C, int RB) {
  return static_cast<size_t>(T) * (C + 2) * 2 + static_cast<size_t>(RB) * (T + 1) * 4;
}
// dst[r][pitch] <- src[(row0 + r) * ld + coff + c], r < rows
__device__ __forceinline__ void attn_load_tile(bf16* dst, const bf16* src, size_t row0, int rows, int ld, int coff, int C,
                                               int pitch) {
  const int c8 = C / 8;
  for (int idx = threadIdx.x; idx < rows * c8; idx += kAttnThreads) {
    const int r = idx / c8, g = idx - r * c8;
    const uint4 v = *reinterpret_cast<const uint4*>(src + (row0 + r) * ld + coff + g * 8);
    uint32_t* d = reinterpret_cast<uint32_t*>(dst + static_cast<size_t>(r) * pitch + g * 8);
    d[0] = v.x;
    d[1] = v.y;
    d[2] = v.z;
    d[3] = v.w;
  }
}
// out[i][j] = scale * sum_c a[i][c] * b[j][c],  i < rows_a, j < T  (tiles [.][pitch] bf16; out [.][sp] fp32)
__device__ __forceinline__ void attn_abt(const bf16* a, const bf16* b, float* out, int rows_a, int T, int C, int pitch,
                                         int sp, float scale) {
  const int pw = pitch / 2;
  for (int item = threadIdx.x; item < rows_a * (T / 4); item += kAttnThreads) {
    const int i = item / (T / 4), j4 = (item - i * (T / 4)) * 4;
    const uint32_t* ap = reinterpret_cast<const uint32_t*>(a + static_cast<size_t>(i) * pitch);
    const uint32_t* bp = reinterpret_cast<const uint32_t*>(b + static_cast<size_t>(j4) * pitch);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int c = 0; c < C / 2; ++c) {
      const float2 av = unpack_bf16x2(ap[c]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 bv = unpack_bf16x2(bp[j * pw + c]);
        acc[j] += av.x * bv.x + av.y * bv.y;
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) out[i * sp + j4 + j] = acc[j] * scale;
  }
}
__global__ void __launch_bounds__(kAttnThreads)
attention_bwd_scores_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ go, float* __restrict__ Pm,
                            float* __restrict__ gSm, int T, int C, int QB, float scale2) {
  extern __shared__ __align__(128) uint8_t smraw[];
  const int pitch = C + 2, sp = T + 1;
  bf16* sx = reinterpret_cast<bf16*>(smraw);                  // [T][pitch]: k, then v
  bf16* sq = sx + static_cast<size_t>(T) * pitch;             // [QB][pitch]: q block, then go block
  float* P = reinterpret_cast<float*>(sq + static_cast<size_t>(QB) * pitch);
  float* gS = P + static_cast<size_t>(QB) * sp;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const size_t row0 = static_cast<size_t>(blockIdx.y) * T;
  const int i0 = blockIdx.x * QB;
  const int nq = min(QB, T - i0);
  attn_load_tile(sx, qkv, row0, T, 3 * C, C, C, pitch);
  attn_load_tile(sq, qkv, row0 + i0, nq, 3 * C, 0, C, pitch);
  __syncthreads();
  attn_abt(sq, sx, P, nq, T, C, pitch, sp, scale2);
  __syncthreads();
  for (int i = warp; i < nq; i += kAttnThreads / 32) {
    float mx = -INFINITY;
    for (int j = lane; j < T; j += 32) mx = fmaxf(mx, P[i * sp + j]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < T; j += 32) {
      const float e = expf(P[i * sp + j] - mx);
      P[i * sp + j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    for (int j = lane; j < T; j += 32) P[i * sp + j] *= inv;
  }
  __syncthreads();
  attn_load_tile(sx, qkv, row0, T, 3 * C, 2 * C, C, pitch);
  attn_load_tile(sq, go, row0 + i0, nq, C, 0, C, pitch);
  __syncthreads();
  attn_abt(sq, sx, gS, nq, T, C, pitch, sp, 1.0f);  // gP
  __syncthreads();
  for (int i = warp; i < nq; i += kAttnThreads / 32) {
    float dot = 0.f;
    for (int j = lane; j < T; j += 32) dot += gS[i * sp + j] * P[i * sp + j];
    dot = warp_sum(dot);
    float* prow = Pm + (row0 + i0 + i) * T;
    float* grow = gSm + (row0 + i0 + i) * T;
    for (int j = lane; j < T; j += 32) {
      const float pv = P[i * sp + j];
      prow[j] = pv;
      grow[j] = pv * (gS[i * sp + j] - dot);
    }
  }
}
// blockIdx.z: 0 -> gq = scale2 gS k ; 1 -> gk = scale2 gS^T q ; 2 -> gv = P^T go.  Rows [r0, r0 + RB) of the output.
__global__ void __launch_bounds__(kAttnThreads)
attention_bwd_grads_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ go, const float* __restrict__ Pm,
                           const float* __restrict__ gSm, bf16* __restrict__ gqkv, int T, int C, int RB, float scale2) {
  extern __shared__ __align__(128) uint8_t smraw[];
  const int pitch = C + 2, sp = T + 1;
  bf16* sx = reinterpret_cast<bf16*>(smraw);  // [T][pitch]
  float* sm = reinterpret_cast<float*>(sx + static_cast<size_t>(T) * pitch);  // [RB][sp]
  const int tid = threadIdx.x;
  const size_t row0 = static_cast<size_t>(blockIdx.y) * T;
  const int r0 = blockIdx.x * RB;
  const int nr = min(RB, T - r0);
  const int z = blockIdx.z;
  const float* M = (z == 2 ? Pm : gSm) + row0 * T;
  if (z == 0) {
    attn_load_tile(sx, qkv, row0, T, 3 * C, C, C, pitch);
    for (int idx = tid; idx < nr * T; idx += kAttnThreads) {
      const int r = idx / T, t = idx - r * T;
      sm[r * sp + t] = M[static_cast<size_t>(r0 + r) * T + t];
    }
  } else {
    if (z == 1) attn_load_tile(sx, qkv, row0, T, 3 * C, 0, C, pitch);
    else attn_load_tile(sx, go, row0, T, C, 0, C, pitch);
    for (int idx = tid; idx < nr * T; idx += kAttnThreads) {  // transposed read: sm[r][t] = M[t][r0 + r]
      const int t = idx / nr, r = idx - t * nr;
      sm[r * sp + t] = M[static_cast<size_t>(t) * T + r0 + r];
    }
  }
  __syncthreads();
  const float scale = (z == 2) ? 1.0f : scale2;
  const int pairs = C / 2, pw = pitch / 2;
  for (int item = tid; item < pairs * (RB / 8); item += kAttnThreads) {
    const int c2 = item % pairs, ib = (item / pairs) * 8;
    float a0[8], a1[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a0[i] = a1[i] = 0.f;
    const uint32_t* bp = reinterpret_cast<const uint32_t*>(sx) + c2;
    for (int t = 0; t < T; ++t) {
      const float2 bv = unpack_bf16x2(bp[static_cast<size_t>(t) * pw]);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float mv = sm[(ib + i) * sp + t];
        a0[i] += mv * bv.x;
        a1[i] += mv * bv.y;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (ib + i < nr)
        *reinterpret_cast<uint32_t*>(gqkv + (row0 + r0 + ib + i) * 3 * C + z * C + 2 * c2) =
            pack_bf16x2(a0[i] * scale, a1[i] * scale);
  }
}

// SiLU and its derivative as separate elementwise passes (VJP path only: the forward stashes the pre-activation).
//   mode 0: out = silu(pre)        mode 1: out = g * silu'(pre)   (g may alias out)
__global__ void silu_elementwise_kernel(const bf16* __restrict__ pre, const bf16* g, bf16* out, long long n8, int mode) {
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < n8;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint4 pv = *reinterpret_cast<const uint4*>(pre + idx * 8);
    uint4 gv = make_uint4(0, 0, 0, 0);
    if (mode == 1) gv = *reinterpret_cast<const uint4*>(g + idx * 8);
    const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w}, gw[4] = {gv.x, gv.y, gv.z, gv.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 x = unpack_bf16x2(pw[j]);
      float r0, r1;
      const float s0 = 1.0f / (1.0f + __expf(-x.x)), s1 = 1.0f / (1.0f + __expf(-x.y));
      if (mode == 0) {
        r0 = x.x * s0;
        r1 = x.y * s1;
      } else {
        const float2 gg = unpack_bf16x2(gw[j]);
        r0 = gg.x * s0 * (1.0f + x.x * (1.0f - s0));
        r1 = gg.y * s1 * (1.0f + x.y * (1.0f - s1));
      }
      o[j] = pack_bf16x2(r0, r1);
    }
    *reinterpret_cast<uint4*>(out + idx * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// Zero-insertion 2x upsample: out[n, 2h, 2w, :] = in[n, h, w, :], every other pixel zero.  The stride-2 conv's input
// gradient is then a stride-1 conv of `out` with the flipped kernel.
__global__ void zero_upsample_kernel(const bf16* __restrict__ in, bf16* __restrict__ out, long long n, int H, int W,
                                     int C) {
  const int c8 = C / 8;
  const long long total = n * (2 * H) * (2 * W) * c8;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(idx % c8);
    long long r = idx / c8;
    const int w2 = static_cast<int>(r % (2 * W));
    r /= 2 * W;
    const int h2 = static_cast<int>(r % (2 * H));
    const long long img = r / (2 * H);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (((w2 | h2) & 1) == 0) v = *reinterpret_cast<const uint4*>(in + ((img * H + (h2 >> 1)) * W + (w2 >> 1)) * C + g * 8);
    *reinterpret_cast<uint4*>(out + idx * 8) = v;
  }
}

// ------------------------------------------------------------------------------------------------ frame variables
// The C variables of one pixel of a frame tensor (fp32 [frames, HW, C]).  The frame kernels below are templates on
// C = 1..8; C = 4 (the shipped configs, exp/downscaling.py:101) moves a pixel as one 16-byte access, any other count
// as C scalar accesses.
template <int C>
struct Vars {
  float v[C];
  __device__ __forceinline__ float& operator[](int c) { return v[c]; }
  __device__ __forceinline__ float operator[](int c) const { return v[c]; }
};
template <int C>
__device__ __forceinline__ Vars<C> load_vars(const float* p) {
  Vars<C> r;
  if constexpr (C == 4) {
    const float4 q = *reinterpret_cast<const float4*>(p);
    r.v[0] = q.x, r.v[1] = q.y, r.v[2] = q.z, r.v[3] = q.w;
  } else {
#pragma unroll
    for (int c = 0; c < C; ++c) r.v[c] = p[c];
  }
  return r;
}
template <int C>
__device__ __forceinline__ void store_vars(float* p, const Vars<C>& r) {
  if constexpr (C == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
  } else {
#pragma unroll
    for (int c = 0; c < C; ++c) p[c] = r.v[c];
  }
}

// Adjoint of the window compose (src/thor/score.py:76-88,111-141): UNet-output cotangent of window i, slot tau is
// the frame cotangent g[win + tau] where that slot is the frame's source, zero elsewhere.  The windows: win_list[i],
// or win_first + i when win_list is null.
// g: fp32 [frames, HW, C] ; cot: bf16 [n, HW, cpad]; one thread writes 8 channels (16 B).
template <int C>
__global__ void compose_adjoint_kernel(const float* __restrict__ g, bf16* __restrict__ cot, int n, int hw, int cpad,
                                       int order_k, int win_first, int win_last_global, int frame_base,
                                       const int* __restrict__ win_list) {
  const int groups = cpad >> 3;
  const long long total = static_cast<long long>(n) * hw * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int gq = static_cast<int>(idx % groups);
    const long long pw = idx / groups;
    const int pix = static_cast<int>(pw % hw);
    const int i = static_cast<int>(pw / hw);
    const int win = win_list ? win_list[i] : win_first + i;
    const auto take = [&](int tau) {
      return tau <= 2 * order_k &&
             ((tau == order_k) || (win == 0 && tau < order_k) || (win == win_last_global && tau > order_k));
    };
    const auto frame = [&](int tau) { return g + (static_cast<long long>(win + tau - frame_base) * hw + pix) * C; };
    float v[8];
    if constexpr (8 % C == 0) {  // the 8 channels are 8 / C whole slots
#pragma unroll
      for (int hf = 0; hf < 8 / C; ++hf) {
        const int tau = (8 / C) * gq + hf;
        const Vars<C> q = take(tau) ? load_vars<C>(frame(tau)) : Vars<C>{};
#pragma unroll
        for (int c = 0; c < C; ++c) v[C * hf + c] = q[c];
      }
    } else {  // the 8 channels straddle slots
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int ch = 8 * gq + e;
        const int tau = ch / C, c = ch - tau * C;
        v[e] = take(tau) ? frame(tau)[c] : 0.f;
      }
    }
    *reinterpret_cast<uint4*>(cot + (static_cast<long long>(i) * hw + pix) * cpad + 8 * gq) =
        make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  }
}

// Adjoint of unfold (src/thor/score.py:68-74): vjp[f] += sum_tau gin[window f - tau][slot tau] over the windows of this
// launch; a frame no such window touches is left as it is.  The windows: pos == null -> the contiguous global windows
// [win_first, win_first + n); else pos[j] = batch index of global window j or -1 (n_win_global entries).
// gin: fp32 [n, HW, cpad] ; vjp: fp32 [frames, HW, C] ; one thread per (local frame f_lo + fo, pixel), fo < nf.
template <int C>
__global__ void unfold_adjoint_kernel(const float* __restrict__ gin, float* __restrict__ vjp, int n, int f_lo, int nf,
                                      int hw, int cpad, int window, int win_first, int frame_base, int n_win_global,
                                      const int* __restrict__ pos) {
  const long long total = static_cast<long long>(nf) * hw;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int pix = static_cast<int>(idx % hw);
    const int fl = f_lo + static_cast<int>(idx / hw);
    const int fg = frame_base + fl;
    Vars<C> acc{};
    bool any = false;
    for (int tau = 0; tau < window; ++tau) {
      const int j = fg - tau;  // global window whose slot tau is this frame
      int i;
      if (pos) {
        if (j < 0 || j >= n_win_global) continue;
        i = pos[j];
      } else {
        i = j - win_first;
        if (i >= n) continue;
      }
      if (i < 0) continue;
      const Vars<C> q = load_vars<C>(gin + (static_cast<long long>(i) * hw + pix) * cpad + tau * C);
#pragma unroll
      for (int c = 0; c < C; ++c) acc[c] += q[c];
      any = true;
    }
    if (!any) continue;
    float* dst = vjp + (static_cast<long long>(fl) * hw + pix) * C;
    Vars<C> o = load_vars<C>(dst);
#pragma unroll
    for (int c = 0; c < C; ++c) o[c] += acc[c];
    store_vars<C>(dst, o);
  }
}

// ------------------------------------------------------------------------------------------------ K6 / K7
// State layout: x, eps, z are fp32 [frames, H, W, C] (Vars<C> per pixel).  Observation y: fp32 [n_obs, C, Hs, Ws]
// exactly as the reference builds it (exp/downscaling.py:129-132: every t_step-th frame, s x s tile means).
struct GuideParams {
  float* x;
  const float* eps;  // unguided window-composed score (K1 compose epilogue)
  float* eps_out;    // mode 1: guided eps
  const float* y;    // null => unconditioned
  float std2[8];     // likelihood std^2 per variable
  float gamma[8];
  float mu, sigma;            // at the time the score was evaluated
  float mu_next, sigma_next;  // mode 0: target of the predictor step
  int t_step, s_step, H, W;
  int frame_global0;  // global index of local frame 0
  int own_lo;         // first local frame this launch updates (blockIdx.y = 0)
  int mode;           // 0: predictor update of x in place; 1: guided eps -> eps_out + partial sum of squares
  float* partials;    // mode 1: one float per CTA
  int* nan_flag;
  const float* vjp;   // exact_grad: J_eps^T g per pixel (UNet vector-Jacobian product), null = closed-form guidance
  float* cot_out;     // mode 2: g = A^T((y - A x0) / var), the cotangent fed to the UNet VJP
  // mode 0, time-sharded, C = 4: the halo PUSH fused into the predictor update (K8, csrc/halo.cu) — the updated pixels
  // of the first / last k owned frames are also stored into the left / right neighbour's mailbox over NVLink, and the
  // last CTA publishes the step counter.  Null pointers: no neighbour on that side / not sharded.
  float4* push_l;          // left neighbour's mailbox slot (receives local frames [own_lo, own_lo + halo_k))
  float4* push_r;          // right neighbour's slot (receives local frames [own_lo + own_n - halo_k, own_lo + own_n))
  unsigned int* flag_l;    // neighbours' step counters
  unsigned int* flag_r;
  unsigned int* push_done; // CTA counter (local)
  unsigned int publish;    // value to publish: step + 1
  int halo_k, own_n;
};

// mode 1: the CTA's sum of eps_guided^2 -> partials[blockIdx.y * gridDim.x + blockIdx.x] (fixed order, no atomics)
__device__ __forceinline__ void block_partial(const GuideParams& p, float sq) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __shared__ float wsum[32];
  sq = warp_sum(sq);
  if (lane == 0) wsum[warp] = sq;
  __syncthreads();
  if (warp == 0) {
    float v = (lane < (blockDim.x >> 5)) ? wsum[lane] : 0.f;
    v = warp_sum(v);
    if (lane == 0) p.partials[blockIdx.y * gridDim.x + blockIdx.x] = v;
  }
}

// The dense tail of the guidance pass, shared by K6 (coarse-grained observations) and K6p (point observations).  Per
// pixel: grad_x log p = (g - sigma J_eps^T g) / mu  (src/thor/score.py:48-60; the second term only with exact_grad);
// eps_guided = eps - sigma * grad  =>  per-pixel correction sigma (g - sigma vjp) / mu.  Mode 0 then updates x in place
// (and, C = 4, stores the boundary frames into the neighbours' halo mailboxes), mode 1 writes eps_guided and the CTA's
// partial sum of its squares, mode 2 writes g alone to cot_out.  The observation policy `Obs` walks this thread's pixels
// (first / end / step, pixel(i) = index within the frame) and gives the likelihood cotangent g(p, i, o) of pixel i at
// element offset o.
template <int C, class Obs>
__device__ __forceinline__ void guide_tail(const GuideParams& p, const Obs& obs, long long fbase) {
  if (p.mode == 2) {
    for (int i = obs.first(); i < obs.end(); i += obs.step()) {
      const long long o = (fbase + obs.pixel(i)) * C;
      store_vars<C>(p.cot_out + o, obs.g(p, i, o));
    }
    return;
  }
  const int lane = threadIdx.x & 31;
  const float inv_mu = 1.0f / p.mu;
  const float sg_mu = p.sigma * inv_mu;
  float sq = 0.f;
  bool bad = false;
#pragma unroll 1  // unrolled, K6p for C = 1 spills around the division slow path; C = 4 is not unrolled either way
  for (int i = obs.first(); i < obs.end(); i += obs.step()) {
    const long long pix_in_frame = obs.pixel(i);
    const long long o = (fbase + pix_in_frame) * C;
    Vars<C> ev = load_vars<C>(p.eps + o);
    Vars<C> gv = obs.g(p, i, o);
    if (p.vjp != nullptr) {
      const Vars<C> jv = load_vars<C>(p.vjp + o);
#pragma unroll
      for (int c = 0; c < C; ++c) gv[c] -= p.sigma * jv[c];
    }
#pragma unroll
    for (int c = 0; c < C; ++c) ev[c] = __fmaf_rn(-sg_mu, gv[c], ev[c]);  // fused even where g is uniform (K6, no vjp)
    if (p.mode == 0) {
      Vars<C> xv = load_vars<C>(p.x + o);
#pragma unroll
      for (int c = 0; c < C; ++c) {
        // x0 = (x - sigma eps)/mu ; x <- mu' x0 + sigma' eps     (src/thor/pipelines.py:41-46)
        xv[c] = p.mu_next * ((xv[c] - p.sigma * ev[c]) * inv_mu) + p.sigma_next * ev[c];
        bad |= !isfinite(xv[c]);
      }
      store_vars<C>(p.x + o, xv);
      if constexpr (C == 4) {
        // boundary frames also go straight into the neighbours' halo mailboxes (peer stores through NVLink)
        const float4 xq = make_float4(xv[0], xv[1], xv[2], xv[3]);
        const long long hw = static_cast<long long>(p.H) * p.W;
        const int own_idx = static_cast<int>(blockIdx.y);
        if (p.push_l != nullptr && own_idx < p.halo_k) p.push_l[own_idx * hw + pix_in_frame] = xq;
        if (p.push_r != nullptr && own_idx >= p.own_n - p.halo_k)
          p.push_r[(own_idx - (p.own_n - p.halo_k)) * hw + pix_in_frame] = xq;
      }
    } else {
      float s = ev[0] * ev[0];  // the pixel's sum first, then the thread's
#pragma unroll
      for (int c = 1; c < C; ++c) s += ev[c] * ev[c];
      sq += s;
      store_vars<C>(p.eps_out + o, ev);
    }
  }
  if (p.mode == 0) {
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(p.nan_flag, 1);
    if (C == 4 && p.push_done != nullptr) {  // fused halo push: fence this CTA's peer stores, the last CTA publishes
      __threadfence_system();
      __syncthreads();
      if (threadIdx.x == 0) {
        const unsigned int total = gridDim.x * gridDim.y;
        if (atomicAdd(p.push_done, 1u) == total - 1) {
          *p.push_done = 0;
          __threadfence_system();
          if (p.flag_l) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.flag_l), "r"(p.publish) : "memory");
          if (p.flag_r) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.flag_r), "r"(p.publish) : "memory");
        }
      }
    }
  } else {
    block_partial(p, sq);
  }
}

// K6's observation policy: the warp's s x s tile, whose pixels all get the same cotangent (the tile's residual / s^2).
template <int C>
struct TileObs {
  int s, h0, w0, W;
  Vars<C> corr;
  __device__ int first() const { return threadIdx.x & 31; }
  __device__ int end() const { return s * s; }
  __device__ int step() const { return 32; }
  __device__ long long pixel(int i) const { return static_cast<long long>(h0 + i / s) * W + (w0 + i % s); }
  __device__ Vars<C> g(const GuideParams&, int, long long) const { return corr; }
};

// The variance source of a guidance kernel.  Per variable (PerObs = false, the default instances): GuideParams::std2,
// and for K6c's point term PointStd2.  Per observation (PerObs = true, c2w_guided_step_obs_std): std^2 of every
// observation tile in y's layout [n_obs, C, Hs, Ws], and of every point entry [n_entries, C]; the per-variable std2
// fields are not read.  Null where the kernel has no such term.
struct ObsStd2 {
  const float* tile;
  const float* entry;
};

// If observed: obs.corr <- the cotangent of observation tile (ty, tx) (obs's pixels) of global frame fg at fbase,
// computed by one warp (every lane gets it): the warp-shuffle tile mean of x0 (lane order, deterministic), then
// g = A^T(err / var) = err / var / s^2 on each pixel of the tile.  Shared by K6 and K6c: both give a tile the same bits.
// The test is taken here rather than by the caller so that K6's 1/mu is computed ahead of the branch and shared with
// guide_tail, as before the block moved here: K6 keeps its instruction schedule and register count.  PerObs: the tile's
// std^2 is read from tile_std2 at y's offset, in the same expression.
template <int C, bool PerObs = false>
__device__ __forceinline__ void tile_cotangent(const GuideParams& p, bool observed, float inv_mu, long long fbase, int fg,
                                               unsigned ty, int tx, TileObs<C>& obs, const float* tile_std2 = nullptr) {
  if (observed) {
    const int lane = threadIdx.x & 31;
    const int s = obs.s;
    Vars<C> acc{};
    for (int i = lane; i < s * s; i += 32) {
      const long long o = (fbase + obs.pixel(i)) * C;
      const Vars<C> xv = load_vars<C>(p.x + o), ev = load_vars<C>(p.eps + o);
#pragma unroll
      for (int c = 0; c < C; ++c) acc[c] += (xv[c] - p.sigma * ev[c]) * inv_mu;
    }
    const float inv_area = 1.0f / static_cast<float>(s * s);
    const int Hs = p.H / s, Ws = p.W / s;
    const int m = fg / p.t_step;
    const float r2 = (p.sigma * inv_mu) * (p.sigma * inv_mu);
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const float mean = warp_sum(acc[c]) * inv_area;
      const long long yi = ((static_cast<long long>(m) * C + c) * Hs + ty) * Ws + tx;
      const float yv = __ldg(p.y + yi);
      const float std2 = PerObs ? __ldg(tile_std2 + yi) : p.std2[c];
      obs.corr[c] = ((yv - mean) / (std2 + p.gamma[c] * r2)) * inv_area;
    }
  }
}

// CTA = one s-row strip of one frame; one warp per s x s observation tile.
template <int C, bool PerObs>
__global__ void guided_step_kernel(const GuideParams p, const ObsStd2 v) {
  const int warp = threadIdx.x >> 5;
  const int s = p.s_step;
  const int fl = p.own_lo + blockIdx.y;
  const int fg = p.frame_global0 + fl;
  const long long fbase = (static_cast<long long>(fl) * p.H) * p.W;
  const bool observed = (p.y != nullptr) && (fg % p.t_step == 0);
  const float inv_mu = 1.0f / p.mu;
  TileObs<C> obs{s, static_cast<int>(blockIdx.x) * s, warp * s, p.W, {}};  // eps_guided = eps - corr (score.py:35)
  tile_cotangent<C, PerObs>(p, observed, inv_mu, fbase, fg, blockIdx.x, warp, obs, v.tile);
  guide_tail<C>(p, obs, fbase);
}

// ---- K6p: point observations (PointObservation: variables observed at single grid points of chosen frames).  The
// host merges every (frame, pixel) into one entry holding ysum = sum(mask * y) and wsum = sum(mask) per variable, so
// A^T((y - A x0)/var) at that pixel is (ysum - wsum * x0)/var — exact, and zero at every other pixel.  CTA = a strip of
// `strip_rows` full rows of one owned frame; an observed frame first scatters the strip's entries (CSR by frame slot
// and strip) into a shared-memory map pixel -> entry, then runs the dense tail above with g computed from the x and
// eps it loads anyway.  Entries are unique per pixel: no atomics, bit-identical from run to run and under sharding.
// PerObs (a std per observation): observations merge only where their std^2 agree, so a pixel may hold a run of
// consecutive entries (never crossing a strip), each with its own std^2 per variable.  The map holds the run's head;
// g adds the run's entries in entry order, still without atomics.
struct PointParams {
  const int* frame_slot;  // [own_n] observed slot of owned frame own_lo + i, or -1
  const int* strip_off;   // [n_slots * n_strips + 1] CSR offsets into the entries
  const int* pix;         // [n_entries] pixel index within the frame
  const float* ysum;      // [n_entries, C]
  const float* wsum;      // [n_entries, C]
  int strip_rows;
};

__device__ __forceinline__ float point_g(const GuideParams& p, float ys, float ws, float x, float e, float std2,
                                         float gamma) {
  const float inv_mu = 1.0f / p.mu;
  const float r2 = (p.sigma * inv_mu) * (p.sigma * inv_mu);
  const float x0 = (x - p.sigma * e) * inv_mu;
  return (ys - ws * x0) / (std2 + gamma * r2);
}

// The CTA's pixels: `npix` pixels from `pix0` on; slot == nullptr on a frame without observations.  PerObs: also the
// entries' pixels, their std^2 [n_entries][C] and the strip's end entry, to walk a run.
template <int C, bool PerObs = false>
struct StripObs {
  const int* slot;
  const float* ysum;
  const float* wsum;
  long long pix0;
  int npix;
  const int* pix = nullptr;
  const float* std2 = nullptr;
  int e_end = 0;
  __device__ int first() const { return threadIdx.x; }
  __device__ int end() const { return npix; }
  __device__ int step() const { return blockDim.x; }
  __device__ long long pixel(int i) const { return pix0 + i; }
  __device__ Vars<C> g(const GuideParams& p, int i, long long o) const {
    Vars<C> r{};
    const int e = slot ? slot[i] : -1;
    if (e < 0) return r;
    const Vars<C> xv = load_vars<C>(p.x + o), ev = load_vars<C>(p.eps + o);
    if constexpr (PerObs) {
#pragma unroll
      for (int c = 0; c < C; ++c) r[c] = -0.0f;  // -0 + v == v for every v: the run's first term is taken as it is
      add_run(p, e, xv, ev, r);
    } else {
      const Vars<C> ys = load_vars<C>(ysum + static_cast<long long>(C) * e);
      const Vars<C> ws = load_vars<C>(wsum + static_cast<long long>(C) * e);
#pragma unroll
      for (int c = 0; c < C; ++c) r[c] = point_g(p, ys[c], ws[c], xv[c], ev[c], p.std2[c], p.gamma[c]);
    }
    return r;
  }
  // PerObs: r += the point term of every entry of the run headed by e (same pixel, within the strip), in entry order.
  __device__ void add_run(const GuideParams& p, int e, const Vars<C>& xv, const Vars<C>& ev, Vars<C>& r) const {
    const int px = pix[e];
#pragma unroll 1
    for (int k = e; k < e_end && pix[k] == px; ++k) {
      const Vars<C> ys = load_vars<C>(ysum + static_cast<long long>(C) * k);
      const Vars<C> ws = load_vars<C>(wsum + static_cast<long long>(C) * k);
      const Vars<C> s2 = load_vars<C>(std2 + static_cast<long long>(C) * k);
#pragma unroll
      for (int c = 0; c < C; ++c) r[c] += point_g(p, ys[c], ws[c], xv[c], ev[c], s2[c], p.gamma[c]);
    }
  }
};

// This CTA's strip and, on an observed frame, its pixel -> entry map in `slot` (PerObs: run heads only).
template <int C, bool PerObs = false>
__device__ __forceinline__ StripObs<C, PerObs> point_strip(const GuideParams& p, const PointParams& q, int* slot,
                                                           const float* entry_std2 = nullptr) {
  const int h0 = blockIdx.x * q.strip_rows;
  StripObs<C, PerObs> obs{nullptr, q.ysum, q.wsum, static_cast<long long>(h0) * p.W, min(q.strip_rows, p.H - h0) * p.W};
  const int os = q.frame_slot[blockIdx.y];
  if (os >= 0) {  // uniform over the CTA
    for (int i = threadIdx.x; i < obs.npix; i += blockDim.x) slot[i] = -1;
    __syncthreads();
    const int* off = q.strip_off + static_cast<long long>(os) * gridDim.x + blockIdx.x;
    const int e0 = off[0], e1 = off[1];
    for (int e = e0 + static_cast<int>(threadIdx.x); e < e1; e += blockDim.x)
      if (!PerObs || e == e0 || q.pix[e - 1] != q.pix[e]) slot[q.pix[e] - static_cast<int>(obs.pix0)] = e;
    __syncthreads();
    obs.slot = slot;
    if constexpr (PerObs) {
      obs.pix = q.pix;
      obs.std2 = entry_std2;
      obs.e_end = e1;
    }
  }
  return obs;
}

template <int C, bool PerObs>
__global__ void __launch_bounds__(256) guided_points_kernel(const GuideParams p, const PointParams q, const ObsStd2 v) {
  __shared__ int slot[C2W_POINT_STRIP_PIX];
  const long long fbase = (static_cast<long long>(p.own_lo + blockIdx.y) * p.H) * p.W;
  guide_tail<C>(p, point_strip<C, PerObs>(p, q, slot, v.entry), fbase);
}

// ---- K6c: a coarse field and point observations in one likelihood (CombinedObservation).  The cotangent is the sum
// of the two terms' own, g = A_c^T((y_c - A_c x0)/var_c) + A_p^T((y_p - A_p x0)/var_p), each with its own std^2 per
// variable (the point term's in PointStd2, gamma shared).  CTA = a strip of q.strip_rows full rows of one owned frame,
// a multiple of s_step so that every observation tile lies inside one strip.  Phase 1, on a frame with f % t_step == 0:
// the strip's tile cotangents (tile_cotangent, one warp per tile in turn) go to shared memory.  Phase 2: point_strip's
// pixel -> entry map, then the dense tail with g = tile term + point term, in that order, each 0 where absent.  Dynamic
// shared memory: [strip_rows * W] ints of map rounded up to 16 bytes, then [(strip_rows / s) * (W / s)][C] floats of
// tile cotangents (combined_smem_bytes).
struct PointStd2 {
  float v[C2W_MAX_VARS];
};

__host__ __device__ __forceinline__ int combined_map_ints(int strip_rows, int W) { return (strip_rows * W + 3) & ~3; }
__host__ __device__ __forceinline__ int combined_smem_bytes(int strip_rows, int W, int s, int C) {
  return 4 * (combined_map_ints(strip_rows, W) + (strip_rows / s) * (W / s) * C);
}

// PerObs: the tile term with tile_cotangent's per-tile std^2, the point term over the pixel's run (StripObs::add_run).
template <int C, bool PerObs = false>
struct CombinedObs {
  StripObs<C, PerObs> pts;
  const float* corr;  // [tiles][C] of this strip; null on a frame without a coarse observation
  const PointStd2& std2;
  int s, tiles_w, W;
  __device__ int first() const { return pts.first(); }
  __device__ int end() const { return pts.end(); }
  __device__ int step() const { return pts.step(); }
  __device__ long long pixel(int i) const { return pts.pixel(i); }
  __device__ Vars<C> g(const GuideParams& p, int i, long long o) const {
    Vars<C> r{};
    if (corr) {
      const int row = i / W;
      const Vars<C> t = load_vars<C>(corr + ((row / s) * tiles_w + (i - row * W) / s) * C);
#pragma unroll
      for (int c = 0; c < C; ++c) r[c] = t[c];
    }
    const int e = pts.slot ? pts.slot[i] : -1;
    if (e < 0) return r;
    const Vars<C> xv = load_vars<C>(p.x + o), ev = load_vars<C>(p.eps + o);
    if constexpr (PerObs) {
      pts.add_run(p, e, xv, ev, r);
    } else {
      const Vars<C> ys = load_vars<C>(pts.ysum + static_cast<long long>(C) * e);
      const Vars<C> ws = load_vars<C>(pts.wsum + static_cast<long long>(C) * e);
#pragma unroll
      for (int c = 0; c < C; ++c) r[c] += point_g(p, ys[c], ws[c], xv[c], ev[c], std2.v[c], p.gamma[c]);
    }
    return r;
  }
};

// PerObs: pstd2 is not read; the variances come from v.
template <int C, bool PerObs>
__global__ void __launch_bounds__(256) guided_combined_kernel(const GuideParams p, const PointParams q,
                                                              const PointStd2 pstd2, const ObsStd2 v) {
  extern __shared__ __align__(16) int combined_smem[];
  const int s = p.s_step, tiles_w = p.W / s;
  const int fl = p.own_lo + blockIdx.y;
  const int fg = p.frame_global0 + fl;
  const long long fbase = (static_cast<long long>(fl) * p.H) * p.W;
  float* corr = reinterpret_cast<float*>(combined_smem + combined_map_ints(q.strip_rows, p.W));
  const bool coarse = fg % p.t_step == 0;
  if (coarse) {  // uniform over the CTA
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float inv_mu = 1.0f / p.mu;
    const int ty0 = blockIdx.x * (q.strip_rows / s);
    const int tiles = (min(q.strip_rows, p.H - static_cast<int>(blockIdx.x) * q.strip_rows) / s) * tiles_w;
    for (int t = warp; t < tiles; t += blockDim.x >> 5) {
      const int ty = ty0 + t / tiles_w, tx = t % tiles_w;
      TileObs<C> tile{s, ty * s, tx * s, p.W, {}};
      tile_cotangent<C, PerObs>(p, true, inv_mu, fbase, fg, ty, tx, tile, v.tile);
      if (lane == 0) store_vars<C>(corr + t * C, tile.corr);
    }
    __syncthreads();
  }
  const CombinedObs<C, PerObs> obs{point_strip<C, PerObs>(p, q, combined_smem, v.entry), coarse ? corr : nullptr, pstd2,
                                   s, tiles_w, p.W};
  guide_tail<C>(p, obs, fbase);
}

// Fold of the window outputs (fp32 [n, hw, cpad], EPI_F32 of the last conv) into the composed score [frames, hw, C]:
// the centre slot of every window, the head slots of window 0 and the tail slots of the last window
// (src/thor/score.py:76-88) — what the K1 compose epilogue does for C = 4.
__global__ void compose_generic_kernel(const float* __restrict__ out32, float* __restrict__ eps, int n, int hw, int cpad,
                                       int C, int k, int win_first, int win_last_global, int frame_base,
                                       const int* __restrict__ win_list) {
  const long long total = static_cast<long long>(n) * hw * C;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % C);
    const long long ip = idx / C;
    const int pix = static_cast<int>(ip % hw), i = static_cast<int>(ip / hw);
    const int win = win_list ? win_list[i] : win_first + i;
    const float* src = out32 + (static_cast<long long>(i) * hw + pix) * cpad + c;
    const int t0 = (win == 0) ? 0 : k, t1 = (win == win_last_global) ? 2 * k : k;
    for (int tau = t0; tau <= t1; ++tau)
      eps[((static_cast<long long>(win + tau - frame_base)) * hw + pix) * C + c] = src[tau * C];
  }
}

// N2 (SURVEY 8(f), optimiser half): torch.optim.AdamW.step() (training_loop.py:384; decoupled weight decay, bias
// correction, eps added to sqrt(v)/sqrt(bias2)) and StandardEMA.update() (src/thor/ema.py:24-27: ema = ema * rate +
// p * (1 - rate), evaluated on the UPDATED parameters) as ONE pass over the flat parameter buffer: reads p, g, m, v,
// ema and writes p, m, v, ema — 36 B per parameter instead of the ~20 separate elementwise passes of the eager
// optimiser + per-tensor EMA loop.  grad_scale multiplies the gradient first (1 / loss_scaling).
struct AdamWParams {
  float lr, beta1, beta2, eps, weight_decay;
  float bias1, bias2_sqrt;  // 1 - beta1^step, sqrt(1 - beta2^step)
  float ema_rate, grad_scale;
};
__device__ __forceinline__ void adamw_ema_one(float& p, float g, float& m, float& v, float* e, const AdamWParams& h) {
  g *= h.grad_scale;
  p *= 1.0f - h.lr * h.weight_decay;
  m = m + (1.0f - h.beta1) * (g - m);            // exp_avg.lerp_(grad, 1 - beta1)
  v = h.beta2 * v + (1.0f - h.beta2) * g * g;    // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
  const float denom = sqrtf(v) / h.bias2_sqrt + h.eps;
  p = p - (h.lr / h.bias1) * (m / denom);        // param.addcdiv_(exp_avg, denom, value=-step_size)
  if (e) *e = *e * h.ema_rate + p * (1.0f - h.ema_rate);
}
__global__ void adamw_ema_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                 float* __restrict__ v, float* __restrict__ ema, long long n, AdamWParams h) {
  const long long n4 = n / 4;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4; i += stride) {
    float4 pp = reinterpret_cast<float4*>(p)[i], mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    const float4 gg = reinterpret_cast<const float4*>(g)[i];
    float4 ee = ema ? reinterpret_cast<float4*>(ema)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    adamw_ema_one(pp.x, gg.x, mm.x, vv.x, ema ? &ee.x : nullptr, h);
    adamw_ema_one(pp.y, gg.y, mm.y, vv.y, ema ? &ee.y : nullptr, h);
    adamw_ema_one(pp.z, gg.z, mm.z, vv.z, ema ? &ee.z : nullptr, h);
    adamw_ema_one(pp.w, gg.w, mm.w, vv.w, ema ? &ee.w : nullptr, h);
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
    if (ema) reinterpret_cast<float4*>(ema)[i] = ee;
  }
  for (long long i = n4 * 4 + blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += stride)
    adamw_ema_one(p[i], g[i], m[i], v[i], ema ? ema + i : nullptr, h);
}

// Deterministic final reduction of the per-CTA partials (fixed order, double accumulate).
__global__ void reduce_partials_kernel(const float* __restrict__ partials, int n, double* __restrict__ out) {
  __shared__ double sh[256];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += static_cast<double>(partials[i]);
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = sh[0];
}

// Philox4x32-10 (counter-based; keyed by seed, counter = (global pixel index, step id)).
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
  const float u1 = (static_cast<float>(a) + 0.5f) * 2.3283064365386963e-10f;  // (0, 1)
  const float u2 = (static_cast<float>(b) + 0.5f) * 2.3283064365386963e-10f;
  const float r = sqrtf(-2.0f * logf(u1));
  float sn, cs;
  sincospif(2.0f * u2, &sn, &cs);
  return make_float2(r * cs, r * sn);
}

// x <- x - (delta * eps + sqrt(2 delta) z) * sigma' ,  delta = tau / mean(eps^2)   (src/thor/pipelines.py:84-87)
// sumsq: the trajectory-global sum of eps^2 (already all-reduced when time-sharded); count = L*C*H*W.
// z == null: draw z on chip with Philox keyed by the GLOBAL pixel index (identical for any sharding): one block of four
// normals per group of four variables, counter word 3 = group index.
template <int C>
__global__ void corrector_update_kernel(float* __restrict__ x, const float* __restrict__ eps,
                                        const float* __restrict__ z, const double* __restrict__ sumsq, double count,
                                        float tau, float sigma_next, long long pix0_global, long long npix,
                                        unsigned long long seed, unsigned int step_id, int* nan_flag) {
  const float delta = tau / static_cast<float>(sumsq[0] / count);
  const float zs = sqrtf(2.0f * delta);
  bool bad = false;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < npix;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    Vars<C> xv = load_vars<C>(x + i * C);
    const Vars<C> ev = load_vars<C>(eps + i * C);
    Vars<C> zv;
    if (z) {
      zv = load_vars<C>(z + i * C);
    } else {
      const unsigned long long g = static_cast<unsigned long long>(pix0_global + i);
#pragma unroll
      for (int b = 0; 4 * b < C; ++b) {
        const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(g), static_cast<uint32_t>(g >> 32), step_id,
                                                 static_cast<uint32_t>(b)),
                                      make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
        const float2 n0 = box_muller(r.x, r.y), n1 = box_muller(r.z, r.w);
        const float n[4] = {n0.x, n0.y, n1.x, n1.y};
#pragma unroll
        for (int e = 0; e < 4 && 4 * b + e < C; ++e) zv[4 * b + e] = n[e];
      }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
      xv[c] -= (delta * ev[c] + zs * zv[c]) * sigma_next;
      bad |= !isfinite(xv[c]);
    }
    store_vars<C>(x + i * C, xv);
  }
  if (bad) atomicOr(nan_flag, 1);
}

}  // namespace c2w
