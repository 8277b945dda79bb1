// Host side of the C-ABI: handle, weight packing, workspace plan and the static launch sequence of the
// ScoreUNet forward (model/nn.py:220-242) over a batch of Markov windows.
#include <stdlib.h>

#include <algorithm>
#include <map>
#include <string>
#include <type_traits>
#include <vector>

#include "c2w_b200.h"
#include "common.cuh"
#include "conv_tcgen05.cuh"
#include "kernels.cuh"
#include "wgrad_tcgen05.cuh"

using namespace c2w;

int c2w_num_sms();

static long long g_launches = 0;  // kernels launched by this library (bench.py's gpu_launches)
void c2w_count_launches(int n) { g_launches += n; }  // for the other translation units (halo.cu)

namespace {

// Optional per-launch CUDA-event timing (bench.py roofline pass): events are recorded on the launch stream around
// every kernel of the forward pass and summed per class when read.
struct TimedSpan {
  int cls;  // 0 = K1 conv/GEMM (tensor cores), 1 = everything else in the forward pass
  cudaEvent_t e0, e1;
};

struct ConvW {
  bf16* w = nullptr;   // [cout_pad, taps * cin_pad], k = tap * cin_pad + c
  float* b = nullptr;  // [cout_pad]
  bf16* wd = nullptr;  // input-gradient weights [cin_pad, taps * cout_pad], k = (8 - tap) * cout_pad + o  (flipped)
  int cin = 0, cout = 0, cin_pad = 0, cout_pad = 0, taps = 0;
  long long gw = -1, gb = -1;  // offsets of weight / bias in the flat gradient buffer (c2w_param_layout)
};
struct BlockW {
  int mod_off = 0;
  long long g_pw = -1, g_pb = -1;  // project.0 weight / bias
  ConvW c1, c2;
};
struct AttnW {
  ConvW qkv, proj;
};
struct LevelW {
  int C = 0, H = 0, W = 0;
  bool attn = false;
  ConvW head, tail;
  std::vector<BlockW> desc, asc;
  std::vector<AttnW> dattn, aattn;
};

enum OpKind { OP_CONV, OP_LN, OP_ATTN, OP_LN_BWD, OP_ATTN_BWD, OP_ZERO_UP, OP_SILU, OP_COPY, OP_WGRAD, OP_COLSUM };
struct Op {
  OpKind kind;
  // conv
  ConvLaunch conv;
  int pix_per_img = 0;
  bool is_final = false;
  // what the launch was built from (the LayerNorm fusion may rebuild it with one N tile per pixel)
  struct ConvSpec {
    bool c3 = false;
    const bf16* in = nullptr;
    int H = 0, W = 0, cin = 0;
    const bf16* wts = nullptr;
    const float* bias = nullptr;
    int cout_pad = 0, mode = 0;
    bf16* out = nullptr;
    int stride = 1;
  } spec;
  // layernorm (forward: in -> out [+ inv]; backward: in = g_y, aux = y stash, res = incoming gradient or null)
  const bf16* in = nullptr;
  bf16* out = nullptr;
  float* inv = nullptr;
  const bf16* aux = nullptr;
  const bf16* res = nullptr;
  int C = 0, H = 0, W = 0, up = 0, mod_off = -1;
  // attention
  int T = 0;
  // training: OP_COPY (in -> out, C*H*W elements per image); OP_WGRAD (dW of one conv: x = spec.in, dy = in; spec.H/W/cin/
  // cout_pad/stride/c3 as in the forward conv) and OP_COLSUM (bias gradient: column sums of `in`, C padded channels)
  long long dst = -1;        // offset in the flat gradient buffer
  long long dst_bias = -1;   // OP_WGRAD: offset of the conv's bias gradient
  int cin_real = 0, cout_real = 0;
  WgradLaunch wg;            // built for `wg_n` images
  int wg_n = -1;
};

struct Plan {
  int n_max = 0;
  bool vjp = false;        // forward ops stash what the backward ops need
  bool per_t = false;      // one diffusion time per sample: mods is [n, total_mod], no LayerNorm fusion
  bool train = false;      // vjp + per_t + parameter gradients (wgrad / bias / modulation / time-MLP ops in `bwd`)
  int n_last = 0;          // images of the last training forward
  const float* t_last = nullptr;
  float* dmods = nullptr;  // [n, total_mod] gradient w.r.t. the modulation vectors
  float* wg_scratch = nullptr;
  size_t wg_scratch_floats = 0;
  float *feat = nullptr, *pre0 = nullptr, *pre1 = nullptr, *demb = nullptr, *dh0 = nullptr;  // time-MLP backward
  float* loss_partials = nullptr;
  float *forc_pad = nullptr, *fvec = nullptr;  // forcing rows padded to float4 lanes [n, forcing_pad]; Wf forcing + bf [n, E]
  float* grad = nullptr;   // flat gradient buffer of the running c2w_train_backward call
  std::vector<Op> ops;
  std::vector<Op> bwd;     // input-gradient pass (vjp plans only), in execution order
  bf16* cot = nullptr;     // UNet-output cotangent [n, HW, cout_pad(window channels)] bf16
  bf16* g0 = nullptr;
  bf16* xin = nullptr;
  float* h0 = nullptr;
  float* emb = nullptr;
  float* mods = nullptr;
  float* out32 = nullptr;
  size_t attn_smem = 0;
};

inline int pad64(int c) { return (c + 63) / 64 * 64; }

}  // namespace

struct c2w_handle {
  c2w_config cfg;
  int nl = 0, cin = 0, cin_pad = 0;
  std::map<std::string, std::vector<float>> raw;
  std::vector<std::pair<std::string, long long>> params;  // (name, numel) in the order they were loaded
  std::map<std::string, long long> param_off;              // name -> offset in the flat gradient buffer (4-float aligned)
  long long param_total = 0;
  bool finalized = false;
  std::vector<void*> allocs;
  float *map0_w = nullptr, *map0_b = nullptr, *map1_w = nullptr, *map1_b = nullptr;
  float *proj_w = nullptr, *proj_b = nullptr;
  long long *row_w = nullptr, *row_b = nullptr;  // per modulation channel: where its project.weight row / bias lives in the flat gradient
  float *mapf_w = nullptr, *mapf_b = nullptr;  // forcing branch: [E, forcing_pad] (columns zero-padded to 4), [E]
  void* refresh_jobs = nullptr;  // c2w_refresh_weights: device table of re-pack jobs (built at the first call)
  int* refresh_first = nullptr;
  int refresh_n = 0, refresh_chunks = 0;
  int forcing_pad = 0;
  const float* forcing = nullptr;  // c2w_set_forcing: device [n, forcing_dim] for the next per-sample forwards
  float* zero_bias = nullptr;  // 512 zeros: the input-gradient convs have no bias
  int total_mod = 0;
  std::vector<LevelW> levels;
  Plan plan;
  int sms = 0;
  bool timing = false;
  bool fuse_ln = true;  // C2W_NO_FUSE_LN=1 keeps every LayerNorm a separate kernel (A/B runs)
  bool fuse_dsilu = true;  // C2W_NO_FUSE_DSILU=1: silu' of the input-gradient pass as a separate elementwise kernel
  bool fuse_dual = true;   // C2W_NO_FUSE_DUAL=1: stashing forward with a separate SiLU pass after conv1
  std::vector<TimedSpan> spans;
  size_t spans_used = 0;
  long long* timeline = nullptr;  // diagnostics build: device [capacity][2] start / end of every K1 launch (c2w_set_timeline)
  int timeline_cap = 0, timeline_used = 0;
};

namespace {

struct Bump {
  uint8_t* base;
  size_t off = 0;
  explicit Bump(void* p) : base(static_cast<uint8_t*>(p)) {}
  template <typename T>
  T* take(size_t count) {
    off = (off + 1023) & ~size_t(1023);
    T* r = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return r;
  }
};

int dev_upload(c2w_handle* h, const void* src, size_t bytes, void** out) {
  void* d = nullptr;
  C2W_CUDA(cudaMalloc(&d, bytes));
  h->allocs.push_back(d);
  C2W_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
  *out = d;
  return C2W_OK;
}

int need(c2w_handle* h, const std::string& name, size_t numel, const std::vector<float>** out) {
  auto it = h->raw.find(name);
  if (it == h->raw.end()) return fail(C2W_ERR_MISSING, "weight '%s' was never loaded", name.c_str());
  if (it->second.size() != numel)
    return fail(C2W_ERR_INVALID, "weight '%s': expected %zu elements, got %zu", name.c_str(), numel, it->second.size());
  *out = &it->second;
  return C2W_OK;
}

// OIHW (or OI1 for Conv1d) fp32 -> bf16 [cout_pad, taps*cin_pad] with k = (r*kw + s)*cin_pad + c; bias zero-padded.
int pack_conv(c2w_handle* h, const std::string& prefix, int cout, int cin, int taps, ConvW* cw) {
  const std::vector<float>*w, *b;
  int rc = need(h, prefix + ".weight", static_cast<size_t>(cout) * cin * taps, &w);
  if (rc) return rc;
  rc = need(h, prefix + ".bias", cout, &b);
  if (rc) return rc;
  cw->cin = cin;
  cw->cout = cout;
  cw->taps = taps;
  cw->gw = h->param_off.count(prefix + ".weight") ? h->param_off[prefix + ".weight"] : -1;
  cw->gb = h->param_off.count(prefix + ".bias") ? h->param_off[prefix + ".bias"] : -1;
  cw->cin_pad = pad64(cin);
  cw->cout_pad = pad64(cout);
  const size_t K = static_cast<size_t>(taps) * cw->cin_pad;
  std::vector<bf16> packed(static_cast<size_t>(cw->cout_pad) * K, __float2bfloat16_rn(0.f));
  for (int o = 0; o < cout; ++o)
    for (int c = 0; c < cin; ++c)
      for (int t = 0; t < taps; ++t)
        packed[o * K + static_cast<size_t>(t) * cw->cin_pad + c] =
            __float2bfloat16_rn((*w)[(static_cast<size_t>(o) * cin + c) * taps + t]);
  std::vector<float> bias(cw->cout_pad, 0.f);
  for (int o = 0; o < cout; ++o) bias[o] = (*b)[o];
  rc = dev_upload(h, packed.data(), packed.size() * sizeof(bf16), reinterpret_cast<void**>(&cw->w));
  if (rc) return rc;
  rc = dev_upload(h, bias.data(), bias.size() * sizeof(float), reinterpret_cast<void**>(&cw->b));
  if (rc) return rc;
  // input-gradient weights: rows = input channels, k = (taps - 1 - t) * cout_pad + o  (spatially flipped kernel)
  const size_t Kd = static_cast<size_t>(taps) * cw->cout_pad;
  std::vector<bf16> packed_d(static_cast<size_t>(cw->cin_pad) * Kd, __float2bfloat16_rn(0.f));
  for (int o = 0; o < cout; ++o)
    for (int c = 0; c < cin; ++c)
      for (int t = 0; t < taps; ++t)
        packed_d[c * Kd + static_cast<size_t>(taps - 1 - t) * cw->cout_pad + o] =
            __float2bfloat16_rn((*w)[(static_cast<size_t>(o) * cin + c) * taps + t]);
  return dev_upload(h, packed_d.data(), packed_d.size() * sizeof(bf16), reinterpret_cast<void**>(&cw->wd));
}

int upload_named(c2w_handle* h, const std::string& name, size_t numel, float** out) {
  const std::vector<float>* v;
  int rc = need(h, name, numel, &v);
  if (rc) return rc;
  return dev_upload(h, v->data(), numel * sizeof(float), reinterpret_cast<void**>(out));
}

template <int C>
void launch_ln_c(const bf16* x, const float* mod, bf16* out, float* inv, long long npix, int H, int W, int up, int sms,
                 cudaStream_t st, long long mod_stride) {
  const int threads = 256;
  long long blocks = (npix + 7) / 8;
  const long long cap = static_cast<long long>(sms) * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  channel_layernorm_kernel<C><<<static_cast<int>(blocks), threads, 0, st>>>(x, mod, out, inv, npix, H, W, up, 1e-5f,
                                                                            mod_stride);
}
template <int C>
void launch_ln_bwd_c(const bf16* gy, const bf16* y, const float* inv, const bf16* gres, bf16* out, long long npix, int H,
                     int W, int down, int sms, cudaStream_t st, float* dmod, int dmod_stride) {
  const int threads = 256;
  if (dmod != nullptr) {  // training: contiguous per-image chunks, per-image column sums of the input gradient
    const int pix = H * W;
    int chunk = pix < 512 ? pix : 512;
    while (pix % chunk != 0) --chunk;
    channel_layernorm_bwd_kernel<C><<<static_cast<int>(npix / chunk), threads, 0, st>>>(gy, y, inv, gres, out, npix, H, W,
                                                                                      down, dmod, dmod_stride, pix, chunk);
    return;
  }
  long long blocks = (npix + 7) / 8;
  const long long cap = static_cast<long long>(sms) * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  channel_layernorm_bwd_kernel<C><<<static_cast<int>(blocks), threads, 0, st>>>(gy, y, inv, gres, out, npix, H, W, down);
}

#define C2W_LN_DISPATCH(C, CALL)                                                                           \
  switch (C) {                                                                                             \
    case 64: CALL(64); break;                                                                              \
    case 128: CALL(128); break;                                                                            \
    case 192: CALL(192); break;                                                                            \
    case 256: CALL(256); break;                                                                            \
    case 320: CALL(320); break;                                                                            \
    case 384: CALL(384); break;                                                                            \
    case 448: CALL(448); break;                                                                            \
    case 512: CALL(512); break;                                                                            \
    default: return fail(C2W_ERR_INVALID, "channel LayerNorm: unsupported C=%d (multiple of 64, <= 512)", C); \
  }

int launch_ln(const bf16* x, const float* mod, bf16* out, float* inv, long long npix, int C, int H, int W, int up,
              int sms, cudaStream_t st, long long mod_stride = 0) {
#define C2W_CALL(CC) launch_ln_c<CC>(x, mod, out, inv, npix, H, W, up, sms, st, mod_stride)
  C2W_LN_DISPATCH(C, C2W_CALL)
#undef C2W_CALL
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

int launch_ln_bwd(const bf16* gy, const bf16* y, const float* inv, const bf16* gres, bf16* out, long long npix, int C,
                  int H, int W, int down, int sms, cudaStream_t st, float* dmod = nullptr, int dmod_stride = 0) {
#define C2W_CALL(CC) launch_ln_bwd_c<CC>(gy, y, inv, gres, out, npix, H, W, down, sms, st, dmod, dmod_stride)
  C2W_LN_DISPATCH(C, C2W_CALL)
#undef C2W_CALL
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

// scratch: fp32 [2][n][T][T] (P and gS)
// cudaFuncAttributeMaxDynamicSharedMemorySize is per device: set it once per (kernel, device) of this process
template <typename K>
int ensure_smem(K kernel, size_t smem, unsigned long long* done) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (!((*done >> (dev & 63)) & 1ull)) {
    C2W_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    *done |= 1ull << (dev & 63);
  }
  (void)smem;
  return C2W_OK;
}

template <int C>
int launch_attention_bwd_mma(const bf16* qkv, const bf16* go, bf16* gqkv, int n, cudaStream_t st) {
  const size_t smem = attention_bwd_mma_smem_bytes(C);
  static unsigned long long done = 0;
  int rc = ensure_smem(attention_bwd_mma_kernel<C>, smem, &done);
  if (rc) return rc;
  attention_bwd_mma_kernel<C><<<n, 256, smem, st>>>(qkv, go, gqkv, 1.0f / sqrtf(static_cast<float>(C)));
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

int launch_attention_bwd(const bf16* qkv, const bf16* go, bf16* gqkv, float* scratch, int n, int T, int C,
                         cudaStream_t st) {
  C2W_REQUIRE(T % 8 == 0 && C % 8 == 0 && scratch, "attention backward: T %% 8 and C %% 8 must be 0 (T=%d C=%d)", T, C);
  {  // 64 tokens (8 x 8 attention level): tensor-core kernel; C2W_ATTN_MMA=0 keeps the CUDA-core kernels (A/B runs)
    static int use_mma = -1;
    if (use_mma < 0) {
      const char* e = getenv("C2W_ATTN_MMA");
      use_mma = (e && e[0] == '0') ? 0 : 1;
    }
    if (use_mma && T == 64) {
      if (C == 512) return launch_attention_bwd_mma<512>(qkv, go, gqkv, n, st);
      if (C == 256) return launch_attention_bwd_mma<256>(qkv, go, gqkv, n, st);
      if (C == 128) return launch_attention_bwd_mma<128>(qkv, go, gqkv, n, st);
    }
  }
  const int QB = std::min(T, kAttnBwdRows);
  const size_t smem1 = attention_bwd_scores_smem(T, C, QB), smem2 = attention_bwd_grads_smem(T, C, QB);
  C2W_REQUIRE(std::max(smem1, smem2) <= static_cast<size_t>(kSmemLimit),
              "attention backward: T=%d C=%d needs %zu B of shared memory", T, C, std::max(smem1, smem2));
  static unsigned long long done1 = 0, done2 = 0;
  int rc = ensure_smem(attention_bwd_scores_kernel, smem1, &done1);
  if (rc) return rc;
  if ((rc = ensure_smem(attention_bwd_grads_kernel, smem2, &done2))) return rc;
  float* Pm = scratch;
  float* gSm = scratch + static_cast<size_t>(n) * T * T;
  const float scale2 = 1.0f / sqrtf(static_cast<float>(C));
  const int nb = (T + QB - 1) / QB;
  attention_bwd_scores_kernel<<<dim3(nb, n), kAttnThreads, smem1, st>>>(qkv, go, Pm, gSm, T, C, QB, scale2);
  C2W_CUDA(cudaGetLastError());
  attention_bwd_grads_kernel<<<dim3(nb, n, 3), kAttnThreads, smem2, st>>>(qkv, go, Pm, gSm, gqkv, T, C, QB, scale2);
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

template <int QB>
int launch_attention_qb(const bf16* qkv, bf16* out, int n, int T, int C, cudaStream_t st) {
  const size_t smem = attention_smem_bytes(T, C, QB);
  C2W_REQUIRE(smem <= static_cast<size_t>(kSmemLimit), "attention: T=%d C=%d needs %zu B of shared memory", T, C, smem);
  static unsigned long long done = 0;
  int rc = ensure_smem(attention_kernel<QB>, smem, &done);
  if (rc) return rc;
  dim3 grid((T + QB - 1) / QB, n);
  attention_kernel<QB><<<grid, kAttnThreads, smem, st>>>(qkv, out, T, C, 1.0f / sqrtf(static_cast<float>(C)));
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

template <int C>
int launch_attention_mma(const bf16* qkv, bf16* out, int n, cudaStream_t st) {
  const size_t smem = attention_mma_smem_bytes(C);
  static unsigned long long done = 0;
  int rc = ensure_smem(attention_mma_kernel<C>, smem, &done);
  if (rc) return rc;
  attention_mma_kernel<C><<<n, 256, smem, st>>>(qkv, out, 1.0f / sqrtf(static_cast<float>(C)));
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

int launch_attention(const bf16* qkv, bf16* out, int n, int T, int C, cudaStream_t st) {
  C2W_REQUIRE(T % 4 == 0 && C % 8 == 0, "attention: T %% 4 and C %% 8 must be 0 (T=%d C=%d)", T, C);
  {  // 64 tokens (8 x 8 attention level): tensor-core kernel; C2W_ATTN_MMA=0 keeps the CUDA-core kernel (A/B runs)
    static int use_mma = -1;
    if (use_mma < 0) {
      const char* e = getenv("C2W_ATTN_MMA");
      use_mma = (e && e[0] == '0') ? 0 : 1;
    }
    if (use_mma && T == 64) {
      if (C == 512) return launch_attention_mma<512>(qkv, out, n, st);
      if (C == 256) return launch_attention_mma<256>(qkv, out, n, st);
      if (C == 128) return launch_attention_mma<128>(qkv, out, n, st);
    }
  }
  // Queries per CTA: the largest block that still gives every SM two CTAs' worth of work (K and V are re-read from L2
  // by every query block of a window, so bigger blocks move less data; smaller ones fill the machine).
  const int sms = c2w_num_sms();
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("C2W_ATTN_QB");
    forced = e ? atoi(e) : 0;
  }
  int qb = 16;
  for (int cand : {64, 32})
    if (static_cast<long long>(n) * ((T + cand - 1) / cand) >= 2LL * sms) {
      qb = cand;
      break;
    }
  if (forced == 16 || forced == 32 || forced == 64) qb = forced;
  switch (qb) {
    case 64: return launch_attention_qb<64>(qkv, out, n, T, C, st);
    case 32: return launch_attention_qb<32>(qkv, out, n, T, C, st);
    default: return launch_attention_qb<16>(qkv, out, n, T, C, st);
  }
}

int grid_for(long long items, int threads, int sms);

// K0: window batch [n, hw, cin_pad] bf16 from the resident trajectory (tiled form for 4-variable frames); f0 and
// win_list as gather_windows_kernel takes them.
int launch_gather(const float* traj, bf16* out, int n, int hw, int C, int w, int cin_pad, int f0, int sms, cudaStream_t st,
                  const int* win_list = nullptr) {
  static int tiled = -1;
  if (tiled < 0) {
    const char* e = getenv("C2W_GATHER_TILED");
    tiled = (e && e[0] == '0') ? 0 : 1;
  }
  if (!win_list && tiled && C == 4 && hw % kGatherPix == 0 && w <= 64) {
    const size_t smem = static_cast<size_t>(kGatherWin + w - 1) * kGatherPix * sizeof(uint2);
    gather_windows_tiled_kernel<<<dim3(hw / kGatherPix, (n + kGatherWin - 1) / kGatherWin), 256, smem, st>>>(traj, out, n, hw, w,
                                                                                                       cin_pad, f0);
  } else {
    const long long items = static_cast<long long>(n) * hw * (cin_pad / 8);
    gather_windows_kernel<<<grid_for(items, 256, sms), 256, 0, st>>>(traj, out, n, hw, C, w * C, cin_pad, f0, win_list);
  }
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

int grid_for(long long items, int threads, int sms) {
  long long b = (items + threads - 1) / threads;
  const long long cap = static_cast<long long>(sms) * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return static_cast<int>(b);
}

// ns samples: t_dev (device, ns values) or the scalar t for all; h0/emb: [ns, E], mods: [ns, total_mod]
int run_modulation(c2w_handle* h, float t, const float* t_dev, int ns, float* h0, float* emb, float* mods,
                   cudaStream_t st) {
  const int E = h->cfg.embedding_dim, nf = h->cfg.noise_features;
  time_embed_kernel<<<ns, 256, nf * sizeof(float), st>>>(t, t_dev, h->map0_w, h->map0_b, h0, E, nf);
  const float* fvec = nullptr;
  if (h->forcing != nullptr && h->plan.per_t && h->forcing_pad > 0) {  // + map_forcing(forcing), model/score.py:65-66
    const int fp = h->forcing_pad;
    pad_rows_kernel<<<ceil_div(static_cast<long long>(ns) * fp, 256), 256, 0, st>>>(h->forcing, h->plan.forc_pad, ns,
                                                                                  h->cfg.forcing_dim, fp);
    matvec_kernel<<<dim3(ceil_div(static_cast<long long>(E) * 32, 256), ns), 256, 0, st>>>(h->mapf_w, h->mapf_b, h->plan.forc_pad,
                                                                                        h->plan.fvec, E, fp, 0);
    fvec = h->plan.fvec;
    g_launches += 2;
  }
  matvec_kernel<<<dim3(ceil_div(static_cast<long long>(E) * 32, 256), ns), 256, 0, st>>>(h->map1_w, h->map1_b, h0, emb, E,
                                                                                      E, 1, fvec);
  if (h->total_mod > 0)  // a network without residual blocks has no modulation projections
    matvec_kernel<<<dim3(ceil_div(static_cast<long long>(h->total_mod) * 32, 256), ns), 256, 0, st>>>(
        h->proj_w, h->proj_b, emb, mods, h->total_mod, E, 0);
  g_launches += h->total_mod > 0 ? 3 : 2;
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

// Lays the workspace out and (if base != null) builds every launch of the forward pass over it.  vjp: the forward
// ops additionally stash (per block) the LayerNorm output + 1/std and the SiLU pre-activation, (per attention block)
// qkv, and the plan gets the input-gradient pass `bwd`.
int build_plan(c2w_handle* h, int n, bool vjp, bool per_t, void* base, size_t* bytes_out, bool train = false) {
  Plan& P = h->plan;
  const bool real = base != nullptr;
  Bump B(base);
  const int nl = h->nl;
  const long long HW0 = static_cast<long long>(h->cfg.height) * h->cfg.width;
  if (real) {
    P.ops.clear();
    P.bwd.clear();
    P.n_max = n;
    P.vjp = vjp;
    P.per_t = per_t;
    P.train = train;
    P.n_last = 0;
  }
  bf16* xin = B.take<bf16>(n * HW0 * h->cin_pad);
  const size_t ns = per_t ? n : 1;  // modulation vectors: one per sample or one for the batch
  float* h0 = B.take<float>(ns * h->cfg.embedding_dim);
  float* emb = B.take<float>(ns * h->cfg.embedding_dim);
  float* mods = B.take<float>(ns * h->total_mod);
  float* out32 = B.take<float>(n * HW0 * h->levels[0].tail.cout_pad);
  float* forc_pad = h->forcing_pad > 0 ? B.take<float>(ns * h->forcing_pad) : nullptr;
  float* fvec = h->forcing_pad > 0 ? B.take<float>(ns * h->cfg.embedding_dim) : nullptr;
  std::vector<bf16*> xs(nl), as(nl), hs(nl), gs(nl), ga(nl), gh(nl);
  size_t up_elems = 0, qkv_elems = 0, att_elems = 0;
  for (int l = 0; l < nl; ++l) {
    const LevelW& L = h->levels[l];
    const size_t e = static_cast<size_t>(n) * L.H * L.W * L.C;
    xs[l] = B.take<bf16>(e);
    as[l] = vjp ? nullptr : B.take<bf16>(e);  // vjp: every LayerNorm output gets its own stash buffer
    hs[l] = B.take<bf16>(e);
    if (vjp) {
      gs[l] = B.take<bf16>(e);
      ga[l] = B.take<bf16>(e);
      gh[l] = B.take<bf16>(e);
    }
    if (l > 0) {
      const LevelW& U = h->levels[l - 1];
      up_elems = std::max(up_elems, static_cast<size_t>(n) * U.H * U.W * L.C);
    }
    if (L.attn) {
      qkv_elems = std::max(qkv_elems, static_cast<size_t>(n) * L.H * L.W * 3 * L.C);
      att_elems = std::max(att_elems, e);
    }
  }
  bf16* up = vjp ? nullptr : B.take<bf16>(up_elems);
  bf16* qkv = vjp ? nullptr : B.take<bf16>(qkv_elems);
  bf16* att = B.take<bf16>(att_elems);
  bf16 *gup = nullptr, *gz = nullptr, *gqkv = nullptr, *gatt = nullptr, *cot = nullptr;
  float* attn_scratch = nullptr;
  if (vjp) {
    size_t sc = 0;
    for (int l = 0; l < nl; ++l)
      if (h->levels[l].attn) {
        const size_t T = static_cast<size_t>(h->levels[l].H) * h->levels[l].W;
        sc = std::max(sc, 2 * static_cast<size_t>(n) * T * T);
      }
    attn_scratch = B.take<float>(sc);
    gup = B.take<bf16>(up_elems);    // gradient w.r.t. the upsampled LayerNorm output of a tail
    gz = B.take<bf16>(up_elems);     // zero-inserted gradient of a stride-2 head
    gqkv = B.take<bf16>(qkv_elems);
    gatt = B.take<bf16>(att_elems);
    cot = B.take<bf16>(n * HW0 * h->levels[0].tail.cout_pad);
  }
  if (train) {  // parameter-gradient scratch: modulation gradients, split-K slabs, time-MLP backward
    const size_t E = h->cfg.embedding_dim, nf = h->cfg.noise_features;
    float* dmods = B.take<float>(static_cast<size_t>(n) * std::max(h->total_mod, 1));
    const size_t wg_floats = 12u * 1024u * 1024u;  // 48 MB: every layer's slabs fit (wgrad_launch_init trims the splits)
    float* wg = B.take<float>(wg_floats);
    float* feat = B.take<float>(n * nf);
    float* pre0 = B.take<float>(n * E);
    float* pre1 = B.take<float>(n * E);
    float* demb = B.take<float>(n * E);
    float* dh0 = B.take<float>(n * E);
    float* lp = B.take<float>(4096);
    if (real) {
      P.dmods = dmods;
      P.wg_scratch = wg;
      P.wg_scratch_floats = wg_floats;
      P.feat = feat;
      P.pre0 = pre0;
      P.pre1 = pre1;
      P.demb = demb;
      P.dh0 = dh0;
      P.loss_partials = lp;
    }
  }
  // per-block stash buffers are taken on the fly below (same order in the sizing and the real pass)
  auto stash = [&](size_t elems) -> bf16* { return B.take<bf16>(elems); };
  auto stash_f = [&](size_t elems) -> float* { return B.take<float>(elems); };

  if (real) {
    P.xin = xin;
    P.h0 = h0;
    P.emb = emb;
    P.mods = mods;
    P.out32 = out32;
    P.forc_pad = forc_pad;
    P.fvec = fvec;
    P.cot = cot;
    P.g0 = vjp ? gs[0] : nullptr;
  }

  // H, W: INPUT image size; stride 2 halves it (heads of levels > 0, model/nn.py:169-176)
  auto make_conv = [&](Op* op, bool c3, const bf16* in, int H, int W, int cin, const bf16* wts, const float* bias,
                       int cout_pad, int mode, bf16* out, bool is_final, int stride, int bn_force = 0) -> int {
    op->kind = OP_CONV;
    op->spec.c3 = c3;
    op->spec.in = in;
    op->spec.H = H;
    op->spec.W = W;
    op->spec.cin = cin;
    op->spec.wts = wts;
    op->spec.bias = bias;
    op->spec.cout_pad = cout_pad;
    op->spec.mode = mode;
    op->spec.out = out;
    op->spec.stride = stride;
    // the fp32 / compose epilogues (the last conv of a pass) store 64-wide tiles only; a wider frame (C * window > 64
    // channels) takes several of them
    const int bn = bn_force ? bn_force : mode == EPI_F32 ? 64 : conv_pick_bn_tiled(cout_pad, c3, n, H, W, stride, h->sms);
    if (!conv_launch_init(&op->conv, c3, in, n, H, W, cin, wts, cout_pad, bn, h->sms, stride))
      return fail(C2W_ERR_INVALID, "cannot build conv launch (n=%d H=%d W=%d cin=%d cout=%d stride=%d) %s", n, H, W, cin,
                  cout_pad, stride, tmap_error_slot());
    op->conv.p.mode = mode;
    op->conv.p.bias = bias;
    if (out && !conv_launch_set_out(&op->conv, out)) return fail(C2W_ERR_CUDA, "cannot encode the output tensor map");
    op->pix_per_img = (H / stride) * (W / stride);
    op->is_final = is_final;
    return C2W_OK;
  };
  auto add_conv = [&](bool c3, const bf16* in, int H, int W, int cin, const ConvW& w, int mode, bf16* out, bool is_final,
                      int stride = 1) -> int {
    if (!real) return C2W_OK;
    Op op;
    int rc = make_conv(&op, c3, in, H, W, cin, w.w, w.b, w.cout_pad, mode, out, is_final, stride);
    if (rc) return rc;
    P.ops.push_back(op);
    return C2W_OK;
  };
  // input-gradient conv: the transposed / flipped weights, no bias; pushed on `unit` (a backward op group)
  auto add_dconv = [&](std::vector<Op>& unit, bool c3, const bf16* gin, int H, int W, const ConvW& w, int mode,
                       bf16* gout, const bf16* aux) -> int {
    if (!real) return C2W_OK;
    Op op;
    // forward cout is this conv's K side, forward cin its N side
    int rc = make_conv(&op, c3, gin, H, W, w.cout_pad, w.wd, h->zero_bias, w.cin_pad, mode, gout, false, 1);
    if (rc) return rc;
    (void)aux;
    unit.push_back(op);
    return C2W_OK;
  };
  // Channel LayerNorm of `in` (+ modulation) -> `out` (+ inv).  When `in` was just produced by a conv whose single N
  // tile holds all C channels of a pixel, the normalisation is done in that conv's epilogue (no extra HBM pass).
  auto add_ln = [&](const bf16* in, bf16* out, float* inv, int C, int H, int W, int upf, int mod_off) {
    if (!real) return;
    // one diffusion time per sample (training): the fused form takes a per-image modulation vector; LayerNorms without
    // modulation (attention, tails) fuse as usual
    const int mod_stride = (per_t && mod_off >= 0) ? h->total_mod : 0;
    if (h->fuse_ln && !P.ops.empty()) {
      Op& prev = P.ops.back();
      if (prev.kind == OP_CONV && !prev.is_final && prev.conv.out_ptr == in && prev.conv.cout_pad == C &&
          prev.conv.p.num_n_tiles != 1 && (C == 128 || C == 256)) {
        // the tile picker split this layer for a fuller last wave; the fused LayerNorm is worth more than that
        Op whole;
        const Op::ConvSpec& sp = prev.spec;
        if (make_conv(&whole, sp.c3, sp.in, sp.H, sp.W, sp.cin, sp.wts, sp.bias, sp.cout_pad, sp.mode, sp.out, false,
                      sp.stride, C) == C2W_OK && conv_launch_can_ln(&whole.conv, upf))
          prev = whole;
      }
      if (prev.kind == OP_CONV && !prev.is_final && prev.conv.out_ptr == in && prev.conv.cout_pad == C &&
          conv_launch_can_ln(&prev.conv, upf) &&
          conv_launch_set_ln(&prev.conv, out, mod_off >= 0 ? mods + mod_off : nullptr, upf, mod_stride)) {
        prev.conv.p.ln_inv = inv;
        return;
      }
    }
    Op op;
    op.kind = OP_LN;
    op.in = in;
    op.out = out;
    op.inv = inv;
    op.C = C;
    op.H = H;
    op.W = W;
    op.up = upf;
    op.mod_off = mod_off;
    P.ops.push_back(op);
  };
  // training: dW (+ bias gradient) of the conv that read `x` (input image H x W) and whose output gradient is `dy`
  auto add_wgrad = [&](std::vector<Op>& unit, bool c3, const bf16* x, const bf16* dy, int H, int W, const ConvW& w,
                       int stride) {
    if (!real || !train) return;
    if (w.gw >= 0) {
      Op op;
      op.kind = OP_WGRAD;
      op.spec.c3 = c3;
      op.spec.in = x;
      op.in = dy;
      op.spec.H = H;
      op.spec.W = W;
      op.spec.cin = w.cin_pad;
      op.spec.cout_pad = w.cout_pad;
      op.spec.stride = stride;
      op.dst = w.gw;
      op.dst_bias = w.gb;  // the bias gradient (column sums of dy) is collected by the same GEMM
      op.cin_real = w.cin;
      op.cout_real = w.cout;
      unit.push_back(op);
    }
  };
  auto add_ln_bwd = [&](std::vector<Op>& unit, const bf16* gy, const bf16* y, const float* inv, const bf16* gres,
                        bf16* out, int C, int H, int W, int down, int mod_off = -1) {
    if (!real) return;
    Op op;
    op.kind = OP_LN_BWD;
    op.mod_off = train ? mod_off : -1;
    op.in = gy;
    op.aux = y;
    op.inv = const_cast<float*>(inv);
    op.res = gres;
    op.out = out;
    op.C = C;
    op.H = H;
    op.W = W;
    op.up = down;
    unit.push_back(op);
  };

  // Backward op groups are collected per forward unit and replayed in reverse unit order.
  std::vector<std::vector<Op>> units;

  auto add_blocks = [&](int l, const std::vector<BlockW>& blocks, const std::vector<AttnW>& attns) -> int {
    const LevelW& L = h->levels[l];
    const size_t e = static_cast<size_t>(n) * L.H * L.W * L.C;
    const size_t npix = static_cast<size_t>(n) * L.H * L.W;
    for (size_t b = 0; b < blocks.size(); ++b) {
      const BlockW& bw = blocks[b];
      // x + conv2(SiLU(conv1(LN(x + proj(emb)))))    model/nn.py:27-28,151-158
      bf16* y = vjp ? stash(e) : as[l];
      bf16* pre = vjp ? stash(e) : nullptr;
      float* inv = vjp ? stash_f(npix) : nullptr;
      // training keeps every block's SiLU output (conv2's wgrad operand) instead of recomputing it from `pre`
      bf16* hsb = train ? stash(e) : hs[l];
      add_ln(xs[l], y, inv, L.C, L.H, L.W, 0, bw.mod_off);
      int rc;
      bool dual_done = false;
      if (vjp && real && h->fuse_dual) {  // pre-activation AND its SiLU as two TMA-stored outputs of conv1's epilogue
        Op op;
        rc = make_conv(&op, true, y, L.H, L.W, L.C, bw.c1.w, bw.c1.b, bw.c1.cout_pad, EPI_BIAS_SILU_DUAL, pre, false, 1);
        if (rc) return rc;
        if (conv_launch_set_out2(&op.conv, hsb)) {
          P.ops.push_back(op);
          dual_done = true;
        }
      }
      if (vjp && dual_done) {
      } else if (vjp) {  // the pre-activation is stashed; SiLU is a separate elementwise pass
        rc = add_conv(true, y, L.H, L.W, L.C, bw.c1, EPI_BIAS, pre, false);
        if (rc) return rc;
        if (real) {
          Op op;
          op.kind = OP_SILU;
          op.aux = pre;
          op.in = nullptr;
          op.out = hsb;
          op.C = L.C;
          op.H = L.H;
          op.W = L.W;
          op.up = 0;
          P.ops.push_back(op);
        }
      } else {
        rc = add_conv(true, y, L.H, L.W, L.C, bw.c1, EPI_BIAS_SILU, hsb, false);
        if (rc) return rc;
      }
      rc = add_conv(true, hsb, L.H, L.W, L.C, bw.c2, EPI_BIAS_RES, xs[l], false);
      if (rc) return rc;
      if (vjp) {
        units.emplace_back();
        std::vector<Op>& u = units.back();
        add_wgrad(u, true, hsb, gs[l], L.H, L.W, bw.c2, 1);  // conv2's input: this block's stashed SiLU output
        if (h->fuse_dsilu) {
          // conv2's input gradient times silu'(pre), written in place over the stashed pre-activation (the epilogue
          // prefetches `pre` like a residual tile), then conv1's input gradient from it
          if ((rc = add_dconv(u, true, gs[l], L.H, L.W, bw.c2, EPI_MUL_DSILU, pre, nullptr))) return rc;
          add_wgrad(u, true, y, pre, L.H, L.W, bw.c1, 1);
          if ((rc = add_dconv(u, true, pre, L.H, L.W, bw.c1, EPI_BIAS, ga[l], nullptr))) return rc;
        } else {
          if ((rc = add_dconv(u, true, gs[l], L.H, L.W, bw.c2, EPI_BIAS, gh[l], nullptr))) return rc;
          if (real) {  // gh *= silu'(pre)
            Op op;
            op.kind = OP_SILU;
            op.aux = pre;
            op.in = gh[l];
            op.out = gh[l];
            op.C = L.C;
            op.H = L.H;
            op.W = L.W;
            op.up = 1;
            u.push_back(op);
          }
          add_wgrad(u, true, y, gh[l], L.H, L.W, bw.c1, 1);
          if ((rc = add_dconv(u, true, gh[l], L.H, L.W, bw.c1, EPI_BIAS, ga[l], nullptr))) return rc;
        }
        add_ln_bwd(u, ga[l], y, inv, gs[l], gs[l], L.C, L.H, L.W, 0, bw.mod_off);
      }
      if (L.attn) {
        // x + proj(attn(qkv(LN(x))))    model/nn.py:50-60
        const AttnW& aw = attns[b];
        const int T = L.H * L.W;
        bf16* ya = vjp ? stash(e) : as[l];
        float* inva = vjp ? stash_f(npix) : nullptr;
        bf16* q = vjp ? stash(3 * e) : qkv;
        bf16* att_s = train ? stash(e) : att;  // training keeps the attention output: it is the proj conv's wgrad operand
        add_ln(xs[l], ya, inva, L.C, L.H, L.W, 0, -1);
        rc = add_conv(false, ya, L.H, L.W, L.C, aw.qkv, EPI_BIAS, q, false);
        if (rc) return rc;
        if (real) {
          Op op;
          op.kind = OP_ATTN;
          op.in = q;
          op.out = att_s;
          op.T = T;
          op.C = L.C;
          P.ops.push_back(op);
          P.attn_smem = std::max(P.attn_smem, attention_smem_bytes(op.T, op.C));
          if (P.attn_smem > static_cast<size_t>(kSmemLimit))
            return fail(C2W_ERR_INVALID, "attention at level %d (T=%d, C=%d) exceeds shared memory", l, op.T, op.C);
        }
        rc = add_conv(false, att_s, L.H, L.W, L.C, aw.proj, EPI_BIAS_RES, xs[l], false);
        if (rc) return rc;
        if (vjp) {
          units.emplace_back();
          std::vector<Op>& u = units.back();
          add_wgrad(u, false, att_s, gs[l], L.H, L.W, aw.proj, 1);
          if ((rc = add_dconv(u, false, gs[l], L.H, L.W, aw.proj, EPI_BIAS, gatt, nullptr))) return rc;
          if (real) {
            Op op;
            op.kind = OP_ATTN_BWD;
            op.inv = attn_scratch;
            op.in = gatt;
            op.aux = q;
            op.out = gqkv;
            op.T = T;
            op.C = L.C;
            u.push_back(op);
          }
          add_wgrad(u, false, ya, gqkv, L.H, L.W, aw.qkv, 1);
          if ((rc = add_dconv(u, false, gqkv, L.H, L.W, aw.qkv, EPI_BIAS, ga[l], nullptr))) return rc;
          add_ln_bwd(u, ga[l], ya, inva, gs[l], gs[l], L.C, L.H, L.W, 0);
        }
      }
    }
    return C2W_OK;
  };

  // descent (model/nn.py:223-229)
  for (int l = 0; l < nl; ++l) {
    const LevelW& L = h->levels[l];
    int rc;
    if (l == 0) {
      rc = add_conv(true, xin, L.H, L.W, h->cin_pad, L.head, EPI_BIAS, xs[0], false);
      if (rc) return rc;
      if (vjp) {  // gradient w.r.t. the window batch, fp32 [n, HW, cin_pad] into out32
        units.emplace_back();
        add_wgrad(units.back(), true, xin, gs[0], L.H, L.W, L.head, 1);
        if ((rc = add_dconv(units.back(), true, gs[0], L.H, L.W, L.head, EPI_F32, nullptr, nullptr))) return rc;
        if (real) units.back().back().conv.p.out_f32 = out32;
      }
    } else {
      const LevelW& U = h->levels[l - 1];
      // training: the skip value xs[l-1] is the head conv's wgrad operand, but the ascent later accumulates into it
      bf16* skip = train ? stash(static_cast<size_t>(n) * U.H * U.W * U.C) : nullptr;
      if (train && real) {
        Op op;
        op.kind = OP_COPY;
        op.in = xs[l - 1];
        op.out = skip;
        op.C = U.C;
        op.H = U.H;
        op.W = U.W;
        P.ops.push_back(op);
      }
      rc = add_conv(true, xs[l - 1], U.H, U.W, U.C, L.head, EPI_BIAS, xs[l], false, 2);
      if (rc) return rc;
      if (vjp) {  // g[l-1] += conv_flipped(zero-upsampled g[l])
        units.emplace_back();
        std::vector<Op>& u = units.back();
        add_wgrad(u, true, skip, gs[l], U.H, U.W, L.head, 2);
        if (real) {
          Op op;
          op.kind = OP_ZERO_UP;
          op.in = gs[l];
          op.out = gz;
          op.H = L.H;
          op.W = L.W;
          op.C = L.C;
          u.push_back(op);
        }
        if ((rc = add_dconv(u, true, gz, U.H, U.W, L.head, EPI_BIAS_RES, gs[l - 1], nullptr))) return rc;
      }
    }
    rc = add_blocks(l, L.desc, L.dattn);
    if (rc) return rc;
  }
  // ascent (model/nn.py:233-240): blocks, then tail = LN -> nearest x2 -> conv, + skip (in place into the skip)
  for (int l = nl - 1; l >= 0; --l) {
    const LevelW& L = h->levels[l];
    int rc = add_blocks(l, L.asc, L.aattn);
    if (rc) return rc;
    if (l > 0) {
      const LevelW& U = h->levels[l - 1];
      const size_t eu = static_cast<size_t>(n) * U.H * U.W * L.C;
      bf16* upl = vjp ? stash(eu) : up;
      float* invt = vjp ? stash_f(static_cast<size_t>(n) * L.H * L.W) : nullptr;
      add_ln(xs[l], upl, invt, L.C, L.H, L.W, 1, -1);
      rc = add_conv(true, upl, U.H, U.W, L.C, L.tail, EPI_BIAS_RES, xs[l - 1], false);
      if (rc) return rc;
      if (vjp) {  // g[l] = LN_bwd(sum_2x2 conv_flipped(g[l-1]))   (xs[l] feeds nothing else)
        units.emplace_back();
        std::vector<Op>& u = units.back();
        add_wgrad(u, true, upl, gs[l - 1], U.H, U.W, L.tail, 1);
        if ((rc = add_dconv(u, true, gs[l - 1], U.H, U.W, L.tail, EPI_BIAS, gup, nullptr))) return rc;
        add_ln_bwd(u, gup, upl, invt, nullptr, gs[l], L.C, L.H, L.W, 1);
      }
    } else {
      rc = add_conv(true, xs[0], L.H, L.W, L.C, L.tail, EPI_F32, nullptr, true);
      if (rc) return rc;
      if (vjp) {
        units.emplace_back();
        add_wgrad(units.back(), true, xs[0], cot, L.H, L.W, L.tail, 1);
        if ((rc = add_dconv(units.back(), true, cot, L.H, L.W, L.tail, EPI_BIAS, gs[0], nullptr))) return rc;
      }
    }
  }
  *bytes_out = B.off + 1024;
  if (real && vjp)
    for (auto it = units.rbegin(); it != units.rend(); ++it)
      for (const Op& op : *it) P.bwd.push_back(op);
  return C2W_OK;
}

struct SpanGuard {
  c2w_handle* h;
  cudaStream_t st;
  TimedSpan* sp = nullptr;
  SpanGuard(c2w_handle* h_, int cls, cudaStream_t st_) : h(h_), st(st_) {
    ++g_launches;
    if (!h->timing) return;
    if (h->spans_used == h->spans.size()) {
      TimedSpan t;
      t.cls = cls;
      cudaEventCreate(&t.e0);
      cudaEventCreate(&t.e1);
      h->spans.push_back(t);
    }
    sp = &h->spans[h->spans_used++];
    sp->cls = cls;
    cudaEventRecord(sp->e0, st);
  }
  ~SpanGuard() {
    if (sp) cudaEventRecord(sp->e1, st);
  }
};

struct FinalSpec {
  int mode;  // EPI_F32 or EPI_COMPOSE
  float* eps = nullptr;
  int order_k = 0, win_first = 0, win_last_global = 0, frame_base = 0;
  const int* win_list = nullptr;  // EPI_COMPOSE over a selection of windows
};

// Runs an op list (the forward pass, or the input-gradient pass) on the first nn windows of the plan.
int run_ops(c2w_handle* h, std::vector<Op>& ops, int nn, const FinalSpec& fs, cudaStream_t st) {
  Plan& P = h->plan;
  for (Op& op : ops) {
    switch (op.kind) {
      case OP_CONV: {
        ConvLaunch L = op.conv;
        const long long m_total = static_cast<long long>(nn) * op.pix_per_img;
        L.p.m_total = static_cast<int>(m_total);
        L.p.num_m_tiles = ceil_div(m_total, kBlockM);
        conv_set_grid(&L, h->sms);
#ifdef C2W_DIAG
        {  // diagnostics build only: timing experiments inside a real step (results are garbage) — C2W_SKIP_LOADS=1/3/4
          static int skip = -1;
          if (skip < 0) {
            const char* e = getenv("C2W_SKIP_LOADS");
            skip = e ? atoi(e) : 0;
          }
          L.p.dbg_skip_loads = skip;
        }
#endif
        if (op.is_final) {
          L.p.mode = fs.mode;
          L.p.out_f32 = P.out32;
          L.p.eps = fs.eps;
          L.p.hw = op.pix_per_img;
          L.p.order_k = fs.order_k;
          L.p.win_first = fs.win_first;
          L.p.win_last_global = fs.win_last_global;
          L.p.frame_base = fs.frame_base;
          L.p.win_list = fs.win_list;
        }
#ifdef C2W_DIAG
        if (h->timeline != nullptr && h->timeline_used < h->timeline_cap) L.p.dbg_timeline = h->timeline + 2 * h->timeline_used++;
#endif
        {
          SpanGuard sg(h, 0, st);
          C2W_CUDA(conv_launch(L, st));
        }
        break;
      }
      case OP_LN: {
        SpanGuard sg(h, 1, st);
        int rc = launch_ln(op.in, op.mod_off >= 0 ? P.mods + op.mod_off : nullptr, op.out, op.inv,
                           static_cast<long long>(nn) * op.H * op.W, op.C, op.H, op.W, op.up, h->sms, st,
                           P.per_t ? h->total_mod : 0);
        if (rc) return rc;
        break;
      }
      case OP_ATTN: {
        SpanGuard sg(h, 1, st);
        int rc = launch_attention(op.in, op.out, nn, op.T, op.C, st);
        if (rc) return rc;
        break;
      }
      case OP_LN_BWD: {
        SpanGuard sg(h, 1, st);
        float* dmod = (P.train && op.mod_off >= 0) ? P.dmods + op.mod_off : nullptr;
        int rc = launch_ln_bwd(op.in, op.aux, op.inv, op.res, op.out, static_cast<long long>(nn) * op.H * op.W, op.C, op.H,
                               op.W, op.up, h->sms, st, dmod, h->total_mod);
        if (rc) return rc;
        break;
      }
      case OP_COPY: {
        SpanGuard sg(h, 1, st);
        C2W_CUDA(cudaMemcpyAsync(op.out, op.in, static_cast<size_t>(nn) * op.H * op.W * op.C * sizeof(bf16),
                                 cudaMemcpyDeviceToDevice, st));
        break;
      }
      case OP_WGRAD: {
        if (op.wg_n != nn) {
          if (!wgrad_launch_init(&op.wg, op.spec.c3, op.spec.in, op.in, nn, op.spec.H, op.spec.W, op.spec.cin,
                                 op.spec.cout_pad, op.spec.stride, h->sms, P.wg_scratch, P.wg_scratch_floats))
            return fail(C2W_ERR_INVALID, "cannot build wgrad launch (n=%d H=%d W=%d cin=%d cout=%d stride=%d conv3x3=%d) %s", nn,
                        op.spec.H, op.spec.W, op.spec.cin, op.spec.cout_pad, op.spec.stride, (int)op.spec.c3,
                        tmap_error_slot());
          op.wg_n = nn;
        }
        SpanGuard sg(h, 0, st);
        ++g_launches;  // GEMM + slab reduction
        C2W_CUDA(wgrad_run(op.wg, P.grad + op.dst, op.cout_real, op.cin_real, 1, 1.0f, st,
                           op.dst_bias >= 0 ? P.grad + op.dst_bias : nullptr));
        break;
      }
      case OP_COLSUM: {
        SpanGuard sg(h, 1, st);
        const long long rows = static_cast<long long>(nn) * op.H * op.W;
        C2W_CUDA(colsum_run(op.in, P.grad + op.dst, rows, op.C, rows, 0, 1.0f, st, op.cout_real));
        break;
      }
      case OP_ATTN_BWD: {
        SpanGuard sg(h, 1, st);
        int rc = launch_attention_bwd(op.aux, op.in, op.out, op.inv, nn, op.T, op.C, st);
        if (rc) return rc;
        break;
      }
      case OP_SILU: {
        SpanGuard sg(h, 1, st);
        const long long n8 = static_cast<long long>(nn) * op.H * op.W * op.C / 8;
        silu_elementwise_kernel<<<grid_for(n8, 256, h->sms), 256, 0, st>>>(op.aux, op.in, op.out, n8, op.up);
        C2W_CUDA(cudaGetLastError());
        break;
      }
      case OP_ZERO_UP: {
        SpanGuard sg(h, 1, st);
        const long long items = static_cast<long long>(nn) * (2 * op.H) * (2 * op.W) * (op.C / 8);
        zero_upsample_kernel<<<grid_for(items, 256, h->sms), 256, 0, st>>>(op.in, op.out, nn, op.H, op.W, op.C);
        C2W_CUDA(cudaGetLastError());
        break;
      }
    }
  }
  return C2W_OK;
}

int run_plan(c2w_handle* h, int nn, const FinalSpec& fs, cudaStream_t st) { return run_ops(h, h->plan.ops, nn, fs, st); }

// Launches a frame kernel of kernels.cuh (guidance, corrector, window adjoints) instantiated for a runtime count of
// variables per frame: launch(std::integral_constant<int, C>{}) for 1 <= C <= C2W_MAX_VARS.
template <class F>
int launch_for_vars(int C, F&& launch) {
  static_assert(C2W_MAX_VARS == 8, "one case per variable count");
  switch (C) {
    case 1: launch(std::integral_constant<int, 1>{}); break;
    case 2: launch(std::integral_constant<int, 2>{}); break;
    case 3: launch(std::integral_constant<int, 3>{}); break;
    case 4: launch(std::integral_constant<int, 4>{}); break;
    case 5: launch(std::integral_constant<int, 5>{}); break;
    case 6: launch(std::integral_constant<int, 6>{}); break;
    case 7: launch(std::integral_constant<int, 7>{}); break;
    case 8: launch(std::integral_constant<int, 8>{}); break;
    default: return fail(C2W_ERR_INVALID, "1 to %d variables per frame (got %d)", C2W_MAX_VARS, C);
  }
  ++g_launches;
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

// The windows of a window-score call: the contiguous global windows [first, first + n) when list is null, else the
// global windows list[0..n) (device array).  pos (device, n_win_global entries, backward of a list only): the place of
// global window j in the list, or -1.
struct WindowSet {
  int first, n;
  const int* list;
  const int* pos;
};

// Gather -> UNet -> fold into eps, in chunks of the bound workspace.  eps == null: no fold, the window outputs stay
// stashed in a VJP workspace for the backward that follows.
int window_score_fwd(c2w_handle* h, const float* traj, int frame_global0, const WindowSet& ws, int n_win_global, float t,
                     float* eps, cudaStream_t st) {
  Plan& P = h->plan;
  const int w = h->cfg.window, k = w / 2, C = h->cfg.frame_channels;
  const int hw = h->cfg.height * h->cfg.width;
  int rc = run_modulation(h, t, nullptr, 1, P.h0, P.emb, P.mods, st);
  if (rc) return rc;
  for (int c0 = 0; c0 < ws.n; c0 += P.n_max) {
    const int nn = std::min(P.n_max, ws.n - c0);
    const int j0 = ws.first + c0;  // first window of the chunk (contiguous windows)
    const int* list = ws.list ? ws.list + c0 : nullptr;
    if ((rc = launch_gather(traj, P.xin, nn, hw, C, w, h->cin_pad, list ? frame_global0 : j0 - frame_global0, h->sms, st,
                            list)))
      return rc;
    ++g_launches;
    FinalSpec fs;
    fs.mode = EPI_F32;
    if (eps && C == 4) {  // the fold is the last conv's epilogue
      fs.mode = EPI_COMPOSE;
      fs.eps = eps;
      fs.order_k = k;
      fs.win_first = j0;
      fs.win_last_global = n_win_global - 1;
      fs.frame_base = frame_global0;
      fs.win_list = list;
    }
    if ((rc = run_plan(h, nn, fs, st))) return rc;
    if (eps && C != 4) {  // any other variable count: the fold as its own pass over the fp32 window outputs
      const long long items = static_cast<long long>(nn) * hw * C;
      compose_generic_kernel<<<grid_for(items, 256, h->sms), 256, 0, st>>>(P.out32, eps, nn, hw, h->levels[0].tail.cout_pad,
                                                                           C, k, j0, n_win_global - 1, frame_global0, list);
      ++g_launches;
      C2W_CUDA(cudaGetLastError());
    }
  }
  return C2W_OK;
}

// Compose adjoint -> input-gradient pass -> unfold adjoint of the windows whose stashing forward has just run (one
// chunk).  vjp (fp32 [n_frames_local, H, W, C]) is accumulated on the frames the windows touch.
int window_score_bwd(c2w_handle* h, const float* cot, int n_frames_local, int frame_global0, const WindowSet& ws,
                     int n_win_global, float* vjp, cudaStream_t st) {
  Plan& P = h->plan;
  const int w = h->cfg.window, k = w / 2;
  const int hw = h->cfg.height * h->cfg.width;
  const int cpad = h->levels[0].tail.cout_pad;
  const long long items = static_cast<long long>(ws.n) * hw * (cpad / 8);
  int rc = launch_for_vars(h->cfg.frame_channels, [&](auto vars) {
    compose_adjoint_kernel<decltype(vars)::value><<<grid_for(items, 256, h->sms), 256, 0, st>>>(
        cot, P.cot, ws.n, hw, cpad, k, ws.first, n_win_global - 1, frame_global0, ws.list);
  });
  if (rc) return rc;
  FinalSpec fs;
  fs.mode = EPI_F32;
  if ((rc = run_ops(h, P.bwd, ws.n, fs, st))) return rc;
  // the local frames the windows can touch: the n + w - 1 of a contiguous range, every one for a list
  const int f_lo = ws.list ? 0 : ws.first - frame_global0;
  const int nf = ws.list ? n_frames_local : ws.n + w - 1;
  const long long items2 = static_cast<long long>(nf) * hw;
  return launch_for_vars(h->cfg.frame_channels, [&](auto vars) {
    unfold_adjoint_kernel<decltype(vars)::value><<<grid_for(items2, 256, h->sms), 256, 0, st>>>(
        P.out32, vjp, ws.n, f_lo, nf, hw, h->cin_pad, w, ws.first, frame_global0, n_win_global, ws.pos);
  });
}

}  // namespace

extern "C" {

int c2w_abi_version(void) { return 3; }

int c2w_struct_size(int which) {
  switch (which) {
    case 0: return static_cast<int>(sizeof(c2w_config));
    case 1: return static_cast<int>(sizeof(c2w_guide));
    case 2: return static_cast<int>(sizeof(c2w_adamw));
    case 3: return static_cast<int>(sizeof(c2w_conv_desc));
    case 4: return static_cast<int>(sizeof(c2w_point_obs));
    default: return -1;
  }
}
const char* c2w_last_error(void) { return error_slot(); }

int c2w_create(const c2w_config* cfg, c2w_handle** out) {
  C2W_REQUIRE(cfg && out, "c2w_create: null argument");
  C2W_REQUIRE(cfg->n_levels >= 1 && cfg->n_levels <= C2W_MAX_LEVELS, "n_levels=%d out of range", cfg->n_levels);
  C2W_REQUIRE(cfg->frame_channels >= 1 && cfg->window >= 1 && (cfg->window % 2) == 1, "window must be odd, got %d",
              cfg->window);
  C2W_REQUIRE(cfg->embedding_dim % 4 == 0 && cfg->noise_features % 2 == 0 && cfg->noise_features <= 256,
              "embedding_dim %% 4 == 0 and even noise_features <= 256 required");
  int H = cfg->height, W = cfg->width;
  for (int l = 0; l < cfg->n_levels; ++l) {
    C2W_REQUIRE(cfg->hidden_channels[l] % 64 == 0 && cfg->hidden_channels[l] <= 512,
                "hidden_channels[%d]=%d: must be a multiple of 64 and <= 512", l, cfg->hidden_channels[l]);
    C2W_REQUIRE(W >= 8 && W <= 128 && 128 % W == 0 && H >= 1, "level %d: width %d must be a power of two in [8,128]", l, W);
    const int th = std::min(H, 128 / W);
    C2W_REQUIRE(H % th == 0 && 128 % (W * th) == 0, "level %d: %dx%d does not tile into 128-pixel row blocks", l, H, W);
    if (l + 1 < cfg->n_levels) {
      C2W_REQUIRE(H % 2 == 0 && W % 2 == 0, "level %d: %dx%d not divisible by the stride", l, H, W);
      H /= 2;
      W /= 2;
    }
  }
  C2W_REQUIRE(cfg->forcing_dim >= 0 && cfg->forcing_dim <= 4096, "forcing_dim=%d out of range", cfg->forcing_dim);
  int sms = c2w_num_sms();
  C2W_REQUIRE(sms > 0, "c2w_create: no CUDA device available (this library has no CPU path)");
  c2w_handle* h = new c2w_handle();
  h->cfg = *cfg;
  h->nl = cfg->n_levels;
  h->cin = cfg->frame_channels * cfg->window;
  h->cin_pad = pad64(h->cin);
  h->sms = sms;
  {
    const char* e = getenv("C2W_NO_FUSE_LN");
    h->fuse_ln = !(e && e[0] == '1');
    const char* e2 = getenv("C2W_NO_FUSE_DSILU");
    h->fuse_dsilu = !(e2 && e2[0] == '1');
    const char* e3 = getenv("C2W_NO_FUSE_DUAL");
    h->fuse_dual = !(e3 && e3[0] == '1');
  }
  *out = h;
  return C2W_OK;
}

void c2w_destroy(c2w_handle* h) {
  if (!h) return;
  for (void* p : h->allocs) cudaFree(p);
  delete h;
}

int c2w_load_weight(c2w_handle* h, const char* name, const float* host_data, int64_t numel) {
  C2W_REQUIRE(h && name && host_data && numel > 0, "c2w_load_weight: bad argument");
  if (h->finalized) return fail(C2W_ERR_STATE, "weights already finalised");
  if (!h->raw.count(name)) h->params.emplace_back(name, static_cast<long long>(numel));
  h->raw[name].assign(host_data, host_data + numel);
  return C2W_OK;
}

int c2w_finalize_weights(c2w_handle* h) {
  C2W_REQUIRE(h, "null handle");
  if (h->finalized) return fail(C2W_ERR_STATE, "weights already finalised");
  const c2w_config& c = h->cfg;
  const int E = c.embedding_dim, nl = h->nl;
  int rc;
  {  // flat gradient layout: parameters in loading order (= state_dict order), each start aligned to 4 floats
    long long off = 0;
    for (auto& pr : h->params) {
      h->param_off[pr.first] = off;
      off += (pr.second + 3) / 4 * 4;
    }
    h->param_total = off;
  }
  if ((rc = upload_named(h, "map_layer0.weight", static_cast<size_t>(E) * c.noise_features, &h->map0_w))) return rc;
  if ((rc = upload_named(h, "map_layer0.bias", E, &h->map0_b))) return rc;
  if ((rc = upload_named(h, "map_layer1.weight", static_cast<size_t>(E) * E, &h->map1_w))) return rc;
  if ((rc = upload_named(h, "map_layer1.bias", E, &h->map1_b))) return rc;
  if (c.forcing_dim > 0) {
    const std::vector<float>*fw, *fb;
    if ((rc = need(h, "map_forcing.weight", static_cast<size_t>(E) * c.forcing_dim, &fw))) return rc;
    if ((rc = need(h, "map_forcing.bias", E, &fb))) return rc;
    h->forcing_pad = (c.forcing_dim + 3) / 4 * 4;
    std::vector<float> padded(static_cast<size_t>(E) * h->forcing_pad, 0.f);
    for (int r = 0; r < E; ++r)
      for (int j = 0; j < c.forcing_dim; ++j) padded[static_cast<size_t>(r) * h->forcing_pad + j] = (*fw)[static_cast<size_t>(r) * c.forcing_dim + j];
    if ((rc = dev_upload(h, padded.data(), padded.size() * sizeof(float), reinterpret_cast<void**>(&h->mapf_w)))) return rc;
    if ((rc = dev_upload(h, fb->data(), E * sizeof(float), reinterpret_cast<void**>(&h->mapf_b)))) return rc;
  }
  h->levels.assign(nl, LevelW());
  std::vector<float> proj_w, proj_b;
  int H = c.height, W = c.width;
  for (int l = 0; l < nl; ++l) {
    LevelW& L = h->levels[l];
    const int rev = nl - 1 - l;
    L.C = c.hidden_channels[l];
    L.H = H;
    L.W = W;
    L.attn = (c.attention_mask >> l) & 1;
    char buf[128];
    if (l == 0) {
      if ((rc = pack_conv(h, "unet.heads.0", L.C, h->cin, 9, &L.head))) return rc;
      snprintf(buf, sizeof buf, "unet.tails.%d", rev);
      if ((rc = pack_conv(h, buf, h->cin, L.C, 9, &L.tail))) return rc;
    } else {
      const int Cu = c.hidden_channels[l - 1];
      snprintf(buf, sizeof buf, "unet.heads.%d.0", l);
      if ((rc = pack_conv(h, buf, L.C, Cu, 9, &L.head))) return rc;
      snprintf(buf, sizeof buf, "unet.tails.%d.2", rev);
      if ((rc = pack_conv(h, buf, Cu, L.C, 9, &L.tail))) return rc;
    }
    const int step = L.attn ? 2 : 1;
    for (int side = 0; side < 2; ++side) {
      std::vector<BlockW>& blocks = side == 0 ? L.desc : L.asc;
      std::vector<AttnW>& attns = side == 0 ? L.dattn : L.aattn;
      for (int b = 0; b < c.hidden_blocks[l]; ++b) {
        snprintf(buf, sizeof buf, "unet.%s.%d.%d", side == 0 ? "descent" : "ascent", side == 0 ? l : rev, b * step);
        const std::string p(buf);
        BlockW bw;
        const std::vector<float>*pw, *pb;
        if ((rc = need(h, p + ".project.0.weight", static_cast<size_t>(L.C) * E, &pw))) return rc;
        if ((rc = need(h, p + ".project.0.bias", L.C, &pb))) return rc;
        bw.mod_off = static_cast<int>(proj_b.size());
        bw.g_pw = h->param_off.count(p + ".project.0.weight") ? h->param_off[p + ".project.0.weight"] : -1;
        bw.g_pb = h->param_off.count(p + ".project.0.bias") ? h->param_off[p + ".project.0.bias"] : -1;
        proj_w.insert(proj_w.end(), pw->begin(), pw->end());
        proj_b.insert(proj_b.end(), pb->begin(), pb->end());
        if ((rc = pack_conv(h, p + ".residue.1", L.C, L.C, 9, &bw.c1))) return rc;
        if ((rc = pack_conv(h, p + ".residue.3", L.C, L.C, 9, &bw.c2))) return rc;
        blocks.push_back(bw);
        if (L.attn) {
          snprintf(buf, sizeof buf, "unet.%s.%d.%d", side == 0 ? "descent" : "ascent", side == 0 ? l : rev, b * step + 1);
          const std::string q(buf);
          AttnW aw;
          if ((rc = pack_conv(h, q + ".qkv", 3 * L.C, L.C, 1, &aw.qkv))) return rc;
          if ((rc = pack_conv(h, q + ".proj_out", L.C, L.C, 1, &aw.proj))) return rc;
          attns.push_back(aw);
        }
      }
    }
    H /= 2;
    W /= 2;
  }
  {
    std::vector<float> z(2048, 0.f);
    if ((rc = dev_upload(h, z.data(), z.size() * sizeof(float), reinterpret_cast<void**>(&h->zero_bias)))) return rc;
  }
  h->total_mod = static_cast<int>(proj_b.size());
  if (h->total_mod > 0) {
    std::vector<long long> row_w(h->total_mod, -1), row_b(h->total_mod, -1);
    for (LevelW& L : h->levels)
      for (std::vector<BlockW>* side : {&L.desc, &L.asc})
        for (BlockW& bw : *side)
          for (int cidx = 0; cidx < L.C; ++cidx) {
            if (bw.g_pw >= 0) row_w[bw.mod_off + cidx] = bw.g_pw + static_cast<long long>(cidx) * E;
            if (bw.g_pb >= 0) row_b[bw.mod_off + cidx] = bw.g_pb + cidx;
          }
    if ((rc = dev_upload(h, row_w.data(), row_w.size() * sizeof(long long), reinterpret_cast<void**>(&h->row_w)))) return rc;
    if ((rc = dev_upload(h, row_b.data(), row_b.size() * sizeof(long long), reinterpret_cast<void**>(&h->row_b)))) return rc;
  }
  if ((rc = dev_upload(h, proj_w.data(), proj_w.size() * sizeof(float), reinterpret_cast<void**>(&h->proj_w)))) return rc;
  if ((rc = dev_upload(h, proj_b.data(), proj_b.size() * sizeof(float), reinterpret_cast<void**>(&h->proj_b)))) return rc;
  h->raw.clear();
  h->finalized = true;
  return C2W_OK;
}

int c2w_total_mod_channels(c2w_handle* h) { return h ? h->total_mod : 0; }

int64_t c2w_launch_count(void) { return g_launches; }

int c2w_set_timing(c2w_handle* h, int enable) {
  C2W_REQUIRE(h, "null handle");
  h->timing = enable != 0;
  h->spans_used = 0;
  return C2W_OK;
}

// Sums the event-timed spans recorded since the last read: ms[0] / n[0] = K1 conv/GEMM launches, ms[1] / n[1] = the
// other forward-pass kernels.  Synchronises on the recorded events.
int c2w_timing_read(c2w_handle* h, double* ms, int64_t* n) {
  C2W_REQUIRE(h && ms && n, "c2w_timing_read: bad argument");
  ms[0] = ms[1] = 0.0;
  n[0] = n[1] = 0;
  for (size_t i = 0; i < h->spans_used; ++i) {
    TimedSpan& s = h->spans[i];
    C2W_CUDA(cudaEventSynchronize(s.e1));
    float t = 0.f;
    C2W_CUDA(cudaEventElapsedTime(&t, s.e0, s.e1));
    ms[s.cls] += t;
    n[s.cls] += 1;
  }
  h->spans_used = 0;
  return C2W_OK;
}

// Diagnostics (-DC2W_DIAG build only): every following K1 launch of this handle writes {first CTA start, last CTA end}
// (%globaltimer, ns) into buf_dev[launch][2]; initialise starts to LLONG_MAX and ends to 0.  Returns the number of slots
// used so far when buf_dev is NULL.
int c2w_set_timeline(c2w_handle* h, long long* buf_dev, int capacity) {
  C2W_REQUIRE(h, "c2w_set_timeline: null handle");
#ifdef C2W_DIAG
  if (buf_dev == nullptr) return h->timeline_used;
  h->timeline = buf_dev;
  h->timeline_cap = capacity;
  h->timeline_used = 0;
  return C2W_OK;
#else
  (void)buf_dev;
  (void)capacity;
  return fail(C2W_ERR_STATE, "c2w_set_timeline needs the diagnostics build (python -m climate2weather_b200.build --diag)");
#endif
}

int64_t c2w_workspace_bytes_ex(c2w_handle* h, int32_t max_windows, int32_t flags) {
  if (!h || !h->finalized || max_windows < 1) {
    fail(C2W_ERR_STATE, "c2w_workspace_bytes: finalise the weights first");
    return -1;
  }
  size_t bytes = 0;
  const bool train = (flags & C2W_WS_TRAIN) != 0;
  if (build_plan(h, max_windows, train || (flags & C2W_WS_VJP) != 0, train || (flags & C2W_WS_PER_SAMPLE_T) != 0, nullptr,
                 &bytes, train))
    return -1;
  return static_cast<int64_t>(bytes);
}
int c2w_bind_workspace_ex(c2w_handle* h, int32_t max_windows, void* dev_ptr, int64_t bytes, int32_t flags) {
  C2W_REQUIRE(h && dev_ptr && max_windows >= 1, "c2w_bind_workspace: bad argument");
  if (!h->finalized) return fail(C2W_ERR_STATE, "finalise the weights first");
  const bool train = (flags & C2W_WS_TRAIN) != 0;
  const bool vjp = train || (flags & C2W_WS_VJP) != 0, per_t = train || (flags & C2W_WS_PER_SAMPLE_T) != 0;
  C2W_REQUIRE(train || !(vjp && per_t),
              "input gradients with per-sample diffusion times need the training workspace (C2W_WS_TRAIN)");
  size_t need_bytes = 0;
  int rc = build_plan(h, max_windows, vjp, per_t, nullptr, &need_bytes, train);
  if (rc) return rc;
  C2W_REQUIRE(static_cast<size_t>(bytes) >= need_bytes, "workspace too small: %lld < %zu", (long long)bytes, need_bytes);
  void* aligned = reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(dev_ptr) + 1023) & ~uintptr_t(1023));
  return build_plan(h, max_windows, vjp, per_t, aligned, &need_bytes, train);
}

int64_t c2w_workspace_bytes(c2w_handle* h, int32_t max_windows) { return c2w_workspace_bytes_ex(h, max_windows, 0); }
int c2w_bind_workspace(c2w_handle* h, int32_t max_windows, void* dev_ptr, int64_t bytes) {
  return c2w_bind_workspace_ex(h, max_windows, dev_ptr, bytes, 0);
}
int64_t c2w_workspace_bytes_vjp(c2w_handle* h, int32_t max_windows) {
  return c2w_workspace_bytes_ex(h, max_windows, C2W_WS_VJP);
}
int c2w_bind_workspace_vjp(c2w_handle* h, int32_t max_windows, void* dev_ptr, int64_t bytes) {
  return c2w_bind_workspace_ex(h, max_windows, dev_ptr, bytes, C2W_WS_VJP);
}

int c2w_op_modulation(c2w_handle* h, float t, float* emb_out, float* mods_out, void* stream) {
  C2W_REQUIRE(h && h->finalized && h->plan.n_max > 0, "c2w_op_modulation: bind a workspace first");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = run_modulation(h, t, nullptr, 1, h->plan.h0, h->plan.emb, h->plan.mods, st);
  if (rc) return rc;
  if (emb_out)
    C2W_CUDA(cudaMemcpyAsync(emb_out, h->plan.emb, h->cfg.embedding_dim * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (mods_out)
    C2W_CUDA(cudaMemcpyAsync(mods_out, h->plan.mods, h->total_mod * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return C2W_OK;
}

static int unet_forward_impl(c2w_handle* h, const float* x_nchw, int32_t n, float t, const float* t_dev, float* out_nchw,
                             void* stream) {
  C2W_REQUIRE(h && x_nchw && out_nchw && n >= 1, "c2w_unet_forward: bad argument");
  if (h->plan.n_max < 1) return fail(C2W_ERR_STATE, "bind a workspace first");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Plan& P = h->plan;
  C2W_REQUIRE((t_dev != nullptr) == P.per_t,
              "per-sample diffusion times need a workspace bound with C2W_WS_PER_SAMPLE_T (and only then)");
  const int hw = h->cfg.height * h->cfg.width;
  const int cout_pad = h->levels[0].tail.cout_pad;
  int rc;
  if (!t_dev && (rc = run_modulation(h, t, nullptr, 1, P.h0, P.emb, P.mods, st))) return rc;
  FinalSpec fs;
  fs.mode = EPI_F32;
  for (int i0 = 0; i0 < n; i0 += P.n_max) {
    const int nn = std::min(P.n_max, n - i0);
    if (t_dev && (rc = run_modulation(h, 0.f, t_dev + i0, nn, P.h0, P.emb, P.mods, st))) return rc;
    dim3 blk(32, 8);
    dim3 g1(ceil_div(hw, 32), ceil_div(h->cin_pad, 32), nn);
    nchw_to_nhwc_bf16_kernel<<<g1, blk, 0, st>>>(x_nchw + static_cast<size_t>(i0) * h->cin * hw, P.xin, h->cin, hw,
                                                 h->cin_pad);
    C2W_CUDA(cudaGetLastError());
    rc = run_plan(h, nn, fs, st);
    if (rc) return rc;
    dim3 g2(ceil_div(hw, 32), ceil_div(cout_pad, 32), nn);
    nhwc_f32_to_nchw_kernel<<<g2, blk, 0, st>>>(P.out32, out_nchw + static_cast<size_t>(i0) * h->cin * hw, h->cin, hw,
                                                cout_pad);
    C2W_CUDA(cudaGetLastError());
  }
  return C2W_OK;
}

int c2w_unet_forward(c2w_handle* h, const float* x_nchw, int32_t n, float t, float* out_nchw, void* stream) {
  return unet_forward_impl(h, x_nchw, n, t, nullptr, out_nchw, stream);
}
int c2w_unet_forward_t(c2w_handle* h, const float* x_nchw, int32_t n, const float* t_dev, float* out_nchw, void* stream) {
  C2W_REQUIRE(t_dev, "c2w_unet_forward_t: null time array");
  return unet_forward_impl(h, x_nchw, n, 0.f, t_dev, out_nchw, stream);
}

int c2w_window_score(c2w_handle* h, const float* traj, int32_t n_frames_local, int32_t frame_global0,
                     int32_t win_first, int32_t n_win, int32_t n_win_global, float t, float* eps, void* stream) {
  C2W_REQUIRE(h && traj && eps, "c2w_window_score: bad argument");
  if (h->plan.n_max < 1) return fail(C2W_ERR_STATE, "bind a workspace first");
  if (h->plan.per_t) return fail(C2W_ERR_STATE, "window scores use one diffusion time: bind a plain workspace");
  const int w = h->cfg.window, C = h->cfg.frame_channels;
  C2W_REQUIRE(n_win >= 1 && win_first >= 0 && win_first + n_win <= n_win_global, "window range [%d,%d) outside [0,%d)",
              win_first, win_first + n_win, n_win_global);
  C2W_REQUIRE(win_first >= frame_global0 && win_first + n_win - 1 + w <= frame_global0 + n_frames_local,
              "windows [%d,%d) need frames outside the local range [%d,%d)", win_first, win_first + n_win,
              frame_global0, frame_global0 + n_frames_local);
  C2W_REQUIRE(C >= 1 && C <= 8, "1 to 8 variables per frame (got %d)", C);
  return window_score_fwd(h, traj, frame_global0, WindowSet{win_first, n_win, nullptr, nullptr}, n_win_global, t, eps,
                          static_cast<cudaStream_t>(stream));
}

// Forward of a SELECTION of windows (global indices win_list_dev[0..n_sel)).  With the coarse-graining likelihood the
// cotangent of the composed score is non-zero on the OBSERVED frames only (every t_step-th, exp/downscaling.py:129-132),
// so only the windows whose centre (or, for the first / last window, edge) frame is observed contribute to the
// vector-Jacobian product: the caller runs this on a VJP workspace (stashing forward, n_sel <= max_windows) for ~1/t_step
// of the windows, followed by c2w_window_score_backward_sel, and on a plain workspace for the others.
// eps != null: the windows' part of the composed score goes into eps (the same fold as c2w_window_score, by list), so
// the two selections together fill it and no window is evaluated twice; eps == null: stash only.
int c2w_window_score_sel(c2w_handle* h, const float* traj, int32_t n_frames_local, int32_t frame_global0,
                         const int32_t* win_list_dev, int32_t n_sel, int32_t n_win_global, float t, float* eps,
                         void* stream) {
  C2W_REQUIRE(h && traj && win_list_dev && n_sel >= 1, "c2w_window_score_sel: bad argument");
  Plan& P = h->plan;
  if (P.n_max < 1 || P.per_t) return fail(C2W_ERR_STATE, "bind a workspace with one diffusion time first");
  C2W_REQUIRE(!P.vjp || n_sel <= P.n_max, "c2w_window_score_sel: %d windows exceed the bound VJP workspace (%d)", n_sel,
              P.n_max);
  C2W_REQUIRE(eps || P.vjp, "c2w_window_score_sel: no output asked for on a plain workspace");
  (void)n_frames_local;
  return window_score_fwd(h, traj, frame_global0, WindowSet{0, n_sel, win_list_dev, nullptr}, n_win_global, t, eps,
                          static_cast<cudaStream_t>(stream));
}

// Adjoint of the selected windows whose stashing forward has JUST run (c2w_window_score_sel, same list): compose adjoint
// -> input-gradient pass -> unfold adjoint; pos_dev[j] = position of global window j in the list or -1 (n_win_global
// entries); vjp (fp32 [n_frames_local, H, W, C]) is ACCUMULATED.
int c2w_window_score_backward_sel(c2w_handle* h, const float* cot, int32_t n_frames_local, int32_t frame_global0,
                                  const int32_t* win_list_dev, const int32_t* pos_dev, int32_t n_sel, int32_t n_win_global,
                                  float* vjp, void* stream) {
  C2W_REQUIRE(h && cot && vjp && win_list_dev && pos_dev && n_sel >= 1, "c2w_window_score_backward_sel: bad argument");
  Plan& P = h->plan;
  if (P.n_max < 1 || !P.vjp) return fail(C2W_ERR_STATE, "bind a VJP workspace first (c2w_bind_workspace_vjp)");
  C2W_REQUIRE(n_sel <= P.n_max, "backward handles one chunk: %d windows, workspace %d", n_sel, P.n_max);
  return window_score_bwd(h, cot, n_frames_local, frame_global0, WindowSet{0, n_sel, win_list_dev, pos_dev}, n_win_global,
                          vjp, static_cast<cudaStream_t>(stream));
}

// J^T g of ScoreUNet.forward w.r.t. its input: forward (stashing) + input-gradient pass, n <= max_windows.
int c2w_unet_vjp(c2w_handle* h, const float* x_nchw, int32_t n, float t, const float* gout_nchw, float* out_nchw,
                 float* gin_nchw, void* stream) {
  C2W_REQUIRE(h && x_nchw && gout_nchw && gin_nchw && n >= 1, "c2w_unet_vjp: bad argument");
  Plan& P = h->plan;
  if (P.n_max < 1 || !P.vjp) return fail(C2W_ERR_STATE, "bind a VJP workspace first (c2w_bind_workspace_vjp)");
  C2W_REQUIRE(n <= P.n_max, "c2w_unet_vjp: %d windows exceed the bound workspace (%d)", n, P.n_max);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int hw = h->cfg.height * h->cfg.width;
  const int cout_pad = h->levels[0].tail.cout_pad;
  int rc = run_modulation(h, t, nullptr, 1, P.h0, P.emb, P.mods, st);
  if (rc) return rc;
  dim3 blk(32, 8);
  dim3 g1(ceil_div(hw, 32), ceil_div(h->cin_pad, 32), n);
  nchw_to_nhwc_bf16_kernel<<<g1, blk, 0, st>>>(x_nchw, P.xin, h->cin, hw, h->cin_pad);
  C2W_CUDA(cudaGetLastError());
  FinalSpec fs;
  fs.mode = EPI_F32;
  if ((rc = run_ops(h, P.ops, n, fs, st))) return rc;
  dim3 g2(ceil_div(hw, 32), ceil_div(cout_pad, 32), n);
  if (out_nchw) {
    nhwc_f32_to_nchw_kernel<<<g2, blk, 0, st>>>(P.out32, out_nchw, h->cin, hw, cout_pad);
    C2W_CUDA(cudaGetLastError());
  }
  nchw_to_nhwc_bf16_kernel<<<g2, blk, 0, st>>>(gout_nchw, P.cot, h->cin, hw, cout_pad);
  C2W_CUDA(cudaGetLastError());
  if ((rc = run_ops(h, P.bwd, n, fs, st))) return rc;
  dim3 g3(ceil_div(hw, 32), ceil_div(h->cin_pad, 32), n);
  nhwc_f32_to_nchw_kernel<<<g3, blk, 0, st>>>(P.out32, gin_nchw, h->cin, hw, h->cin_pad);
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

// Input-gradient pass of the windows whose forward c2w_window_score has JUST run on a VJP workspace (one chunk:
// n_win <= max_windows).  cot: fp32 [n_frames_local, H, W, C] cotangent w.r.t. the composed score; vjp (same shape)
// is ACCUMULATED: vjp[f] += sum over the windows of this call of d eps / d traj[f] ^T cot.
int c2w_window_score_backward(c2w_handle* h, const float* cot, int32_t n_frames_local, int32_t frame_global0,
                              int32_t win_first, int32_t n_win, int32_t n_win_global, float* vjp, void* stream) {
  C2W_REQUIRE(h && cot && vjp, "c2w_window_score_backward: bad argument");
  Plan& P = h->plan;
  if (P.n_max < 1 || !P.vjp) return fail(C2W_ERR_STATE, "bind a VJP workspace first (c2w_bind_workspace_vjp)");
  const int w = h->cfg.window;
  C2W_REQUIRE(n_win >= 1 && n_win <= P.n_max, "backward handles one chunk: %d windows, workspace %d", n_win, P.n_max);
  C2W_REQUIRE(win_first >= frame_global0 && win_first + n_win - 1 + w <= frame_global0 + n_frames_local,
              "windows [%d,%d) need frames outside the local range [%d,%d)", win_first, win_first + n_win,
              frame_global0, frame_global0 + n_frames_local);
  return window_score_bwd(h, cot, n_frames_local, frame_global0, WindowSet{win_first, n_win, nullptr, nullptr},
                          n_win_global, vjp, static_cast<cudaStream_t>(stream));
}

int c2w_set_forcing(c2w_handle* h, const float* forcing_dev) {
  C2W_REQUIRE(h, "c2w_set_forcing: null handle");
  C2W_REQUIRE(forcing_dev == nullptr || h->cfg.forcing_dim > 0, "c2w_set_forcing: the network has no forcing branch (forcing_dim = 0)");
  h->forcing = forcing_dev;
  return C2W_OK;
}

// Re-packs every weight from a DEVICE copy of the parameters in the flat layout of c2w_param_layout (after an optimiser
// step: the buffer optim.AdamW steps on, no host round trip, no re-allocation): bf16 tensor-core operands of all convs,
// biases, modulation projections, time MLP.
int c2w_refresh_weights(c2w_handle* h, const float* flat_dev, void* stream) {
  C2W_REQUIRE(h && flat_dev, "c2w_refresh_weights: bad argument");
  if (!h->finalized) return fail(C2W_ERR_STATE, "finalise the weights first");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!h->refresh_jobs) {  // the job table is a function of the layout only: built and uploaded once
    std::vector<RefreshJob> jobs;
    auto copy = [&](long long src, float* dst, long long n) {
      RefreshJob j{};
      j.src = src, j.n = n, j.fdst = dst, j.kind = 1;
      j.chunks = static_cast<int>((n + kRefreshChunk - 1) / kRefreshChunk);
      jobs.push_back(j);
    };
    auto conv = [&](const ConvW& w) -> int {
      if (w.gw < 0 || w.gb < 0) return fail(C2W_ERR_MISSING, "a conv has no slot in the flat parameter layout");
      RefreshJob j{};
      j.src = w.gw, j.n = static_cast<long long>(w.cout) * w.cin * w.taps, j.wp = w.w, j.wd = w.wd, j.kind = 0;
      j.cout = w.cout, j.cin = w.cin, j.taps = w.taps, j.cin_pad = w.cin_pad, j.cout_pad = w.cout_pad;
      if (w.taps > 9) return fail(C2W_ERR_INVALID, "weight re-pack handles up to 9 taps (got %d)", w.taps);
      j.chunks = ((w.cout + kRefreshTile - 1) / kRefreshTile) * ((w.cin + kRefreshTile - 1) / kRefreshTile);
      jobs.push_back(j);
      copy(w.gb, w.b, w.cout);
      return C2W_OK;
    };
    const int E = h->cfg.embedding_dim;
    int rc;
    for (LevelW& L : h->levels) {
      if ((rc = conv(L.head)) || (rc = conv(L.tail))) return rc;
      for (int side = 0; side < 2; ++side) {
        std::vector<BlockW>& blocks = side == 0 ? L.desc : L.asc;
        std::vector<AttnW>& attns = side == 0 ? L.dattn : L.aattn;
        for (BlockW& bw : blocks) {
          if ((rc = conv(bw.c1)) || (rc = conv(bw.c2))) return rc;
          C2W_REQUIRE(bw.g_pw >= 0 && bw.g_pb >= 0, "a modulation projection has no slot in the flat parameter layout");
          copy(bw.g_pw, h->proj_w + static_cast<size_t>(bw.mod_off) * E, static_cast<long long>(L.C) * E);
          copy(bw.g_pb, h->proj_b + bw.mod_off, L.C);
        }
        for (AttnW& aw : attns)
          if ((rc = conv(aw.qkv)) || (rc = conv(aw.proj))) return rc;
      }
    }
    if (h->cfg.forcing_dim > 0) {  // forcing branch: weight rows re-padded, bias copied
      auto iw = h->param_off.find("map_forcing.weight"), ib = h->param_off.find("map_forcing.bias");
      C2W_REQUIRE(iw != h->param_off.end() && ib != h->param_off.end(), "map_forcing has no slot in the flat layout");
      RefreshJob j{};
      j.src = iw->second, j.n = static_cast<long long>(E) * h->forcing_pad, j.fdst = h->mapf_w, j.kind = 2;
      j.cin = h->cfg.forcing_dim, j.cin_pad = h->forcing_pad;
      j.chunks = static_cast<int>((j.n + kRefreshChunk - 1) / kRefreshChunk);
      jobs.push_back(j);
      copy(ib->second, h->mapf_b, E);
    }
    struct { const char* name; float* dst; long long n; } mlp[4] = {
        {"map_layer0.weight", h->map0_w, static_cast<long long>(E) * h->cfg.noise_features}, {"map_layer0.bias", h->map0_b, E},
        {"map_layer1.weight", h->map1_w, static_cast<long long>(E) * E}, {"map_layer1.bias", h->map1_b, E}};
    for (auto& m : mlp) {
      auto it = h->param_off.find(m.name);
      C2W_REQUIRE(it != h->param_off.end(), "parameter '%s' has no slot in the flat layout", m.name);
      copy(it->second, m.dst, m.n);
    }
    std::vector<int> first(jobs.size());
    long long chunks = 0;
    for (size_t i = 0; i < jobs.size(); ++i) {
      first[i] = static_cast<int>(chunks);
      chunks += jobs[i].chunks;
    }
    RefreshJob* dj = nullptr;
    int* df = nullptr;
    C2W_CUDA(cudaMalloc(&dj, jobs.size() * sizeof(RefreshJob)));
    h->allocs.push_back(dj);
    C2W_CUDA(cudaMalloc(&df, first.size() * sizeof(int)));
    h->allocs.push_back(df);
    C2W_CUDA(cudaMemcpy(dj, jobs.data(), jobs.size() * sizeof(RefreshJob), cudaMemcpyHostToDevice));
    C2W_CUDA(cudaMemcpy(df, first.data(), first.size() * sizeof(int), cudaMemcpyHostToDevice));
    h->refresh_jobs = dj;
    h->refresh_first = df;
    h->refresh_n = static_cast<int>(jobs.size());
    h->refresh_chunks = static_cast<int>(chunks);
  }
  const int grid = std::min(h->refresh_chunks, 16 * h->sms);
  refresh_weights_kernel<<<grid, 256, 0, st>>>(static_cast<const RefreshJob*>(h->refresh_jobs), h->refresh_first,
                                               h->refresh_n, h->refresh_chunks, flat_dev);
  ++g_launches;
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

// ---------------------------------------------------------------------------------------------- training step (N2)
int64_t c2w_param_total(c2w_handle* h) { return (h && h->finalized) ? h->param_total : -1; }

int c2w_param_layout(c2w_handle* h, const char* name, int64_t* offset, int64_t* numel) {
  C2W_REQUIRE(h && name && offset && numel, "c2w_param_layout: bad argument");
  if (!h->finalized) return fail(C2W_ERR_STATE, "finalise the weights first");
  auto it = h->param_off.find(name);
  if (it == h->param_off.end()) return fail(C2W_ERR_MISSING, "no parameter named '%s'", name);
  *offset = it->second;
  for (auto& pr : h->params)
    if (pr.first == name) *numel = pr.second;
  return C2W_OK;
}

// Forward of the training step: ScoreUNet.forward with one diffusion time per sample (src/thor/pipelines.py:27-35),
// stashing what the backward needs.  n <= max_windows of a C2W_WS_TRAIN workspace (one chunk: backward follows).
int c2w_train_forward(c2w_handle* h, const float* x_nchw, int32_t n, const float* t_dev, float* out_nchw, void* stream) {
  C2W_REQUIRE(h && x_nchw && t_dev && out_nchw && n >= 1, "c2w_train_forward: bad argument");
  Plan& P = h->plan;
  if (P.n_max < 1 || !P.train) return fail(C2W_ERR_STATE, "bind a training workspace first (C2W_WS_TRAIN)");
  C2W_REQUIRE(n <= P.n_max, "c2w_train_forward: %d samples exceed the bound workspace (%d)", n, P.n_max);
  int rc = unet_forward_impl(h, x_nchw, n, 0.f, t_dev, out_nchw, stream);
  if (rc) return rc;
  P.n_last = n;
  P.t_last = t_dev;
  return C2W_OK;
}

// Backward of the training step (training_loop.py:378 `fabric.backward(loss)`): gout = d loss / d output (fp32 NCHW) ->
// input-gradient pass (K1 with flipped weights) + weight gradients (K10) + bias / modulation / time-MLP gradients,
// written into the flat fp32 buffer grad_flat (layout: c2w_param_layout; accumulate != 0 adds to it).
int c2w_train_backward(c2w_handle* h, const float* gout_nchw, int32_t n, float* gin_nchw, float* grad_flat,
                       int32_t accumulate, void* stream) {
  C2W_REQUIRE(h && gout_nchw && grad_flat && n >= 1, "c2w_train_backward: bad argument");
  Plan& P = h->plan;
  if (P.n_max < 1 || !P.train) return fail(C2W_ERR_STATE, "bind a training workspace first (C2W_WS_TRAIN)");
  C2W_REQUIRE(n == P.n_last && P.t_last != nullptr, "c2w_train_backward: call c2w_train_forward on the same %d samples first", n);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int hw = h->cfg.height * h->cfg.width;
  const int cout_pad = h->levels[0].tail.cout_pad;
  const int E = h->cfg.embedding_dim, nf = h->cfg.noise_features, TM = h->total_mod;
  if (!accumulate) C2W_CUDA(cudaMemsetAsync(grad_flat, 0, static_cast<size_t>(h->param_total) * sizeof(float), st));
  if (TM > 0) C2W_CUDA(cudaMemsetAsync(P.dmods, 0, static_cast<size_t>(n) * TM * sizeof(float), st));
  dim3 blk(32, 8);
  dim3 g2(ceil_div(hw, 32), ceil_div(cout_pad, 32), n);
  nchw_to_nhwc_bf16_kernel<<<g2, blk, 0, st>>>(gout_nchw, P.cot, h->cin, hw, cout_pad);
  ++g_launches;
  C2W_CUDA(cudaGetLastError());
  P.grad = grad_flat;
  FinalSpec fs;
  fs.mode = EPI_F32;
  int rc = run_ops(h, P.bwd, n, fs, st);
  P.grad = nullptr;
  if (rc) return rc;
  if (gin_nchw) {
    dim3 g3(ceil_div(hw, 32), ceil_div(h->cin_pad, 32), n);
    nhwc_f32_to_nchw_kernel<<<g3, blk, 0, st>>>(P.out32, gin_nchw, h->cin, hw, h->cin_pad);
    C2W_CUDA(cudaGetLastError());
  }
  // ---- modulation projections and the time MLP (model/nn.py:149; model/score.py:59-67): tiny fp32 products
  auto off = [&](const char* nm) -> long long {
    auto it = h->param_off.find(nm);
    return it == h->param_off.end() ? -1 : it->second;
  };
  auto blocks1d = [](long long items) { return static_cast<int>((items + 255) / 256); };
  if (TM > 0) {
    // all 30 project Linears in one launch: dW_p[c][e] += sum_s dmod[s][c] emb[s][e], db_p[c] += sum_s dmod[s][c]
    proj_grad_kernel<<<blocks1d(static_cast<long long>(TM) * E), 256, 0, st>>>(P.dmods, TM, P.emb, E, n, grad_flat, h->row_w,
                                                                              h->row_b);
    g_launches += 12;  // this block: projections, embedding gradient, two Linear layers of the time MLP
    // d emb = dmods . W_proj  ([n, TM] x [TM, E]);  emb = silu(pre1), pre1 = W1 h0 + b1;  h0 = silu(pre0), pre0 = W0 feat + b0
    C2W_CUDA(cudaMemsetAsync(P.demb, 0, static_cast<size_t>(n) * E * sizeof(float), st));
    gemm_nn_f32_kernel<<<dim3(blocks1d(static_cast<long long>(n) * E), 32), 256, 0, st>>>(P.dmods, TM, h->proj_w, E, P.demb, E,
                                                                                         n, TM, E);
    matvec_kernel<<<dim3(ceil_div(static_cast<long long>(E) * 32, 256), n), 256, 0, st>>>(
        h->map1_w, h->map1_b, P.h0, P.pre1, E, E, 0, (h->forcing != nullptr && h->forcing_pad > 0) ? P.fvec : nullptr);
    dsilu_f32_kernel<<<blocks1d(static_cast<long long>(n) * E), 256, 0, st>>>(P.demb, P.pre1, static_cast<long long>(n) * E);
    const long long o1w = off("map_layer1.weight"), o1b = off("map_layer1.bias");
    const long long o0w = off("map_layer0.weight"), o0b = off("map_layer0.bias");
    if (o1w >= 0)
      gemm_tn_f32_kernel<<<blocks1d(static_cast<long long>(E) * E), 256, 0, st>>>(P.demb, E, P.h0, E, grad_flat + o1w, E, n, E,
                                                                                  E, 1);
    if (o1b >= 0) colsum_f32_kernel<<<blocks1d(E), 256, 0, st>>>(P.demb, E, grad_flat + o1b, n, E, 1);
    if (h->forcing != nullptr && h->forcing_pad > 0) {  // emb = silu(pre1 + Wf f + bf): same d pre1
      const long long ofw = off("map_forcing.weight"), ofb = off("map_forcing.bias");
      const int F = h->cfg.forcing_dim;
      if (ofw >= 0)
        gemm_tn_f32_kernel<<<blocks1d(static_cast<long long>(E) * F), 256, 0, st>>>(P.demb, E, P.forc_pad, h->forcing_pad,
                                                                                  grad_flat + ofw, F, n, E, F, 1);
      if (ofb >= 0) colsum_f32_kernel<<<blocks1d(E), 256, 0, st>>>(P.demb, E, grad_flat + ofb, n, E, 1);
    }
    gemm_nn_f32_kernel<<<blocks1d(static_cast<long long>(n) * E), 256, 0, st>>>(P.demb, E, h->map1_w, E, P.dh0, E, n, E, E);
    time_features_kernel<<<n, 128, 0, st>>>(P.t_last, P.feat, nf);
    matvec_kernel<<<dim3(ceil_div(static_cast<long long>(E) * 32, 256), n), 256, 0, st>>>(h->map0_w, h->map0_b, P.feat, P.pre0,
                                                                                          E, nf, 0);
    dsilu_f32_kernel<<<blocks1d(static_cast<long long>(n) * E), 256, 0, st>>>(P.dh0, P.pre0, static_cast<long long>(n) * E);
    if (o0w >= 0)
      gemm_tn_f32_kernel<<<blocks1d(static_cast<long long>(E) * nf), 256, 0, st>>>(P.dh0, E, P.feat, nf, grad_flat + o0w, nf, n,
                                                                                   E, nf, 1);
    if (o0b >= 0) colsum_f32_kernel<<<blocks1d(E), 256, 0, st>>>(P.dh0, E, grad_flat + o0b, n, E, 1);
    C2W_CUDA(cudaGetLastError());
  }
  return C2W_OK;
}

// mean((out - eps)^2) * loss_scale and its cotangent (src/thor/pipelines.py:27-35 + `.mean()`, training_loop.py:377):
// gout = 2 loss_scale (out - eps) / numel; loss_sum_dev (device double) receives sum((out - eps)^2).
int c2w_dsm_loss_grad(const float* out, const float* eps, float* gout, int64_t numel, float loss_scale, float* partials4096,
                      double* loss_sum_dev, void* stream) {
  C2W_REQUIRE(out && eps && gout && partials4096 && loss_sum_dev && numel >= 1, "c2w_dsm_loss_grad: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = static_cast<int>(std::min<long long>(4096, (numel + 255) / 256));
  dsm_loss_grad_kernel<<<grid, 256, 0, st>>>(out, eps, gout, partials4096, numel, 2.0f * loss_scale / static_cast<float>(numel));
  reduce_partials_kernel<<<1, 256, 0, st>>>(partials4096, grid, loss_sum_dev);
  g_launches += 2;
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

// One denoising-score-matching training step up to the gradients (training_loop.py:372-378 for one accumulation round):
// forward on xt (already noised: xt = mu(t) x + sigma(t) eps), loss + cotangent, backward.  out_nchw / gout_nchw are
// caller-owned work buffers of x's shape (the prediction and its cotangent).
int c2w_train_step(c2w_handle* h, const float* xt_nchw, int32_t n, const float* t_dev, const float* eps_nchw,
                   float* out_nchw, float* gout_nchw, float loss_scale, float* grad_flat, int32_t accumulate,
                   double* loss_sum_dev, void* stream) {
  C2W_REQUIRE(h && xt_nchw && t_dev && eps_nchw && out_nchw && gout_nchw && grad_flat && loss_sum_dev, "c2w_train_step: bad argument");
  int rc = c2w_train_forward(h, xt_nchw, n, t_dev, out_nchw, stream);
  if (rc) return rc;
  const int64_t numel = static_cast<int64_t>(n) * h->cin * h->cfg.height * h->cfg.width;
  if ((rc = c2w_dsm_loss_grad(out_nchw, eps_nchw, gout_nchw, numel, loss_scale, h->plan.loss_partials, loss_sum_dev, stream)))
    return rc;
  return c2w_train_backward(h, gout_nchw, n, nullptr, grad_flat, accumulate, stream);
}

int c2w_traj_pack(const float* nchw, float* fhwc, int64_t frames, int32_t C, int32_t hw, void* stream) {
  C2W_REQUIRE(nchw && fhwc && frames >= 1, "c2w_traj_pack: bad argument");
  nchw_to_fhwc_kernel<<<grid_for(frames * hw, 256, c2w_num_sms()), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      nchw, fhwc, frames, C, hw);
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}
int c2w_traj_unpack(const float* fhwc, float* nchw, int64_t frames, int32_t C, int32_t hw, void* stream) {
  C2W_REQUIRE(nchw && fhwc && frames >= 1, "c2w_traj_unpack: bad argument");
  fhwc_to_nchw_kernel<<<grid_for(frames * hw, 256, c2w_num_sms()), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      fhwc, nchw, frames, C, hw);
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

int c2w_normalize_pack(const float* src, float* fhwc, int64_t frames, int32_t C, int32_t hw, int32_t clhw,
                       const float* shift, const float* scale, int32_t field, void* stream) {
  C2W_REQUIRE(src && fhwc && shift && scale && frames >= 1 && C >= 1 && hw >= 1, "c2w_normalize_pack: bad argument");
  const int grid = grid_for(frames * hw, 256, c2w_num_sms());
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool vec = C == 4 && hw % 4 == 0 && (reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(fhwc) |
                                             reinterpret_cast<uintptr_t>(shift) | reinterpret_cast<uintptr_t>(scale)) % 16 == 0;
  if (vec)
    normalize_pack4_kernel<<<grid_for(frames * hw / 4, 256, c2w_num_sms()), 256, 0, st>>>(src, fhwc, frames, hw, clhw,
                                                                                          shift, scale, field);
  else if (C == 4) normalize_pack_kernel<4><<<grid, 256, 0, st>>>(src, fhwc, frames, C, hw, clhw, shift, scale, field);
  else normalize_pack_kernel<0><<<grid, 256, 0, st>>>(src, fhwc, frames, C, hw, clhw, shift, scale, field);
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}
int c2w_unpack_unnormalize(const float* fhwc, float* dst, int64_t frames, int32_t C, int32_t hw, int32_t clhw,
                           const float* shift, const float* scale, int32_t field, void* stream) {
  C2W_REQUIRE(dst && fhwc && shift && scale && frames >= 1 && C >= 1 && hw >= 1, "c2w_unpack_unnormalize: bad argument");
  const int grid = grid_for(frames * hw, 256, c2w_num_sms());
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool vec = C == 4 && hw % 4 == 0 && (reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(fhwc) |
                                             reinterpret_cast<uintptr_t>(shift) | reinterpret_cast<uintptr_t>(scale)) % 16 == 0;
  if (vec)
    unpack_unnormalize4_kernel<<<grid_for(frames * hw / 4, 256, c2w_num_sms()), 256, 0, st>>>(fhwc, dst, frames, hw, clhw,
                                                                                              shift, scale, field);
  else if (C == 4) unpack_unnormalize_kernel<4><<<grid, 256, 0, st>>>(fhwc, dst, frames, C, hw, clhw, shift, scale, field);
  else unpack_unnormalize_kernel<0><<<grid, 256, 0, st>>>(fhwc, dst, frames, C, hw, clhw, shift, scale, field);
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

int c2w_adamw_ema_step(float* p, const float* g, float* m, float* v, float* ema, int64_t n, const c2w_adamw* hp,
                       void* stream) {
  C2W_REQUIRE(p && g && m && v && hp && n >= 1, "c2w_adamw_ema_step: bad argument");
  C2W_REQUIRE(hp->step >= 1 && hp->beta1 >= 0.f && hp->beta1 < 1.f && hp->beta2 >= 0.f && hp->beta2 < 1.f,
              "c2w_adamw_ema_step: step must be >= 1 and betas in [0, 1)");
  C2W_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(ema)) & 15) == 0,
              "c2w_adamw_ema_step: buffers must be 16-byte aligned");
  AdamWParams h;
  h.lr = hp->lr;
  h.beta1 = hp->beta1;
  h.beta2 = hp->beta2;
  h.eps = hp->eps;
  h.weight_decay = hp->weight_decay;
  h.bias1 = static_cast<float>(1.0 - pow(static_cast<double>(hp->beta1), static_cast<double>(hp->step)));
  h.bias2_sqrt = static_cast<float>(sqrt(1.0 - pow(static_cast<double>(hp->beta2), static_cast<double>(hp->step))));
  h.ema_rate = hp->ema_rate;
  h.grad_scale = hp->grad_scale;
  adamw_ema_kernel<<<grid_for((n + 3) / 4, 256, c2w_num_sms()), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      p, g, m, v, ema, n, h);
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

// GuideParams and the variable count C from a c2w_guide: the checks and fields both guidance entry points share (`what`
// names the caller).
static int guide_params(const c2w_guide* g, const char* what, GuideParams& p, int& C) {
  C2W_REQUIRE(g && g->x && g->eps && g->nan_flag, "%s: bad argument", what);
  C2W_REQUIRE(g->mode != 1 || (g->eps_out && g->partials), "mode 1 needs eps_out and partials");
  C2W_REQUIRE(g->own_n >= 1, "own_n must be positive");
  C = g->channels == 0 ? 4 : g->channels;
  C2W_REQUIRE(C >= 1 && C <= C2W_MAX_VARS, "%s: 1 to %d variables per frame (got %d)", what, C2W_MAX_VARS, C);
  C2W_REQUIRE(C == 4 || g->halo == nullptr, "%s: the fused halo push handles 4 variables per frame", what);
  p.x = g->x;
  p.eps = g->eps;
  p.eps_out = g->eps_out;
  p.y = g->y;
  for (int i = 0; i < C2W_MAX_VARS; ++i) {
    p.std2[i] = g->std2[i];
    p.gamma[i] = g->gamma[i];
  }
  p.mu = g->mu;
  p.sigma = g->sigma;
  p.mu_next = g->mu_next;
  p.sigma_next = g->sigma_next;
  p.t_step = g->t_step;
  p.s_step = g->s_step;
  p.H = g->H;
  p.W = g->W;
  p.frame_global0 = g->frame_global0;
  p.own_lo = g->own_lo;
  p.mode = g->mode;
  p.partials = g->partials;
  p.nan_flag = g->nan_flag;
  p.vjp = g->vjp;
  p.cot_out = g->cot_out;
  p.push_l = p.push_r = nullptr;
  p.flag_l = p.flag_r = p.push_done = nullptr;
  p.publish = 0;
  p.halo_k = g->halo_k;
  p.own_n = g->own_n;
  if (g->halo != nullptr && g->mode == 0) {  // fused halo push (csrc/halo.cu)
    C2W_REQUIRE(g->halo_k >= 1 && g->own_n >= g->halo_k, "%s: fused halo push needs 1 <= halo_k <= own_n", what);
    void *sl, *sr, *fl, *fr, *dn;
    uint32_t pub;
    int rc = c2w_halo_push_targets(static_cast<c2w_halo*>(g->halo), &sl, &sr, &fl, &fr, &dn, &pub);
    if (rc) return rc;
    p.push_l = static_cast<float4*>(sl);
    p.push_r = static_cast<float4*>(sr);
    p.flag_l = static_cast<unsigned int*>(fl);
    p.flag_r = static_cast<unsigned int*>(fr);
    p.push_done = (sl || sr) ? static_cast<unsigned int*>(dn) : nullptr;
    p.publish = pub;
  }
  return C2W_OK;
}

static PointParams point_params(const c2w_point_obs* obs) {
  PointParams q;
  q.frame_slot = obs->frame_slot;
  q.strip_off = obs->strip_off;
  q.pix = obs->pix;
  q.ysum = obs->ysum;
  q.wsum = obs->wsum;
  q.strip_rows = obs->strip_rows;
  return q;
}

// The bodies of c2w_guided_step, c2w_guided_step_points and c2w_guided_step_combined: their argument checks, then
// the per-variable (PerObs = false) or per-observation (c2w_guided_step_obs_std) instance of K6, K6p or K6c.
extern "C++" {
template <bool PerObs>
static int guided_coarse(const c2w_guide* g, const ObsStd2& v, void* stream) {
  C2W_REQUIRE(g->s_step >= 1 && g->H % g->s_step == 0 && g->W % g->s_step == 0 && g->W / g->s_step <= 32,
              "s_step=%d must divide %dx%d with at most 32 tiles per row", g->s_step, g->H, g->W);
  C2W_REQUIRE(g->mode != 2 || (g->cot_out && g->y), "mode 2 needs cot_out and an observation");
  C2W_REQUIRE(g->t_step >= 1, "own_n and t_step must be positive");
  GuideParams p;
  int C;
  int rc = guide_params(g, "c2w_guided_step", p, C);
  if (rc) return rc;
  dim3 grid(g->H / g->s_step, g->own_n);
  return launch_for_vars(C, [&](auto vars) {
    guided_step_kernel<decltype(vars)::value, PerObs>
        <<<grid, 32 * (g->W / g->s_step), 0, static_cast<cudaStream_t>(stream)>>>(p, v);
  });
}

template <bool PerObs>
static int guided_points(const c2w_guide* g, const c2w_point_obs* obs, const ObsStd2& v, void* stream) {
  C2W_REQUIRE(obs->frame_slot && obs->strip_off, "c2w_guided_step_points: bad argument");
  C2W_REQUIRE(obs->n_slots == 0 || (obs->pix && obs->ysum && obs->wsum), "c2w_guided_step_points: entries missing");
  C2W_REQUIRE(g->H >= 1 && g->W >= 1 && obs->strip_rows >= 1 && obs->strip_rows * g->W <= C2W_POINT_STRIP_PIX,
              "c2w_guided_step_points: strip of %d rows of %d pixels exceeds %d pixels", obs->strip_rows, g->W,
              C2W_POINT_STRIP_PIX);
  C2W_REQUIRE(g->mode != 2 || g->cot_out, "mode 2 needs cot_out");
  GuideParams p;
  int C;
  int rc = guide_params(g, "c2w_guided_step_points", p, C);
  if (rc) return rc;
  PointParams q = point_params(obs);
  dim3 grid((g->H + obs->strip_rows - 1) / obs->strip_rows, g->own_n);
  return launch_for_vars(C, [&](auto vars) {
    guided_points_kernel<decltype(vars)::value, PerObs><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(p, q, v);
  });
}

template <bool PerObs>
static int guided_combined(const c2w_guide* g, const c2w_point_obs* obs, const float* point_std2, const ObsStd2& v,
                           void* stream) {
  C2W_REQUIRE(obs->frame_slot && obs->strip_off, "c2w_guided_step_combined: bad argument");
  C2W_REQUIRE(obs->n_slots == 0 || (obs->pix && obs->ysum && obs->wsum), "c2w_guided_step_combined: entries missing");
  C2W_REQUIRE(g->y, "c2w_guided_step_combined: needs the coarse observation y");
  C2W_REQUIRE(g->H >= 1 && g->W >= 1, "c2w_guided_step_combined: empty %dx%d grid", g->H, g->W);
  C2W_REQUIRE(g->s_step >= 1 && g->H % g->s_step == 0 && g->W % g->s_step == 0 && g->W / g->s_step <= 32,
              "s_step=%d must divide %dx%d with at most 32 tiles per row", g->s_step, g->H, g->W);
  C2W_REQUIRE(g->t_step >= 1, "own_n and t_step must be positive");
  C2W_REQUIRE(obs->strip_rows >= 1 && obs->strip_rows % g->s_step == 0 &&
                  static_cast<long long>(obs->strip_rows) * g->W <= C2W_COMBINED_STRIP_PIX,
              "c2w_guided_step_combined: strip of %d rows of %d pixels must be a multiple of s_step=%d and at most %d "
              "pixels", obs->strip_rows, g->W, g->s_step, C2W_COMBINED_STRIP_PIX);
  C2W_REQUIRE(g->mode != 2 || g->cot_out, "mode 2 needs cot_out");
  GuideParams p;
  int C;
  int rc = guide_params(g, "c2w_guided_step_combined", p, C);
  if (rc) return rc;
  PointParams q = point_params(obs);
  PointStd2 ps;
  for (int i = 0; i < C2W_MAX_VARS; ++i) ps.v[i] = i < C && !PerObs ? point_std2[i] : 0.f;
  const int smem = combined_smem_bytes(obs->strip_rows, g->W, g->s_step, C);
  dim3 grid((g->H + obs->strip_rows - 1) / obs->strip_rows, g->own_n);
  cudaError_t attr = cudaSuccess;
  rc = launch_for_vars(C, [&](auto vars) {
    const auto kernel = guided_combined_kernel<decltype(vars)::value, PerObs>;
    if (smem > 48 * 1024) attr = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (attr == cudaSuccess) kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(p, q, ps, v);
  });
  C2W_CUDA(attr);
  return rc;
}
}  // extern "C++"

int c2w_guided_step(const c2w_guide* g, void* stream) {
  C2W_REQUIRE(g, "c2w_guided_step: bad argument");
  return guided_coarse<false>(g, ObsStd2{}, stream);
}

int c2w_guided_step_points(const c2w_guide* g, const c2w_point_obs* obs, void* stream) {
  C2W_REQUIRE(g && obs, "c2w_guided_step_points: bad argument");
  return guided_points<false>(g, obs, ObsStd2{}, stream);
}

int c2w_guided_step_combined(const c2w_guide* g, const c2w_point_obs* obs, const float* point_std2, void* stream) {
  C2W_REQUIRE(g && obs && point_std2, "c2w_guided_step_combined: bad argument");
  return guided_combined<false>(g, obs, point_std2, ObsStd2{}, stream);
}

int c2w_guided_step_obs_std(const c2w_guide* g, const c2w_point_obs* obs, const float* coarse_std2,
                            const float* entry_std2, void* stream) {
  C2W_REQUIRE(g, "c2w_guided_step_obs_std: bad argument");
  C2W_REQUIRE((g->y == nullptr) == (coarse_std2 == nullptr),
              "c2w_guided_step_obs_std: the coarse term needs both g->y and coarse_std2, or neither");
  C2W_REQUIRE((obs == nullptr) == (entry_std2 == nullptr),
              "c2w_guided_step_obs_std: the point term needs both obs and entry_std2, or neither");
  C2W_REQUIRE(g->y || obs, "c2w_guided_step_obs_std: no observation term (needs g->y or obs)");
  const ObsStd2 v{coarse_std2, entry_std2};
  if (obs == nullptr) return guided_coarse<true>(g, v, stream);
  if (g->y == nullptr) return guided_points<true>(g, obs, v, stream);
  return guided_combined<true>(g, obs, nullptr, v, stream);
}

int c2w_reduce_partials(const float* partials, int32_t n, double* sumsq, void* stream) {
  C2W_REQUIRE(partials && sumsq && n >= 1, "c2w_reduce_partials: bad argument");
  reduce_partials_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(partials, n, sumsq);
  ++g_launches;
  C2W_CUDA(cudaGetLastError());
  return C2W_OK;
}

int c2w_corrector_update_c(float* x, const float* eps, const float* z, const double* sumsq, double count, float tau,
                           float sigma_next, int64_t pix0_global, int64_t npix, int32_t channels, uint64_t seed,
                           uint32_t step_id, int32_t* nan_flag, void* stream) {
  C2W_REQUIRE(x && eps && sumsq && nan_flag && npix >= 1 && count > 0, "c2w_corrector_update: bad argument");
  C2W_REQUIRE(channels >= 1 && channels <= C2W_MAX_VARS, "c2w_corrector_update: 1 to %d variables per frame (got %d)",
              C2W_MAX_VARS, channels);
  return launch_for_vars(channels, [&](auto vars) {
    corrector_update_kernel<decltype(vars)::value><<<grid_for(npix, 256, c2w_num_sms()), 256, 0,
                                                     static_cast<cudaStream_t>(stream)>>>(
        x, eps, z, sumsq, count, tau, sigma_next, pix0_global, npix, seed, step_id, nan_flag);
  });
}

int c2w_corrector_update(float* x, const float* eps, const float* z, const double* sumsq, double count, float tau,
                         float sigma_next, int64_t pix0_global, int64_t npix, uint64_t seed, uint32_t step_id,
                         int32_t* nan_flag, void* stream) {
  return c2w_corrector_update_c(x, eps, z, sumsq, count, tau, sigma_next, pix0_global, npix, 4, seed, step_id, nan_flag,
                                stream);
}

// ---------------------------------------------------------------------------------------------- op-level hooks
int c2w_op_layernorm(const void* x, const float* mod, void* out, int64_t npix, int C, int H, int W, int upsample,
                     void* stream) {
  C2W_REQUIRE(x && out && npix >= 1, "c2w_op_layernorm: bad argument");
  return launch_ln(static_cast<const bf16*>(x), mod, static_cast<bf16*>(out), nullptr, npix, C, H, W, upsample, c2w_num_sms(),
                   static_cast<cudaStream_t>(stream));
}
int c2w_op_layernorm_bwd(const void* gy, const void* y, const float* inv, const void* gres, void* out, int64_t npix,
                         int C, int H, int W, int down, void* stream) {
  C2W_REQUIRE(gy && y && inv && out && npix >= 1, "c2w_op_layernorm_bwd: bad argument");
  return launch_ln_bwd(static_cast<const bf16*>(gy), static_cast<const bf16*>(y), inv, static_cast<const bf16*>(gres),
                       static_cast<bf16*>(out), npix, C, H, W, down, c2w_num_sms(), static_cast<cudaStream_t>(stream));
}
int c2w_op_layernorm_inv(const void* x, const float* mod, void* out, float* inv, int64_t npix, int C, void* stream) {
  C2W_REQUIRE(x && out && inv && npix >= 1, "c2w_op_layernorm_inv: bad argument");
  return launch_ln(static_cast<const bf16*>(x), mod, static_cast<bf16*>(out), inv, npix, C, 1, 1, 0, c2w_num_sms(),
                   static_cast<cudaStream_t>(stream));
}
int c2w_op_attention_bwd(const void* qkv, const void* go, void* gqkv, float* scratch, int n, int T, int C,
                         void* stream) {
  C2W_REQUIRE(qkv && go && gqkv && scratch && n >= 1, "c2w_op_attention_bwd: bad argument");
  return launch_attention_bwd(static_cast<const bf16*>(qkv), static_cast<const bf16*>(go), static_cast<bf16*>(gqkv),
                              scratch, n, T, C, static_cast<cudaStream_t>(stream));
}
int c2w_op_attention(const void* qkv, void* out, int n, int T, int C, void* stream) {
  C2W_REQUIRE(qkv && out && n >= 1, "c2w_op_attention: bad argument");
  return launch_attention(static_cast<const bf16*>(qkv), static_cast<bf16*>(out), n, T, C,
                          static_cast<cudaStream_t>(stream));
}
int c2w_op_gather_windows(const float* traj, void* out, int n, int hw, int C, int window, int cin_pad, int frame0,
                          void* stream) {
  C2W_REQUIRE(traj && out && n >= 1 && cin_pad % 8 == 0 && cin_pad >= C * window, "c2w_op_gather_windows: bad argument");
  return launch_gather(traj, static_cast<bf16*>(out), n, hw, C, window, cin_pad, frame0, c2w_num_sms(),
                       static_cast<cudaStream_t>(stream));
}

// ---- weight-gradient kernels, op level (parity tests of single kernels; the training step launches the same kernels)
int c2w_op_wgrad(const void* x, const void* dy, int32_t n_img, int32_t H, int32_t W, int32_t cin_pad, int32_t cout_pad,
                 int32_t stride, int32_t conv3x3, float* scratch, int64_t scratch_floats, float* dw, float* db,
                 int32_t cin, int32_t cout, int32_t accumulate, void* stream) {
  C2W_REQUIRE(x && dy && dw && scratch && n_img >= 1 && cin >= 1 && cout >= 1 && cin <= cin_pad && cout <= cout_pad,
              "c2w_op_wgrad: bad argument");
  const int sms = c2w_num_sms();
  C2W_REQUIRE(sms > 0, "c2w_op_wgrad: no CUDA device");
  WgradLaunch L;
  if (!wgrad_launch_init(&L, conv3x3 != 0, static_cast<const __nv_bfloat16*>(x), static_cast<const __nv_bfloat16*>(dy), n_img,
                         H, W, cin_pad, cout_pad, stride ? stride : 1, sms, scratch, static_cast<size_t>(scratch_floats)))
    return fail(C2W_ERR_INVALID, "c2w_op_wgrad: cannot build launch (n=%d H=%d W=%d cin=%d cout=%d stride=%d; channel "
                "counts must be multiples of 64, output images multiples of 8 x 8, GEMM rows a multiple of 64; scratch "
                "%lld floats) %s", n_img, H, W, cin_pad, cout_pad, stride, (long long)scratch_floats, tmap_error_slot());
  C2W_CUDA(wgrad_run(L, dw, cout, cin, accumulate, 1.0f, static_cast<cudaStream_t>(stream), db));
  return C2W_OK;
}

int c2w_op_colsum(const void* x_bf16, float* out, int64_t rows, int32_t C, int64_t rows_per_group, int32_t out_stride,
                  float scale, void* stream) {
  C2W_REQUIRE(x_bf16 && out && rows >= 1 && C >= 2 && C % 2 == 0 && rows_per_group >= 1,
              "c2w_op_colsum: bad argument");
  C2W_CUDA(colsum_run(static_cast<const __nv_bfloat16*>(x_bf16), out, rows, C, rows_per_group, out_stride, scale,
                      static_cast<cudaStream_t>(stream)));
  return C2W_OK;
}

}  // extern "C"
