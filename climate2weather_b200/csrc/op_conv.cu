// Op-level C-ABI entry for K1 (used by the parity tests and by tools/; the engine calls
// conv_launch_init/conv_launch directly with prebuilt tensor maps).
#include "c2w_b200.h"
#include "common.cuh"
#include "conv_tcgen05.cuh"

using namespace c2w;

static int g_num_sms = 0;

int c2w_num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  return g_num_sms;
}

extern "C" {

int c2w_conv_tile_width(int cout_pad, int conv3x3, int n_img, int H, int W, int stride, int num_sms) {
  if (cout_pad < 64 || cout_pad % 64 != 0 || n_img < 1 || H < 1 || W < 1 || (stride != 1 && stride != 2) || num_sms < 2)
    return fail(C2W_ERR_INVALID, "c2w_conv_tile_width: bad argument");
  return conv_pick_bn_tiled(cout_pad, conv3x3 != 0, n_img, H, W, stride, num_sms);
}

int c2w_op_conv_ex(const c2w_conv_desc* d, void* stream) {
  C2W_REQUIRE(d && d->x && d->w_packed && d->bias, "c2w_op_conv_ex: null argument");
  C2W_REQUIRE(d->mode == EPI_BIAS || d->mode == EPI_BIAS_SILU || d->mode == EPI_BIAS_RES || d->mode == EPI_F32 ||
                  d->mode == EPI_MUL_DSILU,
              "c2w_op_conv_ex: unsupported mode %d", d->mode);
  const int sms = c2w_num_sms();
  C2W_REQUIRE(sms > 0, "c2w_op_conv_ex: no CUDA device");
  const int bn = d->bn ? d->bn : d->mode == EPI_F32 ? 64 : conv_pick_bn(d->cout_pad);  // fp32 output: 64-wide tiles only
  const int stride = d->stride ? d->stride : 1;
  ConvLaunch L;
  if (!conv_launch_init(&L, d->conv3x3 != 0, static_cast<const __nv_bfloat16*>(d->x), d->n_img, d->H, d->W, d->cin,
                        static_cast<const __nv_bfloat16*>(d->w_packed), d->cout_pad, bn,
                        d->max_ctas > 0 ? d->max_ctas : sms, stride, d->variant))
    return fail(C2W_ERR_INVALID, "c2w_op_conv_ex: cannot build launch (n=%d H=%d W=%d cin=%d cout=%d bn=%d stride=%d "
                "variant=%d)", d->n_img, d->H, d->W, d->cin, d->cout_pad, bn, stride, d->variant);
  L.p.mode = d->mode;
  L.p.bias = d->bias;
  L.p.out_f32 = d->out_f32;
#ifdef C2W_DIAG
  L.p.dbg_skip_loads = d->skip_loads;
  L.p.dbg_stats = reinterpret_cast<long long*>(d->stats);
#else
  C2W_REQUIRE(d->skip_loads == 0 && d->stats == nullptr,
              "c2w_op_conv_ex: skip_loads / stats are diagnostics of the -DC2W_DIAG build (libc2w_b200_diag.so); the "
              "shipped kernels carry no instrumentation");
#endif
  if (d->mode != EPI_F32) {
    C2W_REQUIRE(d->out, "c2w_op_conv_ex: bf16 output modes need `out`");
    C2W_REQUIRE((d->mode != EPI_BIAS_RES && d->mode != EPI_MUL_DSILU) || d->res == d->out,
                "modes 2 and 5 work in place: res must equal out");
    if (!conv_launch_set_out(&L, static_cast<__nv_bfloat16*>(d->out)))
      return fail(C2W_ERR_CUDA, "c2w_op_conv_ex: cannot encode the output tensor map");
  }
  if (d->ln_out) {
    if (!conv_launch_set_ln(&L, static_cast<__nv_bfloat16*>(d->ln_out), d->ln_mod, d->ln_upsample))
      return fail(C2W_ERR_INVALID, "fused LayerNorm needs bn == cout_pad in {64,128,256}, a bf16 output mode and "
                  "(upsampled) tiles made of whole rows of one image");
  }
  C2W_CUDA(conv_launch(L, static_cast<cudaStream_t>(stream)));
  return C2W_OK;
}

// x: bf16 NHWC [n_img, H, W, cin]  (conv3x3 != 0)   or   bf16 [n_img*H*W, cin] row-major (conv3x3 == 0)
// w_packed: bf16 [cout_pad, taps*cin] with k = (r*3+s)*cin + c ; bias: fp32 [cout_pad]
// mode: EpiMode (0 bias, 1 bias+silu, 2 bias+residual, 4 fp32 out); res/out: bf16 [M, cout_pad]
// bn: N tile (0 = pick) ; max_ctas: 0 = one per SM.  Stride 1, kernel variant picked like the engine does.
int c2w_op_conv(const void* x, int n_img, int H, int W, int cin, const void* w_packed, int cout_pad,
                const float* bias, int mode, const void* res, void* out, float* out_f32, int conv3x3, int bn,
                int max_ctas, void* stream) {
  c2w_conv_desc d;
  memset(&d, 0, sizeof(d));
  d.x = x;
  d.n_img = n_img;
  d.H = H;
  d.W = W;
  d.cin = cin;
  d.stride = 1;
  d.conv3x3 = conv3x3;
  d.w_packed = w_packed;
  d.cout_pad = cout_pad;
  d.bias = bias;
  d.mode = mode;
  d.res = res;
  d.out = out;
  d.out_f32 = out_f32;
  d.bn = bn;
  d.variant = -1;
  d.max_ctas = max_ctas;
  return c2w_op_conv_ex(&d, stream);
}

}  // extern "C"
