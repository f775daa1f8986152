// Generic device-op layer of the C ABI (include/ltb200.h, "ltb_ctx / ltb_op_*"): the MuseTalk networks (diffusers
// UNet2DConditionModel / AutoencoderKL and the Whisper encoder — third-party graphs the reference only wraps,
// avatars/musetalk/models/{unet,vae}.py, avatars/musetalk/whisper/audio2feature.py) are assembled by the Python host
// code out of these operators, captured ONCE into a CUDA graph and replayed per step.  Every op is asynchronous on the
// context's stream; device memory is owned by the context.
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/ltb200.h"
#include "conv_halo.h"
#include "ltb_internal.h"
#include "ops.h"

using namespace ltb;

struct ltb_ctx {
  int device = 0;
  cudaStream_t st = nullptr;
  std::mutex mu;                // guards `allocs` (a model ctx is shared by every session thread that uploads / frees)
  std::vector<void*> allocs;
  float* zero_bias = nullptr;   // 16384 zeros (bias of bias-free GEMMs)
  float* gn_ws = nullptr;       // GroupNorm statistics workspace
  float* splitk_ws = nullptr;   // fp32 split-K workspace (zero between uses)
  long long launches = 0;
  bool capturing = false;
  long long capture_launches = 0;
};
struct ltb_graph {
  cudaGraph_t g = nullptr;
  cudaGraphExec_t exec = nullptr;
  long long launches = 0;
};

// the calling thread may be a fresh render / inference / process thread whose current device is 0
#define LTB_CTX_ENTER(c)                                                                          \
  do {                                                                                            \
    int _cur = -1;                                                                                \
    if (cudaGetDevice(&_cur) != cudaSuccess || _cur != (c)->device) LTB_CUDA(cudaSetDevice((c)->device)); \
  } while (0)

static const int kZeroBias = 16384;
static const int kGnWsFloats = 64 * 64 * 2;
static const size_t kSplitKWsFloats = (size_t)16 << 20;  // ksplit * M * Cout floats

extern "C" {

int ltb_ctx_create(ltb_ctx** out) {
  if (!out) return LTB_FAIL("null argument");
  auto* c = new ltb_ctx();
  cudaError_t e = cudaGetDevice(&c->device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->zero_bias), kZeroBias * sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(c->zero_bias, 0, kZeroBias * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->gn_ws), kGnWsFloats * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->splitk_ws), kSplitKWsFloats * sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(c->splitk_ws, 0, kSplitKWsFloats * sizeof(float));
  if (e != cudaSuccess) {
    delete c;
    return LTB_FAIL(std::string("ctx create: ") + cudaGetErrorString(e));
  }
  *out = c;
  return 0;
}

int ltb_ctx_destroy(ltb_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->st);
  for (void* p : c->allocs) cudaFree(p);
  cudaFree(c->zero_bias);
  cudaFree(c->gn_ws);
  cudaFree(c->splitk_ws);
  cudaStreamDestroy(c->st);
  delete c;
  return 0;
}

int ltb_ctx_stream(ltb_ctx* c, void** stream) {
  if (!c || !stream) return LTB_FAIL("null argument");
  LTB_CTX_ENTER(c);
  *stream = static_cast<void*>(c->st);
  return 0;
}
int ltb_ctx_sync(ltb_ctx* c) {
  if (!c) return LTB_FAIL("null ctx");
  LTB_CTX_ENTER(c);
  LTB_CUDA(cudaStreamSynchronize(c->st));
  return 0;
}
int ltb_ctx_launch_count(ltb_ctx* c, long long* n) {
  if (!c || !n) return LTB_FAIL("null argument");
  LTB_CTX_ENTER(c);
  *n = c->launches;
  return 0;
}

int ltb_dev_alloc(ltb_ctx* c, size_t bytes, int zero, void** dptr) {
  if (!c || !dptr) return LTB_FAIL("null argument");
  LTB_CTX_ENTER(c);
  void* p = nullptr;
  LTB_CUDA(cudaMalloc(&p, bytes ? bytes : 16));
  if (zero) LTB_CUDA(cudaMemset(p, 0, bytes ? bytes : 16));
  {
    std::lock_guard<std::mutex> lk(c->mu);
    c->allocs.push_back(p);
  }
  *dptr = p;
  return 0;
}
int ltb_dev_free(ltb_ctx* c, void* dptr) {
  if (!c || !dptr) return 0;
  LTB_CTX_ENTER(c);
  {
    std::lock_guard<std::mutex> lk(c->mu);
    size_t i = 0;
    while (i < c->allocs.size() && c->allocs[i] != dptr) ++i;
    if (i == c->allocs.size()) return LTB_FAIL("dev_free: pointer not owned by this context");
    c->allocs.erase(c->allocs.begin() + i);
  }
  cudaFree(dptr);
  return 0;
}
int ltb_h2d(ltb_ctx* c, void* dst_dev, const void* src_host, size_t bytes, int sync) {
  if (!c) return LTB_FAIL("null ctx");
  LTB_CTX_ENTER(c);
  LTB_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, c->st));
  if (sync) LTB_CUDA(cudaStreamSynchronize(c->st));
  return 0;
}
int ltb_d2h(ltb_ctx* c, void* dst_host, const void* src_dev, size_t bytes, int sync) {
  if (!c) return LTB_FAIL("null ctx");
  LTB_CTX_ENTER(c);
  LTB_CUDA(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, c->st));
  if (sync) LTB_CUDA(cudaStreamSynchronize(c->st));
  return 0;
}
int ltb_set_i32(ltb_ctx* c, void* dptr, int value) {
  if (!c || !dptr) return LTB_FAIL("null argument");
  LTB_CTX_ENTER(c);
  LTB_CUDA(launch_set_int(static_cast<int*>(dptr), value, c->st));
  c->launches += 1;
  return 0;
}

// ---- graph capture ------------------------------------------------------------------------------
int ltb_capture_begin(ltb_ctx* c) {
  if (!c) return LTB_FAIL("null ctx");
  LTB_CTX_ENTER(c);
  if (c->capturing) return LTB_FAIL("already capturing");
  LTB_CUDA(cudaStreamBeginCapture(c->st, cudaStreamCaptureModeThreadLocal));
  c->capturing = true;
  c->capture_launches = c->launches;
  return 0;
}
int ltb_capture_end(ltb_ctx* c, ltb_graph** out) {
  if (!c || !out) return LTB_FAIL("null argument");
  LTB_CTX_ENTER(c);
  if (!c->capturing) return LTB_FAIL("not capturing");
  c->capturing = false;
  auto* g = new ltb_graph();
  cudaError_t e = cudaStreamEndCapture(c->st, &g->g);
  if (e == cudaSuccess) e = cudaGraphInstantiate(&g->exec, g->g, 0);
  if (e != cudaSuccess) {
    if (g->g) cudaGraphDestroy(g->g);
    delete g;
    return LTB_FAIL(std::string("graph capture/instantiate: ") + cudaGetErrorString(e));
  }
  g->launches = c->launches - c->capture_launches;
  c->launches = c->capture_launches;  // captured launches did not execute
  *out = g;
  return 0;
}
int ltb_graph_launch(ltb_ctx* c, ltb_graph* g) {
  if (!c || !g) return LTB_FAIL("null argument");
  LTB_CTX_ENTER(c);
  LTB_CUDA(cudaGraphLaunch(g->exec, c->st));
  c->launches += g->launches;
  return 0;
}
int ltb_graph_destroy(ltb_graph* g) {
  if (!g) return 0;
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->g) cudaGraphDestroy(g->g);
  delete g;
  return 0;
}

// ---- ops ----------------------------------------------------------------------------------------
int ltb_op_conv2d(ltb_ctx* c, const ltb_conv_op* d) {
  if (!c || !d || !d->in || !d->w || !d->out) return LTB_FAIL("conv2d: null argument");
  LTB_CTX_ENTER(c);
  if (d->KH * d->KW > kMaxTaps) return LTB_FAIL("conv2d: kernel too large");
  pdl_set_enabled(pdl_default());   // the calling thread may have run a w2l profiling pass with PDL off
  if (d->Cout > kZeroBias && !d->bias) return LTB_FAIL("conv2d: Cout too large for the implicit zero bias");
  ConvParams p;
  std::memset(&p, 0, sizeof(p));
  p.in = static_cast<const __half*>(d->in);
  p.N = d->N;
  p.IH = d->IH;
  p.IW = d->IW;
  p.ICtot = d->ICtot;
  p.ic_off = d->ic_off;
  p.Cin = d->Cin;
  p.sy = d->sy;
  p.sx = d->sx;
  p.GH = d->OH;
  p.GW = d->OW;
  p.out = static_cast<__half*>(d->out);
  p.OH = d->OH;
  p.OW = d->OW;
  p.OCtot = d->OCtot;
  p.oc_off = d->oc_off;
  p.osy = p.osx = 1;
  p.Cout = d->Cout;
  p.res = static_cast<const __half*>(d->res);
  p.RCtot = d->RCtot;
  p.rc_off = d->rc_off;
  p.w = static_cast<const __half*>(d->w);
  p.Ktot = d->Ktot;
  p.bias = d->bias ? d->bias : c->zero_bias;
  p.relu = d->relu;
  p.M = d->N * d->OH * d->OW;
  p.nphases = 1;
  p.ph[0].ntaps = d->KH * d->KW;
  p.ph[0].koff = d->w_koff;
  for (int kh = 0; kh < d->KH; ++kh)
    for (int kw = 0; kw < d->KW; ++kw) {
      p.ph[0].dy[kh * d->KW + kw] = (signed char)(kh - d->pad_t);
      p.ph[0].dx[kh * d->KW + kw] = (signed char)(kw - d->pad_l);
    }
  if (d->upsample2x) {
    if (d->KH != 3 || d->KW != 3 || d->sy != 1 || d->sx != 1 || d->pad_t != 1 || d->pad_l != 1 || d->OH != 2 * d->IH || d->OW != 2 * d->IW ||
        d->Ktot != 16 * d->Cin || !d->w_tap || d->zbatch > 1)
      return LTB_FAIL("conv2d: upsample2x needs a 3x3 s1 p1 conv, OH = 2*IH, OW = 2*IW and the 16-slice weights");
    // four sub-pixel phases over the low-resolution grid: phase (a, b) reads rows {-1, 0} (a = 0) or {0, +1} (a = 1)
    p.GH = d->IH;
    p.GW = d->IW;
    p.M = d->N * d->IH * d->IW;
    p.osy = p.osx = 2;
    p.nphases = 4;
    p.upconv = 1;
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b) {
        ConvPhase& ph = p.ph[a * 2 + b];
        ph.ntaps = 4;
        ph.koff = (a * 2 + b) * 4 * d->Cin;
        ph.ooy = a;
        ph.oox = b;
        for (int ry = 0; ry < 2; ++ry)
          for (int rx = 0; rx < 2; ++rx) {
            ph.dy[ry * 2 + rx] = (signed char)(ry - 1 + a);
            ph.dx[ry * 2 + rx] = (signed char)(rx - 1 + b);
          }
      }
    if (!conv_halo_supported(p)) return LTB_FAIL("conv2d: upsample2x: geometry not supported by the halo kernel (Cout % 64, Cin % 8)");
  }
  p.zbatch = d->zbatch;
  p.zdiv = d->zdiv > 0 ? d->zdiv : 1;
  p.in_zo = d->in_zo;
  p.in_zi = d->in_zi;
  p.w_zo = d->w_zo;
  p.w_zi = d->w_zi;
  p.out_zo = d->out_zo;
  p.out_zi = d->out_zi;
  cudaError_t e;
  const bool want_stats = d->gn_stats != nullptr && d->gn_groups > 0 && d->gn_hw > 0 && (p.M % d->gn_hw) == 0 && d->zbatch <= 1;
  bool stats_fused = false;
  const bool one_by_one = (d->KH == 1 && d->KW == 1);
  if ((d->w_tap || one_by_one) && d->zbatch <= 1 && !d->no_halo && conv_halo_supported(p)) {
    HaloPlan pl;
    if (conv_halo_make_plan(p, static_cast<const __half*>(d->w_tap), &pl) != 0) return LTB_FAIL("conv2d: tensor map creation failed");
    if (want_stats && d->oc_off == 0 && d->OCtot == d->Cout && conv_halo_gn_fusable(pl, d->Cout, d->gn_groups, d->gn_hw)) {
      // GroupNorm statistics of the output are accumulated by the conv epilogue
      LTB_CUDA(cudaMemsetAsync(d->gn_stats, 0, (size_t)(p.M / d->gn_hw) * d->gn_groups * 2 * sizeof(float), c->st));
      pl.hp.gn_stats = static_cast<float*>(d->gn_stats);
      pl.hp.gn_groups = d->gn_groups;
      pl.hp.gn_cpg = d->Cout / d->gn_groups;
      pl.hp.gn_hw = d->gn_hw;
      pl.hp.gn_images = p.M / d->gn_hw;
      stats_fused = true;
    }
    e = launch_conv_halo(pl, c->st);
  } else {
    e = launch_conv_gather(p, c->st, c->splitk_ws, kSplitKWsFloats);
  }
  if (e != cudaSuccess) return LTB_FAIL(std::string("conv2d launch: ") + cudaGetErrorString(e));
  c->launches += 1;
  if (want_stats && !stats_fused) {
    // fallback: separate statistics pass over the freshly written output
    e = launch_gn_stats(static_cast<const __half*>(d->out), p.M / d->gn_hw, d->gn_hw, d->Cout, d->OCtot, d->oc_off, d->gn_groups,
                        static_cast<float*>(d->gn_stats), c->st);
    if (e != cudaSuccess) return LTB_FAIL(std::string("conv2d gn_stats: ") + cudaGetErrorString(e));
    c->launches += 1;
  }
  return 0;
}

int ltb_op_w_tap_major(ltb_ctx* c, const void* w, void* wt, int cout, int cin) {
  if (!c || !w || !wt) return LTB_FAIL("null argument");
  LTB_CTX_ENTER(c);
  LTB_CUDA(launch_w_tap_major(static_cast<const __half*>(w), static_cast<__half*>(wt), cout, cin, c->st));
  c->launches += 1;
  return 0;
}

int ltb_op_groupnorm(ltb_ctx* c, const void* x, int N, int HW, int C, int Ctot, int c_off, int groups, float eps, const float* gamma,
                     const float* beta, int silu, void* out, int OCtot, int oc_off) {
  if (!c || !x || !out || !gamma || !beta) return LTB_FAIL("groupnorm: null argument");
  LTB_CTX_ENTER(c);
  if ((size_t)N * groups * 2 > (size_t)kGnWsFloats) return LTB_FAIL("groupnorm: batch too large for the statistics workspace");
  cudaError_t e = launch_groupnorm(static_cast<const __half*>(x), N, HW, C, Ctot, c_off, groups, eps, gamma, beta, silu,
                                   static_cast<__half*>(out), OCtot, oc_off, c->gn_ws, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("groupnorm: ") + cudaGetErrorString(e));
  c->launches += 2;
  return 0;
}
int ltb_op_groupnorm_apply(ltb_ctx* c, const void* x, int N, int HW, int C, int Ctot, int c_off, int groups, float eps, const void* stats,
                           const float* gamma, const float* beta, int silu, void* out, int OCtot, int oc_off) {
  if (!c || !x || !out || !gamma || !beta || !stats) return LTB_FAIL("groupnorm_apply: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_gn_apply(static_cast<const __half*>(x), N, HW, C, Ctot, c_off, groups, eps, static_cast<const float*>(stats), gamma,
                                  beta, silu, static_cast<__half*>(out), OCtot, oc_off, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("groupnorm_apply: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_layernorm(ltb_ctx* c, const void* x, int rows, int C, float eps, const float* gamma, const float* beta, void* out) {
  if (!c || !x || !out) return LTB_FAIL("layernorm: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_layernorm(static_cast<const __half*>(x), rows, C, eps, gamma, beta, static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("layernorm: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_softmax(ltb_ctx* c, const void* x, int rows, int cols, int ld, int valid, float scale, void* out) {
  if (!c || !x || !out) return LTB_FAIL("softmax: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_softmax(static_cast<const __half*>(x), rows, cols, ld, valid, scale, static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("softmax: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_geglu(ltb_ctx* c, const void* h, long long rows, int H, void* out) {
  if (!c || !h || !out) return LTB_FAIL("geglu: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_geglu(static_cast<const __half*>(h), (size_t)rows, H, static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("geglu: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_eltwise(ltb_ctx* c, const void* x, const void* y, long long n, long long period, int act, void* out) {
  if (!c || !x || !out) return LTB_FAIL("eltwise: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_eltwise(static_cast<const __half*>(x), static_cast<const __half*>(y), (size_t)n, (size_t)period, act,
                                 static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("eltwise: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_upsample2x(ltb_ctx* c, const void* x, int N, int H, int W, int C, void* out) {
  if (!c || !x || !out) return LTB_FAIL("upsample2x: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_upsample2x(static_cast<const __half*>(x), N, H, W, C, static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("upsample2x: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_copy_channels(ltb_ctx* c, const void* src, long long rows, int C, int SCtot, int sc_off, void* dst, int DCtot, int dc_off) {
  if (!c || !src || !dst) return LTB_FAIL("copy_channels: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_copy_channels(static_cast<const __half*>(src), (size_t)rows, C, SCtot, sc_off, static_cast<__half*>(dst), DCtot,
                                       dc_off, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("copy_channels: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_transpose_heads(ltb_ctx* c, const void* v, int B, int n_keys, int Ctot, int c_off, int heads, int d, int n_pad, void* vt) {
  if (!c || !v || !vt) return LTB_FAIL("transpose_heads: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_transpose_heads(static_cast<const __half*>(v), B, n_keys, Ctot, c_off, heads, d, n_pad, static_cast<__half*>(vt),
                                         c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("transpose_heads: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_attention(ltb_ctx* c, const void* q, int q_pitch, const void* k, int kv_pitch, int kv_rows, const void* vt, int n_pad, int B, int heads,
                     int nq, int valid, int d, float scale, void* out, int out_pitch) {
  if (!c || !q || !k || !vt || !out) return LTB_FAIL("attention: null argument");
  if (!attn_fused_supported(d, q_pitch, kv_pitch, n_pad)) return LTB_FAIL("attention: unsupported head dim / pitch (d % 16 == 0, d <= 160, pitches % 8 == 0)");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_attn_fused(static_cast<const __half*>(q), q_pitch, static_cast<const __half*>(k), kv_pitch, kv_rows,
                                    static_cast<const __half*>(vt), n_pad, B, heads, nq, valid, d, scale, static_cast<__half*>(out), out_pitch, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("attention: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
// ---- UltraLight / HuBERT ops (SURVEY 8 row f4)
int ltb_op_dwconv3x3(ltb_ctx* c, const void* x, int N, int IH, int IW, int ICtot, int ic_off, int C, const void* w_tap, const float* bias, int stride,
                     int relu, void* out, int OCtot, int oc_off) {
  if (!c || !x || !w_tap || !bias || !out) return LTB_FAIL("dwconv3x3: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_dwconv3x3(static_cast<const __half*>(x), N, IH, IW, ICtot, ic_off, C, static_cast<const __half*>(w_tap), bias, stride, relu,
                                   static_cast<__half*>(out), OCtot, oc_off, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("dwconv3x3 (C, pitches, offsets % 8 == 0; stride 1 | 2): ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_upsample_bilinear2x(ltb_ctx* c, const void* x, int N, int H, int W, int ICtot, int ic_off, int C, void* out, int OCtot, int oc_off) {
  if (!c || !x || !out) return LTB_FAIL("upsample_bilinear2x: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_upsample_bilinear2x(static_cast<const __half*>(x), N, H, W, ICtot, ic_off, C, static_cast<__half*>(out), OCtot, oc_off, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("upsample_bilinear2x: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_ul_prep(ltb_ctx* c, const void* faces_u8, int nf, const void* d_index, int B, void* out) {
  if (!c || !faces_u8 || !d_index || !out || nf < 1 || B < 1) return LTB_FAIL("ul_prep: bad argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_ul_prep(static_cast<const uint8_t*>(faces_u8), nf, static_cast<const int*>(d_index), B, static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("ul_prep: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_head_sigmoid255(ltb_ctx* c, const void* x, const float* w3x32, const float* b3, long long npix, float* pred) {
  if (!c || !x || !w3x32 || !b3 || !pred) return LTB_FAIL("head_sigmoid255: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_w2l_head(static_cast<const __half*>(x), w3x32, b3, pred, (int)npix, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("head_sigmoid255: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_ul_paste(ltb_ctx* c, const void* frames, const void* faces, const void* coords, const float* pred, void* out, int nf, int H, int W,
                    int index, int explicit_idx, int slot0, int count) {
  if (!c || !frames || !faces || !coords || !pred || !out || nf < 1 || count < 1) return LTB_FAIL("ul_paste: bad argument");
  if (explicit_idx >= nf) return LTB_FAIL("ul_paste: frame index out of range");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_ul_paste(static_cast<const uint8_t*>(frames), static_cast<const uint8_t*>(faces), static_cast<const int*>(coords), pred,
                                  static_cast<uint8_t*>(out), nf, H, W, index, explicit_idx, slot0, count, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("ul_paste: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_ul_paste_region(ltb_ctx* c, const void* faces, const void* coords, const float* pred, void* out, int nf, int rh, int rw, int index,
                           int explicit_idx, int slot0, int count) {
  if (!c || !faces || !coords || !pred || !out || nf < 1 || count < 1 || rh < 1 || rw < 1) return LTB_FAIL("ul_paste_region: bad argument");
  if (explicit_idx >= nf) return LTB_FAIL("ul_paste_region: frame index out of range");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_ul_paste_region(static_cast<const uint8_t*>(faces), static_cast<const int*>(coords), pred, static_cast<uint8_t*>(out), nf,
                                         rh, rw, index, explicit_idx, slot0, count, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("ul_paste_region: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_hubert_conv0(ltb_ctx* c, const float* pcm, int n, const float* w, const float* bias, int C, float* stats, void* out) {
  if (!c || !pcm || !w || !stats || !out) return LTB_FAIL("hubert_conv0: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_hubert_conv0(pcm, n, w, bias, C, stats, static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("hubert_conv0: ") + cudaGetErrorString(e));
  c->launches += 2;
  return 0;
}
int ltb_op_hubert_pos_conv(ltb_ctx* c, const void* h, int T, int D, int groups, int K, const void* w, const float* bias, void* out) {
  if (!c || !h || !w || !bias || !out) return LTB_FAIL("hubert_pos_conv: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_hubert_pos_conv(static_cast<const __half*>(h), T, D, groups, K, static_cast<const __half*>(w), bias, static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("hubert_pos_conv (K = 128, D / groups = 64, out != h): ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_hubert_slice(ltb_ctx* c, const void* hidden, int Tc, int T, int D, int B, int R, float start, float mult, int win_l, float* out_f32,
                        void* out_nhwc) {
  if (!c || !hidden || (!out_f32 && !out_nhwc)) return LTB_FAIL("hubert_slice: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_hubert_slice(static_cast<const __half*>(hidden), Tc, T, D, B, R, start, mult, win_l, out_f32, static_cast<__half*>(out_nhwc), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("hubert_slice: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_vae_post(ltb_ctx* c, const void* x, long long npix, int Ctot, void* out_u8) {
  if (!c || !x || !out_u8) return LTB_FAIL("vae_post: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_vae_post(static_cast<const __half*>(x), (size_t)npix, Ctot, static_cast<uint8_t*>(out_u8), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("vae_post: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_bgr_to_i420(ltb_ctx* c, const void* bgr_u8, int N, int H, int W, void* out_i420) {
  if (!c || !bgr_u8 || !out_i420) return LTB_FAIL("bgr_to_i420: null argument");
  LTB_CTX_ENTER(c);
  if (N <= 0 || H <= 0 || W <= 0 || (H & 1) || (W & 3)) return LTB_FAIL("bgr_to_i420: needs even height and a width that is a multiple of 4");
  cudaError_t e = launch_bgr_to_i420(static_cast<const uint8_t*>(bgr_u8), N, H, W, static_cast<uint8_t*>(out_i420), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("bgr_to_i420: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_stamp_pixels(ltb_ctx* c, void* frames_u8, int N, int H, int W, const void* pix_yx, int n, int b, int g, int r) {
  if (!c || !frames_u8 || (!pix_yx && n > 0)) return LTB_FAIL("stamp_pixels: null argument");
  if (N < 0 || n < 0 || H <= 0 || W <= 0) return LTB_FAIL("stamp_pixels: bad size");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_stamp_pixels(static_cast<uint8_t*>(frames_u8), N, H, W, static_cast<const int*>(pix_yx), n, b, g, r, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("stamp_pixels: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_vae_pre(ltb_ctx* c, const void* img_u8, int N, int H, int W, int half_mask, void* out) {
  if (!c || !img_u8 || !out) return LTB_FAIL("vae_pre: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_vae_pre(static_cast<const uint8_t*>(img_u8), N, H, W, half_mask, static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("vae_pre: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_gather_rows(ltb_ctx* c, const void* table, int n, const void* d_index, int B, long long row_elems, void* out) {
  if (!c || !table || !d_index || !out) return LTB_FAIL("gather_rows: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_gather_rows(static_cast<const __half*>(table), n, static_cast<const int*>(d_index), B, (size_t)row_elems,
                                     static_cast<__half*>(out), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("gather_rows: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_whisper_logmel(ltb_ctx* c, const void* pcm_f32, int n, const void* fb_f32, void* logspec_ws, void* gmax_ws, void* out_f16,
                          void* out_f32) {
  if (!c || !pcm_f32 || !fb_f32 || !logspec_ws || !gmax_ws || !out_f16) return LTB_FAIL("whisper_logmel: null argument");
  LTB_CTX_ENTER(c);
  cudaError_t e = launch_whisper_logmel(static_cast<const float*>(pcm_f32), n, static_cast<const float*>(fb_f32),
                                        static_cast<float*>(logspec_ws), static_cast<int*>(gmax_ws), static_cast<__half*>(out_f16),
                                        static_cast<float*>(out_f32), c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("whisper_logmel: ") + cudaGetErrorString(e));
  c->launches += 3;
  return 0;
}
int ltb_op_whisper_slice(ltb_ctx* c, const void* const* hidden5, int T, int D, int B, float start, float mult, void* out,
                         int out_rows_per_frame) {
  if (!c || !hidden5 || !out) return LTB_FAIL("whisper_slice: null argument");
  LTB_CTX_ENTER(c);
  if (D % 8 != 0 || out_rows_per_frame < 50) return LTB_FAIL("whisper_slice: bad shape");
  cudaError_t e = launch_whisper_slice(reinterpret_cast<const __half* const*>(hidden5), T, D, B, start, mult, static_cast<__half*>(out),
                                       out_rows_per_frame, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("whisper_slice: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}
int ltb_op_mt_paste(ltb_ctx* c, const ltb_mt_paste_op* d) {
  if (!c || !d) return LTB_FAIL("mt_paste: null argument");
  LTB_CTX_ENTER(c);
  MtPasteArgs a;
  a.frames = static_cast<const uint8_t*>(d->frames);
  a.coords = static_cast<const int*>(d->coords);
  a.crop = static_cast<const int*>(d->crop);
  a.masks = static_cast<const uint8_t*>(d->masks);
  a.mask_off = static_cast<const long long*>(d->mask_off);
  a.pred = static_cast<const uint8_t*>(d->pred);
  a.out = static_cast<uint8_t*>(d->out);
  a.nf = d->nf;
  a.H = d->H;
  a.W = d->W;
  a.index = d->index;
  a.explicit_idx = d->explicit_idx;
  a.slot0 = d->slot0;
  a.S = d->pred_hw > 0 ? d->pred_hw : 256;
  a.body = static_cast<const uint8_t*>(d->body);
  a.rh = d->region_h;
  a.rw = d->region_w;
  if (!a.body && !a.frames) return LTB_FAIL("mt_paste: frames == NULL (frame-free avatar): set body to its body crops for the region form");
  if (a.body && (a.rh < 1 || a.rw < 1)) return LTB_FAIL("mt_paste: the region form needs region_h, region_w >= the crop boxes");
  cudaError_t e = launch_mt_paste(a, d->count, c->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("mt_paste: ") + cudaGetErrorString(e));
  c->launches += 1;
  return 0;
}

}  // extern "C"
