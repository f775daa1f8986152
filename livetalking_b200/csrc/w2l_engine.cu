// wav2lip256 engine: weight blob -> layer plan -> CUDA-graph replay, behind the C ABI of include/ltb200.h.
//
// Data layout in HBM (per session, batch B):
//   faces/frames/coords : resident u8 / int32 avatar assets (uploaded once)
//   img_pad   [B,262,264,8]   fp16   zero-bordered 8-channel image (3 masked + 3 full + 2 zero) for the 7x7 stem
//   cat0..7   [B,h,w,Cdec+Cskip] fp16 NHWC  : U-Net skip concat buffers; the decoder block writes channels [0,Cdec),
//                                             the matching encoder block writes [Cdec, Cdec+Cskip)  (torch.cat is gone)
//   tmp ring  fp16 NHWC                      : intra-block activations
//   pred      [B,256,256,3]   f32            : sigmoid*255, the reference's inference_batch return layout
//   frames_out[B,H,W,3]       u8             : composited frames
// Reference topology: avatars/wav2lip/models/wav2lip_v2.py:12-91, forward :123-163.
#include <algorithm>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/ltb200.h"
#include "conv_halo.h"
#include "ltb_internal.h"
#include "stem_umma.h"

namespace ltb {

// ------------------------------------------------------------------------------------------------ errors
static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }

bool pdl_default() {   // process-wide default: on unless LTB_NO_PDL is set
  static const bool on = [] {
    const char* e = std::getenv("LTB_NO_PDL");
    return !(e && e[0] && e[0] != '0');
  }();
  return on;
}
static thread_local int g_pdl = -1;   // current setting of the launching thread (-1: default)
bool pdl_enabled() { return g_pdl < 0 ? pdl_default() : g_pdl == 1; }
void pdl_set_enabled(bool on) { g_pdl = on ? 1 : 0; }
int fail(const char* file, int line, const std::string& msg) {
  const char* base = std::strrchr(file, '/');
  g_last_error = std::string(base ? base + 1 : file) + ":" + std::to_string(line) + ": " + msg;
  return 1;
}

// ------------------------------------------------------------------------------------------------ layer table
struct LDef {
  char kind;  // 'c' conv, 't' transposed conv
  int cin, cout, k, sy, sx, pad;
  bool res;
};
// execution order: audio encoder (0..12), face encoder (13..32), decoder (33..52), output_block.0 (53)
static const LDef kLayers[54] = {
    // audio_encoder, wav2lip_v2.py:41-58
    {'c', 1, 32, 3, 1, 1, 1, false},   {'c', 32, 32, 3, 1, 1, 1, true},    {'c', 32, 32, 3, 1, 1, 1, true},
    {'c', 32, 64, 3, 3, 1, 1, false},  {'c', 64, 64, 3, 1, 1, 1, true},    {'c', 64, 64, 3, 1, 1, 1, true},
    {'c', 64, 128, 3, 3, 3, 1, false}, {'c', 128, 128, 3, 1, 1, 1, true},  {'c', 128, 128, 3, 1, 1, 1, true},
    {'c', 128, 256, 3, 3, 2, 1, false}, {'c', 256, 256, 3, 1, 1, 1, true}, {'c', 256, 512, 3, 1, 1, 0, false},
    {'c', 512, 512, 1, 1, 1, 0, false},
    // face_encoder_blocks, wav2lip_v2.py:12-39
    {'c', 6, 16, 7, 1, 1, 3, false},
    {'c', 16, 32, 3, 2, 2, 1, false},  {'c', 32, 32, 3, 1, 1, 1, true},    {'c', 32, 32, 3, 1, 1, 1, true},
    {'c', 32, 64, 3, 2, 2, 1, false},  {'c', 64, 64, 3, 1, 1, 1, true},    {'c', 64, 64, 3, 1, 1, 1, true},
    {'c', 64, 64, 3, 1, 1, 1, true},
    {'c', 64, 128, 3, 2, 2, 1, false}, {'c', 128, 128, 3, 1, 1, 1, true},  {'c', 128, 128, 3, 1, 1, 1, true},
    {'c', 128, 256, 3, 2, 2, 1, false}, {'c', 256, 256, 3, 1, 1, 1, true}, {'c', 256, 256, 3, 1, 1, 1, true},
    {'c', 256, 512, 3, 2, 2, 1, false}, {'c', 512, 512, 3, 1, 1, 1, true},
    {'c', 512, 512, 3, 2, 2, 1, false}, {'c', 512, 512, 3, 1, 1, 1, true},
    {'c', 512, 512, 4, 1, 1, 0, false}, {'c', 512, 512, 1, 1, 1, 0, false},
    // face_decoder_blocks, wav2lip_v2.py:60-87
    {'c', 512, 512, 1, 1, 1, 0, false},
    {'t', 1024, 512, 4, 1, 1, 0, false}, {'c', 512, 512, 3, 1, 1, 1, true},
    {'t', 1024, 512, 3, 2, 2, 1, false}, {'c', 512, 512, 3, 1, 1, 1, true},
    {'t', 1024, 512, 3, 2, 2, 1, false}, {'c', 512, 512, 3, 1, 1, 1, true}, {'c', 512, 512, 3, 1, 1, 1, true},
    {'t', 768, 384, 3, 2, 2, 1, false},  {'c', 384, 384, 3, 1, 1, 1, true}, {'c', 384, 384, 3, 1, 1, 1, true},
    {'t', 512, 256, 3, 2, 2, 1, false},  {'c', 256, 256, 3, 1, 1, 1, true}, {'c', 256, 256, 3, 1, 1, 1, true},
    {'t', 320, 128, 3, 2, 2, 1, false},  {'c', 128, 128, 3, 1, 1, 1, true}, {'c', 128, 128, 3, 1, 1, 1, true},
    {'t', 160, 64, 3, 2, 2, 1, false},   {'c', 64, 64, 3, 1, 1, 1, true},   {'c', 64, 64, 3, 1, 1, 1, true},
    // output_block.0, wav2lip_v2.py:89
    {'c', 80, 32, 3, 1, 1, 1, false},
};
constexpr int kNumLayers = 54;
constexpr size_t kSplitKFloats = (size_t)8 << 20;  // 8M floats: ksplit * M * Cout of the small-spatial layers (<= 10 x 1024 x 512)
constexpr int kStem = 13, kConvT4 = 34;

// expected packed sizes (elements) of layer i's weight matrix [rows][K]
static void packed_dims(int i, int* rows, int* K) {
  const LDef& L = kLayers[i];
  if (i == 0) {
    *rows = 32;
    *K = 9;
  } else if (i == kStem) {
    *rows = 16;
    *K = 7 * 64;
  } else if (i == kConvT4) {
    *rows = 16 * 512;
    *K = 1024;
  } else {
    *rows = L.cout;
    *K = L.k * L.k * L.cin;
  }
}

// ------------------------------------------------------------------------------------------------ geometry helpers
static void phases_conv(ConvParams& p, int KH, int KW, int pad, int cin) {
  p.nphases = 1;
  ConvPhase& ph = p.ph[0];
  ph.ntaps = KH * KW;
  ph.koff = 0;
  ph.ooy = ph.oox = 0;
  for (int kh = 0; kh < KH; ++kh)
    for (int kw = 0; kw < KW; ++kw) {
      ph.dy[kh * KW + kw] = (signed char)(kh - pad);
      ph.dx[kh * KW + kw] = (signed char)(kw - pad);
    }
  (void)cin;
}

// ConvTranspose2d(k=3, s=2, p=1, op=1): out[2g+a] gathers (d=0,k=1) for a=0 and (d=0,k=2),(d=+1,k=0) for a=1.
static const int kTd[2][2] = {{0, 0}, {0, 1}};
static const int kTk[2][2] = {{1, 0}, {2, 0}};
static const int kTn[2] = {1, 2};
static void phases_convT(ConvParams& p, int cin) {
  p.nphases = 4;
  int koff = 0;
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      ConvPhase& ph = p.ph[a * 2 + b];
      ph.ntaps = kTn[a] * kTn[b];
      ph.koff = koff;
      ph.ooy = a;
      ph.oox = b;
      int t = 0;
      for (int i = 0; i < kTn[a]; ++i)
        for (int j = 0; j < kTn[b]; ++j, ++t) {
          ph.dy[t] = (signed char)kTd[a][i];
          ph.dx[t] = (signed char)kTd[b][j];
        }
      koff += ph.ntaps * cin;
    }
}

// host-side packing of PyTorch-layout float weights into the kernels' K-major fp16 rows (used by ltb_conv2d_f16;
// the model path receives rows already packed by livetalking_b200/w2l_pack.py, which follows the same order)
static void pack_conv_w(const float* w, int cout, int cin, int KH, int KW, std::vector<__half>& out) {
  out.resize((size_t)cout * KH * KW * cin);
  for (int co = 0; co < cout; ++co)
    for (int kh = 0; kh < KH; ++kh)
      for (int kw = 0; kw < KW; ++kw)
        for (int ci = 0; ci < cin; ++ci)
          out[((size_t)co * KH * KW + kh * KW + kw) * cin + ci] = __float2half(w[(((size_t)co * cin + ci) * KH + kh) * KW + kw]);
}
static void pack_convT_w(const float* w, int cin, int cout, std::vector<__half>& out) {
  out.resize((size_t)cout * 9 * cin);
  for (int co = 0; co < cout; ++co) {
    size_t k = 0;
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b)
        for (int i = 0; i < kTn[a]; ++i)
          for (int j = 0; j < kTn[b]; ++j) {
            const int kh = kTk[a][i], kw = kTk[b][j];
            for (int ci = 0; ci < cin; ++ci, ++k)
              out[(size_t)co * 9 * cin + k] = __float2half(w[(((size_t)ci * cout + co) * 3 + kh) * 3 + kw]);
          }
  }
}

// ------------------------------------------------------------------------------------------------ objects
struct BlobEntry {
  char name[40];
  uint32_t dtype;  // 0 = f16, 1 = f32
  uint32_t pad;
  uint64_t offset;
  uint64_t nbytes;
};
struct BlobHeader {
  char magic[8];  // "LTBW2L1"
  uint32_t n_entries;
  uint32_t header_bytes;
};

}  // namespace ltb

using namespace ltb;

struct ltb_w2l_model {
  int device = 0;
  uint8_t* blob = nullptr;
  bool owns = false;
  size_t nbytes = 0;
  const __half* w[kNumLayers] = {nullptr};
  __half* wt[kNumLayers] = {nullptr};  // tap-major [9][Cout][Cin] copies for the halo kernel (3x3 / sub-pixel ConvT layers)
  const float* w0 = nullptr;  // layer 0 weights (f32 [32][9])
  const float* bias[kNumLayers] = {nullptr};
  const float* head_w = nullptr;
  const float* head_b = nullptr;
};

struct ltb_w2l_avatar {
  int device = 0;
  int n = 0, H = 0, W = 0;
  uint8_t* faces = nullptr;
  uint8_t* frames = nullptr;   // nullptr: frame-free avatar (the host keeps the frames; only region outputs are produced)
  int* coords = nullptr;
  std::vector<int> coords_host;
  int rh_max = 0, rw_max = 0;  // largest paste rectangle: the per-slot pitch of region outputs
};

namespace ltb {
struct Tensor {
  __half* p = nullptr;
  int H = 0, W = 0, C = 0;  // C = pixel pitch (total channels)
};
struct Op {
  int type;  // 0 = conv (gather kernel), 1 = prep, 2 = audio conv0, 3 = head, 4 = conv (halo kernel), 5 = stem (tensor-core),
             // 6 = mel of the resident PCM chunk (skipped when the host supplies mel windows)
  ConvParams cp;
  int halo = -1;    // index into the session's halo plans (type 4)
  int branch = 0;   // 1 = audio-encoder branch: runs on the side stream, concurrently with the face encoder
  bool join = false;  // first op that consumes the audio branch's result
};
struct LayerOut {
  const __half* p;
  int H, W, C, Ctot, c_off;
};
}  // namespace ltb

struct ltb_w2l_session {
  ltb_w2l_model* m = nullptr;
  ltb_w2l_avatar* a = nullptr;
  int device = 0;   // copied from the model: entry points and the destructor must not dereference a model that may be gone
  int B = 0, l = 10, r = 10, fps = 25, flags = 0;
  cudaStream_t st = nullptr;
  cudaStream_t st2 = nullptr;  // audio-encoder branch (forked/joined with events; becomes a parallel branch of the graph)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  std::vector<void*> allocs;
  __half* img_pad = nullptr;
  // Threading (avatars/base_avatar.py:469-501): the reference drives one session from three threads — render() calls
  // asr.run_step (-> ltb_w2l_mel_step), inference() calls inference_batch (-> ltb_w2l_infer / paste_batch), process_frames()
  // calls paste_back_frame (-> ltb_w2l_paste*).  `mu` serialises every entry point that enqueues on `st` (each holds it
  // from its first enqueue to its synchronise, so multi-call sequences such as H2D(mel) -> set_int -> graph launch cannot be
  // interleaved); the feature extractor has its OWN stream, buffers and mutex (`mu_asr`), so run_step never touches the
  // forward's mel input and never waits for a forward pass.
  std::mutex mu, mu_asr;
  float* mel = nullptr;           // forward input: written by ltb_w2l_infer (host windows) or by the in-graph mel kernels
  float* pcm = nullptr;           // resident PCM window of the in-graph mel (step_async / step_e2e_async)
  int pcm_cap = 0;
  double* mel_spec = nullptr;
  double* mel_mel = nullptr;
  cudaStream_t st_asr = nullptr;  // ltb_w2l_mel_step only
  float* asr_pcm = nullptr;
  float* asr_mel = nullptr;
  double* asr_spec = nullptr;
  double* asr_melf = nullptr;
  float* pred = nullptr;
  float* pred_scratch = nullptr;  // one host-supplied prediction (ltb_w2l_paste_pred)
  uint8_t* frames_out = nullptr;
  uint8_t* frames_out2 = nullptr;        // second composite buffer: D2H of step i overlaps the kernels of step i+1
  cudaStream_t st_copy = nullptr;
  cudaEvent_t ev_paste[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
  bool copied_valid[2] = {false, false};
  unsigned e2e_seq = 0;
  int* d_index = nullptr;
  SlotDesc* d_slots = nullptr;      // LTB_SESSION_SLOTS: per-slot (face, frame, rectangle) descriptors, rewritten before every step
  float* h_mel_stage = nullptr;     // pinned staging for the B mel windows of a cross-session batch
  SlotDesc* h_slots = nullptr;      // pinned staging for the descriptors
  float* splitk_ws[2] = {nullptr, nullptr};  // one fp32 split-K workspace per stream (main, audio branch)
  std::vector<Op> ops;
  std::vector<HaloPlan> halo_plans;
  StemParams stem;
  LayerOut louts[kNumLayers];
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t gexec = nullptr;
  cudaGraph_t graph_mel = nullptr;       // same forward with the mel kernels heading the audio branch
  cudaGraphExec_t gexec_mel = nullptr;
  long long launches = 0;      // guarded by mu
  long long launches_asr = 0;  // guarded by mu_asr
  int graph_nodes = 0;
  bool pdl = true;   // conv kernels use programmatic dependent launch
};

namespace ltb {

static int dev_alloc(ltb_w2l_session* s, size_t bytes, void** out, bool zero) {
  void* p = nullptr;
  LTB_CUDA(cudaMalloc(&p, bytes));
  if (zero) LTB_CUDA(cudaMemset(p, 0, bytes));
  s->allocs.push_back(p);
  *out = p;
  return 0;
}

// Every entry point may be called from a thread whose current CUDA device is not the session's (the reference starts
// fresh render / inference / process threads, which default to device 0).
static inline int enter(const ltb_w2l_session* s) {
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess || cur != s->device) LTB_CUDA(cudaSetDevice(s->device));
  return 0;
}

static int parse_blob(ltb_w2l_model* m, const uint8_t* host_header, size_t nbytes) {
  if (nbytes < sizeof(BlobHeader)) return LTB_FAIL("weight blob too small");
  BlobHeader h;
  std::memcpy(&h, host_header, sizeof(h));
  if (std::memcmp(h.magic, "LTBW2L1", 7) != 0) return LTB_FAIL("bad weight blob magic");
  if (h.header_bytes > nbytes || h.header_bytes < sizeof(BlobHeader) + (size_t)h.n_entries * sizeof(BlobEntry))
    return LTB_FAIL("bad weight blob header");
  const BlobEntry* ent = reinterpret_cast<const BlobEntry*>(host_header + sizeof(BlobHeader));
  auto find = [&](const std::string& name, uint32_t dtype, size_t expect_bytes, const void** out) -> int {
    for (uint32_t i = 0; i < h.n_entries; ++i) {
      if (name == ent[i].name) {
        if (ent[i].dtype != dtype) return LTB_FAIL("blob entry " + name + ": wrong dtype");
        if (ent[i].nbytes != expect_bytes)
          return LTB_FAIL("blob entry " + name + ": expected " + std::to_string(expect_bytes) + " bytes, got " +
                          std::to_string(ent[i].nbytes));
        if (ent[i].offset % 256 != 0 || ent[i].offset + ent[i].nbytes > nbytes) return LTB_FAIL("blob entry " + name + ": bad offset");
        *out = m->blob + ent[i].offset;
        return 0;
      }
    }
    return LTB_FAIL("blob entry " + name + " missing");
  };
  for (int i = 0; i < kNumLayers; ++i) {
    int rows, K;
    packed_dims(i, &rows, &K);
    char nm[40];
    const void* p = nullptr;
    std::snprintf(nm, sizeof(nm), "L%02d.w", i);
    if (i == 0) {
      if (find(nm, 1, (size_t)rows * K * 4, &p)) return 1;
      m->w0 = static_cast<const float*>(p);
    } else {
      if (find(nm, 0, (size_t)rows * K * 2, &p)) return 1;
      m->w[i] = static_cast<const __half*>(p);
    }
    std::snprintf(nm, sizeof(nm), "L%02d.b", i);
    if (find(nm, 1, (size_t)rows * 4, &p)) return 1;
    m->bias[i] = static_cast<const float*>(p);
  }
  const void* p = nullptr;
  if (find("head.w", 1, 96 * 4, &p)) return 1;
  m->head_w = static_cast<const float*>(p);
  if (find("head.b", 1, 3 * 4, &p)) return 1;
  m->head_b = static_cast<const float*>(p);
  return 0;
}

// fill the generic part of a ConvParams
static ConvParams conv_base(const __half* in, int N, int IH, int IW, int ICtot, int ic_off, int Cin, __half* out, int OH,
                            int OW, int OCtot, int oc_off, int Cout, const __half* w, int Ktot, const float* bias, bool relu) {
  ConvParams p;
  std::memset(&p, 0, sizeof(p));
  p.in = in;
  p.N = N;
  p.IH = IH;
  p.IW = IW;
  p.ICtot = ICtot;
  p.ic_off = ic_off;
  p.Cin = Cin;
  p.sy = p.sx = 1;
  p.GH = OH;
  p.GW = OW;
  p.out = out;
  p.OH = OH;
  p.OW = OW;
  p.OCtot = OCtot;
  p.oc_off = oc_off;
  p.osy = p.osx = 1;
  p.Cout = Cout;
  p.w = w;
  p.Ktot = Ktot;
  p.bias = bias;
  p.relu = relu ? 1 : 0;
  p.M = N * OH * OW;
  p.nphases = 1;
  return p;
}

static int out_dim(int in, int k, int s, int pad) { return (in + 2 * pad - k) / s + 1; }

struct View {
  __half* p;
  int H, W, Ctot, c_off, C;
};

static int build_plan(ltb_w2l_session* s) {
  const int B = s->B;
  const ltb_w2l_model* m = s->m;
  const bool keep = (s->flags & LTB_SESSION_KEEP_LAYERS) != 0;

  // concat buffers: {h, Cdec, Cskip}
  const int catH[8] = {1, 4, 8, 16, 32, 64, 128, 256};
  const int catD[8] = {512, 512, 512, 512, 384, 256, 128, 64};
  const int catS[8] = {512, 512, 512, 256, 128, 64, 32, 16};
  __half* cat[8];
  for (int i = 0; i < 8; ++i) {
    void* p;
    if (dev_alloc(s, (size_t)B * catH[i] * catH[i] * (catD[i] + catS[i]) * 2, &p, true)) return 1;
    cat[i] = static_cast<__half*>(p);
  }
  // temp ring (largest intra-block activation: [B,256,256,64])
  const size_t tmp_bytes = (size_t)B * 256 * 256 * 64 * 2;
  __half* ring[2] = {nullptr, nullptr};
  int ring_next = 0;
  auto new_tmp = [&](int H, int W, int C, View* v) -> int {
    void* p = nullptr;
    if (keep) {
      if (dev_alloc(s, (size_t)B * H * W * C * 2, &p, true)) return 1;
    } else {
      if (!ring[ring_next]) {
        if (dev_alloc(s, tmp_bytes, &p, true)) return 1;
        ring[ring_next] = static_cast<__half*>(p);
      }
      p = ring[ring_next];
      ring_next ^= 1;
    }
    *v = View{static_cast<__half*>(p), H, W, C, 0, C};
    return 0;
  };
  // the audio encoder keeps its own small ring so it never aliases the face branch
  __half* aring[2] = {nullptr, nullptr};
  int aring_next = 0;
  auto new_atmp = [&](int H, int W, int C, View* v) -> int {
    void* p = nullptr;
    if (keep) {
      if (dev_alloc(s, (size_t)B * H * W * C * 2, &p, true)) return 1;
    } else {
      if (!aring[aring_next]) {
        if (dev_alloc(s, (size_t)B * 80 * 16 * 32 * 2, &p, true)) return 1;
        aring[aring_next] = static_cast<__half*>(p);
      }
      p = aring[aring_next];
      aring_next ^= 1;
    }
    *v = View{static_cast<__half*>(p), H, W, C, 0, C};
    return 0;
  };
  auto cat_dec = [&](int i) { return View{cat[i], catH[i], catH[i], catD[i] + catS[i], 0, catD[i]}; };
  auto cat_skip = [&](int i) { return View{cat[i], catH[i], catH[i], catD[i] + catS[i], catD[i], catS[i]}; };
  auto cat_all = [&](int i) { return View{cat[i], catH[i], catH[i], catD[i] + catS[i], 0, catD[i] + catS[i]}; };

  auto record = [&](int li, const View& v) {
    s->louts[li] = LayerOut{v.p, v.H, v.W, v.C, v.Ctot, v.c_off};
  };
  // route a conv to the halo-resident TMA kernel when its geometry allows, else to the generic gather kernel
  auto push_conv = [&](int li, const ConvParams& p) {
    Op o;
    o.type = 0;
    o.cp = p;
    const bool gemm1x1 = (p.nphases == 1 && p.ph[0].ntaps == 1);
    if (!(s->flags & LTB_SESSION_NO_HALO) && (m->wt[li] || gemm1x1) && conv_halo_supported(p)) {
      HaloPlan pl;
      if (conv_halo_make_plan(p, m->wt[li], &pl) == 0) {
        o.type = 4;
        o.halo = (int)s->halo_plans.size();
        s->halo_plans.push_back(pl);
      }
    }
    s->ops.push_back(o);
  };
  // regular conv block li: in -> out (+res)
  auto add_conv = [&](int li, const View& in, const View& out, const View* res) -> int {
    const LDef& L = kLayers[li];
    if (in.C != L.cin || out.C != L.cout) return LTB_FAIL("plan: channel mismatch at layer " + std::to_string(li));
    const int OH = out_dim(in.H, L.k, L.sy, L.pad), OW = out_dim(in.W, L.k, L.sx, L.pad);
    if (OH != out.H || OW != out.W) return LTB_FAIL("plan: spatial mismatch at layer " + std::to_string(li));
    ConvParams p = conv_base(in.p, B, in.H, in.W, in.Ctot, in.c_off, L.cin, out.p, OH, OW, out.Ctot, out.c_off, L.cout,
                             m->w[li], L.k * L.k * L.cin, m->bias[li], true);
    p.sy = L.sy;
    p.sx = L.sx;
    phases_conv(p, L.k, L.k, L.pad, L.cin);
    if (res) {
      p.res = res->p;
      p.RCtot = res->Ctot;
      p.rc_off = res->c_off;
    }
    push_conv(li, p);
    record(li, out);
    return 0;
  };
  auto add_convT = [&](int li, const View& in, const View& out) -> int {
    const LDef& L = kLayers[li];
    if (in.C != L.cin || out.C != L.cout || out.H != 2 * in.H) return LTB_FAIL("plan: convT mismatch at layer " + std::to_string(li));
    ConvParams p = conv_base(in.p, B, in.H, in.W, in.Ctot, in.c_off, L.cin, out.p, out.H, out.W, out.Ctot, out.c_off, L.cout,
                             m->w[li], 9 * L.cin, m->bias[li], true);
    p.GH = in.H;
    p.GW = in.W;
    p.M = B * in.H * in.W;
    p.osy = p.osx = 2;
    phases_convT(p, L.cin);
    push_conv(li, p);
    record(li, out);
    return 0;
  };

  // ---- audio branch first (so the fork precedes the face path): mel of the resident PCM chunk, then audio conv0
  {
    Op o;
    std::memset(&o.cp, 0, sizeof(o.cp));
    o.type = 6;
    o.branch = 1;
    s->ops.push_back(o);
  }
  View a_prev;
  if (new_atmp(80, 16, 32, &a_prev)) return 1;
  {
    Op o;
    std::memset(&o.cp, 0, sizeof(o.cp));
    o.type = 2;
    o.cp.out = a_prev.p;
    o.branch = 1;
    s->ops.push_back(o);
    record(0, a_prev);
  }
  // ---- audio encoder 1..12
  {
    int H = 80, W = 16;
    for (int li = 1; li <= 12; ++li) {
      const LDef& L = kLayers[li];
      const int OH = out_dim(H, L.k, L.sy, L.pad), OW = out_dim(W, L.k, L.sx, L.pad);
      View o;
      if (new_atmp(OH, OW, L.cout, &o)) return 1;
      if (add_conv(li, a_prev, o, L.res ? &a_prev : nullptr)) return 1;
      s->ops.back().branch = 1;
      a_prev = o;
      H = OH;
      W = OW;
    }
  }
  const View audio_emb = a_prev;  // [B,1,1,512]
  // ---- prep (faces -> padded 8-channel fp16 image)
  {
    Op o;
    std::memset(&o.cp, 0, sizeof(o.cp));
    o.type = 1;
    s->ops.push_back(o);
  }

  // ---- face encoder
  // stem (layer 13): 7 row-taps, each K block = 8 consecutive pixels x 8 channels of the padded image
  {
    const View out = cat_skip(7);
    ConvParams p = conv_base(s->img_pad, B, 262, 264, 8, 0, 64, out.p, 256, 256, out.Ctot, out.c_off, 16, m->w[kStem], 7 * 64,
                             m->bias[kStem], true);
    p.nphases = 1;
    p.ph[0].ntaps = 7;
    for (int t = 0; t < 7; ++t) {
      p.ph[0].dy[t] = (signed char)t;
      p.ph[0].dx[t] = 0;
    }
    Op so;
    so.type = 0;
    so.cp = p;
    if (!(s->flags & LTB_SESSION_NO_HALO) && m->wt[kStem] &&
        stem_make_plan(s->img_pad, B, m->wt[kStem], m->bias[kStem], out.p, out.Ctot, out.c_off, &s->stem) == 0)
      so.type = 5;
    s->ops.push_back(so);
    record(kStem, out);
  }
  {
    // blocks 1..7 : first layer strided from the previous skip slice, last layer writes the skip slice
    const int first[8] = {13, 14, 17, 21, 24, 27, 29, 31};
    const int last[8] = {13, 16, 20, 23, 26, 28, 30, 32};
    for (int b = 1; b < 8; ++b) {
      View prev = cat_skip(8 - b);  // output of block b-1 lives in cat[7-(b-1)]
      for (int li = first[b]; li <= last[b]; ++li) {
        const LDef& L = kLayers[li];
        const int OH = out_dim(prev.H, L.k, L.sy, L.pad), OW = out_dim(prev.W, L.k, L.sx, L.pad);
        View o;
        if (li == last[b]) {
          o = cat_skip(7 - b);
        } else {
          if (new_tmp(OH, OW, L.cout, &o)) return 1;
        }
        if (add_conv(li, prev, o, L.res ? &prev : nullptr)) return 1;
        prev = o;
      }
    }
  }
  // ---- decoder
  {
    // block 0: 1x1 conv on the audio embedding -> cat0[0:512]
    if (add_conv(33, audio_emb, cat_dec(0), nullptr)) return 1;
    s->ops.back().join = true;
    // block 1: ConvT(1024->512, k4, s1, p0) on a 1x1 map == 1x1 conv with 16*512 outputs laid out [4,4,512]
    View t;
    if (new_tmp(4, 4, 512, &t)) return 1;
    {
      const View in = cat_all(0);
      ConvParams p = conv_base(in.p, B, 1, 1, in.Ctot, 0, 1024, t.p, 1, 1, 16 * 512, 0, 16 * 512, m->w[kConvT4], 1024,
                               m->bias[kConvT4], true);
      p.ph[0].ntaps = 1;
      p.ph[0].dy[0] = p.ph[0].dx[0] = 0;
      push_conv(kConvT4, p);
      record(kConvT4, t);
    }
    if (add_conv(35, t, cat_dec(1), &t)) return 1;
    const int firstT[8] = {0, 0, 36, 38, 41, 44, 47, 50};
    const int lastC[8] = {0, 0, 37, 40, 43, 46, 49, 52};
    for (int b = 2; b < 8; ++b) {
      View o;
      const View in = cat_all(b - 1);
      if (new_tmp(in.H * 2, in.W * 2, kLayers[firstT[b]].cout, &o)) return 1;
      if (add_convT(firstT[b], in, o)) return 1;
      View prev = o;
      for (int li = firstT[b] + 1; li <= lastC[b]; ++li) {
        View oo;
        if (li == lastC[b]) {
          oo = cat_dec(b);
        } else {
          if (new_tmp(prev.H, prev.W, kLayers[li].cout, &oo)) return 1;
        }
        if (add_conv(li, prev, oo, &prev)) return 1;
        prev = oo;
      }
    }
  }
  // ---- output block: conv 80->32 on cat7, then 1x1 head + sigmoid
  View h;
  if (new_tmp(256, 256, 32, &h)) return 1;
  if (add_conv(53, cat_all(7), h, nullptr)) return 1;
  if (!keep && s->ops.back().type == 4 && s->halo_plans[s->ops.back().halo].BN == 32) {
    // fuse the 1x1 head + sigmoid into the epilogue of layer 53 (its 32-channel activations are never stored)
    HaloParams& hp = s->halo_plans[s->ops.back().halo].hp;
    hp.head_w = m->head_w;
    hp.head_b = m->head_b;
    hp.head_out = s->pred;
  } else {
    Op o;
    std::memset(&o.cp, 0, sizeof(o.cp));
    o.type = 3;
    o.cp.in = h.p;
    s->ops.push_back(o);
  }
  return 0;
}

static const char* op_name(const Op& o) {
  switch (o.type) {
    case 0: return "conv";
    case 1: return "prep_faces";
    case 2: return "audio_conv0";
    case 3: return "head";
    case 4: return "conv_halo";
    case 5: return "stem_umma";
    case 6: return "mel";
  }
  return "?";
}

// enqueue the forward plan on the session stream (reads the step's first avatar index from *d_index).
// events (optional): ops.size()+1 events recorded around every op (profiling pass only).
static int run_ops(ltb_w2l_session* s, bool with_mel, cudaEvent_t* events = nullptr) {
  pdl_set_enabled(s->pdl && events == nullptr);   // the per-op profiling pass times kernels in isolation
  size_t i = 0;
  const bool branches = (events == nullptr);  // the profiling pass serialises everything on the main stream
  bool forked = false;
  for (const Op& o : s->ops) {
    if (events) cudaEventRecord(events[i], s->st);
    cudaStream_t st = s->st;
    if (branches && o.branch == 1) {
      if (!forked) {
        if (cudaEventRecord(s->ev_fork, s->st) != cudaSuccess || cudaStreamWaitEvent(s->st2, s->ev_fork, 0) != cudaSuccess)
          return LTB_FAIL("stream fork failed");
        forked = true;
      }
      st = s->st2;
    }
    if (branches && o.join && forked) {
      if (cudaEventRecord(s->ev_join, s->st2) != cudaSuccess || cudaStreamWaitEvent(s->st, s->ev_join, 0) != cudaSuccess)
        return LTB_FAIL("stream join failed");
      forked = false;
    }
    cudaError_t e = cudaSuccess;
    switch (o.type) {
      case 0: e = launch_conv_gather(o.cp, st, s->splitk_ws[st == s->st2 ? 1 : 0], kSplitKFloats); break;
      case 1: e = launch_w2l_prep_faces(s->a->faces, s->a->n, s->d_index, s->B, s->img_pad, st, s->d_slots); break;
      case 2: e = launch_w2l_audio_conv0(s->mel, s->m->w0, s->m->bias[0], o.cp.out, s->B, st); break;
      case 3: e = launch_w2l_head(o.cp.in, s->m->head_w, s->m->head_b, s->pred, s->B * 65536, st); break;
      case 4: e = launch_conv_halo(s->halo_plans[o.halo], st); break;
      case 5: e = launch_stem(s->stem, st); break;
      case 6:
        if (with_mel) e = launch_mel_step(s->pcm, s->pcm_cap, s->B, s->l, s->fps, s->mel_spec, s->mel_mel, s->mel, st);
        break;
    }
    if (e != cudaSuccess) return LTB_FAIL(std::string("kernel launch failed (") + op_name(o) + "): " + cudaGetErrorString(e));
    ++i;
  }
  if (forked) return LTB_FAIL("plan error: audio branch never joined");
  if (events) cudaEventRecord(events[i], s->st);
  return 0;
}

}  // namespace ltb

// ==================================================================================================== C ABI
extern "C" {

int ltb_version(void) { return 100; }
const char* ltb_last_error(void) { return g_last_error.c_str(); }

int ltb_device_count(int* count) {
  LTB_CUDA(cudaGetDeviceCount(count));
  return 0;
}
int ltb_set_device(int device) {
  LTB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  LTB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return LTB_FAIL(std::string("libltb200 needs an sm_100a GPU (B200); found ") + prop.name);
  return 0;
}

int ltb_host_alloc(size_t nbytes, void** out) {
  LTB_CUDA(cudaHostAlloc(out, nbytes, cudaHostAllocDefault));
  return 0;
}
int ltb_host_free(void* p) {
  LTB_CUDA(cudaFreeHost(p));
  return 0;
}

static void model_free(ltb_w2l_model* m) {
  for (int i = 0; i < kNumLayers; ++i)
    if (m->wt[i]) cudaFree(m->wt[i]);
  if (m->owns && m->blob) cudaFree(m->blob);
  delete m;
}

static int model_from(ltb_w2l_model* m, const uint8_t* header_host, size_t nbytes, ltb_w2l_model** out) {
  if (parse_blob(m, header_host, nbytes)) {
    model_free(m);
    return 1;
  }
  // tap-major weight copies for the halo kernel: every 3x3 p1 conv (stride 1, and stride 2 for the parity-plane path) and every k3 s2 ConvT
  for (int i = 1; i < kNumLayers; ++i) {
    const LDef& L = kLayers[i];
    const bool conv3 = L.kind == 'c' && L.k == 3 && L.pad == 1 && L.cin >= 16 && ((L.sy == 1 && L.sx == 1) || (L.sy == 2 && L.sx == 2));
    const bool convt = L.kind == 't' && L.k == 3;
    if (!conv3 && !convt) continue;
    const size_t bytes = (size_t)L.cout * 9 * L.cin * 2;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&m->wt[i]), bytes);
    if (e == cudaSuccess)
      e = convt ? launch_w_tap_major_convT(m->w[i], m->wt[i], L.cout, L.cin, nullptr)
                : launch_w_tap_major(m->w[i], m->wt[i], L.cout, L.cin, nullptr);
    if (e != cudaSuccess) {
      model_free(m);
      return LTB_FAIL(std::string("tap-major weight copy: ") + cudaGetErrorString(e));
    }
  }
  {  // stem: [16][7][64] -> [7][16][64]
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&m->wt[kStem]), (size_t)16 * 7 * 64 * 2);
    if (e == cudaSuccess) e = launch_w_tap_major(m->w[kStem], m->wt[kStem], 16, 64, nullptr, 7);
    if (e != cudaSuccess) {
      model_free(m);
      return LTB_FAIL(std::string("stem weight copy: ") + cudaGetErrorString(e));
    }
  }
  if (cudaDeviceSynchronize() != cudaSuccess) {
    model_free(m);
    return LTB_FAIL("tap-major weight copy failed");
  }
  *out = m;
  return 0;
}

int ltb_w2l_model_create(const void* blob, size_t nbytes, ltb_w2l_model** out) {
  if (!blob || !out) return LTB_FAIL("null argument");
  auto* m = new ltb_w2l_model();
  LTB_CUDA(cudaGetDevice(&m->device));
  m->nbytes = nbytes;
  m->owns = true;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&m->blob), nbytes);
  if (e == cudaSuccess) e = cudaMemcpy(m->blob, blob, nbytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    delete m;
    return LTB_FAIL(std::string("weight upload: ") + cudaGetErrorString(e));
  }
  return model_from(m, static_cast<const uint8_t*>(blob), nbytes, out);
}

int ltb_w2l_model_create_from_device(void* blob_dev, size_t nbytes, ltb_w2l_model** out) {
  if (!blob_dev || !out) return LTB_FAIL("null argument");
  if (nbytes < sizeof(BlobHeader)) return LTB_FAIL("weight blob too small");
  BlobHeader h;
  LTB_CUDA(cudaMemcpy(&h, blob_dev, sizeof(h), cudaMemcpyDeviceToHost));
  if (h.header_bytes > nbytes || h.header_bytes > (1u << 24)) return LTB_FAIL("bad weight blob header");
  std::vector<uint8_t> header(h.header_bytes);
  LTB_CUDA(cudaMemcpy(header.data(), blob_dev, h.header_bytes, cudaMemcpyDeviceToHost));
  auto* m = new ltb_w2l_model();
  LTB_CUDA(cudaGetDevice(&m->device));
  m->nbytes = nbytes;
  m->owns = false;
  m->blob = static_cast<uint8_t*>(blob_dev);
  return model_from(m, header.data(), nbytes, out);
}

int ltb_w2l_model_destroy(ltb_w2l_model* m) {
  if (!m) return 0;
  model_free(m);
  return 0;
}

int ltb_w2l_avatar_destroy(ltb_w2l_avatar* a);

int ltb_w2l_avatar_create(const uint8_t* faces, const uint8_t* frames, const int32_t* coords, int n, int H, int W,
                          ltb_w2l_avatar** out) {
  if (!faces || !coords || !out || n <= 0 || H <= 0 || W <= 0) return LTB_FAIL("bad avatar arguments");
  int rh_max = 0, rw_max = 0;
  for (int i = 0; i < n; ++i) {
    const int y1 = coords[i * 4], y2 = coords[i * 4 + 1], x1 = coords[i * 4 + 2], x2 = coords[i * 4 + 3];
    if (y1 < 0 || x1 < 0 || y2 > H || x2 > W || y2 <= y1 || x2 <= x1)
      return LTB_FAIL("avatar coords[" + std::to_string(i) + "] outside the frame");
    rh_max = std::max(rh_max, y2 - y1);
    rw_max = std::max(rw_max, x2 - x1);
  }
  auto* a = new ltb_w2l_avatar();
  a->n = n;
  a->H = H;
  a->W = W;
  a->rh_max = rh_max;
  a->rw_max = rw_max;
  a->coords_host.assign(coords, coords + (size_t)n * 4);
  cudaError_t e = cudaGetDevice(&a->device);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&a->faces), (size_t)n * 65536 * 3);
  if (e == cudaSuccess && frames) e = cudaMalloc(reinterpret_cast<void**>(&a->frames), (size_t)n * H * W * 3);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&a->coords), (size_t)n * 4 * sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpy(a->faces, faces, (size_t)n * 65536 * 3, cudaMemcpyHostToDevice);
  if (e == cudaSuccess && frames) e = cudaMemcpy(a->frames, frames, (size_t)n * H * W * 3, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(a->coords, coords, (size_t)n * 4 * sizeof(int), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    ltb_w2l_avatar_destroy(a);
    return LTB_FAIL(std::string("avatar upload: ") + cudaGetErrorString(e));
  }
  *out = a;
  return 0;
}

int ltb_w2l_avatar_region_max(const ltb_w2l_avatar* a, int* rh_max, int* rw_max) {
  if (!a || !rh_max || !rw_max) return LTB_FAIL("null argument");
  *rh_max = a->rh_max;
  *rw_max = a->rw_max;
  return 0;
}

int ltb_mem_get_info(size_t* free_bytes, size_t* total_bytes) {
  if (!free_bytes || !total_bytes) return LTB_FAIL("null argument");
  LTB_CUDA(cudaMemGetInfo(free_bytes, total_bytes));
  return 0;
}

int ltb_w2l_avatar_destroy(ltb_w2l_avatar* a) {
  if (!a) return 0;
  cudaFree(a->faces);
  cudaFree(a->frames);
  cudaFree(a->coords);
  delete a;
  return 0;
}

int ltb_w2l_session_destroy(ltb_w2l_session* s) {
  if (!s) return 0;
  cudaSetDevice(s->device);
  if (s->st) cudaStreamSynchronize(s->st);
  if (s->st_asr) {
    cudaStreamSynchronize(s->st_asr);
    cudaStreamDestroy(s->st_asr);
  }
  if (s->gexec) cudaGraphExecDestroy(s->gexec);
  if (s->graph) cudaGraphDestroy(s->graph);
  if (s->gexec_mel) cudaGraphExecDestroy(s->gexec_mel);
  if (s->graph_mel) cudaGraphDestroy(s->graph_mel);
  for (void* p : s->allocs) cudaFree(p);
  if (s->h_slots) cudaFreeHost(s->h_slots);
  if (s->h_mel_stage) cudaFreeHost(s->h_mel_stage);
  if (s->st_copy) cudaStreamSynchronize(s->st_copy);
  for (int i = 0; i < 2; ++i) {
    if (s->ev_paste[i]) cudaEventDestroy(s->ev_paste[i]);
    if (s->ev_copied[i]) cudaEventDestroy(s->ev_copied[i]);
  }
  if (s->st_copy) cudaStreamDestroy(s->st_copy);
  if (s->ev_fork) cudaEventDestroy(s->ev_fork);
  if (s->ev_join) cudaEventDestroy(s->ev_join);
  if (s->st2) cudaStreamDestroy(s->st2);
  if (s->st) cudaStreamDestroy(s->st);
  delete s;
  return 0;
}

int ltb_w2l_session_create(ltb_w2l_model* m, ltb_w2l_avatar* a, int batch, int stride_left, int stride_right, int fps,
                           int flags, ltb_w2l_session** out) {
  if (!m || !a || !out) return LTB_FAIL("null argument");
  if (batch < 1 || batch > 64) return LTB_FAIL("batch must be in [1,64]");
  if (fps <= 0 || stride_left < 0 || stride_right < 0) return LTB_FAIL("bad fps/stride");
  auto* s = new ltb_w2l_session();
  s->m = m;
  s->a = a;
  s->device = m->device;
  s->B = batch;
  s->l = stride_left;
  s->r = stride_right;
  s->fps = fps;
  s->flags = flags;
  s->pdl = !(flags & LTB_SESSION_NO_PDL) && pdl_default();
  auto bail = [&](int) {
    ltb_w2l_session_destroy(s);
    return 1;
  };
  if (m->device != a->device) return bail(LTB_FAIL("model and avatar live on different devices"));
  if (cudaSetDevice(m->device) != cudaSuccess) return bail(LTB_FAIL("cudaSetDevice failed"));
  if (cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking) != cudaSuccess) return bail(LTB_FAIL("stream create failed"));
  if (cudaStreamCreateWithFlags(&s->st2, cudaStreamNonBlocking) != cudaSuccess) return bail(LTB_FAIL("stream create failed"));
  if (cudaStreamCreateWithFlags(&s->st_asr, cudaStreamNonBlocking) != cudaSuccess) return bail(LTB_FAIL("stream create failed"));
  if (cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming) != cudaSuccess)
    return bail(LTB_FAIL("event create failed"));
  void* p;
  s->pcm_cap = (stride_left + stride_right + 2 * batch) * 320;
  if (flags & LTB_SESSION_MEL_ONLY) {
    // feature extractor only (sessions whose frames are produced by a shared cross-session batch): no activation arena, no
    // layer plan, no graphs — a few hundred KB instead of ~0.9 GB
    if (dev_alloc(s, (size_t)batch * 80 * 16 * 4, &p, true)) return bail(1);
    s->asr_mel = static_cast<float*>(p);
    if (dev_alloc(s, (size_t)s->pcm_cap * 4, &p, true)) return bail(1);
    s->asr_pcm = static_cast<float*>(p);
    if (dev_alloc(s, mel_scratch_spec_doubles(s->pcm_cap) * 8, &p, true)) return bail(1);
    s->asr_spec = static_cast<double*>(p);
    if (dev_alloc(s, mel_scratch_mel_doubles(s->pcm_cap) * 8, &p, true)) return bail(1);
    s->asr_melf = static_cast<double*>(p);
    *out = s;
    return 0;
  }
  if (dev_alloc(s, (size_t)batch * 262 * 264 * 8 * 2, &p, true)) return bail(1);
  s->img_pad = static_cast<__half*>(p);
  if (dev_alloc(s, (size_t)batch * 80 * 16 * 4, &p, true)) return bail(1);
  s->mel = static_cast<float*>(p);
  if (dev_alloc(s, (size_t)s->pcm_cap * 4, &p, true)) return bail(1);
  s->pcm = static_cast<float*>(p);
  if (dev_alloc(s, mel_scratch_spec_doubles(s->pcm_cap) * 8, &p, true)) return bail(1);
  s->mel_spec = static_cast<double*>(p);
  if (dev_alloc(s, mel_scratch_mel_doubles(s->pcm_cap) * 8, &p, true)) return bail(1);
  s->mel_mel = static_cast<double*>(p);
  if (dev_alloc(s, (size_t)batch * 80 * 16 * 4, &p, true)) return bail(1);
  s->asr_mel = static_cast<float*>(p);
  if (dev_alloc(s, (size_t)s->pcm_cap * 4, &p, true)) return bail(1);
  s->asr_pcm = static_cast<float*>(p);
  if (dev_alloc(s, mel_scratch_spec_doubles(s->pcm_cap) * 8, &p, true)) return bail(1);
  s->asr_spec = static_cast<double*>(p);
  if (dev_alloc(s, mel_scratch_mel_doubles(s->pcm_cap) * 8, &p, true)) return bail(1);
  s->asr_melf = static_cast<double*>(p);
  if (dev_alloc(s, (size_t)batch * 65536 * 3 * 4, &p, true)) return bail(1);
  s->pred = static_cast<float*>(p);
  if (dev_alloc(s, (size_t)65536 * 3 * 4, &p, true)) return bail(1);
  s->pred_scratch = static_cast<float*>(p);
  // composite output: full frames, or (frame-free avatar) the packed paste rectangles [batch][rh_max][rw_max][3]
  const size_t out_px = a->frames ? (size_t)a->H * a->W : (size_t)a->rh_max * a->rw_max;
  if (dev_alloc(s, (size_t)batch * out_px * 3, &p, true)) return bail(1);
  s->frames_out = static_cast<uint8_t*>(p);
  if (dev_alloc(s, 256, &p, true)) return bail(1);
  s->d_index = static_cast<int*>(p);
  if (flags & LTB_SESSION_SLOTS) {
    // every slot starts on the session avatar's frame 0 (the warm-up pass and the graph capture read the table)
    if (dev_alloc(s, (size_t)batch * sizeof(SlotDesc), &p, true)) return bail(1);
    s->d_slots = static_cast<SlotDesc*>(p);
    if (cudaHostAlloc(reinterpret_cast<void**>(&s->h_slots), (size_t)batch * sizeof(SlotDesc), cudaHostAllocDefault) != cudaSuccess ||
        cudaHostAlloc(reinterpret_cast<void**>(&s->h_mel_stage), (size_t)batch * 1280 * sizeof(float), cudaHostAllocDefault) != cudaSuccess)
      return bail(LTB_FAIL("pinned staging allocation failed"));
    for (int i = 0; i < batch; ++i)
      s->h_slots[i] = SlotDesc{a->faces, a->frames, a->coords_host[0], a->coords_host[1], a->coords_host[2], a->coords_host[3]};
    if (cudaMemcpy(s->d_slots, s->h_slots, (size_t)batch * sizeof(SlotDesc), cudaMemcpyHostToDevice) != cudaSuccess)
      return bail(LTB_FAIL("slot table upload failed"));
  }
  for (int i = 0; i < 2; ++i) {
    if (dev_alloc(s, kSplitKFloats * sizeof(float), &p, true)) return bail(1);
    s->splitk_ws[i] = static_cast<float*>(p);
  }
  if (build_plan(s)) return bail(1);
  // warm-up (also the reference's warm_up, wav2lip_avatar.py:90-96): one eager pass
  if (launch_set_int(s->d_index, 0, s->st) != cudaSuccess) return bail(LTB_FAIL("set_int launch failed"));
  if (run_ops(s, true)) return bail(1);
  cudaError_t e = cudaStreamSynchronize(s->st);
  if (e != cudaSuccess) return bail(LTB_FAIL(std::string("warm-up forward failed: ") + cudaGetErrorString(e)));
  if (!(flags & (LTB_SESSION_NO_GRAPH | LTB_SESSION_KEEP_LAYERS))) {
    // capture the whole forward into CUDA graphs (with and without the mel kernels); the per-step index lives in device
    // memory.  If the driver refuses programmatic edges in a captured graph, capture again without PDL.
    for (int attempt = 0; attempt < 2; ++attempt) {
      bool ok = true;
      std::string why;
      for (int with_mel = 0; with_mel < 2 && ok; ++with_mel) {
        cudaGraph_t* g = with_mel ? &s->graph_mel : &s->graph;
        cudaGraphExec_t* ge = with_mel ? &s->gexec_mel : &s->gexec;
        e = cudaStreamBeginCapture(s->st, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) return bail(LTB_FAIL(std::string("graph capture begin: ") + cudaGetErrorString(e)));
        const int rc = run_ops(s, with_mel != 0);
        e = cudaStreamEndCapture(s->st, g);
        if (rc || e != cudaSuccess) {
          ok = false;
          why = std::string("graph capture: ") + (rc ? ltb_last_error() : cudaGetErrorString(e));
          break;
        }
        e = cudaGraphInstantiate(ge, *g, 0);
        if (e == cudaSuccess) e = cudaGraphLaunch(*ge, s->st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s->st);
        if (e != cudaSuccess) {
          ok = false;
          why = std::string("graph instantiate/warm-up: ") + cudaGetErrorString(e);
        }
      }
      if (ok) break;
      cudaGetLastError();
      if (s->gexec) cudaGraphExecDestroy(s->gexec);
      if (s->graph) cudaGraphDestroy(s->graph);
      if (s->gexec_mel) cudaGraphExecDestroy(s->gexec_mel);
      if (s->graph_mel) cudaGraphDestroy(s->graph_mel);
      s->gexec = s->gexec_mel = nullptr;
      s->graph = s->graph_mel = nullptr;
      if (attempt == 1 || !s->pdl) return bail(LTB_FAIL(why));
      s->pdl = false;
    }
  }
  *out = s;
  return 0;
}

int ltb_w2l_mel_step(ltb_w2l_session* s, const float* pcm, int nsamples, float* out_mel) {
  if (!s || !pcm) return LTB_FAIL("null argument");
  const int expect = (s->l + s->r + 2 * s->B) * 320;
  if (nsamples != expect) return LTB_FAIL("mel_step: expected " + std::to_string(expect) + " samples, got " + std::to_string(nsamples));
  if (enter(s)) return 1;
  // MelASR.run_step runs on the render thread, concurrently with inference_batch on the inference thread: own stream,
  // own PCM / scratch / output buffers — nothing here is read or written by the forward pass
  std::lock_guard<std::mutex> lk(s->mu_asr);
  LTB_CUDA(cudaMemcpyAsync(s->asr_pcm, pcm, (size_t)nsamples * 4, cudaMemcpyHostToDevice, s->st_asr));
  cudaError_t e = launch_mel_step(s->asr_pcm, nsamples, s->B, s->l, s->fps, s->asr_spec, s->asr_melf, s->asr_mel, s->st_asr);
  if (e != cudaSuccess) return LTB_FAIL(std::string("mel kernels: ") + cudaGetErrorString(e));
  s->launches_asr += 1;
  if (out_mel) LTB_CUDA(cudaMemcpyAsync(out_mel, s->asr_mel, (size_t)s->B * 1280 * 4, cudaMemcpyDeviceToHost, s->st_asr));
  LTB_CUDA(cudaStreamSynchronize(s->st_asr));
  return 0;
}

int ltb_w2l_set_pcm(ltb_w2l_session* s, const float* pcm, int nsamples) {
  if (!s || !pcm) return LTB_FAIL("null argument");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  const int expect = (s->l + s->r + 2 * s->B) * 320;
  if (nsamples != expect) return LTB_FAIL("set_pcm: expected " + std::to_string(expect) + " samples, got " + std::to_string(nsamples));
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  LTB_CUDA(cudaMemcpyAsync(s->pcm, pcm, (size_t)nsamples * 4, cudaMemcpyHostToDevice, s->st));
  LTB_CUDA(cudaStreamSynchronize(s->st));
  return 0;
}

static int need_frames(const ltb_w2l_avatar* a, const char* what) {
  if (a->frames) return 0;
  return LTB_FAIL(std::string(what) + ": the avatar was created frame-free (frames == NULL); use the *_region entry points");
}

static int forward_enqueue(ltb_w2l_session* s, int index, bool with_mel) {
  if (index < 0) return LTB_FAIL("negative index");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  if (launch_set_int(s->d_index, index, s->st) != cudaSuccess) return LTB_FAIL("set_int launch failed");
  if (s->gexec) {
    LTB_CUDA(cudaGraphLaunch(with_mel ? s->gexec_mel : s->gexec, s->st));
  } else {
    if (run_ops(s, with_mel)) return 1;
  }
  s->launches += (long long)s->ops.size() + (with_mel ? 1 : 0);   // set_int + every op but the mel slot (+ the fused mel kernel)
  return 0;
}

int ltb_w2l_infer(ltb_w2l_session* s, int index, const float* mel, float* pred_out) {
  if (!s) return LTB_FAIL("null session");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  if (mel) LTB_CUDA(cudaMemcpyAsync(s->mel, mel, (size_t)s->B * 1280 * 4, cudaMemcpyHostToDevice, s->st));
  if (forward_enqueue(s, index, false)) return 1;
  if (pred_out) LTB_CUDA(cudaMemcpyAsync(pred_out, s->pred, (size_t)s->B * 65536 * 3 * 4, cudaMemcpyDeviceToHost, s->st));
  LTB_CUDA(cudaStreamSynchronize(s->st));
  return 0;
}

int ltb_w2l_paste(ltb_w2l_session* s, int slot, int idx, uint8_t* out_frame) {
  if (!s || !out_frame) return LTB_FAIL("null argument");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  if (slot < 0 || slot >= s->B) return LTB_FAIL("paste: slot out of range");
  if (idx < 0 || idx >= s->a->n) return LTB_FAIL("paste: idx out of range");
  if (need_frames(s->a, "ltb_w2l_paste")) return 1;
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  const size_t fb = (size_t)s->a->H * s->a->W * 3;
  cudaError_t e = launch_w2l_paste(s->a->frames, s->a->coords, s->a->n, s->a->H, s->a->W, s->pred, slot, 0, idx, 1,
                                   s->frames_out + (size_t)slot * fb, s->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("paste kernel: ") + cudaGetErrorString(e));
  s->launches += 1;
  LTB_CUDA(cudaMemcpyAsync(out_frame, s->frames_out + (size_t)slot * fb, fb, cudaMemcpyDeviceToHost, s->st));
  LTB_CUDA(cudaStreamSynchronize(s->st));
  return 0;
}

int ltb_w2l_paste_pred(ltb_w2l_session* s, const float* pred, int idx, uint8_t* out_frame) {
  if (!s || !pred || !out_frame) return LTB_FAIL("null argument");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  if (idx < 0 || idx >= s->a->n) return LTB_FAIL("paste: idx out of range");
  if (need_frames(s->a, "ltb_w2l_paste_pred")) return 1;
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  const size_t fb = (size_t)s->a->H * s->a->W * 3;
  LTB_CUDA(cudaMemcpyAsync(s->pred_scratch, pred, (size_t)65536 * 3 * 4, cudaMemcpyHostToDevice, s->st));
  cudaError_t e = launch_w2l_paste(s->a->frames, s->a->coords, s->a->n, s->a->H, s->a->W, s->pred_scratch, 0, 0, idx, 1,
                                   s->frames_out, s->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("paste kernel: ") + cudaGetErrorString(e));
  s->launches += 1;
  LTB_CUDA(cudaMemcpyAsync(out_frame, s->frames_out, fb, cudaMemcpyDeviceToHost, s->st));
  LTB_CUDA(cudaStreamSynchronize(s->st));
  return 0;
}

static int paste_batch_enqueue(ltb_w2l_session* s, int index, uint8_t* dst = nullptr) {
  cudaError_t e = launch_w2l_paste(s->a->frames, s->a->coords, s->a->n, s->a->H, s->a->W, s->pred, 0, index, -1, s->B,
                                   dst ? dst : s->frames_out, s->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("paste kernel: ") + cudaGetErrorString(e));
  s->launches += 1;
  return 0;
}

int ltb_w2l_paste_batch(ltb_w2l_session* s, int index, uint8_t* out_frames) {
  if (!s) return LTB_FAIL("null session");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  if (index < 0) return LTB_FAIL("negative index");
  if (need_frames(s->a, "ltb_w2l_paste_batch")) return 1;
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  if (paste_batch_enqueue(s, index)) return 1;
  if (out_frames) {
    LTB_CUDA(cudaMemcpyAsync(out_frames, s->frames_out, (size_t)s->B * s->a->H * s->a->W * 3, cudaMemcpyDeviceToHost, s->st));
    LTB_CUDA(cudaStreamSynchronize(s->st));
  }
  return 0;
}

int ltb_w2l_infer_paste(ltb_w2l_session* s, int index, const float* mel, uint8_t* out_frames) {
  if (!s || !mel || !out_frames) return LTB_FAIL("null argument");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  if (need_frames(s->a, "ltb_w2l_infer_paste")) return 1;
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  LTB_CUDA(cudaMemcpyAsync(s->mel, mel, (size_t)s->B * 1280 * 4, cudaMemcpyHostToDevice, s->st));
  if (forward_enqueue(s, index, false)) return 1;
  if (paste_batch_enqueue(s, index)) return 1;
  LTB_CUDA(cudaMemcpyAsync(out_frames, s->frames_out, (size_t)s->B * s->a->H * s->a->W * 3, cudaMemcpyDeviceToHost, s->st));
  LTB_CUDA(cudaStreamSynchronize(s->st));
  return 0;
}

// Shared by both slot forms: validate the requests, stage the per-slot descriptors and mel windows, enqueue the forward.
// region: slots may come from frame-free avatars of any frame size, but every rectangle must fit the session's region pitch.
static int slots_forward_enqueue(ltb_w2l_session* s, const ltb_w2l_slot* slots, int nslots, bool region, const char* what) {
  if (!s->d_slots) return LTB_FAIL(std::string(what) + ": session was not created with LTB_SESSION_SLOTS");
  if (nslots < 1 || nslots > s->B) return LTB_FAIL(std::string(what) + ": 1 <= nslots <= batch");
  const int H = s->a->H, W = s->a->W;
  for (int i = 0; i < nslots; ++i) {
    const ltb_w2l_avatar* a = slots[i].avatar;
    const std::string slot = std::string(what) + ": slot " + std::to_string(i);
    if (!a || !slots[i].mel) return LTB_FAIL(slot + " has a null avatar / mel");
    if (a->device != s->device) return LTB_FAIL(slot + ": avatar lives on another device");
    if (slots[i].idx < 0 || slots[i].idx >= a->n) return LTB_FAIL(slot + ": frame index out of range");
    if (region) {
      const int* c = &a->coords_host[(size_t)slots[i].idx * 4];
      if (c[1] - c[0] > s->a->rh_max || c[3] - c[2] > s->a->rw_max)
        return LTB_FAIL(slot + ": paste rectangle larger than the session avatar's largest (the region pitch)");
    } else {
      if (a->H != H || a->W != W) return LTB_FAIL(slot + ": all avatars of a batch must share the frame size of the session's avatar");
      if (need_frames(a, what)) return 1;
    }
  }
  for (int i = 0; i < s->B; ++i) {
    const ltb_w2l_slot& q = slots[i < nslots ? i : nslots - 1];   // unused slots repeat the last request (results discarded)
    const ltb_w2l_avatar* a = q.avatar;
    const int* c = &a->coords_host[(size_t)q.idx * 4];
    const uint8_t* frame = a->frames ? a->frames + (size_t)q.idx * a->H * a->W * 3 : nullptr;
    s->h_slots[i] = SlotDesc{a->faces + (size_t)q.idx * 65536 * 3, frame, c[0], c[1], c[2], c[3]};
    std::memcpy(s->h_mel_stage + (size_t)i * 1280, q.mel, 1280 * sizeof(float));
  }
  LTB_CUDA(cudaMemcpyAsync(s->d_slots, s->h_slots, (size_t)s->B * sizeof(SlotDesc), cudaMemcpyHostToDevice, s->st));
  LTB_CUDA(cudaMemcpyAsync(s->mel, s->h_mel_stage, (size_t)s->B * 1280 * 4, cudaMemcpyHostToDevice, s->st));
  return forward_enqueue(s, 0, false);
}

int ltb_w2l_infer_slots(ltb_w2l_session* s, const ltb_w2l_slot* slots, int nslots, uint8_t* out_frames) {
  if (!s || !slots || !out_frames) return LTB_FAIL("null argument");
  if (need_frames(s->a, "ltb_w2l_infer_slots")) return 1;
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  if (slots_forward_enqueue(s, slots, nslots, false, "infer_slots")) return 1;
  const int H = s->a->H, W = s->a->W;
  cudaError_t e = launch_w2l_paste(nullptr, nullptr, 0, H, W, s->pred, 0, 0, -1, nslots, s->frames_out, s->st, s->d_slots);
  if (e != cudaSuccess) return LTB_FAIL(std::string("paste kernel: ") + cudaGetErrorString(e));
  s->launches += 1;
  LTB_CUDA(cudaMemcpyAsync(out_frames, s->frames_out, (size_t)nslots * H * W * 3, cudaMemcpyDeviceToHost, s->st));
  LTB_CUDA(cudaStreamSynchronize(s->st));
  return 0;
}

// ---- region forms (any avatar; the only composite forms for a frame-free one) ----
static int region_enqueue_d2h(ltb_w2l_session* s, const float* pred, int index, int explicit_idx, int count, uint8_t* out,
                              int rh, int rw, const SlotDesc* slots) {
  cudaError_t e = launch_w2l_paste_region(s->a->coords, s->a->n, pred, 0, index, explicit_idx, count, s->frames_out, rh, rw, s->st,
                                          slots);
  if (e != cudaSuccess) return LTB_FAIL(std::string("region paste kernel: ") + cudaGetErrorString(e));
  s->launches += 1;
  LTB_CUDA(cudaMemcpyAsync(out, s->frames_out, (size_t)count * rh * rw * 3, cudaMemcpyDeviceToHost, s->st));
  LTB_CUDA(cudaStreamSynchronize(s->st));
  return 0;
}

int ltb_w2l_infer_paste_region(ltb_w2l_session* s, int index, const float* mel, uint8_t* out_regions) {
  if (!s || !mel || !out_regions) return LTB_FAIL("null argument");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  LTB_CUDA(cudaMemcpyAsync(s->mel, mel, (size_t)s->B * 1280 * 4, cudaMemcpyHostToDevice, s->st));
  if (forward_enqueue(s, index, false)) return 1;
  return region_enqueue_d2h(s, s->pred, index, -1, s->B, out_regions, s->a->rh_max, s->a->rw_max, nullptr);
}

int ltb_w2l_infer_slots_region(ltb_w2l_session* s, const ltb_w2l_slot* slots, int nslots, uint8_t* out_regions) {
  if (!s || !slots || !out_regions) return LTB_FAIL("null argument");
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  if (slots_forward_enqueue(s, slots, nslots, true, "infer_slots_region")) return 1;
  return region_enqueue_d2h(s, s->pred, 0, -1, nslots, out_regions, s->a->rh_max, s->a->rw_max, s->d_slots);
}

int ltb_w2l_paste_pred_region(ltb_w2l_session* s, const float* pred, int idx, uint8_t* out_region) {
  if (!s || !pred || !out_region) return LTB_FAIL("null argument");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  if (idx < 0 || idx >= s->a->n) return LTB_FAIL("paste: idx out of range");
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  const int* c = &s->a->coords_host[(size_t)idx * 4];
  LTB_CUDA(cudaMemcpyAsync(s->pred_scratch, pred, (size_t)65536 * 3 * 4, cudaMemcpyHostToDevice, s->st));
  return region_enqueue_d2h(s, s->pred_scratch, 0, idx, 1, out_region, c[1] - c[0], c[3] - c[2], nullptr);
}

int ltb_w2l_mel_resident(ltb_w2l_session* s) {
  if (!s) return LTB_FAIL("null session");
  if (s->ops.empty()) return LTB_FAIL("this session was created with LTB_SESSION_MEL_ONLY: it has no network");
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  cudaError_t e = launch_mel_step(s->pcm, s->pcm_cap, s->B, s->l, s->fps, s->mel_spec, s->mel_mel, s->mel, s->st);
  if (e != cudaSuccess) return LTB_FAIL(std::string("mel kernels: ") + cudaGetErrorString(e));
  s->launches += 1;
  return 0;
}

int ltb_w2l_step_async(ltb_w2l_session* s, int index) {
  if (!s) return LTB_FAIL("null session");
  if (need_frames(s->a, "ltb_w2l_step_async")) return 1;
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  if (forward_enqueue(s, index, true)) return 1;
  return paste_batch_enqueue(s, index);
}

int ltb_w2l_forward_async(ltb_w2l_session* s, int index) {
  if (!s) return LTB_FAIL("null session");
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  return forward_enqueue(s, index, false);
}

int ltb_w2l_profile_ops(ltb_w2l_session* s, int index, int max_ops, int* n_ops, float* ms, double* flops, int* kinds) {
  if (!s || !n_ops) return LTB_FAIL("null argument");
  const int n = (int)s->ops.size();
  *n_ops = n;
  if (!ms) return 0;
  if (max_ops < n) return LTB_FAIL("profile_ops: buffer too small");
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) LTB_CUDA(cudaEventCreate(&e));
  if (launch_set_int(s->d_index, index, s->st) != cudaSuccess) return LTB_FAIL("set_int launch failed");
  int rc = run_ops(s, true, ev.data());
  if (!rc && cudaStreamSynchronize(s->st) != cudaSuccess) rc = LTB_FAIL("profile pass failed");
  for (int i = 0; i < n && !rc; ++i) {
    cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
    const Op& o = s->ops[i];
    if (kinds) kinds[i] = o.type;
    if (flops) {
      double f = 0;
      if (o.type == 0 || o.type == 4 || o.type == 5) {
        for (int p = 0; p < o.cp.nphases; ++p) f += 2.0 * o.cp.M * o.cp.Cout * (double)o.cp.ph[p].ntaps * o.cp.Cin;
      }
      flops[i] = f;
    }
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return rc;
}

int ltb_w2l_e2e_acquire(ltb_w2l_session* s) {
  if (!s) return LTB_FAIL("null session");
  if (enter(s)) return 1;
  cudaEvent_t ev = nullptr;
  {
    std::lock_guard<std::mutex> lk(s->mu);
    const int slot = (int)(s->e2e_seq & 1u);
    if (s->copied_valid[slot]) ev = s->ev_copied[slot];
  }
  if (ev) LTB_CUDA(cudaEventSynchronize(ev));   // step seq-2 (same host buffers) fully drained
  return 0;
}

int ltb_w2l_step_e2e_async(ltb_w2l_session* s, int index, const float* pcm_host, int nsamples, uint8_t* frames_host) {
  if (!s || !pcm_host || !frames_host) return LTB_FAIL("null argument");
  const int expect = (s->l + s->r + 2 * s->B) * 320;
  if (nsamples != expect) return LTB_FAIL("step_e2e: expected " + std::to_string(expect) + " samples");
  if (need_frames(s->a, "ltb_w2l_step_e2e_async")) return 1;
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  if (!s->st_copy) {
    LTB_CUDA(cudaStreamCreateWithFlags(&s->st_copy, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      LTB_CUDA(cudaEventCreateWithFlags(&s->ev_paste[i], cudaEventDisableTiming));
      LTB_CUDA(cudaEventCreateWithFlags(&s->ev_copied[i], cudaEventDisableTiming));
    }
    void* p = nullptr;
    if (dev_alloc(s, (size_t)s->B * s->a->H * s->a->W * 3, &p, true)) return 1;
    s->frames_out2 = static_cast<uint8_t*>(p);
  }
  const int slot = (int)(s->e2e_seq & 1u);
  uint8_t* dev_frames = slot ? s->frames_out2 : s->frames_out;
  // the paste kernel of this step must not overwrite the buffer while the copy of step-2 is still draining it
  if (s->copied_valid[slot]) LTB_CUDA(cudaStreamWaitEvent(s->st, s->ev_copied[slot], 0));
  LTB_CUDA(cudaMemcpyAsync(s->pcm, pcm_host, (size_t)nsamples * 4, cudaMemcpyHostToDevice, s->st));
  if (forward_enqueue(s, index, true)) return 1;
  if (paste_batch_enqueue(s, index, dev_frames)) return 1;
  LTB_CUDA(cudaEventRecord(s->ev_paste[slot], s->st));
  LTB_CUDA(cudaStreamWaitEvent(s->st_copy, s->ev_paste[slot], 0));
  LTB_CUDA(cudaMemcpyAsync(frames_host, dev_frames, (size_t)s->B * s->a->H * s->a->W * 3, cudaMemcpyDeviceToHost, s->st_copy));
  LTB_CUDA(cudaEventRecord(s->ev_copied[slot], s->st_copy));
  s->copied_valid[slot] = true;
  ++s->e2e_seq;
  return 0;
}

int ltb_w2l_sync(ltb_w2l_session* s) {
  if (!s) return LTB_FAIL("null session");
  if (enter(s)) return 1;
  std::lock_guard<std::mutex> lk(s->mu);
  LTB_CUDA(cudaStreamSynchronize(s->st));
  if (s->st_copy) LTB_CUDA(cudaStreamSynchronize(s->st_copy));
  return 0;
}

int ltb_w2l_stream(ltb_w2l_session* s, void** cuda_stream) {
  if (!s || !cuda_stream) return LTB_FAIL("null argument");
  *cuda_stream = static_cast<void*>(s->st);
  return 0;
}

int ltb_w2l_launch_count(ltb_w2l_session* s, long long* n) {
  if (!s || !n) return LTB_FAIL("null argument");
  {
    std::lock_guard<std::mutex> lk(s->mu);
    *n = s->launches;
  }
  {
    std::lock_guard<std::mutex> lk(s->mu_asr);
    *n += s->launches_asr;
  }
  return 0;
}

int ltb_w2l_num_layers(void) { return kNumLayers; }

int ltb_w2l_layer_shape(ltb_w2l_session* s, int layer, int* H, int* W, int* C) {
  if (!s || layer < 0 || layer >= kNumLayers) return LTB_FAIL("bad layer");
  *H = s->louts[layer].H;
  *W = s->louts[layer].W;
  *C = s->louts[layer].C;
  return 0;
}

int ltb_w2l_layer_read(ltb_w2l_session* s, int layer, void* out_f16, size_t nbytes) {
  if (!s || layer < 0 || layer >= kNumLayers || !out_f16) return LTB_FAIL("bad layer");
  if (!(s->flags & LTB_SESSION_KEEP_LAYERS)) return LTB_FAIL("session was not created with LTB_SESSION_KEEP_LAYERS");
  const LayerOut& lo = s->louts[layer];
  const size_t rows = (size_t)s->B * lo.H * lo.W;
  if (nbytes != rows * lo.C * 2) return LTB_FAIL("layer_read: wrong buffer size");
  LTB_CUDA(cudaStreamSynchronize(s->st));
  LTB_CUDA(cudaMemcpy2D(out_f16, (size_t)lo.C * 2, lo.p + lo.c_off, (size_t)lo.Ctot * 2, (size_t)lo.C * 2, rows,
                        cudaMemcpyDeviceToHost));
  return 0;
}

static int conv2d_f16_impl(const ltb_conv_desc* d, const void* in_f16, const float* w_f32, const float* bias_f32,
                           const void* res_f16, void* out_f16, int reps, float* ms_out);

int ltb_conv2d_f16(const ltb_conv_desc* d, const void* in_f16, const float* w_f32, const float* bias_f32,
                   const void* res_f16, void* out_f16) {
  return conv2d_f16_impl(d, in_f16, w_f32, bias_f32, res_f16, out_f16, 0, nullptr);
}

int ltb_conv2d_f16_timed(const ltb_conv_desc* d, const void* in_f16, const float* w_f32, const float* bias_f32,
                         const void* res_f16, void* out_f16, int reps, float* ms_per_launch) {
  if (reps < 1 || !ms_per_launch) return LTB_FAIL("conv2d_f16_timed: reps >= 1 and a result pointer are required");
  return conv2d_f16_impl(d, in_f16, w_f32, bias_f32, res_f16, out_f16, reps, ms_per_launch);
}

static int conv2d_f16_impl(const ltb_conv_desc* d, const void* in_f16, const float* w_f32, const float* bias_f32,
                           const void* res_f16, void* out_f16, int reps, float* ms_out) {
  if (!d || !in_f16 || !w_f32 || !bias_f32 || !out_f16) return LTB_FAIL("null argument");
  if (d->has_res && !res_f16) return LTB_FAIL("has_res set but res is null");
  int OH, OW, Ktot;
  std::vector<__half> wp;
  if (d->transposed) {
    if (d->KH != 3 || d->KW != 3) return LTB_FAIL("transposed conv: only k=3,s=2,p=1,op=1");
    OH = d->IH * 2;
    OW = d->IW * 2;
    Ktot = 9 * d->Cin;
    pack_convT_w(w_f32, d->Cin, d->Cout, wp);
  } else {
    if (d->KH * d->KW > kMaxTaps) return LTB_FAIL("kernel too large");
    OH = out_dim(d->IH, d->KH, d->sy, d->pad);
    OW = out_dim(d->IW, d->KW, d->sx, d->pad);
    Ktot = d->KH * d->KW * d->Cin;
    pack_conv_w(w_f32, d->Cout, d->Cin, d->KH, d->KW, wp);
  }
  if (OH <= 0 || OW <= 0) return LTB_FAIL("empty output");
  const size_t in_b = (size_t)d->N * d->IH * d->IW * d->Cin * 2, out_b = (size_t)d->N * OH * OW * d->Cout * 2;
  __half *din = nullptr, *dout = nullptr, *dw = nullptr, *dres = nullptr, *dwt = nullptr;
  float* dbias = nullptr;
  float* dws = nullptr;
  int rc = 0;
  auto cleanup = [&]() {
    cudaFree(din);
    cudaFree(dout);
    cudaFree(dw);
    cudaFree(dres);
    cudaFree(dwt);
    cudaFree(dws);
    cudaFree(dbias);
  };
#define CK(x)                                                             \
  do {                                                                    \
    cudaError_t _e = (x);                                                 \
    if (_e != cudaSuccess) {                                              \
      rc = LTB_FAIL(std::string(#x) + ": " + cudaGetErrorString(_e));     \
      cleanup();                                                          \
      return rc;                                                          \
    }                                                                     \
  } while (0)
  CK(cudaMalloc(&din, in_b));
  CK(cudaMalloc(&dout, out_b));
  CK(cudaMalloc(&dw, wp.size() * 2));
  CK(cudaMalloc(&dbias, (size_t)d->Cout * 4));
  CK(cudaMemcpy(din, in_f16, in_b, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dw, wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dbias, bias_f32, (size_t)d->Cout * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(dout, 0xFF, out_b));  // NaN pattern: unwritten outputs are caught by the test
  if (d->has_res) {
    CK(cudaMalloc(&dres, out_b));
    CK(cudaMemcpy(dres, res_f16, out_b, cudaMemcpyHostToDevice));
  }
  ConvParams p = conv_base(din, d->N, d->IH, d->IW, d->Cin, 0, d->Cin, dout, OH, OW, d->Cout, 0, d->Cout, dw, Ktot, dbias,
                           d->relu != 0);
  if (d->transposed) {
    p.GH = d->IH;
    p.GW = d->IW;
    p.M = d->N * d->IH * d->IW;
    p.osy = p.osx = 2;
    phases_convT(p, d->Cin);
  } else {
    p.sy = d->sy;
    p.sx = d->sx;
    phases_conv(p, d->KH, d->KW, d->pad, d->Cin);
  }
  if (d->has_res) {
    p.res = dres;
    p.RCtot = d->Cout;
    p.rc_off = 0;
  }
  const bool can_halo = conv_halo_supported(p);
  if (d->force_path == 2 && !can_halo) {
    cleanup();
    return LTB_FAIL("force_path=2 but this geometry is not supported by the halo kernel");
  }
  if (d->force_path != 1 && can_halo) {
    CK(cudaMalloc(&dwt, wp.size() * 2));
    if (d->KH == 3)
      CK(d->transposed ? launch_w_tap_major_convT(dw, dwt, d->Cout, d->Cin, nullptr) : launch_w_tap_major(dw, dwt, d->Cout, d->Cin, nullptr));
    HaloPlan pl;
    if (conv_halo_make_plan(p, dwt, &pl) != 0) {
      cleanup();
      return LTB_FAIL("halo plan / tensor map creation failed");
    }
    CK(launch_conv_halo(pl, nullptr));
    if (reps > 0) {   // back-to-back launches of the same plan between two events (kernel development aid)
      cudaEvent_t e0, e1;
      CK(cudaEventCreate(&e0));
      CK(cudaEventCreate(&e1));
      for (int i = 0; i < 3; ++i) CK(launch_conv_halo(pl, nullptr));
      CK(cudaEventRecord(e0, nullptr));
      for (int i = 0; i < reps; ++i) CK(launch_conv_halo(pl, nullptr));
      CK(cudaEventRecord(e1, nullptr));
      CK(cudaEventSynchronize(e1));
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, e0, e1));
      *ms_out = ms / reps;
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
    }
  } else {
    CK(cudaMalloc(&dws, ((size_t)1 << 22) * sizeof(float)));
    CK(cudaMemset(dws, 0, ((size_t)1 << 22) * sizeof(float)));
    CK(launch_conv_gather(p, nullptr, dws, (size_t)1 << 22));
    if (reps > 0) {
      cudaEvent_t e0, e1;
      CK(cudaEventCreate(&e0));
      CK(cudaEventCreate(&e1));
      CK(cudaEventRecord(e0, nullptr));
      for (int i = 0; i < reps; ++i) CK(launch_conv_gather(p, nullptr, dws, (size_t)1 << 22));
      CK(cudaEventRecord(e1, nullptr));
      CK(cudaEventSynchronize(e1));
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, e0, e1));
      *ms_out = ms / reps;
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
    }
  }
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out_f16, dout, out_b, cudaMemcpyDeviceToHost));
#undef CK
  cleanup();
  return 0;
}

}  // extern "C"
