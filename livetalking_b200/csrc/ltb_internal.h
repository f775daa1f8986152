// Internal declarations shared by the engine translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include <atomic>
#include <cstdlib>
#include <utility>
#include <string>

#include "conv_params.h"

namespace ltb {

// ---- error plumbing (C ABI returns int status; message via ltb_last_error) ----
void set_error(const std::string& msg);
int fail(const char* file, int line, const std::string& msg);
#define LTB_FAIL(msg) ::ltb::fail(__FILE__, __LINE__, (msg))
#define LTB_CUDA(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      cudaGetLastError(); /* clear the (non-sticky) error: the next launch check must not see it */ \
      return LTB_FAIL(std::string(#expr) + ": " + cudaGetErrorString(_e));                     \
    }                                                                                          \
  } while (0)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: configure each kernel once per device, thread-safely
struct SmemConfigOnce {
  std::atomic<unsigned long long> done{0};  // bit d = configured on device d
  template <typename K>
  cudaError_t ensure(K kernel, int bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const unsigned long long bit = 1ull << (dev & 63);
    if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
    return e;
  }
};

// Programmatic dependent launch of the conv kernels (they all call pdl_wait() before touching activations): overlaps a
// kernel's prologue (barrier init, TMEM allocation, descriptor prefetch, resident-weight loads) with its predecessor's tail.
// Thread-local switch so that a session can capture its graph with or without it (LTB_NO_PDL=1 disables it globally).
bool pdl_default();
bool pdl_enabled();
void pdl_set_enabled(bool on);

template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// Ordinary (fully serialised) launch with the same call shape.  The element-wise / norm / paste kernels use it: they call
// griddepcontrol.launch_dependents first thing, which lets a PDL-launched successor (a conv kernel: it executes griddepcontrol.wait
// before it touches activations) run its prologue under this kernel's tail — but they are never started early themselves, so their
// own loads (some through the non-coherent path: const __restrict__) need no special care.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel_plain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.numAttrs = 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// cross-session batching: one descriptor per batch slot (device memory, rewritten before every step), so that ONE forward /
// paste launch serves frames of different sessions (different avatars, unrelated frame indices)
struct SlotDesc {
  const uint8_t* face;    // u8 [256,256,3] BGR crop of this slot
  const uint8_t* frame;   // u8 [H,W,3] full frame the prediction is pasted into (nullptr: frame-free avatar, region paste)
  int y1, y2, x1, x2;     // paste rectangle (wav2lip coords.pkl order)
};

// ---- kernel launchers ----
// splitk_ws: optional zero-initialised fp32 workspace (one per stream) enabling split-K for small-M deep-K layers
cudaError_t launch_conv_gather(const ConvParams& p, cudaStream_t st, float* splitk_ws = nullptr, size_t splitk_ws_floats = 0);
int conv_gather_pick_bn(const ConvParams& p);

// wav2lip-specific small kernels (w2l_small.cu)
// faces u8 [nf,256,256,3] BGR -> padded fp16 [B,262,264,8]: ch0-2 = face/255 with rows >= 128 zeroed, ch3-5 = face/255
// the first avatar index of the step is read from device memory (*d_index) so that a captured CUDA graph can be replayed
cudaError_t launch_w2l_prep_faces(const uint8_t* faces, int nfaces, const int* d_index, int B, __half* img_pad, cudaStream_t st,
                                  const SlotDesc* slots = nullptr);   // slots != nullptr: face of slot b = slots[b].face
cudaError_t launch_set_int(int* p, int v, cudaStream_t st);
// mel f32 [B,80,16] -> fp16 NHWC [B,80,16,32]: conv3x3 p1 (1->32) + folded BN + ReLU
cudaError_t launch_w2l_audio_conv0(const float* mel, const float* w9x32, const float* bias, __half* out, int B, cudaStream_t st);
// x fp16 [npix,32] -> pred f32 [npix,3] = sigmoid(W x + b) * 255 ; optional u8 copy (truncation)
cudaError_t launch_w2l_head(const __half* x, const float* w3x32, const float* b3, float* pred, int npix, cudaStream_t st);

// mel.cu : PCM f32 [nsamp] -> mel windows f32 [B,80,16] (float64 arithmetic, see mel.cu)
cudaError_t launch_mel_step(const float* pcm, int nsamp, int B, int stride_left_chunks, int fps, double* scratch_spec,
                            double* scratch_mel, float* out, cudaStream_t st);
size_t mel_scratch_spec_doubles(int nsamp);
size_t mel_scratch_mel_doubles(int nsamp);

// paste.cu : wav2lip paste-back for `count` frames in one launch.
//   frame index of job i = explicit_idx (>= 0, count must be 1) or mirror_index(nf, index + i); prediction slot = slot0 + i
cudaError_t launch_w2l_paste(const uint8_t* frames, const int* coords, int nf, int H, int W, const float* pred, int slot0,
                             int index, int explicit_idx, int count, uint8_t* out, cudaStream_t st, const SlotDesc* slots = nullptr);
// same jobs, region form: job i writes only its paste rectangle (h, w) into out[i][0:h][0:w] of a packed u8 [count][rh][rw][3]
// buffer (rh >= h, rw >= w); no frame is read
cudaError_t launch_w2l_paste_region(const int* coords, int nf, const float* pred, int slot0, int index, int explicit_idx, int count,
                                    uint8_t* out, int rh, int rw, cudaStream_t st, const SlotDesc* slots = nullptr);

}  // namespace ltb
