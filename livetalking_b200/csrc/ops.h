// Launchers of the bandwidth-bound operators (ops.cu) and the MuseTalk blend composite (mt_paste.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace ltb {

cudaError_t launch_groupnorm(const __half* x, int N, int HW, int C, int Ctot, int c_off, int groups, float eps, const float* gamma,
                             const float* beta, int silu, __half* out, int OCtot, int oc_off, float* stats_ws, cudaStream_t st);
cudaError_t launch_gn_stats(const __half* x, int N, int HW, int C, int Ctot, int c_off, int groups, float* stats, cudaStream_t st);
cudaError_t launch_gn_apply(const __half* x, int N, int HW, int C, int Ctot, int c_off, int groups, float eps, const float* stats,
                            const float* gamma, const float* beta, int silu, __half* out, int OCtot, int oc_off, cudaStream_t st);
cudaError_t launch_layernorm(const __half* x, int rows, int C, float eps, const float* gamma, const float* beta, __half* out,
                             cudaStream_t st);
cudaError_t launch_softmax(const __half* x, int rows, int cols, int ld, int valid, float scale, __half* out, cudaStream_t st);
cudaError_t launch_geglu(const __half* h, size_t rows, int H, __half* out, cudaStream_t st);
cudaError_t launch_eltwise(const __half* x, const __half* y, size_t n, size_t period, int act, __half* out, cudaStream_t st);
cudaError_t launch_upsample2x(const __half* x, int N, int H, int W, int C, __half* out, cudaStream_t st);
cudaError_t launch_copy_channels(const __half* src, size_t rows, int C, int SCtot, int sc_off, __half* dst, int DCtot, int dc_off,
                                 cudaStream_t st);
cudaError_t launch_transpose_heads(const __half* v, int B, int n_keys, int Ctot, int c_off, int heads, int d, int n_pad, __half* vt,
                                   cudaStream_t st);
// softmax(scale * Q K^T) V in one kernel (attn_fused.cu); head dim d % 16 == 0, d <= 160
bool attn_fused_supported(int d, int q_pitch, int kv_pitch, int n_pad);
cudaError_t launch_attn_fused(const __half* q, int q_pitch, const __half* k, int kv_pitch, int kv_rows, const __half* vt, int n_pad, int B, int H,
                              int nq, int valid, int d, float scale, __half* out, int out_pitch, cudaStream_t st);
// ---- UltraLight / HuBERT (ultralight.cu, hubert.cu)
cudaError_t launch_dwconv3x3(const __half* x, int N, int IH, int IW, int ICtot, int ic_off, int C, const __half* w, const float* bias, int stride,
                             int relu, __half* out, int OCtot, int oc_off, cudaStream_t st);
cudaError_t launch_upsample_bilinear2x(const __half* x, int N, int H, int W, int ICtot, int ic_off, int C, __half* out, int OCtot, int oc_off,
                                       cudaStream_t st);
cudaError_t launch_ul_prep(const uint8_t* faces, int nf, const int* d_index, int B, __half* out, cudaStream_t st);
cudaError_t launch_ul_paste(const uint8_t* frames, const uint8_t* faces, const int* coords, const float* pred, uint8_t* out, int nf, int H, int W,
                            int index, int explicit_idx, int slot0, int count, cudaStream_t st);
// region form: job j's bbox rectangle into out[j][0:h][0:w] of a packed u8 [count][rh][rw][3] buffer, no frame read
cudaError_t launch_ul_paste_region(const uint8_t* faces, const int* coords, const float* pred, uint8_t* out, int nf, int rh, int rw, int index,
                                   int explicit_idx, int slot0, int count, cudaStream_t st);
cudaError_t launch_hubert_conv0(const float* pcm, int n, const float* w, const float* bias, int C, float* stats, __half* out, cudaStream_t st);
cudaError_t launch_hubert_pos_conv(const __half* h, int T, int D, int groups, int K, const __half* w, const float* bias, __half* out,
                                   cudaStream_t st);
cudaError_t launch_hubert_slice(const __half* hidden, int Tc, int T, int D, int B, int R, float start, float mult, int win_l, float* out_f32,
                                __half* out_nhwc, cudaStream_t st);
cudaError_t launch_vae_post(const __half* x, size_t npix, int Ctot, uint8_t* out, cudaStream_t st);
// uint8 BGR [N,H,W,3] -> planar I420 [N, H*3/2, W] (OpenCV COLOR_BGR2YUV_I420 arithmetic); H even, W % 4 == 0
cudaError_t launch_bgr_to_i420(const uint8_t* bgr, int N, int H, int W, uint8_t* out, cudaStream_t st);
cudaError_t launch_stamp_pixels(uint8_t* frames, int N, int H, int W, const int* pix, int n, int b, int g, int r, cudaStream_t st);
cudaError_t launch_vae_pre(const uint8_t* img, int N, int H, int W, int half_mask, __half* out, cudaStream_t st);
cudaError_t launch_gather_rows(const __half* table, int n, const int* d_index, int B, size_t row_elems, __half* out, cudaStream_t st);

// Whisper front-end (whisper.cu)
cudaError_t launch_whisper_logmel(const float* pcm, int n, const float* fb, float* logspec_ws, int* gmax, __half* out16, float* out32,
                                  cudaStream_t st);
cudaError_t launch_whisper_slice(const __half* const* hidden5, int T, int D, int B, float start, float mult, __half* out,
                                 int out_rows_per_frame, cudaStream_t st);

// MuseTalk paste-back (mt_paste.cu): resize + insert + blendLinear, `count` frames per launch
struct MtPasteArgs {
  const uint8_t* frames;     // [nf,H,W,3]
  const int* coords;         // [nf,4] = (x1,y1,x2,y2)           (musetalk_avatar.py:157)
  const int* crop;           // [nf,4] = (x_s,y_s,x_e,y_e)       (myutil.py:7)
  const uint8_t* masks;      // concatenated 3-channel masks, frame i at mask_off[i], size (y_e-y_s) x (x_e-x_s) x 3
  const long long* mask_off;
  const uint8_t* pred;       // [B,S,S,3] u8 BGR (VAE decode output)
  uint8_t* out;              // [count,H,W,3]
  int nf, H, W;
  int index, explicit_idx, slot0;
  int S;                     // prediction side: 256 (reference), 512 for the 64x64-latent configuration
  const uint8_t* body;       // != nullptr: region form (frame-free avatar): body crops packed like the masks; out is [count][rh][rw][3]
  int rh, rw;
};
cudaError_t launch_mt_paste(const MtPasteArgs& a, int count, cudaStream_t st);

}  // namespace ltb
