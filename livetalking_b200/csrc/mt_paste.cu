// MuseTalk paste-back composite (replaces the CPU OpenCV path of MuseReal.paste_back_frame,
// avatars/musetalk_avatar.py:154-164 -> get_image_blending, avatars/musetalk/myutil.py:4-25):
//   res   = cv2.resize(pred.astype(u8), (x2-x1, y2-y1))                       8-bit INTER_LINEAR, fixed point (see paste.cu)
//   large = body[y_s:y_e, x_s:x_e].copy(); large[y1-y_s:y2-y_s, x1-x_s:x2-x_s] = res
//   m     = cvtColor(mask, BGR2GRAY) / 255      (15-bit fixed point: (3735 B + 19235 G + 9798 R + 16384) >> 15)
//   body[y_s:y_e, x_s:x_e] = blendLinear(large, body_crop, m, 1-m) = sat_u8(rint((large*m + body*(1-m)) / (m + (1-m) + 1e-5)))
// Byte work, bit-exact with OpenCV; one thread per output pixel of the full frame (copy outside the crop box), or of the crop box
// alone in the region form.
#include "ltb_internal.h"
#include "ops.h"
#include "ptx_sm100.cuh"

namespace ltb {

__device__ __forceinline__ int mirror_index_m(int size, int index) {
  const int turn = index / size, res = index % size;
  return (turn % 2 == 0) ? res : size - res - 1;
}

__device__ __forceinline__ void cv_tap_m(int d, double scale, int src_len, bool clamp_taps, int& s, int& w0, int& w1) {
  float f = (float)__dadd_rn(__dmul_rn((double)d + 0.5, scale), -0.5);
  int si = (int)floorf(f);
  f = __fsub_rn(f, (float)si);
  if (clamp_taps) {
    if (si < 0) {
      si = 0;
      f = 0.f;
    }
    if (si >= src_len - 1) {
      si = src_len - 1;
      f = 0.f;
    }
  }
  s = si;
  w0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
  w1 = __float2int_rn(__fmul_rn(f, 2048.f));
}

// cv2.resize(pred_u8 SxSx3, (dw, dh)) sampled at (dy, dx), channel c   (S = 256, or 512 for BASELINE configs[4])
__device__ __forceinline__ int resized_px(const uint8_t* __restrict__ pred, int S, int dw, int dh, int dy, int dx, int c) {
  const size_t row = (size_t)S * 3;
  if (dw == S && dh == S) return pred[(size_t)dy * row + dx * 3 + c];
  if (2 * dw == S && 2 * dh == S) {   // exact 2x shrink: OpenCV's INTER_LINEAR takes the 2x2 area path
    const uint8_t* p = pred + (size_t)(2 * dy) * row + 2 * dx * 3 + c;
    return (p[0] + p[3] + p[row] + p[row + 3] + 2) >> 2;
  }
  int sy, b0, b1, sx, a0, a1;
  cv_tap_m(dy, 1.0 / ((double)dh / (double)S), S, false, sy, b0, b1);
  cv_tap_m(dx, 1.0 / ((double)dw / (double)S), S, true, sx, a0, a1);
  const int sy0 = min(max(sy, 0), S - 1), sy1 = min(max(sy + 1, 0), S - 1), sx1 = min(sx + 1, S - 1);
  const uint8_t* r0 = pred + (size_t)sy0 * row;
  const uint8_t* r1 = pred + (size_t)sy1 * row;
  const int S0 = r0[sx * 3 + c] * a0 + r0[sx1 * 3 + c] * a1;
  const int S1 = r1[sx * 3 + c] * a0 + r1[sx1 * 3 + c] * a1;
  const int v = (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2;
  return min(max(v, 0), 255);
}

// blendLinear(large, body, m, 1-m) at one pixel of the crop box: the per-pixel arithmetic shared by the full-frame and the region
// kernels.  mk / body: this pixel of the mask and of the original frame; (fy, fx): its position relative to the bbox (x1, y1).
__device__ __forceinline__ void mt_blend_px(const MtPasteArgs& a, int job, int x1, int y1, int x2, int y2, int fy, int fx, const uint8_t* mk,
                                            const uint8_t* body, uint8_t px[3]) {
  const int gray = (mk[0] * 3735 + mk[1] * 19235 + mk[2] * 9798 + 16384) >> 15;
  const float m = (float)((double)gray / 255.0);          // (mask_image/255).astype(np.float32)
  const float w2 = __fsub_rn(1.f, m);
  const float den = __fadd_rn(__fadd_rn(m, w2), 1e-5f);
  const bool in_face = (fy >= 0 && fy < y2 - y1 && fx >= 0 && fx < x2 - x1);
  const uint8_t* pred = a.pred + (size_t)(a.slot0 + job) * a.S * a.S * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float fl = in_face ? (float)resized_px(pred, a.S, x2 - x1, y2 - y1, fy, fx, c) : (float)body[c];
    const float num = __fadd_rn(__fmul_rn(fl, m), __fmul_rn((float)body[c], w2));
    const int v = __float2int_rn(__fdiv_rn(num, den));
    px[c] = (uint8_t)min(max(v, 0), 255);
  }
}

__global__ void __launch_bounds__(256) mt_paste_kernel(const MtPasteArgs a) {
  pdl_launch_dependents();   // a PDL-launched successor (the conv kernels) may start its prologue now; it waits before reading
  const int job = blockIdx.z, y = blockIdx.y;
  const int x = blockIdx.x * 256 + threadIdx.x;
  if (x >= a.W) return;
  const int idx = a.explicit_idx >= 0 ? a.explicit_idx : mirror_index_m(a.nf, a.index + job);
  const int x1 = a.coords[idx * 4 + 0], y1 = a.coords[idx * 4 + 1], x2 = a.coords[idx * 4 + 2], y2 = a.coords[idx * 4 + 3];
  const int xs = a.crop[idx * 4 + 0], ys = a.crop[idx * 4 + 1], xe = a.crop[idx * 4 + 2], ye = a.crop[idx * 4 + 3];
  const uint8_t* body = a.frames + (((size_t)idx * a.H + y) * a.W + x) * 3;
  uint8_t* o = a.out + (((size_t)job * a.H + y) * a.W + x) * 3;
  uint8_t px[3] = {body[0], body[1], body[2]};
  if (y >= ys && y < ye && x >= xs && x < xe) {
    const uint8_t* mk = a.masks + a.mask_off[idx] + ((size_t)(y - ys) * (xe - xs) + (x - xs)) * 3;
    mt_blend_px(a, job, x1, y1, x2, y2, y - y1, x - x1, mk, body, px);
  }
  o[0] = px[0];
  o[1] = px[1];
  o[2] = px[2];
}

// Region form for frame-free avatars: job j writes only its blended crop box, out[j][0:ye-ys][0:xe-xs] of a packed [count][rh][rw][3]
// buffer.  The original pixels come from the body crops, packed like the masks (same shape, same offsets); no frame is read.
__global__ void __launch_bounds__(256) mt_paste_region_kernel(const MtPasteArgs a) {
  pdl_launch_dependents();
  const int job = blockIdx.z, dy = blockIdx.y;
  const int dx = blockIdx.x * 256 + threadIdx.x;
  const int idx = a.explicit_idx >= 0 ? a.explicit_idx : mirror_index_m(a.nf, a.index + job);
  const int xs = a.crop[idx * 4 + 0], ys = a.crop[idx * 4 + 1], xe = a.crop[idx * 4 + 2], ye = a.crop[idx * 4 + 3];
  if (dy >= ye - ys || dx >= xe - xs) return;
  const int x1 = a.coords[idx * 4 + 0], y1 = a.coords[idx * 4 + 1], x2 = a.coords[idx * 4 + 2], y2 = a.coords[idx * 4 + 3];
  const size_t off = a.mask_off[idx] + ((size_t)dy * (xe - xs) + dx) * 3;
  uint8_t px[3];
  mt_blend_px(a, job, x1, y1, x2, y2, ys + dy - y1, xs + dx - x1, a.masks + off, a.body + off, px);
  uint8_t* o = a.out + (((size_t)job * a.rh + dy) * a.rw + dx) * 3;
  o[0] = px[0];
  o[1] = px[1];
  o[2] = px[2];
}

cudaError_t launch_mt_paste(const MtPasteArgs& a, int count, cudaStream_t st) {
  if (a.body) {
    dim3 grid((a.rw + 255) / 256, a.rh, count);
    return launch_kernel_plain(mt_paste_region_kernel, dim3(grid), dim3(256), 0, st, a);
  }
  dim3 grid((a.W + 255) / 256, a.H, count);
  return launch_kernel_plain(mt_paste_kernel, dim3(grid), dim3(256), 0, st, a);
}

}  // namespace ltb
