// UltraLight path kernels (SURVEY 8 row f4): the pieces of avatars/ultralight/unet.py and avatars/ultralight_avatar.py that are
// not dense GEMMs.  The pointwise (1x1) and dense 3x3 convolutions of the U-Net run on the tcgen05 conv kernels; here:
//   * depthwise 3x3 + folded BN + ReLU (InvertedResidual's middle conv, unet.py:18-26)            — HBM/L2-bound, fp32 accumulate
//   * bilinear x2 upsample, align_corners=True (Up.up, unet.py:76) written into a channel slice of the concat buffer
//   * LightReal.inference_batch's input glue (ultralight_avatar.py:146-160): 168x168 u8 crops -> [B,160,160,16] fp16
//   * LightReal.paste_back_frame (ultralight_avatar.py:171-184): crop border + prediction -> cv2.resize -> bbox, bit-exact u8
#include "cv_resize.cuh"
#include "ltb_internal.h"
#include "ops.h"
#include "ptx_sm100.cuh"

namespace ltb {

// ------------------------------------------------------------------------------------------------ depthwise 3x3
// x [N,IH,IW] pixels of ICtot halves (channels [ic_off, ic_off+C)), w tap-major [9][C] fp16 (BN folded), bias fp32 [C];
// out [N,OH,OW] pixels of OCtot halves.  pad 1, stride s.  One thread = 8 channels of one output pixel.
__global__ void __launch_bounds__(256) dwconv3x3_kernel(const __half* __restrict__ x, int N, int IH, int IW, int ICtot, int ic_off, int C,
                                                        const __half* __restrict__ w, const float* __restrict__ bias, int stride, int relu,
                                                        __half* __restrict__ out, int OH, int OW, int OCtot, int oc_off) {
  pdl_launch_dependents();   // a PDL-launched successor (the conv kernels) may start its prologue now; it waits before reading
  const int cg = C >> 3;
  const size_t total = (size_t)N * OH * OW * cg;
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (size_t)gridDim.x * 256) {
    const int c8 = (int)(i % cg) * 8;
    const size_t pix = i / cg;
    const int ox = (int)(pix % OW), oy = (int)((pix / OW) % OH), n = (int)(pix / ((size_t)OW * OH));
    float acc[8];
    {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + c8)), b1 = __ldg(reinterpret_cast<const float4*>(bias + c8 + 4));
      acc[0] = b0.x, acc[1] = b0.y, acc[2] = b0.z, acc[3] = b0.w, acc[4] = b1.x, acc[5] = b1.y, acc[6] = b1.z, acc[7] = b1.w;
    }
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = oy * stride + ky - 1;
      if (iy < 0 || iy >= IH) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int ix = ox * stride + kx - 1;
        if (ix < 0 || ix >= IW) continue;
        const uint4 xv = __ldg(reinterpret_cast<const uint4*>(x + (((size_t)n * IH + iy) * IW + ix) * ICtot + ic_off + c8));
        const uint4 wv = __ldg(reinterpret_cast<const uint4*>(w + (size_t)(ky * 3 + kx) * C + c8));
        const __half2* xh = reinterpret_cast<const __half2*>(&xv);
        const __half2* wh = reinterpret_cast<const __half2*>(&wv);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 a = __half22float2(xh[q]), b = __half22float2(wh[q]);
          acc[2 * q] = fmaf(a.x, b.x, acc[2 * q]);
          acc[2 * q + 1] = fmaf(a.y, b.y, acc[2 * q + 1]);
        }
      }
    }
    uint4 o;
    __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float a = acc[2 * q], b = acc[2 * q + 1];
      if (relu) a = fmaxf(a, 0.f), b = fmaxf(b, 0.f);
      oh[q] = __floats2half2_rn(fminf(fmaxf(a, -65504.f), 65504.f), fminf(fmaxf(b, -65504.f), 65504.f));
    }
    *reinterpret_cast<uint4*>(out + pix * OCtot + oc_off + c8) = o;
  }
}

cudaError_t launch_dwconv3x3(const __half* x, int N, int IH, int IW, int ICtot, int ic_off, int C, const __half* w, const float* bias, int stride,
                             int relu, __half* out, int OCtot, int oc_off, cudaStream_t st) {
  if (C % 8 || ICtot % 8 || ic_off % 8 || OCtot % 8 || oc_off % 8 || (stride != 1 && stride != 2)) return cudaErrorInvalidValue;
  const int OH = (IH + 2 - 3) / stride + 1, OW = (IW + 2 - 3) / stride + 1;
  const size_t total = (size_t)N * OH * OW * (C / 8);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  return launch_kernel_plain(dwconv3x3_kernel, dim3(blocks), dim3(256), 0, st, x, N, IH, IW, ICtot, ic_off, C, w, bias, stride, relu, out, OH, OW, OCtot, oc_off);
}

// ------------------------------------------------------------------------------------------------ bilinear x2, align_corners=True
// F.interpolate(x, scale_factor=2, mode='bilinear', align_corners=True): src = dst * (in-1)/(out-1); fp32 lerp, fp16 out.
__global__ void __launch_bounds__(256) upsample_bilinear2x_kernel(const __half* __restrict__ x, int N, int H, int W, int ICtot, int ic_off, int C,
                                                                  __half* __restrict__ out, int OCtot, int oc_off) {
  pdl_launch_dependents();   // a PDL-launched successor (the conv kernels) may start its prologue now; it waits before reading
  const int cg = C >> 3, OH = 2 * H, OW = 2 * W;
  const float sy = OH > 1 ? (float)(H - 1) / (float)(OH - 1) : 0.f, sx = OW > 1 ? (float)(W - 1) / (float)(OW - 1) : 0.f;
  const size_t total = (size_t)N * OH * OW * cg;
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (size_t)gridDim.x * 256) {
    const int c8 = (int)(i % cg) * 8;
    const size_t pix = i / cg;
    const int ox = (int)(pix % OW), oy = (int)((pix / OW) % OH), n = (int)(pix / ((size_t)OW * OH));
    const float fy = sy * (float)oy, fx = sx * (float)ox;
    const int y0 = (int)fy, x0 = (int)fx;
    const int y1 = y0 + (y0 < H - 1 ? 1 : 0), x1 = x0 + (x0 < W - 1 ? 1 : 0);
    const float ly = fy - (float)y0, lx = fx - (float)x0;
    const __half* base = x + (size_t)n * H * W * ICtot + ic_off + c8;
    const uint4 v00 = __ldg(reinterpret_cast<const uint4*>(base + ((size_t)y0 * W + x0) * ICtot));
    const uint4 v01 = __ldg(reinterpret_cast<const uint4*>(base + ((size_t)y0 * W + x1) * ICtot));
    const uint4 v10 = __ldg(reinterpret_cast<const uint4*>(base + ((size_t)y1 * W + x0) * ICtot));
    const uint4 v11 = __ldg(reinterpret_cast<const uint4*>(base + ((size_t)y1 * W + x1) * ICtot));
    const __half2 *a = reinterpret_cast<const __half2*>(&v00), *b = reinterpret_cast<const __half2*>(&v01),
                  *c = reinterpret_cast<const __half2*>(&v10), *d = reinterpret_cast<const __half2*>(&v11);
    uint4 o;
    __half2* oh = reinterpret_cast<__half2*>(&o);
    const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float2 fa = __half22float2(a[q]), fb = __half22float2(b[q]), fc = __half22float2(c[q]), fd = __half22float2(d[q]);
      oh[q] = __floats2half2_rn(w00 * fa.x + w01 * fb.x + w10 * fc.x + w11 * fd.x, w00 * fa.y + w01 * fb.y + w10 * fc.y + w11 * fd.y);
    }
    *reinterpret_cast<uint4*>(out + pix * OCtot + oc_off + c8) = o;
  }
}

cudaError_t launch_upsample_bilinear2x(const __half* x, int N, int H, int W, int ICtot, int ic_off, int C, __half* out, int OCtot, int oc_off,
                                       cudaStream_t st) {
  if (C % 8 || ICtot % 8 || ic_off % 8 || OCtot % 8 || oc_off % 8) return cudaErrorInvalidValue;
  const size_t total = (size_t)N * 4 * H * W * (C / 8);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  return launch_kernel_plain(upsample_bilinear2x_kernel, dim3(blocks), dim3(256), 0, st, x, N, H, W, ICtot, ic_off, C, out, OCtot, oc_off);
}

// ------------------------------------------------------------------------------------------------ LightReal input glue
// faces u8 [nf,168,168,3] BGR -> [B,160,160,16] fp16: ch 0-2 = centre crop [4:164,4:164] / 255, ch 3-5 = the same with the filled
// cv2.rectangle((5,5,150,145)) = columns [5,154], rows [5,149] zeroed, ch 6-15 = 0 (K padding of the first 1x1 conv).
__global__ void __launch_bounds__(256) ul_prep_kernel(const uint8_t* __restrict__ faces, int nf, const int* __restrict__ d_index, int B,
                                                      __half* __restrict__ out) {
  pdl_launch_dependents();   // a PDL-launched successor (the conv kernels) may start its prologue now; it waits before reading
  const int total = B * 160 * 160;
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= total) return;
  const int x = i % 160, y = (i / 160) % 160, b = i / 25600;
  const int idx = mirror_index_p(nf, *d_index + b);
  const uint8_t* p = faces + (((size_t)idx * 168 + (y + 4)) * 168 + (x + 4)) * 3;
  const bool masked = (x >= 5 && x <= 154 && y >= 5 && y <= 149);
  uint4 lo = make_uint4(0, 0, 0, 0), hi = make_uint4(0, 0, 0, 0);
  __half* h = reinterpret_cast<__half*>(&lo);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float v = __fdiv_rn((float)p[c], 255.f);      // float32 array / 255.0 (ultralight_avatar.py:157-158)
    h[c] = __float2half_rn(v);
    h[3 + c] = masked ? __float2half_rn(0.f) : __float2half_rn(v);
  }
  uint4* o = reinterpret_cast<uint4*>(out + (size_t)i * 16);
  o[0] = lo;
  o[1] = hi;
}

cudaError_t launch_ul_prep(const uint8_t* faces, int nf, const int* d_index, int B, __half* out, cudaStream_t st) {
  return launch_kernel_plain(ul_prep_kernel, dim3((B * 25600 + 255) / 256), dim3(256), 0, st, faces, nf, d_index, B, out);
}

// ------------------------------------------------------------------------------------------------ LightReal.paste_back_frame
struct UlPasteArgs {
  const uint8_t* frames;  // [nf,H,W,3]
  const uint8_t* faces;   // [nf,168,168,3]
  const int* coords;      // [nf,4] = (x1,y1,x2,y2)
  const float* pred;      // [B,160,160,3] = sigmoid * 255
  uint8_t* out;           // [count,H,W,3]
  int nf, H, W, index, explicit_idx, slot0;
};

// pixel (sy, sx), channel c of crop_img_ori after `crop_img_ori[4:164, 4:164] = pred_frame.astype(np.uint8)`
__device__ __forceinline__ int ul_src(const uint8_t* __restrict__ face, const float* __restrict__ pred, int sy, int sx, int c) {
  if (sy >= 4 && sy < 164 && sx >= 4 && sx < 164) return trunc_u8(pred[((sy - 4) * 160 + (sx - 4)) * 3 + c]);
  return face[(sy * 168 + sx) * 3 + c];
}

// pixel (dy, dx) of cv2.resize(crop_img_ori, (dw, dh)): the per-pixel arithmetic shared by the full-frame and the region kernels
__device__ __forceinline__ void ul_resize_px(const uint8_t* __restrict__ face, const float* __restrict__ pred, int dy, int dx, int dw, int dh,
                                             uint8_t px[3]) {
  constexpr int S = 168;
  if (dw == S && dh == S) {
#pragma unroll
    for (int c = 0; c < 3; ++c) px[c] = (uint8_t)ul_src(face, pred, dy, dx, c);
  } else if (2 * dw == S && 2 * dh == S) {   // exact 2x shrink: OpenCV's INTER_LINEAR takes the 2x2 area path
#pragma unroll
    for (int c = 0; c < 3; ++c)
      px[c] = (uint8_t)((ul_src(face, pred, 2 * dy, 2 * dx, c) + ul_src(face, pred, 2 * dy, 2 * dx + 1, c) + ul_src(face, pred, 2 * dy + 1, 2 * dx, c) +
                         ul_src(face, pred, 2 * dy + 1, 2 * dx + 1, c) + 2) >> 2);
  } else {
    int sy, b0, b1, sx, a0, a1;
    cv_tap(dy, 1.0 / ((double)dh / (double)S), S, false, sy, b0, b1);
    cv_tap(dx, 1.0 / ((double)dw / (double)S), S, true, sx, a0, a1);
    const int sy0 = min(max(sy, 0), S - 1), sy1 = min(max(sy + 1, 0), S - 1), sx1 = min(sx + 1, S - 1);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int S0 = ul_src(face, pred, sy0, sx, c) * a0 + ul_src(face, pred, sy0, sx1, c) * a1;
      const int S1 = ul_src(face, pred, sy1, sx, c) * a0 + ul_src(face, pred, sy1, sx1, c) * a1;
      const int v = (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2;
      px[c] = (uint8_t)min(max(v, 0), 255);
    }
  }
}

__global__ void __launch_bounds__(256) ul_paste_kernel(const UlPasteArgs a) {
  pdl_launch_dependents();   // a PDL-launched successor (the conv kernels) may start its prologue now; it waits before reading
  const int job = blockIdx.z, y = blockIdx.y;
  const int x = blockIdx.x * 256 + threadIdx.x;
  if (x >= a.W) return;
  const int idx = a.explicit_idx >= 0 ? a.explicit_idx : mirror_index_p(a.nf, a.index + job);
  const int x1 = a.coords[idx * 4 + 0], y1 = a.coords[idx * 4 + 1], x2 = a.coords[idx * 4 + 2], y2 = a.coords[idx * 4 + 3];
  const uint8_t* body = a.frames + (((size_t)idx * a.H + y) * a.W + x) * 3;
  uint8_t* o = a.out + (((size_t)job * a.H + y) * a.W + x) * 3;
  uint8_t px[3] = {body[0], body[1], body[2]};
  if (y >= y1 && y < y2 && x >= x1 && x < x2)
    ul_resize_px(a.faces + (size_t)idx * 168 * 168 * 3, a.pred + (size_t)(a.slot0 + job) * 160 * 160 * 3, y - y1, x - x1, x2 - x1, y2 - y1, px);
  o[0] = px[0];
  o[1] = px[1];
  o[2] = px[2];
}

cudaError_t launch_ul_paste(const uint8_t* frames, const uint8_t* faces, const int* coords, const float* pred, uint8_t* out, int nf, int H, int W,
                            int index, int explicit_idx, int slot0, int count, cudaStream_t st) {
  UlPasteArgs a{frames, faces, coords, pred, out, nf, H, W, index, explicit_idx, slot0};
  dim3 grid((W + 255) / 256, H, count);
  return launch_kernel_plain(ul_paste_kernel, dim3(grid), dim3(256), 0, st, a);
}

// Region form for frame-free avatars: job j writes only its bbox rectangle, out[j][0:dh][0:dw] of a packed [count][rh][rw][3] buffer;
// no frame is read (a.frames, a.H, a.W unused).
__global__ void __launch_bounds__(256) ul_paste_region_kernel(const UlPasteArgs a, int rh, int rw) {
  pdl_launch_dependents();
  const int job = blockIdx.z, dy = blockIdx.y;
  const int dx = blockIdx.x * 256 + threadIdx.x;
  const int idx = a.explicit_idx >= 0 ? a.explicit_idx : mirror_index_p(a.nf, a.index + job);
  const int x1 = a.coords[idx * 4 + 0], y1 = a.coords[idx * 4 + 1], x2 = a.coords[idx * 4 + 2], y2 = a.coords[idx * 4 + 3];
  if (dy >= y2 - y1 || dx >= x2 - x1) return;
  uint8_t px[3];
  ul_resize_px(a.faces + (size_t)idx * 168 * 168 * 3, a.pred + (size_t)(a.slot0 + job) * 160 * 160 * 3, dy, dx, x2 - x1, y2 - y1, px);
  uint8_t* o = a.out + (((size_t)job * rh + dy) * rw + dx) * 3;
  o[0] = px[0];
  o[1] = px[1];
  o[2] = px[2];
}

cudaError_t launch_ul_paste_region(const uint8_t* faces, const int* coords, const float* pred, uint8_t* out, int nf, int rh, int rw, int index,
                                   int explicit_idx, int slot0, int count, cudaStream_t st) {
  UlPasteArgs a{nullptr, faces, coords, pred, out, nf, 0, 0, index, explicit_idx, slot0};
  dim3 grid((rw + 255) / 256, rh, count);
  return launch_kernel_plain(ul_paste_region_kernel, dim3(grid), dim3(256), 0, st, a, rh, rw);
}

}  // namespace ltb
