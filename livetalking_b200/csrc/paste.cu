// wav2lip paste-back composite (replaces the CPU OpenCV path of LipReal.paste_back_frame,
// avatars/wav2lip_avatar.py:141-147):
//     combine = frame.copy(); res = cv2.resize(pred.astype(np.uint8), (x2-x1, y2-y1)); combine[y1:y2, x1:x2] = res
// Integer/byte work, bit-exact with OpenCV's 8-bit INTER_LINEAR: 11-bit fixed-point taps computed with the same
// float32/float64 expression order, int32 horizontal pass, ((b0*(S0>>4))>>16 + (b1*(S1>>4))>>16 + 2)>>2 vertical
// pass, and the INTER_AREA 2x2 box average OpenCV silently substitutes for an exact 2x decimation.
// HBM-bound: 2*H*W*3 bytes per frame; one thread = 4 output pixels (12 contiguous bytes).
#include "cv_resize.cuh"
#include "ltb_internal.h"

namespace ltb {

// One pixel of cv2.resize(pred.astype(u8), (dw, dh)) at (dy, dx) of the paste rectangle: the per-pixel arithmetic shared by the
// full-frame kernels and the region kernel.  The row taps depend on dy only and are set up once per row.
struct W2LRowTaps {
  bool same, area;
  int dy, sy0, sy1, b0, b1;
  double scale_x;
};

__device__ __forceinline__ W2LRowTaps w2l_row_taps(int dy, int dw, int dh) {
  W2LRowTaps t;
  t.same = (dw == 256 && dh == 256);
  t.area = (dw == 128 && dh == 128);
  t.dy = dy;
  int sy = 0;
  t.b0 = 2048;
  t.b1 = 0;
  if (!t.same && !t.area) cv_tap(dy, 1.0 / ((double)dh / 256.0), 256, false, sy, t.b0, t.b1);
  t.sy0 = min(max(sy, 0), 255);
  t.sy1 = min(max(sy + 1, 0), 255);
  t.scale_x = 1.0 / ((double)dw / 256.0);
  return t;
}

__device__ __forceinline__ void w2l_resize_px(const float* pred, const W2LRowTaps& t, int dx, int v3[3]) {
  if (t.same) {
    const float* p = pred + ((size_t)t.dy * 256 + dx) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) v3[c] = trunc_u8(p[c]);
  } else if (t.area) {
    const float* p = pred + ((size_t)(2 * t.dy) * 256 + 2 * dx) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c)
      v3[c] = (trunc_u8(p[c]) + trunc_u8(p[3 + c]) + trunc_u8(p[768 + c]) + trunc_u8(p[771 + c]) + 2) >> 2;
  } else {
    int sx, a0, a1;
    cv_tap(dx, t.scale_x, 256, true, sx, a0, a1);
    const int sx1 = min(sx + 1, 255);
    const float* r0 = pred + (size_t)t.sy0 * 768;
    const float* r1 = pred + (size_t)t.sy1 * 768;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int S0 = trunc_u8(r0[sx * 3 + c]) * a0 + trunc_u8(r0[sx1 * 3 + c]) * a1;
      const int S1 = trunc_u8(r1[sx * 3 + c]) * a0 + trunc_u8(r1[sx1 * 3 + c]) * a1;
      const int v = (((t.b0 * (S0 >> 4)) >> 16) + ((t.b1 * (S1 >> 4)) >> 16) + 2) >> 2;
      v3[c] = min(max(v, 0), 255);
    }
  }
}

struct PasteArgs {
  const uint8_t* frames;  // [nf,H,W,3]
  const int* coords;      // [nf,4] = (y1,y2,x1,x2)
  const float* pred;      // [B,256,256,3]
  uint8_t* out;           // [count,H,W,3]
  int nf, H, W;
  int index;         // first avatar index (mirror_index applied) when explicit_idx < 0
  int explicit_idx;  // >= 0: use this frame index for the (single) job
  int slot0;         // first prediction slot
  const SlotDesc* slots;  // != nullptr: job j pastes into slots[j].frame at slots[j]'s rectangle (cross-session batch)
};

__global__ void __launch_bounds__(256) w2l_paste_kernel(const PasteArgs a) {
  const int job = blockIdx.z;
  const int y = blockIdx.y;
  const int xg = (blockIdx.x * 256 + threadIdx.x) * 4;
  if (xg >= a.W) return;
  int y1, y2, x1, x2;
  const uint8_t* frow;
  if (a.slots) {
    const SlotDesc sd = a.slots[job];
    y1 = sd.y1, y2 = sd.y2, x1 = sd.x1, x2 = sd.x2;
    frow = sd.frame + (size_t)y * a.W * 3;
  } else {
    const int idx = a.explicit_idx >= 0 ? a.explicit_idx : mirror_index_p(a.nf, a.index + job);
    y1 = a.coords[idx * 4 + 0], y2 = a.coords[idx * 4 + 1], x1 = a.coords[idx * 4 + 2], x2 = a.coords[idx * 4 + 3];
    frow = a.frames + ((size_t)idx * a.H + y) * a.W * 3;
  }
  uint8_t* orow = a.out + ((size_t)job * a.H + y) * a.W * 3;
  const float* pred = a.pred + (size_t)(a.slot0 + job) * 256 * 256 * 3;
  const int npx = min(4, a.W - xg);
  uint8_t px[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) px[i] = (i < npx * 3) ? frow[xg * 3 + i] : 0;
  if (y >= y1 && y < y2 && xg + npx > x1 && xg < x2) {
    const W2LRowTaps t = w2l_row_taps(y - y1, x2 - x1, y2 - y1);
    for (int i = 0; i < npx; ++i) {
      const int x = xg + i;
      if (x < x1 || x >= x2) continue;
      int v3[3];
      w2l_resize_px(pred, t, x - x1, v3);
      for (int c = 0; c < 3; ++c) px[i * 3 + c] = (uint8_t)v3[c];
    }
  }
  if (npx == 4 && ((a.W * 3) % 4 == 0)) {
    uint32_t* o32 = reinterpret_cast<uint32_t*>(orow + xg * 3);
    const uint32_t* p32 = reinterpret_cast<const uint32_t*>(px);
    o32[0] = p32[0];
    o32[1] = p32[1];
    o32[2] = p32[2];
  } else {
    for (int i = 0; i < npx * 3; ++i) orow[xg * 3 + i] = px[i];
  }
}

// Vectorised variant for 16-byte aligned rows (W % 16 == 0): one thread = 16 output pixels = three 128-bit loads and stores;
// the kernel above issued 12 single-byte loads per thread and ran at ~1.6 TB/s.  Same integer arithmetic, bit for bit.
__global__ void __launch_bounds__(256) w2l_paste_vec_kernel(const PasteArgs a, int groups_per_row, int total_groups) {
  for (int gidx = blockIdx.x * 256 + threadIdx.x; gidx < total_groups; gidx += gridDim.x * 256) {
    const int xg = (gidx % groups_per_row) * 16;
    const int yj = gidx / groups_per_row;
    const int y = yj % a.H, job = yj / a.H;
    int y1, y2, x1, x2;
    const uint4* frow;
    if (a.slots) {
      const SlotDesc sd = a.slots[job];
      y1 = sd.y1, y2 = sd.y2, x1 = sd.x1, x2 = sd.x2;
      frow = reinterpret_cast<const uint4*>(sd.frame + (size_t)y * a.W * 3 + (size_t)xg * 3);
    } else {
      const int idx = a.explicit_idx >= 0 ? a.explicit_idx : mirror_index_p(a.nf, a.index + job);
      const int4 cb = __ldg(reinterpret_cast<const int4*>(a.coords) + idx);   // (y1, y2, x1, x2)
      y1 = cb.x, y2 = cb.y, x1 = cb.z, x2 = cb.w;
      frow = reinterpret_cast<const uint4*>(a.frames + ((size_t)idx * a.H + y) * a.W * 3 + (size_t)xg * 3);
    }
    uint4* orow = reinterpret_cast<uint4*>(a.out + ((size_t)job * a.H + y) * a.W * 3 + (size_t)xg * 3);
    uint32_t w[12];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const uint4 v = __ldg(frow + i);
      w[4 * i] = v.x;
      w[4 * i + 1] = v.y;
      w[4 * i + 2] = v.z;
      w[4 * i + 3] = v.w;
    }
    if (y >= y1 && y < y2 && xg + 16 > x1 && xg < x2) {
      const float* pred = a.pred + (size_t)(a.slot0 + job) * 256 * 256 * 3;
      const W2LRowTaps t = w2l_row_taps(y - y1, x2 - x1, y2 - y1);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int x = xg + i;
        if (x < x1 || x >= x2) continue;
        int v3[3];
        w2l_resize_px(pred, t, x - x1, v3);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int bi = i * 3 + c;   // static after unrolling: byte bi of the 48-byte group
          w[bi >> 2] = (w[bi >> 2] & ~(0xFFu << ((bi & 3) * 8))) | ((uint32_t)v3[c] << ((bi & 3) * 8));
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) orow[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
  }
}

cudaError_t launch_w2l_paste(const uint8_t* frames, const int* coords, int nf, int H, int W, const float* pred, int slot0,
                             int index, int explicit_idx, int count, uint8_t* out, cudaStream_t st, const SlotDesc* slots) {
  PasteArgs a;
  a.slots = slots;
  a.frames = frames;
  a.coords = coords;
  a.pred = pred;
  a.out = out;
  a.nf = nf;
  a.H = H;
  a.W = W;
  a.index = index;
  a.explicit_idx = explicit_idx;
  a.slot0 = slot0;
  if (W % 16 == 0 && (reinterpret_cast<uintptr_t>(frames) % 16) == 0 && (reinterpret_cast<uintptr_t>(out) % 16) == 0 &&
      (reinterpret_cast<uintptr_t>(coords) % 16) == 0) {
    const int gpr = W / 16;
    const long long total = (long long)gpr * H * count;
    if (total < (1ll << 31)) {
      int blocks = (int)((total + 255) / 256);
      if (blocks > 148 * 16) blocks = 148 * 16;
      w2l_paste_vec_kernel<<<blocks, 256, 0, st>>>(a, gpr, (int)total);
      return cudaGetLastError();
    }
  }
  dim3 grid((W + 1023) / 1024, H, count);
  w2l_paste_kernel<<<grid, 256, 0, st>>>(a);
  return cudaGetLastError();
}

// Region form for frame-free avatars: only the paste rectangle of job j, written to out[j][0:dh][0:dw] of a packed
// [count][rh][rw][3] buffer.  No frame is read; the host writes the rectangle into its own copy of the frame.  One thread = one pixel.
__global__ void __launch_bounds__(256) w2l_paste_region_kernel(const PasteArgs a, int rh, int rw) {
  const int job = blockIdx.z;
  const int dy = blockIdx.y;
  const int dx = blockIdx.x * 256 + threadIdx.x;
  int y1, y2, x1, x2;
  if (a.slots) {
    const SlotDesc sd = a.slots[job];
    y1 = sd.y1, y2 = sd.y2, x1 = sd.x1, x2 = sd.x2;
  } else {
    const int idx = a.explicit_idx >= 0 ? a.explicit_idx : mirror_index_p(a.nf, a.index + job);
    y1 = a.coords[idx * 4 + 0], y2 = a.coords[idx * 4 + 1], x1 = a.coords[idx * 4 + 2], x2 = a.coords[idx * 4 + 3];
  }
  const int dw = x2 - x1, dh = y2 - y1;
  if (dy >= dh || dx >= dw) return;
  const float* pred = a.pred + (size_t)(a.slot0 + job) * 256 * 256 * 3;
  int v3[3];
  w2l_resize_px(pred, w2l_row_taps(dy, dw, dh), dx, v3);
  uint8_t* o = a.out + (((size_t)job * rh + dy) * rw + dx) * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c) o[c] = (uint8_t)v3[c];
}

cudaError_t launch_w2l_paste_region(const int* coords, int nf, const float* pred, int slot0, int index, int explicit_idx, int count,
                                    uint8_t* out, int rh, int rw, cudaStream_t st, const SlotDesc* slots) {
  PasteArgs a{};
  a.slots = slots;
  a.coords = coords;
  a.pred = pred;
  a.out = out;
  a.nf = nf;
  a.index = index;
  a.explicit_idx = explicit_idx;
  a.slot0 = slot0;
  dim3 grid((rw + 255) / 256, rh, count);
  w2l_paste_region_kernel<<<grid, 256, 0, st>>>(a, rh, rw);
  return cudaGetLastError();
}

}  // namespace ltb
