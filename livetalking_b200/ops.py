"""Python handle over the generic device-op layer of the C ABI (``ltb_ctx`` / ``ltb_op_*``, include/ltb200.h).

A ``Ctx`` owns a CUDA stream and device memory; ``DevTensor`` is a (pointer, shape) view — NHWC fp16 activations or raw
byte buffers.  Ops enqueue kernels asynchronously; ``capture()`` records a sequence of ops into a CUDA graph that is
replayed with ``Graph.launch()``.  No computation happens in Python."""
from __future__ import annotations

import contextlib
import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _capi
from ._capi import ConvOp, MtPasteOp, check, lib


class DevTensor:
    __slots__ = ("ptr", "shape", "dtype", "nbytes", "pitch", "c_off", "stats")

    def __init__(self, ptr: int, shape: Sequence[int], dtype=np.float16, pitch: Optional[int] = None, c_off: int = 0):
        self.ptr = int(ptr)
        self.shape = tuple(int(s) for s in shape)
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.pitch = int(pitch) if pitch is not None else self.shape[-1]   # elements between consecutive pixels / rows
        self.c_off = int(c_off)                                            # first channel inside the pitch
        self.stats = None                                                  # (DevTensor, groups): GroupNorm statistics produced with the tensor

    @property
    def C(self) -> int:
        return self.shape[-1]

    @property
    def rows(self) -> int:
        return int(np.prod(self.shape[:-1]))

    def offset(self, elems: int) -> int:
        return self.ptr + elems * self.dtype.itemsize


class Graph:
    def __init__(self, ctx: "Ctx", handle):
        self.ctx, self._h = ctx, handle

    def launch(self):
        check(lib().ltb_graph_launch(self.ctx._h, self._h))

    def close(self):
        if self._h:
            lib().ltb_graph_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Ctx:
    """One CUDA stream + scratch workspaces + a list of owned allocations.  Not internally serialised across multi-call
    sequences: a ctx belongs to ONE session and thread role (``lock`` is what a session holds around h2d -> launch -> d2h);
    weights uploaded through a model's ctx are immutable and may be read from any other ctx's stream."""

    def __init__(self):
        import threading
        self._h = C.c_void_p()
        check(lib().ltb_ctx_create(C.byref(self._h)))
        self.lock = threading.RLock()

    # ---- memory
    def alloc(self, shape, dtype=np.float16, zero: bool = False) -> DevTensor:
        t = DevTensor(0, shape, dtype)
        p = C.c_void_p()
        check(lib().ltb_dev_alloc(self._h, t.nbytes, int(zero), C.byref(p)))
        t.ptr = p.value
        return t

    def free(self, t: DevTensor):
        check(lib().ltb_dev_free(self._h, C.c_void_p(t.ptr)))

    def upload(self, arr: np.ndarray, dtype=None) -> DevTensor:
        arr = np.ascontiguousarray(arr, dtype=dtype)
        t = self.alloc(arr.shape, arr.dtype)
        check(lib().ltb_h2d(self._h, C.c_void_p(t.ptr), arr.ctypes.data_as(C.c_void_p), arr.nbytes, 1))
        return t

    def h2d(self, t: DevTensor, arr: np.ndarray, sync: bool = True):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= t.nbytes, (arr.nbytes, t.nbytes)
        check(lib().ltb_h2d(self._h, C.c_void_p(t.ptr), arr.ctypes.data_as(C.c_void_p), arr.nbytes, int(sync)))

    def download(self, t: DevTensor, out: Optional[np.ndarray] = None, sync: bool = True) -> np.ndarray:
        if out is None:
            out = np.empty(t.shape, t.dtype)
        check(lib().ltb_d2h(self._h, out.ctypes.data_as(C.c_void_p), C.c_void_p(t.ptr), t.nbytes, int(sync)))
        return out

    def download_slice(self, t: DevTensor) -> np.ndarray:
        """Dense copy of a channel-sliced view (pitch > C): gathers through a temporary."""
        if t.pitch == t.C and t.c_off == 0:
            return self.download(t)
        tmp = self.alloc(t.shape, t.dtype)
        self.copy_channels(t, tmp)
        out = self.download(tmp)
        self.free(tmp)
        return out

    def set_i32(self, t: DevTensor, value: int):
        check(lib().ltb_set_i32(self._h, C.c_void_p(t.ptr), int(value)))

    def sync(self):
        check(lib().ltb_ctx_sync(self._h))

    @property
    def cuda_stream(self) -> int:
        p = C.c_void_p()
        check(lib().ltb_ctx_stream(self._h, C.byref(p)))
        return p.value or 0

    @property
    def launch_count(self) -> int:
        n = C.c_longlong(0)
        check(lib().ltb_ctx_launch_count(self._h, C.byref(n)))
        return n.value

    @contextlib.contextmanager
    def capture(self):
        """with ctx.capture() as g: <ops> ; afterwards g.graph is the instantiated CUDA graph."""
        holder = type("Capture", (), {"graph": None})()
        check(lib().ltb_capture_begin(self._h))
        try:
            yield holder
        except Exception:
            h = C.c_void_p()
            lib().ltb_capture_end(self._h, C.byref(h))
            if h:
                lib().ltb_graph_destroy(h)
            raise
        h = C.c_void_p()
        check(lib().ltb_capture_end(self._h, C.byref(h)))
        holder.graph = Graph(self, h)

    # ---- ops
    def conv(self, x: DevTensor, w: "ConvWeight", out: DevTensor, *, N: int, IH: int, IW: int, OH: int, OW: int, stride=(1, 1),
             pad=(0, 0), res: Optional[DevTensor] = None, relu: bool = False, cin: Optional[int] = None, no_halo: bool = False,
             zbatch: int = 0, zdiv: int = 1, in_z=(0, 0), w_z=(0, 0), out_z=(0, 0), w_ptr: Optional[int] = None,
             ktot: Optional[int] = None, cout: Optional[int] = None, in_ptr: Optional[int] = None, out_ptr: Optional[int] = None,
             gn_stats: Optional[DevTensor] = None, gn_groups: int = 0, gn_hw: int = 0, upsample2x: bool = False):
        d = ConvOp()
        d.in_ = in_ptr if in_ptr is not None else x.ptr
        d.w = w_ptr if w_ptr is not None else w.w.ptr
        d.w_tap = (w.w_tap.ptr if (w is not None and w.w_tap is not None and w_ptr is None) else None)
        d.bias = (w.bias.ptr if (w is not None and w.bias is not None) else None)
        d.res = res.ptr if res is not None else None
        d.out = out_ptr if out_ptr is not None else out.ptr
        d.N, d.IH, d.IW = N, IH, IW
        d.ICtot, d.ic_off = x.pitch, x.c_off
        d.Cin = cin if cin is not None else w.cin
        d.OH, d.OW = OH, OW
        d.Cout = cout if cout is not None else w.cout
        d.OCtot, d.oc_off = out.pitch, out.c_off
        d.RCtot, d.rc_off = (res.pitch, res.c_off) if res is not None else (0, 0)
        d.KH, d.KW = (w.kh, w.kw) if w is not None else (1, 1)
        d.sy, d.sx = stride
        d.pad_t, d.pad_l = pad
        d.Ktot = ktot if ktot is not None else w.ktot
        d.w_koff = 0
        d.relu = int(relu)
        d.no_halo = int(no_halo)
        d.zbatch, d.zdiv = zbatch, zdiv
        d.in_zo, d.in_zi = in_z
        d.w_zo, d.w_zi = w_z
        d.out_zo, d.out_zi = out_z
        d.gn_stats = gn_stats.ptr if gn_stats is not None else None
        d.gn_groups, d.gn_hw = gn_groups, gn_hw
        if upsample2x:          # fused nearest-2x upsample + 3x3 conv: the 16-slice weights of ConvWeight.upconv()
            up = w.upconv(self)
            d.w, d.w_tap, d.Ktot, d.upsample2x = up[0].ptr, up[1].ptr, 16 * w.cin, 1
        check(lib().ltb_op_conv2d(self._h, C.byref(d)))

    def groupnorm(self, x: DevTensor, N: int, HW: int, groups: int, eps: float, gamma: DevTensor, beta: DevTensor, silu: bool,
                  out: DevTensor):
        check(lib().ltb_op_groupnorm(self._h, C.c_void_p(x.ptr), N, HW, x.C, x.pitch, x.c_off, groups, eps, C.c_void_p(gamma.ptr),
                                     C.c_void_p(beta.ptr), int(silu), C.c_void_p(out.ptr), out.pitch, out.c_off))

    def groupnorm_apply(self, x: DevTensor, N: int, HW: int, groups: int, eps: float, stats: DevTensor, gamma: DevTensor, beta: DevTensor,
                        silu: bool, out: DevTensor):
        check(lib().ltb_op_groupnorm_apply(self._h, C.c_void_p(x.ptr), N, HW, x.C, x.pitch, x.c_off, groups, eps, C.c_void_p(stats.ptr),
                                           C.c_void_p(gamma.ptr), C.c_void_p(beta.ptr), int(silu), C.c_void_p(out.ptr), out.pitch, out.c_off))

    def layernorm(self, x: DevTensor, rows: int, Cc: int, eps: float, gamma: DevTensor, beta: DevTensor, out: DevTensor):
        check(lib().ltb_op_layernorm(self._h, C.c_void_p(x.ptr), rows, Cc, eps, C.c_void_p(gamma.ptr), C.c_void_p(beta.ptr),
                                     C.c_void_p(out.ptr)))

    def softmax(self, x: DevTensor, rows: int, cols: int, valid: int, scale: float):
        check(lib().ltb_op_softmax(self._h, C.c_void_p(x.ptr), rows, cols, cols, valid, scale, C.c_void_p(x.ptr)))

    def geglu(self, h: DevTensor, rows: int, H: int, out: DevTensor):
        check(lib().ltb_op_geglu(self._h, C.c_void_p(h.ptr), rows, H, C.c_void_p(out.ptr)))

    def eltwise(self, x: DevTensor, y: Optional[DevTensor], n: int, period: int, act: int, out: DevTensor):
        check(lib().ltb_op_eltwise(self._h, C.c_void_p(x.ptr), C.c_void_p(y.ptr) if y is not None else None, n, period, act,
                                   C.c_void_p(out.ptr)))

    def upsample2x(self, x: DevTensor, N: int, H: int, W: int, out: DevTensor):
        check(lib().ltb_op_upsample2x(self._h, C.c_void_p(x.ptr), N, H, W, x.C, C.c_void_p(out.ptr)))

    def copy_channels(self, src: DevTensor, dst: DevTensor, rows: Optional[int] = None):
        check(lib().ltb_op_copy_channels(self._h, C.c_void_p(src.ptr), rows if rows is not None else src.rows, src.C, src.pitch,
                                         src.c_off, C.c_void_p(dst.ptr), dst.pitch, dst.c_off))

    def transpose_heads(self, v_ptr: int, B: int, n_keys: int, Ctot: int, heads: int, d: int, n_pad: int, vt: DevTensor):
        check(lib().ltb_op_transpose_heads(self._h, C.c_void_p(v_ptr), B, n_keys, Ctot, 0, heads, d, n_pad, C.c_void_p(vt.ptr)))

    def attention(self, q_ptr: int, q_pitch: int, k_ptr: int, kv_pitch: int, kv_rows: int, vt: DevTensor, n_pad: int, B: int, heads: int, nq: int,
                  valid: int, d: int, scale: float, out: DevTensor):
        """out = softmax(scale * Q K^T) V, one kernel (csrc/attn_fused.cu)."""
        check(lib().ltb_op_attention(self._h, C.c_void_p(q_ptr), q_pitch, C.c_void_p(k_ptr), kv_pitch, kv_rows, C.c_void_p(vt.ptr), n_pad, B,
                                     heads, nq, valid, d, scale, C.c_void_p(out.ptr), out.pitch))

    # ---- UltraLight / HuBERT ops (SURVEY 8 row f4)
    def dwconv3x3(self, x: DevTensor, N: int, IH: int, IW: int, w_tap: DevTensor, bias: DevTensor, stride: int, relu: bool, out: DevTensor):
        check(lib().ltb_op_dwconv3x3(self._h, C.c_void_p(x.ptr), N, IH, IW, x.pitch, x.c_off, x.C, C.c_void_p(w_tap.ptr), C.c_void_p(bias.ptr),
                                     stride, int(relu), C.c_void_p(out.ptr), out.pitch, out.c_off))

    def upsample_bilinear2x(self, x: DevTensor, N: int, H: int, W: int, out: DevTensor):
        check(lib().ltb_op_upsample_bilinear2x(self._h, C.c_void_p(x.ptr), N, H, W, x.pitch, x.c_off, x.C, C.c_void_p(out.ptr), out.pitch,
                                               out.c_off))

    def ul_prep(self, faces_u8: DevTensor, nf: int, d_index: DevTensor, B: int, out: DevTensor):
        check(lib().ltb_op_ul_prep(self._h, C.c_void_p(faces_u8.ptr), nf, C.c_void_p(d_index.ptr), B, C.c_void_p(out.ptr)))

    def head_sigmoid255(self, x: DevTensor, w3x32: DevTensor, b3: DevTensor, npix: int, pred: DevTensor):
        check(lib().ltb_op_head_sigmoid255(self._h, C.c_void_p(x.ptr), C.c_void_p(w3x32.ptr), C.c_void_p(b3.ptr), npix, C.c_void_p(pred.ptr)))

    def ul_paste(self, frames: DevTensor, faces: DevTensor, coords: DevTensor, pred: DevTensor, out: DevTensor, nf: int, H: int, W: int,
                 index: int, explicit_idx: int, slot0: int, count: int):
        check(lib().ltb_op_ul_paste(self._h, C.c_void_p(frames.ptr), C.c_void_p(faces.ptr), C.c_void_p(coords.ptr), C.c_void_p(pred.ptr),
                                    C.c_void_p(out.ptr), nf, H, W, index, explicit_idx, slot0, count))

    def ul_paste_region(self, faces: DevTensor, coords: DevTensor, pred: DevTensor, out: DevTensor, nf: int, rh: int, rw: int, index: int,
                        explicit_idx: int, slot0: int, count: int):
        check(lib().ltb_op_ul_paste_region(self._h, C.c_void_p(faces.ptr), C.c_void_p(coords.ptr), C.c_void_p(pred.ptr), C.c_void_p(out.ptr),
                                           nf, rh, rw, index, explicit_idx, slot0, count))

    def hubert_conv0(self, pcm: DevTensor, n: int, w: DevTensor, bias: Optional[DevTensor], Cc: int, stats: DevTensor, out: DevTensor):
        check(lib().ltb_op_hubert_conv0(self._h, C.c_void_p(pcm.ptr), n, C.c_void_p(w.ptr), C.c_void_p(bias.ptr) if bias is not None else None,
                                        Cc, C.c_void_p(stats.ptr), C.c_void_p(out.ptr)))

    def hubert_pos_conv(self, h: DevTensor, T: int, D: int, groups: int, K: int, w: DevTensor, bias: DevTensor, out: DevTensor):
        check(lib().ltb_op_hubert_pos_conv(self._h, C.c_void_p(h.ptr), T, D, groups, K, C.c_void_p(w.ptr), C.c_void_p(bias.ptr),
                                           C.c_void_p(out.ptr)))

    def hubert_slice(self, hidden: DevTensor, Tc: int, T: int, D: int, B: int, R: int, start: float, mult: float, win_l: int,
                     out_f32: Optional[DevTensor], out_nhwc: Optional[DevTensor]):
        check(lib().ltb_op_hubert_slice(self._h, C.c_void_p(hidden.ptr), Tc, T, D, B, R, float(start), float(mult), win_l,
                                        C.c_void_p(out_f32.ptr) if out_f32 is not None else None,
                                        C.c_void_p(out_nhwc.ptr) if out_nhwc is not None else None))

    def bgr_to_i420(self, frames_u8: DevTensor, N: int, H: int, W: int, out_u8: DevTensor):
        """uint8 BGR [N,H,W,3] -> planar I420 [N, H*3/2, W] (encoder hand-off; cv2.COLOR_BGR2YUV_I420 arithmetic)."""
        check(lib().ltb_op_bgr_to_i420(self._h, C.c_void_p(frames_u8.ptr), N, H, W, C.c_void_p(out_u8.ptr)))

    def stamp_pixels(self, frames_u8: DevTensor, N: int, H: int, W: int, pix_yx: DevTensor, color_bgr=(128, 128, 128)):
        """Write `color_bgr` into the pixels pix_yx (int32 (n, 2) = (y, x)) of every frame: the resident form of cv2.putText's
        thickness-1 LINE_8 rasterisation (livetalking_b200/watermark.py)."""
        n = int(pix_yx.shape[0])
        check(lib().ltb_op_stamp_pixels(self._h, C.c_void_p(frames_u8.ptr), N, H, W, C.c_void_p(pix_yx.ptr), n, int(color_bgr[0]),
                                        int(color_bgr[1]), int(color_bgr[2])))

    def vae_post(self, x: DevTensor, npix: int, out_u8: DevTensor):
        check(lib().ltb_op_vae_post(self._h, C.c_void_p(x.ptr), npix, x.pitch, C.c_void_p(out_u8.ptr)))

    def vae_pre(self, img_u8: DevTensor, N: int, H: int, W: int, half_mask: bool, out: DevTensor):
        check(lib().ltb_op_vae_pre(self._h, C.c_void_p(img_u8.ptr), N, H, W, int(half_mask), C.c_void_p(out.ptr)))

    def gather_rows(self, table: DevTensor, n: int, d_index: DevTensor, B: int, row_elems: int, out: DevTensor):
        check(lib().ltb_op_gather_rows(self._h, C.c_void_p(table.ptr), n, C.c_void_p(d_index.ptr), B, row_elems, C.c_void_p(out.ptr)))

    def w_tap_major(self, w: DevTensor, wt: DevTensor, cout: int, cin: int):
        check(lib().ltb_op_w_tap_major(self._h, C.c_void_p(w.ptr), C.c_void_p(wt.ptr), cout, cin))

    def mt_paste(self, op: MtPasteOp):
        check(lib().ltb_op_mt_paste(self._h, C.byref(op)))

    def close(self):
        if self._h:
            lib().ltb_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ConvWeight:
    """Device-resident conv / linear weights in the kernels' layout: fp16 [Cout][KH*KW*Cin] (+ tap-major copy for 3x3)."""

    def __init__(self, ctx: Ctx, w: np.ndarray, bias: Optional[np.ndarray], *, pad_cin: Optional[int] = None,
                 pad_cout: Optional[int] = None, tap_major: bool = True):
        w = np.asarray(w, dtype=np.float32)
        if w.ndim == 2:
            w = w[:, :, None, None]
        cout, cin, kh, kw = w.shape
        cin_p = pad_cin or cin
        cout_p = pad_cout or cout
        if cin_p != cin or cout_p != cout:
            wp = np.zeros((cout_p, cin_p, kh, kw), np.float32)
            wp[:cout, :cin] = w
            w = wp
        self.cout, self.cin, self.kh, self.kw = cout_p, cin_p, kh, kw
        self.ktot = kh * kw * cin_p
        packed = np.ascontiguousarray(w.transpose(0, 2, 3, 1)).reshape(cout_p, self.ktot).astype(np.float16)
        self.w = ctx.upload(packed)
        b = np.zeros(cout_p, np.float32)
        if bias is not None:
            b[:cout] = np.asarray(bias, np.float32)
        self.bias = ctx.upload(b)
        self.w_tap = None
        self._w_f32 = w if (kh == 3 and kw == 3) else None       # kept for upconv() (dropped after the first use)
        self._upconv = None
        if tap_major and kh == 3 and kw == 3 and cin_p >= 16:
            self.w_tap = ctx.alloc((9, cout_p, cin_p), np.float16)
            ctx.w_tap_major(self.w, self.w_tap, cout_p, cin_p)

    def upconv_supported(self) -> bool:
        return self.kh == 3 and self.kw == 3 and self.cout % 64 == 0 and self.cin >= 16 and self.cin % 8 == 0

    def upconv(self, ctx: "Ctx"):
        """Weights of `conv3x3(nearest_upsample_2x(x))` as four 2x2 sub-pixel convs over x (diffusers Upsample2D).

        Output pixel (2y+a, 2x+b) reads up[2y+a+dy-1, 2x+b+dx-1] = x[(2y+a+dy-1)//2, ...]: for a = 0 the kernel rows {0} fall on
        input row y-1 and {1,2} on row y; for a = 1 rows {0,1} fall on y and {2} on y+1 (same for columns).  So
        V[a,b][ry,rx] = sum of the w[dy,dx] that land on the (ry,rx)-th row/column of the 2x2 footprint — summed in fp32, then
        rounded to fp16 once.  2.25x fewer MACs than the conv on the upsampled map and no upsampled tensor.
        Returns (phase-major [Cout][16][Cin], view-major [16][Cout][Cin] in the slice order of conv_halo.cu's upconv plan)."""
        if self._upconv is None:
            w = self._w_f32                                              # (cout, cin, 3, 3) float32 (already padded)
            rows = {0: ([0], [1, 2]), 1: ([0, 1], [2])}
            V = {}
            for a in (0, 1):
                for b in (0, 1):
                    for ry in (0, 1):
                        for rx in (0, 1):
                            V[(a, b, ry, rx)] = sum(w[:, :, dy, dx] for dy in rows[a][ry] for dx in rows[b][rx])
            phase_major = np.stack([V[(a, b, ry, rx)] for a in (0, 1) for b in (0, 1) for ry in (0, 1) for rx in (0, 1)], 1)   # (cout,16,cin)
            # view-major order: (phase, ry, rx) per slice — see the stage table in conv_halo_make_plan
            p00, p01, p11, p10 = (0, 0), (0, 1), (1, 1), (1, 0)
            order = [(p00, 1, 1), (p01, 1, 0), (p11, 0, 0), (p10, 0, 1),
                     (p00, 0, 1), (p01, 0, 0), (p01, 1, 1), (p11, 0, 1),
                     (p11, 1, 0), (p10, 1, 1), (p00, 1, 0), (p10, 0, 0),
                     (p00, 0, 0), (p01, 0, 1), (p11, 1, 1), (p10, 1, 0)]
            view_major = np.stack([V[(ph[0], ph[1], ry, rx)] for ph, ry, rx in order], 0)                                       # (16,cout,cin)
            self._upconv = (ctx.upload(np.ascontiguousarray(phase_major).astype(np.float16)),
                            ctx.upload(np.ascontiguousarray(view_major).astype(np.float16)))
            self._w_f32 = None
        return self._upconv
