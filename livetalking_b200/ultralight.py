"""UltraLight avatar path on the B200 engine (SURVEY §8 row f4) — replaces the per-avatar U-Net of
avatars/ultralight/unet.py (``Model(6, 'hubert')``) and the glue of ``LightReal.inference_batch`` / ``paste_back_frame``
(avatars/ultralight_avatar.py:141-184).

The network is MobileNet-style: every InvertedResidual is 1x1 conv -> depthwise 3x3 -> 1x1 conv with BatchNorm after each
(unet.py:7-37).  BatchNorm (eval) is folded into the preceding convolution at load time; the 1x1 convs (97 % of the FLOPs) and the
two dense stride-2 3x3 convs of the audio branch run on the tcgen05 implicit-GEMM kernels, the depthwise convs / bilinear
upsampling / input glue / paste-back on the HBM-bound kernels of csrc/ultralight.cu.  ``torch.cat`` never copies: producers write
straight into channel slices of the concat buffers.  One CUDA graph per (session, batch size)."""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np

from .musetalk import Builder, _Replay, _ceil16, _np
from ._capi import LtbError
from .engine import mirror_index
from .ops import ConvWeight, Ctx, DevTensor

CH = [32, 64, 128, 256, 512]          # unet.py:188
FACE, CROP, INSET = 160, 168, 4       # network input side, stored crop side, crop[4:164] (ultralight_avatar.py:148)
BN_EPS = 1e-5


def _fold(sd, conv_w: np.ndarray, conv_b: Optional[np.ndarray], bn: str):
    """conv (+bias) followed by eval BatchNorm -> (w', b'):  y = (conv(x) + b - mean) * gamma / sqrt(var + eps) + beta."""
    g, beta, mean, var = (_np(sd[f"{bn}.{k}"]) for k in ("weight", "bias", "running_mean", "running_var"))
    s = g / np.sqrt(var + BN_EPS)
    b = beta - mean * s if conv_b is None else beta + (conv_b - mean) * s
    return conv_w * s.reshape(-1, *([1] * (conv_w.ndim - 1))), b.astype(np.float32)


class _IR:
    """One InvertedResidual (unet.py:7-37) with folded BatchNorms, channel counts padded to multiples of 16."""

    def __init__(self, ctx: Ctx, sd, p: str, inp: int, oup: int, stride: int, res: bool, expand: int = 2):
        hid = inp * expand
        self.inp_p, self.hid_p, self.oup, self.stride, self.res = _ceil16(inp), _ceil16(hid), oup, stride, res
        assert oup % 16 == 0
        w1, b1 = _fold(sd, _np(sd[p + ".conv.0.weight"]), None, p + ".conv.1")
        self.pw1 = ConvWeight(ctx, w1, b1, pad_cin=self.inp_p, pad_cout=self.hid_p, tap_major=False)
        wd, bd = _fold(sd, _np(sd[p + ".conv.3.weight"]), None, p + ".conv.4")              # (hid, 1, 3, 3)
        wt = np.zeros((9, self.hid_p), np.float16)
        wt[:, :hid] = wd.reshape(hid, 9).T
        bt = np.zeros(self.hid_p, np.float32)
        bt[:hid] = bd
        self.dw_w, self.dw_b = ctx.upload(wt), ctx.upload(bt)
        w2, b2 = _fold(sd, _np(sd[p + ".conv.6.weight"]), None, p + ".conv.7")
        self.pw2 = ConvWeight(ctx, w2, b2, pad_cin=self.hid_p, tap_major=False)


class UltraLightModel:
    """Device-resident ``Model(6, 'hubert')`` built from its state_dict (``ultralight.pth``, ultralight_avatar.py:69-70)."""

    def __init__(self, ctx: Ctx, sd: Dict):
        self.ctx = ctx
        ir = lambda p, i, o, s=1, r=False: _IR(ctx, sd, p, i, o, s, r)  # noqa: E731
        dc = lambda p, i, o, s: [ir(p + ".double_conv.0", i, o, s), ir(p + ".double_conv.1", o, o, 1, True)]  # noqa: E731  (DoubleConvDW)
        a = "audio_model"
        self.a1, self.a2 = ir(a + ".conv1", 16, CH[1]), ir(a + ".conv2", CH[1], CH[2])
        self.a3 = ConvWeight(ctx, *_fold(sd, _np(sd[a + ".conv3.weight"]), _np(sd[a + ".conv3.bias"]), a + ".bn3"))
        self.a4 = ir(a + ".conv4", CH[3], CH[3], 1, True)
        self.a5 = ConvWeight(ctx, *_fold(sd, _np(sd[a + ".conv5.weight"]), _np(sd[a + ".conv5.bias"]), a + ".bn5"), tap_major=False)
        self.a6, self.a7 = ir(a + ".conv6", CH[4], CH[4], 1, True), ir(a + ".conv7", CH[4], CH[4], 1, True)
        self.fuse = dc("fuse_conv.0", CH[4] * 2, CH[4], 1) + dc("fuse_conv.1", CH[4], CH[3], 1)
        self.inc = ir("inc.inconv.0", 6, CH[0])
        self.down = [dc(f"down{i + 1}.maxpool_conv.0", CH[i], CH[i + 1], 2) for i in range(4)]
        self.up = [dc(f"up{i + 1}.conv", c_in, c_out, 1)
                   for i, (c_in, c_out) in enumerate(((CH[4], CH[3] // 2), (CH[3], CH[2] // 2), (CH[2], CH[1] // 2), (CH[1], CH[0])))]
        self.head_w = ctx.upload(_np(sd["outc.conv.weight"]).reshape(3, CH[0]).astype(np.float32))
        self.head_b = ctx.upload(_np(sd["outc.conv.bias"]).astype(np.float32))
        ctx.sync()

    # ---- emitters (ops go to the builder's ctx = the session's stream; weights are read-only)
    @staticmethod
    def _ir(b: Builder, blk: _IR, x: DevTensor, out: Optional[DevTensor] = None) -> DevTensor:
        ctx = b.ctx
        N, H, W, _ = x.shape
        rows = N * H * W
        h1 = b.new(N, H, W, blk.hid_p)
        ctx.conv(x, blk.pw1, h1, N=1, IH=1, IW=rows, OH=1, OW=rows, relu=True)
        OH, OW = (H - 1) // blk.stride + 1, (W - 1) // blk.stride + 1
        h2 = b.new(N, OH, OW, blk.hid_p)
        ctx.dwconv3x3(h1, N, H, W, blk.dw_w, blk.dw_b, blk.stride, True, h2)
        if out is None:
            out = b.new(N, OH, OW, blk.oup)
        orow = N * OH * OW
        ctx.conv(h2, blk.pw2, out, N=1, IH=1, IW=orow, OH=1, OW=orow, res=x if blk.res else None)
        return out

    def _dc(self, b: Builder, blks: List[_IR], x: DevTensor, out: Optional[DevTensor] = None) -> DevTensor:
        for i, blk in enumerate(blks):
            x = self._ir(b, blk, x, out if i == len(blks) - 1 else None)
        return x

    def emit(self, b: Builder, img16: DevTensor, audio16: DevTensor, pred: DevTensor, taps: Optional[dict] = None):
        """img16 (B,160,160,16) fp16 NHWC (6 real channels), audio16 (B,32,32,16) -> pred f32 (B,160,160,3) = sigmoid x 255.
        Model.forward, unet.py:208-226."""
        ctx = b.ctx
        B = img16.shape[0]
        view = lambda buf, c0, c: DevTensor(buf.ptr, buf.shape[:3] + (c,), pitch=buf.shape[3], c_off=c0)  # noqa: E731
        # concat buffers: [upsampled | skip] (torch.cat([x1, x2]), unet.py:88) and [x5 | audio] (unet.py:217)
        cat = [b.new(B, FACE >> i, FACE >> i, 2 * CH[i]) for i in range(4)]                  # up4..up1 inputs at 160, 80, 40, 20
        cat5 = b.new(B, 10, 10, 2 * CH[4])
        skips = [view(cat[i], CH[i], CH[i]) for i in range(4)]                              # x1..x4 live in the second half
        x = self._ir(b, self.inc, img16, skips[0])
        for i in range(3):
            x = self._dc(b, self.down[i], x, skips[i + 1])
        x5 = self._dc(b, self.down[3], x, view(cat5, 0, CH[4]))
        # audio branch, AudioConvHubert.forward (unet.py:164-181)
        a = self._ir(b, self.a2, self._ir(b, self.a1, audio16))
        a3 = b.new(B, 16, 16, CH[3])
        ctx.conv(a, self.a3, a3, N=B, IH=32, IW=32, OH=16, OW=16, stride=(2, 2), pad=(1, 1), relu=True)
        a4 = self._ir(b, self.a4, a3)
        a5 = b.new(B, 10, 10, CH[4])
        ctx.conv(a4, self.a5, a5, N=B, IH=16, IW=16, OH=10, OW=10, stride=(2, 2), pad=(3, 3), relu=True, no_halo=True)
        af = self._ir(b, self.a7, self._ir(b, self.a6, a5), view(cat5, CH[4], CH[4]))
        f = self._dc(b, self.fuse, cat5)
        if taps is not None:
            taps.update(x5=x5, audio=af, fuse=f)
        # Up.forward x 4 (unet.py:81-90): sizes are exact doubles, so the F.pad is a no-op
        for i in range(4):
            lvl = 3 - i
            H = FACE >> (lvl + 1)
            ctx.upsample_bilinear2x(f, B, H, H, view(cat[lvl], 0, CH[lvl]))
            f = self._dc(b, self.up[i], cat[lvl])
            if taps is not None:
                taps[f"u{i + 1}"] = f
        ctx.head_sigmoid255(f, self.head_w, self.head_b, B * FACE * FACE, pred)
        return pred


class UltraLightAvatar:
    """Avatar assets resident in HBM (replaces load_avatar's lists, ultralight_avatar.py:63-82): full frames, 168x168 face crops,
    bbox (x1,y1,x2,y2) — and, as in the reference, the avatar's OWN network (``ultralight.pth`` lives in the avatar directory).

    frames_resident=False: a frame-free avatar — crops and boxes only (``frames`` is None); sessions composite the bbox rectangle
    (the *_region methods) and the host writes it into a copy of its own frame (engine.paste_region)."""

    def __init__(self, ctx: Ctx, model: UltraLightModel, frames, faces, coords, frames_resident: bool = True):
        self.frames_resident = bool(frames_resident)
        if self.frames_resident:
            frames = np.ascontiguousarray(np.asarray(frames), np.uint8)
            self.n, self.H, self.W = frames.shape[0], frames.shape[1], frames.shape[2]
        else:
            self.n, (self.H, self.W) = len(frames), np.shape(frames[0])[:2]
        faces = np.ascontiguousarray(np.asarray(faces), np.uint8)
        if faces.shape != (self.n, CROP, CROP, 3):
            raise ValueError(f"UltraLight face crops must be ({self.n},{CROP},{CROP},3) uint8, got {faces.shape}")
        self.coords_host = np.ascontiguousarray(np.asarray(coords), np.int32).reshape(self.n, 4)
        for x1, y1, x2, y2 in self.coords_host:
            if not (0 <= x1 < x2 <= self.W and 0 <= y1 < y2 <= self.H):
                raise ValueError("avatar bbox outside the frame")
        c = self.coords_host
        self.region_max = (int((c[:, 3] - c[:, 1]).max()), int((c[:, 2] - c[:, 0]).max()))
        self.ctx, self.model = ctx, model
        self.frames = ctx.upload(frames) if self.frames_resident else None
        self.faces, self.coords = ctx.upload(faces), ctx.upload(self.coords_host)

    def box(self, idx: int):
        """(y1, y2, x1, x2) of frame idx: the order engine.paste_region takes."""
        x1, y1, x2, y2 = (int(v) for v in self.coords_host[idx])
        return (y1, y2, x1, x2)


class UltraLightSession:
    """One avatar stream at a fixed batch size: captured prep + U-Net + head graph, paste-back buffers."""

    def __init__(self, avatar: UltraLightAvatar, batch: int, keep_taps: bool = False, ctx: Optional[Ctx] = None):
        self.avatar, self.B = avatar, int(batch)
        self._own_ctx = ctx is None
        ctx = self.ctx = Ctx() if ctx is None else ctx
        B = self.B
        self.builder = Builder(ctx)
        self.d_index = ctx.alloc((4,), np.int32, zero=True)
        self.audio16 = ctx.alloc((B, 32, 32, 16), np.float16, zero=True)           # NHWC view of audiofeat.reshape(16, 32, 32)
        self.img16 = ctx.alloc((B, FACE, FACE, 16), np.float16, zero=True)
        self.pred = ctx.alloc((B, FACE, FACE, 3), np.float32, zero=True)
        out_hw = (avatar.H, avatar.W) if avatar.frames_resident else avatar.region_max
        self.frames_out = ctx.alloc((B, *out_hw, 3), np.uint8, zero=True)
        self.taps = {} if keep_taps else None
        self._paste_ctx = None

        def emit():
            ctx.ul_prep(avatar.faces, avatar.n, self.d_index, B, self.img16)
            avatar.model.emit(self.builder, self.img16, self.audio16, self.pred, self.taps)

        emit()
        ctx.sync()
        temps, self.builder.temps = self.builder.temps, []
        self.builder.new = _Replay(temps)
        with ctx.capture() as cap:
            emit()
        self.graph = cap.graph

    # ---- LightReal.inference_batch (ultralight_avatar.py:141-169)
    def infer_async(self, index: int, audio_feats: Optional[np.ndarray] = None):
        """audio_feats: (B, 16, 1024) float (the HubertASR windows) or None when audio16 is already resident."""
        if audio_feats is not None:
            a = np.asarray(audio_feats, np.float32)
            if a.shape != (self.B, 16, 1024):
                raise ValueError(f"audio features must be ({self.B},16,1024), got {a.shape}")
            self.ctx.h2d(self.audio16, np.ascontiguousarray(a.transpose(0, 2, 1)).astype(np.float16), sync=False)
        self.ctx.set_i32(self.d_index, index)
        self.graph.launch()

    def infer(self, index: int, audio_feats: Optional[np.ndarray] = None, want_pred: bool = True):
        with self.ctx.lock:
            self.infer_async(index, audio_feats)
            if want_pred:
                return self.ctx.download(self.pred)              # float32 (B,160,160,3) = pred * 255, as the reference returns
            self.ctx.sync()
            return None

    # ---- LightReal.paste_back_frame (ultralight_avatar.py:171-184)
    def _need_frames(self, what: str):
        if not self.avatar.frames_resident:
            raise LtbError(f"{what}: the avatar was created frame-free (frames_resident=False); use the *_region methods")

    def paste_batch_async(self, index: int):
        a = self.avatar
        self._need_frames("paste_batch")
        self.ctx.ul_paste(a.frames, a.faces, a.coords, self.pred, self.frames_out, a.n, a.H, a.W, index, -1, 0, self.B)

    def paste_batch(self, index: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        with self.ctx.lock:
            self.paste_batch_async(index)
            return self.ctx.download(self.frames_out, out)

    def infer_paste(self, index: int, audio_feats: Optional[np.ndarray] = None, out: Optional[np.ndarray] = None) -> np.ndarray:
        """inference_batch + B x paste_back_frame as one engine round: (B, H, W, 3) uint8 composited frames."""
        self._need_frames("infer_paste")
        with self.ctx.lock:
            self.infer_async(index, audio_feats)
            self.paste_batch_async(index)
            return self.ctx.download(self.frames_out, out)

    def paste_pred(self, pred_frame: np.ndarray, idx: int) -> np.ndarray:
        """paste_back_frame for a host prediction (160,160,3) — the reference's exact argument; own small ctx (process_frames thread)."""
        self._need_frames("paste_pred")
        a = self.avatar
        pc, p = self._paste_scratch(pred_frame, idx, "paste_pred")
        with pc.lock:
            pc.h2d(self._pred_scratch, p, sync=False)
            pc.ul_paste(a.frames, a.faces, a.coords, self._pred_scratch, self._paste_out, a.n, a.H, a.W, 0, idx, 0, 1)
            return pc.download(self._paste_out)

    def _paste_scratch(self, pred_frame, idx: int, what: str):
        a = self.avatar
        p = np.ascontiguousarray(pred_frame, np.float32)
        if p.shape != (FACE, FACE, 3):
            raise ValueError(f"{what}: prediction must be ({FACE},{FACE},3), got {p.shape}")
        if not 0 <= idx < a.n:
            raise ValueError(f"{what}: idx out of range")
        if self._paste_ctx is None:
            self._paste_ctx = Ctx()
            self._pred_scratch = self._paste_ctx.alloc((1, FACE, FACE, 3), np.float32)
            self._paste_out = self._paste_ctx.alloc((a.H, a.W, 3) if a.frames_resident else (*a.region_max, 3), np.uint8)
        return self._paste_ctx, p

    # ---- region forms (frame-free avatars): rectangles + their boxes (y1, y2, x1, x2); engine.paste_region does the host half
    def infer_paste_region(self, index: int, audio_feats: Optional[np.ndarray] = None, out: Optional[np.ndarray] = None):
        """infer_paste with region output: -> (regions uint8 (B, rh_max, rw_max, 3), boxes); slot i's rectangle is
        regions[i, :y2-y1, :x2-x1] of frame mirror_index(n, index + i)."""
        a = self.avatar
        rh, rw = a.region_max
        packed = DevTensor(self.frames_out.ptr, (self.B, rh, rw, 3), np.uint8)     # fits: every box lies inside the frame
        with self.ctx.lock:
            self.infer_async(index, audio_feats)
            self.ctx.ul_paste_region(a.faces, a.coords, self.pred, packed, a.n, rh, rw, index, -1, 0, self.B)
            regions = self.ctx.download(packed, out)
        return regions, [a.box(mirror_index(a.n, index + i)) for i in range(self.B)]

    def paste_pred_region(self, pred_frame: np.ndarray, idx: int):
        """paste_pred with region output: -> (region uint8 (y2-y1, x2-x1, 3), box (y1, y2, x1, x2))."""
        a = self.avatar
        pc, p = self._paste_scratch(pred_frame, idx, "paste_pred_region")
        box = a.box(idx)
        h, w = box[1] - box[0], box[3] - box[2]
        region = DevTensor(self._paste_out.ptr, (h, w, 3), np.uint8)
        with pc.lock:
            pc.h2d(self._pred_scratch, p, sync=False)
            pc.ul_paste_region(a.faces, a.coords, self._pred_scratch, region, a.n, h, w, 0, idx, 0, 1)
            return pc.download(region), box

    def step_async(self, index: int):
        self._need_frames("step_async")
        self.infer_async(index, None)
        self.paste_batch_async(index)

    def close(self):
        if getattr(self, "graph", None) is not None:
            self.graph.close()
            self.graph = None
        if self._paste_ctx is not None:
            self._paste_ctx.close()
            self._paste_ctx = None
        if self._own_ctx and self.ctx is not None:
            self.ctx.close()
        self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def unet_gflop_per_frame() -> float:
    """Algorithmic GFLOP (2 x MAC) of one Model(6,'hubert') forward at 160x160 (real channel counts, no padding)."""
    fl = 0.0

    def ir(inp, oup, H, s=1):
        nonlocal fl
        hid, O = 2 * inp, H // s
        fl += 2.0 * H * H * inp * hid + 2.0 * O * O * 9 * hid + 2.0 * O * O * hid * oup
        return O

    def dc(inp, oup, H, s):
        O = ir(inp, oup, H, s)
        return ir(oup, oup, O)

    ir(6, CH[0], 160)
    H = 160
    for i in range(4):
        H = dc(CH[i], CH[i + 1], H, 2)
    ir(16, CH[1], 32), ir(CH[1], CH[2], 32)
    fl += 2.0 * 16 * 16 * 9 * CH[2] * CH[3]
    ir(CH[3], CH[3], 16)
    fl += 2.0 * 10 * 10 * 9 * CH[3] * CH[4]
    ir(CH[4], CH[4], 10), ir(CH[4], CH[4], 10)
    dc(2 * CH[4], CH[4], 10, 1), dc(CH[4], CH[3], 10, 1)
    for i, (ci, co) in enumerate(((CH[4], CH[3] // 2), (CH[3], CH[2] // 2), (CH[2], CH[1] // 2), (CH[1], CH[0]))):
        dc(ci, co, 20 << i, 1)
    fl += 2.0 * 160 * 160 * CH[0] * 3
    return fl / 1e9
