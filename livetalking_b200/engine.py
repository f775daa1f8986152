"""Python handles over the C ABI (include/ltb200.h): model / avatar / session objects holding opaque
engine pointers.  numpy arrays in, numpy arrays out; all device memory is owned by libltb200."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _capi
from ._capi import LtbError, check, lib  # noqa: F401


def set_device(device: int) -> None:
    check(lib().ltb_set_device(int(device)))


def device_count() -> int:
    n = C.c_int(0)
    check(lib().ltb_device_count(C.byref(n)))
    return n.value


def mem_get_info() -> tuple:
    """(free, total) bytes of the current device (cudaMemGetInfo)."""
    free, total = C.c_size_t(0), C.c_size_t(0)
    check(lib().ltb_mem_get_info(C.byref(free), C.byref(total)))
    return free.value, total.value


# Share of the device's free memory (at load time) that an avatar's full frames may take.  Above it an avatar is created
# frame-free: the frames stay in host RAM, as the reference keeps them, and the device composites only the paste rectangle.
FRAMES_DEVICE_SHARE = 0.25
# Frames below this size are uploaded without asking the device: a session's own activation arena is ~0.9 GB, so on a device
# that can run one at all, 64 MiB of frames cannot decide between the two residencies.
FRAMES_ALWAYS_RESIDENT_BYTES = 64 << 20


def frames_fit_device(frames_nbytes: int) -> bool:
    """The residency rule of the avatar plugins: True = upload the full frames, False = create the avatar frame-free."""
    if frames_nbytes <= FRAMES_ALWAYS_RESIDENT_BYTES:
        return True
    free, _total = mem_get_info()
    return frames_nbytes <= FRAMES_DEVICE_SHARE * free


def paste_region(frame: np.ndarray, region: np.ndarray, box) -> np.ndarray:
    """Host half of a frame-free composite: a fresh, writable copy of `frame` with `region` written at box = (y1, y2, x1, x2)."""
    y1, y2, x1, x2 = (int(v) for v in box)
    out = np.array(frame, copy=True)
    out[y1:y2, x1:x2] = region[:y2 - y1, :x2 - x1]
    return out


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _carr(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


class W2LModel:
    """wav2lip256 weights resident on the current device (replaces load_model, wav2lip_avatar.py:59-70)."""

    def __init__(self, blob: Optional[bytes] = None, *, device_ptr: int = 0, nbytes: int = 0, keepalive=None):
        self._h = C.c_void_p()
        self._keep = keepalive
        if blob is not None:
            buf = (C.c_char * len(blob)).from_buffer_copy(blob)
            check(lib().ltb_w2l_model_create(C.cast(buf, C.c_void_p), len(blob), C.byref(self._h)))
        else:
            check(lib().ltb_w2l_model_create_from_device(C.c_void_p(device_ptr), nbytes, C.byref(self._h)))

    @classmethod
    def from_state_dict(cls, sd) -> "W2LModel":
        from .w2l_pack import pack_state_dict
        return cls(pack_state_dict(sd))

    def close(self):
        if self._h:
            lib().ltb_w2l_model_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class W2LAvatar:
    """Avatar assets resident in HBM (replaces load_avatar's host lists, wav2lip_avatar.py:72-88).

    frames_resident=False: a frame-free avatar.  Only faces and coords go to the device; `frames` stays the caller's host
    sequence (not copied), and sessions composite only the paste rectangle (the *_region methods), which the host writes into a
    copy of its own frame (paste_region)."""

    def __init__(self, faces: Sequence[np.ndarray], frames: Sequence[np.ndarray], coords: Sequence[Sequence[int]],
                 frames_resident: bool = True):
        self.faces = _carr(np.asarray(faces), np.uint8)
        self.coords = _carr(np.asarray(coords), np.int32)
        self.frames_resident = bool(frames_resident)
        n = self.faces.shape[0]
        if self.faces.shape != (n, 256, 256, 3):
            raise ValueError(f"faces must be (n,256,256,3) uint8, got {self.faces.shape}")
        if self.frames_resident:
            self.frames = _carr(np.asarray(frames), np.uint8)
            shape = self.frames.shape
        else:
            self.frames = frames
            shapes = {np.shape(f) for f in frames}
            shape = (len(frames), *shapes.pop()) if len(shapes) == 1 else (len(frames), "mixed")
        if len(shape) != 4 or shape[0] != n or shape[3] != 3:
            raise ValueError(f"frames must be (n,H,W,3) uint8, got {shape}")
        if self.coords.shape != (n, 4):
            raise ValueError(f"coords must be (n,4), got {self.coords.shape}")
        self.n, self.H, self.W = n, shape[1], shape[2]
        self._h = C.c_void_p()
        check(lib().ltb_w2l_avatar_create(_ptr(self.faces), _ptr(self.frames) if self.frames_resident else None, _ptr(self.coords),
                                          n, self.H, self.W, C.byref(self._h)))
        rh, rw = C.c_int(0), C.c_int(0)
        check(lib().ltb_w2l_avatar_region_max(self._h, C.byref(rh), C.byref(rw)))
        self.region_max = (rh.value, rw.value)

    def close(self):
        if self._h:
            lib().ltb_w2l_avatar_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def mirror_index(size: int, index: int) -> int:
    """utils/image.py:26-32 — the frame a batch slot composites (as the engine's kernels compute it)."""
    turn, res = divmod(index, size)
    return res if turn % 2 == 0 else size - res - 1


class PinnedBuffer:
    """Page-locked host memory exposed as a numpy array (e2e path: async H2D / D2H)."""

    def __init__(self, shape, dtype):
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self._p = C.c_void_p()
        check(lib().ltb_host_alloc(self.nbytes, C.byref(self._p)))
        buf = (C.c_char * self.nbytes).from_address(self._p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype).reshape(self.shape)

    def close(self):
        if self._p:
            self.array = None
            lib().ltb_host_free(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class W2LSession:
    """One avatar stream: activation arena + stream + layer plan for a fixed batch size."""

    def __init__(self, model: W2LModel, avatar: W2LAvatar, batch: int, stride_left: int = 10, stride_right: int = 10,
                 fps: int = 25, keep_layers: bool = False, no_graph: bool = False, no_halo: bool = False, no_pdl: bool = False,
                 slots: bool = False, mel_only: bool = False):
        self.model, self.avatar = model, avatar
        self.batch, self.l, self.r, self.fps = int(batch), int(stride_left), int(stride_right), int(fps)
        flags = ((_capi.LTB_SESSION_KEEP_LAYERS if keep_layers else 0) | (_capi.LTB_SESSION_NO_GRAPH if no_graph else 0) |
                 (_capi.LTB_SESSION_NO_HALO if no_halo else 0) | (_capi.LTB_SESSION_NO_PDL if no_pdl else 0) |
                 (_capi.LTB_SESSION_SLOTS if slots else 0) | (_capi.LTB_SESSION_MEL_ONLY if mel_only else 0))
        self._h = C.c_void_p()
        check(lib().ltb_w2l_session_create(model._h, avatar._h, self.batch, self.l, self.r, self.fps, flags,
                                           C.byref(self._h)))

    # --- mel.py:46-63 + audio.py:45-51
    def mel_step(self, pcm: np.ndarray, want_output: bool = True) -> Optional[np.ndarray]:
        pcm = _carr(pcm, np.float32).reshape(-1)
        out = np.empty((self.batch, 80, 16), np.float32) if want_output else None
        check(lib().ltb_w2l_mel_step(self._h, _ptr(pcm), pcm.size, _ptr(out)))
        return out

    def set_pcm(self, pcm: np.ndarray) -> None:
        """Upload the PCM window read by the device-resident step (mel_resident / step_async)."""
        pcm = _carr(pcm, np.float32).reshape(-1)
        check(lib().ltb_w2l_set_pcm(self._h, _ptr(pcm), pcm.size))

    # --- wav2lip_avatar.py:116-139
    def infer(self, index: int, mel: Optional[np.ndarray] = None, want_pred: bool = True) -> Optional[np.ndarray]:
        if mel is not None:
            mel = _carr(mel, np.float32)
            if mel.size != self.batch * 80 * 16:
                raise ValueError(f"mel must hold {self.batch}x80x16 values, got shape {mel.shape}")
        out = np.empty((self.batch, 256, 256, 3), np.float32) if want_pred else None
        check(lib().ltb_w2l_infer(self._h, int(index), _ptr(mel), _ptr(out)))
        return out

    # --- wav2lip_avatar.py:141-147
    def paste(self, slot: int, idx: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        if out is None:
            out = np.empty((self.avatar.H, self.avatar.W, 3), np.uint8)
        check(lib().ltb_w2l_paste(self._h, int(slot), int(idx), _ptr(out)))
        return out

    def paste_pred(self, pred: np.ndarray, idx: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        """paste_back_frame for a host-side prediction (float32 [256,256,3], as inference_batch returns)."""
        pred = _carr(pred, np.float32)
        if pred.shape != (256, 256, 3):
            raise ValueError(f"pred must be (256,256,3), got {pred.shape}")
        if out is None:
            out = np.empty((self.avatar.H, self.avatar.W, 3), np.uint8)
        check(lib().ltb_w2l_paste_pred(self._h, _ptr(pred), int(idx), _ptr(out)))
        return out

    def paste_batch(self, index: int, out: Optional[np.ndarray] = None, to_host: bool = True) -> Optional[np.ndarray]:
        if to_host and out is None:
            out = np.empty((self.batch, self.avatar.H, self.avatar.W, 3), np.uint8)
        check(lib().ltb_w2l_paste_batch(self._h, int(index), _ptr(out) if to_host else None))
        return out

    def infer_paste(self, index: int, mel: np.ndarray, out: Optional[np.ndarray] = None) -> np.ndarray:
        """inference_batch in fused mode: mel windows in, `batch` composited frames out (one engine call)."""
        mel = _carr(mel, np.float32)
        if mel.size != self.batch * 80 * 16:
            raise ValueError(f"mel must hold {self.batch}x80x16 values, got shape {mel.shape}")
        if out is None:
            out = np.empty((self.batch, self.avatar.H, self.avatar.W, 3), np.uint8)
        check(lib().ltb_w2l_infer_paste(self._h, int(index), _ptr(mel), _ptr(out)))
        return out

    def infer_slots(self, requests, out: Optional[np.ndarray] = None) -> np.ndarray:
        """Cross-session batch: requests = [(W2LAvatar, frame_idx, mel (80,16) float32), ...] (1..batch of them, any mix of
        avatars of this session's frame size) -> composited frames uint8 (n, H, W, 3).  One forward + paste launch."""
        n = len(requests)
        arr = (_capi.W2LSlot * n)()
        keep = []
        for i, (av, idx, mel) in enumerate(requests):
            m = _carr(mel, np.float32)
            if m.size != 1280:
                raise ValueError(f"slot {i}: mel window must be (80,16), got {m.shape}")
            keep.append(m)
            arr[i].avatar, arr[i].idx, arr[i].mel = av._h, int(idx), m.ctypes.data_as(C.c_void_p)
        if out is None:
            out = np.empty((n, self.avatar.H, self.avatar.W, 3), np.uint8)
        check(lib().ltb_w2l_infer_slots(self._h, arr, n, _ptr(out)))
        return out

    # --- region forms (frame-free avatars): rectangles + their boxes; engine.paste_region puts one into a frame copy
    def infer_paste_region(self, index: int, mel: np.ndarray, out: Optional[np.ndarray] = None):
        """infer_paste for a frame-free avatar: -> (regions uint8 (batch, rh_max, rw_max, 3), boxes int32 (batch, 4)); slot i's
        rectangle is regions[i, :y2-y1, :x2-x1] of boxes[i] = (y1, y2, x1, x2) of frame mirror_index(n, index + i)."""
        mel = _carr(mel, np.float32)
        if mel.size != self.batch * 80 * 16:
            raise ValueError(f"mel must hold {self.batch}x80x16 values, got shape {mel.shape}")
        rh, rw = self.avatar.region_max
        if out is None:
            out = np.empty((self.batch, rh, rw, 3), np.uint8)
        check(lib().ltb_w2l_infer_paste_region(self._h, int(index), _ptr(mel), _ptr(out)))
        n = self.avatar.n
        boxes = self.avatar.coords[[mirror_index(n, index + i) for i in range(self.batch)]]
        return out, boxes

    def infer_slots_region(self, requests, out: Optional[np.ndarray] = None):
        """infer_slots with region output: -> [(region view (h, w, 3), box (y1, y2, x1, x2)), ...], one per request.  Slot avatars
        may be frame-free and of any frame size; every box must fit this session's avatar's region_max."""
        n = len(requests)
        arr = (_capi.W2LSlot * n)()
        keep = []
        for i, (av, idx, mel) in enumerate(requests):
            m = _carr(mel, np.float32)
            if m.size != 1280:
                raise ValueError(f"slot {i}: mel window must be (80,16), got {m.shape}")
            keep.append(m)
            arr[i].avatar, arr[i].idx, arr[i].mel = av._h, int(idx), m.ctypes.data_as(C.c_void_p)
        rh, rw = self.avatar.region_max
        if out is None:
            out = np.empty((n, rh, rw, 3), np.uint8)
        check(lib().ltb_w2l_infer_slots_region(self._h, arr, n, _ptr(out)))
        res = []
        for i, (av, idx, _m) in enumerate(requests):
            box = av.coords[int(idx)]
            res.append((out[i, :box[1] - box[0], :box[3] - box[2]], box))
        return res

    def paste_pred_region(self, pred: np.ndarray, idx: int):
        """paste_pred for a frame-free avatar: -> (region uint8 (y2-y1, x2-x1, 3), box (y1, y2, x1, x2)) of frame idx."""
        pred = _carr(pred, np.float32)
        if pred.shape != (256, 256, 3):
            raise ValueError(f"pred must be (256,256,3), got {pred.shape}")
        if not 0 <= int(idx) < self.avatar.n:
            raise ValueError(f"idx {idx} out of range")
        box = self.avatar.coords[int(idx)]
        out = np.empty((box[1] - box[0], box[3] - box[2], 3), np.uint8)
        check(lib().ltb_w2l_paste_pred_region(self._h, _ptr(pred), int(idx), _ptr(out)))
        return out, box

    def mel_resident(self) -> None:
        check(lib().ltb_w2l_mel_resident(self._h))

    def profile_ops(self, index: int = 0):
        """One eager profiling pass: (ms, flops, kinds) per op of the forward plan."""
        n = C.c_int(0)
        check(lib().ltb_w2l_profile_ops(self._h, int(index), 0, C.byref(n), None, None, None))
        ms = np.zeros(n.value, np.float32)
        fl = np.zeros(n.value, np.float64)
        kinds = np.zeros(n.value, np.int32)
        check(lib().ltb_w2l_profile_ops(self._h, int(index), n.value, C.byref(n), _ptr(ms), _ptr(fl), _ptr(kinds)))
        return ms, fl, kinds

    def step_async(self, index: int) -> None:
        check(lib().ltb_w2l_step_async(self._h, int(index)))

    def forward_async(self, index: int) -> None:
        """U-Net forward only (no mel, no paste-back), enqueued without synchronising."""
        check(lib().ltb_w2l_forward_async(self._h, int(index)))

    def step_e2e_async(self, index: int, pcm_pinned: np.ndarray, frames_pinned: np.ndarray) -> None:
        """Pipelined host-to-host step (pinned buffers): H2D PCM -> mel -> forward -> paste -> D2H frames on a copy stream."""
        check(lib().ltb_w2l_step_e2e_async(self._h, int(index), _ptr(pcm_pinned), int(pcm_pinned.size), _ptr(frames_pinned)))

    def e2e_acquire(self) -> None:
        """Wait until the host buffers of the step issued two calls ago are free again."""
        check(lib().ltb_w2l_e2e_acquire(self._h))

    def sync(self) -> None:
        check(lib().ltb_w2l_sync(self._h))

    @property
    def cuda_stream(self) -> int:
        p = C.c_void_p()
        check(lib().ltb_w2l_stream(self._h, C.byref(p)))
        return p.value or 0

    @property
    def launch_count(self) -> int:
        n = C.c_longlong(0)
        check(lib().ltb_w2l_launch_count(self._h, C.byref(n)))
        return n.value

    # --- debug
    def layer_output(self, layer: int) -> np.ndarray:
        H, W, Cc = C.c_int(), C.c_int(), C.c_int()
        check(lib().ltb_w2l_layer_shape(self._h, layer, C.byref(H), C.byref(W), C.byref(Cc)))
        out = np.empty((self.batch, H.value, W.value, Cc.value), np.float16)
        check(lib().ltb_w2l_layer_read(self._h, layer, _ptr(out), out.nbytes))
        return out

    def close(self):
        if self._h:
            lib().ltb_w2l_session_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def conv2d_f16(x_nhwc: np.ndarray, w: np.ndarray, bias: np.ndarray, *, stride=(1, 1), pad: int = 0, transposed: bool = False,
               relu: bool = True, res: Optional[np.ndarray] = None, force_path: int = 0, reps: int = 0):
    """Stand-alone tensor-core conv (test hook).  x: (N,H,W,Cin) fp16; w: PyTorch layout float32.
    reps > 0: also time `reps` back-to-back launches -> (out, ms_per_launch)."""
    x = _carr(x_nhwc, np.float16)
    w = _carr(w, np.float32)
    bias = _carr(bias, np.float32)
    N, IH, IW, Cin = x.shape
    if transposed:
        Cout, KH, KW = w.shape[1], w.shape[2], w.shape[3]
        OH, OW = IH * 2, IW * 2
    else:
        Cout, KH, KW = w.shape[0], w.shape[2], w.shape[3]
        OH = (IH + 2 * pad - KH) // stride[0] + 1
        OW = (IW + 2 * pad - KW) // stride[1] + 1
    d = _capi.ConvDesc(N, IH, IW, Cin, Cout, KH, KW, stride[0], stride[1], pad, int(transposed), int(relu),
                       int(res is not None), force_path)
    out = np.empty((N, OH, OW, Cout), np.float16)
    if res is not None:
        res = _carr(res, np.float16)
        assert res.shape == out.shape
    if reps > 0:
        ms = C.c_float(0.0)
        check(lib().ltb_conv2d_f16_timed(C.byref(d), _ptr(x), _ptr(w), _ptr(bias), _ptr(res), _ptr(out), int(reps), C.byref(ms)))
        return out, ms.value
    check(lib().ltb_conv2d_f16(C.byref(d), _ptr(x), _ptr(w), _ptr(bias), _ptr(res), _ptr(out)))
    return out
