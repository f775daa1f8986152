"""Wav2Lip avatar plugin on the B200 engine — drop-in for avatars/wav2lip_avatar.py.

Module surface used by app.py:128-151 (unchanged): ``load_model(path)``, ``load_avatar(avatar_id)``,
``warm_up(batch_size, model, modelres)`` and the class registered as ``("avatar", "wav2lip")`` constructed with
``opt, model, avatar``.  ``LipReal`` keeps the reference class's hooks:

    inference_batch(index, audiofeat_batch) -> iterable of B per-frame results      (wav2lip_avatar.py:116-139)
    paste_back_frame(pred_frame, idx)       -> H x W x 3 uint8 BGR, fresh & writable (wav2lip_avatar.py:141-147)

By default the per-frame result is an opaque ``EngineFrame`` (the reference treats it as opaque,
base_avatar.py:374-376, 433): the whole batch is composited on the GPU right after the forward pass and copied back
once; ``paste_back_frame`` then only hands out the finished frame.  With ``opt.ltb_return_pred = True`` the plugin
returns the reference's exact data instead (float32 (B,256,256,3) predictions; paste on demand).

Frame-free avatars: ``make_avatar`` uploads the full frames only while they fit ``engine.frames_fit_device`` (a fixed share of
the device's free memory at load time).  A larger avatar keeps its frames in host RAM, as the reference does; the device then
composites only the paste rectangle, and ``paste_back_frame`` writes it into a fresh copy of ``frame_list_cycle[idx]``.  Every
mode below works with either residency and hands ``BaseAvatar`` the same frames.

Cross-session batching (``opt.ltb_cross_session = True`` or ``LTB_CROSS_SESSION=1``): the session owns no network; its
frames are slot requests to a scheduler shared by all sessions of the model (plugin/batcher.py), which packs up to
``LTB_MUX_BATCH`` (16) frames of different sessions into one forward + paste launch.  The session's own ``batch_size`` can
then be small (low latency) without under-filling the GPU.
"""
from __future__ import annotations

import glob
import os
import pickle

import numpy as np

from .. import avatar_pack, engine
from .batcher import CrossSessionBatcher
from .mel_asr import MelASR

try:
    from avatars.base_avatar import BaseAvatar            # the reference's runtime, unchanged
    from registry import register
    from utils.image import mirror_index, read_imgs
    from utils.logger import logger
except Exception as _e:  # pragma: no cover - only when imported outside LiveTalking without stubs
    raise ImportError("livetalking_b200.plugin.wav2lip_avatar must be imported inside LiveTalking (or with stubs for "
                      "avatars.base_avatar / registry / utils): " + repr(_e))


class AvatarPayload(tuple):
    """(frame_list_cycle, face_list_cycle, coord_list_cycle) as the reference returns it, plus the resident copy."""
    engine_avatar = None


class EngineFrame:
    """One composited frame of a batch, produced on the GPU; opaque to BaseAvatar."""
    __slots__ = ("frame", "idx")

    def __init__(self, frame, idx):
        self.frame, self.idx = frame, idx


class EngineRegion:
    """Frame-free form of EngineFrame: the composited paste rectangle of frame idx and its box (y1, y2, x1, x2)."""
    __slots__ = ("region", "box", "idx")

    def __init__(self, region, box, idx):
        self.region, self.box, self.idx = region, box, idx


class _RegionMux:
    """A slots session of a frame-free avatar as a CrossSessionBatcher mux: one (region, box) per request."""

    def __init__(self, session):
        self.session, self.batch = session, session.batch

    def infer_slots(self, requests):
        return self.session.infer_slots_region(requests)


def load_model(path):
    """wav2lip_avatar.py:59-70 — checkpoint["state_dict"] (optional 'module.' prefixes) -> resident engine weights."""
    import torch
    engine.set_device(int(os.environ.get("LTB_DEVICE", "0")))
    logger.info("Load checkpoint from: {}".format(path))
    checkpoint = torch.load(path, map_location="cpu")
    sd = checkpoint["state_dict"] if "state_dict" in checkpoint else checkpoint
    return engine.W2LModel.from_state_dict({k.replace("module.", ""): v for k, v in sd.items()})


def load_avatar(avatar_id):
    """wav2lip_avatar.py:72-88 — same on-disk format; additionally uploads the assets once.  A packed ``avatar.ltbav``
    (``python -m livetalking_b200.avatar_pack``) next to the image folders is preferred: one sequential read, no PNG decodes."""
    avatar_path = f"./data/avatars/{avatar_id}"
    packed = os.path.join(avatar_path, "avatar.ltbav")
    if os.path.exists(packed):
        return make_avatar(*avatar_pack.load_packed(packed).wav2lip_lists())
    with open(f"{avatar_path}/coords.pkl", "rb") as f:
        coord_list_cycle = pickle.load(f)
    key = lambda x: int(os.path.splitext(os.path.basename(x))[0])  # noqa: E731
    frame_list_cycle = read_imgs(sorted(glob.glob(os.path.join(f"{avatar_path}/full_imgs", "*.[jpJP][pnPN]*[gG]")), key=key))
    face_list_cycle = read_imgs(sorted(glob.glob(os.path.join(f"{avatar_path}/face_imgs", "*.[jpJP][pnPN]*[gG]")), key=key))
    return make_avatar(frame_list_cycle, face_list_cycle, coord_list_cycle)


def make_avatar(frame_list_cycle, face_list_cycle, coord_list_cycle, frames_resident=None) -> AvatarPayload:
    """frames_resident: None = the residency rule (engine.frames_fit_device); False forces a frame-free avatar."""
    if frames_resident is None:
        frames_resident = engine.frames_fit_device(sum(np.asarray(f).nbytes for f in frame_list_cycle))
    payload = AvatarPayload((frame_list_cycle, face_list_cycle, coord_list_cycle))
    if frames_resident:
        payload.engine_avatar = engine.W2LAvatar(face_list_cycle, frame_list_cycle, coord_list_cycle)
    else:
        payload.engine_avatar = engine.W2LAvatar(face_list_cycle, frame_list_cycle, coord_list_cycle, frames_resident=False)
    return payload


def warm_up(batch_size, model, modelres):
    """wav2lip_avatar.py:90-96 — the engine warms every session when it is created; nothing to do per model."""
    logger.info("warmup model... (engine sessions warm up at creation)")


_BATCHER_LOCK = __import__("threading").Lock()


def shared_batcher(model, eng_avatar) -> CrossSessionBatcher:
    """One scheduler per (model, frame size), or per (model, region capacity) for frame-free avatars: created by the first
    session that asks, shared by all later ones."""
    with _BATCHER_LOCK:
        table = getattr(model, "_ltb_batchers", None)
        if table is None:
            table = model._ltb_batchers = {}
        frame_free = not getattr(eng_avatar, "frames_resident", True)
        key = ("region", *eng_avatar.region_max) if frame_free else (eng_avatar.H, eng_avatar.W)
        if key not in table:
            mux = engine.W2LSession(model, eng_avatar, int(os.environ.get("LTB_MUX_BATCH", "16")), slots=True)
            table[key] = CrossSessionBatcher(_RegionMux(mux) if frame_free else mux, float(os.environ.get("LTB_MUX_WAIT_MS", "4")))
        return table[key]


@register("avatar", "wav2lip")
class LipReal(BaseAvatar):
    def __init__(self, opt, model, avatar):
        super().__init__(opt)
        self.model = model
        self.frame_list_cycle, self.face_list_cycle, self.coord_list_cycle = avatar
        eng_avatar = getattr(avatar, "engine_avatar", None)
        if eng_avatar is None:   # a plain tuple from somewhere else: upload now
            eng_avatar = engine.W2LAvatar(self.face_list_cycle, self.frame_list_cycle, self.coord_list_cycle)
        self._engine_avatar = eng_avatar
        self._frame_free = not getattr(eng_avatar, "frames_resident", True)
        self._return_pred = bool(getattr(opt, "ltb_return_pred", False))
        cross = bool(getattr(opt, "ltb_cross_session", False)) or os.environ.get("LTB_CROSS_SESSION", "0") == "1"
        self._batcher = None
        if cross and not self._return_pred:
            self._batcher = shared_batcher(model, eng_avatar)
            # feature extractor only: the forward pass of this session's frames runs in the shared cross-session batch
            self.engine_session = engine.W2LSession(model, eng_avatar, self.batch_size, opt.l, opt.r, opt.fps, mel_only=True)
        else:
            self.engine_session = engine.W2LSession(model, eng_avatar, self.batch_size, opt.l, opt.r, opt.fps)
        self.asr = MelASR(opt, self, self.engine_session)
        self.asr.warm_up()
        # page-locked output ring for the fused mode: a D2H into pageable memory runs at a few GB/s, pinned at PCIe speed.  A buffer
        # is reused after `ring` more batches; res_frame_queue holds at most 2 batches (base_avatar.py:86) plus the one being
        # produced and the one being pasted, so 4 is the minimum safe depth.
        self._ring, self._ring_pos = [], 0
        if self._batcher is None and not self._return_pred:
            shape = (self.batch_size, *(eng_avatar.region_max if self._frame_free else (eng_avatar.H, eng_avatar.W)), 3)
            try:
                self._ring = [engine.PinnedBuffer(shape, np.uint8) for _ in range(max(4, int(os.environ.get("LTB_PIN_RING", "4"))))]
            except Exception as e:   # pinned memory exhausted: fall back to pageable output buffers
                logger.warning("pinned output ring unavailable (%r): using pageable buffers", e)
                self._ring = []

    def close(self):
        """Release this session's engine objects (arena, graphs, streams, pinned ring).  The shared cross-session scheduler
        and the avatar assets belong to the model / payload and stay."""
        sess, self.engine_session = getattr(self, "engine_session", None), None
        if sess is not None:
            sess.close()
        for b in getattr(self, "_ring", []):
            b.close()
        self._ring = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _next_out(self):
        if not self._ring:
            return None
        buf = self._ring[self._ring_pos % len(self._ring)].array
        self._ring_pos += 1
        return buf

    def inference_batch(self, index, audiofeat_batch):
        mel = np.asarray(audiofeat_batch, dtype=np.float32)                      # (B, 80, 16)
        length = len(self.face_list_cycle)
        if self._batcher is not None:
            idxs = [mirror_index(length, index + i) for i in range(self.batch_size)]
            frames = self._batcher.submit([(self._engine_avatar, idxs[i], mel[i]) for i in range(self.batch_size)])
            if self._frame_free:
                return [EngineRegion(*frames[i], idxs[i]) for i in range(self.batch_size)]
            return [EngineFrame(frames[i], idxs[i]) for i in range(self.batch_size)]
        if self._return_pred:
            return self.engine_session.infer(index, mel, want_pred=True)        # float32 (B,256,256,3), as the reference
        if self._frame_free:
            regions, boxes = self.engine_session.infer_paste_region(index, mel, out=self._next_out())
            return [EngineRegion(regions[i], boxes[i], mirror_index(length, index + i)) for i in range(self.batch_size)]
        frames = self.engine_session.infer_paste(index, mel, out=self._next_out())   # (B,H,W,3) uint8: one engine call, one D2H
        return [EngineFrame(frames[i], mirror_index(length, index + i)) for i in range(self.batch_size)]

    def paste_back_frame(self, pred_frame, idx: int):
        if isinstance(pred_frame, (EngineFrame, EngineRegion)) and pred_frame.idx != idx:
            raise ValueError(f"paste_back_frame: frame was composited for idx {pred_frame.idx}, asked for {idx}")
        if isinstance(pred_frame, EngineFrame):
            return np.array(pred_frame.frame, copy=True)                          # fresh, writable, owned by Python
        if isinstance(pred_frame, EngineRegion):
            return engine.paste_region(self.frame_list_cycle[idx], pred_frame.region, pred_frame.box)
        if self._frame_free:
            region, box = self.engine_session.paste_pred_region(np.asarray(pred_frame, dtype=np.float32), idx)
            return engine.paste_region(self.frame_list_cycle[idx], region, box)
        return self.engine_session.paste_pred(np.asarray(pred_frame, dtype=np.float32), idx)
