"""UltraLight avatar plugin on the B200 engine — drop-in for avatars/ultralight_avatar.py (SURVEY §8 row f4).

Module surface used by app.py (unchanged): ``load_model(opt)``, ``load_avatar(avatar_id)``, ``warm_up(batch_size, avatar, modelres)``
and the class registered as ``("avatar", "ultralight")``.  ``LightReal`` keeps the reference hooks:

    inference_batch(index, audiofeat_batch) -> B predictions                               (ultralight_avatar.py:141-169)
    paste_back_frame(pred_frame, idx)       -> H x W x 3 uint8 BGR, fresh and writable    (ultralight_avatar.py:171-184)

Default (fused) mode: ``inference_batch`` runs prep + U-Net + paste-back on the device and returns B ``EngineFrame`` tokens that
already hold the composited frames; ``paste_back_frame`` hands the matching one out.  ``opt.ltb_return_pred = True`` restores the
reference's exact data flow (float32 (B,160,160,3) predictions x 255, pasted per frame from the host).

Frame-free avatars: ``make_avatar`` uploads the full frames only while they fit ``engine.frames_fit_device``; otherwise the device
holds the crops and boxes only, composites just the bbox rectangle, and ``paste_back_frame`` writes it into a fresh copy of
``frame_list_cycle[idx]``.  Both modes work with either residency and hand ``BaseAvatar`` the same frames."""
from __future__ import annotations

import glob
import os
import pickle

import numpy as np

from .. import engine
from ..hubert import HubertEncoder, HubertFeatures
from ..ops import Ctx
from ..ultralight import FACE, UltraLightAvatar, UltraLightModel, UltraLightSession
from .hubert_asr import HubertASR

try:
    from avatars.base_avatar import BaseAvatar
    from registry import register
    from utils.image import mirror_index, read_imgs
    from utils.logger import logger
except Exception as _e:  # pragma: no cover
    raise ImportError("livetalking_b200.plugin.ultralight_avatar must be imported inside LiveTalking (or with stubs): " + repr(_e))


class EngineFrame:
    """A composited frame produced by the fused inference_batch, tagged with the avatar frame index it was pasted into."""
    __slots__ = ("frame", "idx")

    def __init__(self, frame, idx):
        self.frame, self.idx = frame, idx


class EngineRegion:
    """Frame-free form of EngineFrame: the composited bbox rectangle of frame idx and its box (y1, y2, x1, x2)."""
    __slots__ = ("region", "box", "idx")

    def __init__(self, region, box, idx):
        self.region, self.box, self.idx = region, box, idx


class EngineAudio:
    """What load_model() returns as ``audio_processor``: the resident HuBERT encoder; sessions build their own extractor graph."""

    def __init__(self, ctx, encoder):
        self.ctx, self.encoder = ctx, encoder


class AvatarPayload(tuple):
    engine_avatar = None


def make_model(hubert_sd) -> tuple:
    engine.set_device(int(os.environ.get("LTB_DEVICE", "0")))
    ctx = Ctx()
    return EngineAudio(ctx, HubertEncoder(ctx, hubert_sd)), None


def load_model(opt=None, hubert_dir="./models/hubert-large-ls960-ft"):
    """ultralight_avatar.py:58-61 / audio2feature.py:7-12: the same HuBERT checkpoint, made resident on the engine."""
    from transformers import HubertModel
    return make_model(HubertModel.from_pretrained(hubert_dir).state_dict())


def make_avatar(unet_sd, frames, faces, coords, ctx: Ctx = None, frames_resident=None) -> AvatarPayload:
    """frames_resident: None = the residency rule (engine.frames_fit_device); False forces a frame-free avatar."""
    if frames_resident is None:
        frames_resident = engine.frames_fit_device(sum(np.asarray(f).nbytes for f in frames))
    ctx = ctx or Ctx()
    net = UltraLightModel(ctx, unet_sd)
    payload = AvatarPayload((net, frames, faces, coords))
    if frames_resident:
        payload.engine_avatar = UltraLightAvatar(ctx, net, frames, faces, coords)
    else:
        payload.engine_avatar = UltraLightAvatar(ctx, net, frames, faces, coords, frames_resident=False)
    return payload


def load_avatar(avatar_id):
    """ultralight_avatar.py:63-82 — same on-disk format (full_imgs/, face_imgs/, coords.pkl, ultralight.pth)."""
    import torch
    p = f"./data/avatars/{avatar_id}"
    engine.set_device(int(os.environ.get("LTB_DEVICE", "0")))
    sd = torch.load(f"{p}/ultralight.pth", map_location="cpu")
    if os.path.exists(f"{p}/avatar.ltbav"):            # packed form (`python -m livetalking_b200.avatar_pack <dir>`: the wav2lip layout —
        from .. import avatar_pack                     # full_imgs / face_imgs / coords.pkl — holds 168x168 crops just as well)
        return make_avatar(sd, *avatar_pack.load_packed(f"{p}/avatar.ltbav").wav2lip_lists())
    with open(f"{p}/coords.pkl", "rb") as f:
        coords = pickle.load(f)
    key = lambda x: int(os.path.splitext(os.path.basename(x))[0])  # noqa: E731
    frames = read_imgs(sorted(glob.glob(os.path.join(f"{p}/full_imgs", "*.[jpJP][pnPN]*[gG]")), key=key))
    faces = read_imgs(sorted(glob.glob(os.path.join(f"{p}/face_imgs", "*.[jpJP][pnPN]*[gG]")), key=key))
    return make_avatar(sd, frames, faces, coords)


def warm_up(batch_size, avatar, modelres):
    """ultralight_avatar.py:85-91 — engine sessions run an eager warm-up pass when they are created."""
    logger.info("warmup model... (engine sessions warm up at creation)")


@register("avatar", "ultralight")
class LightReal(BaseAvatar):
    def __init__(self, opt, model, avatar):
        super().__init__(opt)
        audio_processor, _ = model
        self.model, self.frame_list_cycle, self.face_list_cycle, self.coord_list_cycle = avatar
        eng_avatar = getattr(avatar, "engine_avatar", None)
        if eng_avatar is None:
            raise RuntimeError("LightReal needs the payload of livetalking_b200.plugin.ultralight_avatar.load_avatar / make_avatar")
        self._engine_avatar = eng_avatar
        self._frame_free = not getattr(eng_avatar, "frames_resident", True)
        self._return_pred = bool(getattr(opt, "ltb_return_pred", False))
        # every session owns its stream + scratch (two: U-Net graph, HuBERT graph); weights / avatar assets are shared
        self.engine_session = UltraLightSession(eng_avatar, self.batch_size)
        self.audio_processor = HubertFeatures(audio_processor.encoder, self.batch_size, opt.l, opt.r)
        self.asr = HubertASR(opt, self, self.audio_processor, audio_feat_length=[4, 4])
        self.asr.warm_up()
        # page-locked output ring for the fused mode (a D2H into pageable memory runs at a few GB/s, pinned at PCIe speed); a buffer is
        # reused after `ring` more batches: res_frame_queue holds at most 2 batches (base_avatar.py:86) + one produced + one pasted
        self._ring, self._ring_pos = [], 0
        if not self._return_pred:
            try:
                shape = (self.batch_size, *(eng_avatar.region_max if self._frame_free else (eng_avatar.H, eng_avatar.W)), 3)
                self._ring = [engine.PinnedBuffer(shape, np.uint8) for _ in range(max(4, int(os.environ.get("LTB_PIN_RING", "4"))))]
            except Exception as e:   # pinned memory exhausted: pageable output buffers
                logger.warning("pinned output ring unavailable (%r): using pageable buffers", e)
                self._ring = []

    def close(self):
        for o in (getattr(self, "engine_session", None), getattr(self, "audio_processor", None)):
            if o is not None:
                o.close()
        self.engine_session = self.audio_processor = None
        for b in getattr(self, "_ring", []):
            b.close()
        self._ring = []

    def _next_out(self):
        if not self._ring:
            return None
        buf = self._ring[self._ring_pos % len(self._ring)].array
        self._ring_pos += 1
        return buf

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _features(self, audiofeat_batch) -> np.ndarray:
        """(B, 16, 1024) float32.  The silence default of HubertASR is B x zeros((10, 1024)) — in the reference its reshape(16,32,32)
        would raise; BaseAvatar never forwards an all-silent batch to inference_batch, but be total: treat it as zero features."""
        out = np.zeros((self.batch_size, 16, 1024), np.float32)
        for i, a in enumerate(audiofeat_batch):
            a = np.asarray(a, np.float32)
            if a.shape == (16, 1024):
                out[i] = a
            elif a.size == 16 * 1024:
                out[i] = a.reshape(16, 1024)
        return out

    def inference_batch(self, index, audiofeat_batch):
        feats = self._features(audiofeat_batch)
        if self._return_pred:
            return self.engine_session.infer(index, feats, want_pred=True)          # float32 (B,160,160,3), as the reference
        length = len(self.face_list_cycle)
        if self._frame_free:
            regions, boxes = self.engine_session.infer_paste_region(index, feats, out=self._next_out())
            return [EngineRegion(regions[i], boxes[i], mirror_index(length, index + i)) for i in range(self.batch_size)]
        frames = self.engine_session.infer_paste(index, feats, out=self._next_out())   # (B,H,W,3) uint8: one engine round, one D2H
        return [EngineFrame(frames[i], mirror_index(length, index + i)) for i in range(self.batch_size)]

    def paste_back_frame(self, pred_frame, idx: int):
        if isinstance(pred_frame, (EngineFrame, EngineRegion)) and pred_frame.idx != idx:
            raise ValueError(f"paste_back_frame: frame was composited for idx {pred_frame.idx}, asked for {idx}")
        if isinstance(pred_frame, EngineFrame):
            return np.array(pred_frame.frame, copy=True)                              # fresh, writable, owned by Python
        if isinstance(pred_frame, EngineRegion):
            return engine.paste_region(self.frame_list_cycle[idx], pred_frame.region, pred_frame.box)
        if self._frame_free:
            region, box = self.engine_session.paste_pred_region(np.asarray(pred_frame, dtype=np.float32), idx)
            return engine.paste_region(self.frame_list_cycle[idx], region, box)
        return self.engine_session.paste_pred(np.asarray(pred_frame, dtype=np.float32), idx)
