"""MuseTalk avatar plugin on the B200 engine — drop-in for avatars/musetalk_avatar.py.

Module surface used by app.py:140-143 (unchanged): ``load_model()``, ``load_avatar(avatar_id)``, ``warm_up(batch_size, model)``
and the class registered as ``("avatar", "musetalk")``.  ``MuseReal`` keeps the reference hooks:

    inference_batch(index, audiofeat_batch) -> (B,256,256,3) uint8 BGR predictions      (musetalk_avatar.py:130-152)
    paste_back_frame(pred_frame, idx)       -> H x W x 3 uint8 BGR, fresh and writable   (musetalk_avatar.py:154-164)

Frame-free avatars: the engine avatar gets the full frames only while they fit ``engine.frames_fit_device`` (a fixed share of the
device's free memory when the avatar is uploaded); otherwise it holds the crop boxes of the frames (what get_image_blending reads),
the device blends only the crop box, and ``paste_back_frame`` writes it into a fresh copy of ``frame_list_cycle[idx]``.  Single-session
and cross-session modes work with either residency and hand ``BaseAvatar`` the same frames.
"""
from __future__ import annotations

import glob
import json
import os
import pickle

import numpy as np

from .. import engine
from ..musetalk import MuseTalkAvatar, MuseTalkBatchSession, MuseTalkModel, MuseTalkSession
from ..ops import Ctx
from ..whisper import WhisperEncoder, WhisperFeatures
from .batcher import CrossSessionBatcher
from .whisper_asr import WhisperASR

try:
    from avatars.base_avatar import BaseAvatar
    from registry import register
    from utils.image import mirror_index, read_imgs
    from utils.logger import logger
except Exception as _e:  # pragma: no cover
    raise ImportError("livetalking_b200.plugin.musetalk_avatar must be imported inside LiveTalking (or with stubs): " + repr(_e))


class EngineModel:
    """What load_model() returns: one engine context holding the UNet + VAE and the Whisper encoder."""

    def __init__(self, ctx, net, whisper):
        self.ctx, self.net, self.whisper = ctx, net, whisper

    def __iter__(self):   # the reference unpacks a 5-tuple (vae, unet, pe, timesteps, audio_processor)
        return iter((self.net, self.net, self.net.pe, 0, self.whisper))


class AvatarPayload(tuple):
    engine_avatar = None
    frames_resident = None       # None: the residency rule decides when the engine avatar is created


def _engine_avatar(model: EngineModel, lists, frames_resident=None) -> MuseTalkAvatar:
    frames, masks, coords, mask_coords, latents = lists
    if frames_resident is None:
        frames_resident = engine.frames_fit_device(sum(np.asarray(f).nbytes for f in frames))
    if frames_resident:
        return MuseTalkAvatar(model.ctx, frames, masks, coords, mask_coords, latents)
    return MuseTalkAvatar(model.ctx, frames, masks, coords, mask_coords, latents, frames_resident=False)


def _load_state_dict(path):
    import torch
    if path.endswith(".safetensors"):
        from safetensors.torch import load_file
        return load_file(path)
    return torch.load(path, map_location="cpu")


def load_model(unet_path="./models/musetalkV15/unet.pth", unet_config="./models/musetalkV15/musetalk.json", vae_dir="./models/sd-vae",
               whisper_dir="./models/whisper"):
    """musetalk_avatar.py:57-67 / utils/utils.py:15-31: the same model files, made resident on the engine."""
    from transformers import WhisperModel
    from ..configs import unet_config_from_json, vae_config_from_json
    with open(unet_config) as f:
        ucfg = unet_config_from_json(json.load(f))
    with open(os.path.join(vae_dir, "config.json")) as f:
        vcfg = vae_config_from_json(json.load(f))
    vae_file = next(p for p in (os.path.join(vae_dir, n) for n in ("diffusion_pytorch_model.safetensors", "diffusion_pytorch_model.bin"))
                    if os.path.exists(p))
    whisper_sd = WhisperModel.from_pretrained(whisper_dir).state_dict()
    return make_model(_load_state_dict(unet_path), _load_state_dict(vae_file), whisper_sd, ucfg, vcfg)


def make_model(unet_sd, vae_sd, whisper_sd, ucfg, vcfg) -> EngineModel:
    engine.set_device(int(os.environ.get("LTB_DEVICE", "0")))
    ctx = Ctx()
    net = MuseTalkModel(ctx, unet_sd, vae_sd, ucfg, vcfg)
    return EngineModel(ctx, net, WhisperEncoder(ctx, whisper_sd))


def load_avatar(avatar_id, model: EngineModel = None):
    """musetalk_avatar.py:69-91 — same on-disk format (full_imgs/, mask/, coords.pkl, mask_coords.pkl, latents.pt)."""
    import torch
    p = f"./data/avatars/{avatar_id}"
    if os.path.exists(f"{p}/avatar.ltbav"):            # packed form (livetalking_b200.avatar_pack): one read, no PNG decodes
        from .. import avatar_pack
        return make_avatar(*avatar_pack.load_packed(f"{p}/avatar.ltbav").musetalk_lists(), model)
    key = lambda x: int(os.path.splitext(os.path.basename(x))[0])  # noqa: E731
    latents = torch.load(f"{p}/latents.pt", map_location="cpu")
    with open(f"{p}/coords.pkl", "rb") as f:
        coords = pickle.load(f)
    with open(f"{p}/mask_coords.pkl", "rb") as f:
        mask_coords = pickle.load(f)
    frames = read_imgs(sorted(glob.glob(os.path.join(f"{p}/full_imgs", "*.[jpJP][pnPN]*[gG]")), key=key))
    masks = read_imgs(sorted(glob.glob(os.path.join(f"{p}/mask", "*.[jpJP][pnPN]*[gG]")), key=key))
    return make_avatar(frames, masks, coords, mask_coords, latents, model)


def make_avatar(frames, masks, coords, mask_coords, latents, model: EngineModel = None, frames_resident=None) -> AvatarPayload:
    """frames_resident: None = the residency rule (engine.frames_fit_device); False forces a frame-free avatar."""
    payload = AvatarPayload((frames, masks, coords, mask_coords, latents))
    payload.frames_resident = frames_resident
    if model is not None:
        payload.engine_avatar = _engine_avatar(model, payload, frames_resident)
    return payload


def warm_up(batch_size, model):
    """musetalk_avatar.py:93-108 — engine sessions run an eager warm-up pass when they are created."""
    logger.info("warmup model... (engine sessions warm up at creation)")


_BATCHER_LOCK = __import__("threading").Lock()


def shared_batcher(model: EngineModel, lat_hw: int, frames_per_session: int) -> CrossSessionBatcher:
    """Cross-session mode (SURVEY 8(f) rank 1): one scheduler per (model, latent size, session batch size), created by the first
    session that asks.  Its mux is a MuseTalkBatchSession: up to LTB_MT_GROUPS sessions' B frames run as ONE UNet + VAE graph."""
    with _BATCHER_LOCK:
        table = getattr(model, "_ltb_batchers", None)
        if table is None:
            table = model._ltb_batchers = {}
        key = (int(lat_hw), int(frames_per_session))
        if key not in table:
            mux = MuseTalkBatchSession(model.net, lat_hw, int(os.environ.get("LTB_MT_GROUPS", "4")), frames_per_session)
            table[key] = CrossSessionBatcher(mux, float(os.environ.get("LTB_MUX_WAIT_MS", "4")))
        return table[key]


@register("avatar", "musetalk")
class MuseReal(BaseAvatar):
    def __init__(self, opt, model, avatar):
        super().__init__(opt)
        self.model = model
        self.frame_list_cycle, self.mask_list_cycle, self.coord_list_cycle, self.mask_coords_list_cycle, self.input_latent_list_cycle = avatar
        eng_avatar = getattr(avatar, "engine_avatar", None)
        if eng_avatar is None:
            # app.py:86-91 calls load_avatar(avatar_id) without the model and shares the payload between sessions: upload once,
            # cache on the payload (a plain tuple from elsewhere cannot carry it and is uploaded per session)
            eng_avatar = _engine_avatar(model, tuple(avatar), getattr(avatar, "frames_resident", None))
            if isinstance(avatar, AvatarPayload):
                avatar.engine_avatar = eng_avatar
        self._engine_avatar = eng_avatar
        self._frame_free = not getattr(eng_avatar, "frames_resident", True)
        cross = bool(getattr(opt, "ltb_cross_session", False)) or os.environ.get("LTB_CROSS_SESSION", "0") == "1"
        self._batcher = shared_batcher(model, eng_avatar.lat_hw, self.batch_size) if cross else None
        # every session owns its stream + scratch (two: UNet/VAE graph, Whisper graph); weights / avatar assets are shared.
        # Cross-session mode: the session keeps only a paste-back context, its UNet/VAE pass runs in the shared batch.
        self.engine_session = MuseTalkSession(model.net, eng_avatar, self.batch_size, paste_only=cross)
        self.audio_processor = WhisperFeatures(model.whisper, self.batch_size, opt.l, opt.r)
        self.asr = WhisperASR(opt, self, self.audio_processor)
        self.asr.warm_up()

    def close(self):
        """Release this session's graphs, streams and device buffers (one WebRTC connection = one session)."""
        for o in (getattr(self, "engine_session", None), getattr(self, "audio_processor", None)):
            if o is not None:
                o.close()
        self.engine_session = self.audio_processor = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def inference_batch(self, index, audiofeat_batch):
        whisper_batch = np.stack(audiofeat_batch)                                   # (B, 50, 384)
        if self._batcher is not None:                                               # one group request of the shared cross-session batch
            return self._batcher.submit([(self._engine_avatar, index, whisper_batch)])[0]
        return self.engine_session.infer(index, whisper_batch)                      # uint8 (B,256,256,3) BGR, as decode_latents

    def paste_back_frame(self, pred_frame, idx: int):
        if self._frame_free:
            region, box = self.engine_session.paste_pred_region(np.asarray(pred_frame).astype(np.uint8), idx)
            return engine.paste_region(self.frame_list_cycle[idx], region, box)
        return self.engine_session.paste_pred(np.asarray(pred_frame).astype(np.uint8), idx)
