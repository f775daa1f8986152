"""Frame-free UltraLight avatars on the CPU.

1. The bbox rectangle (the crop with [4:164] replaced by the prediction, resized by oracle/paste_ref.py) + engine.paste_region equals
   the reference's full-frame LightReal.paste_back_frame (ultralight_avatar.py:171-184, run with cv2) bit for bit, over random frame
   sizes and boxes, edge-touching, odd, identity (168²) and exact-halving (84²) ones included.
2. The unmodified three-thread render loop drives a frame-free LightReal (fused and ltb_return_pred) whose engine is a fake defined
   here with no frames at all; every emitted frame equals the oracle frame for its own audio window."""
import threading
import time

import numpy as np
import pytest

import ref_runtime as RR
import test_ultralight_threads as T

from livetalking_b200 import engine
from oracle import paste_ref as P
from oracle import ultralight_ref as U


def region_of(pred, crop_u8, bbox):
    """LightReal's composite restricted to the bbox: (y2-y1, x2-x1, 3) and the box in paste_region's (y1, y2, x1, x2) order."""
    x1, y1, x2, y2 = (int(v) for v in bbox)
    crop = crop_u8.copy()
    crop[4:164, 4:164] = np.asarray(pred).astype(np.uint8)
    return P.resize_linear_u8(crop, x2 - x1, y2 - y1), (y1, y2, x1, x2)


def test_region_plus_host_paste_equals_reference_full_frame_paste():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(11)
    for H, W in [(200, 260), (301, 517), (1080, 1920), (97, 171)]:
        frame = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        boxes = [b for b in [(0, 0, 168, 168), (W - 84, H - 84, W, H)] if min(b) >= 0 and b[2] <= W and b[3] <= H] + [(0, 0, W, H), (5, 5, 6, 6)]
        while len(boxes) < 14:
            x1, y1 = int(rng.integers(0, W - 1)), int(rng.integers(0, H - 1))
            boxes.append((x1, y1, int(rng.integers(x1 + 1, W + 1)), int(rng.integers(y1 + 1, H + 1))))
        for bbox in boxes:
            crop = rng.integers(0, 256, (168, 168, 3), dtype=np.uint8)
            pred = rng.uniform(0, 255.99, (160, 160, 3)).astype(np.float32)
            region, box = region_of(pred, crop, bbox)
            want = U.lightreal_paste(pred, frame, crop, bbox, resize=lambda img, wh: cv2.resize(img, wh))
            assert np.array_equal(engine.paste_region(frame, region, box), want), ((H, W), bbox)


class FrameFreeAvatar:
    """Stands in for UltraLightAvatar(..., frames_resident=False): crops and boxes only, no frames."""

    def __init__(self, ctx, model, frames, faces, coords, frames_resident=True):
        assert frames_resident is False
        self.frames_resident = False
        self.faces = np.asarray(faces).copy()
        self.coords = [tuple(int(v) for v in c) for c in coords]
        self.n, (self.H, self.W) = len(faces), np.shape(frames[0])[:2]
        self.region_max = (max(c[3] - c[1] for c in self.coords), max(c[2] - c[0] for c in self.coords))
        self.model = model


class RegionSession(T.FakeSession):
    """The region methods of UltraLightSession with oracle arithmetic; the inherited full-frame ones fail (no frames)."""

    def infer_paste_region(self, index, feats=None, out=None):
        self.infer(index, feats, want_pred=False)
        a = self.avatar
        rh, rw = a.region_max
        regions = np.zeros((self.B, rh, rw, 3), np.uint8) if out is None else out
        boxes = []
        for i in range(self.B):
            j = U.mirror_index(a.n, index + i)
            r, box = region_of(self._pred[i], a.faces[j], a.coords[j])
            regions[i, :r.shape[0], :r.shape[1]] = r
            boxes.append(box)
        return regions, boxes

    def paste_pred_region(self, pred, idx):
        return region_of(pred, self.avatar.faces[idx], self.avatar.coords[idx])


@pytest.mark.parametrize("return_pred", [False, True], ids=["fused", "reference_pred"])
def test_frame_free_lightreal_render_loop_matches_oracle(tmp_path, monkeypatch, return_pred):
    rng = np.random.default_rng(4)
    faces = [rng.integers(0, 256, (168, 168, 3), dtype=np.uint8) for _ in range(T.N_AV)]
    frames = [rng.integers(0, 256, (T.H, T.W, 3), dtype=np.uint8) for _ in range(T.N_AV)]
    coords = [(0, 10 + 2 * i, 140 + i, 150 + 2 * i) for i in range(T.N_AV - 2)] + [(40, 30, 208, 198), (T.W - 84, T.H - 84, T.W, T.H)]
    pristine = [f.copy() for f in frames]
    with RR.reference_runtime(str(tmp_path)) as rt:
        UL = rt.load_ultralight()
        for name, fake in (("UltraLightSession", RegionSession), ("UltraLightAvatar", FrameFreeAvatar), ("UltraLightModel", T.FakeModel),
                           ("HubertFeatures", T.FakeHubertFeatures), ("Ctx", T.FakeCtx)):
            monkeypatch.setattr(UL, name, fake)
        payload = UL.make_avatar({"weights": 1}, frames, faces, coords, frames_resident=False)
        assert isinstance(payload.engine_avatar, FrameFreeAvatar)
        model = (UL.EngineAudio(T.FakeCtx(), encoder=object()), None)
        avatar = rt.registry.create("avatar", "ultralight", opt=RR.make_opt(batch_size=T.B, ltb_return_pred=return_pred), model=model,
                                    avatar=payload)
        sink = RR.RecordingSink()
        avatar.output, avatar.tts = sink, RR.NullTTS()
        pulled = [rt.AudioFrameData(data=np.zeros(320, np.float32), type=1, userdata={}) for _ in range(20)]
        RR.spy_audio_frames(avatar.asr, pulled)
        quit_event = threading.Event()
        render = threading.Thread(target=avatar.render, args=(quit_event,))
        feeder = threading.Thread(target=RR.feed_bursts, args=(avatar, [90, 70, 110, 50]))
        render.start()
        feeder.start()
        t0 = time.time()
        while len(sink.frames) < 220 and time.time() - t0 < 120:
            time.sleep(0.02)
        quit_event.set()
        render.join(timeout=30)
        feeder.join(timeout=30)
        assert not render.is_alive()
        n = len(sink.frames)
        assert n >= 200, f"only {n} frames emitted"
        exp = T.replay_expected(pulled, n, faces, pristine, coords)
        n_speech = 0
        for j in range(min(n, len(exp))):
            assert np.array_equal(sink.frames[j], exp[j]), f"frame {j}: does not match the oracle frame for its own audio window / index"
            n_speech += int(not np.array_equal(exp[j], T.watermark(pristine[rt.mirror_index(T.N_AV, j)].copy())))
        assert n_speech >= 40
        avatar.close()


def test_ultralight_residency_rule(tmp_path, monkeypatch):
    """make_avatar asks engine.frames_fit_device: above the share of free memory the avatar is created frame-free."""
    made = []

    def recording_avatar(ctx, model, frames, faces, coords, frames_resident=True):
        made.append(frames_resident)
        return object()

    big = [np.zeros((1080, 1920, 3), np.uint8)] * 12
    with RR.reference_runtime(str(tmp_path)) as rt:
        UL = rt.load_ultralight()
        for name, fake in (("UltraLightAvatar", recording_avatar), ("UltraLightModel", T.FakeModel), ("Ctx", T.FakeCtx)):
            monkeypatch.setattr(UL, name, fake)
        for free, want in [(180 << 30, True), (200 << 20, False)]:
            monkeypatch.setattr(engine, "mem_get_info", lambda free=free: (free, 180 << 30))
            UL.make_avatar({}, big, [np.zeros((168, 168, 3), np.uint8)] * 12, [(0, 0, 168, 168)] * 12)
            assert made[-1] is want
