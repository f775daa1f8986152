"""Frame-free MuseTalk avatars on the CPU.

1. The blended crop box — oracle/paste_ref.py's mt_paste_back run on the body crop alone, boxes shifted into it — written into a copy
   of the frame by engine.paste_region equals the reference's full-frame get_image_blending (avatars/musetalk/myutil.py:4-25, run with
   cv2 as MuseReal.paste_back_frame drives it, and its stored output in mt_blend_golden.npz) bit for bit, over random frame sizes,
   crop boxes touching the frame edges, odd sizes and 256² / 512² predictions.
2. The unmodified three-thread render loop drives frame-free MuseReal sessions (single and cross-session) whose engine is a fake
   defined here with no frames at all; every emitted frame equals the oracle frame for its own audio window.
3. The residency rule picks frame-free above the share of free device memory, also for an avatar loaded without the model."""
import os

import numpy as np
import pytest

import ref_runtime as RR
import test_musetalk_threads as T
from test_oracle_paste import mt_blend_case

from livetalking_b200 import engine
from oracle import paste_ref as P


def region_of(pred_u8, frame, bbox, mask, crop):
    """get_image_blending restricted to the crop box: the oracle on the body crop, boxes shifted -> (region, (y_s, y_e, x_s, x_e))."""
    xs, ys, xe, ye = (int(v) for v in crop)
    x1, y1, x2, y2 = (int(v) for v in bbox)
    body = np.ascontiguousarray(frame[ys:ye, xs:xe])
    return P.mt_paste_back(pred_u8, body, (x1 - xs, y1 - ys, x2 - xs, y2 - ys), mask, (0, 0, xe - xs, ye - ys)), (ys, ye, xs, xe)


def reference_blend(cv2, pred_u8, frame, bbox, mask, crop):
    """MuseReal.paste_back_frame -> get_image_blending (myutil.py:4-25) on the full frame, with OpenCV."""
    x1, y1, x2, y2 = bbox
    xs, ys, xe, ye = crop
    body = frame.copy()
    res_frame = cv2.resize(pred_u8.astype(np.uint8), (x2 - x1, y2 - y1))
    face_large = body[ys:ye, xs:xe].copy()
    face_large[y1 - ys:y2 - ys, x1 - xs:x2 - xs] = res_frame
    mask_image = cv2.cvtColor(mask, cv2.COLOR_BGR2GRAY)
    mask_image = (mask_image / 255).astype(np.float32)
    body[ys:ye, xs:xe] = cv2.blendLinear(face_large, body[ys:ye, xs:xe], mask_image, 1 - mask_image)
    return body


def random_case(rng, H, W, S):
    xs, ys = int(rng.integers(0, W // 3)), int(rng.integers(0, H // 3))
    xe, ye = int(rng.integers(xs + 8, W + 1)), int(rng.integers(ys + 8, H + 1))
    if rng.random() < 0.4:                                            # crop box on the frame edges
        xs, ys, xe, ye = (0 if rng.random() < 0.5 else xs), (0 if rng.random() < 0.5 else ys), W, H
    x1, y1 = int(rng.integers(xs, xe - 4)), int(rng.integers(ys, ye - 4))
    x2, y2 = int(rng.integers(x1 + 1, xe + 1)), int(rng.integers(y1 + 1, ye + 1))
    mask = rng.integers(0, 256, (ye - ys, xe - xs, 3), dtype=np.uint8)
    return rng.integers(0, 256, (S, S, 3), dtype=np.uint8), (x1, y1, x2, y2), mask, (xs, ys, xe, ye)


@pytest.mark.parametrize("S", [256, 512])
def test_region_plus_host_paste_equals_reference_blend(S):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(S)
    for H, W in [(180, 240), (301, 517), (720, 1280), (97, 131)]:
        frame = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        for _ in range(8):
            pred, bbox, mask, crop = random_case(rng, H, W, S)
            region, box = region_of(pred, frame, bbox, mask, crop)
            got = engine.paste_region(frame, region, box)
            assert np.array_equal(got, reference_blend(cv2, pred, frame, bbox, mask, crop)), ((H, W), bbox, crop)
    # the identity (S x S bbox) and exact-halving cases of cv2.resize
    frame = rng.integers(0, 256, (S + 40, S + 60, 3), dtype=np.uint8)
    for bbox, crop in [((20, 10, 20 + S, 10 + S), (0, 0, S + 60, S + 40)), ((5, 7, 5 + S // 2, 7 + S // 2), (3, 2, S // 2 + 30, S // 2 + 33))]:
        pred, _b, _m, _c = random_case(rng, S + 40, S + 60, S)
        mask = rng.integers(0, 256, (crop[3] - crop[1], crop[2] - crop[0], 3), dtype=np.uint8)
        region, box = region_of(pred, frame, bbox, mask, crop)
        assert np.array_equal(engine.paste_region(frame, region, box), reference_blend(cv2, pred, frame, bbox, mask, crop))


def test_region_plus_host_paste_equals_stored_reference_output(golden_dir):
    frame, pred, bbox, crop, masks = mt_blend_case()
    want = np.load(os.path.join(golden_dir, "mt_blend_golden.npz"))["want"]
    for mask, ref_out in zip(masks, want):
        region, box = region_of(pred, frame, bbox, mask, crop)
        assert np.array_equal(engine.paste_region(frame, region, box), ref_out)


class FrameFreeAvatar:
    """Stands in for MuseTalkAvatar(..., frames_resident=False): body crops (the crop box of every frame) instead of frames."""

    def __init__(self, ctx, frames, masks, coords, crops, latents, frames_resident=True):
        assert frames_resident is False
        self.frames_resident = False
        self.crops = [tuple(int(v) for v in c) for c in crops]
        self.body = [np.ascontiguousarray(f[ys:ye, xs:xe]).copy() for f, (xs, ys, xe, ye) in zip(frames, self.crops)]
        self.masks, self.coords, self.latents = list(masks), [tuple(c) for c in coords], list(latents)
        self.n, (self.H, self.W), self.lat_hw = len(frames), np.shape(frames[0])[:2], 32


class RegionSession(T.FakeSession):
    """paste_pred_region of MuseTalkSession with oracle arithmetic on the body crop; the inherited paste_pred fails (no frames)."""

    def paste_pred_region(self, pred_u8, idx):
        a = self.avatar
        xs, ys, xe, ye = a.crops[idx]
        x1, y1, x2, y2 = a.coords[idx]
        region = P.mt_paste_back(np.asarray(pred_u8, np.uint8), a.body[idx], (x1 - xs, y1 - ys, x2 - xs, y2 - ys), a.masks[idx],
                                 (0, 0, xe - xs, ye - ys))
        return region, (ys, ye, xs, xe)


def _patch(monkeypatch, MT):
    T._patch(monkeypatch, MT)
    monkeypatch.setattr(MT, "MuseTalkSession", RegionSession)
    monkeypatch.setattr(MT, "MuseTalkAvatar", FrameFreeAvatar)


def test_frame_free_musereal_render_loop(tmp_path, monkeypatch):
    assets = T.make_assets(3)
    with RR.reference_runtime(str(tmp_path)) as rt:
        MT = rt.load_musetalk()
        _patch(monkeypatch, MT)
        model = MT.EngineModel(T.FakeCtx(), net=object(), whisper=object())
        payload = MT.make_avatar(*[list(a) for a in assets], model, frames_resident=False)
        assert isinstance(payload.engine_avatar, FrameFreeAvatar)
        avatar = rt.registry.create("avatar", "musetalk", opt=RR.make_opt(batch_size=T.B), model=model, avatar=payload)
        (sink,), (pulled,) = T._run(rt, [avatar])
        T._check(rt, sink, pulled, assets)
        avatar.close()


def test_frame_free_musereal_cross_session(tmp_path, monkeypatch):
    all_assets = [T.make_assets(30 + s) for s in range(2)]
    T.FakeBatchSession.instances.clear()
    with RR.reference_runtime(str(tmp_path)) as rt:
        MT = rt.load_musetalk()
        _patch(monkeypatch, MT)
        model = MT.EngineModel(T.FakeCtx(), net=object(), whisper=object())
        avatars = [rt.registry.create("avatar", "musetalk", opt=RR.make_opt(batch_size=T.B, ltb_cross_session=True, sessionid=s), model=model,
                                      avatar=MT.make_avatar(*[list(a) for a in all_assets[s]], model, frames_resident=False))
                   for s in range(2)]
        assert avatars[0]._batcher is avatars[1]._batcher and all(a._frame_free for a in avatars)
        sinks, spies = T._run(rt, avatars)
        for s in range(2):
            T._check(rt, sinks[s], spies[s], all_assets[s])
        avatars[0]._batcher.close()
        for av in avatars:
            av.close()


def test_musetalk_residency_rule(tmp_path, monkeypatch):
    """make_avatar (with the model) and MuseReal (payload loaded without it, as app.py does) both apply engine.frames_fit_device."""
    made = []

    def recording_avatar(ctx, frames, masks, coords, crops, latents, frames_resident=True):
        made.append(frames_resident)
        return FrameFreeAvatar(ctx, frames, masks, coords, crops, latents, False) if not frames_resident else \
            T.FakeAvatar(ctx, frames, masks, coords, crops, latents)

    n = 12
    big = ([np.zeros((1080, 1920, 3), np.uint8)] * n, [np.zeros((200, 230, 3), np.uint8)] * n, [(70, 40, 200, 180)] * n,
           [(30, 10, 260, 210)] * n, [np.zeros((1, 8, 32, 32), np.float32)] * n)
    with RR.reference_runtime(str(tmp_path)) as rt:
        MT = rt.load_musetalk()
        T._patch(monkeypatch, MT)
        monkeypatch.setattr(MT, "MuseTalkAvatar", recording_avatar)
        model = MT.EngineModel(T.FakeCtx(), net=object(), whisper=object())
        for free, want in [(180 << 30, True), (200 << 20, False)]:
            monkeypatch.setattr(engine, "mem_get_info", lambda free=free: (free, 180 << 30))
            MT.make_avatar(*big, model)
            assert made[-1] is want
            payload = MT.make_avatar(*big)                                 # app.py:86-91: no model at load time
            assert payload.engine_avatar is None
            av = rt.registry.create("avatar", "musetalk", opt=RR.make_opt(batch_size=T.B), model=model, avatar=payload)
            assert made[-1] is want and av._frame_free is (not want)
            av.close()
