"""Frame-free wav2lip avatars on the CPU: the device composites only the paste rectangle and the host writes it into a copy of
its own frame.

1. The region (oracle/paste_ref.py restricted to the box) + engine.paste_region equals the reference's full-frame paste glue
   (wav2lip_avatar.py:141-147, run with cv2) bit for bit, over random frame sizes and boxes, edge-touching and odd ones included.
2. The unmodified three-thread render loop drives a frame-free LipReal (fused, ltb_return_pred and cross-session); every emitted
   frame equals the oracle frame for its own audio window.  The engine is a fake defined here whose avatar has no frames at all.
3. The residency rule: with a patched free-memory reading, load_avatar uploads the frames below the share and goes frame-free
   above it."""
import pickle
import threading
import time
import types

import numpy as np
import pytest

import ref_runtime as RR
import test_base_avatar_threads as T

from livetalking_b200 import engine
from oracle import paste_ref as P


def reference_paste_back(cv2, pred, frame, box):
    """LipReal.paste_back_frame of the reference (wav2lip_avatar.py:141-147), on full frames."""
    y1, y2, x1, x2 = box
    combine_frame = frame.copy()
    res = cv2.resize(pred.astype(np.uint8), (x2 - x1, y2 - y1))
    combine_frame[y1:y2, x1:x2] = res
    return combine_frame


def random_boxes(rng, H, W, n):
    boxes = [(0, H, 0, W), (0, min(H, 256), 0, min(W, 256)), (H - min(H, 128), H, W - min(W, 128), W)]    # frame edges, 256², 128²
    while len(boxes) < n:
        y1, x1 = int(rng.integers(0, H - 1)), int(rng.integers(0, W - 1))
        boxes.append((y1, int(rng.integers(y1 + 1, H + 1)), x1, int(rng.integers(x1 + 1, W + 1))))
    return boxes


def test_region_plus_host_paste_equals_reference_full_frame_paste():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(7)
    for H, W in [(97, 131), (256, 256), (301, 517), (720, 1280), (131, 97)]:
        frame = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        for box in random_boxes(rng, H, W, 12):
            pred = rng.uniform(0, 255.999, (256, 256, 3)).astype(np.float32)
            y1, y2, x1, x2 = box
            region = P.resize_linear_u8(pred.astype(np.uint8), x2 - x1, y2 - y1)
            got = engine.paste_region(frame, region, box)
            assert got.flags.writeable and got.flags.owndata and got is not frame
            assert np.array_equal(got, reference_paste_back(cv2, pred, frame, box)), ((H, W), box)


class FrameFreeAvatar:
    """Stands in for engine.W2LAvatar(..., frames_resident=False): faces and boxes only, no frames."""

    def __init__(self, faces, frames, coords, frames_resident=True):
        assert frames_resident is False
        self.frames_resident = False
        self.faces = np.asarray(faces).copy()
        self.coords = np.asarray(coords, np.int32)
        self.n, (self.H, self.W) = len(faces), np.shape(frames[0])[:2]
        self.region_max = (int((self.coords[:, 1] - self.coords[:, 0]).max()), int((self.coords[:, 3] - self.coords[:, 2]).max()))


class RegionSession(T.FakeSession):
    """The region methods of engine.W2LSession with oracle arithmetic (the rectangle only).  The inherited full-frame methods
    fail for a FrameFreeAvatar, which has no frames."""

    def _region(self, pred, av, idx):
        y1, y2, x1, x2 = av.coords[idx]
        return P.resize_linear_u8(np.asarray(pred).astype(np.uint8), int(x2 - x1), int(y2 - y1))

    def infer_paste_region(self, index, mel, out=None):
        self.infer(index, mel, want_pred=False)
        a = self.avatar
        rh, rw = a.region_max
        regions = np.zeros((self.batch, rh, rw, 3), np.uint8) if out is None else out
        idxs = [P.mirror_index(a.n, index + i) for i in range(self.batch)]
        for i, j in enumerate(idxs):
            r = self._region(self._pred[i], a, j)
            regions[i, :r.shape[0], :r.shape[1]] = r
        return regions, a.coords[idxs]

    def paste_pred_region(self, pred, idx):
        return self._region(pred, self.avatar, idx), self.avatar.coords[idx]

    def infer_slots_region(self, requests):
        assert 1 <= len(requests) <= self.batch
        time.sleep(0.004)
        self.slot_batches.append(len({id(av) for av, _i, _m in requests}))
        return [(self._region(T.fake_net(av.faces[idx], np.asarray(mel, np.float32).reshape(80, 16)), av, idx), av.coords[idx])
                for av, idx, mel in requests]


def run_session(rt, avatar, sink, bursts, seed=0):
    """-> (chunks run_step pulled, quit event, render thread, feeder thread), threads not started yet."""
    pulled = [rt.AudioFrameData(data=np.zeros(320, np.float32), type=1, userdata={}) for _ in range(20)]
    RR.spy_audio_frames(avatar.asr, pulled)
    avatar.output, avatar.tts = sink, RR.NullTTS()
    quit_event = threading.Event()
    return (pulled, quit_event, threading.Thread(target=avatar.render, args=(quit_event,)),
            threading.Thread(target=RR.feed_bursts, args=(avatar, bursts, 320, seed)))


@pytest.mark.parametrize("return_pred", [False, True], ids=["fused", "reference_pred"])
def test_frame_free_render_loop_matches_oracle(tmp_path, monkeypatch, return_pred):
    faces, frames, coords = T.make_assets(3)
    pristine = [f.copy() for f in frames]
    with RR.reference_runtime(str(tmp_path)) as rt:
        monkeypatch.setattr(engine, "W2LSession", RegionSession)
        monkeypatch.setattr(engine, "W2LAvatar", FrameFreeAvatar)
        payload = rt.plugin_w2l.make_avatar(frames, faces, coords, frames_resident=False)
        assert isinstance(payload.engine_avatar, FrameFreeAvatar)
        avatar = rt.registry.create("avatar", "wav2lip", opt=RR.make_opt(batch_size=T.B, ltb_return_pred=return_pred), model=object(),
                                    avatar=payload)
        sink = RR.RecordingSink()
        pulled, quit_event, render, feeder = run_session(rt, avatar, sink, [90, 70, 110, 50])
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
        exp, aud = T.replay_expected(pulled, n, faces, pristine, coords, T.fake_net)
        n_speech = 0
        for j in range(min(n, len(exp))):
            assert np.array_equal(sink.frames[j], exp[j]), f"frame {j}: does not match the oracle frame for its own audio window / index"
            n_speech += int(any(c.type == 0 for c in aud[j]))
        assert n_speech >= 40


def test_frame_free_cross_session_render_loops(tmp_path, monkeypatch):
    """Two frame-free sessions (different frame sizes, same region capacity) and one full-frame session: the frame-free ones share
    one region scheduler, keyed by capacity; every session gets exactly its own frames."""
    assets = [T.make_assets(20 + s) for s in range(3)]
    # session 1: a different frame size with the same largest box as session 0 -> same region scheduler
    f1 = [np.ascontiguousarray(np.pad(f, ((0, 8), (0, 24), (0, 0)))) for f in assets[1][1]]
    assets[1] = (assets[1][0], f1, assets[1][2])
    pristine = [[f.copy() for f in a[1]] for a in assets]
    with RR.reference_runtime(str(tmp_path)) as rt:

        def avatar_factory(faces, frames, coords, frames_resident=True):
            return FrameFreeAvatar(faces, frames, coords, frames_resident) if not frames_resident else T.FakeAvatar(faces, frames, coords)

        monkeypatch.setattr(engine, "W2LSession", RegionSession)
        monkeypatch.setattr(engine, "W2LAvatar", avatar_factory)
        monkeypatch.setenv("LTB_MUX_BATCH", "8")
        monkeypatch.setattr(T, "B", 2)                               # replay_expected reads the module-level batch size
        model = types.SimpleNamespace()
        avatars, sinks, logs, threads, quits = [], [], [], [], []
        for s in range(3):
            faces, frames, coords = assets[s]
            payload = rt.plugin_w2l.make_avatar(frames, faces, coords, frames_resident=(s == 2))
            av = rt.registry.create("avatar", "wav2lip", opt=RR.make_opt(batch_size=2, ltb_cross_session=True, sessionid=s), model=model,
                                    avatar=payload)
            sink = RR.RecordingSink()
            pulled, quit_event, render, feeder = run_session(rt, av, sink, [60, 50], 100 + s)
            quits.append(quit_event)
            avatars.append(av)
            sinks.append(sink)
            logs.append(pulled)
            threads += [render, feeder]
        region_batcher = avatars[0]._batcher
        assert avatars[1]._batcher is region_batcher and avatars[2]._batcher is not region_batcher
        assert len(model._ltb_batchers) == 2
        for t in threads:
            t.start()
        t0 = time.time()
        while min(len(s.frames) for s in sinks) < 70 and time.time() - t0 < 120:
            time.sleep(0.02)
        for q in quits:
            q.set()
        for t in threads:
            t.join(timeout=30)
        for b in model._ltb_batchers.values():
            b.close()
        for s in range(3):
            n = len(sinks[s].frames)
            assert n >= 60
            exp, _aud = T.replay_expected(logs[s], n, assets[s][0], pristine[s], assets[s][2], T.fake_net)
            for j in range(min(n, len(exp))):
                assert np.array_equal(sinks[s].frames[j], exp[j]), f"session {s} frame {j}"
        assert region_batcher.batches > 0 and isinstance(region_batcher.mux.session, RegionSession)


def test_residency_rule_follows_free_device_memory(tmp_path, monkeypatch):
    """load_avatar uploads the full frames while they take at most FRAMES_DEVICE_SHARE of the free memory, else goes frame-free."""
    import cv2
    n, H, W = 12, 1080, 1920
    root = tmp_path / "data" / "avatars" / "big"
    (root / "full_imgs").mkdir(parents=True)
    (root / "face_imgs").mkdir()
    frame, face = np.full((H, W, 3), 90, np.uint8), np.full((256, 256, 3), 30, np.uint8)
    for i in range(n):
        cv2.imwrite(str(root / "full_imgs" / f"{i:08d}.png"), frame)
        cv2.imwrite(str(root / "face_imgs" / f"{i:08d}.png"), face)
    with open(root / "coords.pkl", "wb") as f:
        pickle.dump([(100, 420, 800, 1120)] * n, f)
    frames_bytes = n * H * W * 3
    assert frames_bytes > engine.FRAMES_ALWAYS_RESIDENT_BYTES
    made = []

    def recording_avatar(faces, frames, coords, frames_resident=True):
        made.append(frames_resident)
        return types.SimpleNamespace(frames_resident=frames_resident)

    with RR.reference_runtime(str(tmp_path)) as rt:
        monkeypatch.setattr(engine, "W2LAvatar", recording_avatar)
        for free, want in [(int(frames_bytes / engine.FRAMES_DEVICE_SHARE) + 1, True), (int(frames_bytes / engine.FRAMES_DEVICE_SHARE) - 1, False),
                           (180 << 30, True), (200 << 20, False)]:
            monkeypatch.setattr(engine, "mem_get_info", lambda free=free: (free, 180 << 30))
            payload = rt.plugin_w2l.load_avatar("big")
            assert made[-1] is want and payload.engine_avatar.frames_resident is want, free
        # small avatars never ask the device (the CPU tests with fake engines build only those)
        monkeypatch.setattr(engine, "mem_get_info", lambda: pytest.fail("queried the device for a small avatar"))
        faces, frames, coords = T.make_assets(0)
        rt.plugin_w2l.make_avatar(frames, faces, coords)
        assert made[-1] is True
