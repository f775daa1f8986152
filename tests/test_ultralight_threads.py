"""SURVEY §8 a15 for the UltraLight plugin (row f4): ``LightReal`` + ``HubertASR`` under the reference's REAL three-thread driving.

Same technique as tests/test_base_avatar_threads.py: the UNMODIFIED ``avatars/base_avatar.py`` runs ``render()`` (which starts the
real ``inference`` and ``process_frames`` threads) against our plugin class; the engine objects are deterministic stand-ins whose
"HuBERT" is a cheap function of the PCM window and whose "U-Net" is a cheap function of (face crop, feature window) — what is under
test is the plugin's plumbing under concurrency: every emitted frame must equal the oracle's frame for ITS OWN audio window and avatar
index (replayed from the spied chunk stream with the reference's window rows, HubertASR's two-batch silence rule, the silence
short-circuit of inference(), the mirror index and the OpenCV-pinned paste-back of oracle/ultralight_ref.py)."""
import threading
import time

import cv2
import numpy as np
import pytest

import ref_runtime as RR

B, N_AV, H, W = 4, 5, 200, 260


def fake_hubert(pcm: np.ndarray) -> np.ndarray:
    """(n,) PCM -> (T, 1024) 'hidden states', T = (n - 80) // 320: row t depends on the samples of its own 20 ms hop only."""
    n = pcm.size
    T = (n - 80) // 320
    hop = np.asarray(pcm[:T * 320], np.float32).reshape(T, 320)
    base = np.stack([hop.mean(1), np.abs(hop).mean(1), hop[:, 0], hop[:, 160]], 1)            # (T, 4)
    return np.tile(base, (1, 256)).astype(np.float32) * np.linspace(0.5, 1.5, 1024, dtype=np.float32)[None, :]


def fake_net(crop_u8: np.ndarray, feat: np.ndarray) -> np.ndarray:
    """(168,168,3) u8 crop + (16,1024) window -> (160,160,3) float32 'prediction' in [0,255], sensitive to both."""
    f = np.asarray(feat, np.float32)
    pat = np.tile(f[:, :160], (10, 1))                                                            # (160,160)
    return np.clip(crop_u8[4:164, 4:164].astype(np.float32) * 0.5 + 300.0 * np.abs(pat[..., None]) + 20.0, 0.0, 255.0).astype(np.float32)


class FakeCtx:
    def close(self):
        pass


class FakeModel:
    def __init__(self, ctx, sd):
        self.sd = sd


class FakeAvatar:
    def __init__(self, ctx, model, frames, faces, coords):
        self.frames, self.faces = np.asarray(frames).copy(), np.asarray(faces).copy()
        self.coords = [tuple(int(v) for v in c) for c in coords]
        self.n, self.H, self.W = len(frames), self.frames.shape[1], self.frames.shape[2]
        self.model = model


class FakeHubertFeatures:
    """livetalking_b200.hubert.HubertFeatures surface: run(pcm) -> (B, 16, 1024) float32 windows."""
    in_infer = None                                            # set by the session fake: counts real overlap of the threads

    def __init__(self, encoder, batch, l=10, r=10, **kw):
        self.B, self.l, self.n = batch, l, (l + r + 2 * batch) * 320
        self.overlaps = 0

    def run(self, pcm):
        from oracle import ultralight_ref as U
        if FakeHubertFeatures.in_infer is not None and FakeHubertFeatures.in_infer.is_set():
            self.overlaps += 1
        time.sleep(0.001)
        pcm = np.asarray(pcm, np.float32)
        assert pcm.size == self.n
        hid = U.trim_features(fake_hubert(pcm), pcm.size)
        return hid[U.window_rows(hid.shape[0], self.B, self.l / 2)].astype(np.float32)

    def close(self):
        pass


class FakeSession:
    """livetalking_b200.ultralight.UltraLightSession surface; oracle arithmetic; sleeps stand in for GPU latency."""

    def __init__(self, avatar, batch, **kw):
        self.avatar, self.B = avatar, batch
        self._mu = threading.Lock()
        self._pred = None
        FakeHubertFeatures.in_infer = threading.Event()

    def infer(self, index, feats=None, want_pred=True):
        from oracle import ultralight_ref as U
        with self._mu:
            FakeHubertFeatures.in_infer.set()
            feats = np.asarray(feats, np.float32).reshape(self.B, 16, 1024).copy()
            time.sleep(0.004)
            a = self.avatar
            self._pred = np.stack([fake_net(a.faces[U.mirror_index(a.n, index + i)], feats[i]) for i in range(self.B)])
            FakeHubertFeatures.in_infer.clear()
            return self._pred.copy() if want_pred else None

    def infer_paste(self, index, feats=None, out=None):
        from oracle import ultralight_ref as U
        self.infer(index, feats, want_pred=False)
        a = self.avatar
        idxs = [U.mirror_index(a.n, index + i) for i in range(self.B)]
        frames = np.stack([U.lightreal_paste(self._pred[i], a.frames[j], a.faces[j], a.coords[j]) for i, j in enumerate(idxs)])
        if out is not None:
            out[...] = frames
            return out
        return frames

    def paste_pred(self, pred, idx):
        from oracle import ultralight_ref as U
        a = self.avatar
        return U.lightreal_paste(np.asarray(pred, np.float32), a.frames[idx], a.faces[idx], a.coords[idx])

    def close(self):
        pass


def watermark(frame):
    cv2.putText(frame, "LiveTalking", (10, 20), cv2.FONT_HERSHEY_SIMPLEX, 0.3, (128, 128, 128), 1)   # base_avatar.py:449
    return frame


def replay_expected(chunks, n_frames, faces, frames, coords, l=10, r=10):
    from oracle import ultralight_ref as U
    exp = []
    index = k = 0
    last_is_silence = True                                        # HubertASR.__init__ (hubert.py:22)
    while len(exp) < n_frames:
        buf = chunks[2 * B * k: 2 * B * k + l + r + 2 * B]
        if len(buf) < l + r + 2 * B:
            break
        out = chunks[2 * B * k + l: 2 * B * k + l + 2 * B]        # the audio inference() pairs with this feature batch (lags by r)
        silent = all(c.type != 0 for c in out)
        # HubertASR decides on the 2B chunks it has just pulled (the NEWEST ones, r chunks ahead of `out`): features are computed
        # unless this pull and the previous one were all silence (hubert.py:40-41).  With 2B < r (this test: 8 < 10; never with the
        # reference's default batch 16) the tail of a burst can still be in `out` when that rule has already switched to the zero
        # default — the reference would then fail in reshape(16,32,32) on its (10,1024) zeros; the plugin feeds zero windows.
        newest = buf[l + r:]
        is_all_silence = all(c.type != 0 for c in newest)
        if not is_all_silence or not last_is_silence:
            pcm = np.concatenate([np.asarray(c.data, np.float32) for c in buf])
            hid = U.trim_features(fake_hubert(pcm), pcm.size)
            feats = hid[U.window_rows(hid.shape[0], B, l / 2)]
        else:
            feats = np.zeros((B, 16, 1024), np.float32)
        last_is_silence = is_all_silence
        for i in range(B):
            idx = U.mirror_index(len(frames), index)
            if silent or all(c.type != 0 for c in out[2 * i: 2 * i + 2]):
                f = frames[idx].copy()
            else:
                f = U.lightreal_paste(fake_net(faces[idx], feats[i]), frames[idx], faces[idx], coords[idx])
            exp.append(watermark(np.ascontiguousarray(f)))
            index += 1
        k += 1
    return exp


@pytest.mark.parametrize("return_pred", [False, True], ids=["fused", "reference_pred"])
def test_lightreal_render_loop_every_frame_matches_its_own_audio_window(tmp_path, monkeypatch, return_pred):
    rng = np.random.default_rng(0)
    faces = [rng.integers(0, 256, (168, 168, 3), dtype=np.uint8) for _ in range(N_AV)]
    frames = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(N_AV)]
    coords = [(20 + i, 10 + 2 * i, 140 + i, 150 + 2 * i) for i in range(N_AV - 1)] + [(40, 30, 208, 198)]     # (x1,y1,x2,y2); last = identity size
    pristine = [f.copy() for f in frames]
    with RR.reference_runtime(str(tmp_path)) as rt:
        UL = rt.load_ultralight()
        for name, fake in (("UltraLightSession", FakeSession), ("UltraLightAvatar", FakeAvatar), ("UltraLightModel", FakeModel),
                           ("HubertFeatures", FakeHubertFeatures), ("Ctx", FakeCtx)):
            monkeypatch.setattr(UL, name, fake)
        payload = UL.make_avatar({"weights": 1}, frames, faces, coords)
        model = (UL.EngineAudio(FakeCtx(), encoder=object()), None)                                # what load_model(opt) returns
        opt = RR.make_opt(batch_size=B, ltb_return_pred=return_pred)
        avatar = rt.registry.create("avatar", "ultralight", opt=opt, model=model, avatar=payload)   # app.py:99
        assert isinstance(avatar, rt.base_avatar.BaseAvatar) and type(avatar.asr).__name__ == "HubertASR"
        host_asr = "avatars.audio_features.base_asr" if rt.reference else "livetalking_b200.plugin.base_asr"
        assert type(avatar.asr).__mro__[1].__module__ == host_asr                                  # the host's own BaseASR
        sink = RR.RecordingSink()
        avatar.output, avatar.tts = sink, RR.NullTTS()
        pulled = [rt.AudioFrameData(data=np.zeros(320, np.float32), type=1, userdata={}) for _ in range(20)]   # warm_up() ran on an empty queue
        RR.spy_audio_frames(avatar.asr, pulled)
        quit_event = threading.Event()
        render = threading.Thread(target=avatar.render, args=(quit_event,))
        render.start()
        feeder = threading.Thread(target=RR.feed_bursts, args=(avatar, [90, 70, 110, 50]))
        feeder.start()
        t0 = time.time()
        while len(sink.frames) < 220 and time.time() - t0 < 120:
            time.sleep(0.02)
        quit_event.set()
        render.join(timeout=30)
        feeder.join(timeout=30)
        assert not render.is_alive(), "render() did not stop"
        n = len(sink.frames)
        assert n >= 200, f"only {n} frames emitted"
        exp = replay_expected(pulled, n, faces, pristine, coords)
        assert len(exp) >= n - B
        n_checked = n_speech = 0
        for j in range(min(n, len(exp))):
            assert np.array_equal(sink.frames[j], exp[j]), f"frame {j}: does not match the oracle frame for its own audio window / index"
            n_checked += 1
            n_speech += int(not np.array_equal(exp[j], watermark(pristine[rt.mirror_index(N_AV, j)].copy())))
        assert n_checked >= 200 and 40 <= n_speech <= n_checked - 20, (n_checked, n_speech)         # both branches exercised
        assert avatar.audio_processor.overlaps > 0          # run_step really computed features while inference_batch was in flight
        avatar.close()
