"""SURVEY §8 a15 for the MuseTalk plugin: ``MuseReal`` + ``WhisperASR`` under the reference's REAL three-thread driving.

Same technique as tests/test_base_avatar_threads.py: the UNMODIFIED ``avatars/base_avatar.py`` runs ``render()`` against our plugin
class; the engine objects are deterministic stand-ins ("Whisper" = a cheap function of the PCM window, "UNet + VAE" = a cheap function
of (latent, feature window)).  Every emitted frame must equal the oracle's frame for ITS OWN audio window and avatar index: replayed
from the spied chunk stream with the silence short-circuit of inference(), the mirror index and the OpenCV-pinned blend paste-back of
oracle/paste_ref.py.  Also run in cross-session mode: two sessions, one shared scheduler, each gets its own frames back."""
import threading
import time

import cv2
import numpy as np

import ref_runtime as RR

B, N_AV, H, W = 4, 5, 220, 300


def fake_whisper(pcm: np.ndarray, batch: int, l: int) -> np.ndarray:
    """PCM window of (l + r + 2B) chunks -> (B, 50, 384) float16: frame i depends on its own two chunks only."""
    ch = np.asarray(pcm, np.float32).reshape(-1, 320)
    out = np.zeros((batch, 50, 384), np.float32)
    for i in range(batch):
        own = ch[l + 2 * i: l + 2 * i + 2].reshape(-1)
        out[i] = np.outer(np.linspace(0.5, 1.5, 50), np.resize(own[::2], 384)).astype(np.float32)
    return out.astype(np.float16)


def fake_net(latent: np.ndarray, feat: np.ndarray) -> np.ndarray:
    """(1,8,32,32) latent + (50,384) window -> (256,256,3) uint8 'decoded image', sensitive to both."""
    lat = np.kron(np.asarray(latent, np.float32)[0, :3].transpose(1, 2, 0), np.ones((8, 8, 1), np.float32))      # (256,256,3)
    f = np.asarray(feat, np.float32)
    pat = np.tile(f[:, :256], (6, 1))[:256]                                                                        # (256,256)
    return np.clip(128.0 + 40.0 * lat + 200.0 * pat[..., None], 0, 255).astype(np.uint8)


class FakeCtx:
    def close(self):
        pass


class FakeAvatar:
    def __init__(self, ctx, frames, masks, coords, crops, latents):
        self.frames = [np.asarray(f).copy() for f in frames]
        self.masks, self.coords, self.crops, self.latents = list(masks), [tuple(c) for c in coords], [tuple(c) for c in crops], list(latents)
        self.n, self.H, self.W, self.lat_hw = len(frames), self.frames[0].shape[0], self.frames[0].shape[1], 32


class FakeWhisperFeatures:
    def __init__(self, enc, batch, l=10, r=10, **kw):
        self.B, self.l, self.n = batch, l, (l + r + 2 * batch) * 320

    def run(self, pcm):
        time.sleep(0.001)
        assert np.asarray(pcm).size == self.n
        return fake_whisper(pcm, self.B, self.l)

    def close(self):
        pass


class FakeSession:
    """livetalking_b200.musetalk.MuseTalkSession surface (infer / paste_pred)."""

    def __init__(self, net, avatar, batch, paste_only=False, **kw):
        self.avatar, self.B, self.paste_only = avatar, batch, paste_only

    def infer(self, index, feats=None, want_pred=True):
        from oracle.paste_ref import mirror_index
        assert not self.paste_only
        time.sleep(0.004)
        a = self.avatar
        return np.stack([fake_net(a.latents[mirror_index(a.n, index + i)], np.asarray(feats)[i]) for i in range(self.B)])

    def paste_pred(self, pred_u8, idx):
        from oracle import paste_ref as P
        a = self.avatar
        time.sleep(0.001)
        return P.mt_paste_back(np.asarray(pred_u8, np.uint8), a.frames[idx], a.coords[idx], a.masks[idx], a.crops[idx])

    def close(self):
        pass


class FakeBatchSession:
    """livetalking_b200.musetalk.MuseTalkBatchSession surface: the mux of the cross-session scheduler."""
    instances = []

    def __init__(self, net, lat_hw, groups, frames_per_session, **kw):
        self.batch, self.Bs, self.sizes = groups, frames_per_session, []
        FakeBatchSession.instances.append(self)

    def infer_slots(self, requests):
        from oracle.paste_ref import mirror_index
        assert 1 <= len(requests) <= self.batch
        time.sleep(0.004)
        self.sizes.append(len(requests))
        return [np.stack([fake_net(av.latents[mirror_index(av.n, index + i)], np.asarray(feats)[i]) for i in range(self.Bs)])
                for av, index, feats in requests]

    def close(self):
        pass


def make_assets(seed):
    rng = np.random.default_rng(seed)
    frames = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(N_AV)]
    coords = [(70 + 2 * i, 40 + i, 200 + 2 * i, 180 + i) for i in range(N_AV)]                  # (x1,y1,x2,y2)
    crops = [(30, 10, 260, 210)] * N_AV                                                        # (x_s,y_s,x_e,y_e)
    soft = (np.clip((np.linspace(0, 1, 200)[:, None] - 0.35) * 4, 0, 1) * 255).astype(np.uint8) * np.ones((1, 230), np.uint8)
    masks = [np.stack([soft, soft, soft], -1)] * N_AV
    latents = [rng.standard_normal((1, 8, 32, 32)).astype(np.float32) for _ in range(N_AV)]
    return frames, masks, coords, crops, latents


def watermark(frame):
    cv2.putText(frame, "LiveTalking", (10, 20), cv2.FONT_HERSHEY_SIMPLEX, 0.3, (128, 128, 128), 1)   # base_avatar.py:449
    return frame


def replay_expected(chunks, n_frames, assets, l=10, r=10):
    from oracle import paste_ref as P
    frames, masks, coords, crops, latents = assets
    exp = []
    index = k = 0
    while len(exp) < n_frames:
        buf = chunks[2 * B * k: 2 * B * k + l + r + 2 * B]
        if len(buf) < l + r + 2 * B:
            break
        out = chunks[2 * B * k + l: 2 * B * k + l + 2 * B]
        silent = all(c.type != 0 for c in out)
        feats = None if silent else fake_whisper(np.concatenate([np.asarray(c.data, np.float32) for c in buf]), B, l)
        for i in range(B):
            idx = P.mirror_index(len(frames), index)
            if silent or all(c.type != 0 for c in out[2 * i: 2 * i + 2]):
                f = frames[idx].copy()
            else:
                f = P.mt_paste_back(fake_net(latents[idx], feats[i]), frames[idx], coords[idx], masks[idx], crops[idx])
            exp.append(watermark(np.ascontiguousarray(f)))
            index += 1
        k += 1
    return exp


def _patch(monkeypatch, MT):
    for name, fake in (("MuseTalkSession", FakeSession), ("MuseTalkAvatar", FakeAvatar), ("WhisperFeatures", FakeWhisperFeatures),
                       ("MuseTalkBatchSession", FakeBatchSession), ("Ctx", FakeCtx)):
        monkeypatch.setattr(MT, name, fake)


def _run(rt, avatars, n_target=220, timeout=150):
    sinks, spies, threads = [], [], []
    quit_event = threading.Event()
    for s, av in enumerate(avatars):
        sink = RR.RecordingSink()
        av.output, av.tts = sink, RR.NullTTS()
        pulled = [rt.AudioFrameData(data=np.zeros(320, np.float32), type=1, userdata={}) for _ in range(20)]
        RR.spy_audio_frames(av.asr, pulled)
        sinks.append(sink)
        spies.append(pulled)
        threads.append(threading.Thread(target=av.render, args=(quit_event,)))
        threads.append(threading.Thread(target=RR.feed_bursts, args=(av, [90, 70, 110, 50]), kwargs={"seed": s}))
    for t in threads:
        t.start()
    t0 = time.time()
    while min(len(s.frames) for s in sinks) < n_target and time.time() - t0 < timeout:
        time.sleep(0.02)
    quit_event.set()
    for t in threads:
        t.join(timeout=40)
    assert not any(t.is_alive() for t in threads), "render() did not stop"
    return sinks, spies


def _check(rt, sink, pulled, assets):
    n = len(sink.frames)
    assert n >= 200, f"only {n} frames emitted"
    exp = replay_expected(pulled, n, assets)
    assert len(exp) >= n - B
    n_checked = n_speech = 0
    for j in range(min(n, len(exp))):
        assert np.array_equal(sink.frames[j], exp[j]), f"frame {j}: does not match the oracle frame for its own audio window / index"
        n_checked += 1
        n_speech += int(not np.array_equal(exp[j], watermark(assets[0][rt.mirror_index(N_AV, j)].copy())))
    assert n_checked >= 200 and 40 <= n_speech <= n_checked - 20, (n_checked, n_speech)


def test_musereal_render_loop_every_frame_matches_its_own_audio_window(tmp_path, monkeypatch):
    assets = make_assets(0)
    with RR.reference_runtime(str(tmp_path)) as rt:
        MT = rt.load_musetalk()
        _patch(monkeypatch, MT)
        model = MT.EngineModel(FakeCtx(), net=object(), whisper=object())
        avatar = rt.registry.create("avatar", "musetalk", opt=RR.make_opt(batch_size=B), model=model,
                                    avatar=MT.make_avatar(*[list(a) for a in assets], model))
        assert isinstance(avatar, rt.base_avatar.BaseAvatar) and type(avatar.asr).__name__ == "WhisperASR"
        (sink,), (pulled,) = _run(rt, [avatar])
        _check(rt, sink, pulled, assets)
        avatar.close()


def test_musereal_cross_session_mode_under_the_real_render_loops(tmp_path, monkeypatch):
    """opt.ltb_cross_session: two sessions (own avatars, own audio) with the reference's own three threads each; their inference_batch
    calls are group requests to ONE shared scheduler; every session still gets exactly its own frames."""
    all_assets = [make_assets(10 + s) for s in range(2)]
    FakeBatchSession.instances.clear()
    with RR.reference_runtime(str(tmp_path)) as rt:
        MT = rt.load_musetalk()
        _patch(monkeypatch, MT)
        model = MT.EngineModel(FakeCtx(), net=object(), whisper=object())
        avatars = [rt.registry.create("avatar", "musetalk", opt=RR.make_opt(batch_size=B, ltb_cross_session=True, sessionid=s), model=model,
                                      avatar=MT.make_avatar(*[list(a) for a in all_assets[s]], model)) for s in range(2)]
        assert avatars[0]._batcher is avatars[1]._batcher and avatars[0].engine_session.paste_only
        sinks, spies = _run(rt, avatars)
        for s in range(2):
            _check(rt, sinks[s], spies[s], all_assets[s])
        mux = FakeBatchSession.instances[0]
        assert len(FakeBatchSession.instances) == 1 and sum(mux.sizes) == avatars[0]._batcher.slots and max(mux.sizes) <= mux.batch
        avatars[0]._batcher.close()
        for av in avatars:
            av.close()
