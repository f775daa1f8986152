"""SURVEY §8 a15 — the plugin under the reference's REAL three-thread driving.

The UNMODIFIED ``avatars/base_avatar.py`` is imported from the reference checkout (fake av / resampy / soundfile only),
``LipReal`` (our plugin class, a subclass of that real ``BaseAvatar``) is constructed through the real registry, a recording
sink replaces the transport, and the real ``render()`` runs — which starts the real ``inference`` and ``process_frames``
threads (avatars/base_avatar.py:469-501) — for >= 200 frames of speech bursts and silence.

Every emitted frame must equal the oracle's frame for ITS OWN audio window and avatar index: the test replays the exact
chunk stream ``run_step`` pulled (spied), rebuilds each step's (l + r + 2B)-chunk buffer, the mel windows (oracle/mel_ref.py),
the silence short-circuit, the mirror index and the paste-back (oracle/paste_ref.py), and compares bit for bit.

CPU variant: the engine session is a deterministic stand-in whose "network" is a cheap function of (face, mel window) —
what is under test is the plugin's plumbing under concurrency, not the CUDA kernels (tests/test_gpu_threads.py runs the same
loop against the real engine on the GPU box)."""
import threading
import time

import cv2
import numpy as np
import pytest

import ref_runtime as RR

B, N_AV, H, W = 4, 6, 120, 160


def fake_net(face_u8: np.ndarray, mel_win: np.ndarray) -> np.ndarray:
    """(256,256,3) u8 face + (80,16) mel window -> (256,256,3) float32 'prediction' in [0,255], sensitive to both inputs."""
    m = np.asarray(mel_win, np.float32)
    pat = np.tile(np.repeat(m, 4, axis=0)[:256, :], (1, 16))[:, :256]                 # (256,256) from the window
    return np.clip(face_u8.astype(np.float32) * 0.5 + 16.0 * (pat[..., None] + 4.0), 0.0, 255.0).astype(np.float32)


def make_assets(seed=0):
    rng = np.random.default_rng(seed)
    faces = [rng.integers(0, 256, (256, 256, 3), dtype=np.uint8) for _ in range(N_AV)]
    frames = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(N_AV)]
    coords = [(10 + i, 90 + i, 20 + 2 * i, 120 + 2 * i) for i in range(N_AV)]          # (y1, y2, x1, x2)
    return faces, frames, coords


class FakeAvatar:
    def __init__(self, faces, frames, coords):
        self.faces = np.asarray(faces).copy()
        self.frames = np.asarray(frames).copy()
        self.coords = [tuple(c) for c in coords]
        self.n, self.H, self.W = len(faces), self.frames.shape[1], self.frames.shape[2]


class FakeSession:
    """Same method surface as livetalking_b200.engine.W2LSession; oracle arithmetic; sleeps stand in for GPU latency so the
    three threads really interleave.  Like the real engine, predictions stay 'on the device' between infer and paste."""

    def __init__(self, model, avatar, batch, l=10, r=10, fps=25, **kw):
        self.avatar, self.batch, self.l, self.r, self.fps = avatar, batch, l, r, fps
        self._pred = None
        self.slot_batches = []
        self._mu = threading.Lock()
        self.concurrent_mel_during_infer = 0
        self._in_infer = False

    def mel_step(self, pcm, want_output=True):
        from oracle import mel_ref
        if self._in_infer:
            self.concurrent_mel_during_infer += 1
        time.sleep(0.001)
        return mel_ref.mel_step(np.asarray(pcm, np.float32), self.batch, self.l, self.r, self.fps).astype(np.float32)

    def infer(self, index, mel=None, want_pred=True):
        from oracle.paste_ref import mirror_index
        with self._mu:
            self._in_infer = True
            mel = np.asarray(mel, np.float32).reshape(self.batch, 80, 16).copy()
            time.sleep(0.004)
            self._pred = np.stack([fake_net(self.avatar.faces[mirror_index(self.avatar.n, index + i)], mel[i]) for i in range(self.batch)])
            self._in_infer = False
            return self._pred.copy() if want_pred else None

    def paste_batch(self, index, out=None, to_host=True):
        from oracle import paste_ref as P
        with self._mu:
            time.sleep(0.002)
            a = self.avatar
            idxs = [P.mirror_index(a.n, index + i) for i in range(self.batch)]
            return np.stack([P.w2l_paste_back(self._pred[i], a.frames[j], a.coords[j]) for i, j in enumerate(idxs)])

    def paste_pred(self, pred, idx, out=None):
        from oracle import paste_ref as P
        return P.w2l_paste_back(np.asarray(pred, np.float32), self.avatar.frames[idx], self.avatar.coords[idx])

    def infer_paste(self, index, mel, out=None):
        self.infer(index, mel, want_pred=False)
        frames = self.paste_batch(index)
        if out is not None:
            out[...] = frames
            return out
        return frames

    def infer_slots(self, requests, out=None):
        """cross-session batch (engine.W2LSession.infer_slots): every slot names its own avatar / frame / mel window"""
        from oracle import paste_ref as P
        assert 1 <= len(requests) <= self.batch
        time.sleep(0.004)
        self.slot_batches.append(len({id(av) for av, _i, _m in requests}))
        return np.stack([P.w2l_paste_back(fake_net(av.faces[idx], np.asarray(mel, np.float32).reshape(80, 16)), av.frames[idx], av.coords[idx])
                         for av, idx, mel in requests])

    def close(self):
        pass


def watermark(frame):
    cv2.putText(frame, "LiveTalking", (10, 20), cv2.FONT_HERSHEY_SIMPLEX, 0.3, (128, 128, 128), 1)   # base_avatar.py:449
    return frame


def replay_expected(chunks, n_frames, faces, frames, coords, net, l=10, r=10, fps=25):
    """chunks: every AudioFrameData the ASR pulled, in order (warm-up included).  -> list of expected frames (watermarked) and,
    per frame, the two chunk records that must accompany it."""
    from oracle import mel_ref
    from oracle import paste_ref as P
    exp, aud = [], []
    index = 0
    k = 0
    while len(exp) < n_frames:
        buf = chunks[2 * B * k: 2 * B * k + l + r + 2 * B]
        if len(buf) < l + r + 2 * B:
            break
        out = chunks[2 * B * k + l: 2 * B * k + l + 2 * B]        # what inference() pairs with this feature batch (output lags by r)
        silent = all(c.type != 0 for c in out)
        mel = None if silent else mel_ref.mel_step(np.concatenate([np.asarray(c.data, np.float32) for c in buf]), B, l, r, fps)
        for i in range(B):
            idx = P.mirror_index(len(frames), index)
            # inference() skips the model only when the WHOLE batch is silent (base_avatar.py:356-360); process_frames() shows the
            # plain avatar frame whenever the frame's OWN two chunks are silent, inferred or not (:409-417)
            if silent or all(c.type != 0 for c in out[2 * i: 2 * i + 2]):
                f = frames[idx].copy()
            else:
                f = P.w2l_paste_back(net(faces[idx], mel[i].astype(np.float32)), frames[idx], coords[idx])
            exp.append(watermark(np.ascontiguousarray(f)))
            aud.append(out[2 * i: 2 * i + 2])
            index += 1
        k += 1
    return exp, aud


@pytest.mark.parametrize("return_pred", [False, True], ids=["fused", "reference_pred"])
def test_render_loop_every_frame_matches_its_own_audio_window(tmp_path, monkeypatch, return_pred):
    faces, frames, coords = make_assets()
    pristine_frames = [f.copy() for f in frames]
    with RR.reference_runtime(str(tmp_path)) as rt:
        from livetalking_b200 import engine
        monkeypatch.setattr(engine, "W2LSession", FakeSession)
        monkeypatch.setattr(engine, "W2LAvatar", FakeAvatar)
        assert rt.plugin_base_asr.REFERENCE_BASE_ASR == rt.reference, "inside LiveTalking the plugin must use the reference's own BaseASR"
        payload = rt.plugin_w2l.make_avatar(frames, faces, coords)
        opt = RR.make_opt(batch_size=B, ltb_return_pred=return_pred)
        avatar = rt.registry.create("avatar", "wav2lip", opt=opt, model=object(), avatar=payload)      # app.py:99
        assert isinstance(avatar, rt.base_avatar.BaseAvatar) and type(avatar).__mro__[1] is rt.base_avatar.BaseAvatar
        sink = RR.RecordingSink()
        avatar.output, avatar.tts = sink, RR.NullTTS()
        warm = [rt.AudioFrameData(data=np.zeros(320, np.float32), type=1, userdata={}) for _ in range(20)]   # warm_up() ran on an empty queue
        pulled = list(warm)
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
        assert sink.started and sink.stopped
        n = len(sink.frames)
        assert n >= 200, f"only {n} frames emitted"
        assert len(sink.audio) >= 2 * n - 2
        exp, aud = replay_expected(pulled, n, faces, pristine_frames, coords, fake_net)
        assert len(exp) >= n - B
        n_speech = n_checked = 0
        for j in range(min(n, len(exp))):
            assert np.array_equal(sink.frames[j], exp[j]), f"frame {j}: does not match the oracle frame for its own audio window / index"
            n_checked += 1
            for t in range(2):                                   # the audio that accompanies frame j is the audio its window was cut for
                if 2 * j + t < len(sink.audio):
                    pcm16, ud = sink.audio[2 * j + t]
                    want = aud[j][t]
                    assert ud == want.userdata
                    assert np.array_equal(pcm16, (np.asarray(want.data) * 32767).astype(np.int16))
            n_speech += int(any(c.type == 0 for c in aud[j]))
        assert n_checked >= 200 and 40 <= n_speech <= n_checked - 20, (n_checked, n_speech)     # both branches exercised
        if hasattr(avatar.engine_session, "concurrent_mel_during_infer"):
            # the three threads really overlapped: run_step computed features while inference_batch was in flight
            assert avatar.engine_session.concurrent_mel_during_infer > 0


def test_short_custom_audio_chunk_does_not_kill_run_step(tmp_path, monkeypatch):
    """ADVICE r1: get_custom_audio_stream hands out a SHORT last chunk (base_avatar.py:303-309); run_step must pad it, not raise."""
    faces, frames, coords = make_assets(1)
    with RR.reference_runtime(str(tmp_path)) as rt:
        from livetalking_b200 import engine
        monkeypatch.setattr(engine, "W2LSession", FakeSession)
        monkeypatch.setattr(engine, "W2LAvatar", FakeAvatar)
        avatar = rt.registry.create("avatar", "wav2lip", opt=RR.make_opt(batch_size=B), model=object(),
                                    avatar=rt.plugin_w2l.make_avatar(frames, faces, coords))
        clip = (0.1 * np.random.default_rng(0).standard_normal(320 * 5 + 123)).astype(np.float32)     # not a multiple of 320
        avatar.custom_audio_cycle[2] = clip
        avatar.custom_audio_index[2] = 0
        avatar.custom_index[2] = 0
        avatar.custom_audiotype = 2
        for _ in range(2):                                       # feat_queue holds 2 batches (base_asr.py:46)
            avatar.asr.run_step()
        assert avatar.custom_audiotype == 1                       # clip exhausted -> back to silence (base_avatar.py:307-308)
        assert avatar.asr.feat_queue.qsize() == 2
        sizes = {np.asarray(avatar.asr.output_queue.get().data).size for _ in range(avatar.asr.output_queue.qsize())}
        assert sizes == {320}


def test_silent_frames_of_a_packed_avatar_take_the_watermark(tmp_path, monkeypatch):
    """ADVICE r1: process_frames draws into frame_list_cycle[idx] on silent frames; packed avatars must hand out writable frames."""
    from livetalking_b200 import avatar_pack as AP
    faces, frames, coords = make_assets(2)
    root = tmp_path / "data" / "avatars" / "packed"
    (root / "full_imgs").mkdir(parents=True)
    (root / "face_imgs").mkdir()
    import pickle
    for i in range(N_AV):
        cv2.imwrite(str(root / "full_imgs" / f"{i:08d}.png"), frames[i])
        cv2.imwrite(str(root / "face_imgs" / f"{i:08d}.png"), faces[i])
    with open(root / "coords.pkl", "wb") as f:
        pickle.dump(coords, f)
    AP.pack_wav2lip(str(root))
    with RR.reference_runtime(str(tmp_path)) as rt:
        from livetalking_b200 import engine
        monkeypatch.setattr(engine, "W2LSession", FakeSession)
        monkeypatch.setattr(engine, "W2LAvatar", FakeAvatar)
        payload = rt.plugin_w2l.load_avatar("packed")            # cwd = tmp_path -> ./data/avatars/packed/avatar.ltbav
        avatar = rt.registry.create("avatar", "wav2lip", opt=RR.make_opt(batch_size=B), model=object(), avatar=payload)
        sink = RR.RecordingSink()
        avatar.output, avatar.tts = sink, RR.NullTTS()
        quit_event = threading.Event()
        th = threading.Thread(target=avatar.render, args=(quit_event,))
        th.start()
        t0 = time.time()
        while len(sink.frames) < 2 * B and time.time() - t0 < 60:
            time.sleep(0.02)
        quit_event.set()
        th.join(timeout=30)
        assert len(sink.frames) >= 2 * B, "process_frames died on the first silent frame"
        for j, f in enumerate(sink.frames[:2 * B]):
            assert np.array_equal(f, watermark(frames[rt.mirror_index(N_AV, j)].copy()))


def test_cross_session_batching_under_the_real_render_loops(tmp_path, monkeypatch):
    """SURVEY §8 f1: three sessions, each with the reference's own three threads, share ONE forward launch per batch of slots;
    every session still gets exactly its own frames."""
    import types
    n_sess = 3
    assets = [make_assets(10 + s) for s in range(n_sess)]
    pristine = [[f.copy() for f in a[1]] for a in assets]
    with RR.reference_runtime(str(tmp_path)) as rt:
        from livetalking_b200 import engine
        monkeypatch.setattr(engine, "W2LSession", FakeSession)
        monkeypatch.setattr(engine, "W2LAvatar", FakeAvatar)
        monkeypatch.setenv("LTB_MUX_BATCH", "8")
        model = types.SimpleNamespace()                            # shared by the sessions, as app.py:99 shares the model
        avatars, sinks, pulled = [], [], []
        for s in range(n_sess):
            faces, frames, coords = assets[s]
            opt = RR.make_opt(batch_size=2, ltb_cross_session=True, sessionid=s)
            av = rt.registry.create("avatar", "wav2lip", opt=opt, model=model, avatar=rt.plugin_w2l.make_avatar(frames, faces, coords))
            sink = RR.RecordingSink()
            av.output, av.tts = sink, RR.NullTTS()
            log = [rt.AudioFrameData(data=np.zeros(320, np.float32), type=1, userdata={}) for _ in range(20)]
            RR.spy_audio_frames(av.asr, log)
            avatars.append(av)
            sinks.append(sink)
            pulled.append(log)
        batcher = avatars[0]._batcher
        assert batcher is not None and all(a._batcher is batcher for a in avatars)
        quit_event = threading.Event()
        renders = [threading.Thread(target=a.render, args=(quit_event,)) for a in avatars]
        feeders = [threading.Thread(target=RR.feed_bursts, args=(a, [60, 50], 320, 100 + i)) for i, a in enumerate(avatars)]
        for t in renders + feeders:
            t.start()
        t0 = time.time()
        while min(len(s.frames) for s in sinks) < 70 and time.time() - t0 < 120:
            time.sleep(0.02)
        quit_event.set()
        for t in renders + feeders:
            t.join(timeout=30)
        batcher.close()
        global B
        old_B, B = B, 2                                            # replay_expected reads the module-level batch size
        try:
            for s in range(n_sess):
                n = len(sinks[s].frames)
                assert n >= 60
                exp, _aud = replay_expected(pulled[s], n, assets[s][0], pristine[s], assets[s][2], fake_net)
                for j in range(min(n, len(exp))):
                    assert np.array_equal(sinks[s].frames[j], exp[j]), f"session {s} frame {j}"
        finally:
            B = old_B
        mux = batcher.mux
        assert max(mux.slot_batches) >= 2, "no batch ever mixed frames of different sessions"
        assert batcher.slots > batcher.batches                      # requests were packed
