"""CPU: host-side logic of the plugin layer (queues, silence synthesis, warm-up, run_step bookkeeping), and equivalence with
the reference's own BaseASR / WhisperASR / HubertASR on the same event sequences (their results are stored in
tests/golden/asr_host_golden.npz by tests/golden/make_golden.py::make_asr_host)."""
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(__file__))
import stubs  # noqa: E402

stubs.install()
from livetalking_b200.plugin import base_asr as B  # noqa: E402


def _feed(asr, n, rng):
    chunks = [rng.standard_normal(320).astype(np.float32) for _ in range(n)]
    for i, c in enumerate(chunks):
        asr.put_audio_frame(c, {"i": i})
    return chunks


def _golden():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "asr_host_golden.npz"))


def _assert_records(frames, types, data, userdata=None):
    assert len(frames) == len(types)
    for k, f in enumerate(frames):
        assert f.type == types[k] and np.array_equal(np.asarray(f.data, np.float32), data[k])
        if userdata is not None:
            assert f.userdata == json.loads(str(userdata[k]))


def _assert_frames(frames, want):
    assert len(frames) == len(want) and all(np.array_equal(x, y) for x, y in zip(frames, want))


def _drain(q):
    return [q.get() for _ in range(q.qsize())]


def test_silence_synthesis_and_warm_up():
    opt = stubs.Opt(batch_size=2)
    a = B.BaseASR(opt)
    assert a.chunk == 320 and a.feat_queue.maxsize == 2
    f = a.get_audio_frame()                             # empty queue -> zeros, type 1 (base_asr.py:66-69)
    assert f.type == 1 and f.data.shape == (320,) and f.data.dtype == np.float32 and not f.data.any()
    rng = np.random.default_rng(0)
    chunks = _feed(a, 25, rng)
    a.warm_up()                                         # l + r = 20 chunks consumed, first l = 10 dropped from output
    assert len(a.frames) == 20 and a.output_queue.qsize() == 10
    out = a.get_audio_out()
    assert out.type == 0 and np.array_equal(out.data, chunks[10]) and out.userdata == {"i": 10}
    a.flush_talk()
    assert a.queue.qsize() == 0


def test_custom_audio_stream_has_priority():
    class Parent:
        custom_audiotype = 2

        def get_custom_audio_stream(self, t):
            return np.full(320, 0.25, np.float32)

    a = B.BaseASR(stubs.Opt(), Parent())
    a.put_audio_frame(np.ones(320, np.float32), {})
    f = a.get_audio_frame()
    assert f.type == 2 and float(f.data[0]) == 0.25      # base_asr.py:59-62


def test_same_behaviour_as_reference_base_asr():
    g = _golden()
    ours = B.BaseASR(stubs.Opt(batch_size=3))
    _feed(ours, 23, np.random.default_rng(5))
    ours.warm_up()
    got = [ours.get_audio_frame() for _ in range(8)]     # drains speech then synthesises silence
    _assert_records(got, g["base_get_type"], g["base_get_data"], g["base_get_ud"])
    assert ours.output_queue.qsize() == int(g["base_outq"])
    _assert_frames(ours.frames, g["base_frames"])


def test_mel_asr_run_step_bookkeeping_with_fake_session():
    """run_step: 2B chunks forwarded, one feature list queued, l+r chunks of context kept (mel.py:36-67, Appendix E)."""
    from livetalking_b200.plugin.mel_asr import MelASR

    class FakeSession:
        def __init__(self):
            self.calls = []

        def mel_step(self, pcm):
            self.calls.append(pcm.copy())
            return np.zeros((2, 80, 16), np.float32)

    opt = stubs.Opt(batch_size=2)
    sess = FakeSession()
    asr = MelASR(opt, None, sess)
    rng = np.random.default_rng(1)
    chunks = _feed(asr, 24, rng)
    asr.warm_up()
    asr.run_step()
    assert asr.feat_queue.qsize() == 1 and asr.output_queue.qsize() == 10 + 4
    feats = asr.feat_queue.get()
    assert len(feats) == 2 and feats[0].shape == (80, 16)
    assert sess.calls[0].size == (10 + 10 + 4) * 320 and np.array_equal(sess.calls[0], np.concatenate(chunks[:24]))
    assert len(asr.frames) == 20 and np.array_equal(asr.frames[0], chunks[4])
    with pytest.raises(RuntimeError):
        MelASR(opt, None, None)                          # no engine session -> loud failure, never a CPU fallback


def test_whisper_asr_run_step_bookkeeping_matches_reference():
    """WhisperASR.run_step (whisper.py:58-76): 2B chunks forwarded, the whole l+r+2B context handed to the feature extractor,
    one list of B (50, 384) arrays queued, l+r chunks kept.  Every queue / buffer must match what the reference's own class
    recorded on the same event sequence (its Audio2Feature replaced by a recorder)."""
    from livetalking_b200.plugin.whisper_asr import WhisperASR

    class FakeFeatures:                                   # stands in for livetalking_b200.whisper.WhisperFeatures
        def __init__(self, B):
            self.B, self.calls = B, []

        def run(self, pcm):
            self.calls.append(pcm.copy())
            return np.zeros((self.B, 50, 384), np.float16)

    B = 3
    opt = stubs.Opt(batch_size=B)
    fake = FakeFeatures(B)
    ours = WhisperASR(opt, None, fake)
    rng = np.random.default_rng(2)
    chunks = _feed(ours, 20 + 2 * B + 2, rng)
    ours.warm_up()
    ours.run_step()
    assert ours.feat_queue.qsize() == 1 and ours.output_queue.qsize() == 10 + 2 * B
    feats = ours.feat_queue.get()
    assert len(feats) == B and feats[0].shape == (50, 384)
    assert fake.calls[0].dtype == np.float32 and np.array_equal(fake.calls[0], np.concatenate(chunks[:20 + 2 * B]))
    assert len(ours.frames) == 20 and np.array_equal(ours.frames[0], chunks[2 * B])
    with pytest.raises(RuntimeError):
        WhisperASR(opt, None, None)                       # no engine object -> loud failure, never a CPU fallback

    g = _golden()
    assert np.array_equal(np.asarray([np.asarray(f).shape for f in feats]), g["whisper_feat_shape"])
    assert np.array_equal(fake.calls[0], g["whisper_pcm"])                              # identical PCM context handed over
    _assert_frames(ours.frames, g["whisper_frames"])
    _assert_records(_drain(ours.output_queue), g["whisper_out_type"], g["whisper_out_data"])


def test_hubert_asr_run_step_bookkeeping_matches_reference():
    """HubertASR.run_step (avatars/audio_features/hubert.py:27-51): 2B chunks forwarded, silence tracking over TWO batches (features
    are computed unless this batch and the previous one were all silence), the whole l+r+2B context handed to the extractor, one
    list of B windows queued, l+r chunks kept.  Every queue / buffer / flag must match what the reference's own class recorded on
    the same event sequence (speech, then two silent steps) with its Audio2Feature replaced by a recorder."""
    from livetalking_b200.plugin.hubert_asr import HubertASR

    class FakeFeatures:                                   # stands in for livetalking_b200.hubert.HubertFeatures
        def __init__(self, B):
            self.B, self.calls = B, []

        def run(self, pcm):
            self.calls.append(pcm.copy())
            return np.ones((self.B, 16, 1024), np.float32)

    Bsz = 3
    opt = stubs.Opt(batch_size=Bsz)

    def drive(asr):
        _feed(asr, 20 + 2 * Bsz, np.random.default_rng(4))
        asr.warm_up()
        shapes = []
        for _step in range(3):                            # speech; silence (previous was speech -> still computed); silence (skipped)
            asr.run_step()
            shapes.append([np.asarray(f).shape for f in asr.feat_queue.get()])
        return shapes

    fake = FakeFeatures(Bsz)
    ours = HubertASR(opt, None, fake, audio_feat_length=[4, 4])
    shapes = drive(ours)
    assert shapes == [[(16, 1024)] * Bsz, [(16, 1024)] * Bsz, [(10, 1024)] * Bsz]
    assert len(fake.calls) == 2 and fake.calls[0].size == (20 + 2 * Bsz) * 320 and ours.last_is_silence
    with pytest.raises(RuntimeError):
        HubertASR(opt, None, None)                        # no engine object -> loud failure, never a CPU fallback

    g = _golden()
    assert np.array_equal(np.asarray(shapes), g["hubert_feat_shapes"])
    assert len(fake.calls) == len(g["hubert_pcm"]) and all(np.array_equal(a, b) for a, b in zip(fake.calls, g["hubert_pcm"]))
    assert ours.last_is_silence == bool(g["hubert_last_is_silence"])
    _assert_frames(ours.frames, g["hubert_frames"])
    _assert_records(_drain(ours.output_queue), g["hubert_out_type"], g["hubert_out_data"])
