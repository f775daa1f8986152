"""Run the plugin under the reference's REAL runtime: the unmodified ``avatars/base_avatar.py`` (its ``render`` /
``inference`` / ``process_frames`` threads, avatars/base_avatar.py:326-501), ``registry.py``, ``utils/image.py`` and
``avatars/audio_features/base_asr.py`` imported from the read-only checkout, with fake ``av`` / ``resampy`` / ``soundfile``
modules injected (the technique of the reference's own tests/test_asr_server.py:57-72 — those three are transport / file
decoding dependencies that the per-frame path never calls).

Used where a LiveTalking checkout is named by the LTB_REFERENCE environment variable; elsewhere ``reference_runtime`` hands out
the host of tests/stubs.py instead, whose ``BaseAvatar`` runs the same three-thread render loop, so the tests run everywhere.
Only the swapped module names (reference modules, the three fakes, the plugin modules) are saved and restored, so the
process-wide stubs other tests install come back afterwards and torch / cv2 stay loaded."""
from __future__ import annotations

import contextlib
import importlib
import os
import sys
import threading
import types

import numpy as np

REF = os.environ.get("LTB_REFERENCE", "")

_REF_MODULES = ("avatars", "avatars.base_avatar", "avatars.audio_features", "avatars.audio_features.base_asr", "registry", "utils",
                "utils.image", "utils.logger")
_PLUGIN_MODULES = ("livetalking_b200.plugin", "livetalking_b200.plugin.base_asr", "livetalking_b200.plugin.mel_asr",
                   "livetalking_b200.plugin.wav2lip_avatar", "livetalking_b200.plugin.whisper_asr",
                   "livetalking_b200.plugin.musetalk_avatar", "livetalking_b200.plugin.hubert_asr",
                   "livetalking_b200.plugin.ultralight_avatar")


def available() -> bool:
    return bool(REF) and os.path.isfile(os.path.join(REF, "avatars", "base_avatar.py"))


def _fake_modules():
    av = types.ModuleType("av")

    class _Frame:                                   # av.AudioFrame / av.VideoFrame: referenced by name only on this path
        @staticmethod
        def from_ndarray(*a, **k):
            raise RuntimeError("fake av module: transports are out of scope of this test")

    av.AudioFrame = av.VideoFrame = _Frame
    resampy = types.ModuleType("resampy")
    resampy.resample = lambda x, sr_orig, sr_new: x
    soundfile = types.ModuleType("soundfile")
    soundfile.read = lambda *a, **k: (np.zeros(0, np.float32), 16000)
    soundfile.write = lambda *a, **k: None
    return {"av": av, "resampy": resampy, "soundfile": soundfile}


def _namespace(reference: bool):
    base = sys.modules["avatars.base_avatar"]
    ns = types.SimpleNamespace(reference=reference, base_avatar=base, registry=importlib.import_module("registry"),
                               AudioFrameData=base.AudioFrameData, mirror_index=importlib.import_module("utils.image").mirror_index,
                               plugin_w2l=importlib.import_module("livetalking_b200.plugin.wav2lip_avatar"),
                               plugin_base_asr=importlib.import_module("livetalking_b200.plugin.base_asr"))
    ns.load_musetalk = lambda: importlib.import_module("livetalking_b200.plugin.musetalk_avatar")
    ns.load_ultralight = lambda: importlib.import_module("livetalking_b200.plugin.ultralight_avatar")
    return ns


@contextlib.contextmanager
def reference_runtime(workdir: str):
    """-> namespace(reference, base_avatar, registry, plugin_w2l, plugin_base_asr, load_musetalk, load_ultralight,
    AudioFrameData, mirror_index): the reference's own runtime when available(), else the host of tests/stubs.py."""
    old_cwd = os.getcwd()
    if not available():
        import stubs
        stubs.install()
        os.chdir(workdir)
        try:
            yield _namespace(reference=False)
        finally:
            os.chdir(old_cwd)
        return
    os.chdir(workdir)                              # utils/logger.py opens ./livetalking.log at import
    fakes = _fake_modules()
    managed = tuple(fakes) + _REF_MODULES + _PLUGIN_MODULES
    saved = {name: sys.modules.get(name) for name in managed}      # only these names are swapped; torch, cv2 ... stay loaded
    for name in _REF_MODULES + _PLUGIN_MODULES:
        sys.modules.pop(name, None)
    sys.modules.update(fakes)
    sys.path.insert(0, REF)
    try:
        base = importlib.import_module("avatars.base_avatar")
        assert os.path.samefile(base.__file__, os.path.join(REF, "avatars", "base_avatar.py")), "not the reference's module"
        yield _namespace(reference=True)
    finally:
        sys.path.remove(REF)
        os.chdir(old_cwd)
        for name in list(sys.modules):             # reference submodules imported on the way (e.g. avatars.audio_features.*)
            if name.split(".")[0] in ("avatars", "utils", "registry") or name in managed:
                sys.modules.pop(name, None)
        for name, mod in saved.items():
            if mod is not None:
                sys.modules[name] = mod
        import livetalking_b200
        if hasattr(livetalking_b200, "plugin") and "livetalking_b200.plugin" not in sys.modules:
            delattr(livetalking_b200, "plugin")


class RecordingSink:
    """Stands in for streamout.* (base_avatar.py:115-124): records what process_frames pushes, in order."""

    def __init__(self):
        self.frames, self.audio, self.lock = [], [], threading.Lock()
        self.started = self.stopped = False

    def start(self):
        self.started = True

    def stop(self):
        self.stopped = True

    def get_buffer_size(self):
        return 0                                   # never throttle render() (base_avatar.py:491-494)

    def push_video_frame(self, frame):
        assert frame.flags.writeable and frame.flags.c_contiguous and frame.dtype == np.uint8
        with self.lock:
            self.frames.append(np.array(frame, copy=True))

    def push_audio_frame(self, frame_i16, userdata):
        with self.lock:
            self.audio.append((np.array(frame_i16, copy=True), dict(userdata or {})))


class NullTTS:
    def render(self, quit_event):                  # base_avatar.py:473
        pass

    def flush_talk(self):
        pass


def make_opt(batch_size=4, **kw):
    opt = types.SimpleNamespace(fps=25, l=10, r=10, batch_size=batch_size, sessionid=0, tts="none", transport="none", customopt=[],
                                W=0, H=0)
    for k, v in kw.items():
        setattr(opt, k, v)
    return opt


def spy_audio_frames(asr, log: list):
    """Record every chunk run_step pulls (render thread only), so that the test can replay the exact stream."""
    orig = asr.get_audio_frame

    def wrapped():
        f = orig()
        log.append(f)
        return f

    asr.get_audio_frame = wrapped


def feed_bursts(avatar, bursts, chunk=320, seed=0, gap_s=0.25):
    """Speech bursts separated by pauses (-> the 10 ms get_audio_frame timeout synthesises silence in between)."""
    import time
    rng = np.random.default_rng(seed)
    cid = 0
    for n in bursts:
        for _ in range(n):
            t = np.arange(chunk) / 16000.0
            tone = 0.3 * np.sin(2 * np.pi * rng.uniform(150, 3000) * t + rng.uniform(0, 6.28))
            data = (tone + 0.05 * rng.standard_normal(chunk)).astype(np.float32)
            avatar.put_audio_frame(data, {"cid": cid})
            cid += 1
        asr = getattr(avatar, "asr", None) or avatar.avatar.asr
        t0 = time.time()
        while not asr.queue.empty() and time.time() - t0 < 30:      # let the session drain the burst, however loaded the box is ...
            time.sleep(0.01)
        time.sleep(gap_s)                                            # ... then stay silent for a while
