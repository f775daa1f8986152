"""Fake-module injection for importing the plugin outside LiveTalking (the technique of the reference's own
tests/test_asr_server.py:57-72): stand-ins for avatars.base_avatar / registry / utils.* so that livetalking_b200.plugin.*
can be imported and run under a render loop without a LiveTalking checkout (and without av/aiortc/resampy...)."""
import logging
import queue
import sys
import threading
import time
import types
from dataclasses import dataclass, field
from queue import Queue

import numpy as np


def install():
    if "avatars.base_avatar" in sys.modules and getattr(sys.modules["avatars.base_avatar"], "_LTB_STUB", False):
        return
    avatars = types.ModuleType("avatars")
    avatars.__path__ = []
    base = types.ModuleType("avatars.base_avatar")
    base._LTB_STUB = True

    @dataclass
    class AudioFrameData:                       # avatars/base_avatar.py:56-61
        data: np.ndarray
        type: int = 0
        userdata: dict = field(default_factory=dict)

    class BaseAvatar:
        """The host side of a LiveTalking session as the plugin meets it (avatars/base_avatar.py): the attributes the plugin
        reads, the audio entry points, custom-audio playback and the three-thread render loop.  render() calls asr.run_step on
        the calling thread; inference() pairs every feature batch with its 2B audio chunks and skips the model for an
        all-silent batch; process_frames() pastes each frame (or takes the avatar / custom frame when the frame's own two
        chunks are silent), stamps the watermark and pushes video and audio to self.output.  The caller sets self.output
        and self.tts."""

        def __init__(self, opt):
            self.opt = opt
            self.sample_rate = 16000
            self.chunk = self.sample_rate // (opt.fps * 2)
            self.sessionid = getattr(opt, "sessionid", 0)
            self.speaking = False
            self.custom_audiotype = 0                # 0 speech, 1 silence, > 1 a custom clip
            self.custom_img_cycle, self.custom_audio_cycle, self.custom_audio_index, self.custom_index = {}, {}, {}, {}
            self.batch_size = opt.batch_size
            self.res_frame_queue = Queue(self.batch_size * 2)

        def get_avatar_length(self):
            return len(self.frame_list_cycle) if hasattr(self, "frame_list_cycle") else 1

        def put_audio_frame(self, audio_chunk, datainfo=None):
            self.asr.put_audio_frame(audio_chunk, {} if datainfo is None else datainfo)

        def flush_talk(self):
            if hasattr(self, "tts"):
                self.tts.flush_talk()
            self.asr.flush_talk()
            self.custom_audiotype = 0

        def init_customindex(self):
            self.custom_audiotype = 0
            for counters in (self.custom_audio_index, self.custom_index):
                for k in counters:
                    counters[k] = 0

        def get_custom_audio_stream(self, audiotype):
            """Next chunk of custom clip `audiotype` (the last one may be short); back to silence once the clip is used up."""
            start = self.custom_audio_index[audiotype]
            clip = self.custom_audio_cycle[audiotype]
            self.custom_audio_index[audiotype] = start + self.chunk
            if start + self.chunk >= clip.shape[0]:
                self.custom_audiotype = 1
            return clip[start:start + self.chunk]

        def inference(self, quit_event):
            n, index, was_speaking = self.get_avatar_length(), 0, False
            while not quit_event.is_set():
                try:
                    feats = self.asr.feat_queue.get(block=True, timeout=1)
                except queue.Empty:
                    continue
                audio = [self.asr.output_queue.get() for _ in range(2 * self.batch_size)]
                speaking = any(a.type == 0 for a in audio)
                if not speaking:
                    results = [None] * self.batch_size
                else:
                    if not was_speaking and self.custom_index.get(1) is not None:
                        index = 0                    # speech after a custom silent clip restarts the avatar cycle
                    results = self.inference_batch(index, feats)
                for i, res in enumerate(results):
                    self.res_frame_queue.put((res, audio[2 * i:2 * i + 2], mirror_index(n, index)))
                    index += 1
                was_speaking = speaking

        def process_frames(self, quit_event):
            import cv2
            self.output.start()
            while not quit_event.is_set():
                try:
                    res, audio, idx = self.res_frame_queue.get(block=True, timeout=1)
                except queue.Empty:
                    continue
                if audio[0].type != 0 and audio[1].type != 0:
                    self.speaking = False
                    kind = audio[0].type
                    if self.custom_index.get(kind) is not None:
                        imgs = self.custom_img_cycle[kind]
                        frame = imgs[mirror_index(len(imgs), self.custom_index[kind])]
                        self.custom_index[kind] += 1
                    else:
                        frame = self.frame_list_cycle[idx]     # drawn on in place: avatar frames must be writable
                else:
                    self.speaking = True
                    try:
                        frame = self.paste_back_frame(res, idx)
                    except Exception as e:                      # noqa: BLE001  one bad frame must not end the session
                        logging.getLogger("livetalking-stub").warning("paste_back_frame error: %r", e)
                        continue
                cv2.putText(frame, "LiveTalking", (10, 20), cv2.FONT_HERSHEY_SIMPLEX, 0.3, (128, 128, 128), 1)
                self.output.push_video_frame(frame)
                for a in audio:
                    self.output.push_audio_frame((a.data * 32767).astype(np.int16), a.userdata)
            self.output.stop()

        def render(self, quit_event):
            self.quit_event = quit_event
            self.init_customindex()
            self.tts.render(quit_event)
            stop_inference, stop_frames = threading.Event(), threading.Event()
            t_inference = threading.Thread(target=self.inference, args=(stop_inference,))
            t_frames = threading.Thread(target=self.process_frames, args=(stop_frames,))
            t_inference.start()
            t_frames.start()
            while not quit_event.is_set():
                self.asr.run_step()
                backlog = self.output.get_buffer_size() if hasattr(self.output, "get_buffer_size") else 0
                if backlog >= 5:                     # the transport is behind: let it drain
                    time.sleep(0.032 * backlog)
            stop_inference.set()                     # frames keeps draining until inference has stopped
            t_inference.join()
            stop_frames.set()
            t_frames.join()

    base.AudioFrameData = AudioFrameData
    base.BaseAvatar = BaseAvatar
    registry = types.ModuleType("registry")
    registry._REG = {}

    def register(category, name):
        def deco(cls):
            registry._REG.setdefault(category, {})[name] = cls
            return cls
        return deco

    def create(category, name, **kw):
        return registry._REG[category][name](**kw)

    registry.register, registry.create = register, create
    utils = types.ModuleType("utils")
    utils.__path__ = []
    image = types.ModuleType("utils.image")

    def mirror_index(size, index):              # utils/image.py:26-32
        turn, res = index // size, index % size
        return res if turn % 2 == 0 else size - res - 1

    def read_imgs(paths):
        import cv2
        return [cv2.imread(p) for p in paths]

    image.mirror_index, image.read_imgs = mirror_index, read_imgs
    logger_mod = types.ModuleType("utils.logger")
    logger_mod.logger = logging.getLogger("livetalking-stub")
    for name, mod in (("avatars", avatars), ("avatars.base_avatar", base), ("registry", registry), ("utils", utils),
                      ("utils.image", image), ("utils.logger", logger_mod)):
        sys.modules[name] = mod


class Opt:
    def __init__(self, batch_size=4, fps=25, l=10, r=10, **kw):
        self.batch_size, self.fps, self.l, self.r = batch_size, fps, l, r
        self.sessionid = 0
        for k, v in kw.items():
            setattr(self, k, v)


def run_three_threads(avatar, sink, quit_event):
    """Test harness for boxes without the reference checkout: drives a plugin avatar with the SAME thread roles and queue
    hand-offs as the reference's render() (avatars/base_avatar.py:469-501) — thread 1 calls asr.run_step in a loop, thread 2
    pairs one feature batch with 2*B audio chunks, skips the model for an all-silent batch and calls inference_batch, thread 3
    calls paste_back_frame (or takes the plain avatar frame for a silent frame) and pushes to the sink.  Blocks until
    quit_event is set.  (tests/test_base_avatar_threads.py runs the real render() where the checkout exists.)"""
    import queue
    import threading

    B, n = avatar.batch_size, len(avatar.frame_list_cycle)
    mirror = sys.modules["utils.image"].mirror_index
    stop2, stop3 = threading.Event(), threading.Event()

    def infer_loop():
        index = 0
        while not stop2.is_set():
            try:
                feats = avatar.asr.feat_queue.get(block=True, timeout=0.5)
            except queue.Empty:
                continue
            audio = [avatar.asr.output_queue.get() for _ in range(2 * B)]
            if all(a.type != 0 for a in audio):
                results = [None] * B
            else:
                results = list(avatar.inference_batch(index, feats))
            for i, r in enumerate(results):
                avatar.res_frame_queue.put((r, audio[2 * i:2 * i + 2], mirror(n, index)))
                index += 1

    def frame_loop():
        while not stop3.is_set():
            try:
                res, audio, idx = avatar.res_frame_queue.get(block=True, timeout=0.5)
            except queue.Empty:
                continue
            if audio[0].type != 0 and audio[1].type != 0:
                frame = np.array(avatar.frame_list_cycle[idx], copy=True)
            else:
                frame = avatar.paste_back_frame(res, idx)
            sink.push_video_frame(frame)
            for a in audio:
                sink.push_audio_frame((np.asarray(a.data) * 32767).astype(np.int16), a.userdata)

    t2, t3 = threading.Thread(target=infer_loop), threading.Thread(target=frame_loop)
    t2.start()
    t3.start()
    while not quit_event.is_set():
        avatar.asr.run_step()
    stop2.set()
    t2.join()
    stop3.set()
    t3.join()
