#!/usr/bin/env python
"""Benchmark of the lip-sync hot path (BASELINE.json metric: lip-sync frames/sec, wav2lip256, 256^2, batch 16).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

One "step" = one pass of the hot path over one batch of 16 frames:
    mel windows (resident PCM) -> wav2lip256 forward -> paste-back of 16 frames into 720p frames.
`value`  : device-timed throughput with every input already resident in HBM.  CUDA events on the engine's stream; the stream
           is GATED (a spin kernel holds it) until all K steps are enqueued, so the device time contains no Python launch jitter.
`e2e`    : the same metric through the C ABI with HOST buffers: pinned PCM -> H2D -> mel -> forward -> paste -> D2H of the 16
           composited frames, every step (ltb_w2l_step_e2e_async, copies pipelined on a second stream).
Extra keys on the same JSON line (all measured in this run):
  roofline          dominant kernels (tcgen05 convs) against the MEASURED burst tensor peak; `sustained` inside it = a >= 2 s
                    forward-only loop against the measured sustained peak
  sustained         the same step loop run for >= 3 s with the clock / power trace
  e2e_plugin        fps through the reference-facing hooks exactly as avatars/base_avatar.py calls them:
                    MelASR features -> LipReal.inference_batch -> 16 x paste_back_frame (host arrays in and out)
  e2e_plugin_threads the same hooks under the reference's three-thread driving (one session, un-paced)
  sessions32        BASELINE configs[3]: 32 concurrent sessions on this GPU, each batch 16 (per-session fps, arena bytes)
  cross_session     the batching scheduler's engine call: 16 slots from 8 different sessions in one forward + paste launch
  musetalk          BASELINE configs[2] (MuseTalk 256x256 batch 8, fp16): value / e2e / roofline of its own
  musetalk512       BASELINE configs[4] (512x512 = 64x64 latents, batch 8) + 8 CONCURRENT sessions per GPU; every rank at N > 1
  torch_eager_b200  the reference network in stock PyTorch on THIS GPU (fp32 = TF32 cuDNN as the reference runs it, and fp16
                    channels_last): the existing Blackwell path to beat
  cpu_baseline      the oracle port on the host cores (N = 1 only)
Under torchrun (N > 1) every rank drives its own GPU with its own session (sessions are independent: weak scaling);
weights are packed on rank 0 and broadcast once with NCCL (the only collective of the design); each rank pins itself to
its GPU's NUMA node; per-rank step times are reported (`per_rank_ms`).
`--impl reference` times the reference's own CPU implementation of the path (the oracle port: CPU PyTorch fp32 +
numpy mel + OpenCV-exact paste) on the host cores; rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "lip-sync frames/sec (wav2lip256, 256x256, batch 16, mel + U-Net fwd + paste-back)"
GFLOP_PER_FRAME = 55.58           # BASELINE.md §2 / SURVEY §8(d): 27.789 GMAC, hooks on the reference module
MT_GFLOP_ONLINE = {32: 800.0, 64: 3314.6}    # UNet + VAE decode per frame at 32x32 / 64x64 latents (SURVEY §8(d))
MT_GFLOP_WHISPER_STEP = 37.0
BATCH = 16
SL, SR, FPS = 10, 10, 25   # opt.l, opt.r (20 ms chunks), opt.fps
FRAME_H, FRAME_W = 720, 1280
BBOX = (200, 520, 480, 800)
WORKLOAD = ("wav2lip256 batch 16, 256x256, 1xB200 per rank, 60 s synthetic 16 kHz sine audio, "
            "mel + U-Net fwd + paste-back into 720p frames (BASELINE.json configs[1])")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        burst = float(d.get("bf16_tflops", 1661.3))
        return {"burst": burst, "sustained": float(d.get("bf16_tflops_sustained", burst)), "hbm": float(d["hbm_gbs"]),
                "src": "MEASURED_PEAKS.json (cuBLAS bf16: best-of-10 burst / 4 s sustained)"}
    return {"burst": 1650.0, "sustained": 1400.0, "hbm": 6650.0, "src": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------ clocks / placement
class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region.  In-process NVML polling (10 ms) when pynvml is there —
    no child process competing with the launch thread — else `nvidia-smi -lms 100`."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device: int):
        self.device, self.samples, self._stop, self.t, self.h, self.nv = device, [], threading.Event(), None, None, None
        self.proc = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(device))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(device: int) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [x for x in vis.split(",") if x.strip() != ""]
            if device < len(ids) and ids[device].strip().isdigit():
                return int(ids[device])
        return device

    def _poll(self):
        nv = self.nv
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM),
                                     nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0, int(reasons(self.h))))
            except Exception:
                pass
            self._stop.wait(0.01)

    def start(self):
        if self.nv is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        import subprocess
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                                          str(self._physical_index(self.device))], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read_smi, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read_smi(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                bits = sum(b for b, v in zip((0x8, 0x40, 0x20, 0x4), f[3:7]) if v.lower().startswith("active"))
                self.samples.append((float(f[0]), float(f[1]), float(f[2]), bits))
            except Exception:
                continue

    def stop(self):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
        self._stop.set()
        if self.t is not None:
            self.t.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"], "samples": 0}
        sm = [s[0] for s in self.samples]
        bits = 0
        for s in self.samples:
            bits |= s[3]
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(min(sm)), "sm_max_mhz": float(max(s[1] for s in self.samples)),
                "power_w_max": round(max(s[2] for s in self.samples), 1), "reasons": sorted(n for b, n in self.REASONS.items() if bits & b),
                "samples": len(sm), "how": "pynvml 10 ms" if self.nv is not None else "nvidia-smi -lms 100"}


def pin_to_gpu_numa(local: int):
    """Bind this rank to the CPUs of its GPU's NUMA node (ranks 4-7 of an 8-GPU box sit on node 1)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(ClockSampler._physical_index(local))
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None
    return None


def step_pcm(audio: np.ndarray, step: int, batch: int = BATCH) -> np.ndarray:
    """The (l + r + 2B) chunk buffer MelASR.run_step would hold at `step` of the 60 s stream (wraps around)."""
    n = (SL + SR + 2 * batch) * 320
    start = (step * 2 * batch * 320) % (audio.size - n)
    return audio[start:start + n]


# ------------------------------------------------------------------------------------------------ reference arm / CPU baseline
class CpuPath:
    """The reference's own CPU implementation of the path (oracle port, see oracle/__init__.py), timed on host cores.
    A 16-frame step is run as 8 reference-style sub-batches of 2 frames (CPU PyTorch conv is pathological at B = 16)."""
    SUB = 2

    def __init__(self, threads: int):
        import torch
        from livetalking_b200 import synth
        from oracle import mel_ref, paste_ref
        from oracle import wav2lip_ref as R
        self.torch, self.mel_ref, self.paste_ref, self.R = torch, mel_ref, paste_ref, R
        self.sd = {k: torch.from_numpy(np.asarray(v)) for k, v in synth.random_state_dict(0).items()}
        for k in list(self.sd):
            if k.endswith("running_var"):
                self.sd[k.replace("running_var", "num_batches_tracked")] = torch.tensor(1)
        self.faces, self.frames, self.coords = synth.synthetic_avatar(n=4, H=FRAME_H, W=FRAME_W, bbox=BBOX)
        self.audio = synth.sine_audio(5.0)
        # the reference's PyTorch CPU path does not scale to all cores of a 128-core host: calibrate the thread count
        best_t, best = threads, None
        for cand in sorted({threads, min(threads, 64), min(threads, 32), min(threads, 16)}, reverse=True):
            torch.set_num_threads(cand)
            self.frames_of(0, self.SUB)
            t0 = time.perf_counter()
            self.frames_of(1, self.SUB)
            d = time.perf_counter() - t0
            if best is None or d < best:
                best, best_t = d, cand
        torch.set_num_threads(best_t)
        self.threads = best_t

    def frames_of(self, step: int, B: int):
        torch, R, P = self.torch, self.R, self.paste_ref
        n = (SL + SR + 2 * B) * 320
        pcm = self.audio[(step * 640) % (self.audio.size - n):][:n]
        mel = self.mel_ref.mel_step(pcm, B, SL, SR, FPS)                                   # MelASR.run_step
        img = P.w2l_build_batch(list(self.faces), step * B, B)                             # inference_batch glue
        out = R.wav2lip_forward(self.sd, torch.from_numpy(mel.astype(np.float32)).reshape(B, 1, 80, 16), torch.from_numpy(img))
        pred = out.numpy().transpose(0, 2, 3, 1) * 255.0
        for i in range(B):                                                                 # paste_back_frame
            idx = P.mirror_index(len(self.faces), step * B + i)
            P.w2l_paste_back(pred[i], self.frames[idx], self.coords[idx])

    def step16(self, step: int):
        for k in range(BATCH // self.SUB):
            self.frames_of(step * (BATCH // self.SUB) + k, self.SUB)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    cpu = CpuPath(cores)
    for w in range(args.warmup):
        cpu.step16(w)
    t0 = time.perf_counter()
    for k in range(args.steps):
        cpu.step16(args.warmup + k)
    dt = time.perf_counter() - t0
    fps = BATCH * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": round(fps, 4), "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(1000.0 * dt / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": BATCH, "sessions_per_gpu": 1, "parallelism": "session-sharded x1",
                   "cpu_arm": "same 16-frame step, run as 8 sub-batches of 2 frames (CPU PyTorch conv is pathological at B = 16)"},
        "cpu_baseline": {"value": round(fps, 4), "unit": "frames/s", "cores": cpu.threads, "kind": "port", "host_cores": cores,
                         "sample": f"{args.steps} steps x 16 frames: numpy mel + CPU PyTorch fp32 wav2lip256 + paste-back (oracle port)"},
        "e2e": {"value": round(fps, 4), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ helpers of our arm
class Gate:
    """Holds a CUDA stream with a spin kernel while the host enqueues the timed work behind it."""

    def __init__(self, torch, stream):
        self.torch, self.stream = torch, stream

    def hold(self, ms: float = 8.0):
        with self.torch.cuda.stream(self.stream):
            self.torch.cuda._sleep(int(ms * 1.9e6))


def timed_steps(torch, stream, gate, enqueue, steps, extra_streams=()):
    """ev0 | K x enqueue | ev1 on `stream`, gated so that the steps are queued before ev0 fires.  -> ms"""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gate.hold(8.0 if steps <= 64 else 20.0)
    for st in extra_streams:                       # other sessions' streams start together with the gated one
        st.wait_stream(stream)
    ev0.record(stream)
    for k in range(steps):
        enqueue(k)
    for st in extra_streams:
        stream.wait_stream(st)
    ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1)


def torch_eager_b200(torch, steps=10):
    """The reference network (oracle restatement, bit-pinned to the unmodified module) in stock PyTorch on this GPU.
    A baseline leg, like cpu_baseline: nothing of the product path goes through it."""
    from livetalking_b200 import synth
    from oracle import wav2lip_ref as R
    out = {}
    sd32 = {k: torch.from_numpy(np.asarray(v)).cuda() for k, v in synth.random_state_dict(0).items()}
    g = torch.Generator(device="cuda").manual_seed(0)
    mel = torch.randn(BATCH, 1, 80, 16, device="cuda", generator=g)
    img = torch.rand(BATCH, 6, 256, 256, device="cuda", generator=g)
    for name, dt, cl in (("fp32_tf32", torch.float32, False), ("fp16_channels_last", torch.float16, True)):
        sd = {k: (v.to(dt) if v.is_floating_point() else v) for k, v in sd32.items()}
        if cl:
            sd = {k: (v.contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v) for k, v in sd.items()}
        m, x = mel.to(dt), img.to(dt)
        if cl:
            x = x.contiguous(memory_format=torch.channels_last)
        with torch.no_grad():
            for _ in range(3):
                R.wav2lip_forward(sd, m, x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                R.wav2lip_forward(sd, m, x)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"frames_per_s": round(BATCH * 1000.0 / ms, 1), "forward_ms": round(ms, 3)}
    out["what"] = ("wav2lip256 forward only (no mel, no paste), B=16, stock PyTorch %s eager on this GPU; cudnn.allow_tf32=%s (PyTorch default, "
                   "what the reference's own GPU path runs)" % (torch.__version__, torch.backends.cudnn.allow_tf32))
    return out


def plugin_e2e(engine, model, av_lists, audio, steps, warmup):
    """fps through the hooks the reference calls (avatars/base_avatar.py:366-376, 433; avatars/audio_features/mel.py:34-67):
    features of the host PCM buffer -> LipReal.inference_batch(index, [B x (80,16)]) -> paste_back_frame(res, idx) x B.
    Serial on one thread (the reference overlaps the three on three threads: this is the conservative number)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import stubs                                                    # stand-in for avatars.base_avatar / registry / utils (no reference checkout here)
    stubs.install()
    from livetalking_b200.plugin import wav2lip_avatar as P
    mirror = sys.modules["utils.image"].mirror_index
    frames, faces, coords = av_lists
    payload = P.make_avatar(frames, faces, coords)
    lip = P.LipReal(stubs.Opt(batch_size=BATCH, fps=FPS, l=SL, r=SR), model, payload)
    n = len(frames)

    def one(k, index):
        mel = lip.engine_session.mel_step(step_pcm(audio, k))       # MelASR.run_step's feature call
        res = lip.inference_batch(index, [mel[i] for i in range(BATCH)])
        out = None
        for i, r in enumerate(res):
            out = lip.paste_back_frame(r, mirror(n, index + i))
        return out

    for k in range(warmup):
        one(k, k * BATCH)
    t0 = time.perf_counter()
    for k in range(steps):
        last = one(k, k * BATCH)
    dt = time.perf_counter() - t0
    assert last.shape == (FRAME_H, FRAME_W, 3) and last.flags.writeable
    lip.engine_session.close()
    payload.engine_avatar.close()
    return {"value": round(BATCH * steps / dt, 1), "unit": "frames/s", "ms_per_step": round(1000.0 * dt / steps, 3),
            "how": "MelASR features + LipReal.inference_batch + 16 x paste_back_frame, host numpy in/out, one thread, wall clock",
            "d2h_bytes_per_step": BATCH * FRAME_H * FRAME_W * 3}


def plugin_threads(engine, model, av_lists, n_frames=480):
    """The same hooks driven the way the reference drives them: three threads (asr.run_step | inference_batch | paste_back_frame,
    avatars/base_avatar.py:469-501) with the reference's bounded queues, speech fed as fast as the session drains it, frames
    pushed to a counting sink.  Un-paced throughput of ONE session through the full host pipeline."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import stubs
    stubs.install()
    from livetalking_b200.plugin import wav2lip_avatar as P
    frames, faces, coords = av_lists
    lip = P.LipReal(stubs.Opt(batch_size=BATCH, fps=FPS, l=SL, r=SR), model, P.make_avatar(frames, faces, coords))

    class Sink:
        n, t_first, t_last = 0, None, None

        def push_video_frame(self, f):
            now = time.perf_counter()
            if self.t_first is None:
                self.t_first = now
            self.t_last = now
            self.n += 1

        def push_audio_frame(self, a, u):
            pass

    sink, quit_event = Sink(), threading.Event()
    rng = np.random.default_rng(0)
    chunk = (0.2 * rng.standard_normal(320)).astype(np.float32)

    def feeder():
        while not quit_event.is_set():
            if lip.asr.queue.qsize() < 4 * BATCH:
                for _ in range(2 * BATCH):
                    lip.asr.put_audio_frame(chunk, {})
            else:
                time.sleep(0.0005)

    th = threading.Thread(target=stubs.run_three_threads, args=(lip, sink, quit_event))
    fd = threading.Thread(target=feeder)
    fd.start()
    th.start()
    t0 = time.time()
    while sink.n < n_frames + 4 * BATCH and time.time() - t0 < 60:
        time.sleep(0.005)
    quit_event.set()
    th.join(timeout=30)
    fd.join(timeout=5)
    n, dt = sink.n, (sink.t_last - sink.t_first) if sink.n > 1 else 1.0
    lip.engine_session.close()
    return {"value": round((n - 1) / dt, 1), "unit": "frames/s", "frames": n,
            "how": "one session, three threads + bounded queues as avatars/base_avatar.py:469-501 (run_step | inference_batch | paste_back_frame), "
                   "speech fed on demand, counting sink, wall clock between first and last frame"}


def sessions_leg(torch, engine, model, av, audio, n_sessions, steps, dist=None, world=1):
    """BASELINE configs[3]: n concurrent sessions on one GPU, each batch 16 on its own stream / arena."""
    free0 = torch.cuda.mem_get_info()[0]
    ss = [engine.W2LSession(model, av, BATCH, SL, SR, FPS) for _ in range(n_sessions)]
    arena = (free0 - torch.cuda.mem_get_info()[0]) / n_sessions
    for s_ in ss:
        s_.set_pcm(step_pcm(audio, 0))
    streams = [torch.cuda.ExternalStream(s_.cuda_stream) for s_ in ss]
    g = Gate(torch, streams[0])
    idx = [0]

    def step_all(_k):
        for s_ in ss:
            s_.step_async(idx[0])
        idx[0] += BATCH

    for k in range(3):
        step_all(k)
    torch.cuda.synchronize()
    ms = timed_steps(torch, streams[0], g, step_all, steps, streams[1:])
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    fps = world * n_sessions * BATCH * steps / (ms / 1000.0)
    for s_ in ss:
        s_.close()
    return {"sessions_per_gpu": n_sessions, "n_gpus": world, "total_sessions": world * n_sessions, "value": round(fps, 1), "unit": "frames/s",
            "per_session_fps": round(fps / (world * n_sessions), 1),
            "realtime_sessions_at_25fps": int(fps // 25), "arena_bytes_per_session": int(arena), "ms_per_round": round(ms / steps, 3),
            "what": "BASELINE configs[3] on one GPU: every session has its own stream, activation arena and CUDA graph; weights / avatar shared"}


def cross_session_leg(engine, model, steps):
    """SURVEY §8 f1: the batching scheduler's engine call — 16 slots taken from 8 DIFFERENT sessions' avatars (2 frames each,
    as sessions running with batch_size 2 would submit them), one forward + paste launch, frames back on the host."""
    from livetalking_b200 import synth
    n_av, per = 8, 2
    avs = []
    for a in range(n_av):
        faces, frames, coords = synth.synthetic_avatar(n=8, H=FRAME_H, W=FRAME_W, bbox=BBOX, seed=100 + a)
        avs.append(engine.W2LAvatar(faces, frames, coords))
    mux = engine.W2LSession(model, avs[0], BATCH, SL, SR, FPS, slots=True)
    rng = np.random.default_rng(0)
    mels = np.clip(rng.standard_normal((BATCH, 80, 16)), -4, 4).astype(np.float32)
    out = engine.PinnedBuffer((BATCH, FRAME_H, FRAME_W, 3), np.uint8)

    def one(k):
        reqs = [(avs[i // per], (k * per + i % per) % 8, mels[i]) for i in range(BATCH)]
        return mux.infer_slots(reqs, out=out.array)

    for k in range(3):
        one(k)
    t0 = time.perf_counter()
    for k in range(steps):
        one(k)
    dt = time.perf_counter() - t0
    mux.close()
    for a in avs:
        a.close()
    return {"value": round(BATCH * steps / dt, 1), "unit": "frames/s", "ms_per_batch": round(1000.0 * dt / steps, 3), "slots": BATCH,
            "sessions_in_batch": n_av, "sessions_at_25fps": int(BATCH * steps / dt // 25),
            "how": "ltb_w2l_infer_slots: 16 slots from 8 avatars per call, host mel windows in, 16 composited 720p frames out (pinned), synchronous"}


class MuseTalkBench:
    """MuseTalk legs.  The model is built ONCE per rank; with N > 1 ranks the synthetic state dicts are generated on rank 0 and
    shipped with one NCCL broadcast (BASELINE configs[4]: "NCCL weight-broadcast init"), exactly like the wav2lip blob."""

    def __init__(self, torch, dist, world, rank):
        from livetalking_b200 import configs, synth
        from livetalking_b200.musetalk import MuseTalkModel
        from livetalking_b200.ops import Ctx
        from livetalking_b200.whisper import WhisperEncoder
        self.torch, self.dist, self.world, self.rank = torch, dist, world, rank
        self.ucfg, self.vcfg = configs.UNetConfig(), configs.VAEConfig()
        t0 = time.time()
        sds = None
        if rank == 0:
            sds = [synth.random_unet_state_dict(self.ucfg), synth.random_vae_state_dict(self.vcfg), synth.random_whisper_state_dict()]
        bcast_s = 0.0
        if world > 1:
            tb = time.time()
            sds = self._broadcast_state_dicts(sds)
            bcast_s = time.time() - tb
        self.ctx = Ctx()
        self.net = MuseTalkModel(self.ctx, sds[0], sds[1], self.ucfg, self.vcfg, with_encoder=False)
        self.wenc = WhisperEncoder(self.ctx, sds[2])
        self.load_s, self.bcast_s = time.time() - t0, bcast_s
        self.audio = synth.sine_audio(10.0)

    def _broadcast_state_dicts(self, sds):
        """rank 0: [dict name -> float32 ndarray] x 3  ->  every rank, through ONE flat NCCL broadcast (+ a small metadata object)."""
        torch, dist = self.torch, self.dist
        meta = [None]
        if self.rank == 0:
            meta = [[[(k, tuple(np.asarray(v).shape)) for k, v in sd.items()] for sd in sds]]
        dist.broadcast_object_list(meta, src=0)
        total = sum(int(np.prod(shape)) if len(shape) else 1 for part in meta[0] for _k, shape in part)
        flat = torch.empty(total, dtype=torch.float32, device="cuda")
        if self.rank == 0:
            host = np.concatenate([np.asarray(v, np.float32).reshape(-1) for sd in sds for v in sd.values()])
            flat.copy_(torch.from_numpy(host))
        dist.broadcast(flat, 0)                    # ~3.7 GB over NVLink / NVSwitch
        if self.rank == 0:
            return sds
        host = flat.cpu().numpy()
        out, o = [], 0
        for part in meta[0]:
            d = {}
            for k, shape in part:
                n = int(np.prod(shape)) if len(shape) else 1
                d[k] = host[o:o + n].reshape(shape)
                o += n
            out.append(d)
        return out

    def _reduce_max(self, ms):
        if self.world == 1:
            return ms
        t = self.torch.tensor([ms], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def leg(self, args, peaks, hw: int, B: int = 8, n_sessions: int = 0, B_sess: int = 2, batch_sessions: int = 0):
        """BASELINE configs[2] (hw = 32: 256x256) / configs[4] (hw = 64: 512x512): the online path the reference runs per step
        (avatars/musetalk_avatar.py:130-164): Whisper features -> PE -> UNet -> VAE decode -> blend paste-back.
        n_sessions > 0: additionally that many CONCURRENT sessions per GPU (own stream / graph / buffers each, batch B_sess)."""
        from livetalking_b200 import synth
        from livetalking_b200.musetalk import MuseTalkAvatar, MuseTalkSession
        from livetalking_b200.whisper import WhisperFeatures
        torch, ctx, net, wenc, audio, world = self.torch, self.ctx, self.net, self.wenc, self.audio, self.world
        frames, masks, coords, crops, latents = synth.synthetic_musetalk_avatar(n=16, hw=hw, seed=self.rank)
        av = MuseTalkAvatar(ctx, frames, masks, coords, crops, latents)
        sess = MuseTalkSession(net, av, B, ctx=ctx)            # device-resident leg: one stream for the whole timed chain
        wf = WhisperFeatures(wenc, B, SL, SR, out=sess.audio_in, out_rows=64, ctx=ctx)
        wf.run_async(step_pcm(audio, 0, B))
        ctx.sync()
        stream = torch.cuda.ExternalStream(ctx.cuda_stream)
        gate = Gate(torch, stream)
        steps, warm = max(5, min(args.steps, 20)), max(3, min(args.warmup, 5))

        def online(k):
            wf.run_async(None)
            sess.step_async(k * B)

        for k in range(warm):
            online(k)
        ctx.sync()
        l0 = ctx.launch_count
        ms = self._reduce_max(timed_steps(torch, stream, gate, online, steps)) / steps
        launches = (ctx.launch_count - l0) // steps
        ms_net = timed_steps(torch, stream, gate, lambda k: sess.infer_async(k * B, None), steps) / steps
        # e2e: host PCM in, host frames out, through the session objects the plugin drives (own ctx per role, as deployed)
        sess2 = MuseTalkSession(net, av, B)
        wf2 = WhisperFeatures(wenc, B, SL, SR)
        S = hw * 8

        def e2e_one(k):
            feats = wf2.run(step_pcm(audio, k, B))                      # WhisperASR.run_step features (H2D PCM, D2H features)
            sess2.infer(k * B, feats, want_pred=False)                  # inference_batch (H2D features)
            return sess2.paste_batch(k * B)                             # B composited frames to the host

        for k in range(warm):
            e2e_one(k)
        t1 = time.perf_counter()
        for k in range(steps):
            e2e_one(k)
        e2e_ms = self._reduce_max((time.perf_counter() - t1) * 1000.0) / steps
        sess2.close()
        wf2.close()
        gf = MT_GFLOP_ONLINE[hw] * B + MT_GFLOP_WHISPER_STEP
        tf = gf / ms
        res = {
            "metric": "lip-sync frames/sec (MuseTalk %dx%d, batch %d, fp16: whisper + PE + UNet + VAE decode + blend paste-back)" % (S, S, B),
            "value": round(world * 1000.0 * B / ms, 2), "unit": "frames/s", "n_gpus": world, "ms_per_step": round(ms, 3), "steps": steps, "warmup": warm,
            "config": {"workload": "MuseTalk %dx%d batch %d, 1xB200 per rank, fp16 (BASELINE.json configs[%d]); online path of "
                                   "avatars/musetalk_avatar.py:130-164, latents pre-encoded" % (S, S, B, 2 if hw == 32 else 4),
                       "weights": "synthetic; rank 0 -> all ranks by one NCCL broadcast (%.1f s)" % self.bcast_s if world > 1 else "synthetic"},
            "e2e": {"value": round(world * 1000.0 * B / e2e_ms, 2), "unit": "frames/s", "h2d_bytes_per_step": int(wf2.n * 4 + B * 50 * 384 * 2),
                    "d2h_bytes_per_step": int(B * 50 * 384 * 2 + B * av.H * av.W * 3),
                    "how": "WhisperFeatures.run(host PCM) + MuseTalkSession.infer(host features) + paste_batch -> host frames, wall clock"},
            "roofline": {"bound": "tensor", "achieved": round(tf, 1), "peak": peaks["burst"], "unit": "TFLOP/s", "frac": round(tf / peaks["burst"], 4),
                         "frac_sustained_peak": round(tf / peaks["sustained"], 4), "algorithmic_gflop_per_step": round(gf, 1),
                         "unet_vae_only_ms": round(ms_net, 3), "traffic": None, "per_gpu": True},
            "gpu_launches_per_step": int(launches), "sessions_at_25fps_per_gpu": int((1000.0 * B / ms) // 25), "model_load_s": round(self.load_s, 1),
        }
        if n_sessions > 0:
            res["concurrent_sessions"] = self._sessions(args, av, hw, n_sessions, B_sess)
        if batch_sessions > 0:
            res["cross_session"] = self._cross_session(args, hw, batch_sessions, B)
            if self.world == 1:                        # single-GPU probe only (a one-sided failure must not strand other ranks in a collective)
                try:                                   # eight sessions per launch (batch 64): how far the batch-size lever goes
                    res["cross_session_x8"] = self._cross_session(args, hw, 2 * batch_sessions, B)
                except Exception as e:
                    res["cross_session_x8"] = {"error": repr(e)[:200]}
        return res

    def _cross_session(self, args, hw, G, Bs):
        """SURVEY 8(f) rank 1 for MuseTalk: G sessions x Bs frames as ONE graph of batch G*Bs (MuseTalkBatchSession): every group has
        its own avatar, frame index and Whisper feature window; aggregate frames/s of one GPU serving G sessions per launch."""
        from livetalking_b200 import synth
        from livetalking_b200.musetalk import MuseTalkAvatar, MuseTalkBatchSession
        from livetalking_b200.whisper import WhisperFeatures
        torch, ctx, world = self.torch, self.ctx, self.world
        avs = [MuseTalkAvatar(ctx, *synth.synthetic_musetalk_avatar(n=16, hw=hw, seed=100 + 8 * self.rank + g)) for g in range(G)]
        bs = MuseTalkBatchSession(self.net, hw, G, Bs, ctx=ctx)
        wfs = [WhisperFeatures(self.wenc, Bs, SL, SR, out=bs.audio_in_of[g], out_rows=64, ctx=ctx) for g in range(G)]
        for g, w_ in enumerate(wfs):
            w_.run_async(step_pcm(self.audio, g, Bs))
        ctx.sync()
        stream = torch.cuda.ExternalStream(ctx.cuda_stream)
        gate = Gate(torch, stream)
        steps = max(5, min(args.steps, 20))

        def one(k):
            for w_ in wfs:
                w_.run_async(None)                    # every session's own Whisper window, every round
            bs.step_async([(avs[g], k * Bs + 3 * g, None) for g in range(G)])

        for k in range(3):
            one(k)
        ctx.sync()
        ms = self._reduce_max(timed_steps(torch, stream, gate, one, steps)) / steps
        fps = 1000.0 * G * Bs / ms
        gf = MT_GFLOP_ONLINE[hw] * G * Bs + MT_GFLOP_WHISPER_STEP * G
        res = {"value": round(world * fps, 2), "unit": "frames/s", "n_gpus": world, "sessions_per_launch": G, "frames_per_session": Bs,
               "ms_per_round": round(ms, 3), "tflops": round(gf / ms, 1), "sessions_at_25fps_per_gpu": int(fps // 25),
               "what": "%d sessions x %d frames in ONE UNet + VAE graph (batch %d), per-session avatar / index / Whisper window, "
                       "blend paste-back per session; device-timed, inputs resident" % (G, Bs, G * Bs)}
        for w_ in wfs:
            w_.close()
        bs.close()
        return res

    def _sessions(self, args, av, hw, n_sessions, B):
        """n concurrent MuseTalk sessions on this GPU (BASELINE configs[4]: 8 sessions per GPU): every session owns its stream,
        CUDA graph and buffers (MuseTalkSession + WhisperFeatures with their own Ctx), weights and avatar are shared."""
        from livetalking_b200.musetalk import MuseTalkSession
        from livetalking_b200.whisper import WhisperFeatures
        torch, world = self.torch, self.world
        free0 = torch.cuda.mem_get_info()[0]
        ss = [MuseTalkSession(self.net, av, B) for _ in range(n_sessions)]
        wfs = [WhisperFeatures(self.wenc, B, SL, SR, out=s_.audio_in, out_rows=64, ctx=s_.ctx) for s_ in ss]
        per_sess = (free0 - torch.cuda.mem_get_info()[0]) / n_sessions
        for w_ in wfs:
            w_.run_async(step_pcm(self.audio, 0, B))
        torch.cuda.synchronize()
        streams = [torch.cuda.ExternalStream(s_.ctx.cuda_stream) for s_ in ss]
        gate = Gate(torch, streams[0])
        steps = max(5, min(args.steps, 20))

        def step_all(k):
            for s_, w_ in zip(ss, wfs):
                w_.run_async(None)
                s_.step_async(k * B)

        for k in range(3):
            step_all(k)
        torch.cuda.synchronize()
        ms = self._reduce_max(timed_steps(torch, streams[0], gate, step_all, steps, streams[1:])) / steps
        fps = n_sessions * B * 1000.0 / ms
        for w_ in wfs:
            w_.close()
        for s_ in ss:
            s_.close()
        return {"sessions_per_gpu": n_sessions, "batch_per_session": B, "n_gpus": world, "value": round(world * fps, 2), "unit": "frames/s",
                "per_session_fps": round(fps / n_sessions, 2), "ms_per_round": round(ms, 3), "bytes_per_session": int(per_sess),
                "what": "%d concurrent %dx%d sessions per GPU, each batch %d on its own stream / graph" % (n_sessions, hw * 8, hw * 8, B)}

    def close(self):
        self.ctx.close()


def ultralight_leg(torch, args):
    """SURVEY 8 row f4: the UltraLight avatar path at the reference's batch size — HuBERT-large features over the (l + r + 2B)-chunk
    window (avatars/audio_features/hubert.py:27-51) + per-avatar U-Net at 160x160 (avatars/ultralight/unet.py) + paste-back into
    720p frames (avatars/ultralight_avatar.py:141-184).  Random-init weights of the real architectures, synthetic avatar."""
    from livetalking_b200 import synth
    from livetalking_b200.hubert import HubertEncoder, HubertFeatures, gflop_per_window
    from livetalking_b200.ops import Ctx
    from livetalking_b200.ultralight import UltraLightAvatar, UltraLightModel, UltraLightSession, unet_gflop_per_frame
    B = BATCH
    t0 = time.time()
    ctx = Ctx()
    enc = HubertEncoder(ctx, synth.random_hubert_state_dict())
    net = UltraLightModel(ctx, synth.random_ultralight_state_dict())
    frames, faces, coords = synth.synthetic_ultralight_avatar(n=16)
    av = UltraLightAvatar(ctx, net, frames, faces, coords)
    sess = UltraLightSession(av, B, ctx=ctx)                         # device-resident leg: one stream for the whole timed chain
    hf = HubertFeatures(enc, B, SL, SR, out_nhwc=sess.audio16, ctx=ctx)
    load_s = time.time() - t0
    audio = synth.sine_audio(10.0)
    hf.run_async(step_pcm(audio, 0, B))
    ctx.sync()
    stream = torch.cuda.ExternalStream(ctx.cuda_stream)
    gate = Gate(torch, stream)
    steps, warm = max(5, min(args.steps, 20)), max(3, min(args.warmup, 5))

    def online(k):
        hf.run_async(None)
        sess.step_async(k * B)

    for k in range(warm):
        online(k)
    ctx.sync()
    l0 = ctx.launch_count
    ms = timed_steps(torch, stream, gate, online, steps) / steps
    launches = (ctx.launch_count - l0) // steps
    ms_net = timed_steps(torch, stream, gate, lambda k: sess.step_async(k * B), steps) / steps
    sess2 = UltraLightSession(av, B)                                  # e2e: the objects the plugin drives (own ctx per role)
    hf2 = HubertFeatures(enc, B, SL, SR)

    from livetalking_b200 import engine
    ring = [engine.PinnedBuffer((B, av.H, av.W, 3), np.uint8) for _ in range(4)]   # the plugin's pinned output ring

    def e2e_one(k):
        feats = hf2.run(step_pcm(audio, k, B))                         # HubertASR.run_step features (H2D PCM, D2H windows)
        return sess2.infer_paste(k * B, feats, out=ring[k % 4].array)  # inference_batch + paste_back_frame x B -> host frames

    for k in range(warm):
        e2e_one(k)
    t1 = time.perf_counter()
    for k in range(steps):
        e2e_one(k)
    e2e_ms = (time.perf_counter() - t1) * 1000.0 / steps
    gf = unet_gflop_per_frame() * B + gflop_per_window(hf.n)
    res = {"metric": "lip-sync frames/sec (UltraLight 160x160, batch %d, fp16: HuBERT-large features + U-Net + paste-back)" % B,
           "value": round(1000.0 * B / ms, 2), "unit": "frames/s", "ms_per_step": round(ms, 3), "steps": steps, "warmup": warm,
           "unet_paste_only_ms": round(ms_net, 3), "algorithmic_gflop_per_step": round(gf, 1), "tflops": round(gf / ms, 1),
           "e2e": {"value": round(1000.0 * B / e2e_ms, 2), "unit": "frames/s", "h2d_bytes_per_step": int(hf2.n * 4 + B * 16 * 1024 * 2),
                   "d2h_bytes_per_step": int(B * 16 * 1024 * 4 + B * av.H * av.W * 3),
                   "how": "HubertFeatures.run(host PCM) + UltraLightSession.infer_paste(host windows) -> host frames, wall clock"},
           "gpu_launches_per_step": int(launches), "sessions_at_25fps_per_gpu": int((1000.0 * B / ms) // 25), "model_load_s": round(load_s, 1),
           "config": {"workload": "UltraLight Model(6,'hubert') at 160x160 + hubert-large (24 layers) over %d samples per step, 720p frames" % hf.n,
                      "weights": "synthetic"}}
    for o in (hf2, sess2, hf, sess, *ring):
        o.close()
    ctx.close()
    return res


# ------------------------------------------------------------------------------------------------ our arm
def dump_outputs(out_dir: str, frames: np.ndarray) -> None:
    """Composited frames (B, H, W, 3) u8 -> out_dir/frames_face.npy: the paste box of every frame, and
    out_dir/frames_sample.npy: 2^20 pixel values of the whole batch at fixed seeded positions; float32, 24 MB together."""
    os.makedirs(out_dir, exist_ok=True)
    y1, y2, x1, x2 = BBOX
    np.save(os.path.join(out_dir, "frames_face.npy"), frames[:, y1:y2, x1:x2].astype(np.float32))
    pos = np.sort(np.random.default_rng(0).choice(frames.size, 1 << 20, replace=False))
    np.save(os.path.join(out_dir, "frames_sample.npy"), frames.reshape(-1)[pos].astype(np.float32))


def run_ours(args):
    import torch
    from livetalking_b200 import engine, synth
    from livetalking_b200.w2l_pack import pack_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    numa = pin_to_gpu_numa(local)
    torch.cuda.set_device(local)
    engine.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks = load_peaks()

    # ---- weights: packed on rank 0, broadcast once over NCCL (NVLink/NVSwitch), adopted in place by every rank
    if rank == 0:
        blob = np.frombuffer(pack_state_dict(synth.random_state_dict(0)), dtype=np.uint8)
        nbytes = torch.tensor([blob.size], dtype=torch.int64, device="cuda")
    else:
        blob, nbytes = None, torch.zeros(1, dtype=torch.int64, device="cuda")
    if world > 1:
        dist.broadcast(nbytes, 0)
    wdev = torch.empty(int(nbytes.item()), dtype=torch.uint8, device="cuda")
    if rank == 0:
        wdev.copy_(torch.from_numpy(blob.copy()))
    if world > 1:
        dist.broadcast(wdev, 0)
    torch.cuda.synchronize()
    model = engine.W2LModel(device_ptr=wdev.data_ptr(), nbytes=wdev.numel(), keepalive=wdev)

    faces, frames, coords = synth.synthetic_avatar(n=64, H=FRAME_H, W=FRAME_W, bbox=BBOX, seed=rank)
    av = engine.W2LAvatar(faces, frames, coords)
    sess = engine.W2LSession(model, av, BATCH, SL, SR, FPS)
    extra = [engine.W2LSession(model, av, BATCH, SL, SR, FPS) for _ in range(max(0, args.sessions - 1))]
    audio = synth.sine_audio(60.0)
    stream = torch.cuda.ExternalStream(sess.cuda_stream)
    xstreams = [torch.cuda.ExternalStream(e.cuda_stream) for e in extra]
    gate = Gate(torch, stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: everything resident (PCM window uploaded once, faces/frames resident), device-timed, gated
    for s_ in [sess] + extra:
        s_.set_pcm(step_pcm(audio, 0))
    idx = [0]

    def step_all(_k):
        for s_ in [sess] + extra:
            s_.step_async(idx[0])
        idx[0] += BATCH

    # clock ramp: an idle GPU needs tens of ms to reach its boost clock; W = 5 steps is 7 ms.  Untimed, before the W warm-up steps.
    t_ramp = time.perf_counter()
    while time.perf_counter() - t_ramp < 0.15:
        step_all(0)
        if idx[0] % (64 * BATCH) == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    idx[0] = 0                     # the ramp ran a timing-dependent number of steps: start the avatar index from a fixed point
    for k in range(args.warmup):
        step_all(k)
    barrier()
    l0 = sess.launch_count
    sampler = ClockSampler(local)
    sampler.start()
    ms = timed_steps(torch, stream, gate, step_all, args.steps, xstreams)
    barrier()
    launches = (sess.launch_count - l0) * args.sessions
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # re-runs the paste-back of the last timed step on that step's prediction, still resident, and copies the frames out
        dump_outputs(args.dump_outputs, sess.paste_batch(idx[0] - BATCH))
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    per_rank = [float(ms)]
    if world > 1:
        allms = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allms, t)
        per_rank = [float(x.item()) for x in allms]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * args.sessions * BATCH * args.steps / (ms_max / 1000.0)

    # ---- sustained: the same loop for >= 3 s, with the clock / power trace
    sustained = None
    if not args.no_sustained:
        n_sus = max(args.steps, int(args.sustained_s * 1000.0 / (ms / args.steps)))
        s2 = ClockSampler(local)
        barrier()
        s2.start()
        ms_sus = timed_steps(torch, stream, gate, step_all, n_sus, xstreams)
        c2 = s2.stop()
        ts = torch.tensor([ms_sus], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        sustained = {"value": round(world * args.sessions * BATCH * n_sus / (float(ts.item()) / 1000.0), 2), "unit": "frames/s", "steps": n_sus,
                     "seconds": round(float(ts.item()) / 1000.0, 3), "ms_per_step": round(float(ts.item()) / n_sus, 4), "clocks": c2}

    # ---- e2e: C-ABI call with HOST buffers; H2D of the PCM window and D2H of the 16 composited frames inside the timed
    # region, pipelined: the D2H of step i (copy stream) overlaps the kernels of step i+1 (two pinned buffer pairs)
    pin_pcm = [engine.PinnedBuffer(((SL + SR + 2 * BATCH) * 320,), np.float32) for _ in range(2)]
    pin_out = [engine.PinnedBuffer((BATCH, FRAME_H, FRAME_W, 3), np.uint8) for _ in range(2)]

    def e2e_step(k, index):
        b = e2e_step.n & 1
        e2e_step.n += 1
        sess.e2e_acquire()                                        # buffer pair b was last used two steps ago: wait until it is drained
        pin_pcm[b].array[:] = step_pcm(audio, k)                  # "TTS" hands over host PCM
        sess.step_e2e_async(index, pin_pcm[b].array, pin_out[b].array)

    e2e_step.n = 0
    for k in range(max(4, args.warmup)):
        e2e_step(k, k * BATCH)
    sess.sync()
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        e2e_step(k, idx[0] + k * BATCH)
    sess.sync()                                                   # every frame of every step is in host memory here
    wall_ms = (time.perf_counter() - t0) * 1000.0
    barrier()
    te = torch.tensor([wall_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * BATCH * args.steps / (float(te.item()) / 1000.0)
    chk = sess.paste_batch(idx[0] + (args.steps - 1) * BATCH)     # the synchronous hooks produce the same frames as the pipelined call
    if not np.array_equal(chk, pin_out[(e2e_step.n - 1) & 1].array):
        raise RuntimeError("pipelined e2e frames differ from the synchronous path")

    # ---- roofline of the dominant kernels (tcgen05 implicit-GEMM convs)
    roof = None
    if rank == 0:
        ms_ops, flops, kinds = sess.profile_ops(idx[0])
        passes = [sess.profile_ops(idx[0])[0] for _ in range(3)]
        med = np.median(np.stack(passes + [ms_ops]), axis=0)
        conv = (kinds == 0) | (kinds == 4) | (kinds == 5)
        algo_flops = GFLOP_PER_FRAME * 1e9 * BATCH
        K = max(20, args.steps)
        for _ in range(3):
            sess.forward_async(idx[0])
        fwd_ms = timed_steps(torch, stream, gate, lambda k: sess.forward_async(idx[0] + k * BATCH), K) / K   # burst window (tens of ms)
        achieved = algo_flops / (fwd_ms / 1000.0) / 1e12
        frac_sus = None
        if not args.no_sustained:
            n_f = int(2000.0 / fwd_ms)
            fwd_sus = timed_steps(torch, stream, gate, lambda k: sess.forward_async(idx[0] + k * BATCH), n_f) / n_f
            frac_sus = {"forward_ms_per_step": round(fwd_sus, 4), "achieved": round(algo_flops / fwd_sus / 1e9, 2), "peak": peaks["sustained"],
                        "frac": round(algo_flops / fwd_sus / 1e9 / peaks["sustained"], 4), "seconds": round(n_f * fwd_sus / 1000.0, 2)}
        traffic = None
        tp = os.path.join(ROOT, "profiles", "conv_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_step")
            except Exception:
                traffic = None
        roof = {"bound": "tensor", "achieved": round(achieved, 2), "peak": peaks["burst"], "unit": "TFLOP/s",
                "frac": round(achieved / peaks["burst"], 4), "traffic": traffic,
                "peak_source": peaks["src"] + "; burst peak for this tens-of-ms window, sustained peak for `sustained`",
                "kernel": "conv_halo_umma + conv_ystack_umma + conv_gather_umma + stem_umma (tcgen05 implicit-GEMM convs): all conv launches of "
                          "one step, timed live as %d back-to-back forward-graph replays (CUDA events, session stream, gated)" % K,
                "forward_ms_per_step": round(fwd_ms, 4), "sustained": frac_sus,
                "conv_ms_per_step_eager_events": round(float(med[conv].sum()), 4),
                "other_ms_per_step_eager_events": round(float(med[~conv].sum()), 4), "algorithmic_gflop_per_step": round(algo_flops / 1e9, 1)}
        if args.dump_ops:
            os.makedirs(os.path.dirname(os.path.abspath(args.dump_ops)), exist_ok=True)
            json.dump({"ops": [(int(k), round(float(m), 4), float(f)) for k, m, f in zip(kinds, med, flops)],
                       "note": "kind(0 conv gather,1 prep,2 audio_conv0,3 head,4 conv halo/ystack,5 stem,6 mel), median ms, algorithmic flops"},
                      open(args.dump_ops, "w"))

    extras = {}

    def guarded(name, fn):
        try:
            extras[name] = fn()
        except Exception as e:                                  # an extra leg must never take the contract line down
            extras[name] = {"error": repr(e)[:300]}

    if rank == 0 and world == 1 and not args.quick and not args.only_musetalk:
        guarded("e2e_plugin", lambda: plugin_e2e(engine, model, (list(frames), list(faces), [tuple(c) for c in coords]), audio,
                                                  max(5, min(args.steps, 20)), 3))
        guarded("e2e_plugin_threads", lambda: plugin_threads(engine, model, (list(frames), list(faces), [tuple(c) for c in coords])))
        guarded("sessions32", lambda: sessions_leg(torch, engine, model, av, audio, 32, max(5, min(args.steps, 20))))
        guarded("cross_session", lambda: cross_session_leg(engine, model, max(5, min(args.steps, 20))))
        guarded("torch_eager_b200", lambda: torch_eager_b200(torch))
    if rank == 0 and world == 1 and not args.quick and not args.no_ultralight:
        guarded("ultralight", lambda: ultralight_leg(torch, args))
    if world > 1 and not args.quick:            # configs[3] at N > 1: 32 sessions on EVERY GPU (aggregate over ranks)
        guarded("sessions32", lambda: sessions_leg(torch, engine, model, av, audio, 32, max(5, min(args.steps, 20)), dist, world))
    if not args.no_musetalk and not args.quick:  # every rank runs the MuseTalk legs (collectives inside): same guard on all ranks
        mt = None
        try:
            mt = MuseTalkBench(torch, dist, world, rank)
            extras["musetalk"] = mt.leg(args, peaks, 32, batch_sessions=4)
            if not args.no_musetalk512:
                extras["musetalk512"] = mt.leg(args, peaks, 64, n_sessions=8, B_sess=2)
        except Exception as e:
            extras.setdefault("musetalk", {"error": repr(e)[:300]})
        finally:
            if mt is not None:
                mt.close()
    if world > 1:
        barrier()

    if rank == 0:
        cores = os.cpu_count() or 1
        cpu = None
        if world == 1 and not args.no_cpu_baseline and not args.quick and not args.only_musetalk:
            c = CpuPath(cores)
            c.frames_of(0, 2)
            t0 = time.perf_counter()
            for r in range(4):
                c.frames_of(r + 1, 2)
            cpu = {"value": round(8 / (time.perf_counter() - t0), 4), "unit": "frames/s", "cores": c.threads, "host_cores": cores, "kind": "port",
                   "sample": "4 reps x 2 frames (+1 warm-up): numpy mel + CPU PyTorch fp32 wav2lip256 + paste-back (oracle port)"}
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_max / args.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 (fp32 accumulate); mel f64; paste u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": BATCH * world * args.sessions, "sessions_per_gpu": args.sessions,
                       "parallelism": f"session-sharded x{world}",
                       "l2": "working set per step (activations ~0.9 GB + 107 MB weights) exceeds the 126 MB L2; no explicit flush",
                       "timing": "CUDA events on the session stream; a spin kernel gates the stream until all steps are enqueued; "
                                 "150 ms untimed clock ramp before the W warm-up steps"},
            "per_rank_ms": [round(x / args.steps, 4) for x in per_rank], "numa": numa,
            "e2e": {"value": round(e2e_value, 2), "unit": "frames/s", "h2d_bytes_per_step": int(pin_pcm[0].nbytes),
                    "d2h_bytes_per_step": int(pin_out[0].nbytes), "how": "ltb_w2l_step_e2e_async, pinned host buffers, wall clock incl. final sync"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof,
            "sustained": sustained,
            "cpu_baseline": cpu,
        }
        line.update(extras)
        print(json.dumps(line))
    for e_ in extra:
        e_.close()
    sess.close()
    av.close()
    model.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-musetalk", action="store_true", help="skip the MuseTalk (configs[2]) leg")
    ap.add_argument("--no-musetalk512", action="store_true", help="skip MuseTalk at 64x64 latents (configs[4]: 512x512, 8 concurrent sessions)")
    ap.add_argument("--musetalk512", action="store_true", help=argparse.SUPPRESS)   # accepted for compatibility: the leg is on by default
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--sustained-s", type=float, default=3.0)
    ap.add_argument("--no-ultralight", action="store_true", help="skip the UltraLight + HuBERT leg")
    ap.add_argument("--only-musetalk", action="store_true", help="development: contract line + the MuseTalk legs only")
    ap.add_argument("--quick", action="store_true", help="contract line only (value / e2e / roofline), no extra legs")
    ap.add_argument("--sessions", type=int, default=1, help="concurrent avatar sessions per GPU in the `value` leg (each batch 16, own stream)")
    ap.add_argument("--dump-ops", default=None, help="write per-op timings (json)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the composited frames of the last timed `value` step to DIR as float32 .npy files")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
