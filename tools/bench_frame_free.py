"""Frame-free vs full-frame avatars, measured on the GPU: HBM bytes per avatar, end-to-end frames/s through the plugin objects, and
D2H bytes per frame, for wav2lip, UltraLight and MuseTalk at 720p and 1080p.

    python tools/bench_frame_free.py [--frames 64] [--steps 30] [--warmup 5] [--kinds wav2lip,ultralight,musetalk] [--out result.json]

End to end = the plugin's inference_batch + batch x paste_back_frame, host numpy in and out, one thread, wall clock: the fused mode
for wav2lip and UltraLight (composite on the device, one D2H), MuseTalk's only mode (predictions to the host, paste_back_frame per
frame).  wav2lip includes MelASR's feature call (bench.py's e2e_plugin); UltraLight and MuseTalk take fixed synthetic features, which
do not depend on the residency.  Both residencies run on the same assets, alternating full / frame-free twice so that the spread
between repeats shows next to the difference.  HBM bytes are the cudaMemGetInfo delta of creating the avatar; D2H bytes are what the
composite copies to the host per frame.  Networks are random-init at the real architectures.  The GPU's name and power limit are
read in the same run and printed with the numbers."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

BATCH, FPS, SL, SR = 16, 25, 10, 10
MT_BATCH = 8
SIZES = {"720p": (720, 1280), "1080p": (1080, 1920)}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]], capture_output=True, text=True, timeout=30)
        name, power = [v.strip() for v in q.stdout.strip().split(",")[:2]]
    except Exception as e:   # noqa: BLE001 - reported, not hidden
        name, power = f"unknown ({e!r})", "unknown"
    return {"gpu": name, "power_limit": power}


def w2l_assets(n, H, W, seed=0):
    """n distinct frames with a ~320x320 mouth box that moves a little, as a talking-head clip's would."""
    rng = np.random.default_rng(seed)
    faces = [rng.integers(0, 256, (256, 256, 3), dtype=np.uint8) for _ in range(n)]
    frames = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(n)]
    coords = []
    for i in range(n):
        y1, x1 = H // 2 - 160 + (i % 7), W // 2 - 160 + (i % 5)
        coords.append((y1, y1 + 316 + (i % 9), x1, x1 + 316 + (i % 9)))
    return frames, faces, coords


def measure(engine, make_payload, make_session, features, mirror, n, B, H, W, steps, warmup, d2h_free, deterministic=True):
    """Both residencies of one avatar kind at one frame size: HBM delta of the avatar, e2e frames/s, D2H bytes per frame."""
    out, payloads = {}, {}
    for resident in (True, False):
        f0 = engine.mem_get_info()[0]
        payloads[resident] = make_payload(resident)
        out["full" if resident else "frame_free"] = {"hbm_bytes_per_avatar": f0 - engine.mem_get_info()[0]}
    sess = {r: make_session(payloads[r]) for r in (True, False)}

    def run(obj, k0, k1):
        last = None
        for k in range(k0, k1):
            index = k * B
            res = obj.inference_batch(index, features(obj))
            for i, r in enumerate(res):
                last = obj.paste_back_frame(r, mirror(n, index + i))
        return last

    check = {}
    for r, obj in sess.items():
        run(obj, 0, warmup)
        check[r] = run(obj, warmup, warmup + 1)
    diff = int(np.abs(check[True].astype(int) - check[False].astype(int)).max())
    # wav2lip's forward is deterministic: the frames must agree bit for bit; the others' networks jitter in the last bits
    assert diff == 0 or not deterministic, "frame-free and full-frame sessions disagree"
    out["max_abs_diff_last_frame"] = diff
    for _rep in range(2):
        for r, obj in sess.items():
            t0 = time.perf_counter()
            run(obj, 0, steps)
            dt = time.perf_counter() - t0
            out["full" if r else "frame_free"].setdefault("e2e_frames_per_s", []).append(round(B * steps / dt, 1))
    out["full"]["d2h_bytes_per_frame"] = H * W * 3
    out["frame_free"]["d2h_bytes_per_frame"] = d2h_free(payloads[False].engine_avatar)
    for obj in sess.values():
        obj.close()
    for p in payloads.values():
        if hasattr(p.engine_avatar, "close"):
            p.engine_avatar.close()
    return out


def w2l_leg(engine, model, P, stubs, mirror, H, W, n, steps, warmup):
    frames, faces, coords = w2l_assets(n, H, W)
    pcm = (0.3 * np.random.default_rng(1).standard_normal((SL + SR + 2 * BATCH) * 320)).astype(np.float32)

    def features(lip):
        mel = lip.engine_session.mel_step(pcm)                      # MelASR.run_step's feature call
        return [mel[i] for i in range(BATCH)]

    return measure(engine, lambda r: P.make_avatar(frames, faces, coords, frames_resident=r),
                   lambda p: P.LipReal(stubs.Opt(batch_size=BATCH, fps=FPS, l=SL, r=SR), model, p), features, mirror, n, BATCH, H, W,
                   steps, warmup, lambda av: av.region_max[0] * av.region_max[1] * 3)


def ul_leg(engine, stubs, mirror, H, W, n, steps, warmup):
    from livetalking_b200 import synth
    from livetalking_b200.plugin import ultralight_avatar as UL
    model = UL.make_model(synth.random_hubert_state_dict())
    sd = synth.random_ultralight_state_dict()
    frames, faces, coords = synth.synthetic_ultralight_avatar(n=n, H=H, W=W, bbox=(W // 2 - 140, H // 2 - 140, W // 2 + 140, H // 2 + 140))
    frames = list(frames)
    feats = [(0.1 * np.random.default_rng(k).standard_normal((16, 1024))).astype(np.float32) for k in range(BATCH)]
    return measure(engine, lambda r: UL.make_avatar(sd, frames, list(faces), coords, frames_resident=r),
                   lambda p: UL.LightReal(stubs.Opt(batch_size=BATCH, fps=FPS, l=SL, r=SR), model, p), lambda _o: feats, mirror, n, BATCH,
                   H, W, steps, warmup, lambda av: av.region_max[0] * av.region_max[1] * 3, deterministic=False)


def mt_leg(engine, stubs, mirror, H, W, n, steps, warmup, model):
    from livetalking_b200 import synth
    from livetalking_b200.plugin import musetalk_avatar as MT
    frames, masks, coords, crops, latents = synth.synthetic_musetalk_avatar(n=n, H=H, W=W, bbox=(W // 2 - 160, H // 2 - 160, W // 2 + 160,
                                                                                                 H // 2 + 160))
    frames = list(frames)
    feats = [(0.1 * np.random.default_rng(k).standard_normal((50, 384))).astype(np.float32) for k in range(MT_BATCH)]
    return measure(engine, lambda r: MT.make_avatar(frames, masks, coords, crops, latents, model, frames_resident=r),
                   lambda p: MT.MuseReal(stubs.Opt(batch_size=MT_BATCH, fps=FPS, l=SL, r=SR), model, p), lambda _o: feats, mirror, n,
                   MT_BATCH, H, W, steps, warmup, lambda av: av.region_max[0] * av.region_max[1] * 3, deterministic=False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64, help="frames per avatar")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--kinds", default="wav2lip,ultralight,musetalk")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import stubs
    stubs.install()
    from livetalking_b200 import engine
    engine.set_device(0)
    mirror = sys.modules["utils.image"].mirror_index
    kinds = args.kinds.split(",")
    result = {**gpu_info(), "frames_per_avatar": args.frames, "steps": args.steps, "batch": {"wav2lip": BATCH, "ultralight": BATCH,
              "musetalk": MT_BATCH}, "how": __doc__.split("\n\n")[1].replace("\n", " ")}
    if "wav2lip" in kinds:
        from livetalking_b200.plugin import wav2lip_avatar as P
        from oracle import wav2lip_ref as R
        model = engine.W2LModel.from_state_dict(R.synth_state_dict(0))
        for name, (H, W) in SIZES.items():
            result.setdefault("wav2lip", {})[name] = w2l_leg(engine, model, P, stubs, mirror, H, W, args.frames, args.steps, args.warmup)
            print("wav2lip", name, json.dumps(result["wav2lip"][name]), flush=True)
        model.close()
    if "ultralight" in kinds:
        for name, (H, W) in SIZES.items():
            result.setdefault("ultralight", {})[name] = ul_leg(engine, stubs, mirror, H, W, args.frames, args.steps, args.warmup)
            print("ultralight", name, json.dumps(result["ultralight"][name]), flush=True)
    if "musetalk" in kinds:
        from livetalking_b200 import configs, synth
        from livetalking_b200.plugin import musetalk_avatar as MT
        ucfg, vcfg = configs.UNetConfig(), configs.VAEConfig()
        model = MT.make_model(synth.random_unet_state_dict(ucfg), synth.random_vae_state_dict(vcfg), synth.random_whisper_state_dict(), ucfg,
                              vcfg)
        for name, (H, W) in SIZES.items():
            result.setdefault("musetalk", {})[name] = mt_leg(engine, stubs, mirror, H, W, args.frames, max(3, args.steps // 3),
                                                             args.warmup, model)
            print("musetalk", name, json.dumps(result["musetalk"][name]), flush=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
