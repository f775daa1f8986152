"""GPU: frame-free avatars composite only the paste rectangle; after the host paste their frames are bit-identical to the
full-frame path on the same assets, index and features.  They allocate no n*H*W*3 frame store and no (batch, H, W, 3) output,
and the full-frame-only entry points refuse them with a message without breaking the session."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def w2l_assets(rng, n, H, W):
    faces = rng.integers(0, 256, (n, 256, 256, 3), dtype=np.uint8)
    frames = rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)
    coords = [(0, 256, 0, 256), (H - 128, H, W - 128, W), (3, H - 5, 7, W - 1)]       # same-size, 2x decimation, edge-touching
    while len(coords) < n:
        y1, x1 = int(rng.integers(0, H - 40)), int(rng.integers(0, W - 40))
        coords.append((y1, int(rng.integers(y1 + 17, min(H, y1 + 333) + 1)), x1, int(rng.integers(x1 + 17, min(W, x1 + 333) + 1))))
    return list(faces), frames, coords


def test_w2l_frame_free_matches_full_frame(w2l_state_dict):
    from livetalking_b200 import engine
    from oracle import paste_ref as P
    engine.set_device(0)
    rng = np.random.default_rng(5)
    H, W, B, n = 301, 517, 8, 11
    faces, frames, coords = w2l_assets(rng, n, H, W)
    model = engine.W2LModel.from_state_dict(w2l_state_dict)
    full = engine.W2LAvatar(faces, frames, coords)
    free = engine.W2LAvatar(faces, list(frames), coords, frames_resident=False)
    assert free.region_max == (max(c[1] - c[0] for c in coords), max(c[3] - c[2] for c in coords)) == full.region_max
    s_full, s_free = engine.W2LSession(model, full, B), engine.W2LSession(model, free, B)
    mel = np.clip(rng.standard_normal((B, 80, 16)), -4, 4).astype(np.float32)
    for index in (0, 5, 17):                                           # 17: mirror_index runs backwards
        want = s_full.infer_paste(index, mel)
        regions, boxes = s_free.infer_paste_region(index, mel)
        for i in range(B):
            idx = P.mirror_index(n, index + i)
            assert tuple(boxes[i]) == tuple(coords[idx])
            assert np.array_equal(engine.paste_region(frames[idx], regions[i], boxes[i]), want[i]), (index, i)
        # return_pred: the host prediction pasted by either residency
        pred = s_full.infer(index, mel)
        for i in (0, B - 1):
            idx = P.mirror_index(n, index + i)
            region, box = s_free.paste_pred_region(pred[i], idx)
            assert region.shape == (box[1] - box[0], box[3] - box[2], 3)
            assert np.array_equal(engine.paste_region(frames[idx], region, box), s_full.paste_pred(pred[i], idx))
    for o in (s_full, s_free, full, free, model):
        o.close()


def test_w2l_frame_free_slots_match_full_frame(w2l_state_dict):
    """Cross-session slots: frame-free avatars of DIFFERENT frame sizes in one region batch, next to a full-frame avatar; each slot
    equals the full-frame slots session's frame after the host paste."""
    from livetalking_b200 import engine
    engine.set_device(0)
    rng = np.random.default_rng(9)
    Bm = 8
    model = engine.W2LModel.from_state_dict(w2l_state_dict)
    a0 = w2l_assets(rng, 5, 300, 400)
    a1 = w2l_assets(rng, 4, 280, 360)
    full0 = engine.W2LAvatar(*a0)
    full1 = engine.W2LAvatar(*a1)
    free0 = engine.W2LAvatar(a0[0], list(a0[1]), a0[2], frames_resident=False)
    free1 = engine.W2LAvatar(a1[0], list(a1[1]), a1[2], frames_resident=False)
    mux0 = engine.W2LSession(model, full0, Bm, slots=True)
    mux1 = engine.W2LSession(model, full1, Bm, slots=True)
    rmux = engine.W2LSession(model, free0, Bm, slots=True)           # free0 has the larger region capacity
    assert all(r >= f for r, f in zip(free0.region_max, free1.region_max))
    mels = np.clip(rng.standard_normal((Bm, 80, 16)), -4, 4).astype(np.float32)
    picks = [(i % 2, (3 * i + 1) % (5 if i % 2 == 0 else 4)) for i in range(Bm)]
    got = rmux.infer_slots_region([((free0, free1)[a], idx, mels[i]) for i, (a, idx) in enumerate(picks)])
    # full-frame references: homogeneous batches (slots do not influence each other, test_gpu_w2l)
    w0 = mux0.infer_slots([(full0, idx, mels[i]) if a == 0 else (full0, 0, mels[i]) for i, (a, idx) in enumerate(picks)])
    w1 = mux1.infer_slots([(full1, idx, mels[i]) if a == 1 else (full1, 0, mels[i]) for i, (a, idx) in enumerate(picks)])
    for i, (a, idx) in enumerate(picks):
        region, box = got[i]
        frame = (a0, a1)[a][1][idx]
        assert np.array_equal(engine.paste_region(frame, region, box), (w0, w1)[a][i]), i
    # a full-frame avatar in a region batch works too; a box larger than the session's pitch is refused
    mixed = rmux.infer_slots_region([(full0, 2, mels[0]), (free0, 2, mels[0])])
    assert np.array_equal(mixed[0][0], mixed[1][0])
    small = engine.W2LSession(model, engine.W2LAvatar(a1[0][:1], [a1[1][0]], [(0, 16, 0, 16)], frames_resident=False), 2, slots=True)
    with pytest.raises(engine.LtbError, match="region pitch"):
        small.infer_slots_region([(free0, 0, mels[0])])
    for o in (small, rmux, mux1, mux0, free1, free0, full1, full0, model):
        o.close()


def test_w2l_frame_free_device_bytes(w2l_state_dict):
    """A frame-free avatar allocates its faces and boxes only; a session of it allocates (batch, rh_max, rw_max, 3) outputs
    instead of (batch, H, W, 3)."""
    from livetalking_b200 import engine
    engine.set_device(0)
    rng = np.random.default_rng(1)
    n, H, W, B = 40, 720, 1280, 16
    faces = list(rng.integers(0, 256, (n, 256, 256, 3), dtype=np.uint8))
    frame = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    frames = [frame] * n
    coords = [(200, 520, 480, 800)] * n
    model = engine.W2LModel.from_state_dict(w2l_state_dict)
    slack = 4 << 20                                                   # cudaMalloc granularity
    f0 = engine.mem_get_info()[0]
    free = engine.W2LAvatar(faces, frames, coords, frames_resident=False)
    d_free = f0 - engine.mem_get_info()[0]
    f0 = engine.mem_get_info()[0]
    full = engine.W2LAvatar(faces, np.stack(frames), coords)
    d_full = f0 - engine.mem_get_info()[0]
    assert d_free <= n * 256 * 256 * 3 + n * 16 + slack, d_free
    assert d_full >= d_free + n * H * W * 3 - slack, (d_full, d_free)
    engine.W2LSession(model, free, B).close()                        # loads the kernels' modules before anything is measured
    f0 = engine.mem_get_info()[0]
    s_free = engine.W2LSession(model, free, B)
    d_sfree = f0 - engine.mem_get_info()[0]
    f0 = engine.mem_get_info()[0]
    s_full = engine.W2LSession(model, full, B)
    d_sfull = f0 - engine.mem_get_info()[0]
    assert d_sfull - d_sfree >= B * (H * W - 320 * 320) * 3 - slack, (d_sfull, d_sfree)
    for o in (s_full, s_free, full, free, model):
        o.close()


def test_w2l_full_frame_entry_points_refuse_frame_free(w2l_state_dict):
    from livetalking_b200 import engine
    from livetalking_b200._capi import lib
    from oracle import paste_ref as P
    engine.set_device(0)
    rng = np.random.default_rng(2)
    H, W, B, n = 260, 320, 4, 6
    faces, frames, coords = w2l_assets(rng, n, H, W)
    model = engine.W2LModel.from_state_dict(w2l_state_dict)
    full = engine.W2LAvatar(faces, frames, coords)
    free = engine.W2LAvatar(faces, list(frames), coords, frames_resident=False)
    s = engine.W2LSession(model, free, B)
    ref = engine.W2LSession(model, full, B)
    mux = engine.W2LSession(model, full, B, slots=True)
    mel = np.clip(rng.standard_normal((B, 80, 16)), -4, 4).astype(np.float32)
    pcm = np.zeros((10 + 10 + 2 * B) * 320, np.float32)
    pcm_pin = engine.PinnedBuffer(pcm.shape, np.float32)
    out_pin = engine.PinnedBuffer((B, H, W, 3), np.uint8)
    calls = {
        "ltb_w2l_infer_paste": lambda: s.infer_paste(0, mel),
        "ltb_w2l_paste_batch": lambda: s.paste_batch(0),
        "ltb_w2l_paste": lambda: s.paste(0, 0),
        "ltb_w2l_paste_pred": lambda: s.paste_pred(np.zeros((256, 256, 3), np.float32), 0),
        "ltb_w2l_step_async": lambda: s.step_async(0),
        "ltb_w2l_step_e2e_async": lambda: s.step_e2e_async(0, pcm_pin.array, out_pin.array),
        "infer_slots": lambda: mux.infer_slots([(free, 0, mel[0])]),
    }
    for name, call in calls.items():
        with pytest.raises(engine.LtbError, match="frame-free") as e:
            call()
        assert name in str(e.value)
    assert lib().ltb_w2l_infer_slots(None, None, 0, None) != 0               # plain null checks still come first
    s.sync()
    regions, boxes = s.infer_paste_region(3, mel)                         # the session is still usable, and correct
    want = ref.infer_paste(3, mel)
    for i in range(B):
        idx = P.mirror_index(n, 3 + i)
        assert np.array_equal(engine.paste_region(frames[idx], regions[i], boxes[i]), want[i])
    for o in (pcm_pin, out_pin, mux, ref, s, full, free, model):
        o.close()


def test_ultralight_frame_free_matches_full_frame():
    """UltraLight: the fused region composite and the region paste of a host prediction, after the host paste, equal the full-frame
    session's paste of the same prediction (and the oracle); the frame-free avatar uploads crops and boxes only; the full-frame
    methods refuse it with a message and leave the session usable."""
    from livetalking_b200 import engine
    from livetalking_b200.ops import Ctx
    from livetalking_b200.ultralight import UltraLightAvatar, UltraLightModel, UltraLightSession
    from oracle import ultralight_ref as U
    engine.set_device(0)
    n, B, H, W = 7, 4, 261, 343
    _img, audio, faces = U.synth_inputs(n, seed=3)
    rng = np.random.default_rng(3)
    frames = rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)
    # (x1,y1,x2,y2): stretch, identity 168², exact halving 84² at the bottom-right edge, full frame, odd sliver, two random
    coords = [(30, 20, 231, 203), (10, 40, 178, 208), (W - 84, H - 84, W, H), (0, 0, W, H), (5, 3, 36, 250), (101, 7, 290, 170),
              (0, 90, 171, 261)]
    feats = audio.numpy().reshape(n, 16, 1024)[:B]
    ctx = Ctx()
    model = UltraLightModel(ctx, U.synth_state_dict(0))
    f0 = engine.mem_get_info()[0]
    free = UltraLightAvatar(ctx, model, list(frames), faces, coords, frames_resident=False)
    assert f0 - engine.mem_get_info()[0] <= n * 168 * 168 * 3 + (4 << 20)
    full = UltraLightAvatar(ctx, model, frames, faces, coords)
    assert free.region_max == (H, W)
    s_free, s_full = UltraLightSession(free, B), UltraLightSession(full, B)
    for index in (0, 5):
        regions, boxes = s_free.infer_paste_region(index, feats)
        pred = s_free.ctx.download(s_free.pred)                          # the prediction the region composite used
        for i in range(B):
            idx = U.mirror_index(n, index + i)
            got = engine.paste_region(frames[idx], regions[i], boxes[i])
            assert np.array_equal(got, s_full.paste_pred(pred[i], idx)), (index, i)
            assert np.array_equal(got, U.lightreal_paste(pred[i], frames[idx], faces[idx], coords[idx])), (index, i)
    host_pred = rng.uniform(0, 255.99, (160, 160, 3)).astype(np.float32)
    for idx in range(n):
        region, box = s_free.paste_pred_region(host_pred, idx)
        assert np.array_equal(engine.paste_region(frames[idx], region, box), s_full.paste_pred(host_pred, idx)), idx
    for call in (lambda: s_free.infer_paste(0, feats), lambda: s_free.paste_batch(0), lambda: s_free.paste_pred(host_pred, 0),
                 lambda: s_free.step_async(0)):
        with pytest.raises(engine.LtbError, match="frame-free"):
            call()
    regions, boxes = s_free.infer_paste_region(2, feats)                 # still usable
    pred = s_free.ctx.download(s_free.pred)
    idx = U.mirror_index(n, 2)
    assert np.array_equal(engine.paste_region(frames[idx], regions[0], boxes[0]), s_full.paste_pred(pred[0], idx))
    s_free.close()
    s_full.close()
    ctx.close()


@pytest.mark.parametrize("hw", [32, 64], ids=["pred256", "pred512"])
def test_musetalk_frame_free_matches_full_frame(hw):
    """MuseTalk (small networks): the blended crop boxes of a frame-free avatar — single session and MuseTalkBatchSession groups —
    after the host paste equal the full-frame paste of the same prediction, bit for bit; the avatar uploads latents, masks and body
    crops but no frames; the full-frame methods refuse it with a message and leave the session usable."""
    from livetalking_b200 import engine
    from livetalking_b200.musetalk import MuseTalkAvatar, MuseTalkBatchSession, MuseTalkModel, MuseTalkSession
    from livetalking_b200.ops import Ctx
    from oracle import musetalk_ref as M
    from oracle import paste_ref as P
    engine.set_device(0)
    ucfg, vcfg = M.UNET_SMALL, M.VAE_SMALL
    S, n, B = hw * 8, 5, 2
    H, W = (300, 400) if hw == 32 else (700, 900)
    rng = np.random.default_rng(hw)
    frames = rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)
    coords, crops, masks = [], [], []
    for i in range(n):
        x1, y1 = int(rng.integers(0, W // 2)), int(rng.integers(0, H // 2))
        x2, y2 = int(rng.integers(x1 + 17, W + 1)), int(rng.integers(y1 + 17, H + 1))
        crop = (0, 0, W, H) if i == 0 else (max(0, x1 - 31), max(0, y1 - 23), min(W, x2 + 41), min(H, y2 + 9))    # frame 0: the whole frame
        coords.append((x1, y1, x2, y2))
        crops.append(crop)
        masks.append(rng.integers(0, 256, (crop[3] - crop[1], crop[2] - crop[0], 3), dtype=np.uint8))
    lat, aud = M.synth_latents_and_audio(n, hw=hw, seed=hw)
    lats = [lat.numpy()[i:i + 1] for i in range(n)]
    aud = aud.numpy()[:B]
    ctx = Ctx()
    model = MuseTalkModel(ctx, M.synth_unet_state_dict(ucfg), M.synth_vae_state_dict(vcfg), ucfg, vcfg, with_encoder=False)
    f0 = engine.mem_get_info()[0]
    free = MuseTalkAvatar(ctx, list(frames), masks, coords, crops, lats, frames_resident=False)
    d_free = f0 - engine.mem_get_info()[0]
    crop_bytes = sum(m.nbytes for m in masks)
    assert d_free <= 2 * crop_bytes + n * hw * hw * 16 * 2 + (16 << 20), d_free        # masks + body crops + latents + boxes
    full = MuseTalkAvatar(ctx, frames, masks, coords, crops, lats)
    assert free.frames is None and free.region_max == (max(c[3] - c[1] for c in crops), max(c[2] - c[0] for c in crops))
    s_free, s_full = MuseTalkSession(model, free, B), MuseTalkSession(model, full, B)

    def same_as_full(region, box, pred_i, idx):
        got = engine.paste_region(frames[idx], region, box)
        assert np.array_equal(got, s_full.paste_pred(pred_i, idx)), idx
        assert np.array_equal(got, P.mt_paste_back(pred_i, frames[idx], coords[idx], masks[idx], crops[idx])), idx

    for index in (0, 4):
        pred = s_free.infer(index, aud)
        regions, boxes = s_free.paste_batch_region(index)
        for i in range(B):
            idx = P.mirror_index(n, index + i)
            assert tuple(boxes[i]) == (crops[idx][1], crops[idx][3], crops[idx][0], crops[idx][2])
            same_as_full(regions[i], boxes[i], pred[i], idx)
    host_pred = rng.integers(0, 256, (S, S, 3), dtype=np.uint8)
    for idx in range(n):
        region, box = s_free.paste_pred_region(host_pred, idx)
        same_as_full(region, box, host_pred, idx)
    for call in (lambda: s_free.paste_batch(0), lambda: s_free.paste(0, 0), lambda: s_free.paste_pred(host_pred, 0),
                 lambda: s_free.step_async(0)):
        with pytest.raises(engine.LtbError, match="frame-free"):
            call()
    region, box = s_free.paste_pred_region(host_pred, 3)                    # still usable
    same_as_full(region, box, host_pred, 3)
    # cross-session groups: a frame-free and a full-frame avatar in one round
    bs = MuseTalkBatchSession(model, hw, 2, B)
    outs = bs.step([(free, 3, aud), (full, 1, aud)])
    pred_b = bs.ctx.download(bs.image_u8)
    assert outs[0].shape == (B, *free.region_max, 3) and outs[1].shape == (B, H, W, 3)
    for i in range(B):
        idx = P.mirror_index(n, 3 + i)
        same_as_full(outs[0][i], free.box(idx), pred_b[i], idx)
        idx = P.mirror_index(n, 1 + i)
        assert np.array_equal(outs[1][i], s_full.paste_pred(pred_b[B + i], idx))
    for o in (bs, s_free, s_full, ctx):
        o.close()
