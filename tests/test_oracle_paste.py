"""CPU: paste-back oracle is bit-exact with OpenCV (the library the reference calls) and with the golden frames."""
import os
import sys
import zlib

import numpy as np
import pytest

from oracle import paste_ref as P

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))


def test_resize_bit_exact_vs_cv2_random_sizes():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(0)
    cases = [(256, 256, 128, 128), (256, 256, 256, 256), (256, 256, 128, 300), (256, 256, 512, 512), (256, 256, 1, 1),
             (256, 256, 255, 257), (256, 256, 64, 64), (256, 256, 321, 320)]
    for _ in range(60):
        cases.append((256, 256, int(rng.integers(2, 520)), int(rng.integers(2, 520))))
    for _ in range(20):
        cases.append((int(rng.integers(8, 300)), int(rng.integers(8, 300)), int(rng.integers(2, 400)), int(rng.integers(2, 400))))
    for sh, sw, dh, dw in cases:
        src = rng.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        assert np.array_equal(cv2.resize(src, (dw, dh)), P.resize_linear_u8(src, dw, dh)), (sh, sw, dh, dw)


def test_paste_matches_golden(golden_dir):
    import make_golden as G
    g = np.load(os.path.join(golden_dir, "paste_golden.npz"))
    pred = G.synth_pred()
    for box, crc, sub in zip(g["boxes"], g["crc32"], g["sub"]):
        out = P.w2l_paste_back(pred, G.synth_frame(300, 300), box)
        assert np.array_equal(out[::3, ::3], sub), box
        assert zlib.crc32(out.tobytes()) == int(crc), box


def test_mirror_index_and_batch_build():
    assert [P.mirror_index(3, i) for i in range(8)] == [0, 1, 2, 2, 1, 0, 0, 1]     # utils/image.py:26-32
    faces = [np.full((256, 256, 3), i * 10, np.uint8) for i in range(3)]
    b = P.w2l_build_batch(faces, 2, 4)
    assert b.shape == (4, 6, 256, 256) and b.dtype == np.float32
    assert np.all(b[:, :3, 128:] == 0) and np.all(b[0, 3:] == np.float32(20 / 255.0)) and np.all(b[1, 3:, :] == np.float32(20 / 255.0))
    assert np.all(b[0, :3, :128] == np.float32(20 / 255.0))


def mt_blend_case():
    """Seeded MuseTalk paste-back case: frame, prediction, bbox, crop, [soft mask, noise mask]."""
    import cv2
    rng = np.random.default_rng(3)
    H, W = 180, 240
    frame = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    pred = rng.integers(0, 256, (256, 256, 3), dtype=np.uint8)
    bbox = (70, 40, 170, 150)            # x1,y1,x2,y2
    crop = (40, 10, 200, 176)            # x_s,y_s,x_e,y_e
    mh, mw = crop[3] - crop[1], crop[2] - crop[0]
    soft = cv2.GaussianBlur((np.arange(mh)[:, None] > mh // 2).astype(np.float32).repeat(mw, 1) * 255, (0, 0), 7).astype(np.uint8)
    masks = [np.stack([soft] * 3, -1), rng.integers(0, 256, (mh, mw, 3), dtype=np.uint8)]
    return frame, pred, bbox, crop, masks


def test_musetalk_blend_matches_cv2_and_reference_function(golden_dir):
    """oracle mt_paste_back vs OpenCV (blendLinear / cvtColor) and vs the output of the reference's own get_image_blending
    (avatars/musetalk/myutil.py) driven as MuseReal.paste_back_frame does (mt_blend_golden.npz)."""
    cv2 = pytest.importorskip("cv2")
    frame, pred, bbox, crop, masks = mt_blend_case()
    want = np.load(os.path.join(golden_dir, "mt_blend_golden.npz"))["want"]
    assert want.shape == (len(masks),) + frame.shape
    for mask, ref_out in zip(masks, want):
        got = P.mt_paste_back(pred, frame, bbox, mask, crop)
        # direct OpenCV composition
        x1, y1, x2, y2 = bbox
        xs, ys, xe, ye = crop
        body = frame.copy()
        large = body[ys:ye, xs:xe].copy()
        large[y1 - ys:y2 - ys, x1 - xs:x2 - xs] = cv2.resize(pred, (x2 - x1, y2 - y1))
        m = (cv2.cvtColor(mask, cv2.COLOR_BGR2GRAY) / 255).astype(np.float32)
        body[ys:ye, xs:xe] = cv2.blendLinear(large, body[ys:ye, xs:xe], m, 1 - m)
        assert np.array_equal(got, body)
        assert np.array_equal(got, ref_out)
