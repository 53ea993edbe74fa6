"""Pins oracle/letterbox_oracle.py (integer restatement of LetterBox + cv2.resize INTER_LINEAR + the predictor's BGR->RGB /
HWC->CHW) to the REAL reference pipeline (fixtures: tests/golden/make_golden.py letterbox, cv2 4.13): bit-exact (CRC) for
every case - downscales, identity, one- and two-axis upscales."""
import os
import zlib

import numpy as np
import pytest
import torch

from _util import GOLD
from oracle import letterbox_oracle as L

GOLDEN = torch.load(os.path.join(GOLD, "letterbox.golden.pt"))


@pytest.mark.parametrize("case", GOLDEN["cases"], ids=lambda c: f"{c['h']}x{c['w']}")
def test_letterbox_oracle_matches_reference(case):
    h, w = case["h"], case["w"]
    img = np.random.default_rng(case["seed"]).integers(0, 256, (h, w, 3), dtype=np.uint8)
    out = L.preprocess_frame(img, (640, 640))
    assert list(out.shape) == case["shape"] and out.dtype == np.uint8
    thumb = out.reshape(3, 40, 16, 40, 16).astype(np.float32).mean((2, 4))
    assert float(np.abs(thumb - case["thumb"].numpy()).max()) == 0.0         # 16x16 block means: localises a mismatch
    assert zlib.crc32(out.tobytes()) == case["crc"]                          # bit-exact


def test_letterbox_params_known_answers():
    """LetterBox.get_params augment.py:1742-1786: 480x640 -> no resize, 80 px of padding top and bottom; 1080x1920 -> 640x360."""
    assert L.letterbox_params((480, 640)) == ((640, 480), 80, 80, 0, 0)
    assert L.letterbox_params((1080, 1920)) == ((640, 360), 140, 140, 0, 0)
    assert L.letterbox_params((333, 500)) == ((640, 426), 107, 107, 0, 0)
    assert L.letterbox_params((100, 37)) == ((237, 640), 0, 0, 201, 202)


def test_resize_matches_cv2_bit_exact():
    """Direct comparison when cv2 is importable (it is in the build container).  The upscales exercise the y-border rule: the two
    clipped row indices keep their fractional weights, so a border row is blended with itself through two truncated products."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(5)
    for (sh, sw, dh, dw) in ((64, 64, 640, 640), (100, 37, 640, 237), (31, 57, 352, 640), (7, 5, 640, 457), (2, 2, 9, 9), (1, 8, 5, 16)):
        img = rng.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        assert np.array_equal(cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR), L.resize_linear_u8(img, dw, dh)), (sh, sw, dh, dw)
    big = np.random.default_rng(6).integers(0, 256, (300, 400, 3), dtype=np.uint8)
    for dw, dh in ((320, 240), (400, 100), (137, 300), (200, 150), (399, 299), (57, 31)):   # downscale / single-axis / exact 2x
        assert np.array_equal(cv2.resize(big, (dw, dh), interpolation=cv2.INTER_LINEAR), L.resize_linear_u8(big, dw, dh)), (dw, dh)


@pytest.mark.parametrize("case", GOLDEN["variants"], ids=lambda c: f"{c['h']}x{c['w']}-{'-'.join(c['kw']) or 'rect'}")
def test_letterbox_variants_match_reference(case):
    """auto (minimum rectangle) / scaleup=False / scale_fill / center=False / non-square target: geometry and pixels of the
    transform itself (HWC, BGR) against the real LetterBox."""
    img = np.random.default_rng(case["seed"]).integers(0, 256, (case["h"], case["w"], 3), dtype=np.uint8)
    prm = L.letterbox_params(img.shape[:2], tuple(case["new_shape"]), **case["kw"])
    assert [list(prm[0]), *prm[1:]] == case["params"]
    out = L.letterbox_frame(img, tuple(case["new_shape"]), **case["kw"])
    assert list(out.shape) == case["shape"]
    assert zlib.crc32(np.ascontiguousarray(out).tobytes()) == case["crc"]


@pytest.mark.parametrize("case", GOLDEN["scale_boxes"], ids=lambda c: f"{c['img0'][0]}x{c['img0'][1]}-{'xywh' if c['xywh'] else 'xyxy'}")
def test_scale_boxes_oracle_matches_reference(case):
    """ops.scale_boxes (+ clip_boxes) of the reference on seeded boxes that straddle the frame: bit-exact fp32."""
    g = torch.Generator().manual_seed(case["seed"])
    img1 = case["img1"]
    b = torch.rand((64, 6), generator=g) * torch.tensor([img1[1], img1[0], img1[1], img1[0], 1, 80]) * 1.1 - 8.0
    out = L.scale_boxes(img1, b[:, :4].numpy(), case["img0"], xywh=case["xywh"])
    assert np.array_equal(out, case["out"].numpy())


def test_scale_coords_oracle_matches_reference():
    """oracle scale_coords == the reference's ops.scale_coords, bit for bit (fixture: tests/golden/make_golden.py scale_coords)."""
    cases = torch.load(os.path.join(GOLD, "scale_coords.golden.pt"))["cases"]
    assert len(cases) == 8
    for c in cases:
        out = L.scale_coords((640, 640), c["coords"].numpy(), c["shape0"], normalize=c["normalize"])
        assert np.array_equal(out, c["out"].numpy()), (c["shape0"], c["normalize"])
