"""TEST INFRASTRUCTURE -- seeded small cases shared by oracle/make_golden.py and the tests.

Inputs and weights are regenerated from seeds (numpy PCG64), only outputs live in tests/golden/.
"""
from __future__ import annotations

import itertools

import numpy as np
import torch

from . import weights

OCR_VOCAB_SMALL = 512


def dbnet_case(h=256, w=256, n=1, seed=11):
    rng = np.random.default_rng(seed)
    # smooth-ish page: low-frequency field + strokes, u8 range mapped like det_batch_forward_default
    img = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    x = img.astype(np.float32) / 127.5 - 1.0
    return img, torch.from_numpy(np.ascontiguousarray(x.transpose(0, 3, 1, 2)))


def ocr_case(n=2, wp=200, seed=12):
    rng = np.random.default_rng(seed)
    img = np.full((n, 48, wp, 3), 0, np.uint8)
    for i in range(n):
        wi = wp - 135 if i == 0 else max(16, (wp - 135) * (i + 1) // (n + 1))
        line = np.clip(235 + 10 * rng.standard_normal((48, wi, 1)), 0, 255).repeat(3, 2)
        for _ in range(wi // 6):
            x0, y0 = rng.integers(0, wi - 4), rng.integers(4, 40)
            line[y0:y0 + rng.integers(2, 8), x0:x0 + rng.integers(1, 4)] = rng.integers(0, 60)
        img[i, :, :wi] = line.astype(np.uint8)
    x = (torch.from_numpy(img).float() - 127.5) / 127.5
    return img, x.permute(0, 3, 1, 2).contiguous()


def lama_case(h=128, w=96, seed=13):
    rng = np.random.default_rng(seed)
    img = rng.uniform(0, 1, (1, 3, h, w)).astype(np.float32)
    mask = np.zeros((1, 1, h, w), np.float32)
    mask[:, :, h // 4: h // 4 + h // 3, w // 5: w // 5 + w // 2] = 1
    mask[:, :, (3 * h) // 4: (3 * h) // 4 + h // 8, (2 * w) // 3: (2 * w) // 3 + w // 5] = 1
    img = img * (1 - mask)
    return torch.from_numpy(img), torch.from_numpy(mask)


def digest(a) -> str:
    """sha256 of an array's dtype, shape and bytes (None -> "none"): how large exact-match fixtures are stored."""
    import hashlib
    if a is None:
        return "none"
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def plain(v):
    """Tuples / numpy scalars -> the JSON types they are stored as (ints stay ints only where they were Python ints)."""
    import json
    return json.loads(json.dumps(v, default=float))


def mpe_masks():
    """Random-rectangle masks plus the all-hole / no-hole corner cases of the MPE table sweep."""
    rng = np.random.default_rng(5)
    out = []
    for (h, w) in ((256, 256), (200, 312), (64, 48)):
        m = np.zeros((h, w), np.float32)
        for _ in range(4):
            y, x = rng.integers(0, h - 8), rng.integers(0, w - 8)
            m[y:y + rng.integers(4, h // 2), x:x + rng.integers(4, w // 2)] = 1
        out.append(m)
    return out + [np.zeros((64, 64), np.float32), np.ones((64, 64), np.float32)]


def quad_boxes():
    """A synthetic page and its text boxes plus two skewed ones, corners in a seeded random order."""
    from mit_b200 import synth
    rng = np.random.default_rng(4)
    page, boxes, _ = synth.make_page(1, 1024, 768, 10)
    extra = [np.array([[100, 100], [400, 130], [390, 190], [95, 160]]), np.array([[50, 50], [90, 60], [70, 400], [30, 390]])]
    return page, [b[rng.permutation(4)] for b in boxes + extra]


def rearrange_images():
    import cv2
    rng = np.random.default_rng(0)
    return [cv2.GaussianBlur(rng.integers(0, 256, shape, dtype=np.uint8), (0, 0), 5) for shape in ((3000, 500, 3), (500, 3300, 3), (1024, 768, 3))]


def rearrange_forward_stub(batch, device=None):
    """Stand-in detector forward for the rearrangement tests: db / mask derived from the batch's channels."""
    import cv2
    batch = np.asarray(batch).astype(np.float32)
    s = batch.shape[1]
    db = np.stack([batch[..., 0] / 255.0, batch[..., 1] / 255.0], 1).astype(np.float32)
    mask = np.stack([cv2.resize(b[..., 2], (s // 2, s // 2)) / 255.0 for b in batch])[:, None].astype(np.float32)
    return db, mask


def contour_case():
    """(probability map, up to 10 of its contours, a random page) for the detector helpers."""
    import cv2
    rng = np.random.default_rng(5)
    prob = cv2.GaussianBlur(rng.random((120, 160)).astype(np.float32), (0, 0), 4)
    cnts, _ = cv2.findContours(((prob > prob.mean()) * 255).astype(np.uint8), cv2.RETR_LIST, cv2.CHAIN_APPROX_SIMPLE)
    cnts = [c.squeeze(1) for c in cnts[:10]]
    img = rng.integers(0, 256, (300, 200, 3), dtype=np.uint8)
    return prob, [c for c in cnts if len(c) >= 3], img


def blob_prob_map():
    """400x600 probability map with rotated / thin / tiny blobs, some below the box threshold."""
    import cv2
    rng = np.random.default_rng(11)
    prob = (0.05 * rng.random((400, 600))).astype(np.float32)
    for _ in range(14):
        cx, cy, w, h, ang = rng.integers(40, 560), rng.integers(40, 360), rng.integers(3, 120), rng.integers(3, 40), rng.uniform(0, 180)
        pts = cv2.boxPoints(((float(cx), float(cy)), (float(w), float(h)), float(ang))).astype(np.int32)
        cv2.fillPoly(prob, [pts], float(rng.uniform(0.55, 0.99)))
    return prob


def refine_page(seed=3, h=768, w=576, n=8):
    """Synthetic page, its text boxes and a raw text mask (the dark strokes dilated 3x3) for mask refinement."""
    import cv2
    from mit_b200 import synth
    page, boxes, _ = synth.make_page(seed, h, w, n)
    raw = cv2.dilate(((page[..., 0] < 100) * 255).astype(np.uint8), np.ones((3, 3), np.uint8))
    return page, boxes, raw


def refine_regions(boxes, k=2):
    import types
    return [types.SimpleNamespace(lines=[b.astype(np.float64) for b in boxes[i:i + k]]) for i in range(0, len(boxes), k)]


REFINE_DISPATCH_CASES = ((3, (768, 576, 8), 0), (9, (640, 480, 6), 20))      # (seed, (h, w, lines), dilation_offset)


def refine_dispatch_case(seed, h, w, n):
    import types
    page, boxes, raw = refine_page(seed, h, w, n)
    line = np.array([[5.0, 5.0], [60.0, 5.0], [60.0, 30.0], [5.0, 30.0]])            # a line without components
    return page, refine_regions(boxes) + [types.SimpleNamespace(lines=[line])], raw


MERGE_PARAMS = (dict(aspect_ratio_tol=1), dict(aspect_ratio_tol=1.3, font_size_ratio_tol=2, char_gap_tolerance=1, char_gap_tolerance2=3))


def merge_random_quads():
    """60 rotated random boxes (int corners) for the text-line merge predicate."""
    rng = np.random.default_rng(8)
    rnd = []
    for t in range(60):
        cx, cy = rng.uniform(200, 500), rng.uniform(200, 500)
        ww, hh = rng.uniform(30, 200), rng.uniform(12, 40)
        if t % 3 == 0:
            ww, hh = hh, ww
        ang = rng.uniform(-0.5, 0.5) if t % 2 else 0.0
        c, s = np.cos(ang), np.sin(ang)
        rnd.append((np.array([[-ww / 2, -hh / 2], [ww / 2, -hh / 2], [ww / 2, hh / 2], [-ww / 2, hh / 2]]) @ np.array([[c, s], [-s, c]]) + [cx, cy]).astype(np.int64))
    return rnd


def merge_random_pages():
    """12 pages of clustered rotated lines ("speech bubbles" of stacked lines + stray lines): per page (corners, colours)."""
    rng = np.random.default_rng(21)
    pages = []
    for _ in range(12):
        pts_list = []
        for blk in range(int(rng.integers(2, 5))):
            bx, by = rng.uniform(100, 900), rng.uniform(100, 700)
            vertical = rng.random() < 0.5
            fs = rng.uniform(18, 40)
            ang = rng.uniform(-0.12, 0.12) if rng.random() < 0.4 else 0.0
            for k in range(int(rng.integers(1, 6))):
                ln = rng.uniform(60, 260)
                w, h = (fs, ln) if vertical else (ln, fs)
                cx, cy = (bx - k * fs * rng.uniform(1.05, 1.6), by + rng.uniform(-8, 8)) if vertical else (bx + rng.uniform(-8, 8), by + k * fs * rng.uniform(1.05, 1.6))
                c, s = np.cos(ang), np.sin(ang)
                pts_list.append((np.array([[-w / 2, -h / 2], [w / 2, -h / 2], [w / 2, h / 2], [-w / 2, h / 2]]) @ np.array([[c, s], [-s, c]]) + [cx, cy]).astype(np.int64))
        cols = [tuple(int(v) for v in rng.integers(0, 256, 6)) for _ in pts_list]
        pages.append((pts_list, cols))
    return pages


def inpaint_case():
    """200x152 random page; mask with two holes, a 130-valued strip and one 127 pixel (the 127 / 128 threshold)."""
    rng = np.random.default_rng(6)
    page = rng.integers(0, 256, (200, 152, 3), dtype=np.uint8)
    mask = np.zeros((200, 152), np.uint8)
    mask[20:50, 10:120] = 255
    mask[120:180, 60:90] = 255
    mask[100:104, 5:40] = 130
    mask[10, 10] = 127
    return page, mask


def detect_variant_stub(quad_cls):
    """`_detect` stand-in for CommonDetector.detect: seeded lines (one of area 1), random raw mask and mask; records its input."""
    async def _detect(self, image, detect_size, text_threshold, box_threshold, unclip_ratio, verbose=False):
        self.seen.append(image.copy())
        h, w = image.shape[:2]
        rng = np.random.default_rng(h * 7919 + w)
        lines = []
        for _ in range(6):
            x0, y0 = int(rng.integers(0, w - 40)), int(rng.integers(0, h - 40))
            bw, bh = int(rng.integers(12, 120)), int(rng.integers(8, 60))
            lines.append(quad_cls(np.array([[x0, y0], [x0 + bw, y0], [x0 + bw, y0 + bh], [x0, y0 + bh]]), "", 0.9))
        lines.append(quad_cls(np.array([[5, 5], [6, 5], [6, 6], [5, 6]]), "", 0.5))
        raw = (rng.random((h, w)) * 255).astype(np.uint8)
        return lines, raw, (rng.random((h, w)) > 0.5).astype(np.uint8) * 255
    return _detect


def detect_variant_cases():
    """(page, invert, gamma, rotate, auto_rotate) for every switch combination on three page sizes."""
    rng = np.random.default_rng(2)
    for (h, w) in ((300, 200), (520, 450), (380, 700)):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        for flags in itertools.product((False, True), repeat=4):
            yield (img,) + flags


def all_weights():
    return dict(dbnet=weights.dbnet_weights(), ocr=weights.ocr_weights(OCR_VOCAB_SMALL),
                lama=weights.lama_weights(9), lama_large=weights.lama_weights(18), mpe=weights.mpe_weights())
