"""Host-side logic (no GPU): geometry / detector post-processing / MPE tables / CTC collapse / rearrangement / the C ABI
surface.  Where a reference helper is the checker, its outputs on seeded inputs are stored under tests/golden."""
import asyncio
import ctypes
import json
import os
import re

import cv2
import numpy as np
import pytest

from mit_b200 import synth
from mit_b200.host import det_post, geometry, mpe, rearrange
from oracle import cases, nets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_header_and_library_agree():
    """Every function declared in include/mitb.h is exported by libmitb.so and bound in mit_b200._lib (no compute calls)."""
    from mit_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "mitb.h")).read()
    declared = set(re.findall(r"\b(mitb_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"mitb_ctx", "mitb_tensor"}
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name)
    assert lib.mitb_ocr_timesteps(647) == 160 and lib.mitb_ocr_timesteps(512) == 127
    assert b"sm_100a" in lib.mitb_version()


def test_no_cpu_fallback():
    """Without a CUDA device context creation fails loudly (and the plugins refuse non-CUDA devices)."""
    import torch
    from mit_b200 import MitbError, plugins
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from mit_b200 import _lib
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.mitb_create(0, ctypes.byref(h)) != 0
    assert b"no CPU fallback" in lib.mitb_last_error(None)
    det = plugins.DBConvNextDetector()
    with pytest.raises(MitbError):
        asyncio.run(det.load("cpu"))
    with pytest.raises(Exception):
        asyncio.run(det.infer(np.zeros((8, 8, 3), np.uint8), 2048, 0.5, 0.7, 2.3))   # infer before load


def test_mpe_tables_match_oracle():
    rng = np.random.default_rng(1)
    for (h, w) in ((256, 256), (120, 312), (64, 48)):
        m = np.zeros((h, w), np.float32)
        for _ in range(4):
            y, x = rng.integers(0, h - 8), rng.integers(0, w - 8)
            m[y:y + rng.integers(4, h // 2), x:x + rng.integers(4, w // 2)] = 1
        a, b = mpe.mpe_tables(m), nets.mpe_tables(m)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    for m in (np.zeros((40, 40), np.float32), np.ones((40, 40), np.float32)):
        a, b = mpe.mpe_tables(m), nets.mpe_tables(m)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_ctc_collapse_matches_oracle():
    from mit_b200.plugins import ctc_collapse
    rng = np.random.default_rng(2)
    idx = rng.integers(0, 4, (5, 60))
    steps = ctc_collapse(idx)
    ref = nets.ctc_greedy(idx, np.zeros(idx.shape, np.float32), np.zeros(idx.shape + (6,), np.float32))
    assert [[int(idx[b, t]) for t in s] for b, s in enumerate(steps)] == [[c[0] for c in l] for l in ref]
    assert [len(s) for s in ctc_collapse(np.zeros((2, 7), np.int64))] == [0, 0]


def test_polygon_helpers():
    sq = np.array([[0, 0], [4, 0], [4, 3], [0, 3]])
    assert geometry.polygon_area(sq) == 12 and geometry.polygon_perimeter(sq) == 14
    assert geometry.hull_area(np.array([[0, 0], [4, 0], [2, 1], [4, 3], [0, 3]])) == 12
    far = sq + np.array([10, 0])
    assert abs(geometry.polygon_distance(sq, far) - 6) < 1e-9
    assert geometry.polygon_distance(sq, sq + 1) == 0 and geometry.polygon_distance(sq, np.array([[1, 1], [2, 1], [2, 2], [1, 2]])) == 0
    diag = np.array([[7, 7], [9, 7], [9, 9], [7, 9]])
    assert abs(geometry.polygon_distance(sq, diag) - 5) < 1e-9        # corner to corner (4,3)->(7,7)


def test_unclip_and_boxes_on_synthetic_prob_map():
    prob = np.zeros((200, 300), np.float32)
    prob[50:80, 40:200] = 0.9
    prob[120:124, 10:14] = 0.9     # too small after unclip filter? (short side 4 -> kept only if >= 3)
    boxes, scores = det_post.boxes_from_prob(prob, 0.5, 0.7, 2.3, 300, 200)
    polys = det_post.polys_from_boxes(boxes, scores, 1.0, 1.0)
    big = [p for p in polys if (p[:, 0].max() - p[:, 0].min()) > 100]
    assert len(big) == 1
    p = big[0]
    # rectangle 160x30 (contour spans 159x29): distance = A*r/L
    d = (159 * 29) * 2.3 / (2 * (159 + 29))
    assert abs((p[:, 0].max() - p[:, 0].min()) - (159 + 2 * d)) <= 2 and abs((p[:, 1].max() - p[:, 1].min()) - (29 + 2 * d)) <= 2
    assert p.sum(axis=1).argmin() == 0                              # starts at the top-left corner


def test_clipper_round_offset_hand_derived_vectors():
    """ClipperOffset (6.4.2) restatement behind `unclip` (dbnet_utils.py:146-152), against vectors derived by hand from the published
    algorithm: square (0,0)-(10,10), delta 2 -> ArcTolerance 0.25 gives pi/acos(1-0.125) = 6.2165 steps per turn, i.e. a 57.91 degree
    rotation per step and round(1.554) = 2 steps per right-angle corner; every vertex = Round(corner + normal*delta), half away from zero:
    corner (0,0): normal (-1,0) -> (-2,0); rotated 57.91 deg -> (-1.063,-1.694) -> (-1,-2); closing normal (0,-1) -> (0,-2); and so on."""
    want = [(-2, 0), (-1, -2), (0, -2), (10, -2), (12, -1), (12, 0), (12, 10), (11, 12), (10, 12), (0, 12), (-2, 11), (-2, 10)]
    sq = [(0, 0), (10, 0), (10, 10), (0, 10)]
    assert det_post.clipper_offset_round(sq, 2.0) == want
    assert det_post.clipper_offset_round(sq[::-1], 2.0) == want                      # FixOrientations: input winding does not matter
    assert det_post.clipper_offset_round(sq + [sq[0]], 2.0) == want                  # closing duplicate stripped by AddPath
    # pyclipper truncates float coordinates toward zero before Clipper sees them
    assert det_post.clipper_offset_round([(0.9, 0.9), (10.9, 0.2), (10.5, 10.7), (0.1, 10.99)], 2.0) == want
    assert det_post.clipper_offset_round([(0, 0), (0, 0), (5, 5)], 2.0) == []        # < 3 distinct vertices: path dropped
    assert det_post.clipper_offset_round(sq, 0) == sq
    # DBNet's use: rectangle 100 x 20, ratio 2.3 -> distance A*r/L = 2000*2.3/240 = 19.1667; sides land on Round(10 - 19.17) = -9,
    # Round(110 + 19.17) = 129, Round(30 + 19.17) = 49; six vertices per corner (round(19.43/4) = 5 arc steps + the closing one)
    box = np.array([[10, 10], [110, 10], [110, 30], [10, 30]], np.float32)
    poly = det_post.clipper_offset_round(box, 2000 * 2.3 / 240)
    xs, ys = [p[0] for p in poly], [p[1] for p in poly]
    assert len(poly) == 24 and (min(xs), max(xs), min(ys), max(ys)) == (-9, 129, -9, 49) and poly[0] == (-9, 10)
    pts, sside = det_post.mini_box(det_post.unclip(box, 2.3))
    assert sside == 58.0 and sorted(map(tuple, np.array(pts).tolist())) == [(-9.0, -9.0), (-9.0, 49.0), (129.0, -9.0), (129.0, 49.0)]


def test_synthetic_page_is_deterministic():
    p1, b1, m1 = synth.make_page(3, 512, 384, 6)
    p2, b2, m2 = synth.make_page(3, 512, 384, 6)
    assert np.array_equal(p1, p2) and np.array_equal(m1, m2) and len(b1) == 6
    assert all(np.array_equal(a, b) for a, b in zip(b1, b2))
    q = synth.make_quads(b1)
    assert [x.direction for x in q] == ["h"] * 3 + ["v"] * 3


def _reference(name):
    """What the reference helpers returned on the seeded inputs of oracle/cases.py (tests/golden, oracle/make_reference_golden.py)."""
    path = os.path.join(ROOT, "tests", "golden", name)
    if name.endswith(".json"):
        with open(path) as f:
            return json.load(f)
    return np.load(path)


def test_quadrilateral_matches_reference():
    page, boxes = cases.quad_boxes()
    want = _reference("ref_host.json")["quadrilateral"]
    assert len(want) == len(boxes)
    for b, ref in zip(boxes, want):
        mine = geometry.Quadrilateral(b, "", 1.0)
        assert mine.pts.tolist() == ref["pts"] and mine.direction == ref["direction"]
        assert abs(mine.aspect_ratio - ref["aspect_ratio"]) < 1e-6 and abs(mine.font_size - ref["font_size"]) < 1e-6
        assert list(mine.aabb) == ref["aabb"]
        assert mine.is_approximate_axis_aligned == ref["axis_aligned"] and abs(mine.angle - ref["angle"]) < 1e-6
        for d in ("h", "v"):
            assert cases.digest(mine.get_transformed_region(page, d, 48)) == ref["region"][d]


def test_rearrange_matches_reference():
    want = _reference("ref_host.json")["rearrange"]
    for img, r in zip(cases.rearrange_images(), want):
        o = rearrange.rearrange_forward(img, cases.rearrange_forward_stub, 1024, 4)
        if r is None:
            assert o[0] is None
        else:
            assert r == [cases.digest(o[0]), cases.digest(o[1])]


def test_detector_helpers_match_reference():
    want = _reference("ref_host.json")
    prob, cnts, img = cases.contour_case()
    assert len(cnts) == len(want["mini_boxes"])
    for c, b in zip(cnts, want["mini_boxes"]):
        a = det_post.mini_box(c)
        assert np.allclose(np.array(a[0]), np.array(b["pts"])) and a[1] == b["sside"]
        assert abs(det_post.box_score(prob, c) - b["score"]) < 1e-12
    for size in (512, 256, 300):
        a, b = det_post.resize_aspect_ratio(img, size, cv2.INTER_LINEAR), want["resize_aspect_ratio"][str(size)]
        assert cases.digest(a[0]) == b["image"] and cases.plain(a[1:]) == b["rest"]


def test_boxes_from_prob_equals_reference_representer():
    """D9 end to end: the reference's own SegDetectorRepresenter.boxes_from_bitmap (dbnet_utils.py:96-144), run with the two absent
    third-party calls adapted (pyclipper.PyclipperOffset -> our Clipper 6.4.2 restatement, shapely Polygon.area/.length -> shoelace /
    perimeter), against host.det_post.boxes_from_prob: contour order, mini boxes, scores, thresholds, unclip call, scale / clip / round /
    roll must agree EXACTLY (boxes int64 and scores)."""
    g = _reference("ref_boxes_from_bitmap.npz")
    prob = cases.blob_prob_map()                               # rotated / thin / tiny blobs, some below box_thresh
    for (dw, dh) in ((600, 400), (1500, 1000)):
        rb, rs = g[f"boxes_{dw}x{dh}"], g[f"scores_{dw}x{dh}"]
        mb, ms = det_post.boxes_from_prob(prob, 0.5, 0.7, 2.3, dw, dh)
        assert rb.shape == mb.shape and len(rb) >= 8
        assert np.array_equal(rb, mb) and np.array_equal(rs, ms)
        assert (mb.reshape(len(mb), -1).sum(1) > 0).sum() >= 3


def test_bench_roofline_object_from_profile():
    """bench.py's roofline block is pure host code: feed it the per-class profile of a recorded run."""
    import json as _json
    import os as _os
    import bench
    prof = _json.loads(open(_os.path.join(bench.ROOT, "profiles", "r01_layers_tma_v13.txt")).read().strip().splitlines()[-1])
    peaks = bench.load_peaks()
    roof = bench.roofline_from_profile(prof, peaks, 1)
    assert roof["kernel"] == "conv_tc" and roof["bound"] == "tensor" and roof["unit"] == "TFLOP/s"
    assert 0.0 < roof["frac"] < 1.0 / 3.0 + 1e-6                       # bf16x3 cannot exceed a third of the bf16 peak
    assert abs(roof["achieved"] * 1e12 * prof["conv_tc"]["ms"] / 1e3 - prof["conv_tc"]["flops"]) < 1e-3 * prof["conv_tc"]["flops"]
    assert roof["traffic"] is None or roof["traffic"] > roof["algorithmic_bytes_per_launch"] * 0.5
    assert set(roof["classes"]) == set(prof)
    assert bench.roofline_from_profile({}, peaks, 1) is None
    _json.dumps(roof)


def test_host_logic_on_empty_and_degenerate_inputs():
    """Edge cases of the host glue: empty detector map, no text lines, all-blank and all-repeat CTC rows, empty shards."""
    import numpy as np
    from mit_b200 import plugins, synth
    from mit_b200.host import det_post, geometry
    from mit_b200.pipeline import shard_indices
    # nothing above threshold -> no boxes, no polygons
    boxes, scores = det_post.boxes_from_prob(np.zeros((64, 48), np.float32), 0.5, 0.7, 2.3, 48, 64)
    assert len(boxes) == 0 and len(scores) == 0
    assert len(det_post.polys_from_boxes(boxes, scores, 1.0, 1.0)) == 0
    # a single saturated blob still yields exactly one box
    prob = np.zeros((64, 96), np.float32); prob[20:40, 10:80] = 0.99
    boxes, scores = det_post.boxes_from_prob(prob, 0.5, 0.7, 2.3, 96, 64)
    assert len(boxes) == 1 and scores[0] > 0.9
    # direction graph / quads of nothing
    assert geometry.generate_text_direction([]) == [] or list(geometry.generate_text_direction([])) == []
    assert len(synth.make_quads([])) == 0
    # CTC collapse: all blank, all the same symbol, alternating with blanks
    idx = np.array([[0, 0, 0, 0], [5, 5, 5, 5], [5, 0, 5, 0], [1, 2, 2, 3]], np.int64)
    kept = plugins.ctc_collapse(idx)
    assert [k.tolist() for k in kept] == [[], [0], [0, 2], [0, 1, 3]]
    # sharding more ranks than pages leaves some ranks empty, never duplicates or drops a page
    parts = [list(shard_indices(3, r, 8)) for r in range(8)]
    assert sorted(sum(parts, [])) == [0, 1, 2] and sum(1 for p in parts if not p) == 5


def test_bench_lama_ffc_figure_from_recorded_launches():
    """The LaMa FFC block figure of the bench line, computed from a recorded per-layer table (profiles/r01_layers_tma_v13.txt)."""
    import json as _json
    import os as _os
    import bench
    lines = open(_os.path.join(bench.ROOT, "profiles", "r01_layers_tma_v13.txt")).read().strip().splitlines()
    prof = _json.loads(lines[-1])
    launches = []
    for ln in lines[2:-1]:
        f = ln.split()
        if len(f) == 7 and f[0].startswith("conv"):
            kind, m, k, n, cnt, ms = f[0], int(f[1]), int(f[2]), int(f[3]), int(f[4]), float(f[5])
            launches += [[kind, m, k, n, ms / cnt]] * cnt
    fig = bench.ffc_block_from_launches(launches, prof, 1, bench.load_peaks())
    assert fig is not None and abs(fig["layers_timed"] - 18) < 1e-9          # 9 blocks x 2 FFC layers per LaMa-MPE page
    assert 300 < fig["us_per_layer"] < 3000 and 0 < fig["hbm_frac"] < 1 and 0 < fig["tensor_frac"] < 1.0 / 3.0
    assert fig["binding_term"] == "tensor"                                    # SURVEY 8d: the fused block is tensor bound
    assert bench.ffc_block_from_launches([], prof, 1, bench.load_peaks()) is None
    _json.dumps(fig)


class _FakeEngine:
    """Stands in for mit_b200.engine.Engine so the plugins' HOST logic can run without a GPU (never part of the product path)."""

    def __init__(self, T=20, V=12):
        self.T, self.V = T, V
        self.calls = []

    def h2d(self, t, dtype=None):
        return t

    def d2h(self, t, scratch=False):
        return t

    def ocr_forward(self, region):
        import numpy as np
        n = region.shape[0]
        rng = np.random.default_rng(5)
        pred = rng.integers(0, self.V, (n, self.T)).astype(np.int32)
        pred[:, ::3] = 0
        logprob = (-rng.random((n, self.T)) * 0.2).astype(np.float32)
        colors = rng.random((n, self.T, 6)).astype(np.float32)
        self.calls.append(("ocr", region.shape))
        return pred, logprob, colors

    def warp_lines(self, page, records, canvas_w, canvas_h=48):
        """Host stand-in for mitb_op_warp_lines_u8: the numpy restatement of the kernel's arithmetic."""
        import numpy as np
        from oracle import warp_ref
        self.calls.append(("warp", len(records), canvas_w))
        return np.stack([warp_ref.warp_line_record(np.asarray(page), r, canvas_w, canvas_h) for r in np.asarray(records)])

    def ctc_collapse(self, pred, logprob, colors):
        """Host stand-in for mitb_op_ctc_collapse (kept steps compacted to the front of each row)."""
        import numpy as np
        from mit_b200 import plugins
        n, T = pred.shape
        counts = np.zeros(n, np.int32)
        steps, chars = np.zeros((n, T), np.int32), np.zeros((n, T), np.int32)
        lp, col = np.zeros((n, T), np.float32), np.zeros((n, T, 6), np.float32)
        for i, st in enumerate(plugins.ctc_collapse(pred)):
            k = len(st)
            counts[i] = k
            steps[i, :k], chars[i, :k], lp[i, :k], col[i, :k] = st, pred[i, st], logprob[i, st], colors[i, st]
        return counts, steps, chars, lp, col

    def mpe_tables_256(self, small):
        import numpy as np
        assert small.shape == (256, 256) and small.dtype == np.uint8
        return np.zeros((1, 256, 256), np.int32), np.zeros((1, 256, 256, 4), np.int32)

    def lama_infer_u8(self, img, mask, rel, direct, composite=True):
        self.calls.append(("lama", img.shape, mask.shape, None if rel is None else rel.shape, composite))
        return (255 - img).copy()


def test_plugin_host_logic_with_a_fake_engine():
    """OCR post-processing (probability / colour statistics, in-place quad mutation) and the inpainter's resize + composite path."""
    import asyncio
    import numpy as np
    from mit_b200 import plugins, synth
    from mit_b200.compat import InpainterConfig, OcrConfig
    page, boxes, mask = synth.make_page(3, 512, 384, 6)
    quads = synth.make_quads(boxes)
    ocr = plugins.Model48pxCTCOCR.__new__(plugins.Model48pxCTCOCR)
    plugins.Model48pxCTCOCR.__init__(ocr)
    ocr.engine = _FakeEngine()
    ocr.dictionary = ["<S>", "</S>", "<SP>"] + [chr(0x3042 + i) for i in range(9)]
    out = asyncio.run(ocr._infer(page, quads, OcrConfig(), False))
    assert len(out) >= 1 and all(q.text and 0 < q.prob <= 1 for q in out)
    assert all(0 <= c <= 255 for q in out for c in (q.fg_r, q.fg_g, q.fg_b, q.bg_r, q.bg_g, q.bg_b))
    # reference arithmetic of the statistics, recomputed per element for the first kept line
    eng = _FakeEngine()
    pred, logprob, colors = eng.ocr_forward(np.zeros((6, 48, 8, 3), np.uint8))
    steps = plugins.ctc_collapse(pred)[0]
    want_prob = np.exp(np.mean([float(v) for v in logprob[0, steps]]))
    assert any(abs(q.prob - want_prob) < 1e-12 for q in out)
    assert ocr.engine.calls[0][0] == "warp"                                          # default path: crops cut on the "device"
    # ... and the reference's own host sequence (cv2 crops) produces the same chunk canvas, hence the same lines
    os.environ["MITB_HOST_CROPS"] = "1"
    try:
        ocr.engine = _FakeEngine()
        out2 = asyncio.run(ocr._infer(page, synth.make_quads(boxes), OcrConfig(), False))
    finally:
        del os.environ["MITB_HOST_CROPS"]
    assert all(c[0] != "warp" for c in ocr.engine.calls) and [(q.text, q.prob) for q in out2] == [(q.text, q.prob) for q in out]

    inp = plugins.LamaMPEInpainter.__new__(plugins.LamaMPEInpainter)
    plugins.LamaMPEInpainter.__init__(inp)
    inp.engine = _FakeEngine()
    page0, mask0 = page.copy(), mask.copy()
    res = asyncio.run(inp._infer(page, mask, InpainterConfig(), 1024, False))           # no resize: device composite
    assert res.shape == page.shape and inp.engine.calls[-1][-1] is True
    res = asyncio.run(inp._infer(page, mask, InpainterConfig(), 256, False))            # resize: host composite with the {0,1} mask
    m01 = (mask0 >= 127)[:, :, None]
    assert res.shape == page.shape and inp.engine.calls[-1][-1] is False
    assert (res[~np.broadcast_to(m01, res.shape)] == page0[~np.broadcast_to(m01, page0.shape)]).all()   # untouched outside the mask
    assert (page == page0).all() and (mask == mask0).all()                               # borrowed inputs were not written


def test_register_swaps_the_reference_registries(monkeypatch):
    """X1: plugins.register() against stand-ins for manga_translator.{detection,ocr,inpainting} that carry the reference's registry
    and cache names (detection/__init__.py:12-27, ocr/__init__.py:11-25, inpainting/__init__.py:13-28) and its Config enums
    (config.py:84-108): the four entries are replaced, stale cached instances are dropped, `get_*` then constructs OUR class with
    no arguments, and other entries are left alone."""
    import enum
    import sys
    import types
    from mit_b200 import compat, plugins

    class Detector(enum.Enum):
        default = "default"
        dbconvnext = "dbconvnext"

    class Ocr(enum.Enum):
        ocr32px = "32px"
        ocr48px_ctc = "48px_ctc"

    class Inpainter(enum.Enum):
        default = "default"
        lama_mpe = "lama_mpe"
        lama_large = "lama_large"

    class Old:
        pass

    det = types.ModuleType("manga_translator.detection")
    det.DETECTORS, det.detector_cache = {Detector.default: Old, Detector.dbconvnext: Old}, {Detector.dbconvnext: Old(), Detector.default: Old()}
    ocr = types.ModuleType("manga_translator.ocr")
    ocr.OCRS, ocr.ocr_cache = {Ocr.ocr32px: Old, Ocr.ocr48px_ctc: Old}, {Ocr.ocr48px_ctc: Old()}
    inp = types.ModuleType("manga_translator.inpainting")
    inp.INPAINTERS, inp.inpainter_cache = {Inpainter.default: Old, Inpainter.lama_mpe: Old, Inpainter.lama_large: Old}, {Inpainter.lama_large: Old()}
    cfg = types.ModuleType("manga_translator.config")
    cfg.Detector, cfg.Ocr, cfg.Inpainter = Detector, Ocr, Inpainter
    root = types.ModuleType("manga_translator")
    root.detection, root.ocr, root.inpainting, root.config = det, ocr, inp, cfg
    for name, mod in (("manga_translator", root), ("manga_translator.detection", det), ("manga_translator.ocr", ocr),
                      ("manga_translator.inpainting", inp), ("manga_translator.config", cfg)):
        monkeypatch.setitem(sys.modules, name, mod)
    monkeypatch.setattr(compat, "HAVE_REFERENCE", True)
    plugins.register()
    assert det.DETECTORS[Detector.dbconvnext] is plugins.DBConvNextDetector and det.DETECTORS[Detector.default] is Old
    assert ocr.OCRS[Ocr.ocr48px_ctc] is plugins.Model48pxCTCOCR and ocr.OCRS[Ocr.ocr32px] is Old
    assert inp.INPAINTERS[Inpainter.lama_mpe] is plugins.LamaMPEInpainter and inp.INPAINTERS[Inpainter.lama_large] is plugins.LamaLargeInpainter
    assert inp.INPAINTERS[Inpainter.default] is Old
    assert Detector.dbconvnext not in det.detector_cache and Detector.default in det.detector_cache
    assert not ocr.ocr_cache and not inp.inpainter_cache
    # the registries construct plugins with no arguments (detection/__init__.py:25-27)
    for cls in (det.DETECTORS[Detector.dbconvnext], ocr.OCRS[Ocr.ocr48px_ctc], inp.INPAINTERS[Inpainter.lama_mpe], inp.INPAINTERS[Inpainter.lama_large]):
        obj = cls()
        with pytest.raises(Exception):
            asyncio.run(obj.infer())                                   # infer before load raises (inference.py:349-350)
    # mask refinement is a module-level import in the orchestrator (manga_translator.py:34): register(mask_refinement=True) rebinds it
    orch = types.ModuleType("manga_translator.manga_translator")
    orch.dispatch_mask_refinement = Old
    root.manga_translator = orch
    monkeypatch.setitem(sys.modules, "manga_translator.manga_translator", orch)
    plugins.register(mask_refinement=True)
    from mit_b200 import mask_refinement
    assert orch.dispatch_mask_refinement is mask_refinement.dispatch
    import inspect
    assert list(inspect.signature(mask_refinement.dispatch).parameters)[:8] == ["text_regions", "raw_image", "raw_mask", "method", "dilation_offset",
                                                                                "ignore_bubble", "verbose", "kernel_size"]      # __init__.py:9
    monkeypatch.setattr(compat, "HAVE_REFERENCE", False)
    from mit_b200 import MitbError
    with pytest.raises(MitbError):
        plugins.register()


def test_detect_variants_and_bubble_filter_standalone():
    """D12 / O10 without the reference package: CommonDetector.detect's border / rotate / invert / gamma variants around a stub `_detect`
    (detection/common.py:12-135) and utils/bubble.is_ignore."""
    from mit_b200 import plugins
    from mit_b200.compat import Quadrilateral
    from mit_b200.host import bubble

    class Stub(plugins.DBConvNextDetector):
        async def _detect(self, image, *a, **k):
            self.seen = image.copy()
            h, w = image.shape[:2]
            q = Quadrilateral(np.array([[10, 20], [60, 20], [60, 40], [10, 40]]), "", 0.9)
            far = Quadrilateral(np.array([[w - 30, h - 30], [w - 5, h - 30], [w - 5, h - 5], [w - 30, h - 5]]), "", 0.8)
            return [q, far], np.full((h // 2, w // 2), 7, np.uint8), None

    det = Stub()
    img = np.full((300, 200, 3), 200, np.uint8)
    img[20:40, 10:60] = 30
    # short side < 400: zero border to a 400 square, results cropped back, lines wholly inside the border dropped
    tl, raw, _ = asyncio.run(det.detect(img, 2048, 0.5, 0.7, 2.3, False, False, False))
    assert det.seen.shape == (400, 400, 3) and (det.seen[:300, :200] == img).all() and det.seen[300:].max() == 0
    assert raw.shape == (300, 200) and len(tl) == 1 and tl[0].pts.max() <= 300
    # inversion and gamma are applied to what the network sees
    asyncio.run(det.detect(img, 2048, 0.5, 0.7, 2.3, True, False, False))
    assert det.seen[25, 20, 0] == 255 - 30
    asyncio.run(det.detect(img, 2048, 0.5, 0.7, 2.3, False, True, False))
    assert det.seen.dtype == np.uint8
    # rotation: the network sees the page rotated clockwise, boxes and mask come back in page coordinates
    big = np.full((500, 450, 3), 200, np.uint8)
    tl, raw, _ = asyncio.run(det.detect(big, 2048, 0.5, 0.7, 2.3, False, False, True))
    assert det.seen.shape == (450, 500, 3) and raw.shape == (250, 225)
    assert all(0 <= p[0] <= 450 and 0 <= p[1] <= 500 for t in tl for p in t.pts)
    # bubble filter: plain white frame -> keep, mixed frame -> ignore, coloured crop -> ignore, parameter out of range -> off
    white = np.full((48, 120, 3), 250, np.uint8)
    mixed = white.copy(); mixed[:, :60] = 5
    colour = white.copy(); colour[10:30, 10:60] = (250, 20, 20)
    assert not bubble.is_ignore(white, 10) and bubble.is_ignore(mixed, 10) and bubble.is_ignore(colour, 10) and not bubble.is_ignore(mixed, 0)


def _random_line_quads(rng, H, W, n):
    """Rotated rectangles with integer corners, some hanging over the page border, some vertical."""
    quads = []
    for t in range(n):
        cx, cy = rng.uniform(0, W), rng.uniform(0, H)
        ww, hh = rng.uniform(40, 500), rng.uniform(20, 80)
        if t % 3 == 0:
            ww, hh = hh, ww
        ang = rng.uniform(-0.35, 0.35) if t % 4 else 0.0
        c, s = np.cos(ang), np.sin(ang)
        pts = np.array([[-ww / 2, -hh / 2], [ww / 2, -hh / 2], [ww / 2, hh / 2], [-ww / 2, hh / 2]]) @ np.array([[c, s], [-s, c]]) + [cx, cy]
        quads.append(pts.astype(np.int64))
    return quads


def test_warp_oracle_equals_cv2():
    """Pins oracle/warp_ref.py (the restatement of OpenCV's warpPerspective the CUDA kernel is checked against) on the installed cv2:
    bit-exact on random line quads, both strip orientations, incl. quads clipped by the page border."""
    from oracle import warp_ref
    rng = np.random.default_rng(11)
    page = rng.integers(0, 256, (700, 900, 3), dtype=np.uint8)
    n_px = 0
    for pts in _random_line_quads(rng, 700, 900, 40):
        q = geometry.Quadrilateral(pts, "", 1.0)
        for d in ("h", "v"):
            (x1, y1, x2, y2), M, (w, h) = geometry.warp_setup(q, 700, 900, d, 48)
            if M is None or x2 <= x1 or y2 <= y1:
                continue
            crop = page[y1:y2, x1:x2]
            ref = cv2.warpPerspective(crop, M, (w, h))
            assert np.array_equal(warp_ref.warp_perspective(crop, M, w, h), ref)
            # ... and the line-record form (what the kernel consumes) reproduces get_transformed_region incl. the rotation
            rec, cw = geometry.warp_record(q, 700, 900, d, 48)
            region = q.get_transformed_region(page, d, 48)
            assert cw == region.shape[1] and region.shape[0] == 48
            line = warp_ref.warp_line_record(page, rec, cw + 135)
            assert np.array_equal(line[:, :cw], region) and not line[:, cw:].any()
            n_px += region.size
    assert n_px > 10 ** 6
    tab = warp_ref.bilinear_itab()
    assert tab[0].tolist() == [32767, 0, 0, 1] and (tab.sum(1) == 32768).all()


def test_traffic_summary_tooling(tmp_path):
    """tools/ncu_traffic.py on the committed ncu launch list (sparse conv launches separated from the dense class, every launch
    classified) and bench.latest_traffic_summary (natural version order, summary of the current CUDA sources preferred)."""
    import importlib.util
    import json as _json
    import bench
    spec = importlib.util.spec_from_file_location("ncu_traffic", os.path.join(ROOT, "tools", "ncu_traffic.py"))
    nt = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(nt)
    src = os.path.join(ROOT, "profiles", "r02_ncu_launches_v17_1page.csv")
    dst = tmp_path / "t.json"
    nt.main(src, str(dst))
    doc = _json.load(open(dst))
    cls = doc["classes"]
    assert cls["conv_tc_sparse"]["launches"] == 27 and cls["conv_tc"]["launches"] > 450           # 12 sparse convs + 12 tile maps + 3 splits
    assert abs(doc["conv_class_dram_bytes_per_page"] - cls["conv_tc"]["dram_bytes"]) < 1 and 30e9 < cls["conv_tc"]["dram_bytes"] < 45e9
    assert abs(sum(c["share_of_time"] for c in cls.values()) - 1.0) < 1e-9 and cls.get("other", {"launches": 0})["launches"] < 20
    d, name = bench.latest_traffic_summary()
    assert name.startswith("r02_ncu_traffic_v") and int(re.search(r"_v(\d+)", name).group(1)) >= 17
    committed = _json.load(open(os.path.join(ROOT, "profiles", name)))
    assert committed["csrc_sha"] == bench.csrc_hash(), "profiles/*_ncu_traffic_*.json was not regenerated for the current CUDA sources"
