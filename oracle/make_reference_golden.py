"""TEST INFRASTRUCTURE -- generates the tests/golden/ref_*.{npz,json} fixtures by running the UNMODIFIED reference code
(imported through oracle/refload.py; MITB_REFERENCE_ROOT names the reference checkout) on the seeded inputs of oracle/cases.py.
The tests that pin the oracle and the host ports on the reference's own code compare against these fixtures, so they run
without the reference tree.  Where the reference code calls a third-party library that is not installed (pyclipper, shapely,
pydensecrf), it runs with that library bound to the repository's restatement, exactly as the tests did when they ran it live.

  python -m oracle.make_reference_golden [section ...]     (default: every section; e.g. `ocr_long` writes ref_ocr_long.npz only)

Large arrays that must match exactly are stored as oracle.cases.digest() values; one dense output is stored as a strided
sample.  No file is larger than 1 MB.
"""
from __future__ import annotations

import asyncio
import importlib
import importlib.util
import itertools
import json
import logging
import os
import sys
import types
import warnings

import numpy as np
import torch

from . import cases, mask_refine_ref as R, nets, refload, weights

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
DBNET_SAMPLE_STRIDE = 3          # every 3rd element of the flattened [1,2,256,512] output (512 % 3 != 0: all columns are hit)
PKG_ROOT = os.path.join(os.path.dirname(os.path.dirname(OUT)), "manga-image-translator_b200")


def _save_npz(name, **arrays):
    np.savez_compressed(os.path.join(OUT, name), **arrays)


def _save_json(name, doc):
    with open(os.path.join(OUT, name), "w") as f:
        json.dump(doc, f, indent=0, sort_keys=True)
        f.write("\n")


# ------------------------------------------------------------------------------------------------ restated third-party libraries
class _Offset:
    def AddPath(self, box, jt, et):
        self.box = box

    def Execute(self, d):
        from mit_b200.host import det_post
        return [det_post.clipper_offset_round(self.box, d)]


_PYCLIPPER = type("pc", (), dict(PyclipperOffset=_Offset, JT_ROUND=1, ET_CLOSEDPOLYGON=2))


class _GeomPolygon:
    """shapely Polygon / MultiPoint bound to host.geometry (area, length, convex hull, distance)."""

    def __init__(self, pts):
        from mit_b200.host import geometry
        self.g = geometry
        self.p = np.asarray(pts, dtype=np.float64).reshape(-1, 2)

    @property
    def area(self):
        return self.g.polygon_area(self.p)

    @property
    def length(self):
        return self.g.polygon_perimeter(self.p)

    @property
    def convex_hull(self):
        return _GeomPolygon(self.g._hull(self.p))

    def distance(self, other):
        return self.g.polygon_distance(self.p, other.p)


def _bind_geometry():
    G = importlib.import_module("manga_translator.utils.generic")
    du = importlib.import_module("manga_translator.detection.default_utils.dbnet_utils")
    saved = (du.pyclipper, du.Polygon, G.Polygon, G.MultiPoint)
    du.pyclipper = _PYCLIPPER
    du.Polygon = G.Polygon = G.MultiPoint = _GeomPolygon

    def restore():
        du.pyclipper, du.Polygon, G.Polygon, G.MultiPoint = saved
    return restore


def _reference_mask_refinement():
    """The reference's own mask_refinement package with shapely.geometry.Polygon and pydensecrf bound to the oracle's restatements."""
    class _Pt:
        def __init__(self, x, y):
            self.x, self.y = x, y

    class Polygon:
        def __init__(self, pts):
            self.p = np.asarray(pts, dtype=np.float64).reshape(-1, 2)

        @property
        def area(self):
            return R.poly_area(self.p) if len(self.p) >= 3 else 0.0

        @property
        def centroid(self):                                     # only ever asked of the component rectangle
            return _Pt(float(self.p[:, 0].mean()), float(self.p[:, 1].mean()))

        def intersection(self, other):                          # `other` is the axis-aligned component rectangle
            x0, y0, x1, y1 = other.p[:, 0].min(), other.p[:, 1].min(), other.p[:, 0].max(), other.p[:, 1].max()
            return Polygon(np.asarray(R.clip_poly_rect(self.p, x0, y0, x1, y1)).reshape(-1, 2))

        def distance(self, pt):
            return R.point_poly_distance(self.p, pt.x, pt.y)

    class DenseCRF2D:
        def __init__(self, w, h, n):
            self.w, self.h, self.n = w, h, n

        def setUnaryEnergy(self, u):
            self.u = np.asarray(u, dtype=np.float32)

        def addPairwiseGaussian(self, sxy, compat, kernel=None, normalization=None):
            self.g = (float(sxy), float(compat))

        def addPairwiseBilateral(self, sxy, srgb, rgbim, compat, kernel=None, normalization=None):
            self.b, self.rgb = (float(sxy), float(srgb), float(compat)), np.asarray(rgbim)

        def inference(self, n):
            assert self.rgb.shape[:2] == (self.h, self.w)
            return R.dense_crf_2d(self.rgb, self.u, n, self.g[0], self.g[1], self.b[0], self.b[1], self.b[2])

    sys.modules["shapely.geometry"].Polygon = Polygon
    dcrf = types.ModuleType("pydensecrf.densecrf")
    dcrf.DenseCRF2D, dcrf.DIAG_KERNEL, dcrf.NO_NORMALIZATION = DenseCRF2D, 1, 0
    putils = types.ModuleType("pydensecrf.utils")
    putils.unary_from_softmax = lambda sm, scale=None, clip=1e-5: (-np.log(np.clip(sm, clip, 1.0))).reshape([sm.shape[0], -1]).astype(np.float32)
    putils.compute_unary = None
    pkg = types.ModuleType("pydensecrf")
    pkg.__path__ = []
    pkg.densecrf, pkg.utils = dcrf, putils
    sys.modules.update({"pydensecrf": pkg, "pydensecrf.densecrf": dcrf, "pydensecrf.utils": putils})
    path = os.path.join(refload.REF_ROOT, "manga_translator", "mask_refinement")
    spec = importlib.util.spec_from_file_location("manga_translator.mask_refinement", os.path.join(path, "__init__.py"), submodule_search_locations=[path])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["manga_translator.mask_refinement"] = mod
    spec.loader.exec_module(mod)
    return mod


# ------------------------------------------------------------------------------------------------ networks
def networks(ref):
    specs = {}
    for name, module, sd in (("dbnet", ref["det"].DBNetConvNext(), None), ("ocr300", ref["ocr"].OCR(["x"] * 300, 768), None)):
        specs[name] = {k: list(v.shape) for k, v in module.state_dict().items() if "num_batches_tracked" not in k and not k.endswith("pe.pe")}
    for nb in (9, 18):
        lf = ref["lama"].LamaFourier(build_discriminator=False, use_mpe=nb == 9, large_arch=nb == 18)
        specs[f"lama{nb}"] = {k: list(v.shape) for k, v in lf.generator.state_dict().items() if "num_batches_tracked" not in k}
        if nb == 9:
            specs["mpe"] = {k: list(v.shape) for k, v in lf.mpe.state_dict().items() if "num_batches_tracked" not in k}
            rel_pos_emb = lf.mpe.rel_pos_emb.weight.detach().numpy()
    _save_json("ref_state_dict_specs.json", specs)

    sd = weights.dbnet_weights(seed=2)
    net = ref["det"].DBNetConvNext().eval()
    net.load_state_dict(sd)
    _, x = cases.dbnet_case(256, 512, seed=21)
    r_db, r_mask = net(x)
    _save_npz("ref_dbnet_256x512.npz", db_sample=r_db.numpy().reshape(-1)[::DBNET_SAMPLE_STRIDE], mask=r_mask.numpy())

    V = 300
    sd = weights.ocr_weights(V, seed=3)
    ocr = ref["ocr"].OCR(weights.synthetic_dictionary(V), 768).eval()
    ocr.load_state_dict(sd, strict=False)
    out = {}
    for wp in (143, 200, 331):
        _, x = cases.ocr_case(3, wp, seed=wp)
        rl, rc = ocr(x)
        dec = ocr.decode(x, [0] * 3, 0)
        chars = np.full((3, max(1, max(len(l) for l in dec))), -1, np.int64)
        for i, l in enumerate(dec):
            chars[i, :len(l)] = [int(c[0]) for c in l]
        out.update({f"logits_{wp}": rl.numpy(), f"colors_{wp}": rc.numpy(), f"decoded_{wp}": chars})
    _save_npz("ref_ocr_widths.npz", **out)

    lf = ref["lama"].LamaFourier(build_discriminator=False, use_mpe=True)
    out = {"rel_pos_emb": rel_pos_emb}
    for i, m in enumerate(cases.mpe_masks()):
        rel, _, direct = lf.load_masked_position_encoding(m)
        out[f"rel_{i}"], out[f"direct_{i}"] = rel, direct
    sd, msd = weights.lama_weights(9, seed=4), weights.mpe_weights(seed=4)
    lf.generator.load_state_dict(sd)
    lf.mpe.load_state_dict(msd)
    lf.eval()
    img, mask = cases.lama_case(88, 120, seed=41)
    out["odd_88x120"] = lf(img.clone(), mask).numpy()
    _save_npz("ref_lama.npz", **out)


OCR_LONG_WIDTHS = (2439, 8196)   # T = 608 (a caption across a 1536 px page, 32 px tall) and T = 2048, the positional table's length
OCR_LONG_TOO_WIDE = 8200         # T = 2049


def ocr_long(ref):
    """The reference OCR on two-line chunks of the longest lines it reads.  Compact per-step results instead of the logits (at T = 2048
    those alone are 2.4 MB): argmax, max log-softmax, top-2 logit margin, clamped colours, and the decoded character ids."""
    V = 300
    ocr = ref["ocr"].OCR(weights.synthetic_dictionary(V), 768).eval()
    ocr.load_state_dict(weights.ocr_weights(V, seed=3), strict=False)
    out = {}
    for wp in OCR_LONG_WIDTHS:
        _, x = cases.ocr_case(2, wp, seed=wp)
        rl, rc = ocr(x)
        lp, idx = rl.log_softmax(2).max(2)
        top2 = rl.topk(2, dim=-1).values
        dec = ocr.decode(x, [0] * 2, 0)
        chars = np.full((2, max(1, max(len(l) for l in dec))), -1, np.int16)
        for i, l in enumerate(dec):
            chars[i, :len(l)] = [int(c[0]) for c in l]
        out.update({f"argmax_{wp}": idx.numpy().astype(np.int16), f"logprob_{wp}": lp.numpy(),
                    f"margin_{wp}": (top2[..., 0] - top2[..., 1]).numpy(), f"colors_{wp}": rc.clamp(0, 1).numpy(), f"decoded_{wp}": chars})
    _, x = cases.ocr_case(2, OCR_LONG_TOO_WIDE, seed=OCR_LONG_TOO_WIDE)
    try:
        ocr(x)
        out["too_wide_raises"] = np.array(False)
    except RuntimeError:                          # x + pe[:, :T] with T = 2049 against a 2048-row table: a shape mismatch
        out["too_wide_raises"] = np.array(True)
    _save_npz("ref_ocr_long.npz", **out)


# ------------------------------------------------------------------------------------------------ the three `_infer` glue paths
def infer_glue(ref):
    from mit_b200 import synth
    U = ref["utils"]
    out = {}
    restore = _bind_geometry()
    try:
        det = ref["det"]
        sd = {k: v.clone() for k, v in weights.dbnet_weights().items()}
        sd["conv_db.binarize.4.bias"] -= 1.0
        net = det.DBNetConvNext().eval()
        net.load_state_dict(sd)
        det.MODEL = net
        me = types.SimpleNamespace(device="cpu", logger=logging.getLogger("ref-det"), model=net)
        for k, (page, detect_size) in enumerate(((synth.make_page(5, 512, 384, 6)[0], 512), (synth.make_page(4, 384, 384, 5)[0], 512))):
            lines, mask, _ = asyncio.run(det.DBConvNextDetector._infer(me, page, detect_size, 0.5, 0.6, 2.3))
            out[f"det{k}_pts"] = np.stack([l.pts for l in lines])
            out[f"det{k}_prob"] = np.array([l.prob for l in lines], np.float64)
            out[f"det{k}_direction"] = np.array([l.direction for l in lines])
            out[f"det{k}_mask"] = mask

        V = cases.OCR_VOCAB_SMALL
        dictionary = weights.synthetic_dictionary(V)
        model = ref["ocr"].OCR(dictionary, 768).eval()
        model.load_state_dict(weights.ocr_weights(V), strict=False)
        common = sys.modules["manga_translator.ocr.common"]
        page, boxes, _ = synth.make_page(3, 512, 384, 6)
        me = types.SimpleNamespace(device="cpu", use_gpu=False, logger=logging.getLogger("ref-ocr"), model=model)
        me._generate_text_direction = lambda bboxes: common.CommonOCR._generate_text_direction(me, bboxes)
        cfg = types.SimpleNamespace(ignore_bubble=0, prob=0.0)
        lines = asyncio.run(ref["ocr"].Model48pxCTCOCR._infer(me, page, [U.Quadrilateral(b.copy(), "", 1.0) for b in boxes], cfg, False))
        out["ocr_pts"] = np.stack([l.pts for l in lines])
        out["ocr_text"] = np.array([l.text for l in lines])
        out["ocr_prob"] = np.array([l.prob for l in lines], np.float64)
        out["ocr_colors"] = np.array([(l.fg_r, l.fg_g, l.fg_b, l.bg_r, l.bg_g, l.bg_b) for l in lines], np.int64)
    finally:
        restore()

    lama = ref["lama"]
    lf = lama.LamaFourier(build_discriminator=False, use_mpe=True)
    lf.generator.load_state_dict(weights.lama_weights(9))
    lf.mpe.load_state_dict(weights.mpe_weights())
    lf.eval()
    me = types.SimpleNamespace(device="cpu", logger=logging.getLogger("ref-inp"), model=lf)
    page, mask = cases.inpaint_case()
    for size in (1024, 128):
        out[f"inpaint_{size}"] = asyncio.run(lama.LamaMPEInpainter._infer(me, page.copy(), mask.copy(), types.SimpleNamespace(inpainting_precision="fp32"), size, False))
    _save_npz("ref_infer_glue.npz", **out)


def detect_variants(ref):
    rc = importlib.import_module("manga_translator.detection.common")

    class RefDet(rc.CommonDetector):
        _detect = cases.detect_variant_stub(ref["utils"].Quadrilateral)

    runs = []
    restore = _bind_geometry()
    try:
        for img, invert, gamma, rotate, auto in cases.detect_variant_cases():
            r = RefDet()
            r.seen = []
            lines, raw, mask = asyncio.run(r.detect(img.copy(), 1024, 0.5, 0.7, 2.3, invert, gamma, rotate, auto))
            runs.append({"seen": [cases.digest(a) for a in r.seen], "lines": [l.pts.tolist() for l in lines],
                         "raw": cases.digest(raw), "mask": cases.digest(mask)})
    finally:
        restore()
    _save_json("ref_detect_variants.json", {"runs": runs})


# ------------------------------------------------------------------------------------------------ host ports (tests/test_host.py)
def host(ref):
    U = ref["utils"]
    doc = {}
    page, boxes = cases.quad_boxes()
    doc["quadrilateral"] = []
    for b in boxes:
        q = U.Quadrilateral(b, "", 1.0)
        doc["quadrilateral"].append({"pts": q.pts.tolist(), "direction": q.direction, "aspect_ratio": float(q.aspect_ratio),
                                     "font_size": float(q.font_size), "aabb": [int(q.aabb.x), int(q.aabb.y), int(q.aabb.w), int(q.aabb.h)],
                                     "axis_aligned": bool(q.is_approximate_axis_aligned), "angle": float(q.angle),
                                     "region": {d: cases.digest(q.get_transformed_region(page, d, 48)) for d in ("h", "v")}})
    doc["rearrange"] = []
    for img in cases.rearrange_images():
        r = U.det_rearrange_forward(img, cases.rearrange_forward_stub, 1024, 4)
        doc["rearrange"].append(None if r[0] is None else [cases.digest(r[0]), cases.digest(r[1])])

    du = importlib.import_module("manga_translator.detection.default_utils.dbnet_utils")
    ip = importlib.import_module("manga_translator.detection.default_utils.imgproc")
    import cv2
    rep = du.SegDetectorRepresenter(0.5, 0.7, unclip_ratio=2.3)
    prob, cnts, img = cases.contour_case()
    doc["mini_boxes"] = []
    for c in cnts:
        pts, sside = rep.get_mini_boxes(c)
        doc["mini_boxes"].append({"pts": np.asarray(pts, np.float64).tolist(), "sside": float(sside), "score": float(rep.box_score_fast(prob, c))})
    doc["resize_aspect_ratio"] = {}
    for size in (512, 256, 300):
        b = ip.resize_aspect_ratio(img, size, cv2.INTER_LINEAR, mag_ratio=1)
        doc["resize_aspect_ratio"][str(size)] = {"image": cases.digest(b[0]), "rest": cases.plain(b[1:])}
    _save_json("ref_host.json", doc)

    saved = (du.pyclipper, du.Polygon)
    du.pyclipper, du.Polygon = _PYCLIPPER, _GeomPolygon
    try:
        prob = cases.blob_prob_map()
        out = {}
        for (dw, dh) in ((600, 400), (1500, 1000)):
            out[f"boxes_{dw}x{dh}"], out[f"scores_{dw}x{dh}"] = rep.boxes_from_bitmap(prob, prob > 0.5, dw, dh)
        _save_npz("ref_boxes_from_bitmap.npz", **out)
    finally:
        du.pyclipper, du.Polygon = saved


# ------------------------------------------------------------------------------------------------ mask refinement
def mask_refinement(ref):
    U = ref["utils"]
    out = {}
    _, boxes, _ = cases.refine_page()
    for i, b in enumerate(boxes + [np.array([[10, 20], [200, 35], [195, 80], [5, 66]])]):
        r = R._Line(U.Quadrilateral, b * (2.0 / 3.0))
        out[f"line{i}_pts"], out[f"line{i}_font_size"], out[f"line{i}_aabb"] = r.pts, np.float64(r.font_size), np.asarray(r.aabb_xywh)
    mod = _reference_mask_refinement()
    for seed, (h, w, n), offset in cases.REFINE_DISPATCH_CASES:
        page, regions, raw = cases.refine_dispatch_case(seed, h, w, n)
        out[f"dispatch_{seed}"] = asyncio.run(mod.dispatch(regions, page, raw.copy(), "fit_text", offset, 0, False, 3))
    _save_npz("ref_mask_refinement.npz", **out)


# ------------------------------------------------------------------------------------------------ text-line merge
def textline_merge(ref):
    U = ref["utils"]
    G = importlib.import_module("manga_translator.utils.generic")
    common = sys.modules["manga_translator.ocr.common"]
    from mit_b200.host import geometry

    class Polygon:
        def __init__(self, pts):
            self.p = np.asarray(pts, dtype=np.float64).reshape(-1, 2)

        def distance(self, other):
            return geometry.polygon_distance(self.p, other.p)

    with open(os.path.join(OUT, "textline_merge.json")) as f:
        known = [[np.array(l) for l in c["lines"]] for c in json.load(f)["cases"]]
    doc = {"predicate": []}
    saved = G.Polygon
    G.Polygon = Polygon
    try:
        for pts_list in known + [cases.merge_random_quads()]:
            quads = [U.Quadrilateral(p, "", 1.0) for p in pts_list]
            for q, p in zip(quads, pts_list):                 # the angled branch asks Quadrilateral.poly_distance (hull polygons)
                q.__dict__["polygon"] = Polygon(geometry._hull(geometry.Quadrilateral(p, "", 1.0).pts))
            doc["predicate"].append(["".join("1" if G.quadrilateral_can_merge_region(quads[u], quads[v], **params) else "0"
                                             for u, v in itertools.combinations(range(len(quads)), 2)) for params in cases.MERGE_PARAMS])
    finally:
        G.Polygon = saved

    path = os.path.join(refload.REF_ROOT, "manga_translator", "textline_merge", "__init__.py")
    spec = importlib.util.spec_from_file_location("manga_translator.textline_merge", path, submodule_search_locations=[os.path.dirname(path)])
    ref_merge = importlib.util.module_from_spec(spec)
    sys.modules["manga_translator.textline_merge"] = ref_merge
    spec.loader.exec_module(ref_merge)
    saved = (G.Polygon, G.MultiPoint, ref_merge.Polygon)
    G.Polygon, G.MultiPoint, ref_merge.Polygon = _GeomPolygon, _GeomPolygon, _GeomPolygon
    doc["pages"] = []
    try:
        for pts_list, cols in cases.merge_random_pages():
            quads = [U.Quadrilateral(p, f"t{i}", 0.9, *c) for i, (p, c) in enumerate(zip(pts_list, cols))]
            for q in quads:
                q.assigned_direction = q.direction
            regions = [([quads.index(q) for q in tl], [int(v) for v in fg], [int(v) for v in bg])
                       for tl, fg, bg in ref_merge.merge_bboxes_text_region(quads, 1000, 800)]
            directions = [[quads.index(q), d] for q, d in common.CommonOCR._generate_text_direction(None, quads)]
            doc["pages"].append({"regions": regions, "directions": directions})
    finally:
        G.Polygon, G.MultiPoint, ref_merge.Polygon = saved
    _save_json("ref_textline_merge.json", doc)


SECTIONS = {f.__name__: f for f in (networks, ocr_long, infer_glue, detect_variants, host, mask_refinement, textline_merge)}


def main(sections=None):
    sections = sections or list(SECTIONS)
    unknown = [s for s in sections if s not in SECTIONS]
    if unknown:
        raise SystemExit(f"unknown section(s) {unknown}; choose from {list(SECTIONS)}")
    warnings.filterwarnings("ignore")
    if PKG_ROOT not in sys.path:
        sys.path.insert(0, PKG_ROOT)
    torch.set_grad_enabled(False)
    ref = refload.load()
    for name in sections:
        SECTIONS[name](ref)
    for f in sorted(os.listdir(OUT)):
        if f.startswith("ref_"):
            print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
