"""Pins the oracle restatement against the unmodified reference modules.  What the reference computed on these seeded inputs is
stored under tests/golden/ref_*.{npz,json} (written by oracle/make_reference_golden.py, which runs the reference code), so the
comparison runs without the reference tree."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import cases, nets, weights

torch.set_grad_enabled(False)


@pytest.fixture(scope="module")
def ref(golden_dir):
    def load(name):
        path = os.path.join(golden_dir, name)
        if name.endswith(".json"):
            with open(path) as f:
                return json.load(f)
        return np.load(path)
    return load


def _check_keys(spec, sd):
    have = {k: list(v.shape) for k, v in sd.items()}
    assert spec == have


def test_state_dict_specs_match_reference(ref):
    specs = ref("ref_state_dict_specs.json")
    _check_keys(specs["dbnet"], weights.dbnet_weights())
    _check_keys(specs["ocr300"], weights.ocr_weights(300))
    for nb in (9, 18):
        _check_keys(specs[f"lama{nb}"], weights.lama_weights(nb))
    _check_keys(specs["mpe"], weights.mpe_weights())
    assert torch.equal(torch.from_numpy(ref("ref_lama.npz")["rel_pos_emb"]), weights.mpe_weights()["rel_pos_emb.weight"])


def test_dbnet_rectangular(ref):
    from oracle.make_reference_golden import DBNET_SAMPLE_STRIDE
    g = ref("ref_dbnet_256x512.npz")
    sd = weights.dbnet_weights(seed=2)
    _, x = cases.dbnet_case(256, 512, seed=21)
    o_db, o_mask = nets.dbnet_forward(sd, x)
    o_db = o_db.numpy().reshape(-1)[::DBNET_SAMPLE_STRIDE]
    assert np.abs(g["db_sample"] - o_db).max() < 1e-4 and np.abs(g["mask"] - o_mask.numpy()).max() < 1e-5


def test_ocr_widths_and_decode(ref):
    g = ref("ref_ocr_widths.npz")
    V = 300
    sd = weights.ocr_weights(V, seed=3)
    for wp in (143, 200, 331):
        _, x = cases.ocr_case(3, wp, seed=wp)
        rl, rc = torch.from_numpy(g[f"logits_{wp}"]), torch.from_numpy(g[f"colors_{wp}"])
        ol, oc = nets.ocr_forward(sd, x)
        assert (rl - ol).abs().max() < 1e-4 and (rc - oc).abs().max() < 1e-5
        idx, lp, col = nets.ocr_top1(sd, x)
        ref_dec = [[int(c) for c in row if c >= 0] for row in g[f"decoded_{wp}"]]
        mine = nets.ctc_greedy(idx.numpy(), lp.numpy(), col.numpy())
        top2 = rl.topk(2, dim=-1).values
        if (top2[..., 0] - top2[..., 1]).min() > 1e-3:
            assert ref_dec == [[c[0] for c in l] for l in mine]


def test_ocr_long_lines(ref):
    """The oracle on the longest lines the reference reads: T = 608 and T = 2048 (its PositionalEncoding has 2048 rows, so the oracle's
    per-call sinusoid_pe(T) is checked against the reference's table at every position), and the reference refuses T = 2049."""
    from oracle.make_reference_golden import OCR_LONG_TOO_WIDE, OCR_LONG_WIDTHS
    g = ref("ref_ocr_long.npz")
    sd = weights.ocr_weights(300, seed=3)
    for wp in OCR_LONG_WIDTHS:
        _, x = cases.ocr_case(2, wp, seed=wp)
        logits, colors = nets.ocr_forward(sd, x)
        assert logits.shape[1] == (wp // 2) // 2 - 1
        lp, idx = logits.log_softmax(2).max(2)
        top2 = logits.topk(2, dim=-1).values
        safe = g[f"margin_{wp}"] > 1e-3
        assert safe.mean() > 0.99
        assert np.array_equal(idx.numpy()[safe], g[f"argmax_{wp}"][safe])
        assert np.abs(lp.numpy() - g[f"logprob_{wp}"]).max() < 1e-4
        assert np.abs((top2[..., 0] - top2[..., 1]).numpy() - g[f"margin_{wp}"]).max() < 2e-4
        assert np.abs(colors.clamp(0, 1).numpy() - g[f"colors_{wp}"]).max() < 1e-5
        # decode: the oracle's argmax on the safe steps, the reference's on the few near-ties
        mixed = np.where(safe, idx.numpy(), g[f"argmax_{wp}"])
        mine = nets.ctc_greedy(mixed, lp.numpy(), colors.clamp(0, 1).numpy())
        assert [[int(c) for c in row if c >= 0] for row in g[f"decoded_{wp}"]] == [[c[0] for c in l] for l in mine]
    assert (OCR_LONG_TOO_WIDE // 2) // 2 - 1 == 2049 and bool(g["too_wide_raises"])


def test_lama_mpe_tables_random_masks(ref):
    g = ref("ref_lama.npz")
    # random rectangles, then the all-hole and no-hole masks (the reference guards the infinite loop, :778)
    for i, m in enumerate(cases.mpe_masks()):
        orel, odirect = nets.mpe_tables(m)
        assert np.array_equal(g[f"rel_{i}"], orel) and np.array_equal(g[f"direct_{i}"], odirect)


def test_lama_odd_spectrum_sizes(ref):
    sd, msd = weights.lama_weights(9, seed=4), weights.mpe_weights(seed=4)
    img, mask = cases.lama_case(88, 120, seed=41)   # bottleneck 11x15: odd FFT lengths
    r = torch.from_numpy(ref("ref_lama.npz")["odd_88x120"])
    rel, direct = nets.mpe_tables(mask[0, 0].numpy())
    o = nets.lama_forward(sd, msd, img, mask, torch.from_numpy(rel)[None], torch.from_numpy(direct)[None])
    assert (r - o).abs().max() < 2e-5


# ---------------------------------------------------------------------------------------------------------------------
# The three `_infer` glue paths: oracle/pipeline_ref.py (what the GPU plugin tests compare the product with) against the reference's own
# `_infer` methods, executed unmodified on the CPU with a duck-typed `self` and the absent third-party libraries bound to the repo's
# restatements (pyclipper -> Clipper 6.4.2 restatement, shapely -> geometry restatements).  Closes the loop: reference `_infer` ==
# pipeline_ref here, plugin == pipeline_ref on the GPU.
def test_detector_infer_glue_equals_reference_code(ref):
    from mit_b200 import synth
    from oracle import pipeline_ref
    g = ref("ref_infer_glue.npz")
    sd = {k: v.clone() for k, v in weights.dbnet_weights().items()}
    sd["conv_db.binarize.4.bias"] -= 1.0
    for k, (page, detect_size) in enumerate(((synth.make_page(5, 512, 384, 6)[0], 512), (synth.make_page(4, 384, 384, 5)[0], 512))):   # pad path; upscale path
        o_lines, o_mask, _, _ = pipeline_ref.detector_infer(sd, page, detect_size, 0.5, 0.6, 2.3)
        r_pts, r_prob, r_dir, r_mask = g[f"det{k}_pts"], g[f"det{k}_prob"], g[f"det{k}_direction"], g[f"det{k}_mask"]
        assert len(r_pts) == len(o_lines) and len(r_pts) > 3
        for pts, prob, d, b in zip(r_pts, r_prob, r_dir, o_lines):
            assert np.array_equal(pts, b.pts) and prob == b.prob and d == b.direction
        # the stored mask and this one come from two fp32 CPU evaluations of the network (possibly on different CPUs): the x*255
        # truncation may flip a pixel by one where the value sits on a boundary, as in the inpainter glue below
        d = np.abs(r_mask.astype(int) - o_mask.astype(int))
        assert r_mask.dtype == o_mask.dtype == np.uint8 and d.max() <= 1 and (d > 0).mean() < 1e-3, (int(d.max()), float((d > 0).mean()))


def test_ocr_infer_glue_equals_reference_code(ref):
    from mit_b200 import synth
    from mit_b200.host import geometry
    from oracle import pipeline_ref
    g = ref("ref_infer_glue.npz")
    V = cases.OCR_VOCAB_SMALL
    dictionary = weights.synthetic_dictionary(V)
    sd = weights.ocr_weights(V)
    page, boxes, _ = synth.make_page(3, 512, 384, 6)
    o_out = pipeline_ref.ocr_infer(sd, dictionary, page, [geometry.Quadrilateral(b.copy(), "", 1.0) for b in boxes], 0.0)
    assert len(g["ocr_pts"]) == len(o_out) >= 4
    for pts, text, prob, colors, b in zip(g["ocr_pts"], g["ocr_text"], g["ocr_prob"], g["ocr_colors"], o_out):
        assert np.array_equal(pts, b.pts) and str(text) == b.text and len(b.text) > 0
        assert abs(prob - b.prob) < 1e-4 * max(prob, 1e-30)            # the two fp32 network evaluations differ by ~1e-5 in log-probability
        assert tuple(int(c) for c in colors) == (b.fg_r, b.fg_g, b.fg_b, b.bg_r, b.bg_g, b.bg_b)


def test_inpainter_infer_glue_equals_reference_code(ref):
    from oracle import pipeline_ref
    g = ref("ref_infer_glue.npz")
    sd, msd = weights.lama_weights(9), weights.mpe_weights()
    page, mask = cases.inpaint_case()                             # incl. the 127 / 128 threshold quirk (SURVEY I2)
    for size in (1024, 128):                                      # no resize; keep-aspect resize + back
        r = g[f"inpaint_{size}"]
        o, _ = pipeline_ref.lama_infer(sd, msd, page.copy(), mask.copy(), size)
        assert r.dtype == o.dtype == np.uint8 and r.shape == page.shape
        d = np.abs(r.astype(int) - o.astype(int))
        assert d.max() <= 1 and (d > 0).mean() < 1e-3, (int(d.max()), float((d > 0).mean()))     # x*255 truncation of fp32 values 2e-5 apart


def test_common_detector_detect_equals_reference_code(ref):
    """D12: the stand-in `CommonDetector.detect` of mit_b200.compat (border for small pages, rotation, inversion, gamma correction,
    auto-rotation; used when the reference package cannot be imported) against the reference's own `detection/common.py` code, both
    wrapped around the same stub `_detect`: identical text lines, raw mask and mask for every combination of the switches."""
    import asyncio
    import importlib.util
    import sys
    from mit_b200 import compat as _compat_loaded
    from mit_b200.host import geometry
    # a second copy of mit_b200/compat.py imported while `manga_translator` is hidden: the stand-in, even where the package is installed
    hidden = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "manga_translator" or k.startswith("manga_translator.")}
    sys.modules["manga_translator"] = None                       # makes `import manga_translator...` raise ImportError
    try:
        spec = importlib.util.spec_from_file_location("mit_b200._compat_standin", _compat_loaded.__file__)
        compat = importlib.util.module_from_spec(spec)
        sys.modules["mit_b200._compat_standin"] = compat
        spec.loader.exec_module(compat)
    finally:
        del sys.modules["manga_translator"]
        sys.modules.update(hidden)
    assert not compat.HAVE_REFERENCE

    class OurDet(compat.OfflineDetector):
        _detect = cases.detect_variant_stub(geometry.Quadrilateral)

        async def _load(self, device):
            pass

        async def _unload(self):
            pass

        async def _infer(self, *a, **k):
            raise AssertionError("not used: `_detect` is stubbed")

    runs = ref("ref_detect_variants.json")["runs"]
    variants = list(cases.detect_variant_cases())
    assert len(runs) == len(variants) == 48
    for want, (img, invert, gamma, rotate, auto) in zip(runs, variants):
        o = OurDet()
        o.seen = []
        ot, oraw, omask = asyncio.run(o.detect(img.copy(), 1024, 0.5, 0.7, 2.3, invert, gamma, rotate, auto))
        assert want["seen"] == [cases.digest(a) for a in o.seen], (img.shape, invert, gamma, rotate, auto)
        assert want["lines"] == [np.asarray(t.pts).tolist() for t in ot]
        assert want["raw"] == cases.digest(oraw) and want["mask"] == cases.digest(omask)
