"""Text-line merge (SURVEY 8f, N3) against the reference's own known-answer tests: tests/golden/textline_merge.json holds the
quadrilaterals and expected groupings of manga_translator's test/test_textline_merge.py (extracted by oracle/make_merge_golden.py)."""
import json
import os

import numpy as np
import pytest

from mit_b200.host import geometry, textline_merge
from mit_b200.host.geometry import Quadrilateral

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "textline_merge.json")
CASES = json.load(open(GOLDEN))["cases"]


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_merge_matches_reference_known_answers(case):
    quads = [Quadrilateral(np.array(l), "", 1) for l in case["lines"]]
    regions = textline_merge.dispatch(quads, case["width"], case["height"])
    got = {tuple(sorted(r.line_indices)) for r in regions}
    want = {tuple(c) for c in case["expected"]}
    assert got == want
    assert sorted(i for r in regions for i in r.line_indices) == list(range(len(quads)))      # a partition of the lines


def test_merge_region_fields_and_ordering():
    # three stacked horizontal lines + one far-away vertical line
    lines = [[[100, 100], [400, 100], [400, 140], [100, 140]], [[100, 150], [400, 150], [400, 190], [100, 190]],
             [[100, 200], [380, 200], [380, 240], [100, 240]], [[900, 100], [940, 100], [940, 500], [900, 500]]]
    quads = [Quadrilateral(np.array(l), f"t{i}", 0.9, 10 * i, 0, 0, 255, 255, 250) for i, l in enumerate(lines)]
    for q in quads:
        q.assigned_direction = q.direction
    regions = textline_merge.dispatch(quads[::-1], 1000, 600)          # shuffled input order
    by_size = sorted(regions, key=lambda r: -len(r.lines))
    assert [len(r.lines) for r in by_size] == [3, 1]
    block = by_size[0]
    assert block.direction == "h" and block.texts == ["t0", "t1", "t2"]                      # top to bottom
    assert block.font_size == 40 and block.angle == 0.0
    assert block.fg_color == (10, 0, 0) and block.bg_color == (255, 255, 250)
    assert 0 < block.prob <= 1 and by_size[1].direction == "v"
    assert textline_merge.dispatch([], 10, 10) == []


@pytest.mark.gpu
def test_device_pair_predicate_equals_host():
    """SURVEY 8f N3 on the device: mitb_op_textline_pairs against the host `can_merge_region` (the port the known-answer tests above
    pin) for EVERY pair of lines of every reference case, under both parameter sets in use (OCR direction graph, text-line merge), and
    on rotated random quads; then the whole merge with the device predicate reproduces the host's (= the reference's) regions."""
    import itertools
    from mit_b200.engine import get_engine
    from mit_b200.host import geometry
    eng = get_engine("cuda:0")
    rng = np.random.default_rng(8)
    sets = [[Quadrilateral(np.array(l), "", 1.0) for l in c["lines"]] for c in CASES]
    rnd = []
    for t in range(80):                                       # clustered so that many pairs pass the distance gates
        cx, cy = rng.uniform(200, 500), rng.uniform(200, 500)
        ww, hh = rng.uniform(30, 200), rng.uniform(12, 40)
        if t % 3 == 0:
            ww, hh = hh, ww
        ang = rng.uniform(-0.5, 0.5) if t % 2 else 0.0
        c, s = np.cos(ang), np.sin(ang)
        pts = np.array([[-ww / 2, -hh / 2], [ww / 2, -hh / 2], [ww / 2, hh / 2], [-ww / 2, hh / 2]]) @ np.array([[c, s], [-s, c]]) + [cx, cy]
        rnd.append(Quadrilateral(pts.astype(np.int64), "", 1.0))
    sets.append(rnd)
    sets.append([Quadrilateral(np.array([[0, 0], [100, 0], [30, 10], [0, 40]]), "", 1.0), rnd[0], rnd[1]])      # a non-convex quad
    n_true = n_pairs = 0
    for quads in sets:
        for params in (dict(aspect_ratio_tol=1), dict(aspect_ratio_tol=1.3, font_size_ratio_tol=2, char_gap_tolerance=1, char_gap_tolerance2=3)):
            got = geometry.can_merge_matrix(quads, eng, **params)
            for u, v in itertools.combinations(range(len(quads)), 2):
                want = geometry.can_merge_region(quads[u], quads[v], **params)
                assert bool(got[u, v]) == bool(want) == bool(got[v, u]), (u, v, params)
                n_true += bool(want)
                n_pairs += 1
    print(f"pair predicate: {n_pairs} pairs, {n_true} mergeable, device == host")
    assert n_true > 50 and n_pairs > 3000
    for case in CASES:
        quads = [Quadrilateral(np.array(l), "", 1) for l in case["lines"]]
        regions = textline_merge.dispatch(quads, case["width"], case["height"], engine=eng)
        assert {tuple(sorted(r.line_indices)) for r in regions} == {tuple(c) for c in case["expected"]}
    assert [d for _, d in geometry.generate_text_direction(rnd, engine=eng)] == [d for _, d in geometry.generate_text_direction(rnd)]


def test_pair_matrix_glue_with_a_fake_engine():
    """Host side of the device pair predicate (no GPU): the feature records, the undecided-pair fallback (value 2 for a non-convex
    quad) and the graph built from the matrix give the same regions as the all-host path."""
    import itertools
    from mit_b200.host import geometry

    class Fake:
        def __init__(self, quads):
            self.q, self.asked = quads, 0

        def textline_pairs(self, feat, params):
            assert feat.shape == (len(self.q), 16) and feat.dtype == np.float64
            n = len(self.q)
            adj = np.zeros((n, n), np.uint8)
            for u, v in itertools.combinations(range(n), 2):
                if not (int(feat[u, 15]) & 2 and int(feat[v, 15]) & 2):
                    adj[u, v] = adj[v, u] = 2                                      # what the kernel reports for a non-convex quad
                    self.asked += 1
                else:
                    adj[u, v] = adj[v, u] = 1 if geometry.can_merge_region(self.q[u], self.q[v], *params) else 0
            return adj

    case = CASES[0]
    quads = [Quadrilateral(np.array(l), "", 1) for l in case["lines"]]
    quads.append(Quadrilateral(np.array([[0, 0], [100, 0], [30, 10], [0, 40]]), "", 1))      # non-convex: decided on the host
    fake = Fake(quads)
    f = geometry.pair_features(quads)
    assert int(f[-1, 15]) & 2 == 0 and all(int(v) & 2 for v in f[:-1, 15])
    assert np.array_equal(f[0, :8], np.asarray(quads[0].pts, float).reshape(-1)) and f[0, 12] == quads[0].font_size
    with_dev = textline_merge.dispatch(quads, case["width"], case["height"], engine=fake)
    host = textline_merge.dispatch(quads, case["width"], case["height"])
    assert [r.line_indices for r in with_dev] == [r.line_indices for r in host] and fake.asked == len(quads) - 1
    assert [d for _, d in geometry.generate_text_direction(quads, engine=fake)] == [d for _, d in geometry.generate_text_direction(quads)]


REFERENCE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_textline_merge.json")


def test_merge_predicate_equals_reference_code():
    """`host.geometry.can_merge_region` against the reference's own `quadrilateral_can_merge_region` (utils/generic.py:653-698), run
    unmodified with shapely's Polygon bound to our polygon-distance restatement (its verdicts are stored in tests/golden): every pair of
    every known-answer case and of a set of rotated random quads, under both parameter sets in use.  Pins the rule cascade and its numpy
    scalar-type semantics (the distance function itself is the restated part)."""
    import itertools
    from oracle import cases
    with open(REFERENCE) as f:
        want_sets = json.load(f)["predicate"]
    sets = [[np.array(l) for l in c["lines"]] for c in CASES] + [cases.merge_random_quads()]
    assert len(sets) == len(want_sets)
    n_true = n_pairs = 0
    for pts_list, want_per_params in zip(sets, want_sets):
        mine = [Quadrilateral(p, "", 1.0) for p in pts_list]
        for params, want in zip(cases.MERGE_PARAMS, want_per_params):
            got = "".join("1" if geometry.can_merge_region(mine[u], mine[v], **params) else "0"
                          for u, v in itertools.combinations(range(len(mine)), 2))
            assert got == want, params
            n_true += want.count("1")
            n_pairs += len(want)
    assert n_true > 50 and n_pairs > 3000


def test_regions_and_direction_graph_equal_reference_code_on_random_pages():
    """Beyond the 11 known-answer cases: the reference's own `merge_bboxes_text_region` (textline_merge/__init__.py:110-181) and
    `CommonOCR._generate_text_direction` (ocr/common.py:12-39), run unmodified with shapely bound to our geometry restatements (their
    results are stored in tests/golden), against `host.textline_merge.merge_text_regions` / `host.geometry.generate_text_direction` on
    random clustered pages of rotated lines."""
    from oracle import cases
    with open(REFERENCE) as f:
        want_pages = json.load(f)["pages"]
    n_regions = 0
    for page, ((pts_list, cols), ref) in enumerate(zip(cases.merge_random_pages(), want_pages)):
        mine = [Quadrilateral(p, f"t{i}", 0.9, *c) for i, (p, c) in enumerate(zip(pts_list, cols))]
        for q in mine:
            q.assigned_direction = q.direction
        want = [(members, tuple(fg), tuple(bg)) for members, fg, bg in ref["regions"]]
        got = [(list(members), tuple(int(v) for v in fg), tuple(int(v) for v in bg)) for members, fg, bg, _ in textline_merge.merge_text_regions(mine, 1000, 800)]
        key = lambda r: tuple(sorted(r[0]))
        assert sorted(map(key, got)) == sorted(map(key, want))                                       # same partition ...
        assert sorted(got, key=key) == sorted(want, key=key), (page, got, want)                      # ... same reading order and colours
        n_regions += len(want)
        rd = [tuple(x) for x in ref["directions"]]
        md = [(mine.index(q), d) for q, d in geometry.generate_text_direction(mine)]
        assert sorted(rd) == sorted(md)
        # the order of whole groups follows networkx's component iteration in both; within a group it must agree
        assert rd == md, (page, rd, md)
    assert len(want_pages) == 12 and n_regions > 30
