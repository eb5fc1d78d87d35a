"""OCR at every line length the reference reads.  Its PositionalEncoding has 2048 rows (model_48px_ctc.py:229), so a chunk of width
wp has T = (wp // 2) // 2 - 1 <= 2048 timesteps: lines up to 8064 px after the resize to 48 px, an aspect ratio of about 168:1.
Attention takes three routes by T (hd = 40): up to 416 the whole K / V sits in shared memory for the hd-40 kernel, up to 565 for the
generic one, beyond that K / V stream through shared memory in chunks under an online softmax.  Each route is compared with a float64
reference, the network with the CPU oracle and with what the reference computed (tests/golden/ref_ocr_long.npz), and the device line
crops, the CTC collapse and the OCR plugin at the same lengths."""
import asyncio
import time

import numpy as np
import pytest
import torch

from oracle import cases, nets, pipeline_ref, weights

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
TOL = 1e-3
ATT_TOL = 2e-5


@pytest.fixture(scope="module")
def eng():
    from mit_b200.engine import get_engine
    return get_engine("cuda:0")


def _timesteps(wp):
    return (wp // 2) // 2 - 1


# ------------------------------------------------------------------------------------------------ attention op
def _attention_ref(qk, v, n, t, heads, hd):
    """softmax(q k^T / sqrt(hd)) v in float64 on the host, per (line, head)."""
    d = heads * hd
    out = torch.empty(n * t, d, dtype=torch.float64)
    for b in range(n):                                      # one line at a time: [heads, t, t] float64 is 268 MB at t = 2048
        rows = slice(b * t, (b + 1) * t)
        q, k, vv = (a.double().reshape(t, heads, hd).transpose(0, 1) for a in (qk[rows, :d], qk[rows, d:], v[rows]))
        out[rows] = (torch.softmax(q @ k.transpose(-1, -2) / hd ** 0.5, -1) @ vv).transpose(0, 1).reshape(t, d)
    return out


def _attention_inputs(regime, n, t, heads, hd, seed):
    g = torch.Generator().manual_seed(seed)
    d = heads * hd
    v = torch.randn(n * t, d, generator=g)
    if regime == "random":
        qk = torch.randn(n * t, 2 * d, generator=g)
    elif regime == "peaked":
        # small integers: every q.k is exact in fp32, so the scores differ from the reference only by the 1/sqrt(hd) rounding; q is
        # scaled so that |score| reaches ~100: exp(100) overflows fp32 without the max subtraction, exp(-100) underflows to 0
        qk = torch.randint(-3, 4, (n * t, 2 * d), generator=g).float()
        smax = 0.0
        for b in range(n):
            q, k = (a.double().reshape(t, heads, hd).transpose(0, 1) for a in (qk[b * t:(b + 1) * t, :d], qk[b * t:(b + 1) * t, d:]))
            smax = max(smax, (q @ k.transpose(-1, -2)).abs().max().item() / hd ** 0.5)
        qk[:, :d] *= float(np.floor(100.0 / smax)) if smax >= 1.0 else 1.0
    elif regime == "same_keys":
        # every key of a (line, head) identical: all scores of a row are equal and the output is the mean of V
        qk = torch.randn(n * t, 2 * d, generator=g)
        k = torch.randn(n, 1, d, generator=g).expand(n, t, d).reshape(n * t, d)
        qk[:, d:] = k
    else:
        raise ValueError(regime)
    return qk, v


def _offset_copy(x, dev):
    """A contiguous device copy of x whose data starts 4 bytes into its storage: not 16-byte aligned, so the hd-40 kernel (float4 loads)
    is not eligible and the generic route runs."""
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=dev)
    y = buf[1:].view(x.shape)
    y.copy_(x)
    assert y.is_contiguous() and y.data_ptr() % 16 != 0
    return y


ATT_T = [1, 2, 31, 32, 33, 57, 160, 416, 417, 565, 566, 1000, 2047, 2048]
ATT_CASES = [(n, t) for t in ATT_T for n in (1, 3)] + [(16, 160), (16, 2048)]


def _check_attention(eng, n, t, heads, hd, routes, seed):
    for regime in ("random", "peaked", "same_keys"):
        qk, v = _attention_inputs(regime, n, t, heads, hd, seed)
        ref = _attention_ref(qk, v, n, t, heads, hd)
        if regime == "same_keys":
            mean = v.double().reshape(n, t, heads * hd).mean(1, keepdim=True).expand(n, t, heads * hd).reshape(n * t, -1)
            assert (ref - mean).abs().max().item() < 1e-12
        scale = max(1.0, ref.abs().max().item())
        for route in routes:
            if route == "aligned":
                qd, vd = qk.to(eng.device), v.to(eng.device)
                assert qd.data_ptr() % 16 == 0 and vd.data_ptr() % 16 == 0
            else:
                qd, vd = _offset_copy(qk, eng.device), _offset_copy(v, eng.device)
            out = eng.attention(qd, vd, n, t, heads, hd).cpu().double()
            err = (out - ref).abs().max().item()
            print(f"attention n={n} T={t} hd={hd} {regime} {route}: max abs err {err:.2e} (scale {scale:.2f})")
            assert torch.isfinite(out).all(), (regime, route)
            assert err <= ATT_TOL * scale, f"{regime} {route}: err {err:.3e} > {ATT_TOL * scale:.3e}"


@pytest.mark.parametrize("n,t", ATT_CASES)
def test_attention_hd40_lengths(eng, n, t):
    """The OCR's attention (8 heads x 40) at every route boundary (416 | 417 for the hd-40 kernel, 565 | 566 for the generic one), at T
    below and across a warp's 32 keys, and at the longest sequence the OCR accepts, on 16-byte aligned and on offset inputs."""
    _check_attention(eng, n, t, 8, 40, ("aligned", "offset"), seed=n * 10007 + t)


@pytest.mark.parametrize("hd", [32, 64])
@pytest.mark.parametrize("t", [1, 33, 417, 566, 1000, 2048])
def test_attention_other_head_dims(eng, hd, t):
    _check_attention(eng, 3, t, 8, hd, ("aligned",), seed=hd * 100003 + t)


def test_attention_head_dim_limit(eng):
    """head_dim > 64: only sequences whose K / V fit in shared memory whole (include/mitb.h); longer ones are refused, not miscomputed."""
    from mit_b200 import MitbError
    _check_attention(eng, 2, 97, 4, 96, ("aligned",), seed=96)
    qk, v = _attention_inputs("random", 1, 2048, 4, 96, 0)
    with pytest.raises(MitbError, match="head_dim <= 64"):
        eng.attention(qk, v, 1, 2048, 4, 96)
    _check_attention(eng, 1, 2048, 8, 40, ("aligned",), seed=1)          # the engine keeps working


# ------------------------------------------------------------------------------------------------ the network
@pytest.fixture
def ocr_small(eng):
    sd = weights.ocr_weights(cases.OCR_VOCAB_SMALL)
    eng.load_ocr(sd, nets.sinusoid_pe(2048))
    yield sd
    eng.unload_ocr()


def _compare_with_oracle(idx, lp, col, logits, o_col, what):
    idx, lp, col = idx.cpu().numpy(), lp.cpu().numpy(), col.cpu().numpy()
    o_lp, o_idx = logits.log_softmax(2).max(2)
    top2 = logits.topk(2, dim=-1).values
    safe = ((top2[..., 0] - top2[..., 1]) > 1e-3).numpy()
    unsafe = int((~safe).sum())
    mism = int((idx != o_idx.numpy()).sum())
    e_lp = float(np.abs(lp - o_lp.numpy())[safe].max())
    e_col = float(np.abs(col - o_col.clamp(0, 1).numpy()).max())
    print(f"{what}: T={idx.shape[1]} logprob err {e_lp:.2e} colour err {e_col:.2e} unsafe steps {unsafe} of {safe.size}, argmax differs at {mism}")
    assert np.array_equal(idx[safe], o_idx.numpy()[safe]), what
    assert unsafe <= safe.size // 50 and mism <= unsafe, (what, unsafe, mism)
    assert e_lp < TOL and e_col < TOL, what


@pytest.mark.parametrize("wp", [1600, 1700, 2439, 8196])
def test_ocr_long_chunk_vs_oracle(eng, ocr_small, wp):
    """Two lines of different widths: T = 399 (hd-40 kernel), 424 (generic kernel), 608 and 2048 (streamed K / V)."""
    _, x = cases.ocr_case(2, wp, seed=wp)
    idx, lp, col = eng.ocr_forward(x)
    assert idx.shape == (2, _timesteps(wp))
    logits, o_col = nets.ocr_forward(ocr_small, x)
    _compare_with_oracle(idx, lp, col, logits, o_col, f"ocr 2x48x{wp}")


def test_ocr_full_chunk_longest_lines(eng, ocr_small):
    """The worst chunk the OCR takes: 16 lines at T = 2048.  Its time is printed for information."""
    _, x = cases.ocr_case(16, 8196, seed=16)
    eng.ocr_forward(x)                                      # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    idx, lp, col = eng.ocr_forward(x)
    torch.cuda.synchronize()
    print(f"ocr 16x48x8196 chunk: {1e3 * (time.perf_counter() - t0):.1f} ms on {torch.cuda.get_device_name()}")
    logits, o_col = nets.ocr_forward(ocr_small, x)
    _compare_with_oracle(idx, lp, col, logits, o_col, "ocr 16x48x8196")


def test_ocr_too_long_raises_and_engine_recovers(eng, ocr_small):
    from mit_b200 import MitbError
    _, x = cases.ocr_case(2, 8200, seed=8200)
    with pytest.raises(MitbError, match="2049 timesteps"):
        eng.ocr_forward(x)
    _, x = cases.ocr_case(2, 8196, seed=8196)
    idx, lp, col = eng.ocr_forward(x)
    logits, o_col = nets.ocr_forward(ocr_small, x)
    _compare_with_oracle(idx, lp, col, logits, o_col, "ocr 2x48x8196 after the refused call")


def test_ocr_long_vs_reference_fixture(eng, golden_dir):
    """The engine against what the reference's own OCR computed at T = 608 and 2048 (oracle/make_reference_golden.py ocr_long)."""
    import os
    from oracle.make_reference_golden import OCR_LONG_WIDTHS
    g = np.load(os.path.join(golden_dir, "ref_ocr_long.npz"))
    eng.load_ocr(weights.ocr_weights(300, seed=3), nets.sinusoid_pe(2048))
    try:
        for wp in OCR_LONG_WIDTHS:
            _, x = cases.ocr_case(2, wp, seed=wp)
            idx, lp, col = [a.cpu().numpy() for a in eng.ocr_forward(x)]
            safe = g[f"margin_{wp}"] > 1e-3
            assert safe.mean() > 0.99
            assert np.array_equal(idx[safe], g[f"argmax_{wp}"][safe])
            e_lp = float(np.abs(lp - g[f"logprob_{wp}"])[safe].max())
            e_col = float(np.abs(col - g[f"colors_{wp}"]).max())
            print(f"ocr 2x48x{wp} vs reference: logprob err {e_lp:.2e} colour err {e_col:.2e}")
            assert e_lp < TOL and e_col < TOL
            mixed = np.where(safe, idx, g[f"argmax_{wp}"])             # the reference's choice on its few near-ties
            dec = nets.ctc_greedy(mixed, lp, col)
            assert [[int(c) for c in row if c >= 0] for row in g[f"decoded_{wp}"]] == [[c[0] for c in l] for l in dec]
    finally:
        eng.unload_ocr()


# ------------------------------------------------------------------------------------------------ CTC collapse, line crops
def test_ctc_collapse_longest_line(eng):
    from mit_b200.plugins import ctc_collapse
    rng = np.random.default_rng(2048)
    n, T = 8, 2048
    idx = rng.integers(0, 4, (n, T)).astype(np.int32)
    idx[0] = 0                                              # all blank
    idx[1] = 7                                              # one run over the whole line: one character
    idx[2] = 0
    for a, b in ((20, 80), (95, 96), (127, 129), (500, 1000), (2016, 2048)):   # runs across the 32-step ballot groups, up to the end
        idx[2, a:b] = 5
    idx[3] = np.where(np.arange(T) % 32 == 31, 0, 9)       # a blank closing every group: 64 kept steps, one per group
    idx[4] = np.arange(T) % 2 + 1                           # alternating symbols: every step kept
    idx[5, :] = 3
    idx[5, 31::32] = 4                                      # the last step of each group differs from its neighbours
    lp = rng.standard_normal((n, T)).astype(np.float32)
    col = rng.random((n, T, 6)).astype(np.float32)
    dev = eng.device
    counts, steps, chars, klp, kcol = [t.cpu().numpy() for t in eng.ctc_collapse(torch.from_numpy(idx).to(dev), torch.from_numpy(lp).to(dev),
                                                                                torch.from_numpy(col).to(dev))]
    host = ctc_collapse(idx)
    assert [len(s) for s in host[:5]] == [0, 1, 5, 64, T]
    for i, st in enumerate(host):
        st = np.asarray(st, dtype=np.int64)
        assert counts[i] == len(st), i
        assert np.array_equal(steps[i, :len(st)], st) and np.array_equal(chars[i, :len(st)], idx[i, st])
        assert np.array_equal(klp[i, :len(st)], lp[i, st]) and np.array_equal(kcol[i, :len(st)], col[i, st])


def test_warp_lines_long_thin_quads(eng):
    """Device crops of a long thin slanted horizontal line and a long thin vertical column into a canvas wider than 4096: bit-exact with
    cv2.warpPerspective (+ rotate) as Quadrilateral.get_transformed_region calls it."""
    from mit_b200.host import geometry
    rng = np.random.default_rng(11)
    H, W = 2048, 1536
    page = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    page_dev = torch.from_numpy(page).to(eng.device)
    lines = [(np.array([[12, 300], [1520, 331], [1520, 347], [12, 316]]), "h"),        # 1508 x 16, slanted
             (np.array([[700, 100], [719, 100], [722, 1900], [703, 1900]]), "v")]       # 20 x 1800
    recs, regions = [], []
    for pts, d in lines:
        q = geometry.Quadrilateral(pts, "", 1.0)
        rec, cw = geometry.warp_record(q, H, W, d, 48)
        reg = q.get_transformed_region(page, d, 48)
        assert rec[11] and rec[12] and reg.shape == (48, cw, 3) and cw > 4096 - 135, (d, reg.shape, cw)
        recs.append(rec)
        regions.append(reg)
    wp = max(r.shape[1] for r in regions) + 135
    assert wp > 4096
    canvas = eng.warp_lines(page_dev, np.stack(recs), wp).cpu().numpy()
    for k, reg in enumerate(regions):
        assert np.array_equal(canvas[k, :, :reg.shape[1]], reg), f"line {k}: {(canvas[k, :, :reg.shape[1]] != reg).sum()} bytes differ"
        assert not canvas[k, :, reg.shape[1]:].any()


# ------------------------------------------------------------------------------------------------ the plugin
PLUGIN_V, PLUGIN_SEED = 512, 2           # a seed whose oracle has no near-tie (top-2 margin <= 1e-3) anywhere in the chunk


def _long_line_page():
    """A 2048 x 1536 page with four ordinary short lines, a caption across the full width 32 px tall and a 24 px wide, 1200 px tall
    column: each about 2400 px long after the resize to 48 px (T > 600 alone).  All six fit in one chunk."""
    from mit_b200 import synth
    page, boxes, _ = synth.make_page(21, 2048, 1536, 4)
    rng = np.random.default_rng(21)
    page = page.copy()
    cap = np.array([[0, 1990], [1535, 1990], [1535, 2021], [0, 2021]])
    col = np.array([[1500, 40], [1523, 40], [1523, 1239], [1500, 1239]])
    for (x0, y0), (x1, y1), horizontal in ((cap[0], cap[2], True), (col[0], col[2], False)):
        page[y0:y1 + 1, x0:x1 + 1] = 235
        step = 24 if horizontal else 20
        for c in range((x1 - x0 if horizontal else y1 - y0) // step):
            for _ in range(4):
                sx = x0 + (c * step if horizontal else 0) + int(rng.integers(2, step - 4 if horizontal else x1 - x0 - 4))
                sy = y0 + (0 if horizontal else c * step) + int(rng.integers(2, y1 - y0 - 4 if horizontal else step - 4))
                page[sy:sy + int(rng.integers(2, 6)), sx:sx + int(rng.integers(1, 4))] = int(rng.integers(0, 60))
    return page, list(boxes) + [cap, col]


def _oracle_chunk_margins(sd, page, quads):
    """Top-2 margins of the oracle per line of the (single) chunk, in the reference's crop and canvas layout."""
    dirs = list(pipeline_ref.generate_text_direction(quads))
    regions = [q.get_transformed_region(page, d, 48) for q, d in dirs]
    wp = (4 * (max(r.shape[1] for r in regions) + 7) // 4) + 128
    canvas = np.zeros((len(regions), 48, wp, 3), np.uint8)
    for i, r in enumerate(regions):
        canvas[i, :, :r.shape[1]] = r
    x = ((torch.from_numpy(canvas).float() - 127.5) / 127.5).permute(0, 3, 1, 2).contiguous()
    logits, _ = nets.ocr_forward(sd, x)
    top2 = logits.topk(2, dim=-1).values
    return [r.shape[1] for r in regions], wp, (top2[..., 0] - top2[..., 1]).numpy()


@pytest.mark.parametrize("host_crops", ["0", "1"])
def test_ocr_plugin_long_lines(monkeypatch, host_crops):
    from mit_b200 import plugins, synth
    from mit_b200.compat import OcrConfig
    monkeypatch.setenv("MITB_HOST_CROPS", host_crops)
    sd, dictionary = weights.ocr_weights(PLUGIN_V, seed=PLUGIN_SEED), weights.synthetic_dictionary(PLUGIN_V)
    page, boxes = _long_line_page()
    widths, wp, margins = _oracle_chunk_margins(sd, page, synth.make_quads(boxes))
    assert len(widths) <= 16 and _timesteps(wp) >= 566, (widths, wp)
    long_lines = [i for i, w in enumerate(widths) if _timesteps(w + 135) >= 566]
    assert len(long_lines) == 2
    # the strings below are compared exactly: no step of the long lines may be a near-tie in the oracle (else this seed is unfit)
    assert all(margins[i].min() > 1e-3 for i in long_lines), [float(margins[i].min()) for i in long_lines]
    plugins.Model48pxCTCOCR.set_state_dict(sd)
    plugins.Model48pxCTCOCR.set_dictionary(dictionary)
    ocr = plugins.Model48pxCTCOCR()
    try:
        asyncio.run(ocr.load("cuda:0"))
        mine = asyncio.run(ocr.infer(page, synth.make_quads(boxes), OcrConfig(prob=0.0)))
        ref = pipeline_ref.ocr_infer(sd, dictionary, page, synth.make_quads(boxes), 0.0)
        assert len(mine) == len(ref) == len(boxes)
        for a, b in zip(mine, ref):
            assert np.array_equal(a.pts, b.pts)
            assert a.text == b.text, (a.text, b.text)
            assert abs(a.prob - b.prob) < 1e-3
            # colours: the mean of int(c * 255) over hundreds of steps; a truncation flipped by a 1e-6 difference may move it by one
            fa, fb = (a.fg_r, a.fg_g, a.fg_b, a.bg_r, a.bg_g, a.bg_b), (b.fg_r, b.fg_g, b.fg_b, b.bg_r, b.bg_g, b.bg_b)
            assert max(abs(u - w) for u, w in zip(fa, fb)) <= 1, (fa, fb)
        asyncio.run(ocr.unload())
    finally:
        plugins.Model48pxCTCOCR.set_state_dict(None)
        plugins.Model48pxCTCOCR.set_dictionary(None)
