#!/usr/bin/env python
"""Headline benchmark: pages/sec for detect (DBNet-ConvNeXt) + OCR (48px CTC, 32 lines/page) + inpaint (LaMa-MPE) on
synthetic 2048x1536 RGB pages -- BASELINE.json `metric`, workload = configs[1] (32 pages per GPU; under torchrun every
rank takes 32 pages of the round-robin shard, i.e. configs[2] at 8 GPUs; weak scaling).

  python bench.py --gpus N --steps K --warmup W                      # ours (hand-written CUDA through the C ABI)
  python bench.py --impl reference --gpus N --steps K --warmup W     # CPU restatement of the reference path (oracle/)
  python bench.py ... --dump-outputs DIR                              # also write the last timed step's results as DIR/*.npy

One JSON line on stdout (rank 0).  `value` = device-resident throughput (inputs staged in HBM, CUDA-event timed, max over
ranks); `e2e` = the same pages through the plugin `infer` calls with pinned HOST buffers (H2D/D2H and host glue inside
the timed region); `roofline` = dominant kernel class from per-launch CUDA events recorded during the timed region;
`cpu_baseline` = the oracle port timed on this box's host cores on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "manga-image-translator_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

PAGE_H, PAGE_W, LINES = 2048, 1536, 32
PAGES_PER_GPU = 32
VOCAB = 46000
METRIC = "pages/sec (2048x1536, detect+OCR+inpaint)"
DUMP_PAGES = 32                                   # --dump-outputs: the first 32 pages of the step (all of them by default)
DUMP_SAMPLES = {"db": 65536, "db_mask": 32768, "inpainted": 131072}     # sampled elements per page: 28 MB at 32 pages

# The plugins get their weights in memory, but constructing one creates its model directory (default ./models).  Point it at a
# temporary directory so that the benchmark writes nothing into the tree it runs from, which may be read-only.
_MODEL_DIR = tempfile.TemporaryDirectory(prefix="mitb_models_")
os.environ.setdefault("MITB_MODEL_DIR", _MODEL_DIR.name)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def build_weights():
    from oracle import weights
    db = weights.dbnet_weights()
    db = {k: v.clone() for k, v in db.items()}
    # random weights emit per-pixel noise; bias the binarize head so that the detector's host post-processing sees a sparse
    # map (a few dozen candidates, like a real page) instead of ~10^6 one-pixel contours: measured on page 0, -8 still leaves
    # 4423 single-pixel contours above 0.5, -11 leaves 46.  Parity tests use unbiased weights; the CPU arm uses these same weights.
    db["conv_db.binarize.4.bias"] -= 11.0
    return dict(dbnet=db, ocr=weights.ocr_weights(VOCAB), dictionary=weights.synthetic_dictionary(VOCAB),
                lama=weights.lama_weights(9), mpe=weights.mpe_weights())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


CPU_THREADS_CAP = 64        # fixed policy: min(64, host cores) torch intra-op threads (128 threads were 2-3x slower on this net mix)
SAMPLE_DESC = ("one FULL 2048x1536 page per step (detect_size/inpainting_size 2048, 32 lines, V=46000): detect incl. cv2 bilateral + OCR + "
               "LaMa-MPE through the oracle port of the reference CPU path, torch CPU fp32")


def cpu_threads():
    return max(1, min(CPU_THREADS_CAP, os.cpu_count() or 1))


def cpu_reference_sample(W, index):
    """One full page of the bench workload through the CPU restatement of the reference path.  Returns seconds."""
    from mit_b200 import synth
    from oracle import pipeline_ref
    page, boxes, mask = synth.make_page(index, PAGE_H, PAGE_W, LINES)
    t0 = time.perf_counter()
    pipeline_ref.detector_infer(W["dbnet"], page, 2048, 0.5, 0.7, 2.3)
    pipeline_ref.ocr_infer(W["ocr"], W["dictionary"], page, synth.make_quads(boxes), 0.0)
    pipeline_ref.lama_infer(W["lama"], W["mpe"], page, mask, 2048)
    return time.perf_counter() - t0


def run_reference(args, rank, world):
    if rank != 0:
        return
    torch.set_grad_enabled(False)
    W = build_weights()
    threads = cpu_threads()
    torch.set_num_threads(threads)
    for i in range(min(args.warmup, 1)):             # one warm-up page (allocator, oneDNN primitive caches); more would only cost minutes
        log(f"[cpu arm] warm-up page: {cpu_reference_sample(W, i):.1f} s")
    t = [cpu_reference_sample(W, 10 + i) for i in range(args.steps)]
    total = sum(t)
    value = args.steps / total
    desc = SAMPLE_DESC + f"; {threads} torch threads (fixed policy min({CPU_THREADS_CAP}, {os.cpu_count()} host cores)), 1 warm-up page"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pages/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "2048x1536 pages, dbnet_convnext + 48px_ctc (32 lines/page, V=46000) + lama_mpe; bounded sample: " + desc,
                   "pages_per_step": 1, "weights": "seeded random (no checkpoints offline)"},
        "cpu_baseline": {"value": value, "unit": "pages/s", "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": "pages/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# GPU bar (SURVEY 8d(2)): the same functional modules (oracle/nets.py, pinned against the reference nn.Modules) moved to the
# B200 and run in eager PyTorch -> cuDNN / cuBLAS / cuFFT library kernels, N=1 per forward as the reference does
# (manga_translator.py:1491-1519), with the reference's own flags: allow_tf32 (manga_translator.py:133-138) and LaMa under
# bf16 autocast (config.py:296-299, inpainting_lama_mpe.py:100-107); and once more in plain fp32.  Device-resident inputs,
# CUDA-event timed, bilateral filter / contours / crops excluded (they are host code in the reference): this is the bar
# for our device-resident `value`.
def _bar_stage(W, dev, index):
    from mit_b200 import synth
    from oracle import nets
    page, boxes, mask = synth.make_page(index, PAGE_H, PAGE_W, LINES)
    x_det = torch.from_numpy(np.ascontiguousarray((page.astype(np.float32) / 127.5 - 1.0).transpose(2, 0, 1)[None])).to(dev)
    quads = synth.make_quads(boxes)
    regions = [q.get_transformed_region(page, q.direction, 48) for q in quads]
    perm = sorted(range(len(regions)), key=lambda i: regions[i].shape[1])
    chunks = []
    for s0 in range(0, len(perm), 16):
        ind = perm[s0:s0 + 16]
        widths = [regions[i].shape[1] for i in ind]
        canvas = np.zeros((len(ind), 48, max(widths) + 7 + 128, 3), np.uint8)
        for i, idx in enumerate(ind):
            canvas[i, :, :widths[i]] = regions[idx]
        x = (torch.from_numpy(canvas).float() - 127.5) / 127.5
        chunks.append(x.permute(0, 3, 1, 2).contiguous().to(dev))
    img = torch.from_numpy(page).permute(2, 0, 1).unsqueeze(0).float() / 255.0
    m = (torch.from_numpy(mask)[None, None].float() / 255.0 >= 0.5).float()
    rel, direct = nets.mpe_tables(m[0, 0].numpy())
    return dict(x_det=x_det, chunks=chunks, img=(img * (1 - m)).to(dev), mask=m.to(dev),
                rel=torch.from_numpy(rel)[None].to(dev), direct=torch.from_numpy(direct)[None].to(dev))


def gpu_bar(W, dev, n_pages, warm_pages=2, modes=("tf32_bf16", "fp32")):
    """pages/s of the eager-PyTorch library path on this GPU, per mode."""
    from oracle import nets
    sd_db = {k: v.to(dev) for k, v in W["dbnet"].items()}
    sd_ocr = {k: v.to(dev) for k, v in W["ocr"].items()}
    sd_lama = {k: v.to(dev) for k, v in W["lama"].items()}
    sd_mpe = {k: v.to(dev) for k, v in W["mpe"].items()}
    staged = [_bar_stage(W, dev, 100 + i) for i in range(4)]       # 4 distinct pages cycled (~0.6 GB of inputs, larger than L2)
    out = {}
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)

    def one_page(sp, autocast):
        db, mask = nets.dbnet_forward(sd_db, sp["x_det"])
        db = db.sigmoid()
        for c in sp["chunks"]:
            nets.ocr_top1(sd_ocr, c)
        if autocast:
            with torch.autocast(device_type="cuda", dtype=torch.bfloat16):
                o = nets.lama_forward(sd_lama, sd_mpe, sp["img"], sp["mask"], sp["rel"], sp["direct"])
        else:
            o = nets.lama_forward(sd_lama, sd_mpe, sp["img"], sp["mask"], sp["rel"], sp["direct"])
        return o.float()

    try:
        for mode in modes:
            tf32 = mode == "tf32_bf16"
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            for i in range(warm_pages):
                one_page(staged[i % len(staged)], tf32)
            torch.cuda.synchronize()
            ms = None
            for _ in range(2):                                 # best of two passes: the bar is the library at its best, not a cold-start artefact
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(n_pages):
                    one_page(staged[i % len(staged)], tf32)
                e1.record()
                torch.cuda.synchronize()
                t = e0.elapsed_time(e1)
                ms = t if ms is None else min(ms, t)
            out[mode] = {"pages_per_s": n_pages / (ms / 1e3), "ms_per_page": ms / n_pages, "pages_timed": n_pages, "passes": 2}
            log(f"[gpu bar] {mode}: {ms / n_pages:.1f} ms/page")
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved
    del sd_db, sd_ocr, sd_lama, sd_mpe, staged
    torch.cuda.empty_cache()
    out["what"] = ("eager PyTorch (cuDNN/cuBLAS/cuFFT) forwards of the same networks, N=1 per forward, device-resident inputs, CUDA events; "
                   "tf32_bf16 = allow_tf32 + LaMa under bf16 autocast (the reference's CUDA defaults), fp32 = allow_tf32 off, no autocast; "
                   "host stages (bilateral, contours, crops, MPE tables) excluded")
    return out


def run_reference_cuda(args, rank, world, local_rank):
    """`--impl reference-cuda`: the library-kernel bar as its own JSON line (rank 0 only; one GPU)."""
    if rank != 0:
        return
    if not torch.cuda.is_available():
        print(json.dumps({"impl": "reference-cuda", "unavailable": "no CUDA device"}), flush=True)
        return
    torch.set_grad_enabled(False)
    dev = f"cuda:{local_rank}"
    torch.cuda.set_device(dev)
    W = build_weights()
    n = max(4, args.steps * 4)
    bar = gpu_bar(W, dev, n, warm_pages=max(2, args.warmup))
    v = bar["tf32_bf16"]
    print(json.dumps({
        "impl": "reference-cuda", "metric": METRIC, "value": v["pages_per_s"], "unit": "pages/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": v["ms_per_page"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "tf32+bf16", "data": "synthetic",
        "config": {"workload": "2048x1536 pages, dbnet_convnext + 48px_ctc (32 lines/page, V=46000) + lama_mpe, device-resident forwards only",
                   "pages_per_step": 1, "weights": "seeded random (no checkpoints offline)"},
        "gpu_bar": bar,
    }), flush=True)


def csrc_hash():
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "manga-image-translator_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh", ".h")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def latest_traffic_summary():
    """Newest profiles/r*_ncu_traffic*.json written by tools/ncu_traffic.py (None when absent)."""
    import glob
    import re
    c = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_traffic*.json")),
               key=lambda p: [int(t) if t.isdigit() else t for t in re.split(r"(\d+)", os.path.basename(p))])      # natural order: v13 after v5
    if not c:
        return None, None
    sha = csrc_hash()
    docs = []
    for path in c:
        with open(path) as f:
            docs.append((json.load(f), os.path.basename(path)))
    for doc, name in reversed(docs):                      # the summary measured on exactly these CUDA sources, if there is one
        if doc.get("csrc_sha") == sha:
            return doc, name
    return docs[-1]


def roofline_from_profile(prof, peaks, pages_timed):
    """`roofline` object of the JSON line from the per-class profile {class: {launches, ms, flops, bytes}} that the library
    recorded with CUDA events around every launch of the timed region (`pages_timed` pages on this rank)."""
    if not prof:
        return None
    total_kernel_ms = sum(v["ms"] for v in prof.values())
    name, top = max(prof.items(), key=lambda kv: kv[1]["ms"])
    sec = top["ms"] / 1e3
    tensor_bound = name.startswith("conv")
    if tensor_bound:
        achieved, peak, unit = top["flops"] / sec / 1e12, peaks["tf_sust"], "TFLOP/s"
    else:
        achieved, peak, unit = top["bytes"] / sec / 1e9, peaks["hbm"], "GB/s"
    # DRAM traffic of the dominant class from the committed ncu pass (dram__bytes_read.sum + dram__bytes_write.sum summed over the
    # class's kernels of one page, cold caches), per launch like `achieved`; null if that summary is not in the tree
    traffic, traffic_src = None, None
    tj, tname = latest_traffic_summary()
    if tensor_bound and tj:
        per_page = top["launches"] / max(1, pages_timed)
        traffic = tj["conv_class_dram_bytes_per_page"] / max(1.0, per_page)
        cur = csrc_hash()
        traffic_src = (f"profiles/{tname} (tools/ncu_traffic.py over an ncu launch list of one page, cold cache, every kernel of the conv ops); "
                       f"measured on csrc {tj.get('csrc_sha', '?')} at {tj.get('git_head', '?')}, "
                       + ("same CUDA sources as this run" if tj.get("csrc_sha") == cur else f"this run's sources are {cur} (re-profile)"))
    return {"kernel": name, "bound": "tensor" if tensor_bound else "hbm", "achieved": achieved, "peak": peak, "unit": unit,
            "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes_per_launch": top["bytes"] / max(1, top["launches"]),
            "algorithmic_flops_per_launch": top["flops"] / max(1, top["launches"]),
            "scheme_ceiling_frac": 1.0 / 3.0 if tensor_bound else 1.0,
            "peak_source": peaks["src"] + (" bf16 sustained" if tensor_bound else " copy"),
            "launches": top["launches"], "avg_launch_ms": top["ms"] / max(1, top["launches"]),
            "share_of_kernel_time": top["ms"] / total_kernel_ms,
            "classes": {k: {"ms": round(v["ms"], 3), "launches": v["launches"],
                            "tflops": round(v["flops"] / max(v["ms"], 1e-9) / 1e9, 2),
                            "gbs": round(v["bytes"] / max(v["ms"], 1e-9) / 1e6, 1)} for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}}


def ffc_block_from_launches(launch_list, prof, pages_timed, peaks, H=None, W=None):
    """BASELINE.json's second figure: the fused LaMa FFC block (`FFC_BN_ACT`, SURVEY 8d) - algorithmic 2*512*h*w*4 B + 5.31 MB of
    weights and 123.3 GFLOP at h x w = 256 x 192 - against the time of every kernel of the 18 FFC layers of a page: the convs
    whose GEMM has M = h*w rows with the FFC (K, N) shapes, the spectral 1x1 conv over the half spectrum (M = h*(w/2+1)) and both
    FFT classes.  `launch_list` = [[kind, M, K, N, ms], ...] from MITB_PROFILE_LAUNCHES."""
    H = H or PAGE_H
    W = W or PAGE_W
    h, w = H // 8, W // 8
    m_sp, m_fu = h * w, h * (w // 2 + 1)
    # generic path: l2g 3x3 and the 1x1 out-conv are separate launches; fused path: one launch with K = 192 + 9*128
    ffc_shapes = {(m_sp, 9 * 512, 128), (m_sp, 9 * 128, 384), (m_sp, 384, 192), (m_fu, 384, 384), (m_sp, 192, 384), (m_sp, 192 + 9 * 128, 384)}
    conv_ms = sum(x[4] for x in launch_list if (x[1], x[2], x[3]) in ffc_shapes)
    fft_ms = sum(v["ms"] for k, v in prof.items() if k.startswith("fft_")) + prof.get("split_halo", {}).get("ms", 0.0)
    layers = float(sum(1 for x in launch_list if (x[1], x[2], x[3]) == (m_sp, 384, 192)))     # one spectral in-conv per FFC layer
    if layers < 1 or conv_ms <= 0:
        return None
    sec_per_layer = (conv_ms + fft_ms) / 1e3 / layers
    bytes_alg = 2 * 512 * h * w * 4 + 5.31e6
    flops_alg = 123.3e9 * (h * w) / (256 * 192)
    gbs, tfs = bytes_alg / sec_per_layer / 1e9, flops_alg / sec_per_layer / 1e12
    t_bytes, t_flops = bytes_alg / (peaks["hbm"] * 1e9), flops_alg / (peaks["tf_sust"] * 1e12)
    return {"unit_of_work": f"FFC_BN_ACT layer at {h}x{w} (SURVEY 8d: {bytes_alg / 1e6:.1f} MB, {flops_alg / 1e9:.1f} GFLOP algorithmic)",
            "layers_timed": layers, "layers_per_page": layers / max(1, pages_timed), "us_per_layer": sec_per_layer * 1e6,
            "achieved_hbm_gbs": gbs, "hbm_frac": gbs / peaks["hbm"], "achieved_tflops": tfs, "tensor_frac": tfs / peaks["tf_sust"],
            "binding_term": "tensor" if t_flops > t_bytes else "hbm", "t_bound_us": max(t_bytes, t_flops) * 1e6,
            "frac_of_bound": max(t_bytes, t_flops) / sec_per_layer,
            "note": "tensor term uses the plain bf16 peak; the bf16x3 operand split needs 3 MMAs per product"}


def mask_refine_figure(pages, n_pages):
    """ms per page of mit_b200.mask_refinement.dispatch (host page + raw mask in, refined host mask out; 32 text lines per page; raw
    mask = the page's dark strokes dilated 3x3, like a text-segmentation map), after one warm-up page.  For scale, the oracle
    restatement of the reference's CPU stage is timed on one page too - its DenseCRF is numpy, not pydensecrf's C++, so that number
    overstates the reference's cost and is labelled as such."""
    import asyncio
    import types
    import cv2
    from mit_b200 import mask_refinement
    from mit_b200.host import geometry
    from oracle import mask_refine_ref
    items = []
    for (page, boxes, _) in pages[:n_pages + 1]:
        raw = cv2.dilate(((page[..., 0] < 100) * 255).astype(np.uint8), np.ones((3, 3), np.uint8))
        regions = [types.SimpleNamespace(lines=[b.astype(np.float64) for b in boxes[i:i + 4]]) for i in range(0, len(boxes), 4)]
        items.append((regions, page, raw))
    asyncio.run(mask_refinement.dispatch(*items[0], "fit_text", 20, 0, False, 3))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for it in items[1:]:
        out = asyncio.run(mask_refinement.dispatch(*it, "fit_text", 20, 0, False, 3))
    torch.cuda.synchronize()
    ms = 1e3 * (time.perf_counter() - t0) / max(1, len(items) - 1)
    t0 = time.perf_counter()
    want = mask_refine_ref.dispatch(items[-1][0], items[-1][1], items[-1][2].copy(), geometry.Quadrilateral, dilation_offset=20, kernel_size=3)
    cpu_ms = 1e3 * (time.perf_counter() - t0)
    inter, union = ((out > 0) & (want > 0)).sum(), ((out > 0) | (want > 0)).sum()
    return {"ms_per_page": ms, "pages": len(items) - 1, "lines_per_page": LINES, "mask_coverage": float((out > 0).mean()),
            "iou_vs_oracle_last_page": float(inter / max(1, union)),
            "cpu_oracle_ms_per_page": cpu_ms,
            "cpu_note": "oracle/mask_refine_ref.py on the host: cv2 for resize / components / bilateral / dilation (IPP default), numpy restatement "
                        "of pydensecrf's C++ DenseCRF - slower than the real library, a scale reference only"}


def c4_figure(hp, n_pages):
    """lama_large (18 FFC blocks, no MPE) on synthetic 2560x1920 pages: the inpainter's device section (uint8 page + mask in HBM ->
    inpainted uint8 page), CUDA events, one warm-up page.  The lama_mpe weights of the main workload are unloaded first."""
    import asyncio
    from mit_b200 import synth
    from oracle import weights
    eng = hp.engine
    asyncio_run = asyncio.run
    asyncio_run(hp.inp.unload())
    eng.load_lama(weights.lama_weights(18))
    try:
        staged = []
        for i in range(n_pages + 1):
            page, _, mask = synth.make_page(100 + i, 2560, 1920, LINES)
            staged.append((torch.from_numpy(page).to(eng.device), torch.from_numpy(mask).to(eng.device)))
        eng.lama_infer_u8(staged[0][0], staged[0][1], None, None, composite=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for pg, mk in staged[1:]:
            eng.lama_infer_u8(pg, mk, None, None, composite=True)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n_pages
    finally:
        eng.unload_lama()
        asyncio_run(hp.inp.load(hp.device))
    return {"ms_per_page": ms, "pages_per_s": 1e3 / ms, "pages": n_pages, "what": "lama_large (18 blocks) at 2560x1920, device resident, "
            "uint8 in / uint8 out incl. pack, blend and composite; bottleneck 320x240x512, FFT 320x240"}


def dump_outputs(results, out_dir):
    """Writes what `HotPath.run_resident` returned for each page of one step, as float32 arrays indexed [page, ...]:
    db / db_mask / inpainted are a fixed seeded sample of elements (the same positions on every page) of the detector's
    probability map [1,2,H,W], its mask [1,1,H/2,W/2] and the inpainted uint8 page [H,W,3]; ocr_* hold every text line in
    chunk order (lines sorted by width, as run_resident feeds them) with the collapsed CTC results compacted to the front
    and zero past ocr_counts.  Total size at most ~40 MB."""
    os.makedirs(out_dir, exist_ok=True)
    results = results[:DUMP_PAGES]
    arrays = {}
    for seed, (name, pick) in enumerate((("db", lambda r: r[0]), ("db_mask", lambda r: r[1]), ("inpainted", lambda r: r[3]))):
        n = pick(results[0]).numel()
        idx = np.sort(np.random.default_rng(seed).choice(n, size=min(DUMP_SAMPLES[name], n), replace=False))
        idx = torch.from_numpy(idx).to(pick(results[0]).device)
        arrays[name] = torch.stack([pick(r).reshape(-1)[idx].float() for r in results]).cpu().numpy()
    lines = [[(c, t) for c in [[x.cpu() for x in chunk] for chunk in r[2]] for t in range(c[0].shape[0])] for r in results]   # (chunk, row) per line
    n_lines = max(len(l) for l in lines)
    T = max(c[1].shape[1] for r in results for c in r[2])
    counts = np.zeros((len(results), n_lines), np.float32)
    steps, chars, logprob = (np.zeros((len(results), n_lines, T), np.float32) for _ in range(3))
    colors = np.zeros((len(results), n_lines, T, 6), np.float32)
    for p, page_lines in enumerate(lines):
        for i, (c, t) in enumerate(page_lines):
            k = int(c[0][t])
            counts[p, i] = k
            for dst, src in ((steps, c[1]), (chars, c[2]), (logprob, c[3]), (colors, c[4])):
                dst[p, i, :k] = src[t, :k].float().numpy()
    arrays.update(ocr_counts=counts, ocr_steps=steps, ocr_chars=chars, ocr_logprob=logprob, ocr_colors=colors)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    log(f"[bench] wrote {len(arrays)} arrays ({sum(a.nbytes for a in arrays.values()) / 1e6:.1f} MB) of the last timed step to {out_dir}")


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from mit_b200 import exchange, synth
    from mit_b200.pipeline import HotPath, ResultExchange, shard_indices
    torch.set_grad_enabled(False)
    os.environ.setdefault("MITB_PROFILE_LAUNCHES", "1")    # per-launch conv list for the LaMa FFC figure
    dev = f"cuda:{local_rank}"
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    W = build_weights()
    hp = HotPath(dev, W["dbnet"], W["ocr"], W["dictionary"], W["lama"], W["mpe"])
    eng = hp.engine
    n_pages = args.pages
    idxs = shard_indices(n_pages * world, rank, world)
    t0 = time.time()
    pages = []
    for i in idxs:
        p, b, m = synth.make_page(i, PAGE_H, PAGE_W, LINES)
        # pinned host buffers: the e2e path copies from these every step
        pp = torch.empty(p.shape, dtype=torch.uint8).pin_memory(); pp.copy_(torch.from_numpy(p))
        pm = torch.empty(m.shape, dtype=torch.uint8).pin_memory(); pm.copy_(torch.from_numpy(m))
        pages.append((pp.numpy(), b, pm.numpy()))
    staged = [hp.stage(p, synth.make_quads(b), m) for p, b, m in pages]
    staged_bytes = sum(s.bytes for s in staged)
    log(f"[rank {rank}] {len(pages)} pages generated+staged in {time.time() - t0:.1f}s ({staged_bytes / 1e9:.2f} GB resident)")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # multi-GPU: fixed-size result records (boxes, scores, OCR text / colours, raw mask, inpainted page) all-gathered over NCCL
    xchg = ResultExchange(dev, len(pages), PAGE_H, PAGE_W) if world > 1 else None

    def resident_step(keep=False):
        kept = []
        for i, sp in enumerate(staged):
            db, dmask, ocr, out = hp.run_resident(sp)
            if keep:                                         # --dump-outputs: hold this step's results (fresh tensors per call)
                kept.append((db, dmask, ocr, out))
            if xchg is not None:                             # N > 1: the page goes into this rank's result record, device to device
                o, nb = xchg.lay.o["page"]
                xchg.buf[i, o:o + nb].copy_(out.reshape(-1))
        if xchg is not None:
            exchange.gather_records(xchg.buf, world)         # the one collective of the path: all ranks' records over NCCL / NVLink
        return kept

    # ---------------- device-resident throughput (`value`)
    # --dump-outputs holds the last timed step's results; the warm-up steps hold theirs too, so that the allocator has that memory
    # cached before the timed region instead of allocating it inside
    dump = args.dump_outputs is not None and rank == 0
    for _ in range(args.warmup):
        resident_step(keep=dump)
    barrier()
    eng.lib.mitb_profile_enable(eng._h, 1)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for step in range(args.steps):
        last = resident_step(keep=dump and step == args.steps - 1)
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clk = clocks.stop() if rank == 0 else None
    launches = eng.launches - launches0
    prof = json.loads(eng.lib.mitb_profile_report(eng._h).decode())
    launch_list = prof.pop("_launches", [])               # per-launch conv list (MITB_PROFILE_LAUNCHES), not a kernel class
    eng.lib.mitb_profile_enable(eng._h, 0)
    value = args.steps * n_pages * world / (ms_total / 1e3)
    # the same region once more WITHOUT the per-launch event pairs of the profiler (they cost ~2 us per launch): informational
    barrier()
    e0.record()
    resident_step()
    e1.record()
    barrier()
    value_unprofiled = n_pages * world / (max_over_ranks(e0.elapsed_time(e1)) / 1e3)
    if dump:
        dump_outputs(last, args.dump_outputs)
    del last

    # ---------------- end-to-end through the plugin API with host buffers (`e2e`)
    def e2e_step():
        items = [(p, synth.make_quads(b), m) for (p, b, m) in pages]
        if world == 1:
            return hp.process_pages(items, workers=args.workers)            # the user-facing call: host arrays in, host results out
        # N > 1: every rank keeps its inpainted pages in HBM, packs one record per page and ONE all-gather brings boxes / text /
        # masks / pages to rank 0 over NVLink; rank 0 reads them back to the host (the only D2H of page-sized results)
        outs = hp.process_pages(items, workers=args.workers, keep_on_device=True)
        xchg.pack(outs)
        got = xchg.exchange(world, rank, n_pages * world)
        if rank == 0:
            eng.d2h_bytes += xchg.gathered_bytes * world
            assert len(got) == n_pages * world
        return got

    e2e_warm = min(args.warmup, 1) if args.fast_e2e else args.warmup
    for _ in range(e2e_warm):
        e2e_step()
    barrier()
    eng.h2d_bytes = eng.d2h_bytes = 0
    if os.environ.get("MITB_E2E_TRACE"):
        from mit_b200.engine import trace_report
        trace_report()                                     # drop the warm-up's numbers
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0)))
    if os.environ.get("MITB_E2E_TRACE"):
        from mit_b200.engine import trace_report
        log(f"[e2e trace] wall {e2e_ms / 1e3:.3f} s over {args.steps} step(s) x {n_pages} pages, {args.workers} workers; seconds summed over threads:")
        for k, (sec, cnt) in trace_report().items():
            log(f"[e2e trace]   {k:24s} {sec:8.3f} s  ({cnt} calls)")
    e2e_value = args.steps * n_pages * world / (e2e_ms / 1e3)
    h2d, d2h = eng.h2d_bytes / args.steps, eng.d2h_bytes / args.steps

    # ---------------- roofline of the dominant kernel class (CUDA events recorded per launch during the timed region)
    roof = roofline_from_profile(prof, load_peaks(), args.steps * n_pages)
    try:
        lama_ffc = ffc_block_from_launches(launch_list, prof, args.steps * n_pages, load_peaks())
    except Exception as ex:                                # the second figure must never cost the headline line
        log(f"[bench] lama_ffc figure unavailable: {ex!r}")
        lama_ffc = None

    # ---------------- reference bars (rank 0, N=1 only): eager-PyTorch library kernels on this GPU, and the oracle port on the host
    bar = cpu = None
    if rank == 0 and world == 1 and not args.no_gpu_bar:
        try:
            bar = gpu_bar(W, dev, 8)
        except Exception as ex:                               # the bar must never cost the headline line
            log(f"[bench] gpu bar unavailable: {ex!r}")
            bar = {"unavailable": repr(ex)}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = cpu_threads()
        torch.set_num_threads(threads)
        cpu_reference_sample(W, 9)                           # warm-up page
        sec = cpu_reference_sample(W, 10)
        cpu = {"value": 1.0 / sec, "unit": "pages/s", "cores": threads, "kind": "port",
               "sample": SAMPLE_DESC + f"; {threads} torch threads (fixed policy min({CPU_THREADS_CAP}, {os.cpu_count()} host cores)), "
                                       "1 warm-up page, 1 timed page"}

    # ---------------- SURVEY 8f N1: mask refinement (the CPU stage between OCR and inpainting in the reference) on the device,
    # through its public call with host buffers; outside the headline regions (BASELINE's metric is detect + OCR + inpaint)
    refine = None
    if rank == 0 and world == 1 and not args.no_mask_refine:
        try:
            refine = mask_refine_figure(pages, 4)
        except Exception as ex:
            log(f"[bench] mask refinement figure unavailable: {ex!r}")
            refine = {"unavailable": repr(ex)}

    # ---------------- BASELINE configs[3] (C4): lama_large at --inpainting-size 2560 on 2560x1920 pages (FFT 320x240), one GPU's share,
    # device resident like `value`; parity at this size: tests/test_gpu_fullsize.py::test_lama_large_2560x1920
    c4 = None
    if rank == 0 and world == 1 and not args.no_c4:
        try:
            c4 = c4_figure(hp, 3)
        except Exception as ex:
            log(f"[bench] C4 figure unavailable: {ex!r}")
            c4 = {"unavailable": repr(ex)}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "pages/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{n_pages} pages 2048x1536 per GPU, dbnet_convnext + 48px_ctc ({LINES} lines/page, V={VOCAB}) + lama_mpe, "
                                   f"round-robin sharded over {world} GPU(s)", "pages_per_step": n_pages * world,
                       "value_region": "resident pages, per-launch CUDA-event profiler ON (feeds `roofline`)" + (", incl. the NCCL all-gather of the result records" if world > 1 else ""),
                       "value_without_profiler": value_unprofiled, "workers": args.workers,
                       "l2": f"inputs larger than L2 ({staged_bytes / 1e9:.1f} GB of staged pages per step)",
                       "lama_decoder": "output-sparse: decoder tiles from which no hole pixel of the final blend pred*mask+(1-mask)*img is reachable are "
                                       "skipped, bit-identical to the dense path (synthetic masks cover ~7 % of a page; MITB_DENSE_TAIL=1 = dense)",
                       "ocr_crops": "cut on the device from the resident page (mitb_op_warp_lines_u8), CTC collapse on the device",
                       "weights": "seeded random (no checkpoints offline); detector binarize bias -11 so the random-weight probability map is sparse "
                                  "(~50 candidate contours per page, like a real page, instead of ~10^6 noise pixels)"},
            "e2e": {"value": e2e_value, "unit": "pages/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "lama_ffc": lama_ffc, "cpu_baseline": cpu, "gpu_bar": bar,
            "mask_refinement": refine, "c4_lama_large_2560": c4,
        }), flush=True)
    hp.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3, help="timed steps (each runs every page once)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--pages", type=int, default=PAGES_PER_GPU, help="pages per GPU per step (BASELINE configs[1]: 32)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-bar", action="store_true")
    ap.add_argument("--no-mask-refine", action="store_true", help="skip the mask-refinement (SURVEY 8f N1) figure")
    ap.add_argument("--no-c4", action="store_true", help="skip the lama_large @ 2560 (BASELINE configs[3]) figure")
    ap.add_argument("--workers", type=int, default=8, help="host threads of the page pipeline in the e2e leg")
    ap.add_argument("--fast-e2e", action="store_true", help="one warm-up step for the e2e leg (development only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                                                          "(float32; inputs are seeded, so runs with the same arguments compare output for output)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.pages < 1:
        ap.error("--steps and --pages must be >= 1, --warmup >= 0")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.impl == "reference-cuda":
        run_reference_cuda(args, rank, world, local_rank)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
