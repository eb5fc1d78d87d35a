"""Turn an ncu launch list of ONE device-resident page into the per-class DRAM traffic summary bench.py reports as
`roofline.traffic`.

  gpurun -- 'ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none \
             --profile-from-start off --csv --log-file gpurun_out/r02_page_launches.csv python tools/profile_page.py'
  python tools/ncu_traffic.py gpurun_out/r02_page_launches.csv profiles/r02_ncu_traffic.json

The JSON records the hash of the CUDA sources it was measured on; bench.py prints whether that still matches the build it times.
"""
import csv
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CLASSES = (  # first match wins; conv_tc = every kernel a dense conv op launches (operand split / halo passes included)
    ("conv_tc", ("conv_tma_kernel", "conv_tc_kernel", "split_pad_kernel", "split_stem8_kernel", "split_halo_kernel", "splitk_reduce", "conv_igemm_kernel",
                 "conv_fewout_kernel", "rowstat_final", "tile_need_kernel")),
    ("conv7_thin", ("conv7_thin_kernel",)),          # (output sparse for LaMa's final conv: see DESIGN 4.4)
    ("fft", ("rfft_rows", "irfft_rows", "fft_cols")),
    ("dwconv7_ln", ("dwconv7_ln_kernel",)),
    ("layernorm", ("layernorm_kernel",)),
    ("attention", ("attention_kernel", "attention40_kernel", "attention_stream_kernel")),
    ("ocr_crops_ctc", ("warp_lines_kernel", "ctc_collapse_kernel")),
    ("need_maps", ("need_from_mask_kernel", "need_pool2_kernel", "need_dilate1_kernel")),
    ("bilateral", ("bilateral17_kernel",)),
    ("convT4_c1", ("convT4_c1_kernel",)),
)


def source_hash():
    h = hashlib.sha256()
    d = os.path.join(ROOT, "manga-image-translator_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh", ".h")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def classify(kernel):
    for cls, pats in CLASSES:
        if any(p in kernel for p in pats):
            return cls
    return "other"


def main(src, dst):
    rows = [r for r in csv.reader(l for l in open(src, errors="replace") if l.startswith('"'))]
    hdr = rows[0]
    ik, im, iv, iu = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
    iid = hdr.index("ID")
    per = {}
    for r in rows[1:]:
        k = per.setdefault(r[iid], {"kernel": r[ik]})
        v = float(r[iv].replace(",", ""))
        u = r[iu].lower()
        if "byte" in u:
            v *= {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}[u]
        elif u in ("ns", "nsecond"):
            v *= 1e-9
        elif u in ("us", "usecond"):
            v *= 1e-6
        elif u in ("ms", "msecond"):
            v *= 1e-3
        k[r[im]] = v
    out = {}
    seq = [per[i] for i in sorted(per, key=lambda x: int(x))]
    for k in seq:
        k["class"] = classify(k["kernel"])
    # output-sparse conv ops (ConvOp::need_px): [split_pad,] tile_need_kernel, conv_tma_kernel - their own class, like in the library's
    # profile (`conv_tc_sparse`), so that `conv_tc` stays the dense class the roofline is quoted on
    for i, k in enumerate(seq):
        if "tile_need_kernel" in k["kernel"]:
            k["class"] = "conv_tc_sparse"
            if i + 1 < len(seq) and "conv_tma_kernel" in seq[i + 1]["kernel"]:
                seq[i + 1]["class"] = "conv_tc_sparse"
            if i > 0 and "split_pad_kernel" in seq[i - 1]["kernel"]:
                seq[i - 1]["class"] = "conv_tc_sparse"
    for k in seq:
        c = out.setdefault(k["class"], {"launches": 0, "time_ms": 0.0, "dram_bytes": 0.0})
        c["launches"] += 1
        c["time_ms"] += 1e3 * k.get("gpu__time_duration.sum", 0.0)
        c["dram_bytes"] += k.get("dram__bytes_read.sum", 0.0) + k.get("dram__bytes_write.sum", 0.0)
    total = sum(c["time_ms"] for c in out.values())
    for c in out.values():
        c["share_of_time"] = c["time_ms"] / total if total else 0.0
    try:
        head = subprocess.run(["git", "-C", ROOT, "rev-parse", "--short", "HEAD"], capture_output=True, text=True).stdout.strip()
    except Exception:  # noqa: BLE001
        head = ""
    doc = {"what": "ncu launch list of one device-resident 2048x1536 page (cold caches, serialised launches): DRAM bytes = dram__bytes_read.sum + "
                   "dram__bytes_write.sum per kernel, summed per class; conv_tc covers every kernel a dense conv op launches",
           "source": os.path.basename(src), "git_head": head, "csrc_sha": source_hash(), "total_time_ms": total, "classes": out,
           "conv_class_dram_bytes_per_page": out.get("conv_tc", {}).get("dram_bytes", 0.0)}
    json.dump(doc, open(dst, "w"), indent=1)
    for name, c in sorted(out.items(), key=lambda kv: -kv[1]["time_ms"]):
        print(f"{name:12s} launches {c['launches']:5d} time {c['time_ms']:8.3f} ms share {100 * c['share_of_time']:5.1f} % dram {c['dram_bytes'] / 1e9:7.3f} GB")
    print(f"total {total:.3f} ms -> {dst}")


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
