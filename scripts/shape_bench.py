"""The opt-in shape columns of measurements_results.csv: the shape kernel next to trace + K5 on the same sets, the measurement CSV with and
without the ten columns, and the host alternative (engine.unpack_masks + OpenCV per mask), with output checks in the same run.

Two workloads, the same as scripts/csv_write_bench.py (synthetic_heads -> engine.paste(frames=None) -> K5):
  micrograph : one 8192 x 8192 frame with ~20 k instances;
  batch      : 64 frames of 1024 x 1024 with ~500 instances each.
Stage times are CUDA events (engine.STAGE_TIMING) over warm repetitions, summed over the frames: trace + K5 is every stage of
engine.measure, the shape pass is shape_list's plan + scan and its kernel.  The CSV end to end is a host clock around formatting the
measurement rows of every frame, D2H included.  The host alternative unpacks a sample of instances one full-frame mask at a time and
computes the columns with oracle/shape.py (numpy + OpenCV); its time per instance is scaled to the workload.  Checks: the sample's
device values against the oracle (exact; the Feret angle within 1e-12 degrees) and the device text against csv.writer over
inference.measure_masks(shape_columns=True).  Prints one JSON line with the GPU name and power limit.

    python scripts/shape_bench.py [--reps 10] [--warmup 3] [--sample 200] [--out file.json]
"""
import argparse
import csv
import io
import json
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepemia_b200 import engine, synthetic as syn  # noqa: E402
from deepemia_b200.functions import inference as inf  # noqa: E402
from oracle import shape as oshape  # noqa: E402

CLASS_NAMES = ["pore", "throat"]
UM_PIX = 0.5


def build(dev, frames, n_per_frame, H, W, seed):
    out = []
    for f in range(frames):
        probs, boxes, _, classes = syn.synthetic_heads(seed + f, n_per_frame, H, W, rmin=4, rmax=30, margin=0)
        s = engine.paste(torch.as_tensor(probs, device=dev), torch.as_tensor(boxes, device=dev), H, W, frames=None)
        out.append((f"img{f:03d}.tif", s, [int(c) % 3 for c in classes[:s.n]]))
    return out


def timed(fn, n_frames):
    """Per stage: device time of one call of fn, summed over the frames (stage_summary averages the frames' calls)."""
    engine.STAGE_TIMING["enabled"] = True
    try:
        fn()
        return {k: v * n_frames for k, v in engine.stage_summary().items()}
    finally:
        engine.STAGE_TIMING["enabled"] = False


def csv_texts(frames, shapes):
    out = []
    for (name, s, classes), shp in zip(frames, shapes):
        fields, cidx = inf._class_table(classes, CLASS_NAMES)
        out.append(engine.measurements_csv_text(s, name, "500", cidx, fields, shape=shp))
    return out


def run(dev, wname, n_frames, n_per_frame, H, W, seed, reps, warmup, sample):
    frames = build(dev, n_frames, n_per_frame, H, W, seed)
    measure = lambda: [engine.measure(s, um_pix=UM_PIX, min_area=engine.default_min_area(H, W)) for _, s, _ in frames]  # noqa: E731
    shape = lambda: [engine.shape_descriptors(s) for _, s, _ in frames]                                                    # noqa: E731
    k5, shp_t, csv_plain, csv_shape, e2e_plain, e2e_shape = [], [], [], [], [], []
    for it in range(warmup + reps):
        a = timed(measure, n_frames)
        shapes = []
        b = timed(lambda: shapes.extend(shape()), n_frames)
        c = timed(lambda: csv_texts(frames, [None] * n_frames), n_frames)
        d = timed(lambda: csv_texts(frames, shapes), n_frames)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        plain_text = csv_texts(frames, [None] * n_frames)
        t1 = time.perf_counter()
        shape_text = csv_texts(frames, shapes)
        t2 = time.perf_counter()
        if it >= warmup:
            k5.append(a); shp_t.append(b); csv_plain.append(c); csv_shape.append(d)
            e2e_plain.append((t1 - t0) * 1e3); e2e_shape.append((t2 - t1) * 1e3)
    med = lambda runs: {k: round(float(np.median([r.get(k, 0.0) for r in runs])), 4) for k in runs[0]}           # noqa: E731
    k5_med, shape_med = med(k5), med(shp_t)
    # output checks: the device text against csv.writer over measure_masks' rows (which measure again: the records are the same)
    rows = []
    for name, s, classes in frames:
        rows += inf.measure_masks(s, classes, (H, W), UM_PIX, name, "500", class_names=CLASS_NAMES, shape_columns=True)
    buf = io.StringIO()
    csv.writer(buf).writerows(rows)
    text_equal = b"".join(shape_text) == buf.getvalue().encode("utf-8")
    plain_prefix = all(b.startswith(a + b",") for pt, st in zip(plain_text, shape_text)
                       for a, b in zip(pt.split(b"\r\n")[:-1], st.split(b"\r\n")[:-1]))
    # the host alternative on a sample of the first frame's instances, checked against the device values
    name, s, _ = frames[0]
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.choice(s.n, min(sample, s.n), replace=False))
    dev_vals = shapes[0].cpu().numpy()
    rec = s.records.cpu().numpy()
    cont_off = s.cont_off.cpu().numpy()
    gate = engine.default_min_area(H, W)
    worst_angle, exact = 0.0, True
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    host_vals = []
    for k in idx.tolist():
        m = engine.unpack_masks(s, [k])[0].cpu().numpy().astype(np.uint8)
        cs, _ = cv2.findContours(m, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
        host_vals.append([oshape.shape_descriptors(c, UM_PIX) if cv2.contourArea(c) >= gate else None for c in cs])
    host_ms = (time.perf_counter() - t0) * 1e3
    for k, hv in zip(idx.tolist(), host_vals):
        for j, v in enumerate(hv):
            r = cont_off[k] + j
            if v is None:
                exact &= bool(rec[r, engine.REC_MEASURED] != 1.0 and np.isnan(dev_vals[r]).all())
                continue
            g = dev_vals[r]
            exact &= bool(all(g[f] == v[f] for f in range(10) if f != 7))
            worst_angle = max(worst_angle, abs(g[7] - v[7]))
    n_inst = sum(s.n for _, s, _ in frames)
    return {"workload": wname, "frames": n_frames, "H": H, "W": W, "instances": n_inst, "rows": len(rows),
            "trace_k5_stage_ms": k5_med, "trace_k5_ms": round(sum(k5_med.values()), 4),
            "shape_stage_ms": shape_med, "shape_ms": round(sum(shape_med.values()), 4),
            "csv_stage_ms_plain": med(csv_plain), "csv_stage_ms_shape": med(csv_shape),
            "csv_e2e_ms_host_clock_plain": round(float(np.median(e2e_plain)), 3),
            "csv_e2e_ms_host_clock_shape": round(float(np.median(e2e_shape)), 3),
            "csv_bytes_plain": sum(len(t) for t in plain_text), "csv_bytes_shape": sum(len(t) for t in shape_text),
            "host_alternative_sample": len(idx), "host_alternative_ms_per_instance": round(host_ms / len(idx), 4),
            "host_alternative_ms_scaled": round(host_ms / len(idx) * n_inst, 1),
            "check": {"text_equal_measure_masks": text_equal, "plain_rows_are_prefixes": plain_prefix,
                      "sample_exact_vs_oracle": exact, "sample_max_angle_diff_deg": worst_angle}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sample", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("shape_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    res = [run(dev, "micrograph_8192", 1, 20000, 8192, 8192, 100, args.reps, args.warmup, args.sample),
           run(dev, "batch_64x1024", 64, 500, 1024, 1024, 1000, args.reps, args.warmup, args.sample)]
    ok = all(r["check"]["text_equal_measure_masks"] and r["check"]["plain_rows_are_prefixes"] and r["check"]["sample_exact_vs_oracle"]
             and r["check"]["sample_max_angle_diff_deg"] <= 1e-12 for r in res)
    line = json.dumps({"bench": "shape", "gpu": gpu, "reps": args.reps, "warmup": args.warmup, "results": res, "outputs_ok": ok})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
