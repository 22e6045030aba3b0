"""Writing the result files: R50_flip_results.csv and measurements_results.csv formatted on the device, per stage, against the host
path (" ".join of the runs + csv.writer, and measure_masks rows + csv.writer), with a byte-equality check in the same run.

Two workloads, the same as scripts/rle_load_bench.py (synthetic_heads -> engine.paste(frames=None) -> K6 and K5):
  micrograph : one 8192 x 8192 frame with ~20 k instances (the config-3a geometry);
  batch      : 64 frames of 1024 x 1024 with ~500 instances each.
Stage times (count, scan, write, D2H of each file) are CUDA events over warm repetitions, summed over the frames.  The end to
end is a host clock around formatting both files of every frame and writing them to a temporary directory; the host path is
timed the same way from the same K6 runs and K5 records.  Prints one JSON line with the GPU name and power limit.

    python scripts/csv_write_bench.py [--reps 10] [--warmup 3] [--out file.json]
"""
import argparse
import csv
import io
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepemia_b200 import engine, synthetic as syn  # noqa: E402
from deepemia_b200.functions import inference as inf  # noqa: E402

CLASS_NAMES = ["pore", "throat"]


def build(dev, frames, n_per_frame, H, W, seed):
    """Per frame: (name, iset measured at um_pix 0.5, classes, run_off, runs)."""
    out = []
    for f in range(frames):
        probs, boxes, _, classes = syn.synthetic_heads(seed + f, n_per_frame, H, W, rmin=4, rmax=30, margin=0)
        s = engine.paste(torch.as_tensor(probs, device=dev), torch.as_tensor(boxes, device=dev), H, W, frames=None)
        engine.measure(s, um_pix=0.5, min_area=engine.default_min_area(H, W))
        run_off, runs = engine.rle_encode(s)
        out.append((f"img{f:03d}.tif", s, [int(c) % 3 for c in classes[:s.n]], run_off, runs))
    return out


def device_files(frames, H, W, tmp):
    rle, meas = [], []
    for name, s, classes, run_off, runs in frames:
        rle.append(engine.rle_csv_text(run_off, runs, name.rsplit(".", 1)[0]))
        fields, cidx = inf._class_table(classes, CLASS_NAMES)
        meas.append(engine.measurements_csv_text(s, name, "500", cidx, fields))
    inf._write_csv(os.path.join(tmp, "R50_flip_results.csv"), ["ImageId", "EncodedPixels"], rle)
    inf._write_csv(os.path.join(tmp, "measurements_results.csv"), inf.CSV_HEADER, meas)


def host_files(frames, H, W, tmp):
    """The host path: K6 runs and K5 records copied back, then Python formatting (the same calls as before the device path)."""
    ids, enc, rows = [], [], []
    for name, s, classes, run_off, runs in frames:
        ro, rn = run_off.cpu().numpy(), runs.cpu().numpy()
        for i in range(s.n):
            ids.append(name.rsplit(".", 1)[0])
            enc.append(" ".join(str(int(v)) for v in rn[ro[i]:ro[i + 1]].reshape(-1)))
        rows += _rows(s, classes, name)
    with open(os.path.join(tmp, "R50_flip_results.csv"), "w", newline="") as f:
        w = csv.writer(f)
        w.writerow(["ImageId", "EncodedPixels"])
        w.writerows(zip(ids, enc))
    with open(os.path.join(tmp, "measurements_results.csv"), "w", newline="") as f:
        w = csv.writer(f)
        w.writerow(inf.CSV_HEADER)
        w.writerows(rows)


def _rows(s, classes, name):
    """measure_masks' loop over already-measured records (its own measure pass is K5, outside the timed formatting)."""
    rec = s.records.cpu().numpy()
    cont_off = s.cont_off.cpu().numpy()
    rows = []
    for k, cls in enumerate(classes):
        cname = CLASS_NAMES[cls] if cls < len(CLASS_NAMES) else f"class_{cls}"
        for j in range(cont_off[k], cont_off[k + 1]):
            if rec[j, engine.REC_MEASURED] != 1.0:
                continue
            m = inf.record_to_dict(rec[j])
            rows.append([f"{name}_{k + 1}", cls, cname] + [m[key] for key in inf.KEY_ORDER] + ["500", name])
    return rows


def run(dev, name, n_frames, n_per_frame, H, W, seed, reps, warmup):
    frames = build(dev, n_frames, n_per_frame, H, W, seed)
    # byte equality against measure_masks itself (it measures again; the records are the same)
    ref_rows = []
    for fname, s, classes, _, _ in frames:
        ref_rows += inf.measure_masks(s, classes, (H, W), 0.5, fname, "500", class_names=CLASS_NAMES)
    stage, dev_e2e, host_e2e = {}, [], []
    with tempfile.TemporaryDirectory() as td:
        dd, hd = os.path.join(td, "device"), os.path.join(td, "host")
        os.makedirs(dd)
        os.makedirs(hd)
        for it in range(warmup + reps):
            engine.STAGE_TIMING["enabled"] = it >= warmup
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            device_files(frames, H, W, dd)
            t1 = time.perf_counter()
            if it >= warmup:
                dev_e2e.append((t1 - t0) * 1e3)
                for k, v in engine.stage_summary().items():
                    stage.setdefault(k, []).append(v * n_frames)       # stage_summary averages the frames' calls
            engine.STAGE_TIMING["enabled"] = False
        for it in range(1 + min(reps, 3)):                              # the host path is slow: fewer repetitions
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            host_files(frames, H, W, hd)
            if it:
                host_e2e.append((time.perf_counter() - t0) * 1e3)
        same = {}
        for f in ("R50_flip_results.csv", "measurements_results.csv"):
            with open(os.path.join(dd, f), "rb") as a, open(os.path.join(hd, f), "rb") as b:
                same[f] = a.read() == b.read()
        buf = io.StringIO()
        w = csv.writer(buf)
        w.writerow(inf.CSV_HEADER)
        w.writerows(ref_rows)
        with open(os.path.join(dd, "measurements_results.csv"), "rb") as a:
            same["measurements_vs_measure_masks"] = a.read() == buf.getvalue().encode()
        sizes = {f: os.path.getsize(os.path.join(dd, f)) for f in ("R50_flip_results.csv", "measurements_results.csv")}
    med = {k: round(float(np.median(v)), 4) for k, v in stage.items()}
    n_inst = sum(s.n for _, s, _, _, _ in frames)
    return {"workload": name, "frames": n_frames, "H": H, "W": W, "instances": n_inst,
            "rows": len(ref_rows), "runs": int(sum(int(r.shape[0]) for *_, r in frames)), "bytes": sizes,
            "stage_ms": med, "device_e2e_ms_host_clock": round(float(np.median(dev_e2e)), 3),
            "host_path_e2e_ms_host_clock": round(float(np.median(host_e2e)), 3),
            "speedup_e2e": round(float(np.median(host_e2e)) / float(np.median(dev_e2e)), 1),
            "byte_equal": same, "byte_equal_all": all(same.values())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("csv_write_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    res = [run(dev, "micrograph_8192", 1, 20000, 8192, 8192, 100, args.reps, args.warmup),
           run(dev, "batch_64x1024", 64, 500, 1024, 1024, 1000, args.reps, args.warmup)]
    line = json.dumps({"bench": "csv_write", "gpu": gpu, "reps": args.reps, "warmup": args.warmup, "results": res,
                       "byte_equal": all(r["byte_equal_all"] for r in res)})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
