"""Reading saved results back: R50_flip_results.csv text -> runs -> instances on the device, per stage, against the host baseline.

Two workloads, built as run_inference builds its file (synthetic_heads -> engine.paste(frames=None) -> K6 -> csv.writer rows):
  micrograph : one 8192 x 8192 frame with ~20 k instances (the config-3a geometry);
  batch      : 64 frames of 1024 x 1024 with ~500 instances each.
Stage times are CUDA events over warm repetitions (the text of one workload fits the 126 MB L2, so after the first pass the
parse reads it from L2: reported as l2_resident).  The load end to end is a host clock around read + parse + decode ending in a
synchronize.  The same run checks that the decoded sets are the canonical form of the source sets and prints one JSON line.

    python scripts/rle_load_bench.py [--reps 10] [--warmup 3] [--out file.json]
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

L2_BYTES = 126 * 2 ** 20


def build(dev, frames, n_per_frame, H, W, seed):
    """(source InstanceSets, file bytes) of `frames` frames written the way run_inference writes R50_flip_results.csv."""
    sets, buf = [], io.StringIO()
    w = csv.writer(buf)
    w.writerow(["ImageId", "EncodedPixels"])
    for f in range(frames):
        probs, boxes, _, _ = syn.synthetic_heads(seed + f, n_per_frame, H, W, rmin=4, rmax=30, margin=0)
        s = engine.paste(torch.as_tensor(probs, device=dev), torch.as_tensor(boxes, device=dev), H, W, frames=None)
        ro, rn = (t.cpu().numpy() for t in engine.rle_encode(s))
        w.writerows((f"img{f:03d}", " ".join(str(int(v)) for v in rn[ro[i]:ro[i + 1]].reshape(-1))) for i in range(s.n))
        sets.append(s)
    return sets, buf.getvalue().encode()


def canonical_meta(bbox, area):
    """emia_meta_from_bbox in numpy: the tight-bbox geometry of from_masks."""
    y0, x0, y1, x1 = bbox.T
    live = area > 0
    wc0 = x0 >> 5
    m = np.stack([y0, wc0, y1 - y0 + 1, (x1 >> 5) - wc0 + 1, x0, x1 + 1, np.ones_like(y0), np.zeros_like(y0)], 1)
    m[~live, :6] = 0
    return m.astype(np.int32)


def parity(dec, src, full):
    """dec == canonical form of src: same runs when encoded again, same bbox / area, tight-bbox meta; with full, every table equal to
    from_masks(unpack_masks(src))."""
    ok = all(torch.equal(a, b) for a, b in zip(engine.rle_encode(dec), engine.rle_encode(src)))
    ok &= torch.equal(dec.bbox, src.bbox) and torch.equal(dec.area, src.area)
    ok &= np.array_equal(dec.meta.cpu().numpy(), canonical_meta(src.bbox.cpu().numpy(), src.area.cpu().numpy()))
    if full:
        ref = engine.from_masks(engine.unpack_masks(src))
        ok &= all(torch.equal(getattr(dec, f), getattr(ref, f)) for f in ("meta", "crop_off", "bbox", "area"))
        ok &= torch.equal(dec.crops[:ref.total_crop_words], ref.crops[:ref.total_crop_words])
    return bool(ok)


def host_baseline(data, H, W, sample=32):
    t0 = time.perf_counter()
    rows = list(csv.reader(io.StringIO(data.decode())))[1:]
    vals = [np.fromstring(r[1], dtype=np.int64, sep=" ") for r in rows]
    parse_ms = (time.perf_counter() - t0) * 1e3
    idx = np.linspace(0, len(vals) - 1, min(sample, len(vals))).astype(int)
    t0 = time.perf_counter()
    for i in idx:
        flat = np.zeros(H * W, np.uint8)
        for s, n in vals[i].reshape(-1, 2):
            flat[s - 1:s - 1 + n] = 1
        flat.reshape(W, H).T.copy()
    per_row_ms = (time.perf_counter() - t0) * 1e3 / len(idx)
    return {"csv_reader_numpy_parse_ms": round(parse_ms, 3), "numpy_full_frame_decode_ms_per_row": round(per_row_ms, 4),
            "numpy_full_frame_decode_sampled_rows": int(len(idx)), "numpy_full_frame_bytes_per_row": H * W}


def run(dev, name, frames, n_per_frame, H, W, seed, reps, warmup, tmp):
    sets, data = build(dev, frames, n_per_frame, H, W, seed)
    path = os.path.join(tmp, f"{name}.csv")
    with open(path, "wb") as f:
        f.write(data)
    n_inst = sum(s.n for s in sets)
    owner = np.repeat(np.arange(frames), [s.n for s in sets])
    rows_of = [np.nonzero(owner == k)[0] if frames > 1 else None for k in range(frames)]

    def load():
        with open(path, "rb") as f:
            d = f.read()
        ids, run_off, runs = engine.rle_parse_csv(d, dev)
        decs = []
        for k in range(frames):
            decs.append(engine._rle_decode(run_off, runs, H, W, rows_of[k])[0])
        torch.cuda.synchronize()
        return decs

    stage, e2e, remeasure = {}, [], []
    for it in range(warmup + reps):
        engine.STAGE_TIMING["enabled"] = it >= warmup
        t0 = time.perf_counter()
        decs = load()
        t1 = time.perf_counter()
        if it >= warmup:
            e2e.append((t1 - t0) * 1e3)
            for k, v in engine.stage_summary().items():
                stage.setdefault(k, []).append(v * (frames if k == "rle_decode" else 1))   # stage_summary averages the frames' calls
        engine.STAGE_TIMING["enabled"] = False
        run_off, runs = _cached_runs(data, dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for k in range(frames):
            engine.measure(engine._rle_decode(run_off, runs, H, W, rows_of[k])[0], um_pix=0.5)
        b.record()
        torch.cuda.synchronize()
        if it >= warmup:
            remeasure.append(a.elapsed_time(b))
    t0 = time.perf_counter()
    with open(path, "rb") as f:
        f.read()
    read_ms = (time.perf_counter() - t0) * 1e3
    med = {k: float(np.median(v)) for k, v in stage.items()}
    pd_ms = med.get("rle_parse", 0.0) + med.get("rle_decode", 0.0)
    ok = all(parity(d, s, full=(H * W * s.n <= 2 ** 31)) for d, s in zip(decs, sets))
    return {"workload": name, "frames": frames, "H": H, "W": W, "instances": n_inst, "text_bytes": len(data),
            "values": 2 * int(_cached_runs(data, dev)[1].shape[0]),
            "l2_resident": len(data) < L2_BYTES,
            "stage_ms": {"h2d_text": round(med.get("rle_h2d", 0.0), 4), "parse": round(med.get("rle_parse", 0.0), 4),
                         "decode_plan_decode": round(med.get("rle_decode", 0.0), 4),
                         "remeasure_decode_measure": round(float(np.median(remeasure)), 4)},
            "load_e2e_ms_host_clock": round(float(np.median(e2e)), 4), "file_read_ms_host": round(read_ms, 4),
            "instances_per_s_parse_decode": round(n_inst / (pd_ms * 1e-3), 1) if pd_ms else None,
            "text_GB_per_s_parse": round(len(data) / (med["rle_parse"] * 1e-3) / 1e9, 3) if med.get("rle_parse") else None,
            "host_baseline": host_baseline(data, H, W), "parity_canonical": ok}


_RUNS = {}


def _cached_runs(data, dev):
    """(run_off, runs) of a file, parsed once (the re-measure stage times decode + measure only)."""
    key = id(data)
    if key not in _RUNS:
        _RUNS[key] = engine.rle_parse_csv(data, dev)[1:]
    return _RUNS[key]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rle_load_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    with tempfile.TemporaryDirectory() as tmp:
        res = [run(dev, "micrograph_8192", 1, 20000, 8192, 8192, 100, args.reps, args.warmup, tmp),
               run(dev, "batch_64x1024", 64, 500, 1024, 1024, 1000, args.reps, args.warmup, tmp)]
    line = json.dumps({"bench": "rle_load", "gpu": gpu, "reps": args.reps, "warmup": args.warmup, "results": res,
                       "parity_canonical": all(r["parity_canonical"] for r in res)})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
