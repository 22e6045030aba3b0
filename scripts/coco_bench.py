"""COCO instance JSON: writing the annotations on the device (engine.coco_annotations_text) and reading a file back
(load_coco_results: json.loads, one H2D copy, counts -> runs, RLE decode), per stage, against the host alternative, with the
outputs checked in the same run.

Two workloads, the same as scripts/csv_write_bench.py (synthetic_heads -> engine.paste(frames=None) -> K6):
  micrograph : one 8192 x 8192 frame with ~20 k instances;
  batch      : 64 frames of 1024 x 1024 with ~500 instances each.
Stage times are CUDA events over warm repetitions, summed over the frames.  The end to end is a host clock that ends in a
device synchronise: for the write, the device texts of every frame joined into coco_instances.json in a temporary directory;
for the read, load_coco_results of that file.  The host alternative (unpack_masks + oracle/coco.py's numpy encoder + json.dumps;
oracle rle_fr_string for the read) is timed the same way on a sample of instances, because unpacking every full-frame mask of the
micrograph takes 20 k x 64 MB: its per-instance time and the projection to the whole workload are reported as such.
Byte equality: the file against json.dumps of the oracle's entries computed from the same K6 runs; the decoded tables against
rle_decode of the runs.  Prints one JSON line with the GPU name and power limit.

    python scripts/coco_bench.py [--reps 10] [--warmup 3] [--sample 200] [--out profiles/r3_coco_bench.json]
"""
import argparse
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
from oracle import coco  # noqa: E402

CLASS_NAMES = ["pore", "throat"]


def build(dev, frames, n_per_frame, H, W, seed):
    """Per frame: (name, iset, classes, scores, run_off, runs)."""
    out = []
    for f in range(frames):
        probs, boxes, scores, classes = syn.synthetic_heads(seed + f, n_per_frame, H, W, rmin=4, rmax=30, margin=0)
        s = engine.paste(torch.as_tensor(probs, device=dev), torch.as_tensor(boxes, device=dev), H, W, frames=None)
        run_off, runs = engine.rle_encode(s)
        out.append((f"img{f:03d}.tif", s, [int(c) % 3 for c in classes[:s.n]], [np.float32(v) for v in scores[:s.n]], run_off, runs))
    return out


def write_file(frames, H, W, path):
    imgs, texts, n_ann, seen = [], [], 0, set()
    for j, (name, s, classes, scores, run_off, runs) in enumerate(frames):
        imgs.append({"id": j + 1, "file_name": name, "height": H, "width": W})
        texts.append(engine.coco_annotations_text(s, run_off, runs, j + 1, classes, scores, n_ann + 1))
        n_ann += s.n
        seen.update(classes)
    inf._write_coco(path, imgs, texts, CLASS_NAMES, seen)


def oracle_file(frames, H, W):
    """json.dumps of the oracle's entries from the K6 runs (area, tight bbox, counts_from_runs)."""
    imgs, anns = [], []
    seen = set()
    for j, (name, s, classes, scores, run_off, runs) in enumerate(frames):
        imgs.append({"id": j + 1, "file_name": name, "height": H, "width": W})
        ro, rn = run_off.cpu().numpy(), runs.cpu().numpy()
        for i in range(s.n):
            r = rn[ro[i]:ro[i + 1]]
            area = int(r[:, 1].sum()) if len(r) else 0
            bbox = [0.0, 0.0, 0.0, 0.0]
            if area:
                f0, f1 = r[:, 0] - 1, r[:, 0] + r[:, 1] - 2
                x0, x1 = f0 // H, f1 // H
                y0, y1 = np.where(x0 == x1, f0 - x0 * H, 0), np.where(x0 == x1, f1 - x1 * H, H - 1)
                bbox = [float(x0.min()), float(y0.min()), float(x1.max() - x0.min() + 1), float(y1.max() - y0.min() + 1)]
            anns.append({"id": len(anns) + 1, "image_id": j + 1, "category_id": classes[i],
                         "segmentation": {"size": [H, W], "counts": coco.rle_to_string(coco.counts_from_runs(r, H, W))},
                         "area": area, "bbox": bbox, "iscrowd": 0, "score": float(scores[i])})
            seen.add(classes[i])
    cats = [{"id": k, "name": n} for k, n in enumerate(CLASS_NAMES)] + \
        [{"id": c, "name": f"class_{c}"} for c in sorted(seen) if c >= len(CLASS_NAMES)]
    return json.dumps({"images": imgs, "annotations": anns, "categories": cats}).encode()


def host_write_sample(s, classes, scores, k):
    """The host alternative for the first k instances of a set: unpack_masks, the numpy encoder, json.dumps."""
    masks = engine.unpack_masks(s, list(range(k))).cpu().numpy()
    return json.dumps([coco.annotation(i + 1, 1, classes[i], masks[i], scores[i]) for i in range(k)])


def host_read_sample(anns):
    return [coco.runs_from_counts(coco.rle_fr_string(a["segmentation"]["counts"])) for a in anns]


def run(dev, name, n_frames, n_per_frame, H, W, seed, reps, warmup, sample):
    frames = build(dev, n_frames, n_per_frame, H, W, seed)
    images = [(f[0], np.broadcast_to(np.zeros(1, np.uint8), (H, W, 3))) for f in frames]
    stage, w_e2e, r_e2e, jl = {}, [], [], []
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "coco_instances.json")
        for it in range(warmup + reps):
            engine.STAGE_TIMING["enabled"] = it >= warmup
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            write_file(frames, H, W, path)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            sets = inf.load_coco_results(path, images)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            with open(path, "rb") as f:
                raw = f.read()
            t3 = time.perf_counter()
            d = json.loads(raw)
            t4 = time.perf_counter()
            if it >= warmup:
                w_e2e.append((t1 - t0) * 1e3)
                r_e2e.append((t2 - t1) * 1e3)
                jl.append((t4 - t3) * 1e3)
                for k, v in engine.stage_summary().items():
                    # stage_summary averages the calls: the write runs once per frame, the read once per frame size
                    stage.setdefault(k, []).append(v * n_frames if k.startswith("coco_ann") else v)
            engine.STAGE_TIMING["enabled"] = False
        nbytes = len(raw)
        same_file = raw == oracle_file(frames, H, W)
        same_sets = True
        for (fname, s, _, _, run_off, runs) in frames:
            ref = engine.rle_decode(run_off, runs, H, W)
            got = sets[fname]
            t = ref.total_crop_words
            same_sets &= got.n == ref.n and got.total_crop_words == t and all(
                torch.equal(getattr(got, f), getattr(ref, f)) for f in ("meta", "crop_off", "bbox", "area")) and \
                torch.equal(got.crops[:t], ref.crops[:t])
    # the host alternative on a sample of the first frame
    _, s0, cl0, sc0, _, _ = frames[0]
    k = min(sample, s0.n, max(1, 2 ** 30 // (H * W)))                  # at most 1 GB of unpacked masks
    hw, hr = [], []
    for it in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        host_write_sample(s0, cl0, sc0, k)
        t1 = time.perf_counter()
        host_read_sample(d["annotations"][:k])
        t2 = time.perf_counter()
        if it:
            hw.append((t1 - t0) * 1e3 / k)
            hr.append((t2 - t1) * 1e3 / k)
    n_inst = sum(f[1].n for f in frames)
    med = {key: round(float(np.median(v)), 4) for key, v in stage.items()}
    med["json_loads"] = round(float(np.median(jl)), 3)
    return {"workload": name, "frames": n_frames, "H": H, "W": W, "instances": n_inst,
            "runs": int(sum(int(f[5].shape[0]) for f in frames)), "bytes": nbytes, "stage_ms": med,
            "write_e2e_ms_host_clock": round(float(np.median(w_e2e)), 3), "load_e2e_ms_host_clock": round(float(np.median(r_e2e)), 3),
            "host_alternative": {"sample_instances": k, "write_ms_per_instance": round(float(np.median(hw)), 4),
                                 "read_ms_per_instance": round(float(np.median(hr)), 4),
                                 "write_ms_projected": round(float(np.median(hw)) * n_inst, 1),
                                 "read_ms_projected": round(float(np.median(hr)) * n_inst, 1)},
            "byte_equal_file": bool(same_file), "decode_equal_rle_decode": bool(same_sets)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sample", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("coco_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    res = [run(dev, "micrograph_8192", 1, 20000, 8192, 8192, 100, args.reps, args.warmup, args.sample),
           run(dev, "batch_64x1024", 64, 500, 1024, 1024, 1000, args.reps, args.warmup, args.sample)]
    line = json.dumps({"bench": "coco", "gpu": gpu, "reps": args.reps, "warmup": args.warmup, "results": res,
                       "exact": all(r["byte_equal_file"] and r["decode_equal_rle_decode"] for r in res)})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
