"""COCO segm evaluation on the device (functions.inference.evaluate_coco -> engine.coco_evaluate) per stage and end to end,
against the numpy restatement of pycocotools' COCOeval (oracle/cocoeval.py) on the same inputs, with the outputs checked in the
same run.  pycocotools itself is not installed; its own time is not measured.

Two workloads, as scripts/coco_bench.py (oracle.cocoeval.synthetic_case: star-polygon GT and perturbed predictions, one category):
  micrograph : one 8192 x 8192 frame, ~20 k GT against ~20 k detections;
  batch      : 64 frames of 1024 x 1024, ~500 GT and ~500 detections each;
each at max_dets (1, 10, 100) (pycocotools' default) and (100, 1000, 30000).  Stage times are CUDA events over warm repetitions
(order, pairs, match, accumulate; "pairs" holds the two host synchronisations that size the cell and pair lists).  The
order stage (the device radix sorts) is also timed alone on 32 k, 320 k and 3.2 M detections (500 per image, one category, scores
on a grid of 1000 values) to show how it grows with the dataset, its output checked against numpy's stable sorts.  The end to end
is a host clock around evaluate_coco that ends in a device synchronise (it includes reading both files); the file load
(json.loads + the device decode of both files) is also timed on its own.  Prints one JSON line with the GPU name and power limit.

    python scripts/cocoeval_bench.py [--reps 5] [--warmup 2] [--out profiles/r3_cocoeval_bench.json]
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
from deepemia_b200 import engine  # noqa: E402
from deepemia_b200.functions import inference as inf  # noqa: E402
from oracle import cocoeval as ce  # noqa: E402

STAGES = ["cocoeval_order", "cocoeval_pairs", "cocoeval_match", "cocoeval_accumulate"]


def run(name, frames, n, seed, reps, warmup, tmp):
    gt, dt = ce.synthetic_case(seed, frames, n, n_cats=1, rmin=4, rmax=30, crowd_frac=0.01)
    gp, dp = os.path.join(tmp, f"{name}_gt.json"), os.path.join(tmp, f"{name}_dt.json")
    with open(gp, "w") as f:
        json.dump(gt, f)
    with open(dp, "w") as f:
        json.dump(dt, f)
    out = []
    for md in [(1, 10, 100), (100, 1000, 30000)]:
        for _ in range(warmup):
            inf.evaluate_coco(gp, dp, max_dets=md)
        torch.cuda.synchronize()
        e2e, load = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            got = inf.evaluate_coco(gp, dp, max_dets=md)
            torch.cuda.synchronize()
            e2e.append((time.perf_counter() - t0) * 1e3)
        for _ in range(reps):
            t0 = time.perf_counter()
            for p in (gp, dp):
                with open(p, "rb") as f:
                    d = json.loads(f.read())
                names = [e["file_name"] for e in gt["images"]]
                inf._decode_coco(p, names, [(e["height"], e["width"]) for e in gt["images"]], d=d)
            torch.cuda.synchronize()
            load.append((time.perf_counter() - t0) * 1e3)
        engine.STAGE_TIMING["enabled"] = True
        per = {s: [] for s in STAGES}
        for _ in range(reps):
            engine.STAGE_TIMING["events"].clear()
            inf.evaluate_coco(gp, dp, max_dets=md)
            torch.cuda.synchronize()
            sums = {}
            for s, a, b in engine.STAGE_TIMING["events"]:
                sums[s] = sums.get(s, 0.0) + a.elapsed_time(b)
            for s in STAGES:
                per[s].append(sums.get(s, 0.0))
        engine.STAGE_TIMING["enabled"] = False
        engine.STAGE_TIMING["events"].clear()
        t0 = time.perf_counter()
        want = ce.evaluate(gt, dt, max_dets=md)
        t_oracle = (time.perf_counter() - t0) * 1e3
        exact = bool(np.array_equal(got["precision"], want["precision"]) and np.array_equal(got["recall"], want["recall"])
                     and got["stats"] == want["stats"])
        out.append({"workload": name, "max_dets": list(md), "n_gt": len(gt["annotations"]), "n_dt": len(dt["annotations"]),
                    "stage_ms": {s: round(float(np.median(v)), 3) for s, v in per.items()},
                    "evaluate_coco_ms": round(float(np.median(e2e)), 2), "file_load_ms": round(float(np.median(load)), 2),
                    "oracle_numpy_ms": round(t_oracle, 1), "stats": got["stats"], "exact": exact})
        print(json.dumps(out[-1]), flush=True)
    return out


def order_scaling(reps, warmup):
    dev = torch.device("cuda:0")
    out = []
    for n in (32_000, 320_000, 3_200_000):
        rng = np.random.default_rng(n)
        score = rng.integers(0, 1000, n) / 1000.0
        img = np.arange(n) // 500                                   # the DT list is in (category, image, file order)
        seg_off = np.concatenate([np.arange(0, n, 500), [n]]).astype(np.int64)
        t = [torch.as_tensor(a, device=dev) for a in (score, np.zeros(n, np.int32), img.astype(np.int32), seg_off)]
        for _ in range(warmup):
            engine.coco_eval_order(t[0], t[1], t[2], t[3], 1, len(seg_off) - 1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms = []
        for _ in range(reps):
            a.record()
            rank, corder, morder = engine.coco_eval_order(t[0], t[1], t[2], t[3], 1, len(seg_off) - 1)
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        want_c = np.argsort(-score, kind="stable")
        want_m = np.lexsort((np.arange(n), -score, img))
        want_r = np.empty(n, np.int64)
        want_r[want_m] = np.arange(n) - seg_off[img[want_m]]
        exact = bool(np.array_equal(corder.cpu().numpy(), want_c) and np.array_equal(morder.cpu().numpy(), want_m)
                     and np.array_equal(rank.cpu().numpy(), want_r))
        out.append({"n_dt": n, "order_ms": round(float(np.median(ms)), 3), "exact": exact})
        print(json.dumps(out[-1]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cocoeval_bench.py needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    with tempfile.TemporaryDirectory() as tmp:
        res = run("micrograph_8192", [(8192, 8192)], 20000, 10, args.reps, args.warmup, tmp)
        res += run("batch_64x1024", [(1024, 1024)] * 64, 500, 11, args.reps, args.warmup, tmp)
    scaling = order_scaling(args.reps, args.warmup)
    line = json.dumps({"bench": "cocoeval", "gpu": gpu, "reps": args.reps, "warmup": args.warmup, "results": res,
                       "order_scaling": scaling, "exact": all(r["exact"] for r in res + scaling)})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
