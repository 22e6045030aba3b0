"""The opt-in neighbours_results.csv: the neighbour pass (engine.neighbours) next to trace + K5 on the same sets, the CSV end to end,
and the host alternative (unpack the masks, scipy.spatial.cKDTree for the centroid nearest neighbour and one Euclidean distance
transform per instance for the edge distance and the touching pairs), with output checks in the same run.

Two workloads, the same as scripts/shape_bench.py (synthetic_heads -> engine.paste(frames=None) -> K5):
  micrograph : one 8192 x 8192 frame with ~20 k instances;
  batch      : 64 frames of 1024 x 1024 with ~500 instances each.
Stage times are CUDA events (engine.STAGE_TIMING) over warm repetitions, summed over the frames: trace + K5 is every stage of
engine.measure; the neighbour pass is moments, plan, scan and search (the cell-list sizing synchronisation falls between the scan
and the search and is not a device stage).  The CSV end to end is a host clock around engine.neighbours + neighbours_csv_text for
every frame, D2H included.  The host alternative runs on a sample of the first frame's instances: per instance, one cKDTree query
and one EDT of the complement of the mask over the instance's bbox grown by its centroid-NN distance, from which the least distance to
every other mask in that window is read; its time per instance is scaled to the workload.  Checks: the device text against csv.writer
over inference.neighbour_rows, and the sample's nearest neighbour, closest neighbour, edge distance and touching count against
oracle/neighbours.py.  Prints one JSON line with the GPU name and power limit.

    python scripts/neighbour_bench.py [--reps 10] [--warmup 3] [--sample 200] [--out file.json]
"""
import argparse
import csv
import io
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
from scipy import ndimage, spatial

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepemia_b200 import engine, synthetic as syn  # noqa: E402
from deepemia_b200.functions import inference as inf  # noqa: E402
from oracle import neighbours as onb  # noqa: E402

CLASS_NAMES = ["pore", "throat", "grain"]
UM_PIX = 0.5


def build(dev, frames, n_per_frame, H, W, seed):
    out = []
    for f in range(frames):
        probs, boxes, _, classes = syn.synthetic_heads(seed + f, n_per_frame, H, W, rmin=4, rmax=30, margin=0)
        s = engine.paste(torch.as_tensor(probs, device=dev), torch.as_tensor(boxes, device=dev), H, W, frames=None)
        fields, cidx = inf._class_table([int(c) % 3 for c in classes[:s.n]], CLASS_NAMES)
        out.append((f"img{f:03d}.tif", s, cidx, fields))
    return out


def timed(fn, n_frames):
    engine.STAGE_TIMING["enabled"] = True
    try:
        fn()
        return {k: v * n_frames for k, v in engine.stage_summary().items()}
    finally:
        engine.STAGE_TIMING["enabled"] = False


def pieces(s):
    meta = s.meta.cpu().numpy()
    off = s.crop_off.cpu().numpy()
    words = s.crops.cpu().numpy().view(np.uint32)
    out = []
    for i in range(s.n):
        ry0, wc0, ch, cw = (int(v) for v in meta[i, :4])
        w = np.ascontiguousarray(words[off[i]:off[i] + ch * cw].reshape(ch, cw))
        m = np.unpackbits(w.view(np.uint8), axis=1, bitorder="little").astype(bool)
        out.append((ry0, wc0 * 32, m) if m.any() else None)
    return out


def host_alternative(s, cidx, listed, idx):
    """Per image: every mask unpacked to the host, centroids and one cKDTree per class; per sampled instance: the tree's nearest
    centroid, and one EDT of the complement of the mask over its bbox grown by that distance, read under the other masks of the class
    whose bboxes meet the window.  Returns (ms for the whole image, ms per sampled instance, {i: (nearest, edge distance)})."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ps = [onb.tight(p) if ok else None for p, ok in zip(pieces(s), listed)]
    cls = np.asarray(cidx)
    cent = np.full((s.n, 2), np.nan)
    box = np.zeros((s.n, 4), np.int64)
    for k in np.nonzero(listed)[0]:
        y0, x0, m = ps[k]
        ys, xs = np.nonzero(m)
        cent[k] = (xs.mean() + x0, ys.mean() + y0)
        box[k] = (y0, x0, y0 + m.shape[0] - 1, x0 + m.shape[1] - 1)
    trees = {}
    for c in np.unique(cls[listed]):
        members = np.nonzero(listed & (cls == c))[0]
        trees[c] = (members, spatial.cKDTree(cent[members]))
    t1 = time.perf_counter()
    out = {}
    for i in idx:
        members, tree = trees[cls[i]]
        if len(members) < 2:
            out[int(i)] = (-1, None)
            continue
        d, j = tree.query(cent[i], k=2)
        nn = int(members[j[1]])
        r = int(np.ceil(d[1])) + 2
        y0, x0, y1, x1 = box[i, 0] - r, box[i, 1] - r, box[i, 2] + r, box[i, 3] + r
        win = np.zeros((y1 - y0 + 1, x1 - x0 + 1), bool)
        py, px, pm = ps[i]
        win[py - y0:py - y0 + pm.shape[0], px - x0:px - x0 + pm.shape[1]] = pm
        dist = ndimage.distance_transform_edt(~win)
        best = None
        near = members[(box[members, 0] <= y1) & (box[members, 2] >= y0) & (box[members, 1] <= x1) & (box[members, 3] >= x0)]
        for k in near:
            if k == i:
                continue
            ky, kx, km = ps[k]
            ys, xs = np.nonzero(km)
            ys, xs = ys + ky - y0, xs + kx - x0
            ok = (ys >= 0) & (ys < win.shape[0]) & (xs >= 0) & (xs < win.shape[1])
            if ok.any():
                v = float(dist[ys[ok], xs[ok]].min())
                best = v if best is None else min(best, v)
        out[int(i)] = (nn, best)
    t2 = time.perf_counter()
    return (t1 - t0) * 1e3, (t2 - t1) * 1e3 / max(len(idx), 1), out


def run(dev, wname, n_frames, n_per_frame, H, W, seed, reps, warmup, sample):
    frames = build(dev, n_frames, n_per_frame, H, W, seed)
    measure = lambda: [engine.measure(s, um_pix=UM_PIX, min_area=engine.default_min_area(H, W)) for _, s, _, _ in frames]  # noqa: E731
    nbs = []
    nb_pass = lambda: nbs.extend(engine.neighbours(s, cidx, UM_PIX) for _, s, cidx, _ in frames)                           # noqa: E731
    k5, nbt, csvt, e2e = [], [], [], []
    for it in range(warmup + reps):
        a = timed(measure, n_frames)
        nbs.clear()
        b = timed(nb_pass, n_frames)
        c = timed(lambda: [engine.neighbours_csv_text(s, nb, name, "500", cidx, fields)
                           for (name, s, cidx, fields), nb in zip(frames, nbs)], n_frames)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        texts = [engine.neighbours_csv_text(s, engine.neighbours(s, cidx, UM_PIX), name, "500", cidx, fields)
                 for name, s, cidx, fields in frames]
        t1 = time.perf_counter()
        if it >= warmup:
            k5.append(a); nbt.append(b); csvt.append(c); e2e.append((t1 - t0) * 1e3)
    med = lambda runs: {k: round(float(np.median([r.get(k, 0.0) for r in runs])), 4) for k in runs[0]}           # noqa: E731
    k5_med, nb_med = med(k5), med(nbt)
    rows = []
    for (name, s, cidx, fields), nb in zip(frames, nbs):
        rows += inf.neighbour_rows(s, nb, name, "500", cidx, fields)
    buf = io.StringIO()
    csv.writer(buf).writerows(rows)
    text_equal = b"".join(texts) == buf.getvalue().encode("utf-8")
    # the sample of the first frame: device values against the oracle, and the host alternative's time
    name, s, cidx, _ = frames[0]
    ints = nbs[0].ints.cpu().numpy()
    vals = nbs[0].values.cpu().numpy()
    listed = ints[:, 0] == 1
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.choice(np.nonzero(listed)[0], min(sample, int(listed.sum())), replace=False))
    want_f, want_i = onb.Neighbours(pieces(s), listed, cidx).rows(UM_PIX, idx)
    exact = bool(np.array_equal(ints[idx, :4], want_i[idx, :4]) and np.array_equal(vals[idx].view(np.int64), want_f[idx].view(np.int64)))
    host_image_ms, host_per_inst, host = host_alternative(s, cidx, listed, idx)
    # the tree finds the same nearest centroid; the EDT edge distance is the Euclidean one, so equal to sqrt(D2) (times um_pix)
    host_agrees = all(host[int(i)][0] == ints[i, 1] and (host[int(i)][1] is None or host[int(i)][1] * UM_PIX == vals[i, 3]) for i in idx)
    n_inst = sum(s.n for _, s, _, _ in frames)
    return {"workload": wname, "frames": n_frames, "H": H, "W": W, "instances": n_inst, "rows": len(rows),
            "touching_rows": int(sum(r[9] > 0 for r in rows)),
            "trace_k5_stage_ms": k5_med, "trace_k5_ms": round(sum(k5_med.values()), 4),
            "neighbour_stage_ms": nb_med, "neighbour_ms": round(sum(nb_med.values()), 4),
            "csv_stage_ms": med(csvt), "neighbours_and_csv_e2e_ms_host_clock": round(float(np.median(e2e)), 3),
            "csv_bytes": sum(len(t) for t in texts),
            "host_alternative_sample": len(idx), "host_alternative_unpack_tree_ms_first_frame": round(host_image_ms, 1),
            "host_alternative_ms_per_instance": round(host_per_inst, 4),
            "host_alternative_ms_scaled": round(host_image_ms * n_frames + host_per_inst * n_inst, 1),
            "check": {"text_equal_neighbour_rows": text_equal, "sample_exact_vs_oracle": exact, "host_alternative_agrees": host_agrees}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sample", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("neighbour_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True).stdout.strip()
    res = [run(dev, "micrograph_8192", 1, 20000, 8192, 8192, 100, args.reps, args.warmup, args.sample),
           run(dev, "batch_64x1024", 64, 500, 1024, 1024, 1000, args.reps, args.warmup, args.sample)]
    ok = all(r["check"]["text_equal_neighbour_rows"] and r["check"]["sample_exact_vs_oracle"] for r in res)
    line = json.dumps({"bench": "neighbour", "gpu": gpu, "reps": args.reps, "warmup": args.warmup, "results": res, "outputs_ok": ok})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
