#!/usr/bin/env python
"""bench.py — throughput of the fused post-head hot path on B200 (BASELINE.json metric: instances measured/sec and
mask MPix/sec; % of HBM roofline).

Workload (BASELINE config 5, SURVEY.md §8d): 2048 synthetic 1024x1024 tiles x ~Poisson(500) Mask R-CNN head outputs
(28x28 probabilities + box + score + class), sharded tile t -> rank t mod G (strong scaling, no data-path collective).
One step = one pass of the whole path over this rank's shard:
    K1 paste + threshold + bit-pack (full-frame bit masks into a reusable HBM arena + bbox crops + bbox + area)
 -> K5 external contours + morphometry  -> K4 deduplicate_masks_smart(0.7) -> overlap + containment rules.
`value`   : device-resident inputs, CUDA-event timed, max over ranks.
`e2e`     : same path through the public API from pinned HOST buffers, H2D of the step's inputs and D2H of the
            measurement table + kept lists inside the timed region.
`roofline`: dominant kernel (K1) algorithmic bytes / its CUDA-event duration vs MEASURED_PEAKS.json hbm_gbs.
`cpu_baseline`: the CPU oracle (port of the reference's numpy/OpenCV path) on a bounded sample of the same tiles, rank 0.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 1024
N_TILES = 2048
MEAN_INST = 500
UM_PIX = 0.5
DEDUP_IOU = 0.7
N_PROTO = 1024


def _prototypes():
    from deepemia_b200 import synthetic as syn
    rng = np.random.default_rng(12345)
    protos = np.zeros((N_PROTO, 28, 28), np.float32)
    for k in range(N_PROTO):
        poly = syn.star_polygon(rng, 0.0, 0.0, 20.0)
        protos[k], _ = syn.head_from_poly(rng, poly)
    return protos


def tile_heads(t):
    """Head outputs of tile t (seed 5000+t): proto ids, boxes, scores, classes.  ~10 % are jittered re-detections."""
    rng = np.random.default_rng(5000 + t)
    n = max(1, int(rng.poisson(MEAN_INST)))
    proto = rng.integers(0, N_PROTO, n)
    cx = rng.uniform(40, W - 40, n); cy = rng.uniform(40, H - 40, n)
    r = rng.uniform(8, 30, n)
    ax = rng.uniform(0.8, 1.0, n); ay = rng.uniform(0.8, 1.0, n)
    ndup = n // 10
    if ndup:
        src = rng.integers(0, n - ndup, ndup)
        dst = np.arange(n - ndup, n)
        proto[dst] = proto[src]; r[dst] = r[src]; ax[dst] = ax[src]; ay[dst] = ay[src]
        cx[dst] = cx[src] + rng.uniform(-1.5, 1.5, ndup); cy[dst] = cy[src] + rng.uniform(-1.5, 1.5, ndup)
    boxes = np.stack([cx - r * ax, cy - r * ay, cx + r * ax, cy + r * ay], 1).astype(np.float32)
    scores = rng.permutation(n).astype(np.float32)
    scores = (0.05 + 0.95 * (scores + rng.uniform(0.1, 0.9, n).astype(np.float32)) / n).astype(np.float32)
    classes = (rng.random(n) < 0.5).astype(np.int32)
    return proto, boxes, scores, classes


def shard(rank, world, n_tiles, variant=0):
    """This rank's tiles of sweep `variant`: tile ids t = rank, rank + world, ... of the 2048-tile sweep; variant v uses the tile
    seeds 5000 + v * n_tiles + t, i.e. a different synthetic data set of the same statistics (the timed steps rotate through
    several variants so that no step sees the per-tile instance counts of its predecessor)."""
    tiles = [t for t in range(n_tiles) if t % world == rank]
    parts = [tile_heads(variant * n_tiles + t) for t in tiles]
    offs = np.zeros(len(tiles) + 1, np.int32)
    offs[1:] = np.cumsum([len(p[0]) for p in parts])
    cat = [np.concatenate([p[k] for p in parts]) for k in range(4)]
    return tiles, offs, cat


def _clock_sampler(path):
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                             stdout=open(path, "w"), stderr=subprocess.DEVNULL)
    except Exception:
        return None
    atexit.register(_stop_sampler, p)       # the sampler never outlives the benchmark, whichever way it ends
    return p


def _stop_sampler(p):
    if p is not None and p.poll() is None:
        p.terminate()
        p.wait()


def _clock_summary(path, gpu_index):
    sm, mx, reasons = [], [], set()
    try:
        for line in open(path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or f[0] != str(gpu_index):
                continue
            sm.append(float(f[1])); mx.append(float(f[2]))
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
    except Exception:
        pass
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    busy = [s for s in sm if s > 0.5 * max(sm)] or sm
    return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


_W = {}


def _worker_init(protos):
    """Once per worker process, OUTSIDE every timed region: single-threaded libraries, imports, the prototype table."""
    os.environ["OMP_NUM_THREADS"] = "1"
    import cv2
    import torch
    cv2.setNumThreads(1)
    torch.set_num_threads(1)
    from deepemia_b200 import synthetic as syn
    from oracle import pipeline
    _W["protos"], _W["syn"], _W["pipeline"] = protos, syn, pipeline


def _oracle_tile(t):
    """One tile of the sweep through the CPU oracle (port of the reference path).  Returns its own compute seconds too."""
    if "protos" not in _W:
        _worker_init(_prototypes())
    proto, boxes, scores, classes = tile_heads(t)
    t0 = time.perf_counter()
    final, rows, masks = _W["pipeline"].run_tile(_W["protos"][proto], boxes, scores, classes, H, W, um_pix=UM_PIX,
                                                 rules=_W["syn"].POLYHIPES_RULES, dedup_iou=DEDUP_IOU)
    dt = time.perf_counter() - t0
    vals = [[float(v) for v in r[3:15]] for r in rows]
    return t, len(proto), final, vals, dt


def _as_written_overhead(t):
    """Seconds per measured instance of what the reference's measurement loop does ON TOP of the computation: the 3-channel
    stack + JPEG dump of every mask (src/functions/inference.py:1153-1162) and the per-instance gc.collect() (:1253), measured
    with a tile's final masks alive as in the reference.  8 instances are enough for a per-instance figure."""
    import gc
    import tempfile
    import cv2
    if "protos" not in _W:
        _worker_init(_prototypes())
    proto, boxes, scores, classes = tile_heads(t)
    _, _, masks = _W["pipeline"].run_tile(_W["protos"][proto], boxes, scores, classes, H, W, um_pix=UM_PIX,
                                          rules=_W["syn"].POLYHIPES_RULES, dedup_iou=DEDUP_IOU)
    k = min(8, len(masks))
    with tempfile.TemporaryDirectory() as d:
        t0 = time.perf_counter()
        for i in range(k):
            m = (np.asarray(masks[i]) > 0).astype(np.uint8) * 255
            cv2.imwrite(os.path.join(d, f"mask_{i}.jpg"), np.stack([m] * 3, axis=-1))
            gc.collect()
        dt = time.perf_counter() - t0
    return dt / max(k, 1), len(masks)


class CpuArm:
    """The CPU oracle over tiles of the sweep: P = all host cores the process may use, one single-threaded worker process per
    core, created ONCE (imports, prototype table and one untimed warm-up tile per worker outside the timed region)."""

    def __init__(self, protos, procs=None):
        import multiprocessing as mp
        try:
            avail = len(os.sched_getaffinity(0))
        except Exception:
            avail = os.cpu_count() or 1
        self.procs = max(1, min(avail, procs or avail))
        self.pool = mp.get_context("spawn").Pool(self.procs, initializer=_worker_init, initargs=(protos,))
        self.warm = self.pool.map_async(_oracle_tile, [N_TILES + 7 + k for k in range(self.procs)], chunksize=1)   # untimed

    def run(self, tiles):
        """(wall seconds of pool.map over `tiles`, results)."""
        self.warm.wait()
        t0 = time.perf_counter()
        res = self.pool.map(_oracle_tile, list(tiles), chunksize=1)
        return time.perf_counter() - t0, res

    def as_written(self):
        sec_per_inst, _ = self.pool.apply(_as_written_overhead, (N_TILES + 3,))
        return sec_per_inst

    def submit(self, fn, arg):
        return self.pool.apply_async(fn, (arg,))

    def close(self):
        self.pool.terminate()


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    protos = _prototypes()
    arm = CpuArm(protos)
    P = arm.procs
    ntl = args.ref_tiles if args.ref_tiles > 0 else 2 * P
    secs, inst, per_tile = [], 0, []
    for s in range(args.warmup + args.steps):
        tiles = [(s * ntl + k) % args.tiles for k in range(ntl)]
        dt, res = arm.run(tiles)
        if s >= args.warmup:
            secs.append(dt); inst += sum(r[1] for r in res); per_tile += [r[4] for r in res]
    arm.close()
    total = sum(secs)
    v = inst / total
    line = {"impl": "reference", "metric": "instances_per_sec", "value": v, "unit": "instances/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(1, args.steps), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"config5 sample: {ntl} of {args.tiles} tiles (1024x1024, ~500 instances) per step, CPU oracle",
                       "processes": P, "tiles_per_step": ntl, "mean_tile_compute_s": float(np.mean(per_tile)) if per_tile else None},
            "cpu_baseline": {"value": v, "unit": "instances/s", "cores": P, "kind": "port",
                             "sample": f"{ntl} tiles x {args.steps} steps on {P} single-threaded worker processes (pool, imports and one warm-up "
                                       "tile per worker outside the timed region), compute only (no JPEG dump / gc.collect)"},
            "e2e": {"value": v, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "mask_mpix_per_sec": v * H * W / 1e6}
    print(json.dumps(line))


DUMP_CAPS = {"tile": 1 << 16, "kept": 1 << 19, "instance": 1 << 19, "record": 1 << 16}   # rows per group: < 40 MB in all
DUMP_MASKS, DUMP_PATCH = 256, 64


def _sample_rows(n, cap, seed):
    """All of 0..n-1, or a fixed seeded sample of `cap` of them in ascending order."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, cap, replace=False))


def dump_outputs(out_dir, res, suffix=""):
    """Write what a caller of the device-resident step receives (`res`: the step's results, finalized) to out_dir/<name>.npy,
    integers as float64 (ids) or float32 (coordinates, counts), so that two builds can be compared output for output.
    Each group of arrays shares its rows; a group longer than DUMP_CAPS is a fixed seeded sample, <group>_rows holds the rows:
        tile:     kept_len [T]                    kept instances per tile
        kept:     kept_idx [K]                    kept instance ids, tile by tile in list order
        instance: bbox [n, 4], area [n]           per pasted instance: (y_min, x_min, y_max, x_max) inclusive (-1: empty), pixels
        record:   records [R, 16], record_inst [R]  morphometry rows (include/emia.h) and the instance of each row
        mask:     mask_patches [k, 64, 64], mask_origin [k, 2]  masks (0 / 1) of DUMP_MASKS seeded instances: the 64 x 64 window
                  at (y, x) = mask_origin, their bbox corner moved into the frame"""
    import torch
    from deepemia_b200 import engine
    os.makedirs(out_dir, exist_ok=True)
    kept_len, kept_idx, bbox, area, rec, rec_inst = [], [], [], [], [], []
    for r in res:
        g, it, m = r["kept"], r["iset"], r["meas"]
        ln, ix, co = g.length.cpu().numpy(), g.idx.cpu().numpy(), g.cap_off_host
        kept_len.append(ln)
        kept_idx += [ix[co[k]:co[k] + ln[k]] for k in range(g.G)]
        bbox.append(it.bbox.cpu().numpy()); area.append(it.area.cpu().numpy())
        rec.append(m.records.cpu().numpy()); rec_inst.append(m.rec_inst.cpu().numpy())
    cat = np.concatenate
    groups = {"tile": {"kept_len": (cat(kept_len), np.float32)},
              "kept": {"kept_idx": (cat(kept_idx), np.float64)},
              "instance": {"bbox": (cat(bbox), np.float32), "area": (cat(area), np.float32)},
              "record": {"records": (cat(rec), np.float64), "record_inst": (cat(rec_inst), np.float64)}}
    out = {}
    for seed, (grp, arrays) in enumerate(groups.items()):
        rows = _sample_rows(len(next(iter(arrays.values()))[0]), DUMP_CAPS[grp], seed)
        out[f"{grp}_rows"] = rows.astype(np.float64)
        out.update({k: a[rows].astype(t) for k, (a, t) in arrays.items()})
    sel = _sample_rows(len(groups["instance"]["area"][0]), DUMP_MASKS, len(groups))
    patches, origins = [], []
    for r in res:
        it, i0 = r["iset"], r["inst0"]
        loc = sel[(sel >= i0) & (sel < i0 + it.n)] - i0
        if not len(loc):
            continue
        P = min(DUMP_PATCH, it.H, it.W)
        full = engine.unpack_masks(it, loc)
        bb = it.bbox[torch.as_tensor(loc, device=it.device)].long()
        y0, x0 = bb[:, 0].clamp(0, it.H - P), bb[:, 1].clamp(0, it.W - P)
        ar = torch.arange(P, device=it.device)
        k = torch.arange(len(loc), device=it.device)
        patches.append(full[k[:, None, None], (y0[:, None] + ar)[:, :, None], (x0[:, None] + ar)[:, None, :]].cpu().numpy())
        origins.append(torch.stack([y0, x0], 1).cpu().numpy())
    out["mask_rows"] = sel.astype(np.float64)
    out["mask_patches"] = cat(patches).astype(np.float32)
    out["mask_origin"] = cat(origins).astype(np.float32)
    for k, a in out.items():
        np.save(os.path.join(out_dir, f"{k}{suffix}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--tiles", type=int, default=N_TILES)
    ap.add_argument("--variant", type=int, default=int(os.environ.get("EMIA_PASTE_VARIANT", "2")))
    ap.add_argument("--arena-gb", type=float, default=32.0)
    ap.add_argument("--ref-tiles", type=int, default=0, help="tiles of the CPU sample (0 = 2 per worker process)")
    ap.add_argument("--shards", type=int, default=4, help="distinct synthetic data sets the steps rotate through")
    ap.add_argument("--batches", type=int, default=1, help="tile batches of the device-resident pass (1: no overlap; the "
                    "latency-bound kernels lose more under the paste kernel's HBM write stream than the overlap hides)")
    ap.add_argument("--e2e-batches", type=int, default=0, help="tile batches of the three-stream pipeline with host inputs (0 = auto)")
    ap.add_argument("--paste-ctas", type=int, default=0, help="resident paste CTAs per SM (0 = kernel default)")
    ap.add_argument("--no-graph", action="store_true", help="enqueue every step kernel by kernel instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-flows", action="store_true", help="skip the config 2 / 3a / 3b / 4 legs")
    ap.add_argument("--flows-only", default="", help="comma list of config2,config3a,config3b,config4: run only those legs")
    ap.add_argument("--workload", default="", help="config3a | config3b: ONE micrograph split over all ranks (torchrun), see bench_flows.run_split_workload")
    ap.add_argument("--breakdown", action="store_true", help="extra untimed pass with per-stage CUDA events (stderr)")
    ap.add_argument("--device-pass-only", action="store_true", help="profiling aid: run only the warm-up + timed device-resident steps")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the results of the last timed device-resident step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.workload:
        import bench_flows
        return bench_flows.run_split_workload(args.workload, args.steps, args.warmup)

    import torch
    import torch.distributed as dist
    from deepemia_b200 import engine, synthetic as syn

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    protos = _prototypes()
    # CPU legs start now, in worker processes, and run beside the GPU measurements (rank 0 of a 1-GPU run only)
    want_cpu = world == 1 and not args.no_cpu_baseline and not args.device_pass_only
    flows = [] if (args.no_flows or world > 1 or args.device_pass_only) else ["config2", "config3a", "config3b", "config4"]
    if args.flows_only:
        flows = [f for f in args.flows_only.split(",") if f]
    arm, legs = None, {}
    if want_cpu:
        import bench_flows
        arm = CpuArm(protos)
        legs = {f: arm.submit(bench_flows.oracle_leg, f) for f in flows if f != "scalebar"}
    if args.flows_only:
        import bench_flows
        out = {}
        for f in flows:
            if f == "scalebar":
                out[f] = bench_flows.run_scalebar_leg(dev, args.steps, args.warmup)
                continue
            out[f] = bench_flows.run_workload(f, dev, args.steps, args.warmup, leg=legs[f].get() if f in legs else None)
        if arm is not None:
            arm.close()
        print(json.dumps(out))
        return

    V = max(1, args.shards)
    shards = []
    d_protos = torch.as_tensor(protos, device=dev)
    for v in range(V):
        tiles, offs, (proto_id, boxes, scores, classes) = shard(rank, world, args.tiles, v)
        d = {"tiles": tiles, "offs": offs, "n": int(offs[-1]),
             "probs": d_protos[torch.as_tensor(proto_id, device=dev)].contiguous(), "boxes": torch.as_tensor(boxes, device=dev),
             "scores": torch.as_tensor(scores, device=dev), "classes": torch.as_tensor(classes, device=dev)}
        shards.append(d)
    pw = engine.pitch_words_for(W)
    frame_bytes = H * pw * 4
    n_max = max(d["n"] for d in shards)
    slots = max(1, min(n_max, int(args.arena_gb * 2**30) // frame_bytes))
    arena = torch.empty((slots, H, pw), dtype=torch.int32, device=dev)
    rules = syn.POLYHIPES_RULES

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    pipe = engine.TilePipeline(H, W, um_pix=UM_PIX, rules=rules, dedup_iou=DEDUP_IOU, frames=arena, variant=args.variant,
                               batches=args.batches, paste_ctas_per_sm=args.paste_ctas, device=dev)

    def step(d, time_k1=False):
        return pipe.run(d["probs"], d["boxes"], d["scores"], d["classes"], d["offs"], time_k1=time_k1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing ----------------
    # set-up (untimed, not a warm-up step of the contract): every shard once, so that the caching allocator has seen every
    # buffer size and the pipeline's capacities cover every shard; a guard that trips is handled as in production (re-run)
    for d in shards:
        for _ in range(3):
            step(d)
            if not pipe.aborted():
                break
    # K1 on its own CUDA events (roofline.achieved): an eager pass over the rotating shards — inside a replayed graph no event
    # can be placed around a single kernel node
    k1_events = []
    for i in range(max(3, min(args.steps, V))):
        d = shards[i % V]
        step(d, time_k1=True)
        k1_events.append((d, list(pipe.k1_events)))
    torch.cuda.synchronize()
    assert not pipe.aborted()
    # the whole sync-free step of every resident shard captured in a CUDA graph (one chain of kernel nodes; shared memory pool)
    graphs, pool, launches_per_step = [], None, 0
    if not args.no_graph:
        for d in shards:
            l0 = engine.LAUNCHES["count"]
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool):
                r = step(d)
            pool = g.pool()
            graphs.append((g, r, pipe._abort))
            launches_per_step = engine.LAUNCHES["count"] - l0

    def timed_step(k):
        if graphs:
            g, r, ab = graphs[k % V]
            g.replay()
            return r, ab
        r = step(shards[k % V])
        return r, pipe._abort

    res = None
    for i in range(args.warmup):
        # keep the previous step's results alive while the next one runs, exactly as the timed loop does
        res, _ = timed_step(i)
    barrier()
    # the clock log goes to a temporary file: the benchmark writes nothing into the source tree (it may be read-only)
    clk_fd, clk_path = tempfile.mkstemp(prefix=f"emia_clocks_rank{rank}_", suffix=".csv")
    os.close(clk_fd)
    atexit.register(os.remove, clk_path)
    sampler = _clock_sampler(clk_path) if rank == 0 else None
    l0 = engine.LAUNCHES["count"]
    x0 = pipe.exact_runs
    barrier()
    step_ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    sticky = torch.zeros(1, dtype=torch.int32, device=dev)
    n_done = 0
    t_host0 = time.perf_counter()
    ev[0].record()
    step_ev[0].record()
    for i in range(args.steps):
        res, ab = timed_step(args.warmup + i)
        sticky.logical_or_(ab)                           # validity of every step, looked at after the timed region
        n_done += shards[(args.warmup + i) % V]["n"]
        step_ev[i + 1].record()
    ev[1].record()
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / args.steps
    barrier()
    aborts = [sticky]
    exact_in_timed = pipe.exact_runs - x0
    assert not any(int(a.item()) for a in aborts), "a capacity guard tripped in the timed region: that step's results are invalid"
    k1_ms = [float(sum(a.elapsed_time(b) for a, b in evs)) for _, evs in k1_events]
    per_step_ms = [step_ev[i].elapsed_time(step_ev[i + 1]) for i in range(args.steps)]
    launches = (launches_per_step * args.steps) if graphs else (engine.LAUNCHES["count"] - l0)
    ms_total = ev[0].elapsed_time(ev[1])
    last = shards[(args.warmup + args.steps - 1) % V]
    for r in res:
        r["meas"].finalize()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res, f"_rank{rank}" if world > 1 else "")
    if args.breakdown and rank == 0:
        # un-overlapped pass (one batch, one stream) with per-stage CUDA events
        d = shards[0]
        engine.STAGE_TIMING["enabled"] = True
        t0 = time.perf_counter()
        engine.run_tiles(d["probs"], d["boxes"], d["scores"], d["classes"], d["offs"], H, W, um_pix=UM_PIX, rules=rules, dedup_iou=DEDUP_IOU,
                         frames=arena, variant=args.variant)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        engine.STAGE_TIMING["enabled"] = False
        summ = engine.stage_summary()
        print(json.dumps({"stage_ms": summ, "sum_ms": sum(summ.values()), "wall_ms": wall}), file=sys.stderr)
    if args.device_pass_only:
        _stop_sampler(sampler)
        if rank == 0:
            print(json.dumps({"device_pass_only": True, "ms_per_step": ms_total / args.steps, "instances_per_step": n_done / args.steps,
                              "per_step_ms": per_step_ms}))
        if world > 1:
            dist.destroy_process_group()
        return
    # K1 alone (nothing else on the GPU), for comparison with its in-pipeline duration
    k1_alone = []
    d0 = shards[0]
    meta0, coff0 = engine.paste_plan(d0["boxes"], H, W)
    words0 = int(coff0[d0["n"]].item())
    crops0 = torch.empty(max(words0, 1), dtype=torch.int32, device=dev)
    for _ in range(4):
        ev[2].record()
        iset_alone = engine.paste(d0["probs"], d0["boxes"], H, W, frames=arena, variant=args.variant, plan=(meta0, coff0, words0), crops_out=crops0)
        ev[3].record()
        torch.cuda.synchronize()
        k1_alone.append(ev[2].elapsed_time(ev[3]))
    k1_alone = k1_alone[1:]
    crop_words = {id(d0): iset_alone.total_crop_words}
    for d in shards[1:]:
        crop_words[id(d)] = int(engine.paste_plan(d["boxes"], H, W)[1][d["n"]].item())
    del iset_alone, crops0
    # crops-only variant of the same step (no full-frame bit masks: what the path itself consumes), as a second roofline line
    pipe_c = engine.TilePipeline(H, W, um_pix=UM_PIX, rules=rules, dedup_iou=DEDUP_IOU, frames=None, variant=args.variant,
                                 batches=1, device=dev)
    for d in shards:
        pipe_c.run(d["probs"], d["boxes"], d["scores"], d["classes"], d["offs"])
        pipe_c.aborted()
    barrier()
    kc_events, n_c = [], 0
    ev[2].record()
    for i in range(args.steps):
        d = shards[i % V]
        pipe_c.run(d["probs"], d["boxes"], d["scores"], d["classes"], d["offs"], time_k1=True)
        kc_events.append(list(pipe_c.k1_events)); n_c += d["n"]
    ev[3].record()
    barrier()
    ms_crops = ev[2].elapsed_time(ev[3]) / args.steps
    k1c_ms = float(np.mean([sum(a.elapsed_time(b) for a, b in evs) for evs in kc_events]))
    assert not pipe_c.aborted()
    del pipe_c
    # ---------------- end-to-end (host buffers) ----------------
    # pinned host copies of two shards.  Tile batches: the H2D copy of batch b+1 runs beside the kernels of batch b, but every batch
    # pays the latency-bound kernels' fixed ~0.4 ms again, so the count is small.  Measured with fp16 head outputs
    # (scripts/e2e_batches_sweep.sh, ms per step): 2048 tiles: 5 / 6 / 8 / 12 / 16 batches -> 36.4 / 36.8 / 34.8 / 36.6 / 37.8;
    # 1024 tiles: 4 / 6 / 8 -> 19.1 / 19.5 / 19.9; 512 tiles: 2 / 3 / 4 / 6 -> 11.5 / 10.9 / 10.9 / 11.3; 256 tiles: 2 / 3 / 4 ->
    # 6.3 / 6.3 / 7.1.  Hence 256 tiles per batch for shards of 1024 tiles and more, 128 below, at least 2 and at most 8.
    E = min(2, V)
    n_tiles = len(shards[0]["tiles"])
    e2e_batches = args.e2e_batches or int(max(2, min(8, round(n_tiles / (256.0 if n_tiles >= 1024 else 128.0)))))
    pipe_e2e = engine.TilePipeline(H, W, um_pix=UM_PIX, rules=rules, dedup_iou=DEDUP_IOU, frames=arena, variant=args.variant,
                                   batches=e2e_batches, paste_ctas_per_sm=args.paste_ctas, device=dev)
    hosts = []
    for d in shards[:E]:
        hosts.append({"offs": d["offs"], "n": d["n"], "probs": d["probs"].cpu().pin_memory(), "boxes": d["boxes"].cpu().pin_memory(),
                      "scores": d["scores"].cpu().pin_memory(), "classes": d["classes"].cpu().pin_memory()})

    def e2e_step(hd, key="probs"):
        r = pipe_e2e.run(hd[key], hd["boxes"], hd["scores"], hd["classes"], hd["offs"], to_host=True)
        torch.cuda.current_stream().synchronize()      # the pinned result buffers are complete
        if pipe_e2e.aborted():                          # the flag travels with the results; re-run with exact sizes
            r = pipe_e2e.run(hd[key], hd["boxes"], hd["scores"], hd["classes"], hd["offs"], to_host=True)
            torch.cuda.current_stream().synchronize()
        return r

    def e2e_leg(key):
        for hd in hosts:
            e2e_step(hd, key)
            e2e_step(hd, key)
        # the whole pipelined step (H2D copies, kernels of the three streams, D2H result copies) of every resident host shard
        # captured in a CUDA graph: per step the host launches one graph and waits for the results
        eg = []
        if not args.no_graph:
            pool_e = None
            for hd in hosts:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool_e):
                    r = pipe_e2e.run(hd[key], hd["boxes"], hd["scores"], hd["classes"], hd["offs"], to_host=True)
                pool_e = g.pool()
                eg.append((g, r, pipe_e2e._abort))

        def one(i):
            if eg:
                g, r, ab = eg[i % E]
                g.replay()
                torch.cuda.current_stream().synchronize()
                assert not int(ab.item()), "a capacity guard tripped in an end-to-end step"
                return r
            return e2e_step(hosts[i % E], key)
        for i in range(max(2, args.warmup)):
            r = one(i)
        barrier()
        wall, n_e = [], 0
        ev[0].record()
        for i in range(args.steps):
            t0 = time.perf_counter()
            r = one(i)
            n_e += hosts[i % E]["n"]
            wall.append(round((time.perf_counter() - t0) * 1e3, 2))
        ev[1].record()
        barrier()
        return ev[0].elapsed_time(ev[1]), n_e, wall, r, hosts[(args.steps - 1) % E]

    def valid_results(res):
        """What a caller reads from the pinned result buffers of a step: the live part of every kept list and the records that
        belong to live list slots (the buffers are capacity-sized; the rest is unspecified)."""
        out = []
        for r in res:
            hst, g = r["host"], r["kept"]
            ln = hst["kept_len"].numpy()
            co = g.cap_off_host
            idx = hst["kept_idx"].numpy()
            out.append(np.concatenate([idx[co[k]:co[k] + ln[k]] for k in range(len(ln))]) if len(ln) else np.zeros(0, np.int32))
            n_rec = int(hst["rec_off"].numpy()[int(co[-1])])
            out.append(hst["records"].numpy()[:n_rec].copy())
            out.append(hst["rec_inst"].numpy()[:n_rec].copy())
        return out

    ms_e2e32, n_e2e32, e2e_wall32, res_h, last_h = e2e_leg("probs")
    ref_valid = valid_results(res_h)
    h2d32 = int(sum(hosts[0][k].numel() * hosts[0][k].element_size() for k in ("probs", "boxes", "scores", "classes")))
    # the same with the head probabilities as fp16 — what the mask head emits under the reference's DEFAULT AMP autocast
    # (inference.py:1392-1396; the synthetic probabilities are fp16-representable, K1 widens them exactly): half the H2D bytes.
    # This is the end-to-end figure of the line (`e2e`); the fp32 transport is reported beside it.
    for hd in hosts:
        hd["probs16"] = hd["probs"].to(torch.float16).pin_memory()
        assert torch.equal(hd["probs16"].to(torch.float32), hd["probs"])
    ms_e2e, n_e2e, e2e_wall, res_h16, _ = e2e_leg("probs16")
    got_valid = valid_results(res_h16)
    same16 = len(ref_valid) == len(got_valid) and all(np.array_equal(a, b) for a, b in zip(ref_valid, got_valid))
    ms_e2e16, n_e2e16 = ms_e2e32, n_e2e32            # (slot names of the reduction below: the second leg is the fp32 one)
    res_h = res_h16
    # the floor of the end-to-end step: the SAME bytes moved (H2D of the fp16 head outputs on one stream, D2H of the results on
    # another) with no kernel in between — (i) by all ranks at once, as in the e2e leg, (ii) by one rank at a time.  On an HGX
    # board two GPUs share one PCIe switch uplink: (i) / (ii) shows how much of the multi-GPU e2e time is the host link.
    d2h_bytes = int(sum(v.numel() * v.element_size() for r in res_h for v in r["host"].values()))
    cp_dev = {k: torch.empty_like(hosts[0][k], device=dev) for k in ("probs16", "boxes", "scores", "classes")}
    cp_out_d = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8, device=dev)
    cp_out_h = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8).pin_memory()
    s_up, s_down = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def copy_only(steps):
        torch.cuda.synchronize()
        ev[2].record()
        for i in range(steps):
            hd = hosts[i % E]
            s_up.wait_stream(torch.cuda.current_stream()); s_down.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s_up):
                for k, t in cp_dev.items():
                    t[:hd[k].shape[0]].copy_(hd[k][:t.shape[0]], non_blocking=True)
            with torch.cuda.stream(s_down):
                cp_out_h.copy_(cp_out_d, non_blocking=True)
            torch.cuda.current_stream().wait_stream(s_up); torch.cuda.current_stream().wait_stream(s_down)
        ev[3].record()
        torch.cuda.synchronize()
        return ev[2].elapsed_time(ev[3]) / steps
    copy_only(2)
    barrier()
    ms_copy_all = copy_only(args.steps)
    barrier()
    ms_copy_solo = 0.0
    for r in range(world):
        if r == rank:
            ms_copy_solo = copy_only(args.steps)
        barrier()
    _stop_sampler(sampler)
    t = torch.tensor([ms_total, ms_e2e, float(np.sum(k1_ms)), ms_e2e16, ms_crops, k1c_ms, ms_copy_all, ms_copy_solo], dtype=torch.float64,
                     device=dev)
    cnt = torch.tensor([float(n_done), float(n_e2e), float(n_e2e16), float(n_c)], dtype=torch.float64, device=dev)
    per_rank = [t.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, t)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    per_rank_ms = [round(float(x[0].item()) / args.steps, 3) for x in per_rank]
    ms_total, ms_e2e, k1_sum, ms_e2e16, ms_crops, k1c_ms, ms_copy_all, ms_copy_solo = t.tolist()
    n_global, n_e2e_g, n_e2e16_g, n_c_g = cnt.tolist()
    if rank == 0:
        ms_step = ms_total / args.steps
        value = n_global / (ms_total * 1e-3)
        e2e_val = n_e2e_g / (ms_e2e * 1e-3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "6650 GB/s (of fallback)"
        # algorithmic bytes of rank 0's timed K1 launches (the steps rotate through shards of slightly different sizes)
        per_inst = 28 * 28 * 4 + 16 + 32 + 8 + 16 + 4
        k1_bytes = float(sum(d["n"] * (per_inst + frame_bytes) + 4.0 * crop_words[id(d)] for d, _ in k1_events))
        k1_rank0 = float(np.sum(k1_ms))
        k1_gbs = k1_bytes / (k1_rank0 * 1e-3) / 1e9
        n_rank0 = float(sum(d["n"] for d, _ in k1_events))
        path_bytes = float(np.mean([d["n"] * (28 * 28 * 4 + 16 + 8 + frame_bytes + 256) + 8.0 * crop_words[id(d)] for d in shards]))  # SURVEY 8d B_inst
        rank0_ms = float(per_rank[0][0].item())
        traffic = None
        try:     # DRAM bytes per instance of the paste kernel from the committed ncu --set full capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "k1_dram_traffic.json")))
            traffic = float(tj["dram_bytes_per_instance"]) * n_rank0 / len(k1_events)
        except Exception:
            pass
        k1_alone_bytes = d0["n"] * (per_inst + frame_bytes) + 4.0 * crop_words[id(d0)]
        crops_bytes = float(np.mean([d["n"] * per_inst + 4.0 * crop_words[id(d)] for d in shards]))
        h2d = int(sum(hosts[0][k].numel() * hosts[0][k].element_size() for k in ("probs16", "boxes", "scores", "classes")))
        d2h = int(sum(v.numel() * v.element_size() for r in res_h for v in r["host"].values()))
        line = {
            "metric": "instances_per_sec", "value": value, "unit": "instances/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"config5: {args.tiles} tiles x ~Poisson(500) instances, 1024x1024, tile t -> rank t mod G",
                       "instances_per_step": n_global / args.steps, "paste_variant": args.variant,
                       "frame_arena_gb": round(slots * frame_bytes / 2**30, 1), "tile_batches": args.batches, "e2e_tile_batches": e2e_batches,
                       "distinct_shards_rotated": V, "cuda_graph": bool(graphs),
                       "host_syncs_per_step": exact_in_timed / args.steps,
                       "host_syncs_note": "measured: TilePipeline runs of the timed region that read sizes back (capacity buckets seeded "
                                          "in the set-up pass; every timed step sees a different synthetic data set than its predecessor)",
                       "host_enqueue_ms_per_step": round(host_enqueue_ms, 3), "paste_ctas_per_sm": args.paste_ctas,
                       "per_step_ms": [round(v, 2) for v in per_step_ms], "per_rank_ms_per_step": per_rank_ms,
                       "e2e_head_probabilities": "fp16 (AMP head output, the reference's default: inference.py:1392-1396), widened exactly in K1",
                       "l2": "per step each rank writes >= 16 GB of frames and re-reads GBs of inputs: far larger than the 126 MB L2",
                       "um_pix": UM_PIX, "dedup_iou": DEDUP_IOU, "rules": "polyhipes_tommy"},
            "mask_mpix_per_sec": value * H * W / 1e6,
            "clocks": _clock_summary(clk_path, local),
            "e2e": {"value": e2e_val, "unit": "instances/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps, "rank0_wall_ms_per_step": e2e_wall, "host_shards_rotated": E,
                    "head_probabilities": "fp16",
                    "copies_only_ms_per_step": {"all_ranks_at_once": ms_copy_all, "one_rank_at_a_time": ms_copy_solo,
                                                "note": "the same H2D + D2H bytes from / to the same pinned buffers with no kernel in between "
                                                        "(max over ranks): the floor the host link sets for this step; when the first exceeds the second "
                                                        "the ranks are sharing PCIe uplinks / host memory bandwidth"}},
            "e2e_fp32_heads": {"value": n_e2e16_g / (ms_e2e16 * 1e-3), "unit": "instances/s", "h2d_bytes_per_step": h2d32,
                               "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e16 / args.steps, "identical_results_to_fp16": bool(same16),
                               "note": "the same step with the 28x28 probabilities transported as fp32 (a predictor run without AMP)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_paste_v2 (K1 paste+threshold+bitpack)", "achieved": k1_gbs, "peak": peak,
                         "unit": "GB/s", "frac": k1_gbs / peak, "traffic": traffic, "algorithmic_bytes": k1_bytes / len(k1_events),
                         "peak_source": peak_src, "k1_ms_per_step": k1_rank0 / len(k1_events), "k1_launches_per_step": len(res),
                         "k1_share_of_step": (k1_rank0 / len(k1_events)) / (rank0_ms / args.steps),
                         "k1_alone_ms": float(np.median(k1_alone)), "k1_alone_gbs": k1_alone_bytes / (float(np.median(k1_alone)) * 1e-3) / 1e9,
                         "note": "achieved = K1 algorithmic bytes of rank 0 / its CUDA-event time on the stream it is launched on, measured in "
                                 "this run over an eager pass of the same rotating shards (one launch per step, nothing overlaps it; the "
                                 "timed steps replay a CUDA graph, where no event fits around one kernel node); traffic = dram__bytes_read+write of the same "
                                 "kernel from profiles/k1_dram_traffic.json (one ncu --set full capture), scaled to this step's instances",
                         "path_achieved_gbs": path_bytes / (rank0_ms / args.steps * 1e-3) / 1e9,
                         "path_frac": path_bytes / (rank0_ms / args.steps * 1e-3) / 1e9 / peak},
            "roofline_crops_only": {"note": "the same step with frames=None: K1 writes only the bbox crops the later kernels read (the "
                                            "full-frame bit masks of the headline step are the drop-in equivalent of Detectron2's N x H x W "
                                            "pred_masks and are not consumed by the path itself)",
                                    "value": n_c_g / (ms_crops * args.steps * 1e-3), "unit": "instances/s", "ms_per_step": ms_crops,
                                    "k1_ms_per_step": k1c_ms, "k1_algorithmic_bytes": crops_bytes,
                                    "k1_achieved_gbs": crops_bytes / (k1c_ms * 1e-3) / 1e9, "k1_frac_of_hbm_peak": crops_bytes / (k1c_ms * 1e-3) / 1e9 / peak},
        }
        if want_cpu:
            ntl = args.ref_tiles if args.ref_tiles > 0 else 2 * arm.procs
            sample = list(range(min(ntl, len(last["tiles"]))))
            for lg in legs.values():          # the flow legs share the worker pool: let them finish before the timed map
                lg.wait()
            # the sampled tiles are the first tiles of shard variant 0; parity against the GPU result of that shard
            dt, cres = arm.run([shards[0]["tiles"][k] for k in sample])
            inst = sum(r[1] for r in cres)
            g_res = pipe.run(d0["probs"], d0["boxes"], d0["scores"], d0["classes"], d0["offs"])
            torch.cuda.synchronize()
            if pipe.aborted():
                g_res = pipe.run(d0["probs"], d0["boxes"], d0["scores"], d0["classes"], d0["offs"])
            first = g_res[0]
            first["meas"].finalize()
            kl = first["kept"].to_lists(); rows_h = first["meas"].rows_to_host()
            ok = True
            for (tt, n_t, final, vals, _) in cres:
                g = shards[0]["tiles"].index(tt)
                got = [k - int(d0["offs"][g]) for k in kl[g]]
                if got != final:
                    ok = False
                    continue
                gv = [r[:12] for _, rr in rows_h[g] for r in rr if r[15] == 1.0]
                if len(gv) != len(vals) or not all(np.allclose(a, np.array(b), rtol=1e-5, atol=0) for a, b in zip(gv, vals)):
                    ok = False
            kept_inst = sum(len(r[2]) for r in cres)
            ovh = arm.as_written()
            line["cpu_baseline"] = {"value": inst / dt, "unit": "instances/s", "cores": arm.procs, "kind": "port",
                                    "sample": f"{len(sample)} of {args.tiles} tiles ({inst} instances) on {arm.procs} single-threaded worker "
                                              f"processes, {dt:.1f} s wall (pool, imports and one warm-up tile per worker outside the timed "
                                              "region), compute only (no per-instance JPEG dump / gc.collect)",
                                    "mean_tile_compute_s": float(np.mean([r[4] for r in cres])),
                                    "single_process_value": inst / float(sum(r[4] for r in cres)),
                                    "as_written_value": inst / (dt + ovh * kept_inst / arm.procs),
                                    "as_written_note": f"compute + {ovh * 1e3:.1f} ms per measured instance for the reference's 3-channel JPEG dump "
                                                       "(inference.py:1153-1162) and per-instance gc.collect() (:1253), measured on 8 instances "
                                                       "with a tile's masks alive and extrapolated",
                                    "parity_vs_gpu_on_sample": bool(ok)}
        for f in flows:
            import bench_flows
            line[f] = bench_flows.run_workload(f, dev, args.steps, args.warmup, leg=legs[f].get() if f in legs else None)
        if flows and not args.flows_only:
            line["scalebar"] = bench_flows.run_scalebar_leg(dev, args.steps, args.warmup)
        print(json.dumps(line))
    if arm is not None:
        arm.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
