"""bench.py --dump-outputs: the files hold exactly what the fused path computes for the last timed step's shard, and --steps
sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from deepemia_b200 import engine, synthetic as syn  # noqa: E402

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_last_steps_results(cuda_device, tmp_path):
    tiles, shards, steps, warmup = 16, 2, 3, 1
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--tiles", str(tiles), "--shards", str(shards), "--steps", str(steps),
           "--warmup", str(warmup), "--arena-gb", "1", "--device-pass-only", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert len(json.loads(r.stdout.strip().splitlines()[-1])["per_step_ms"]) == steps
    d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= 64 << 20

    # the same shard through the fused path directly
    _, offs, (proto_id, boxes, scores, classes) = bench.shard(0, 1, tiles, (warmup + steps - 1) % shards)
    protos = torch.as_tensor(bench._prototypes(), device=cuda_device)
    t = [protos[torch.as_tensor(proto_id, device=cuda_device)].contiguous()] + \
        [torch.as_tensor(a, device=cuda_device) for a in (boxes, scores, classes)]
    iset, kept, meas = engine.run_tiles(*t, offs, bench.H, bench.W, um_pix=bench.UM_PIX, rules=syn.POLYHIPES_RULES,
                                        dedup_iou=bench.DEDUP_IOU)
    kl = kept.to_lists()
    n = int(offs[-1])
    for grp, size in (("tile", tiles), ("kept", sum(map(len, kl))), ("instance", n), ("record", meas.n_records)):
        assert np.array_equal(d[f"{grp}_rows"], np.arange(size)), grp        # small enough to be dumped whole
    assert np.array_equal(d["kept_len"], [len(l) for l in kl])
    assert np.array_equal(d["kept_idx"], np.concatenate(kl))
    assert np.array_equal(d["bbox"], iset.bbox.cpu().numpy()) and np.array_equal(d["area"], iset.area.cpu().numpy())
    assert np.array_equal(d["records"], meas.records.cpu().numpy())
    assert np.array_equal(d["record_inst"], meas.rec_inst.cpu().numpy())
    sel = d["mask_rows"].astype(np.int64)
    assert len(sel) == bench.DUMP_MASKS and len(np.unique(sel)) == len(sel) and sel.max() < n
    full = engine.unpack_masks(iset, sel).cpu().numpy()
    P = bench.DUMP_PATCH
    for k, (y, x) in enumerate(d["mask_origin"].astype(np.int64)):
        assert np.array_equal(d["mask_patches"][k], full[k, y:y + P, x:x + P]), k
    assert d["mask_patches"].any()
