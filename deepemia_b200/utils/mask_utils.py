"""Mirror of the reference's src/utils/mask_utils.py (functions on the hot path), computing in libemia.so."""
import numpy as np
import torch

from .. import engine
from . import _bridge

MIN_CRYSTAL_SIZE = 2      # DefaultThresholds.MIN_CRYSTAL_SIZE (src/utils/constants.py) — only used by the column gate (Q5)


def rle_encoding(x):
    """rle_encoding (src/utils/mask_utils.py:17-35): column-major, 1-indexed [start, length, start, length, ...]."""
    iset = _bridge.upload([np.asarray(x) == 1])
    _, runs = engine.rle_encode(iset)
    return [int(v) for v in runs.cpu().numpy().reshape(-1)]


def rle_decoding(rle, shape):
    """Companion of rle_encoding, not a function of the reference (which only writes the format): [start, length, ...] (a list of
    ints or the space-separated EncodedPixels string) -> H x W uint8 0/1 mask.  Raises EmiaError on a malformed run list."""
    H, W = (int(s) for s in shape[:2])
    vals = np.asarray([int(v) for v in rle.split()] if isinstance(rle, str) else list(rle), np.int64)
    if vals.size % 2:
        raise engine._lib.EmiaError(f"rle_decoding: odd number of values ({vals.size})")
    dev = engine._need_cuda(None)
    run_off = torch.tensor([0, vals.size // 2], dtype=torch.int64, device=dev)
    runs = torch.as_tensor(vals.reshape(-1, 2), device=dev).contiguous()
    return engine.unpack_masks(engine.rle_decode(run_off, runs, H, W))[0].cpu().numpy()


def postprocess_masks(ori_mask, ori_score, image, min_crys_size=None):
    """postprocess_masks (src/utils/mask_utils.py:38-84): column gate (Q5), fill holes, closing with the 3x3 cross, first-come
    overlap removal, masks with more than one component zeroed but kept (Q6).  Returns a list of uint8 H x W masks."""
    if min_crys_size is None:
        min_crys_size = MIN_CRYSTAL_SIZE
    if len(ori_mask) == 0 or np.asarray(ori_score).all() < 0.5:
        return []
    iset = _bridge.upload(ori_mask)
    out, gated = engine.postprocess_masks(iset, _bridge.one_group(iset.n, iset.device), min_crys_size)
    keep = gated.to_lists()[0]
    return _bridge.download(out, keep, np.uint8)
