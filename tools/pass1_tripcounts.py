#!/usr/bin/env python
"""Dynamic trip counts of enc_pass1_fused_kernel on the benchmark's inputs, computed on the CPU (no GPU needed):
per pyramid level, the (warp, image) tasks of pass 1 and the (warp, GT) pairs that pass the warp-box cull test, with and
without the layout hint.  Together with the SASS of the kernel this splits the kernel's warp instructions into the fixed
cost of a task and the cost of its pairs (profiles/r03_pass1_breakdown.md).

    python tools/pass1_tripcounts.py [--batch 32]"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dan_b200 import synthetic  # noqa: E402
from oracle import reference_np as R  # noqa: E402


def warp_lanes(n, grids):
    """[nwarps, 32] anchor index of every lane (n = padding), as warp_anchor() / enc_warp_map_kernel assign them."""
    nw = (n + 31) // 32
    idx = np.arange(nw)[:, None] * 32 + np.arange(32)[None, :]
    for start, w, h in grids:
        wbeg, wcnt, tpb = start // 32, w * h // 32, w // 8
        j = np.arange(wcnt)
        base = start + (j // tpb) * 4 * w + (j % tpb) * 8
        lane = np.arange(32)
        idx[wbeg:wbeg + wcnt] = base[:, None] + (lane[None, :] >> 3) * w + (lane[None, :] & 7)
    idx[idx >= n] = n
    return idx


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    args = ap.parse_args()
    cfg = synthetic.pyramid_config("s3fd", (640, 640))
    ay0, ax0, ay1, ax1, _ = [np.asarray(v) for v in synthetic.build_anchors(R.AnchorEncoder(0.4, 0.4, [0.1, 0.1, 0.2, 0.2]), cfg)]
    n = ay0.shape[0]
    sizes = [h * w for h, w in cfg["layer_shapes"]]
    starts = np.cumsum([0] + sizes)
    grids = [(int(starts[i]), w, h) for i, (h, w) in enumerate(cfg["layer_shapes"])
             if starts[i] % 32 == 0 and w % 8 == 0 and h % 4 == 0]
    gts = [synthetic.gen_faces(i, 50) for i in range(args.batch)]
    ms = np.array([len(g) for g in gts])
    print("N = %d anchors, %d warps; batch %d: GTs per image mean %.1f (min %d, max %d), %.1f chunks of 32 per image"
          % (n, (n + 31) // 32, args.batch, ms.mean(), ms.min(), ms.max(), np.mean((ms + 31) // 32)))
    pad = lambda v, f: np.append(v, f)  # noqa: E731
    for label, gl in (("layout hint", grids), ("no hint", [])):
        lanes = warp_lanes(n, gl)
        valid = lanes < n
        y0 = np.where(valid, pad(ay0, 0)[lanes], np.inf).min(1)
        x0 = np.where(valid, pad(ax0, 0)[lanes], np.inf).min(1)
        y1 = np.where(valid, pad(ay1, 0)[lanes], -np.inf).max(1)
        x1 = np.where(valid, pad(ax1, 0)[lanes], -np.inf).max(1)
        first = lanes[:, 0]
        level = np.searchsorted(starts, first, side="right") - 1
        pairs = np.zeros(len(first))
        for g in gts:
            g = g.astype(np.float32)
            dy = np.minimum(y1[:, None], g[None, :, 2]) - np.maximum(y0[:, None], g[None, :, 0])
            dx = np.minimum(x1[:, None], g[None, :, 3]) - np.maximum(x0[:, None], g[None, :, 1])
            pairs += ((dy >= -1) & (dx >= -1)).sum(1)
        print("\n%s: %.0f (warp, GT) pairs per image, %.2f per (warp, image) task" % (label, pairs.sum() / args.batch,
                                                                                    pairs.sum() / args.batch / len(first)))
        print("%-8s %8s %7s %12s %16s" % ("level", "stride", "warps", "pairs/img", "pairs per task"))
        for lv in range(len(sizes)):
            sel = level == lv
            if sel.any():
                print("%-8d %8d %7d %12.0f %16.3f" % (lv, cfg["layer_strides"][lv], sel.sum(), pairs[sel].sum() / args.batch,
                                                     pairs[sel].mean() / args.batch))


if __name__ == "__main__":
    main()
