#!/usr/bin/env python
"""Warp timeline of enc_pass1_fused_kernel on the benchmark's encode (batch 32, 640^2, mining, layout hint).

Uses a copy of the library built with -DDAN_PASS1_TIMELINE (lane 0 of every warp records the global timer at its start
and end):  bash tools/variant.sh timeline -DDAN_PASS1_TIMELINE;  python tools/pass1_timeline.py build/variants/libdan_timeline.so
Prints, per pyramid level, the warps' durations and when the last of them ended, and the kernel's span."""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["DAN_B200_LIB"] = sys.argv[1]
import torch  # noqa: E402
from dan_b200 import _lib, functional as F, synthetic  # noqa: E402
from dan_b200.utility import anchor_manipulator as am  # noqa: E402


def main():
    L = _lib.lib()
    L.dan_debug_pass1_timeline.argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_int32]
    dev = torch.device("cuda", 0)
    ps = [0.1, 0.1, 0.2, 0.2]
    enc = am.AnchorEncoder(0.4, 0.4, ps)
    cfg = synthetic.pyramid_config("s3fd", (640, 640))
    a = synthetic.build_anchors(enc, cfg)
    params = F.encode_params(0.4, 0.4, ps, match_mining=True, pyramid=enc.pyramid)
    cat, offs = synthetic.to_csr([synthetic.gen_faces(i, 50) for i in range(32)])
    gt, off = torch.from_numpy(cat).to(dev), torch.from_numpy(offs).to(dev)
    n = a[0].numel()
    starts = np.cumsum([0] + [h * w for h, w in cfg["layer_shapes"]])
    nchunks = (n + 127) // 128
    for _ in range(5):
        _, ms = F.encode_batch(params, *a[:4], a[4], gt, off, profile=True)
    warps = 65536
    buf = (ctypes.c_ulonglong * (3 * warps))()
    _lib.check(L.dan_debug_pass1_timeline(buf, warps))
    t = np.frombuffer(buf, dtype=np.uint64).reshape(-1, 3).astype(np.float64)
    used = t[:, 1] > 0
    # (entries of an earlier, larger launch may remain beyond this one's warps: keep the last launch's time window)
    last = t[used, 1].max()
    live = used & (t[:, 0] >= last - 1e6)
    t = t[live]
    t0 = t[:, 0].min()
    imgs = (t[:, 2].astype(np.uint64) & 0xffffffff).astype(int)
    from_end = (t[:, 2].astype(np.uint64) >> 32).astype(int)
    first_anchor = (nchunks - 1 - from_end) * 128
    level = np.searchsorted(starts, first_anchor, side="right") - 1
    dur = (t[:, 1] - t[:, 0]) / 1e3
    print("pass 1 by CUDA events (last rep): %.1f us; warps recorded %d; span of the warp timeline %.1f us"
          % (1e3 * ms[0], len(t), (t[:, 1].max() - t0) / 1e3))
    print("%-6s %6s %6s %10s %10s %12s %12s" % ("level", "warps", "imgs", "mean us", "max us", "last start", "last end"))
    for lv in range(len(starts) - 1):
        s = level == lv
        if s.any():
            print("%-6d %6d %6.1f %10.2f %10.2f %12.2f %12.2f" % (lv, s.sum(), imgs[s].mean(), dur[s].mean(), dur[s].max(),
                                                               (t[s, 0].max() - t0) / 1e3, (t[s, 1].max() - t0) / 1e3))
    q = np.percentile((t[:, 1] - t0) / 1e3, [50, 90, 99, 100])
    print("warp end times (us after the first start): p50 %.1f p90 %.1f p99 %.1f max %.1f" % tuple(q))


if __name__ == "__main__":
    main()
