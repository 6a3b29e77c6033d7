"""detect_face through dan_detect_face_batch_top: the old entry point against the new one at top 1125 (the same kernels),
and the select path for k > 8192 at larger tops.  One JSON line per configuration.

    python tools/bench_detect_face_top.py [--reps 3] [--out profiles/r07_detect_face_top.jsonl]

Configurations: S3FD anchors (border 0) at 1024^2 (N = 87 360) and 1600^2 (N = 213 294); B = 32 (four distinct images of
synthetic.gen_predictions, 300 faces at most, repeated over the batch); fp32 and bf16 predictions; shrink 1.
  top 1125           old  dan_detect_face_batch      new  dan_detect_face_batch_top (functional.detect_face_batch);
                     old and new alternate, and after every timed pair their rows and indices are compared bit for bit
  top 9000, 16384, 98302 (k = min(N - 1, top))       new only (the old entry point refuses top > 8192); after every
                     repetition the rows and indices are compared bit for bit with an eager call made before the timing
Each call is captured in a CUDA graph and timed with CUDA events around --iters replays.  The inputs of B = 32 exceed the
126 MB L2 at 1600^2 (bf16: 82 MB of logits and offsets) and stay partly in it at 1024^2.  The card's name, power limit
and max SM clock are read in the same run (nvidia-smi, read-only query)."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dan_b200 import _lib as L, functional as F, synthetic  # noqa: E402
from dan_b200.utility import anchor_manipulator as am  # noqa: E402

PS = [0.1, 0.1, 0.2, 0.2]
SIZES = [(1024, 1024), (1600, 1600)]
B = 32
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}
DISTINCT = 4
TOP_SMALL = 1125
TOPS_LARGE = [9000, 16384, 98302]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def capture(fn):
    fn()                                          # warm-up outside the graph (kernel attributes, workspace sizes)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            out = fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    return g, out


def time_graph(g, iters):
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def old_call(cls, loc, anchors, top, ws):
    """dan_detect_face_batch, the entry point limited to top <= 8192"""
    n = cls.shape[1]
    det = torch.empty((B, top, 5), dtype=torch.float32, device=cls.device)
    idx = torch.empty((B, top), dtype=torch.int32, device=cls.device)
    nb = L.lib().dan_detect_face_batch_workspace_bytes(n, B)
    ps = (ctypes.c_float * 4)(*PS)
    L.check(L.lib().dan_detect_face_batch(L.pred_dtype(cls, "cls_pred"), L.dev_ptr(cls, cls.dtype), L.dev_ptr(loc, cls.dtype),
                                          *[L.dev_ptr(a) for a in anchors], n, B, ps, 1.0, top, L.dev_ptr(det), L.dev_ptr(idx),
                                          L.dev_ptr(ws), nb, L.stream_ptr()))
    return det, idx


def same(a, b):
    return torch.equal(a[0].view(torch.int32), b[0].view(torch.int32)) and torch.equal(a[1], b[1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "r07_detect_face_top.jsonl"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    L.lib()
    dev = torch.device("cuda", 0)
    gpu = card()
    enc = am.AnchorEncoder(None, None, PS)
    lines = []

    def emit(line):
        print(json.dumps(line), flush=True)
        lines.append(line)

    for size in SIZES:
        a = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd", size, border=0.))[:4]
        n = a[0].numel()
        an = np.stack([v.cpu().numpy() for v in a], -1)
        preds = [synthetic.gen_predictions(i, an, size=size, max_faces=300) for i in range(DISTINCT)]
        cls32 = torch.from_numpy(np.stack([preds[i % DISTINCT][0] for i in range(B)])).to(dev)
        loc32 = torch.from_numpy(np.stack([preds[i % DISTINCT][1] for i in range(B)])).to(dev)
        for name, dt in DTYPES.items():
            cls, loc = cls32.to(dt).contiguous(), loc32.to(dt).contiguous()
            ws_old = torch.empty(L.lib().dan_detect_face_batch_workspace_bytes(n, B), dtype=torch.uint8, device=dev)
            ws_new = L.Workspace()
            g_old, out_old = capture(lambda: old_call(cls, loc, a, TOP_SMALL, ws_old))
            g_new, out_new = capture(lambda: F.detect_face_batch(cls, loc, a, 1.0, TOP_SMALL, PS, workspace=ws_new)[:2])
            t_old, t_new = [], []
            for _ in range(args.reps):
                t_old.append(time_graph(g_old, 50))
                t_new.append(time_graph(g_new, 50))
                if not same(out_old, out_new):
                    raise RuntimeError("%s %s top %d: the new entry point's rows differ from the old one's" % (size, name, TOP_SMALL))
            emit({"card": gpu, "image": "%dx%d" % size, "N": n, "B": B, "dtype": name, "top": TOP_SMALL, "k": TOP_SMALL,
                  "path": "small", "iters": 50, "old_ms": [round(v, 4) for v in t_old], "new_ms": [round(v, 4) for v in t_new],
                  "new_over_old_median": round(float(np.median(t_new) / np.median(t_old)), 3),
                  "verified": "rows and indices of old and new bit-identical after every timed pair"})
            del g_old, g_new
            for top in TOPS_LARGE:
                k = min(n - 1, top)
                ref = [t.clone() for t in F.detect_face_batch(cls, loc, a, 1.0, top, PS)[:2]]
                ws = L.Workspace()
                g, out = capture(lambda: F.detect_face_batch(cls, loc, a, 1.0, top, PS, workspace=ws)[:2])
                t = []
                for _ in range(args.reps):
                    t.append(time_graph(g, 10))
                    if not same(out, ref):
                        raise RuntimeError("%s %s top %d: graph replay differs from the eager call" % (size, name, top))
                emit({"card": gpu, "image": "%dx%d" % size, "N": n, "B": B, "dtype": name, "top": top, "k": k,
                      "path": "large", "iters": 10, "new_ms": [round(v, 4) for v in t],
                      "workspace_mb": round(L.lib().dan_detect_face_top_workspace_bytes(n, B, top) / 2**20, 1),
                      "verified": "rows and indices bit-identical to an eager call after every repetition"})
                del g
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
