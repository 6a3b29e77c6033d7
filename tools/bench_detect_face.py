"""The per-pass detect_face chain of the evaluation scripts, old against new, one JSON line per configuration.

    python tools/bench_detect_face.py [--reps 3] [--out profiles/r05_detect_face_bench.jsonl]

  old  functional.softmax (fp32 logits: a bf16 head's logits are widened first) -> functional.decode_batch ->
       B x functional.detect_face_select, one image per call
  new  functional.detect_face_batch, one call for the batch (logits and offsets in their own dtype)

Configurations: S3FD anchors (border 0) at 640^2, 1024^2 and 1600^2; B = 1 and 32; fp32 and bf16 predictions (G3:
synthetic.gen_predictions, 300 faces at most; four distinct images repeated over the batch); top = 1125, shrink 1.
Each chain is captured in a CUDA graph (no host work and no host read inside the timed window) and timed with CUDA
events around --iters replays; old and new alternate, --reps times each.  After every timed pair the rows and indices
of the new call are compared bit for bit with the old chain's.  B = 1 inputs stay in the 126 MB L2 between replays;
B = 32 inputs at 1024^2 and 1600^2 exceed it.  The card's name, power limit and max SM clock are read in the same run
(nvidia-smi, read-only query)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dan_b200 import _lib, functional as F, synthetic  # noqa: E402
from dan_b200.utility import anchor_manipulator as am  # noqa: E402

PS = [0.1, 0.1, 0.2, 0.2]
TOP = 1125
SIZES = [(640, 640), (1024, 1024), (1600, 1600)]
BATCHES = [1, 32]
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}
DISTINCT = 4


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "r05_detect_face_bench.jsonl"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    _lib.lib()
    dev = torch.device("cuda", 0)
    gpu = card()
    enc = am.AnchorEncoder(None, None, PS)
    lines = []
    for size in SIZES:
        a = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd", size, border=0.))[:4]
        n = a[0].numel()
        an = np.stack([v.cpu().numpy() for v in a], -1)
        preds = [synthetic.gen_predictions(i, an, size=size, max_faces=300) for i in range(DISTINCT)]
        for B in BATCHES:
            cls32 = torch.from_numpy(np.stack([preds[i % DISTINCT][0] for i in range(B)])).to(dev)
            loc32 = torch.from_numpy(np.stack([preds[i % DISTINCT][1] for i in range(B)])).to(dev)
            for name, dt in DTYPES.items():
                cls, loc = cls32.to(dt), loc32.to(dt)
                ws = _lib.Workspace()

                def old():
                    scores = F.softmax(cls.float())[..., 1]
                    boxes = F.decode_batch(loc, *a, PS)
                    rows = [F.detect_face_select(boxes[b], scores[b], 1.0, TOP)[:2] for b in range(B)]
                    return torch.stack([r[0] for r in rows]), torch.stack([r[1] for r in rows])

                def new():
                    return F.detect_face_batch(cls, loc, a, 1.0, TOP, PS, workspace=ws)[:2]
                g_old, out_old = capture(old)
                g_new, out_new = capture(new)
                iters = 100 if B == 1 else 20
                t_old, t_new = [], []
                for _ in range(args.reps):
                    t_old.append(time_graph(g_old, iters))
                    t_new.append(time_graph(g_new, iters))
                    if not (torch.equal(out_old[0].view(torch.int32), out_new[0].view(torch.int32))
                            and torch.equal(out_old[1], out_new[1])):
                        raise RuntimeError("%s B=%d %s: rows differ from the old chain" % (size, B, name))
                line = {"card": gpu, "image": "%dx%d" % size, "N": n, "B": B, "dtype": name, "top": TOP, "iters": iters,
                        "old_ms": [round(v, 4) for v in t_old], "new_ms": [round(v, 4) for v in t_new],
                        "speedup_median": round(float(np.median(t_old) / np.median(t_new)), 2),
                        "verified": "rows and indices bit-identical to the old chain after every timed pair"}
                print(json.dumps(line), flush=True)
                lines.append(line)
                del g_old, g_new
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
