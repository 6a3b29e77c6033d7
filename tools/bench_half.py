"""fp32 vs fp16 vs bf16 predictions on bench.py's workload (B = 32, 640x640, G3 predictions, threshold 0.01, top-k 5000,
NMS 0.3 -> 750), one JSON line on stdout.

    python tools/bench_half.py [--reps 3] [--iters 40] [--steps 200]

Per dtype, alternating fp32 / fp16 / bf16 for --reps repetitions:
  postprocess  CUDA events around --iters replays of a CUDA graph that holds one dan_postprocess_batch_typed launch per
               input set; the sets (device-resident logits + offsets) together exceed the 126 MB L2 in every dtype.
  e2e          HotPath.step fed from pinned host memory as in bench.py's `e2e` leg: GT and logits copied in, the box offsets
               left in pinned host memory (rows of passing anchors read in place), the detection slab copied out; copy-in,
               compute and copy-out on three streams, inputs prefetched 3 steps ahead.  One compute stream (bench.py
               runs several), so the rate is below bench.py's.
Every half run's slabs are checked bit for bit against the fp32 run on the widened (`.float()`) half inputs.  The card's
name, power limit and max SM clock are read in the same run (nvidia-smi, read-only query)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dan_b200 import _lib, functional as F, pipeline, synthetic  # noqa: E402
from dan_b200.utility import anchor_manipulator as am  # noqa: E402

B, IMAGE, PS = 32, (640, 640), [0.1, 0.1, 0.2, 0.2]
DTYPES = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--sets", type=int, default=12)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    _lib.lib()
    dev = torch.device("cuda", 0)
    gpu = card()
    enc = am.AnchorEncoder(0.4, 0.4, PS)
    a_train = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd", IMAGE))
    a_eval = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd", IMAGE, border=0.))
    N = a_eval[0].numel()
    enc_params = F.encode_params(0.4, 0.4, PS, match_mining=True, pyramid=enc.pyramid)
    pp = F.postprocess_params(2, IMAGE, 0.01, 0, 5000, 750, 0.3, prior_scaling=PS)
    an = np.stack([a.cpu().numpy() for a in a_eval[:4]], -1)
    gts = [synthetic.gen_faces(i, 50) for i in range(B)]
    preds = [synthetic.gen_predictions(i, an, max_faces=300) for i in range(B)]
    R = args.sets
    host = []                                  # per set: gt, offs and the fp32 predictions (pinned)
    for r in range(R):
        order = [(i + r) % B for i in range(B)]
        cat, offs = synthetic.to_csr([gts[i] for i in order])
        host.append({"gt": torch.from_numpy(cat).pin_memory(), "offs": torch.from_numpy(offs).pin_memory(),
                     "cls": torch.from_numpy(np.stack([preds[i][0] for i in order])).pin_memory(),
                     "loc": torch.from_numpy(np.stack([preds[i][1] for i in order])).pin_memory()})
    dev_in = {}
    for name, dt in DTYPES.items():
        dev_in[name] = []
        for h in host:
            d = {"gt": h["gt"].to(dev), "offs": h["offs"].to(dev), "cls": h["cls"].to(dev).to(dt), "loc": h["loc"].to(dev).to(dt)}
            d["cls_host"] = d["cls"].cpu().pin_memory()
            d["loc_host"] = d["loc"].cpu().pin_memory()
            dev_in[name].append(d)
    hps = [pipeline.HotPath(a_train[:4], a_train[4], enc_params, pp, anchors_eval=a_eval[:4]) for _ in range(R)]
    ws = _lib.Workspace()
    outs = [F.postprocess_batch(pp, dev_in["fp32"][r]["cls"], loc_pred=dev_in["fp32"][r]["loc"], anchors=a_eval[:4], workspace=ws)
            for r in range(R)]

    # references: the fp32 path on the widened half inputs
    ref_pp, ref_slab = {}, {}
    for name in ("fp16", "bf16"):
        ref_pp[name], ref_slab[name] = [], []
        for r, d in enumerate(dev_in[name]):
            det = F.postprocess_batch(pp, d["cls"].float(), loc_pred=d["loc"].float(), anchors=a_eval[:4], workspace=ws)
            ref_pp[name].append(torch.cat([det.boxes.flatten(), det.scores.flatten()]).view(torch.int32).clone())
            hps[r].step(d["gt"], d["offs"], d["cls"].float(), d["loc"].float())
            ref_slab[name].append(hps[r]._slab.buf.view(torch.int32).clone())
    torch.cuda.synchronize()

    def capture(fn):
        fn()                                      # warm-up outside the graph (kernel attributes, workspace size)
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        return g

    pp_graph, step_graphs = {}, {}
    for name in DTYPES:
        def all_sets(name=name):
            for r, d in enumerate(dev_in[name]):
                F.postprocess_batch(pp, d["cls"], loc_pred=d["loc"], anchors=a_eval[:4], workspace=ws, out=tuple(outs[r]))
        pp_graph[name] = capture(all_sets)
        step_graphs[name] = [capture(lambda r=r, d=d: hps[r].step(d["gt"], d["offs"], d["cls"], d["loc_host"]))
                             for r, d in enumerate(dev_in[name])]

    def check_pp(name):
        if name in ref_pp:
            for r in range(R):
                got = torch.cat([outs[r].boxes.flatten(), outs[r].scores.flatten()]).view(torch.int32)
                if not torch.equal(got, ref_pp[name][r]):
                    raise RuntimeError("%s postprocess set %d differs from fp32 on the widened inputs" % (name, r))

    def check_slabs(name):
        if name in ref_slab:
            for r in range(R):
                if not torch.equal(hps[r]._slab.buf.view(torch.int32), ref_slab[name][r]):
                    raise RuntimeError("%s e2e set %d: slab differs from fp32 on the widened inputs" % (name, r))

    def time_pp(name):
        g = pp_graph[name]
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        check_pp(name)
        return e0.elapsed_time(e1) / (args.iters * R)

    slab_words = hps[0]._slab.buf.numel()
    NB, PREFETCH = 4, 3
    h_out = [torch.empty(slab_words, dtype=torch.float32).pin_memory() for _ in range(NB)]
    main_s = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    ev_in = [torch.cuda.Event() for _ in range(R)]
    ev_done = [torch.cuda.Event() for _ in range(R)]
    ev_out = [torch.cuda.Event() for _ in range(NB)]

    def e2e_run(name, n_steps):
        sets = dev_in[name]

        def copy_in(k):
            d = sets[k % R]
            with torch.cuda.stream(s_in):
                s_in.wait_event(ev_done[k % R])
                d["gt"].copy_(host[k % R]["gt"], non_blocking=True)
                d["offs"].copy_(host[k % R]["offs"], non_blocking=True)
                d["cls"].copy_(d["cls_host"], non_blocking=True)
                ev_in[k % R].record(s_in)
        for r in range(R):
            ev_done[r].record(main_s)
        for k in range(min(PREFETCH, n_steps)):
            copy_in(k)
        for k in range(n_steps):
            if k + PREFETCH < n_steps:
                copy_in(k + PREFETCH)
            main_s.wait_event(ev_in[k % R])
            step_graphs[name][k % R].replay()
            ev_done[k % R].record(main_s)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_done[k % R])
                ev_out[k % NB].synchronize()
                h_out[k % NB].copy_(hps[k % R]._slab.buf, non_blocking=True)
                ev_out[k % NB].record(s_out)
            if k >= NB - 1:
                ev_out[(k - (NB - 1)) % NB].synchronize()
        for ev in ev_out:
            ev.synchronize()
        torch.cuda.synchronize()

    def time_e2e(name):
        e2e_run(name, 2 * R)
        t0 = time.perf_counter()
        e2e_run(name, args.steps)
        dt = time.perf_counter() - t0
        check_slabs(name)
        return B * args.steps / dt

    res = {name: {"pp_ms": [], "e2e": []} for name in DTYPES}
    for _ in range(args.reps):
        for name in DTYPES:
            res[name]["pp_ms"].append(time_pp(name))
            res[name]["e2e"].append(time_e2e(name))
    thr = float(pp.select_threshold)
    out = {"card": gpu, "workload": "B=%d, %dx%d, N=%d, G3, threshold 0.01, top-k 5000, NMS 0.3 -> 750" % (B, IMAGE[0], IMAGE[1], N),
           "sets": R, "reps": args.reps, "pp_iters": args.iters, "e2e_steps": args.steps,
           "verified": "fp16 / bf16 outputs and slabs of every set bit-identical to fp32 on the widened inputs"}
    for name, dt in DTYPES.items():
        esz = torch.empty(0, dtype=dt).element_size()
        pp_ms = res[name]["pp_ms"]
        # rows of anchors whose (widened) score passes the threshold: the ones the kernels read in place
        rows = float(np.mean([int((torch.softmax(d["cls"].float(), -1)[..., 1] > thr).sum()) for d in dev_in[name]]))
        h2d_copied = sum(int(host[0][k].numel() * host[0][k].element_size()) for k in ("gt", "offs")) + B * N * 2 * esz
        out[name] = {
            "postprocess_ms_per_batch": [round(v, 5) for v in pp_ms],
            "postprocess_img_per_s": [round(B / (v * 1e-3)) for v in pp_ms],
            "e2e_img_per_s": [round(v) for v in res[name]["e2e"]],
            "h2d_copied_bytes_per_step": h2d_copied,
            "h2d_rows_read_in_place_per_step": rows,
            "h2d_bytes_per_step": int(h2d_copied + 4 * esz * rows),
            "device_input_mb_all_sets": round(R * B * N * 6 * esz / 1e6, 1),
        }
    print(json.dumps(out))


if __name__ == "__main__":
    main()
