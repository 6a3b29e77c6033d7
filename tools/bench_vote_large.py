"""bbox_vote timed on both paths: the small kernel (capacity <= 8192) and the large one (capacity > 8192), B images per
launch, one CTA each.  The workloads alternate, each repetition times every workload once in a CUDA graph with CUDA
events; the card's name, power limit and max SM clock are read in the same run (nvidia-smi, read-only query).

    python tools/bench_vote_large.py [out.jsonl] [--batch B] [--reps R]

Workloads (synthetic.gen_vote_dets(i, n, n / 56, 0.6), ragged counts):
    small_6750        the small kernel at 6 750 rows (6 passes of 1125)
    large_6750_cap8193  the same input with capacity 8193: the large kernel on the same rows
    large_11250 / large_20000 / large_70000   10 passes, about 18, about 62
The outputs of small_6750 and large_6750_cap8193 are compared bit for bit after every repetition."""
import json, os, subprocess, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dan_b200 import _lib as L, functional as F, synthetic


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def workload(B, n, cap, dev):
    dets = [synthetic.gen_vote_dets(1000 * n + i, n, max(n // 56, 1), 0.6) for i in range(B)]
    cap = max([cap] + [d.shape[0] for d in dets])
    batch = np.zeros((B, cap, 5), np.float32)
    for i, d in enumerate(dets):
        batch[i, :d.shape[0]] = d
    x = torch.from_numpy(batch).to(dev)
    c = torch.tensor([d.shape[0] for d in dets], dtype=torch.int32, device=dev)
    ws = L.Workspace()
    fn = lambda: F.bbox_vote_batch(x, c, 0.3, 750, details=True, workspace=ws)
    fn()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            out = fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    # the graph replays on x, c and ws: they live as long as it does
    return dict(graph=g, out=out, x=x, c=c, ws=ws, rows=int(c.float().mean()), cap=cap)


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
    args = sys.argv[1:]
    path = args[0] if args and not args[0].startswith("--") else None
    B = int(args[args.index("--batch") + 1]) if "--batch" in args else 32
    reps = int(args[args.index("--reps") + 1]) if "--reps" in args else 3
    dev = torch.device("cuda", 0)
    who = card()
    spec = [("small_6750", 6750, 0), ("large_6750_cap8193", 6750, 8193), ("large_11250", 11250, 0),
            ("large_20000", 20000, 0), ("large_70000", 70000, 0)]
    W = {name: workload(B, n, cap, dev) for name, n, cap in spec}
    times = {name: [] for name, _, _ in spec}
    for _ in range(reps):
        for name, _, _ in spec:
            ms = time_graph(W[name]["graph"], 3)
            times[name].append(round(time_graph(W[name]["graph"], max(3, min(50, int(200 / max(ms, 1e-3))))), 4))
        a, b = W["small_6750"]["out"], W["large_6750_cap8193"]["out"]
        w = a[2].shape[1]
        same = (torch.equal(a[0].view(torch.int32), b[0].view(torch.int32)) and torch.equal(a[1], b[1]) and
                torch.equal(a[2], b[2][:, :w]) and torch.equal(a[3], b[3][:, :w]))
        assert same, "small and large paths differ on the same input"
    lines = []
    for name, n, _ in spec:
        w = W[name]
        rec = {"card": who, "workload": name, "B": B, "rows_mean": w["rows"], "capacity": w["cap"],
               "path": "small" if w["cap"] <= 8192 else "large", "ms_per_batch": times[name],
               "groups_mean": round(float(w["out"][1].float().mean()), 1)}
        if name.startswith("large_6750"):
            rec["verified"] = "out, count, order and assign bit-identical to small_6750 after every repetition"
        lines.append(json.dumps(rec))
    print("\n".join(lines))
    if path:
        with open(path, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
