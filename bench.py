#!/usr/bin/env python
"""bench.py -- images/sec of the DAN anchor hot path (match + encode + decode + top-k + NMS) at 640^2.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

One "step" = one pass of the hot path over one batch of synthetic images PER GPU (weak scaling):
  training side    S3FD 640x640 pyramid (34 125 anchors), encode_anchors(match_mining=True), thresholds 0.4/0.4,
                   G1 ground truth with <= 50 faces / image                      (BASELINE.json configs[1])
  evaluation side  decode + softmax + threshold 0.01 + top-k 5000 + NMS 0.3 -> 750 on G3 predictions
                   (parse_by_class semantics, configs[3] at 640^2)
  N > 1            images are sharded per rank (configs[4]: 8 x 32 = 256 images); ONE ncclAllGather of the
                   fixed-capacity detection slabs per step, enqueued behind the NMS kernel inside the step's CUDA graph.
`value` is timed with inputs resident in HBM (CUDA events, the step replayed as a CUDA graph, rotating input/output
buffer sets larger than L2); `e2e` is timed through the public python API with HOST (pinned) buffers, H2D and D2H
copies inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/sec anchor match+encode+decode+NMS @640^2"
UNIT = "images/s"
IMAGE = (640, 640)
PP = (0.01, 0, 5000, 750, 0.3)      # select_threshold, min_size, keep_topk, nms_topk, nms_threshold
CPU_CFG = dict(kind="s3fd", size=IMAGE, pos=0.4, ign=0.4, mining=True, max_gt=50, max_faces=300, pp=PP)
# kernels of one step (the memset node aside): enc_pass1, enc_pass2_find, enc_pass2_apply, enc_pass3, nms_greedy
# (+ the NCCL kernel at N > 1)
KERNELS_PER_STEP = 5
DUMP_LIMIT_BYTES = 64 << 20


def workload_config(batch, n_gpus):
    """The `config` object: identical in both arms (the driver compares them)."""
    return {"workload": "S3FD 640x640 (34125 anchors): mining encode of <=50 GT faces/image + decode/threshold 0.01/"
                        "top-k 5000/NMS 0.3->750 of G3 predictions, batch %d per GPU" % batch,
            "images_per_gpu": batch, "global_batch": batch * n_gpus, "num_anchors": 34125,
            "parallelism": "per-image sharding, dp%d" % n_gpus}


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline (the ONLY place bench.py touches oracle/)
# --------------------------------------------------------------------------------------------------
def cpu_measure(images, steps, warmup, procs=None):
    """The reference's CPU path (oracle/cpu_path.py) on all host cores: `steps` timed passes over `images` images."""
    from oracle import cpu_path, native
    native.build()
    procs = procs or os.cpu_count() or 1
    idx = list(range(images))
    cpu_path.generate_inputs(CPU_CFG, idx, procs)
    pool = cpu_path.CpuPool(CPU_CFG, procs)
    for _ in range(warmup):
        pool.run(idx)
    walls, busy = [], 0.0
    for _ in range(steps):
        w, n, b = pool.run(idx)
        walls.append(w)
        busy += b
    pool.close()
    total = sum(walls)
    lib = os.path.join("oracle", "_ref", "libsmm_ref.so") if pool.impl == "reference" else os.path.join("oracle", "liboracle_native.so")
    return {"value": images * steps / total, "ms_per_step": 1e3 * total / steps, "cores": procs, "impl": pool.impl,
            "images": images, "core_seconds_per_image": busy / (images * steps), "matcher_library": lib}


def cpu_kind(r):
    """"reference": the matcher is the reference's own functor compiled from /root/reference (oracle/_ref); the TF graph
    ops around it are restated in numpy either way (TensorFlow 1.8 is not installable)."""
    return "reference" if r["impl"] == "reference" else "port"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    procs = os.cpu_count() or 1
    images = min(args.batch, max(2 * procs, 8))
    r = cpu_measure(images, args.steps, max(args.warmup, 1), procs)
    sample = ("%d images/step x %d steps, %d worker processes (one image per task); numpy fp32 restatement of the TF graph ops"
              " + %s SmallMiningMatch (%s, loaded by the worker processes) + restated tf.nn.top_k / non_max_suppression "
              "(TF 1.8 is not installable)"
              % (images, args.steps, procs, "the reference's own compiled" if r["impl"] == "reference" else "ported", r["matcher_library"]))
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": max(args.warmup, 1), "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.batch, args.gpus),
            "run": {"cpu_sample_images_per_step": images, "native_so_loaded": [r["matcher_library"]]},
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": procs, "kind": cpu_kind(r), "sample": sample},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.path):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_mhz_max_seen": max(sm), "sm_max_mhz": max(smax), "samples": len(sm),
                "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------------
# the CUDA arm
# --------------------------------------------------------------------------------------------------
def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def fp32_peak():
    """Non-FMA FP32 issue rate (instructions/s): calibrated on the box with tools/fp32_peak.cu, else 148 x 128 x 1.965 GHz."""
    try:
        return (1e12 * json.load(open(os.path.join(ROOT, "profiles", "r01_fp32_peak.json")))["fp32_nonfma_tinstr_s"],
                "measured (profiles/r01_fp32_peak.json, tools/fp32_peak.cu)")
    except Exception:
        return 37.2e12, "nominal 148 SM x 128 lanes x 1.965 GHz"


def ncu_traffic():
    """dram bytes/launch per kernel from the committed ncu --set full capture (profiles/), else None."""
    path = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except Exception:
            return None
    return None


def _cpulist(text):
    out = []
    for part in text.strip().split(","):
        if part:
            lo, _, hi = part.partition("-")
            out.extend(range(int(lo), int(hi or lo) + 1))
    return out


def gpu_numa_nodes(local_world):
    """NUMA node of every local GPU (sysfs, via the PCI address NVML reports); None where the platform does not say."""
    nodes = [None] * local_world
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip().isdigit()]
        for i in range(local_world):
            phys = int(visible[i]) if i < len(visible) else i
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            path = "/sys/bus/pci/devices/%s/numa_node" % bus.lower()[-12:]
            if os.path.exists(path):
                v = int(open(path).read().strip())
                nodes[i] = v if v >= 0 else None
        pynvml.nvmlShutdown()
    except Exception:
        pass
    return nodes


def pin_rank_to_cores(local_rank, local_world):
    """Give every rank of the node its own slice of the host cores BEFORE it allocates pinned memory, on the NUMA node its
    GPU hangs off when sysfs says which: the pinned buffers are then first-touched next to the GPU's PCIe root and the
    copies of the ranks do not all cross the socket interconnect or share one memory controller.
    Returns (cores given to the rank, NUMA node or None)."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
        nodes = gpu_numa_nodes(local_world)
        node = nodes[local_rank]
        mine = None
        if node is not None:
            path = "/sys/devices/system/node/node%d/cpulist" % node
            local = [c for c in _cpulist(open(path).read()) if c in allowed] if os.path.exists(path) else []
            sharers = [r for r in range(local_world) if nodes[r] == node]
            per = len(local) // max(len(sharers), 1)
            if per >= 1:
                k = sharers.index(local_rank)
                mine = local[k * per:(k + 1) * per]
        if not mine:
            node = None
            per = max(1, len(allowed) // max(local_world, 1))
            mine = allowed[local_rank * per:(local_rank + 1) * per] or allowed
        os.sched_setaffinity(0, mine)
        return len(mine), node
    except (AttributeError, OSError, ValueError):
        return None, None


def log(msg):
    """Progress on stderr (DAN_BENCH_VERBOSE=1): where a multi-rank run is, should it ever stall."""
    if os.environ.get("DAN_BENCH_VERBOSE"):
        sys.stderr.write("[bench rank %s %.1fs] %s\n" % (os.environ.get("RANK", "0"), time.time() - _T0, msg))
        sys.stderr.flush()


_T0 = time.time()


def step_outputs(hp, image_ids):
    """What HotPath.step() handed its caller in the step that last used `hp`: the encode outputs and the detections, as
    float32 host arrays (labels, counts and indices are integers below 2^24, exact in float32).  Above DUMP_LIMIT_BYTES
    a fixed, seeded sample of the images is kept; `image_id` names the synthetic image of every row."""
    import numpy as np
    import torch
    counts, scores, boxes = hp._slab.views()
    targets, labels, enc_scores, matched = hp._enc_out[:4]
    out = {"enc_targets": targets, "enc_labels": labels, "enc_scores": enc_scores, "enc_matched_gt": matched,
           "det_boxes": boxes, "det_scores": scores, "det_counts": counts, "det_anchor_index": hp._aux[0], "det_keep_pos": hp._aux[1]}
    n = len(image_ids)
    per_image = 8 + sum(4 * t[0].numel() for t in out.values())
    keep = min(n, DUMP_LIMIT_BYTES // per_image)
    rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    idx = torch.from_numpy(rows).to(boxes.device)
    res = {name: t.index_select(0, idx).float().cpu().numpy() for name, t in out.items()}
    res["image_id"] = np.asarray(image_ids, np.float64)[rows]
    return res


def run_cuda(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    B = args.batch

    # ---- CPU baseline first (rank 0, N == 1 only): needs fork, so it runs before CUDA is initialised ----------
    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        procs = os.cpu_count() or 1
        images = max(4 * procs, 32)
        r = cpu_measure(images, 5, 1, procs)
        cpu_base = {"value": r["value"], "unit": UNIT, "cores": procs, "kind": cpu_kind(r),
                    "sample": "%d images x 5 passes after 1 warm-up pass (%.0f core-seconds), %d worker processes; numpy restatement + %s "
                              "SmallMiningMatch (%s); %.1f ms per image per core"
                              % (images, r["core_seconds_per_image"] * images * 5, procs,
                                 "reference-compiled" if r["impl"] == "reference" else "ported", r["matcher_library"],
                                 1e3 * r["core_seconds_per_image"])}
    cores_per_rank, numa_node = pin_rank_to_cores(local_rank, local_world) if world > 1 else (None, None)

    import numpy as np
    import torch
    import torch.distributed as dist
    from dan_b200 import _lib, functional as F, pipeline, synthetic
    from dan_b200.utility import anchor_manipulator as am

    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback for the product path"
    _lib.lib()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    log("process group ready")
    # ---- anchors, parameters ----------------------------------------------------------------------------------
    ps = [0.1, 0.1, 0.2, 0.2]
    enc = am.AnchorEncoder(0.4, 0.4, ps)
    a_train = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd", IMAGE))
    a_eval = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd", IMAGE, border=0.))
    N = a_train[0].numel()
    # (layout hint: the 160^2 / 80^2 / 40^2 levels are one-anchor-per-cell grids; results do not depend on it)
    enc_params = F.encode_params(0.4, 0.4, ps, match_mining=True, pyramid=None if args.no_layout_hint else enc.pyramid)
    pp_params = F.postprocess_params(2, IMAGE, *PP, prior_scaling=ps)

    # ---- synthetic inputs: B distinct images per rank; buffer set r holds them rolled by r ----------------------
    an = np.stack([a.cpu().numpy() for a in a_eval[:4]], -1)
    base = rank * B
    gts = [synthetic.gen_faces(base + i, 50) for i in range(B)]
    preds = [synthetic.gen_predictions(base + i, an, max_faces=300) for i in range(B)]
    per_set = B * N * (8 + 16 + 44)          # cls + loc in, encode outputs out
    R = args.sets if args.sets > 0 else max(4, int(np.ceil(3.0 * 126e6 / per_set)))
    # `inflight` consecutive steps are in flight at a time, each on its own stream with its own workspaces (different
    # buffer sets, no shared state): the fused sort + NMS kernel and the compensation pass run one CTA per image, i.e. on
    # 32 of the 148 SMs, and their latency would otherwise leave most of the GPU idle
    L = max(1, args.inflight)
    R = (R + L - 1) // L * L                  # a set always runs on the same lane
    ws_lanes = [(_lib.Workspace(), _lib.Workspace()) for _ in range(L)]
    slab_words = pipeline.DetectionSlab.words_for(B, pp_params.num_classes - 1, pp_params.nms_topk)
    # the detection exchange (N > 1): "p2p" = the NMS kernel stores its slab rows into every rank's receive buffer over
    # NVLink (CUDA IPC) and a one-warp kernel waits for the arrival flags; "nccl" = one ncclAllGather per step, one
    # communicator per lane (collectives of one communicator must not run concurrently, the lanes do)
    peers, gathers = None, [None] * L
    gather_fallback = None
    if world > 1 and args.gather == "p2p":
        # CUDA IPC can be unavailable (some container / vGPU set-ups): every rank then falls back to the NCCL gather.  The
        # ranks agree on the outcome so that none of them is left waiting in the other path.
        try:
            peers = pipeline.PeerExchange(rank, world, dev, slab_words, num_sets=R)
            ok, why = 1, ""
        except Exception as e:      # noqa: BLE001 (reported in the JSON line)
            peers, ok, why = None, 0, "%s: %s" % (type(e).__name__, e)
        agreed = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(agreed, op=dist.ReduceOp.MIN)
        if int(agreed.item()) == 0:
            if peers is not None:
                peers.close()
                peers = None
            gather_fallback = why or "another rank could not map the peer buffers"
            log("peer exchange unavailable (%s): falling back to ncclAllGather" % gather_fallback)
    if world > 1 and peers is None:
        gathers = [pipeline.DeviceGather(rank, world, dev) for _ in range(L)]
    sets = []
    for r in range(R):
        order = [(i + r) % B for i in range(B)]
        cat, offs = synthetic.to_csr([gts[i] for i in order])
        h = {"gt": torch.from_numpy(cat).pin_memory(), "offs": torch.from_numpy(offs).pin_memory(),
             "cls": torch.from_numpy(np.stack([preds[i][0] for i in order])).pin_memory(),
             "loc": torch.from_numpy(np.stack([preds[i][1] for i in order])).pin_memory()}
        d = {k: v.to(dev) for k, v in h.items()}
        recv = None
        if peers is not None:
            recv = peers.recv(r)
        elif world > 1:
            recv = torch.zeros(world * slab_words, dtype=torch.float32, device=dev)
        hp = pipeline.HotPath(a_train[:4], a_train[4], enc_params, pp_params, anchors_eval=a_eval[:4],
                              workspaces=ws_lanes[r % L], overlap=not args.no_overlap, device_gather=gathers[r % L],
                              recv_buffer=None if peers is not None else recv, peer_exchange=peers, peer_set=r)
        sets.append({"host": h, "dev": d, "hp": hp, "recv": recv, "total_gt": int(offs[-1]), "image_id": [base + i for i in order]})
    total_gt_mean = float(np.mean([s["total_gt"] for s in sets]))

    # kernels of this library per step: enc_pass1, enc_pass2_find, enc_pass2_apply, enc_pass3, nms_greedy (+ the warp table of
    # the layout hint, + the one-warp wait of the peer exchange at N > 1; the NCCL gather's kernel is not ours)
    launches_per_step = KERNELS_PER_STEP + (1 if enc_params.num_grids > 0 else 0) + (1 if peers is not None else 0)
    log("inputs and exchange ready")
    def run_set(s, profile=False, host_loc=False):
        """host_loc: the box offsets stay in the pinned host buffer and the NMS kernel reads the rows it needs in place"""
        return s["hp"].step(s["dev"]["gt"], s["dev"]["offs"], s["dev"]["cls"], s["host" if host_loc else "dev"]["loc"], profile=profile)

    # warm-up outside graphs (sizes the workspace, sets kernel attributes, opens the NCCL channels), then capture one
    # CUDA graph per set; at N > 1 the graph contains the all-gather of the step's detection slab
    for s in sets:
        run_set(s)
    torch.cuda.synchronize()
    log("eager warm-up done")
    def capture(host_loc):
        out = []
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for s in sets:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):
                    run_set(s, host_loc=host_loc)
                out.append(g)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        return out
    graphs = [] if args.no_graph else capture(False)
    graphs_hl = []                              # captured before the end-to-end leg that uses them

    log("graphs captured")
    main = torch.cuda.current_stream()
    lanes = [torch.cuda.Stream() for _ in range(L)]

    def lane_of(k, serial=False):
        return lanes[0] if serial else lanes[(k % R) % L]

    def step(k, serial=False, host_loc=False):
        """Enqueue step k on its lane's stream (serial=True: every step on lane 0, one after the other)."""
        with torch.cuda.stream(lane_of(k, serial)):
            if graphs:
                (graphs_hl if host_loc else graphs)[k % R].replay()
            else:
                run_set(sets[k % R], host_loc=host_loc)

    def fork():
        for ln in lanes:
            ln.wait_stream(main)

    def drain():
        for ln in lanes:
            main.wait_stream(ln)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(n):
        fork()
        for k in range(n):
            step(k)
            if k % 256 == 255:
                torch.cuda.synchronize()
        drain()
        torch.cuda.synchronize()

    # ---- device-resident timing: W warm-up steps, then exactly K steps between barrier+sync ----------------------
    # warm-up: at least W steps AND ~0.5 s of load so that the SM clocks have ramped up from idle.  Every rank runs
    # the same number of steps (the collective is part of a step): the time-based part is sized on rank 0.
    W, K = max(args.warmup, 3), args.steps
    run_steps(W)
    t0 = time.time()
    run_steps(4 * R)
    per_step_s = max((time.time() - t0) / (4 * R), 1e-6)
    plan = torch.tensor([int(0.5 / per_step_s), int(1.0 / per_step_s)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.broadcast(plan, src=0)
    n_ramp, n_tail = int(plan[0].item()), int(plan[1].item())
    run_steps(n_ramp)
    log("clock ramp done")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
        time.sleep(0.3)

    host_enqueue_us = [0.0]

    def timed(serial):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        drain()
        barrier()
        e0.record()
        fork()
        h0 = time.perf_counter()
        for k in range(K):
            step(W + k, serial=serial)
        host_enqueue_us[0] = 1e6 * (time.perf_counter() - h0) / K      # host time to enqueue one step (not a GPU time)
        drain()
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    dumped = None
    try:
        serial_ms = timed(True) if L > 1 else None       # one step at a time: the latency of a step
        elapsed_ms = timed(False)
        log("timed regions done: %.3f ms/step" % (elapsed_ms / K))
        if args.dump_outputs and rank == 0:
            last = sets[(W + K - 1) % R]                 # the buffer set of the last timed step
            dumped = step_outputs(last["hp"], last["image_id"])
        run_steps(n_tail)                                # keep the GPU busy a little longer: the clock sampler sees the loaded state
    finally:
        clocks = sampler.stop() if sampler else None     # never leave nvidia-smi running
    t = torch.tensor([elapsed_ms, serial_ms if serial_ms is not None else elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms, serial_ms = float(t[0].item()), float(t[1].item())
    value = world * B * K / (elapsed_ms * 1e-3)

    # ---- the steps in flight must not disturb each other: every set's outputs after a pipelined run are compared
    # bit for bit with the outputs of the same set run alone
    def outputs(s):
        return list(s["hp"]._enc_out[:4]) + [s["hp"]._slab.buf]
    fork()
    for r in range(R):
        step(r, serial=True)
    drain()
    torch.cuda.synchronize()
    alone = [[t.clone() for t in outputs(s)] for s in sets]
    for s in sets:
        for t in outputs(s):
            t.fill_(-7)
    torch.cuda.synchronize()
    run_steps(2 * R)
    for r, s in enumerate(sets):
        for a, b in zip(alone[r], outputs(s)):
            if not torch.equal(a, b):
                raise RuntimeError("set %d: outputs with %d steps in flight differ from the serial run" % (r, L))
    alone_slabs = [a[-1] for a in alone]
    del alone

    log("in-flight outputs verified")
    # ---- N > 1: what every rank received must be what every rank sent.  Each rank checksums its own slab of every set;
    # the checksums travel separately (torch.distributed, outside any timed region) and are compared with checksums of
    # the received slabs; the rank's own slot must be bit-identical to its send buffer.
    gather_check = None
    if world > 1:
        weights = torch.arange(slab_words, device=dev, dtype=torch.int64) % 65521 + 1

        def checksum(x):
            v = x.view(torch.int32).to(torch.int64)
            return torch.stack([v.sum(), (v * weights).sum()])
        mine = torch.stack([checksum(s["hp"]._slab.buf) for s in sets])                    # [R, 2]
        allsums = torch.empty((world,) + tuple(mine.shape), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allsums, mine)
        for r, s in enumerate(sets):
            for q in range(world):
                got = checksum(s["recv"][q * slab_words:(q + 1) * slab_words])
                if not torch.equal(got, allsums[q, r]):
                    raise RuntimeError("rank %d, set %d: the slab received from rank %d differs from what it sent" % (rank, r, q))
            if not torch.equal(s["recv"][rank * slab_words:(rank + 1) * slab_words], s["hp"]._slab.buf):
                raise RuntimeError("rank %d, set %d: own slot of the gathered buffer differs from the send slab" % (rank, r))
        per_rank = [int(v[0].sum()) for v in sets[0]["hp"].gathered()]
        gather_check = {"verified": "checksums of all %d x %d received slabs equal the senders' on every rank" % (world, R),
                        "detections_per_rank_set0": per_rank}

    log("gather verified")
    # ---- end to end: host buffers in, results out, every step ----------------------------------------------------
    # Software pipeline over three streams: while step k computes, the inputs of step k+1 cross PCIe on the copy-in stream
    # and the results of step k-1 are read back.  Every step's inputs come from pinned host memory and every step's
    # result lands in pinned host memory inside the timed region.  full=True also returns the encode outputs (targets,
    # labels, scores, matched boxes: 44 B/anchor), which the reference produces in host RAM (dataset_common.py:150,178).
    NB = 4                                    # result buffers on the host: the host reads the result of step k - (NB - 1)
    PREFETCH = 3                              # inputs of step k + PREFETCH are enqueued while step k is (R >= 4 buffer sets)
    h_out = [torch.empty(slab_words, dtype=torch.float32).pin_memory() for _ in range(NB)]
    h_enc = [None] * NB
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    ev_in = [torch.cuda.Event() for _ in range(R)]
    ev_done = [torch.cuda.Event() for _ in range(R)]
    ev_out = [torch.cuda.Event() for _ in range(NB)]

    def e2e_run(n_steps, full, host_loc):
        copied = ("gt", "offs", "cls") if host_loc else ("gt", "offs", "cls", "loc")

        def copy_in(k):
            s = sets[k % R]
            with torch.cuda.stream(s_in):
                s_in.wait_event(ev_done[k % R])            # the set's previous user has finished
                for name in copied:
                    s["dev"][name].copy_(s["host"][name], non_blocking=True)
                ev_in[k % R].record(s_in)
        drain()
        for r in range(R):
            ev_done[r].record(main)
        fork()
        ahead = max(1, min(PREFETCH, R - 1))
        for k in range(min(ahead, n_steps)):
            copy_in(k)
        for k in range(n_steps):
            if k + ahead < n_steps:
                copy_in(k + ahead)
            lane_of(k).wait_event(ev_in[k % R])
            step(k, host_loc=host_loc)
            ev_done[k % R].record(lane_of(k))
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_done[k % R])
                ev_out[k % NB].synchronize()                  # the host consumed this pinned buffer NB steps ago
                h_out[k % NB].copy_(sets[k % R]["hp"]._slab.buf, non_blocking=True)
                if full:
                    for dst, src in zip(h_enc[k % NB], sets[k % R]["hp"]._enc_out[:4]):
                        dst.copy_(src, non_blocking=True)
                ev_out[k % NB].record(s_out)
            if k >= NB - 1:
                ev_out[(k - (NB - 1)) % NB].synchronize()     # the result of step k - (NB - 1) is on the host now
        for ev in ev_out:
            ev.synchronize()
        torch.cuda.synchronize()

    def e2e_measure(full, host_loc):
        e2e_run(4, full, host_loc)
        barrier()
        t0 = time.perf_counter()
        e2e_run(K, full, host_loc)
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    def nbytes(s, names):
        return sum(int(s["host"][n].numel() * s["host"][n].element_size()) for n in names)
    d2h = slab_words * 4
    # (a) every input tensor copied to the device, as in round 1
    h2d_all = nbytes(sets[0], ("gt", "offs", "cls", "loc"))
    e2e_all_s = e2e_measure(False, False)
    e2e_copy_all = {"value": world * B * K / e2e_all_s, "unit": UNIT, "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_all_s / K, "h2d_gbs_per_gpu": h2d_all * K / e2e_all_s / 1e9,
                    "note": "all of GT, logits AND box offsets copied to the device every step (26 MB): bound by PCIe"}
    # (b) host-resident geometry: GT and logits are copied; the box offsets stay in the pinned host buffer and the NMS kernel
    # fetches, in place over PCIe, only the rows of the anchors that pass the score threshold.  Same results, bit for bit
    # (checked below against the device-resident run).
    if not args.no_graph:
        graphs_hl.extend(capture(True))
    for s in sets:
        s["hp"]._slab.buf.fill_(-7)
    e2e_s = e2e_measure(False, True)
    for r, s in enumerate(sets[:max(4, K)]):              # (the sets the two runs above have touched)
        if not torch.equal(alone_slabs[r], s["hp"]._slab.buf):
            raise RuntimeError("set %d: detections with the box offsets read from host memory differ from the device-resident run" % r)
    thr = float(pp_params.select_threshold)
    rows = float(np.mean([int((torch.softmax(s["dev"]["cls"], -1)[..., 1] > thr).sum().item()) for s in sets[:4]]))
    h2d_copied = nbytes(sets[0], ("gt", "offs", "cls"))
    h2d = int(h2d_copied + 16 * rows)
    e2e = {"value": world * B * K / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "ms_per_step": 1e3 * e2e_s / K, "h2d_gbs_per_gpu": h2d * K / e2e_s / 1e9,
           "h2d_copied_bytes_per_step": h2d_copied, "h2d_rows_read_in_place_per_step": rows,
           "returns": "detection slab (counts, boxes, scores); the encode targets stay on the device, where a training "
                      "loop consumes them",
           "verified": "detection slabs of all sets bit-identical to the device-resident run",
           "note": "per step: GT boxes and logits copied in from pinned host memory (8.7 MB); the box offsets (17.5 MB) stay in "
                   "pinned host memory and the NMS kernel reads the ~3 % of rows whose score passes the threshold in place over "
                   "PCIe (dan_postprocess_batch, host-resident geometry); hot path; detection slab copied out to pinned host "
                   "memory; copies of neighbouring steps overlap the compute (3 streams). e2e_copy_all is the same with all "
                   "26 MB copied"}
    h_enc = [[torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in sets[0]["hp"]._enc_out[:4]] for _ in range(NB)]
    d2h_full = d2h + sum(int(t.numel() * t.element_size()) for t in sets[0]["hp"]._enc_out[:4])
    e2e_full_s = e2e_measure(True, True)
    e2e_full = {"value": world * B * K / e2e_full_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_full,
                "ms_per_step": 1e3 * e2e_full_s / K,
                "returns": "detection slab AND the encode outputs (targets, labels, scores, matched boxes) in pinned host memory, "
                           "as the reference's input pipeline produces them (dataset_common.py:150,178-186)"}
    h_enc = [None] * NB

    log("e2e done")
    # ---- per-kernel CUDA-event durations (profile entry points), cold buffers --------------------------------------
    prof = {}
    reps = max(10, R)
    for k in range(reps):
        _, det, ms = run_set(sets[k % R], profile=True)
        for name, v in ms.items():
            prof.setdefault(name, []).append(v)
    kernel_ms = {name: statistics.mean(v[2:]) for name, v in prof.items()}
    kernel_ms.pop("pp_filter", None)          # two classes: the filter runs inside nms_greedy_kernel
    step_kernel_sum = sum(kernel_ms.values())
    longest = max(kernel_ms, key=kernel_ms.get)

    # ---- roofline of the STEP (SURVEY.md 8(d)): per stage t = max(bytes / BW_HBM, flops / P_FP32) on the ALGORITHMIC
    # work, summed over the stages, against the measured time of a step
    peak_hbm, peak_src = measured_hbm_peak()
    p_fp32, fp32_src = fp32_peak()
    # candidates per image K (after threshold / top-k): where fewer than nms_topk boxes were kept, the first filler row
    # of the keep list sits at position K
    last = sets[(reps - 1) % R]["hp"]
    cnts = last._slab.views()[0].reshape(-1).cpu().numpy()
    keep = last._aux[1].reshape(len(cnts), -1).cpu().numpy()
    Ks = np.array([keep[i, cnts[i]] if cnts[i] < pp_params.nms_topk else pp_params.keep_topk for i in range(len(cnts))], dtype=np.float64)
    enc_bytes = B * (44.0 * N) + 16.0 * total_gt_mean + 17.0 * N       # 44N + 16M + 17N/B per image
    enc_flops = N * (20.0 * total_gt_mean + 30.0 * B)                  # N (20 M + 30) per image, non-FMA flops
    pp_bytes = B * 24.0 * N + float(np.sum(20.0 * np.minimum(cnts, pp_params.nms_topk)))   # 24 N + 20 K_out per image
    pp_flops = 40.0 * N * B
    nms_flops = float(np.sum(16.0 * Ks * (Ks - 1.0) / 2.0))            # 16 K (K-1) / 2 per image
    nms_bytes = 20.0 * float(np.sum(Ks))

    def stage(nbytes, flops):
        t_h, t_f = 1e6 * nbytes / (peak_hbm * 1e9), 1e6 * flops / p_fp32
        return {"bytes": nbytes, "flops": flops, "t_hbm_us": t_h, "t_fp32_us": t_f, "bound": "hbm" if t_h >= t_f else "fp32",
                "t_roofline_us": max(t_h, t_f)}
    stages = {"encode": stage(enc_bytes, enc_flops), "decode_filter": stage(pp_bytes, pp_flops), "nms": stage(nms_bytes, nms_flops)}
    t_roof_us = sum(st["t_roofline_us"] for st in stages.values())
    step_us = 1e3 * elapsed_ms / K
    traffic = ncu_traffic() or {}
    step_bytes = enc_bytes + pp_bytes
    p1_gbs = enc_bytes / (kernel_ms["enc_pass1"] * 1e-3) / 1e9
    roofline = {
        # the step against the roofline: images/s of the measured step vs images/s at which the algorithmic work of the
        # three stages would run at the binding peak of each stage (encode, NMS: non-FMA FP32 issue rate; filter: HBM)
        "bound": "fp32 (encode, nms) + hbm (decode_filter), per stage",
        "achieved": B * 1e6 / step_us, "peak": B * 1e6 / t_roof_us, "unit": "images/s per GPU",
        "frac": t_roof_us / step_us,
        "t_roofline_us": t_roof_us, "t_step_us": step_us, "stages": stages,
        "mean_candidates_per_image": float(np.mean(Ks)),
        "peak_hbm_gbs": peak_hbm, "peak_hbm_source": peak_src, "peak_fp32_tinstr_s": p_fp32 / 1e12, "peak_fp32_source": fp32_src,
        "serial_frac": (t_roof_us / (1e3 * serial_ms / K)) if serial_ms else None,
        "kernel": longest, "kernel_ms": kernel_ms[longest],
        # HBM view: algorithmic bytes of the whole step over the step time, and of the kernel that writes all encode outputs
        "hbm": {"step_bytes": step_bytes, "step_achieved_gbs": step_bytes / (step_us * 1e-6) / 1e9,
                "step_frac": step_bytes / (step_us * 1e-6) / 1e9 / peak_hbm,
                "enc_pass1": {"algorithmic_bytes_per_launch": enc_bytes, "kernel_ms": kernel_ms["enc_pass1"], "achieved_gbs": p1_gbs,
                              "frac": p1_gbs / peak_hbm}},
        "traffic": traffic.get("enc_pass1_fused_kernel"),
        "fp32_dense_equivalent": {"flops_per_step": enc_flops, "kernel": "enc_pass1", "kernel_ms": kernel_ms["enc_pass1"],
                                  "achieved_tflops": enc_flops / (kernel_ms["enc_pass1"] * 1e-3) / 1e12,
                                  "frac": enc_flops / (kernel_ms["enc_pass1"] * 1e-3) / p_fp32},
    }

    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": workload_config(B, world),
                "run": {"l2_policy": "%d rotating input/output buffer sets (%.0f MB) > 126 MB L2" % (R, R * per_set / 1e6),
                        "cuda_graph": not args.no_graph, "two_stream_overlap": not args.no_overlap, "steps_in_flight": L,
                        "inflight_outputs": "bit-identical to the serial run (checked on all sets)",
                        "mean_gt_per_image": total_gt_mean / B, "host_enqueue_us_per_step": host_enqueue_us[0],
                        "gather": None if world == 1 else (
                            "peer stores: the NMS kernel writes its slab rows into every rank's receive buffer over NVLink "
                            "(dan_postprocess_batch_peers) + a one-warp wait on the arrival flags, inside each step's CUDA graph"
                            if peers is not None else "ncclAllGather inside each step's CUDA graph (dan_gather_detections)"),
                        "gather_fallback": gather_fallback, "gather_check": gather_check, "host_cores_per_rank": cores_per_rank, "numa_node_rank0": numa_node,
                        "native_so_loaded": [os.path.relpath(_lib.LIB_PATH, ROOT)]},
                "clocks": clocks, "e2e": e2e, "e2e_copy_all": e2e_copy_all, "e2e_full": e2e_full, "gpu_launches": launches_per_step * K,
                "roofline": roofline, "cpu_baseline": cpu_base,
                "kernel_ms": kernel_ms, "step_kernel_ms_sum": step_kernel_sum,
                "serial": {"ms_per_step": serial_ms / K, "value": world * B * K / (serial_ms * 1e-3), "unit": UNIT,
                           "note": "same K steps with one step in flight (step latency); `value` has %d steps in flight" % L}}
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        # Teardown: the CUDA graphs hold references to the lanes' NCCL communicators, and ncclCommDestroy blocks while a
        # captured graph still uses the communicator - release the graphs first, then the communicators.
        torch.cuda.synchronize()
        dist.barrier()
        graphs.clear()
        for s in sets:
            s["hp"] = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        for g in gathers:
            if g is not None:
                g.close()
        if peers is not None:
            for s in sets:
                s["recv"] = None
            dist.barrier()
            peers.close()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="images per GPU per step")
    ap.add_argument("--sets", type=int, default=0, help="rotating buffer sets (0 = enough for 3x L2)")
    ap.add_argument("--inflight", type=int, default=10, help="steps in flight (each on its own stream and workspaces)")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"], help="detection exchange at N > 1")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="run encode and postprocess on one stream")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-layout-hint", action="store_true", help="encode without the pyramid layout hint (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one (rank 0's encode outputs and detections, "
                         "float32, at most 64 MB) as DIR/<name>.npy; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs needs the CUDA arm")
    if args.impl == "reference":
        return run_reference(args)
    return run_cuda(args)


if __name__ == "__main__":
    sys.exit(main())
