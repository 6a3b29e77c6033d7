"""The bench.py contract (one JSON line per run, the keys the driver reads) checked without a GPU: the reference arm runs on
the CPU, and the committed final line of the CUDA arm (profiles/) is checked for the same keys."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMMON = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
          "dtype", "data", "config", "e2e", "cpu_baseline"]


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    line = json.loads(lines[-1])
    for k in COMMON:
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "images/s"
    assert line["config"]["workload"].startswith("S3FD 640x640") and line["scaling"] == "weak" and line["vs_baseline"] is None
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1


def test_committed_cuda_line_has_the_contract_keys():
    path = os.path.join(ROOT, "profiles", "r02_final_bench.json")
    if not os.path.exists(path):
        path = os.path.join(ROOT, "profiles", "r02_mid_bench.json")
    line = json.load(open(path))
    for k in COMMON + ["clocks", "gpu_launches", "roofline", "e2e_full", "run", "serial"]:
        assert k in line, k
    assert line["gpu_launches"] in (5 * line["steps"], 6 * line["steps"]) and line["dtype"] == "f32" and line["data"] == "synthetic"
    r = line["roofline"]
    # the roofline describes the step: per-stage max(hbm, fp32) times summed over the stages, against the step time
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and abs(r["frac"] - r["t_roofline_us"] / r["t_step_us"]) < 1e-9
    assert set(r["stages"]) == {"encode", "decode_filter", "nms"}
    assert abs(sum(st["t_roofline_us"] for st in r["stages"].values()) - r["t_roofline_us"]) < 1e-6
    assert r["stages"]["decode_filter"]["bound"] == "hbm" and r["stages"]["encode"]["bound"] == "fp32"
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert line["e2e_full"]["d2h_bytes_per_step"] > line["e2e"]["d2h_bytes_per_step"]
    assert set(line["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"}
    assert line["clocks"]["reasons"] == [] or "sw_power_cap" in "".join(line["clocks"]["reasons"])
    ref = json.load(open(os.path.join(ROOT, "profiles", os.path.basename(path).replace("_bench.json", "_bench_reference_arm.json"))))
    assert ref["config"] == line["config"]          # the driver compares the two arms' config objects


def test_rank_pinning_helpers():
    """bench.py's host-side helpers for N > 1: cpulist parsing and the per-rank core slices (no GPU, no NVML needed: without
    NUMA information every rank gets its own slice of the allowed cores, and the affinity is restored afterwards)."""
    sys.path.insert(0, ROOT)
    import bench
    assert bench._cpulist("0-3,8,10-11\n") == [0, 1, 2, 3, 8, 10, 11] and bench._cpulist("") == []
    assert bench.gpu_numa_nodes(2) in ([None, None], ) or all(v is None or v >= 0 for v in bench.gpu_numa_nodes(2))
    if hasattr(os, "sched_getaffinity"):
        before = os.sched_getaffinity(0)
        try:
            n0, node0 = bench.pin_rank_to_cores(0, 2)
            mine0 = os.sched_getaffinity(0)
            os.sched_setaffinity(0, before)
            n1, node1 = bench.pin_rank_to_cores(1, 2)
            mine1 = os.sched_getaffinity(0)
            assert n0 == len(mine0) >= 1 and n1 == len(mine1) >= 1 and mine0 <= before and mine1 <= before
            if len(before) >= 2 and node0 is None and node1 is None:
                assert not (mine0 & mine1)
        finally:
            os.sched_setaffinity(0, before)


def test_step_outputs_for_dump(monkeypatch):
    """--dump-outputs: every output of the step as float32 with one row per image (image_id float64), and above the size
    limit the same seeded sample of the images on every call."""
    sys.path.insert(0, ROOT)
    import bench
    from dan_b200 import pipeline

    class Step(object):
        pass
    B, N, K = 6, 40, 5
    gen = torch.Generator().manual_seed(0)
    hp = Step()
    hp._slab = pipeline.DetectionSlab(B, 1, K, "cpu")
    hp._slab.buf.copy_(torch.rand(hp._slab.words, generator=gen))
    hp._slab.views()[0].copy_(torch.arange(B, dtype=torch.int32).view(B, 1))
    hp._enc_out = (torch.rand(B, N, 4, generator=gen), torch.randint(-1, 2, (B, N), generator=gen), torch.rand(B, N, generator=gen),
                   torch.rand(B, N, 4, generator=gen), None)
    hp._aux = tuple(torch.randint(-1, 5000, (B, 1, K), dtype=torch.int32, generator=gen) for _ in range(2))
    ids = [100 + i for i in range(B)]
    full = bench.step_outputs(hp, ids)
    assert set(full) == {"enc_targets", "enc_labels", "enc_scores", "enc_matched_gt", "det_boxes", "det_scores", "det_counts",
                         "det_anchor_index", "det_keep_pos", "image_id"}
    assert full["image_id"].dtype == np.float64 and all(v.dtype == np.float32 for k, v in full.items() if k != "image_id")
    assert all(v.shape[0] == B for v in full.values())
    np.testing.assert_array_equal(full["enc_labels"], hp._enc_out[1].numpy())
    np.testing.assert_array_equal(full["det_counts"][:, 0], np.arange(B))
    np.testing.assert_array_equal(full["det_keep_pos"], hp._aux[1].numpy())

    per_image = sum(v[0].nbytes for v in full.values())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 3 * per_image + 1)
    a, b = bench.step_outputs(hp, ids), bench.step_outputs(hp, ids)
    assert a["image_id"].shape == (3,) and sum(v.nbytes for v in a.values()) <= bench.DUMP_LIMIT_BYTES
    rows = (a["image_id"] - 100).astype(np.int64)
    for name in full:
        np.testing.assert_array_equal(a[name], b[name])
        np.testing.assert_array_equal(a[name], full[name][rows])
