"""Times the device SSIM (ops.frame_ssim, bmv_frame_ssim) and what it adds to an evaluate loop at the C2 frame.

    python tools/ssim_bench.py [--out FILE] [--reps 200]

Prints one JSON document (and writes it to --out):
  * card: device name, power limit and max SM clock (nvidia-smi query only), read in the same run;
  * kernel: ops.frame_ssim at 960x544 and 1920x1088, win_size 7 and 101, data_range 2, no crop.  `reps` launches are
    captured in one CUDA graph and timed with CUDA events over several replays (the graph removes the Python / ctypes
    enqueue cost, which is larger than the kernel).  The launches rotate through distinct (pred, gt) pairs that
    together exceed the 126 MB L2, so every launch streams its frame from HBM.  Rate = algorithmic bytes (24 B per
    pixel: pred and gt, fp32 RGB, read once) over time, against the 6550 GB/s a B200 copy kernel measured and the
    7.7 TB/s data-sheet peak.  Each size / window is also checked against the float64 oracle;
  * frame: C2 (bench.py's workload: 960x544, 6 source views, K = 4) FrameGraph replay alone, replay + PsnrAccumulator,
    and replay + FrameEvaluator (PSNR and SSIM), per frame, with the ground truth uploaded from pinned host memory every
    frame as a loader would deliver it;
  * host: the float64 scipy restatement (oracle/ssim_oracle.frame_ssim) on this machine's CPU, with its core count.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from boostmvsnerfs_b200 import network, ops, sinks  # noqa: E402
from boostmvsnerfs_b200.config import RenderConfig  # noqa: E402
from boostmvsnerfs_b200.graph import FrameGraph  # noqa: E402
from boostmvsnerfs_b200.synth import batch_to, make_scene  # noqa: E402
from oracle import ssim_oracle as SSO  # noqa: E402

L2_BYTES = 126e6
MEASURED_GBS, DATASHEET_GBS = 6550.0, 7700.0


def card():
    info = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info.update(zip(("name", "power_limit", "clocks_max_sm"), (s.strip() for s in q.split(","))))
    except (OSError, IndexError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"unavailable: {exc}"
    return info


def time_kernel(H, W, win, reps, repeats):
    pair_bytes = 24 * H * W
    n_pairs = int(L2_BYTES // pair_bytes) * 2 + 2          # > 2x the L2 in all
    g = torch.Generator(device="cuda").manual_seed(H + win)
    gts = [torch.rand(H * W, 3, device="cuda", generator=g) for _ in range(n_pairs)]
    preds = [(t + 0.05 * torch.randn(t.shape, device="cuda", generator=g)).clamp_(0, 1) for t in gts]
    out = torch.empty(1, device="cuda", dtype=torch.float64)
    for i in range(n_pairs):                                  # warm-up: every pair once, eager
        ops.frame_ssim(preds[i], gts[i], H, W, win_size=win, out=out)
    torch.cuda.synchronize()
    want = SSO.frame_ssim(preds[0].cpu().numpy().reshape(H, W, 3), gts[0].cpu().numpy().reshape(H, W, 3), win, 2.0)
    got = ops.frame_ssim(preds[0], gts[0], H, W, win_size=win).item()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        ops.frame_ssim(preds[i % n_pairs], gts[i % n_pairs], H, W, win_size=win, out=out)
    e1.record()
    torch.cuda.synchronize()
    eager_us = e0.elapsed_time(e1) / reps * 1e3
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.frame_ssim(preds[0], gts[0], H, W, win_size=win, out=out)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(reps):
            ops.frame_ssim(preds[i % n_pairs], gts[i % n_pairs], H, W, win_size=win, out=out)
    graph.replay()
    torch.cuda.synchronize()
    us = []
    for _ in range(repeats):
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        us.append(e0.elapsed_time(e1) / reps * 1e3)
    med = statistics.median(us)
    return {"H": H, "W": W, "win_size": win, "launches_per_replay": reps, "distinct_pairs": n_pairs,
            "working_set_MB": round(n_pairs * pair_bytes / 1e6, 1), "us_per_launch_graph": [round(u, 2) for u in us],
            "us_per_launch_graph_median": round(med, 2), "us_per_launch_eager": round(eager_us, 2),
            "algorithmic_bytes": pair_bytes, "GB_per_s": round(pair_bytes / (med * 1e-6) / 1e9, 1),
            "fraction_of_measured_6550_GBps": round(pair_bytes / (med * 1e-6) / 1e9 / MEASURED_GBS, 4),
            "fraction_of_datasheet_7700_GBps": round(pair_bytes / (med * 1e-6) / 1e9 / DATASHEET_GBS, 4),
            "ssim_device": got, "ssim_oracle_f64": want, "abs_err": abs(got - want)}


def time_frames(steps):
    H, W = 544, 960
    rc = RenderConfig.enerf_eval(4)
    torch.manual_seed(0)
    net = network.BoostEnerfNetwork(preprocess=True, rc=rc).eval().cuda()
    net.view_selection_outputs = {"synth_0": [0, 7, 12, 19]}
    batch = batch_to(make_scene(H=H, W=W, n_views=6, seed=0), "cuda")
    rs = np.random.RandomState(0)
    batch["rgb_1"] = torch.from_numpy(rs.rand(1, H * W, 3).astype(np.float32)).pin_memory()
    fg = FrameGraph(net)
    res = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, make in (("replay", None), ("replay+PsnrAccumulator", lambda: sinks.PsnrAccumulator(rc)),
                       ("replay+FrameEvaluator(psnr,ssim)", lambda: sinks.FrameEvaluator(rc))):
        ev = make() if make else None
        for _ in range(3):
            out = fg(batch, cameras_unchanged=True)
            if ev:
                ev.evaluate(out, batch)
        torch.cuda.synchronize()
        ev = make() if make else None
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            out = fg(batch, cameras_unchanged=True)
            if ev:
                ev.evaluate(out, batch)
        e1.record()
        torch.cuda.synchronize()
        res[name] = {"ms_per_frame_events": round(e0.elapsed_time(e1) / steps, 4),
                     "ms_per_frame_wall": round((time.perf_counter() - t0) / steps * 1e3, 4)}
        if ev:
            res[name]["summary"] = ev.summarize()
    base = res["replay"]["ms_per_frame_events"]
    for name in list(res)[1:]:
        res[name]["added_us_per_frame"] = round((res[name]["ms_per_frame_events"] - base) * 1e3, 1)
    return {"workload": "C2 960x544, 6 source views, K=4, FrameGraph replay", "steps": steps, **res}


def time_host():
    rs = np.random.RandomState(0)
    res = {"cpu_count": os.cpu_count(), "implementation": "oracle/ssim_oracle.frame_ssim: float64, scipy.ndimage.uniform_filter"}
    for H, W, n in ((544, 960, 3), (1088, 1920, 2)):
        gt = rs.rand(H, W, 3).astype(np.float32)
        pred = np.clip(gt + 0.05 * rs.randn(H, W, 3), 0, 1).astype(np.float32)
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            SSO.frame_ssim(pred, gt, 7, 2.0)
            ts.append((time.perf_counter() - t0) * 1e3)
        res[f"{W}x{H}_w7_ms"] = round(min(ts), 1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--frames", type=int, default=100)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ssim_bench.py measures the GPU kernel: it needs a CUDA device")
    torch.cuda.set_device(0)
    doc = {"card": card(),
           "kernel": [time_kernel(H, W, win, a.reps, a.repeats) for H, W in ((544, 960), (1088, 1920)) for win in (7, 101)],
           "frame": time_frames(a.frames),
           "host": time_host()}
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
