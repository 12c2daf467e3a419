#!/usr/bin/env python
"""Benchmark of the per-frame rendering hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C2|C1|C4]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one boosted frame (`Network.forward`) of the configuration BASELINE.json's metric is
quoted on: ENeRF + BoostMVSNeRFs, K=4 cost volumes, 960x540 run as 960x544 (H and W must be
multiples of 32, SURVEY.md §7), N=6 synthetic source views, random-init weights.
Rank 0 prints ONE JSON line; see DESIGN.md §Measurement for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (H, W, n_views, K, view-selection indices into C(n_views,3))
    "C1": dict(H=256, W=320, n_views=3, K=1, k_best=[0]),
    "C2": dict(H=544, W=960, n_views=6, K=4, k_best=[0, 7, 12, 19]),
    "C4": dict(H=1088, W=1920, n_views=6, K=8, k_best=[0, 3, 7, 9, 12, 15, 17, 19]),
    # MVSNeRF backbone + boost, 128 depth planes / samples, bf16 cost volume (BASELINE config 3)
    "C3": dict(H=544, W=960, n_views=6, K=4, k_best=[0, 7, 12, 19], backbone="mvsnerf", D=128),
    # ScanNet_plus-shaped sequence (BASELINE config 5): 1296x968 -> 1312x992, K=6; each step renders the NEXT novel view
    # of a 64-view trajectory, every view with its own K selected triples (one selection-agnostic graph)
    "C5": dict(H=992, W=1312, n_views=6, K=6, k_best=[0, 3, 7, 12, 15, 19], sequence=64),
}
CPU_SAMPLE_SIZES = [(544, 960), (384, 640), (288, 480), (256, 320), (128, 192), (64, 96)]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget-s", type=float, default=40.0)
    ap.add_argument("--stage-report", action="store_true", help="print the per-stage table to stderr")
    ap.add_argument("--mlp-engine", default=None, choices=["mma", "fma", "umma", "cublas"], help="override Network.mlp_engine")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true",
                    help="skip timing the reference's op sequence (oracle restatement) as eager PyTorch on this GPU (N=1 leg)")
    ap.add_argument("--no-strict", action="store_true", help="skip the strict-fp32 timing / parity legs")
    ap.add_argument("--ref-budget-s", type=float, default=300.0, help="time budget of the --impl reference run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (a fixed sample above 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the reference arm picks its frame size from a time budget: its outputs are not the same from run to run
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dump_dir, outs, limit=DUMP_LIMIT_BYTES):
    """Writes every tensor of `outs` (the outputs of the last timed step) as dump_dir/<name>.npy, float32 (float64 for
    integer or boolean outputs), so that two builds run with the same arguments can be compared output for output.
    Above `limit` bytes in all, every array is cut to a fixed, seeded sample of its flattened elements (the same sample
    for the same shapes) holding the same fraction of each array."""
    import numpy as np
    import torch
    arrays = {}
    for k, v in outs.items():
        if not torch.is_tensor(v):
            continue
        v = v.detach().cpu()
        arrays[k] = v.float().numpy() if v.is_floating_point() else v.double().numpy()
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(dump_dir, exist_ok=True)
    for k, a in sorted(arrays.items()):
        if total > limit:
            m = max(1, a.size * limit // total)
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, m, replace=False))]
        np.save(os.path.join(dump_dir, f"{k}.npy"), a)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = str(index), [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", self.index], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        threading.Thread(target=self._pump, daemon=True).start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.1] or [r for _, r in self.rows[-3:]]
        sm, reasons, mx, pw = [], set(), None, []
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx = float(r[2]); pw.append(float(r[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------ stage timing
class StageTimer:
    """CUDA-event brackets around the named stages of Network._render_frame, recorded on torch's
    current stream (the one libbmv launches on)."""

    def __init__(self):
        import torch
        self.torch = torch
        self.records, self.enabled = [], False

    def __call__(self, name):
        return _Stage(self, name)

    def summary(self):
        agg = {}
        for name, e0, e1 in self.records:
            a = agg.setdefault(name, [0.0, 0])
            a[0] += e0.elapsed_time(e1)
            a[1] += 1
        return agg


class KernelTimer:
    """CUDA events recorded right around each libbmv enqueue (hook: _lib.kernel_timer), so a kernel's
    duration is not inflated by host-side gaps when the stream runs dry."""

    def __init__(self, torch):
        self.torch, self.records, self.enabled, self._e0 = torch, [], False, None

    def before(self, name):
        if self.enabled:
            self._e0 = self.torch.cuda.Event(enable_timing=True)
            self._e0.record()

    def after(self, name):
        if self.enabled:
            e1 = self.torch.cuda.Event(enable_timing=True)
            e1.record()
            self.records.append((name, self._e0, e1))

    def summary(self):
        agg = {}
        for name, e0, e1 in self.records:
            a = agg.setdefault(name, [])
            a.append(e0.elapsed_time(e1))
        return agg


class _Stage:
    def __init__(self, timer, name):
        self.t, self.name = timer, name

    def __enter__(self):
        if self.t.enabled:
            self.e0 = self.t.torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *a):
        if self.t.enabled:
            e1 = self.t.torch.cuda.Event(enable_timing=True)
            e1.record()
            self.t.records.append((self.name, self.e0, e1))
        return False


def algorithmic_bytes(wl, rc, volume_bytes=4):
    """Compulsory HBM traffic per LAUNCH of each hand-written kernel (SURVEY.md §8(d); DESIGN.md).
    volume_bytes: storage size of a cost-volume element K1 writes (4 = fp32, the survey's figure; 2 = the fp16
    volume K1 emits when conv0 of the regulariser runs on libbmv's fp16-operand tensor-core kernel)."""
    H, W, K = wl["H"], wl["W"], wl["K"]
    S_v = rc.cost_volume_input_views
    out = {}
    for i in range(rc.num):
        C = int(32 * 2 ** (-i))
        hs, ws = int(H * rc.im_feat_scale[i]), int(W * rc.im_feat_scale[i])
        h, w, D = int(H * rc.volume_scale[i]), int(W * rc.volume_scale[i]), rc.volume_planes[i]
        planes = 0 if i == 0 else D * h * w * 4
        out[f"cost_volume_l{i}"] = S_v * C * hs * ws * 4 + planes + C * D * h * w * volume_bytes
        out[f"depth_regression_l{i}"] = D * h * w * 4 + (planes if i else D * 4) + 2 * h * w * 4
        if rc.render_if[i]:
            rs = rc.render_scale[i]
            Hr, Wr = int(H * rs), int(W * rs)
            R, S = Hr * Wr, rc.num_samples[i]
            Cf = rc.nerf_model_feat_ch[i]
            reads = 8 * D * h * w * 4 + S_v * (Cf + 3) * Hr * Wr * 4 + 4 * h * w * 4 + R * 8 * 4
            writes = R * S * 8 * 4 + R * S * S_v * (Cf + 7) * 4 + 2 * R * S * 4
            out[f"raygen_fetch_l{i}"] = reads + writes
            out[f"render_fused_l{i}"] = reads + R * S * (16 + 4 + 4)
            out[f"composite_blend_l{i}"] = R * (K * S * 24 + 12 + 4 + 4 * S)
    return out


# DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum, MB per launch) of the kernels `roofline` can name, from the
# committed `ncu --set full` captures (profiles/round1g_ncu_full_kernels.csv, round1j_ncu_full_conv_tma.csv,
# round1l_ncu_tcgen05.csv).  Traffic
# below the algorithmic bytes = part of the input / output was served by the 126 MB L2 (producer and consumer adjacent).
NCU_TRAFFIC_MB = {}
NCU_TRAFFIC_SOURCE = None


def load_ncu_traffic():
    """DRAM bytes per launch of the named kernels: profiles/ncu_traffic.json, written by tools/ncu_traffic.py from an
    `ncu --set full` capture of THIS build (the file records the capture it came from and the library digest)."""
    global NCU_TRAFFIC_MB, NCU_TRAFFIC_SOURCE
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        d = json.load(open(path))
        from boostmvsnerfs_b200 import build as _build
        if d.get("csrc_digest") != _build._digest()[:16]:          # a capture of ANOTHER build says nothing about this one
            NCU_TRAFFIC_MB, NCU_TRAFFIC_SOURCE = {}, {"stale": True, "captured_for": d.get("csrc_digest")}
            return
        NCU_TRAFFIC_MB = {k: float(v) for k, v in d.get("traffic_mb", {}).items()}
        NCU_TRAFFIC_SOURCE = {k: d.get(k) for k in ("capture", "csrc_digest", "when", "workload")}
    except (OSError, ValueError):
        NCU_TRAFFIC_MB, NCU_TRAFFIC_SOURCE = {}, None


def conv_kernel_bytes(wl, rc, volume_bytes=4, heads_entry="bmv_conv3d_k3", fpn_mid=False):
    """Compulsory HBM bytes of each libbmv convolution launch of one frame, keyed by entry point, in launch
    order (FPN: stem, half-resolution step, full-resolution step; per cascade level: conv0, conv1, conv2, heads /
    conv9T, conv11T).  All K chains (N views) are batched in one launch.  heads_entry: the entry point the merged
    heads run on (bmv_conv3d_k3_umma when the inference plan routes them to the tcgen05 kernel)."""
    H, W, K, N = wl["H"], wl["W"], wl["K"], wl["n_views"]
    px = N * H * W
    # stem: image in, c0 + the (N,H,W,4) colour image out.  cuDNN route of conv1.x / conv2.x: c0 fp32 + its space-to-depth
    # copy; tensor-core route (csrc/conv2d_mma.cu): c0 and every tensor up to the top layer in fp16, laterals read fp16
    lat = 2 if fpn_mid else 4                     # bytes per lateral-input element of the two top-down steps
    out = {"bmv_fpn_stem": [("fpn_stem", px * (3 * 4 + 4 * 4 + (8 * 2 if fpn_mid else 16 * 4)))],
           "bmv_fpn_topdown_smooth": [("fpn_topdown_smooth_half", px // 4 * (32 // 4 * 4 + 16 * lat + 32 * 4 + 16 * 4)),
                                      ("fpn_topdown_smooth_full", px * (32 // 4 * 4 + 8 * lat + 8 * 4))],
           "bmv_conv3d_k3": [], "bmv_convT3d_k3s2": []}
    if fpn_mid:      # conv1.0 (reads c0 through space-to-depth), conv1.1, conv2.0, conv2.1 + top layer (fp32 out)
        out["bmv_conv2d_k3"] = [("fpn_conv1_0", px * 8 * 2 + px // 4 * 16 * 2), ("fpn_conv1_1", px // 4 * 16 * (2 + 2)),
                                ("fpn_conv2_0", px // 4 * 16 * 2 + px // 16 * 32 * 2), ("fpn_conv2_1_top", px // 16 * 32 * (2 + 4))]
    out.setdefault(heads_entry, [])
    for i in range(rc.num):
        C = int(32 * 2 ** (-i))
        vox = K * rc.volume_planes[i] * int(H * rc.volume_scale[i]) * int(W * rc.volume_scale[i])
        a = volume_bytes      # activations between libbmv kernels are fp16 exactly when the cost volume is
        out["bmv_conv3d_k3"] += [(f"conv0_l{i}", vox * (C * volume_bytes + 8 * a)), (f"conv1_l{i}", vox * 8 * a + vox // 8 * 16 * a),
                                 (f"conv2_l{i}", vox // 8 * 16 * (a + 4))]
        out[heads_entry] += [(f"heads_l{i}", vox * (8 * a + 9 * 4))]
        out["bmv_convT3d_k3s2"] += [(f"conv9T_l{i}", vox // 64 * 32 * 4 + vox // 8 * 16 * (4 + a)),
                                    (f"conv11T_l{i}", vox // 8 * 16 * a + vox * 8 * a * 2)]
    return out


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_rate(wl, rc, steps, warmup, budget_s, state_dict=None, keep=None):
    """Times the oracle restatement of the reference's CPU path (oracle/enerf_oracle.py,
    kind="port": the reference is pure Python/PyTorch and cannot travel to the GPU box) with all
    host threads, on a bounded sample: the same K/N configuration at the largest listed
    resolution whose estimated cost fits the budget (the workload's own resolution when that fits).
    Returns (rays_per_s, ms_per_step, sample, cores, (h, w)).  state_dict: weights to load (the GPU arm's, so the
    frame can double as the parity reference); keep: dict that receives the last frame's outputs."""
    import torch
    from boostmvsnerfs_b200.modules import EnerfModules
    from boostmvsnerfs_b200.synth import make_scene
    from oracle import enerf_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    net = EnerfModules(rc).eval()
    if state_dict is not None:
        net.load_state_dict({k: v.detach().cpu() for k, v in state_dict.items()}, strict=True)
    kb = torch.tensor([wl["k_best"]])

    def run(h, w):
        scene = make_scene(H=h, W=w, n_views=wl["n_views"], seed=0)
        t0 = time.perf_counter()
        with torch.no_grad():
            out = O.boost_enerf_forward(net, scene, rc, kb)
        dt = time.perf_counter() - t0
        if keep is not None:
            keep.clear()
            keep.update({k: v for k, v in out.items()})
            keep["_size"] = (h, w)
        return dt

    run(64, 96)                                   # thread-pool / allocator warm-up
    t_probe = run(128, 192)
    rate = 128 * 192 / t_probe                    # rays/s estimate (roughly resolution independent)
    per_step_budget = budget_s / max(1, steps + warmup)
    size = CPU_SAMPLE_SIZES[-1]
    for h, w in [(wl["H"], wl["W"])] + CPU_SAMPLE_SIZES:
        if h <= wl["H"] and w <= wl["W"] and 1.1 * h * w / rate <= per_step_budget:  # margin over the small-frame probe (which under-estimates the rate)
            size = (h, w)
            break
    for _ in range(warmup):
        run(*size)
    ts = [run(*size) for _ in range(steps)]
    dt = sum(ts) / len(ts)
    sample = (f"{steps} frame(s) of K={wl['K']} N={wl['n_views']} at {size[1]}x{size[0]} "
              f"({size[0] * size[1]} rays) through oracle.boost_enerf_forward, torch {torch.__version__} CPU")
    return size[0] * size[1] / dt, dt * 1e3, sample, cores, size


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from boostmvsnerfs_b200.config import RenderConfig
    wl = WORKLOADS[args.workload]
    rc = RenderConfig.enerf_eval(wl["K"])
    rate, ms, sample, cores, size = cpu_reference_rate(wl, rc, max(1, args.steps), args.warmup, budget_s=args.ref_budget_s)
    full = (size[0], size[1]) == (wl["H"], wl["W"])
    line = {"impl": "reference", "metric": "rays_per_sec", "value": rate, "unit": "rays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, wl),
            # what each timed step actually was: the workload's own frame when (steps + warmup) of them fit the time
            # budget, else the same K / N at a smaller resolution (rays/s is roughly resolution independent)
            "step_sample": {"resolution": [size[1], size[0]], "full_workload_frame": full},
            "cpu_baseline": {"value": rate, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(name, wl):
    seq = (f"; sequence of {wl['sequence']} novel views over the same source images, a new target camera and a new selection "
           f"of K triples per step" if wl.get("sequence") else "")
    return {"workload": f"{name}: ENeRF + BoostMVSNeRFs K={wl['K']} cost volumes, {wl['W']}x{wl['H']} "
                        f"(960x540 padded to /32 for C2), N={wl['n_views']} source views, 3 views per volume, "
                        f"levels (64 planes @1/8, 8 planes @1/2), 2 samples/ray, random-init weights{seq}",
            "e2e_inputs": "pinned host: N source images + cameras + near/far, uploaded every step (graph mode: on a copy "
                          "stream while the previous frame renders, FrameGraph.prefetch); rays generated on device; "
                          "rgb + depth read back to pinned host memory every step",
            "l2": "no explicit flush: one frame streams ~3 GB through HBM (volumes 4x67 MB per level, fetched "
                  "features 4x221 MB), far above the 126 MB L2",
            "timing": "CUDA events on the launch stream around exactly `steps` frames, max over ranks"}


# ------------------------------------------------------------------------------------------ GPU arm
def main_ours(args):
    import torch
    import torch.distributed as dist
    from boostmvsnerfs_b200 import _lib, network
    from boostmvsnerfs_b200.config import RenderConfig
    from boostmvsnerfs_b200.synth import batch_to, make_scene

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    wl = WORKLOADS[args.workload]
    rc = RenderConfig.enerf_eval(wl["K"])
    torch.manual_seed(0)
    net = network.BoostEnerfNetwork(preprocess=True, rc=rc).eval().to(dev)
    net.view_selection_outputs = {"synth_0": wl["k_best"]}
    if args.mlp_engine:
        net.mlp_engine = args.mlp_engine
    timer = StageTimer()
    net.stage_timer = timer
    ktimer = KernelTimer(torch)
    _lib.kernel_timer = ktimer
    # replicas: every rank renders its own frames (different seeds) — SURVEY.md §8(e) "sequence mode"
    host = make_scene(H=wl["H"], W=wl["W"], n_views=wl["n_views"], seed=rank)
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in host.items()}
    batch = batch_to(host, dev)
    rays_per_frame = wl["H"] * wl["W"]
    # ---- sequence workloads (BASELINE config 5): every step renders the NEXT novel view of an n_seq-view trajectory over
    # the same source images; each view has its own target camera and its own K selected triples
    n_seq = int(wl.get("sequence", 0))
    seq_host, seq_dev = [], []
    if n_seq:
        import itertools
        import numpy as np
        from boostmvsnerfs_b200.synth import _look_at
        net.generate_rays = True                              # rays follow the per-view camera: generated on the device
        n_tri = len(list(itertools.combinations(range(wl["n_views"]), 3)))
        rs = np.random.RandomState(1234 + rank)
        for j in range(n_seq):
            ang = 2.0 * np.pi * j / n_seq
            eye = np.array([0.25 * np.cos(ang), 0.1 * np.sin(ang), 0.15 * np.sin(2 * ang)])
            tar_ext = torch.from_numpy(np.linalg.inv(_look_at(eye, np.array([0.0, 0.0, 5.0])))[None].astype(np.float32))
            hj = {k: v for k, v in host.items() if not k.startswith("rays_")}
            hj["tar_ext"] = tar_ext.pin_memory()
            hj["meta"] = {"scene": ["synth"], "tar_view": torch.tensor([j]), "frame_id": torch.tensor([j])}
            net.view_selection_outputs[f"synth_{j}"] = sorted(int(v) for v in rs.choice(n_tri, wl["K"], replace=False))
            seq_host.append(hj)
            dj = {k: v for k, v in batch.items() if not k.startswith("rays_")}
            dj["tar_ext"] = tar_ext.to(dev)
            dj["meta"] = hj["meta"]
            seq_dev.append(dj)

    def dev_batch(j):
        return seq_dev[j % n_seq] if n_seq else batch

    def host_batch(j):
        return seq_host[j % n_seq] if n_seq else host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    clocks = ClockSampler(local)
    clocks.start()                     # before the warm-up: the sampler's start-up must not steal host time from the timed loop
    for j in range(args.warmup):
        net(dev_batch(j))
    vol_dtype = str(getattr(net, "last_volume_dtype", torch.float32)).replace("torch.", "")
    # ---- device-resident timing: NO profiling hooks inside this region
    net.stage_timer = None
    _lib.kernel_timer = None
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    for j in range(args.steps):
        out = net(dev_batch(j))
    e1.record()
    t_host = (time.time() - t_wall0) / args.steps * 1e3        # host time to ENQUEUE one frame
    barrier()
    t_wall1 = time.time()
    eager_out = {k: v.detach().cpu() for k, v in out.items()} if args.dump_outputs else None
    launches = (_lib.launch_count() - l0) / args.steps
    ms = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    clk = clocks.stop(t_wall0, t_wall1)
    # ---- instrumented pass (same frames): CUDA events around every stage and every libbmv enqueue.
    # Kept out of the timed region above because ~60 event records per frame cost host time.
    net.stage_timer = timer
    _lib.kernel_timer = ktimer
    timer.enabled, timer.records = True, []
    ktimer.enabled, ktimer.records = True, []
    barrier()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for j in range(args.steps):
        net(dev_batch(j))
    pe1.record()
    barrier()
    ms_instrumented = pe0.elapsed_time(pe1) / args.steps
    timer.enabled = False
    ktimer.enabled = False
    net.stage_timer = None
    _lib.kernel_timer = None
    stages = timer.summary()

    # ---- end to end: pinned host inputs -> H2D -> forward -> D2H of the frame, every step.
    # The rays of a full target image are a pure function of (tar_ext, tar_ixt, H, W): they are generated on
    # the device (SURVEY.md §8 f3) instead of being uploaded, so the host batch carries images + cameras only.
    net.generate_rays = True
    host = {k: v for k, v in host.items() if not k.startswith("rays_")}
    h2d = sum(v.numel() * v.element_size() for k, v in host.items() if torch.is_tensor(v))
    res_host = {k: torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory() for k in ("rgb_level1", "depth_level1")}
    d2h = sum(v.numel() * v.element_size() for v in res_host.values())
    for j in range(2):
        o = net(batch_to(host_batch(j), dev, non_blocking=True))
    barrier()
    e0.record()
    for j in range(args.steps):
        o = net(batch_to(host_batch(j), dev, non_blocking=True))
        for k, v in res_host.items():
            v.copy_(o[k], non_blocking=True)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1) / args.steps)

    # ---- CUDA-graph replay of the frame (boostmvsnerfs_b200/graph.py): same kernels, one graph launch
    graph_res = None
    try:
        from boostmvsnerfs_b200.graph import FrameGraph
        fg = FrameGraph(net)
        for j in range(max(2, args.warmup)):
            fg(dev_batch(j))
        barrier()
        e0.record()
        for j in range(args.steps):
            # single frame: same batch object every step; sequence: a new camera + selection per step (device-resident
            # cameras are read back: one host sync per frame); includes the D2D refresh of the static inputs
            og = fg(dev_batch(j), cameras_unchanged=not n_seq)
        e1.record()
        barrier()
        ms_graph = max_over_ranks(e0.elapsed_time(e1) / args.steps)
        default_out = {k: v.detach().float().cpu() for k, v in og.items()}
        for j in range(2):
            og = fg(host_batch(j))
        barrier()
        fg.prefetch(host_batch(0))
        e0.record()
        for j in range(args.steps):
            og = fg(host_batch(j))                           # waits for this frame's upload, D2D into the static buffers, replay
            fg.prefetch(host_batch(j + 1))                   # H2D upload of the NEXT frame (pinned host batch) overlaps this replay
            fg.read_back(og, res_host)                       # D2H of THIS frame's rgb + depth overlaps the next replay
        fg.wait_read_back()                                  # the last frame's transfer is inside the timed region
        e1.record()
        barrier()
        ms_graph_e2e = max_over_ranks(e0.elapsed_time(e1) / args.steps)
        graph_res = {"ms_per_step": ms_graph, "value": world * rays_per_frame / (ms_graph * 1e-3),
                     "e2e_ms_per_step": ms_graph_e2e, "e2e_value": world * rays_per_frame / (ms_graph_e2e * 1e-3),
                     "captured_graphs": len(fg._cache)}
    except Exception as exc:                                 # report, never hide
        graph_res = {"error": f"{type(exc).__name__}: {exc}"}
        default_out = None

    # ---- strict-fp32 leg: the SAME frame with TF32-class arithmetic switched off (cuDNN fp32 convolutions, fp32 cost
    # volume): the path the 1e-4 parity tests check.  Timed through the same FrameGraph entry point.
    strict_res, strict_out = None, None
    if not args.no_strict and not n_seq:
        old_flags = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            from boostmvsnerfs_b200.graph import FrameGraph
            fgs = FrameGraph(net)
            n_strict = max(2, min(args.steps, 5))
            for _ in range(2):
                fgs(batch)
            barrier()
            e0.record()
            for _ in range(n_strict):
                os_ = fgs(batch, cameras_unchanged=True)
            e1.record()
            barrier()
            ms_strict = max_over_ranks(e0.elapsed_time(e1) / n_strict)
            strict_out = {k: v.detach().float().cpu() for k, v in os_.items()}
            strict_res = {"ms_per_step": ms_strict, "value": world * rays_per_frame / (ms_strict * 1e-3), "steps": n_strict,
                          "cost_volume_storage": str(getattr(net, "last_volume_dtype", None)).replace("torch.", ""),
                          "what": "torch.backends.cudnn.allow_tf32 = False: every kept convolution on cuDNN fp32, fp32 cost "
                                  "volume, hand-written K1-K5 unchanged; CUDA-graph replay"}
            del fgs
        except Exception as exc:
            strict_res = {"error": f"{type(exc).__name__}: {exc}"}
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_flags

    # ---- single-frame latency mode: the SAME frame sharded over the ranks (SURVEY.md §8(e))
    sharded = None
    if world > 1:
        from boostmvsnerfs_b200.dist import make_sharded_graph
        net.stage_timer = None
        keep_gen = net.generate_rays
        net.generate_rays = False
        same = batch_to(make_scene(H=wl["H"], W=wl["W"], n_views=wl["n_views"], seed=0), dev)
        with torch.no_grad():
            one = {k: v.clone() for k, v in net(dict(same)).items()}          # this rank alone renders the same frame
        sharded = {"scaling": "strong",
                   "what": "ONE frame: chain blocks over ranks, row-slab all-to-all of the regularised volumes + depth maps, "
                           "row tiles rendered by one launch per rank, NCCL all-gather of the frame; kernels and collectives "
                           "replayed as one CUDA graph per rank (dist.make_sharded_graph)"}
        for label, shard_feats in (("replicated_fpn", False), ("sharded_fpn_fp16_gather", True)):
            try:
                sg = make_sharded_graph(net, shard_features=shard_feats)
                for _ in range(max(2, args.warmup)):
                    so = sg(same, cameras_unchanged=False)
                barrier()
                e0.record()
                for _ in range(args.steps):
                    so = sg(same, cameras_unchanged=True)
                e1.record()
                barrier()
                ms_sh = max_over_ranks(e0.elapsed_time(e1) / args.steps)
                err, over = {}, {}
                for k in one:
                    d = (so[k].float() - one[k].float()).abs()
                    rng = one[k].float().abs().max().clamp_min(1e-12)
                    err[k] = max_over_ranks(float(d.max() / rng))
                    # a sample on a frustum edge flips its visibility count under a 1-ulp change of the depth map (a chain
                    # computed alone on a rank takes other cuDNN algorithms than in a batch of K): the count tells a
                    # handful of such rays from a systematic difference
                    over[k] = int(max_over_ranks(float((d > 1e-4 * rng).sum())))
                sharded[label] = {"ms_per_frame": ms_sh, "rays_per_sec": rays_per_frame / (ms_sh * 1e-3), "max_err_vs_single": err,
                                  "elements_over_1e-4_of_range": over}
                so = None
                sg.close()                                   # a live graph with NCCL work would hang destroy_process_group
                del sg
            except Exception as exc:
                sharded[label] = {"error": f"{type(exc).__name__}: {exc}"}
        best = min((v["ms_per_frame"] for v in sharded.values() if isinstance(v, dict) and "ms_per_frame" in v), default=None)
        sharded["ms_per_frame"] = best
        sharded["rays_per_sec"] = rays_per_frame / (best * 1e-3) if best else None
        net.generate_rays = keep_gen

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant hand-written kernel
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    alg = algorithmic_bytes(wl, rc, volume_bytes=2 if vol_dtype == "float16" else 4)
    launches_per_stage = {k: (wl["K"] if not k.startswith("composite") else 1) for k in alg}
    kernels, step_ms_stage = {}, {}
    # per-launch kernel durations by (entry point, order within the frame) -> stage name
    ksum = ktimer.summary()
    per_kernel = {}
    order = {"bmv_cost_volume_var": ["cost_volume_l0", "cost_volume_l1"],
             "bmv_depth_regression": ["depth_regression_l0", "depth_regression_l1"],
             "bmv_render_rays": [f"render_fused_l{i}" for i in range(rc.num) if rc.render_if[i]],
             "bmv_render_rays_mma": [f"render_fused_l{i}" for i in range(rc.num) if rc.render_if[i]],
             "bmv_render_rays_umma": [f"render_fused_l{i}" for i in range(rc.num) if rc.render_if[i]],
             # all K chains of a level in ONE launch (csrc/render_multi.cu / render_multi_umma.cu)
             "bmv_render_rays_multi": [f"render_fused_l{i}" for i in range(rc.num) if rc.render_if[i]],
             "bmv_render_rays_multi_umma": [f"render_fused_l{i}" for i in range(rc.num) if rc.render_if[i]],
             "bmv_raygen_sample_fetch": [f"raygen_fetch_l{i}" for i in range(rc.num) if rc.render_if[i]],
             "bmv_composite_blend": [f"composite_blend_l{i}" for i in range(rc.num) if rc.render_if[i]]}
    if ksum.get("bmv_cost_volume_var_multi"):
        # level 0: ONE launch for the K chains; every unique source view is read once, K volumes are written
        order["bmv_cost_volume_var"] = ["cost_volume_l1"]
        order["bmv_cost_volume_var_multi"] = ["cost_volume_l0"]
        C0 = 32
        hs0, ws0 = int(wl["H"] * rc.im_feat_scale[0]), int(wl["W"] * rc.im_feat_scale[0])
        h0, w0, D0 = int(wl["H"] * rc.volume_scale[0]), int(wl["W"] * rc.volume_scale[0]), rc.volume_planes[0]
        vb = 2 if vol_dtype == "float16" else 4
        # stored per chain like the other entries (the accounting below multiplies by K)
        alg["cost_volume_l0"] = (wl["n_views"] * C0 * hs0 * ws0 * 4) // wl["K"] + C0 * D0 * h0 * w0 * vb
    for entry, names in order.items():
        ts = ksum.get(entry, [])
        per_frame = len(ts) // max(1, args.steps)
        if not ts or per_frame % len(names):
            continue
        per_name = per_frame // len(names)
        for nm in names:
            launches_per_stage[nm] = per_name              # chain-batched kernels launch once per level
        for f in range(args.steps):
            for j, nm in enumerate(names):
                per_kernel.setdefault(nm, []).extend(ts[f * per_frame + j * per_name:f * per_frame + (j + 1) * per_name])
    for name, (tot_ms, cnt) in stages.items():
        step_ms_stage[name] = tot_ms / args.steps
        if name in alg:
            per_launch_ms = tot_ms / (args.steps * launches_per_stage[name])
            if per_kernel.get(name):
                per_launch_ms = sum(per_kernel[name]) / len(per_kernel[name])
            # alg[] is per chain; a chain-batched kernel processes all K chains of the level in one launch
            units = 1 if name.startswith("composite") else wl["K"]
            nbytes = alg[name] * units // launches_per_stage[name]
            gbs = nbytes / (per_launch_ms * 1e-3) / 1e9
            kernels[name] = {"ms_per_launch": per_launch_ms, "launches_per_step": launches_per_stage[name],
                             "algorithmic_bytes": nbytes, "achieved_gbs": gbs, "frac": gbs / peak_gbs,
                             "share_of_step": per_launch_ms * launches_per_stage[name] / ms}
    # libbmv convolution kernels (one launch each per frame), same accounting
    heads_entry = "bmv_conv3d_k3_umma" if ksum.get("bmv_conv3d_k3_umma") else "bmv_conv3d_k3"
    for entry, layers in conv_kernel_bytes(wl, rc, 2 if vol_dtype == "float16" else 4, heads_entry, bool(ksum.get("bmv_conv2d_k3"))).items():
        ts = ksum.get(entry, [])
        if len(ts) != len(layers) * args.steps:
            continue
        for j, (nm, nbytes) in enumerate(layers):
            per_launch_ms = sum(ts[j::len(layers)]) / args.steps
            gbs = nbytes / (per_launch_ms * 1e-3) / 1e9
            kernels[nm] = {"ms_per_launch": per_launch_ms, "launches_per_step": 1, "algorithmic_bytes": nbytes,
                           "achieved_gbs": gbs, "frac": gbs / peak_gbs, "share_of_step": per_launch_ms / ms}
    for name, k in kernels.items():
        if name.startswith("render_fused"):
            # the fused gather+MLP kernel is compute bound, not HBM bound: 14.6 kFMA per sample (csrc/nerf_mlp.cuh).
            # Reported as fp32-equivalent FLOP/s against the fp32 FMA peak (148 SMs x 128 FMA/clk x clocks.max.sm);
            # the tensor-core engines spend 3 fp16 MMAs per fp32 product (csrc/render_multi_umma.cu, render_multi.cu).
            lvl = int(name[-1])
            samples = int(wl["H"] * rc.render_scale[lvl]) * int(wl["W"] * rc.render_scale[lvl]) * rc.num_samples[lvl]
            flops = samples * 2 * 14600.0 * (wl["K"] / k["launches_per_step"])      # a launch renders K / launches chains
            peak_tf = 148 * 128 * 2 * (clk.get("sm_max_mhz") or 1965.0) * 1e6 / 1e12
            k.update({"bound": "fp32_fma", "tflops": flops / (k["ms_per_launch"] * 1e-3) / 1e12,
                      "peak_tflops_fp32": peak_tf})
            k["frac_fp32_peak"] = k["tflops"] / peak_tf
        else:
            k["bound"] = "hbm"
    # `roofline`: the DOMINANT kernel of the step (largest share of the frame).  That is the fused gather+MLP kernel: its
    # Linear layers run on the tensor cores, so it is reported against the measured dense tensor peak with its ALGORITHMIC
    # flops (2 x 14.6 kMAC per sample, DESIGN.md 3; the kernel spends 3 fp16 MMAs per fp32 product and ~6 k CUDA-core
    # instructions per sample on the gather / splits / activations, which is what actually bounds it).
    # `roofline_hbm`: the dominant HBM-bound hand-written kernel, against the measured copy bandwidth.
    def _share(n):
        return kernels[n]["ms_per_launch"] * kernels[n]["launches_per_step"]
    hbm_kernels = {n: k for n, k in kernels.items() if k["bound"] == "hbm"}
    # north_star names the cost-volume build (K1) as the HBM kernel to judge: report the K1 launch with the largest share
    # (the dominant HBM-bound kernel of any kind is in `roofline_hbm_dominant`)
    k1 = {n: k for n, k in hbm_kernels.items() if n.startswith("cost_volume")}
    dom_hbm_any = max(hbm_kernels, key=_share) if hbm_kernels else None
    dom_hbm = max(k1, key=_share) if k1 else dom_hbm_any
    dom = max(kernels, key=_share) if kernels else None
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 2250.0)))
    tf_src = ("measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)" if "bf16_tflops_sustained" in peaks
              else "fallback 2250 TFLOP/s dense bf16 (B200_PROFILING.md)")

    load_ncu_traffic()

    def _traffic(n):
        # the capture is of ONE workload (C2 unless the file says otherwise): no traffic figure for another frame size
        if (NCU_TRAFFIC_SOURCE or {}).get("workload", "C2") != args.workload:
            return None
        return NCU_TRAFFIC_MB[n] * 1e6 if n in NCU_TRAFFIC_MB else None

    def _hbm_obj(n):
        return {"kernel": n, "bound": "hbm", "achieved": kernels[n]["achieved_gbs"], "peak": peak_gbs, "unit": "GB/s",
                "frac": kernels[n]["frac"], "traffic": _traffic(n), "peak_source": peak_src, "launch_ms": kernels[n]["ms_per_launch"],
                "algorithmic_bytes": kernels[n]["algorithmic_bytes"], "share_of_step": kernels[n]["share_of_step"]}
    roofline = None
    if dom and kernels[dom]["bound"] == "fp32_fma":
        k = kernels[dom]
        roofline = {"kernel": dom, "bound": "tensor", "achieved": k["tflops"], "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": k["tflops"] / peak_tf, "traffic": _traffic(dom), "peak_source": tf_src, "launch_ms": k["ms_per_launch"],
                    "algorithmic_flops": k["tflops"] * 1e12 * k["ms_per_launch"] * 1e-3, "share_of_step": k["share_of_step"],
                    "engine": net.mlp_engine}
    elif dom:
        roofline = _hbm_obj(dom)
    roofline_hbm = _hbm_obj(dom_hbm) if dom_hbm else None
    roofline_hbm_dominant = _hbm_obj(dom_hbm_any) if dom_hbm_any else None
    hand_ms = sum(step_ms_stage.get(k, 0.0) for k in alg)
    eager = {"ms_per_step": ms, "value": world * rays_per_frame / (ms * 1e-3), "e2e_ms_per_step": ms_e2e,
             "e2e_value": world * rays_per_frame / (ms_e2e * 1e-3)}
    # headline = the faster of the two public entry points (Network.forward / FrameGraph.__call__), chosen
    # separately for the device-resident number and for the end-to-end number; both modes are listed in full
    execution, timed_out = "value: eager (stream launches)", eager_out
    if graph_res and "error" not in graph_res and graph_res["ms_per_step"] < ms:
        ms, execution, timed_out = graph_res["ms_per_step"], "value: cuda_graph replay (FrameGraph)", default_out
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, timed_out)
    if graph_res and "error" not in graph_res and graph_res["e2e_ms_per_step"] < ms_e2e:
        ms_e2e, execution = graph_res["e2e_ms_per_step"], execution + "; e2e: cuda_graph replay (FrameGraph)"
    else:
        execution += "; e2e: eager (stream launches)"
    # kernel shares refer to the REPORTED step (the graph replay when it is the faster entry point): the per-launch times
    # were taken in the eager instrumented pass (same kernels, same durations), whose step is longer by the host gaps
    for k in kernels.values():
        k["share_of_step"] = k["ms_per_launch"] * k["launches_per_step"] / ms
    for obj in (roofline, roofline_hbm, roofline_hbm_dominant):
        if obj:
            obj["share_of_step"] = kernels[obj["kernel"]]["share_of_step"]
    line = {
        "metric": "rays_per_sec", "value": world * rays_per_frame / (ms * 1e-3), "unit": "rays/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "ms_per_frame": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        # what the timed (default) path computes in: with torch defaults (cudnn.allow_tf32) the FPN / U-Net convolutions run
        # with fp16 operands and fp32 accumulation and K1 stores a range-scaled fp16 volume (TF32-class, like the reference's
        # own cuDNN convolutions under the same defaults); K1-K5 arithmetic, the MLP (split-fp16 = fp32-class) and K4 are fp32
        "dtype": ("f16-operand/f32-accum convs + scaled-f16 cost volume (TF32-class), f32 elsewhere" if vol_dtype == "float16"
                  else "f32"),
        "data": "synthetic",
        "config": workload_config(args.workload, wl),
        "run": {"execution": execution, "cost_volume_storage": vol_dtype,
                "parallelism": ("single GPU" if world == 1 else f"{world} frame replicas, no data-path collective"),
                "ncu_traffic_source": NCU_TRAFFIC_SOURCE},
        "strict_fp32": strict_res,
        "e2e": {"value": world * rays_per_frame / (ms_e2e * 1e-3), "unit": "rays/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "eager": eager, "cuda_graph": graph_res,
        "gpu_launches": launches, "clocks": clk, "roofline": roofline, "roofline_hbm": roofline_hbm, "roofline_hbm_dominant": roofline_hbm_dominant, "kernels": kernels, "frame_sharded": sharded,
        "stage_ms_per_step": step_ms_stage, "hand_written_ms_per_step": hand_ms,
        "stage_ms_note": "eager instrumented pass: when the GPU outruns the Python enqueue (host_enqueue_ms_per_step >= "
                         "eager ms_per_step) the stage where the stream runs dry is inflated by the host gap; "
                         "libbmv_kernel_ms_per_step (events right around each launch) and the graph replay are not",
        "host_enqueue_ms_per_step": t_host, "instrumented_ms_per_step": ms_instrumented,
        # stages that mix libbmv tensor-core convolution kernels with kept cuDNN layers
        "mixed_library_stage_ms_per_step": {k: v for k, v in step_ms_stage.items() if k.startswith(("cost_reg", "nerf", "feature"))},
        # device time of every libbmv entry point per frame (CUDA events around each launch, instrumented pass)
        "libbmv_kernel_ms_per_step": {e: sum(ts) / args.steps for e, ts in sorted(ksum.items())},
        "libbmv_launches_per_step": {e: len(ts) / args.steps for e, ts in sorted(ksum.items())},
    }
    def _errs(out, ref):
        """Per output: max |a - b| over the frame, the reference's dynamic range max|b|, and their ratio."""
        res = {}
        for k, b in ref.items():
            if k.startswith("_") or k not in out:
                continue
            a = out[k].float().cpu().reshape(-1)
            b = b.float().cpu().reshape(-1)
            rng = float(b.abs().max())
            d = (a - b).abs()
            err = float(d.max())
            # a sample on a frustum edge can flip its visibility count under a 1-ulp change of the depth map (SURVEY.md
            # 10.13; tests/test_gpu_precision.py shows each flip sits on an edge): the element counts tell a handful of
            # such rays from a systematic error
            res[k] = {"max_abs_err": err, "ref_range": rng, "err_over_range": err / max(rng, 1e-30), "elements": d.numel(),
                      "elements_over_1e-4_of_range": int((d > 1e-4 * rng).sum()), "elements_over_1e-2_of_range": int((d > 1e-2 * rng).sum()),
                      "p99.99_err_over_range": float(torch.quantile(d[::max(1, d.numel() // 4000000)], 0.9999)) / max(rng, 1e-30)}
        return res

    cpu_frame = {}
    if world == 1 and not args.no_cpu_baseline:
        rate, cms, sample, cores, size = cpu_reference_rate(wl, rc, 1, 0, args.cpu_budget_s, state_dict=net.state_dict(),
                                                            keep=cpu_frame)
        line["cpu_baseline"] = {"value": rate, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample,
                                "ms_per_step": cms}
        # the CPU frame doubles as the parity reference when it is the workload's own frame (same weights, same scene)
        if cpu_frame.get("_size") == (wl["H"], wl["W"]):
            par = {"reference": "oracle.boost_enerf_forward on the host, fp32, same weights and scene as the timed frames",
                   "definition": "max |ours - ref| / max |ref| per output tensor"}
            if default_out is not None:
                par["default_path"] = _errs(default_out, cpu_frame)
            if strict_out is not None:
                par["strict_fp32_path"] = _errs(strict_out, cpu_frame)
            line["parity_vs_cpu_baseline"] = par
        else:
            line["parity_vs_cpu_baseline"] = {"skipped": "the CPU sample is not the workload's own frame "
                                                         f"({cpu_frame.get('_size')}); raise --cpu-budget-s"}
    if world == 1 and not args.no_torch_gpu_baseline:
        # the reference's own eager-PyTorch op sequence on the same GPU, batch and weights: the
        # "reference single-GPU PyTorch path" of north_star (SURVEY.md §8(d)); with torch defaults (TF32 convolutions)
        # and with TF32 off, each also compared with the CPU frame: the evidence for "TF32-class"
        from oracle import enerf_oracle as O
        kb = torch.tensor([wl["k_best"]], device=dev)
        old_flags = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        tg = {}
        for label, tf32 in (("torch_defaults_tf32_convs", True), ("tf32_off", False)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = False if not tf32 else old_flags[1]
            with torch.no_grad():
                for _ in range(2):
                    ro = O.boost_enerf_forward(net, dict(batch), rc, kb)
                torch.cuda.synchronize()
                e0.record()
                n_ref = max(3, min(args.steps, 10)) if tf32 else 2
                for _ in range(n_ref):
                    ro = O.boost_enerf_forward(net, dict(batch), rc, kb)
                e1.record()
                torch.cuda.synchronize()
            ms_ref = e0.elapsed_time(e1) / n_ref
            tg[label] = {"ms_per_step": ms_ref, "value": rays_per_frame / (ms_ref * 1e-3), "unit": "rays/s", "steps": n_ref,
                         "speedup_of_ours": ms_ref / ms, "speedup_of_ours_e2e": ms_ref / ms_e2e}
            if cpu_frame.get("_size") == (wl["H"], wl["W"]):
                tg[label]["err_vs_cpu_frame"] = _errs({k: v.detach() for k, v in ro.items()}, cpu_frame)
            del ro
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_flags
        tg["what"] = ("oracle.boost_enerf_forward (the reference's op sequence as eager PyTorch, cuDNN/cuBLAS) on the same "
                      "GPU, weights and batch; north_star's >=20x target is against torch_defaults_tf32_convs")
        line["torch_gpu_reference_path"] = tg
    if args.stage_report:
        for k, v in sorted(step_ms_stage.items(), key=lambda kv: -kv[1]):
            print(f"  {k:24s} {v:9.3f} ms/step", file=sys.stderr)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------ MVSNeRF arm (config 3)
def mvs_workload_config(name, wl):
    return {"workload": f"{name}: MVSNeRF + BoostMVSNeRFs K={wl['K']} cost volumes, {wl['W']}x{wl['H']} (960x540 padded to /32), "
                        f"N={wl['n_views']} source views, {wl['D']} depth planes and samples per ray, bf16 cost volume, "
                        "random-init weights",
            "e2e_inputs": "pinned host: N source images + cameras + rays (R,8), uploaded every step; rgb + depth read back",
            "l2": "no explicit flush: one frame streams > 5 GB through HBM (4 x 556 MB cost volumes alone)",
            "timing": "CUDA events on the launch stream around exactly `steps` frames, max over ranks"}


def mvs_cpu_rate(wl, rc, budget_s, steps=1):
    """oracle.boost_mvsnerf_forward on the host at the largest listed resolution that fits the budget (the full C3 frame
    takes ~11 minutes on 8 cores: BASELINE.md)."""
    import torch
    from boostmvsnerfs_b200.modules_mvs import MvsnerfModules
    from boostmvsnerfs_b200.synth import make_scene
    from oracle import mvsnerf_oracle as M
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    net = MvsnerfModules().eval()
    kb = torch.tensor([wl["k_best"]])

    def run(h, w):
        scene = make_scene(H=h, W=w, n_views=wl["n_views"], seed=0, render_scales=(1.0,), mvs_near_far_cols=True)
        t0 = time.perf_counter()
        with torch.no_grad():
            M.boost_mvsnerf_forward(net, scene, rc, kb)
        return time.perf_counter() - t0
    t_probe = run(32, 64)
    rate = 32 * 64 / t_probe
    size = (32, 64)
    for h, w in [(wl["H"], wl["W"]), (288, 480), (128, 192), (64, 96)]:
        if 1.3 * h * w / rate <= budget_s / max(1, steps):
            size = (h, w)
            break
    ts = [run(*size) for _ in range(steps)]
    dt = sum(ts) / len(ts)
    sample = (f"{steps} frame(s) of K={wl['K']} N={wl['n_views']} D=S={wl['D']} at {size[1]}x{size[0]} ({size[0] * size[1]} rays) "
              f"through oracle.boost_mvsnerf_forward, torch {torch.__version__} CPU")
    return size[0] * size[1] / dt, dt * 1e3, sample, cores, size


def main_mvs(args):
    import torch
    from boostmvsnerfs_b200 import _lib
    from boostmvsnerfs_b200.config import RenderConfig
    from boostmvsnerfs_b200.network_mvs import BoostMvsnerfNetwork
    from boostmvsnerfs_b200.synth import batch_to, make_scene
    wl = WORKLOADS[args.workload]
    rc = RenderConfig.mvsnerf_eval(wl["K"], wl["D"])
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            rate, ms, sample, cores, size = mvs_cpu_rate(wl, rc, args.ref_budget_s / max(1, args.steps + args.warmup), 1)
            print(json.dumps({"impl": "reference", "metric": "rays_per_sec", "value": rate, "unit": "rays/s", "n_gpus": args.gpus,
                              "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                              "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": mvs_workload_config(args.workload, wl),
                              "step_sample": {"resolution": [size[1], size[0]], "full_workload_frame": size == (wl["H"], wl["W"])},
                              "cpu_baseline": {"value": rate, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
                              "e2e": {"value": rate, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    torch.manual_seed(0)
    net = BoostMvsnerfNetwork(preprocess=True, rc=rc).eval().to(dev)
    net.view_selection_outputs = {"synth_0": wl["k_best"]}
    net.volume_dtype = torch.bfloat16
    net.mlp_engine = args.mlp_engine if args.mlp_engine in ("umma", "cublas") else "umma"
    host = make_scene(H=wl["H"], W=wl["W"], n_views=wl["n_views"], seed=rank, render_scales=(1.0,), mvs_near_far_cols=True)
    host = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in host.items()}
    batch = batch_to(host, dev)
    rays_per_frame = wl["W"] * wl["H"]
    timer = StageTimer()
    ktimer = KernelTimer(torch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(max(1, args.warmup)):
        out = net(dict(batch))
    clocks = ClockSampler(local)
    clocks.start()
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.time()
    e0.record()
    for _ in range(args.steps):
        out = net(dict(batch))
    e1.record()
    barrier()
    tw1 = time.time()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    ms = e0.elapsed_time(e1) / args.steps
    launches = (_lib.launch_count() - l0) / args.steps
    clk = clocks.stop(tw0, tw1)
    # instrumented pass
    net.stage_timer, _lib.kernel_timer = timer, ktimer
    timer.enabled = ktimer.enabled = True
    for _ in range(max(1, min(args.steps, 3))):
        net(dict(batch))
    barrier()
    n_inst = max(1, min(args.steps, 3))
    net.stage_timer, _lib.kernel_timer = None, None
    stages = {k: v[0] / n_inst for k, v in timer.summary().items()}
    ksum = {k: sum(v) / n_inst for k, v in ktimer.summary().items()}
    kcnt = {k: len(v) / n_inst for k, v in ktimer.summary().items()}
    # end to end: pinned host batch uploaded, rgb + depth read back, every step
    h2d = sum(v.numel() * v.element_size() for v in host.values() if torch.is_tensor(v))
    res_host = {k: torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory() for k in ("rgb_level0", "depth_level0")}
    d2h = sum(v.numel() * v.element_size() for v in res_host.values())
    barrier()
    e0.record()
    for _ in range(args.steps):
        o = net(batch_to(host, dev, non_blocking=True))
        for k, v in res_host.items():
            v.copy_(o[k], non_blocking=True)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1) / args.steps
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
    S, K = wl["D"], wl["K"]
    h, w = wl["H"] // 4 + 48, wl["W"] // 4 + 48
    kernels = {}
    if ksum.get("bmv_mvs_render_umma"):
        per = ksum["bmv_mvs_render_umma"] / K
        flops = 2.0 * 125696.0 * rays_per_frame * S          # MACs per sample of the 6x128 MLP (unpadded), per chain
        kernels["render_fused"] = {"ms_per_launch": per, "launches_per_step": K, "algorithmic_flops": flops,
                                   "tflops": flops / (per * 1e-3) / 1e12, "frac": flops / (per * 1e-3) / 1e12 / peak_tf,
                                   "bound": "tensor", "share_of_step": ksum["bmv_mvs_render_umma"] / ms}
    if ksum.get("bmv_cost_volume_var_img"):
        per = ksum["bmv_cost_volume_var_img"] / K
        nbytes = 41 * S * h * w * 2 + 3 * (32 + 3) * (wl["H"] // 4) * (wl["W"] // 4) * 4
        kernels["cost_volume_img"] = {"ms_per_launch": per, "launches_per_step": K, "algorithmic_bytes": nbytes,
                                      "achieved_gbs": nbytes / (per * 1e-3) / 1e9, "frac": nbytes / (per * 1e-3) / 1e9 / peak_gbs,
                                      "bound": "hbm", "share_of_step": ksum["bmv_cost_volume_var_img"] / ms}
    dom = max(kernels, key=lambda n: kernels[n]["share_of_step"]) if kernels else None
    roofline = None
    if dom:
        k = kernels[dom]
        roofline = ({"kernel": dom, "bound": "tensor", "achieved": k["tflops"], "peak": peak_tf, "unit": "TFLOP/s", "frac": k["frac"],
                     "traffic": None, "launch_ms": k["ms_per_launch"], "share_of_step": k["share_of_step"]} if k["bound"] == "tensor" else
                    {"kernel": dom, "bound": "hbm", "achieved": k["achieved_gbs"], "peak": peak_gbs, "unit": "GB/s", "frac": k["frac"],
                     "traffic": None, "launch_ms": k["ms_per_launch"], "share_of_step": k["share_of_step"]})
    line = {"metric": "rays_per_sec", "value": world * rays_per_frame / (ms * 1e-3), "unit": "rays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "ms_per_frame": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16 cost volume, f16-operand/f32-accum fused MLP (TF32-class), cuDNN TF32 convolutions, f32 elsewhere"
                     if net.mlp_engine == "umma" else "bf16 cost volume, f32 MLP (cuBLAS)",
            "data": "synthetic", "config": mvs_workload_config(args.workload, wl),
            "run": {"mlp_engine": net.mlp_engine, "execution": "eager (stream launches)",
                    "parallelism": "single GPU" if world == 1 else f"{world} frame replicas, no data-path collective"},
            "e2e": {"value": world * rays_per_frame / (ms_e2e * 1e-3), "unit": "rays/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clk, "roofline": roofline, "kernels": kernels,
            "stage_ms_per_step": stages, "libbmv_kernel_ms_per_step": ksum, "libbmv_launches_per_step": kcnt,
            "peak_mem_GB": torch.cuda.max_memory_allocated() / 1e9}
    if world == 1 and not args.no_cpu_baseline:
        rate, cms, sample, cores, size = mvs_cpu_rate(wl, rc, args.cpu_budget_s)
        line["cpu_baseline"] = {"value": rate, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample, "ms_per_step": cms}
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse_args()
    if WORKLOADS[a.workload].get("backbone") == "mvsnerf":
        main_mvs(a)
    elif a.impl == "reference":
        main_reference(a)
    else:
        main_ours(a)
