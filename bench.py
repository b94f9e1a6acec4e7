#!/usr/bin/env python
"""bench.py — frames/s of MaGNet's multi-view matching hot path on B200 (BASELINE.json metric).

One *step* = one pass of the hot path over one batch of synthetic frames per GPU:
    source repack (NCHW -> PIXC: pixel-major features + Gaussians) + camera table  [once per batch, timed]
    N_iter = 3 x ( fused sampler + warp + bilinear sample + consistency + view fusion kernel
                   -> Gaussian update kernel on a fixed synthetic G-Net output )
A *frame* is one reference image's full matching loop (SURVEY §8 d).  Workload at N=1 is BASELINE.json
configs[1]: 640x480 (quarter-res grid 120x160), 4 source views, 64 hypotheses, batch 8 per GPU; N>1 is weak
scaling (each rank owns its own batch of 8; the path has no data-path collective, SURVEY §8 e).

  value     whole-job frames/s, inputs resident in HBM, device-timed (CUDA events), max over ranks
  e2e       same loop through the reference-facing drop-in API (sample_depths + est_costvolume_CW +
            gaussian_update) with pinned HOST buffers: H2D of every input and D2H of the result inside the
            timed region
  roofline  dominant kernel (cost volume): algorithmic bytes / its CUDA-event duration vs measured HBM peak
  cpu_baseline / --impl reference
            the reference's CPU path — its operator sequence as the ATen port oracle/torch_ref.py, pinned bit for bit
            to the reference's own outputs (tests/test_oracle_golden.py) — timed on this box's host cores on a bounded
            sample (1-frame batches)

--dump-outputs DIR writes what the last timed step computed, as float32 .npy files: pred_gmm.npy (B,2,H,W), the
Gaussians after the N_iter iterations, and cost_volume.npy (B,D,H,W), the cost volume of the last iteration.  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "frames/sec (640x480, 4 views, 64 hyp)"
N_ITER = 3
WORKLOADS = {
    "cfg2": "scannet-640x480(q120x160)-V4-D64-B8",
    "cfg3": "kitti-1216x352(q88x304)-V4-D64-B4",
}


def algorithmic_bytes(B, V, D, C, HW, fused=True):
    """SURVEY §8(d): every tensor read or written once, fp32.  S = 2 (mu, sigma) when the sampler is fused,
    D when d_volume is read."""
    S = 2 if fused else D
    return 4 * B * HW * (C + V * C + 2 * V + 3 + S + D)


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload, kind=""):
    """DRAM bytes per launch of the timed cost kernel from the committed ncu --set full capture (profiles/traffic.json:
    keys "<config>:mma" for the tensor-core kernel, "<config>" for the global-gather kernel, "<config>:tma" for the
    TMA-staged one), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(workload + (":" + kind if kind else ""))
    except Exception:
        return None


class ClockSampler:
    """Samples SM clock / throttle reasons DURING the timed region (pynvml; nvidia-smi as a fallback)."""

    def __init__(self, index=0, period=0.004):
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None

    def _decode(self, mask):
        n = self._nvml
        names = {
            "hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(n, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        return {k for k, bit in names.items() if mask & bit}

    def _loop(self):
        n = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM))
                try:
                    mask = n.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                self.reasons |= self._decode(mask)
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self._nvml is not None:
            self._stop.clear()
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
            self._thr = None

    def report(self):
        if self._nvml is None:
            try:
                import subprocess
                out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=10).stdout
                cur, mx = [float(x) for x in out.strip().split(",")]
                return {"sm_mhz": cur, "sm_max_mhz": mx, "reasons": [], "samples": 1, "how": "nvidia-smi after the timed region"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "how": "unavailable"}
        s = sorted(self.samples)
        med = s[len(s) // 2] if s else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s),
                "how": "pynvml, %.0f ms period, during the timed region(s)" % (self.period * 1e3)}


def pin_to_gpu_cpus(index):
    """Pin this process to the CPU cores NVML reports as local to GPU ``index`` (the NUMA node the GPU hangs off): with
    8 ranks on a two-socket host the launch threads otherwise wander across sockets.  Returns the core count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
        allowed = set(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def reference_ops():
    """The reference's cost-volume function for the baseline legs: its ATen port oracle/torch_ref.py, bit-identical to
    models.submodules.homography.est_costvolume_CW — kind "port".  The sampler (MAGNET.py:154-156) and the update
    (MAGNET.py:60-69) are inlined in the reference's forward; they are issued here as the same ATen expressions."""
    from oracle import torch_ref
    return torch_ref.cost_volume_cw, "port", "oracle/torch_ref.py"


def cpu_reference_frames(frames_cfg, steps, warmup, threads=None, budget_s=None):
    """Time the reference's CPU path (sampler -> est_costvolume_CW -> Gaussian update, N_ITER iterations) on 1-frame
    batches of the same workload.  Returns (frames/s, info)."""
    from magnet_b200.synthetic import make_config
    from oracle import torch_ref
    cost_fn, kind, where = reference_ops()
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm must use every host core it may run on.  One thread per
    # PHYSICAL core (what torch picks by default): 128 threads on the 64-core / 128-thread GPU host were
    # measured 8x slower than 64 (oversubscribed hyper-threads).
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or avail
    except Exception:
        phys = avail
    torch.set_num_threads(threads or max(1, min(avail, phys)))
    cores = torch.get_num_threads()
    inp = make_config(frames_cfg, seed=1, B=1)
    klist = [float(v) for v in inp.k.tolist()]
    g = torch.Generator().manual_seed(5)
    raw = torch.randn(1, 2, *inp.ref_feat.shape[2:], generator=g) * 0.1

    def one_frame():
        pred = inp.ref_gmms
        for _ in range(N_ITER):
            dvol = torch_ref.sample_depth_candidates(pred, klist)
            cost_fn(dvol, inp.ref_feat, inp.nghbr_feat, inp.ref_gmms, inp.nghbr_gmms, inp.R, inp.t,
                    inp.is_valid, inp.cam_intrins, inp.thres)
            pred = torch_ref.gaussian_update(raw, pred)
        return pred

    with torch.no_grad():
        for _ in range(warmup):
            one_frame()
        t0 = time.perf_counter()
        done = 0
        for _ in range(steps):
            one_frame()
            done += 1
            if budget_s is not None and time.perf_counter() - t0 > budget_s:
                break
        dt = time.perf_counter() - t0
    what = "ATen port of the reference operator sequence (%s)" % where
    info = {"cores": cores, "os_cpu_count": os.cpu_count(), "frames": done, "seconds": dt, "kind": kind,
            "sample": f"{done} x 1-frame batch of {WORKLOADS[frames_cfg]} (B=1), {N_ITER} iterations each, "
                      f"{what}, {cores} threads"}
    return done / dt, info


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir, outputs):
    """One float32 DIR/<name>.npy per output (every rank computes the same work: rank 0 writes)."""
    import numpy as np
    total = sum(t.numel() * 4 for t in outputs.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy().astype(np.float32, copy=False))


def run_reference_arm(args, rank):
    if rank != 0:
        return
    fps, info = cpu_reference_frames(args.config, max(1, args.steps), max(0, min(args.warmup, 1)), budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": info["frames"], "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * info["seconds"] / max(1, info["frames"]),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.config], "n_iter": N_ITER, "device": "host CPU"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": info["cores"], "kind": info["kind"], "sample": info["sample"]},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--variant", default="auto", choices=["auto", "direct", "cells", "cells_noreuse", "tma", "mma"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gnet", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()

    from magnet_b200 import dist as md
    rank, local_rank, world = md.env_world()
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: magnet_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    md.init_process_group("nccl", device_id=dev)
    K, W = max(1, args.steps), max(3, args.warmup)

    import magnet_b200
    from magnet_b200 import _lib, ops
    from magnet_b200.synthetic import make_config
    variant = {"auto": _lib.VARIANT_AUTO, "direct": _lib.VARIANT_DIRECT, "cells": _lib.VARIANT_CELLS,
               "cells_noreuse": _lib.VARIANT_CELLS_NOREUSE, "tma": _lib.VARIANT_TMA, "mma": _lib.VARIANT_MMA}[args.variant]

    # Weak scaling = the SAME work on every GPU: all ranks build the same seeded batch (each owns its own copy).  With
    # per-rank seeds the step time followed the poses drawn (the kernel's cost depends on how many bilinear cells a
    # depth range crosses): +4 % on rank 1, +10 % on one of ranks 2-3 at the same 1965 MHz — that data variance, not
    # the software, was the 0.91 "scaling efficiency" of round 1 (profiles/r2_scaling.md).
    inp = make_config(args.config, seed=1)
    B, V, D = inp.B, inp.V, inp.D
    C, H, Wd = inp.ref_feat.shape[1], inp.ref_feat.shape[2], inp.ref_feat.shape[3]
    HW = H * Wd
    g = inp.to(dev)
    klist = [float(v) for v in inp.k.tolist()]
    karr = ops.k_array(klist)
    gen = torch.Generator().manual_seed(5)
    raw = (torch.randn(B, 2, H, Wd, generator=gen) * 0.1).to(dev)     # stand-in G-Net output (fixed)
    is_valid_d = inp.is_valid.to(dev)
    intM_d = inp.cam_intrins['intM'].to(dev)
    rays_d = inp.cam_intrins['unit_ray_array_2D'].to(dev).contiguous()
    # production (auto): the tensor-core kernel on fp16 hi/lo planes when C == 64; TMA-staged kernel: PIXC;
    # global-gather kernels: TILED32
    split = variant == _lib.VARIANT_MMA or (variant == _lib.VARIANT_AUTO and C == 64 and V <= 16)
    pixc = variant == _lib.VARIANT_TMA
    layout = _lib.SRC_SPLIT16 if split else (_lib.SRC_PIXC if pixc else _lib.SRC_TILED32)
    kind = "mma" if split else ("tma" if pixc else "")
    ref_split = None
    if split:
        src_packed = torch.empty(int(_lib.lib().magnet_split16_bytes(V * B, H, Wd)), device=dev, dtype=torch.uint8)
        ref_split = torch.empty(int(_lib.lib().magnet_split16_bytes(B, H, Wd)), device=dev, dtype=torch.uint8)
    elif pixc:
        src_packed = torch.empty(V * B, H, Wd, C + 4, device=dev)
    else:
        src_packed = torch.empty(V * B, H, (Wd + 31) // 32, C // 4, 32, 4, device=dev)
    cv = torch.empty(B, D, H, Wd, device=dev)
    ev_pairs = []

    def hot_step(record=False):
        """repack + camera table + N_ITER x (fused cost kernel -> update kernel); everything device-resident."""
        if split:                                           # both feature sets, once per step
            ops.repack_split16(g.nghbr_feat, g.nghbr_gmms, out=src_packed)
            ops.repack_split16(g.ref_feat, out=ref_split)
        elif pixc:
            ops.repack_pixc(g.nghbr_feat, g.nghbr_gmms, out=src_packed)
        else:
            ops.repack_tiled32(g.nghbr_feat, out=src_packed)
        cams = ops.pack_cameras(intM_d, g.R, g.t, is_valid_d)
        pred = g.ref_gmms
        if record:
            # let the host run ahead of the device (a ~0.15 ms spin kernel): otherwise the first e0..e1 interval of a
            # step also contains the time the host needs to marshal and enqueue the launch (the GPU idles between the
            # event and the kernel) and the "kernel time" reads 10 % high
            torch.cuda._sleep(300000)
        for _ in range(N_ITER):
            if record:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            ops.cost_volume(g.ref_feat, src_packed, rays_d, cams, V=V, src_layout=layout, consistency=True,
                            src_gmm=g.nghbr_gmms, kappa=float(inp.thres), ref_gmm=pred, k=karr, out=cv, variant=variant,
                            ref_split=ref_split)
            if record:
                e1.record()
                ev_pairs.append((e0, e1))
            pred = ops.gaussian_update(raw, pred)
        return pred

    def timed(fn, steps, sampler=None):
        md.barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.start()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            fn()
        e.record()
        torch.cuda.synchronize()
        if sampler:
            sampler.stop()
        md.barrier()
        own["ms"] = s.elapsed_time(e)
        return md.max_over_ranks(own["ms"], device=dev)

    own = {"ms": 0.0}
    try:
        full_affinity = os.sched_getaffinity(0)
    except AttributeError:
        full_affinity = None
    affinity = pin_to_gpu_cpus(local_rank)                           # each rank on the cores next to its GPU
    sampler = ClockSampler(index=local_rank)                         # every rank watches its own GPU
    with torch.no_grad():
        for _ in range(W):
            hot_step()
        l0 = _lib.launch_count()
        hot_step()
        launches_per_step = _lib.launch_count() - l0
        torch.cuda.synchronize()
        # The step is launch-latency sensitive (8 short kernels): capture it once per rank in a CUDA graph (SURVEY §7
        # step 5) and time K replays — one host call per step, identical kernels and arguments.
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                graph_pred = hot_step()
        torch.cuda.current_stream().wait_stream(side)
        eager_pred = hot_step()
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize()
        graph_ok = bool(torch.equal(graph_pred, eager_pred))
        ms_total = timed(graph.replay, K, sampler)
        # the graph's output buffers hold the last timed step's results until the next replay or eager step
        outputs = {"pred_gmm": graph_pred.cpu(), "cost_volume": cv.cpu()} if args.dump_outputs else None
        own_ms_step = own["ms"] / K
        launches = launches_per_step * K
        # spread: the same K-step region repeated (median / min / max of the max-over-ranks time per step)
        reps = sorted(timed(graph.replay, K) / K for _ in range(20))
        ms_eager = timed(hot_step, min(K, 50)) / min(K, 50)          # the same step, launched eagerly (one host call per kernel)
        # eager + instrumented: CUDA events around every cost-kernel launch (a graph has no per-kernel events)
        timed(lambda: hot_step(record=True), min(K, 50))
    ms_step = ms_total / K
    frames_per_s = world * B * 1e3 / ms_step
    kern_ms = sum(a.elapsed_time(b) for a, b in ev_pairs) / max(1, len(ev_pairs))
    # per-rank view of the max-over-ranks number: this rank's own step time, cost-kernel time and SM clock under load.
    # (No collective and one graph launch per step: what separates the ranks is the GPU each one runs on.)
    if len(sampler.samples) < 5:
        with torch.no_grad():
            sampler.start()
            t_end = time.time() + 1.0
            while time.time() < t_end:
                graph.replay()
            torch.cuda.synchronize()
            sampler.stop()
    own_clock = sampler.report()
    per_rank_rows = md.gather_over_ranks([own_ms_step, kern_ms, own_clock["sm_mhz"] or 0.0], device=dev)
    per_rank = {"ms_per_step": [r[0] for r in per_rank_rows], "kernel_ms": [r[1] for r in per_rank_rows],
                "sm_mhz_under_load": [r[2] for r in per_rank_rows]}
    repeats = {"regions": len(reps), "median_ms_per_step": reps[len(reps) // 2], "min_ms_per_step": reps[0],
               "max_ms_per_step": reps[-1], "eager_ms_per_step": ms_eager, "graph_equals_eager": graph_ok,
               "cpu_affinity": affinity}
    # ---- loop including the real G-Net convolutions (PyTorch / cuDNN), reported beside the headline --------
    with_gnet = None
    if not args.no_gnet:
        torch.backends.cudnn.benchmark = True                      # as the reference's drivers set it (train_MaGNet.py:56)
        torch.manual_seed(0)
        head = magnet_b200.GNET(ch_in=256 + D).to(dev).eval()
        x_d3 = torch.randn(B, 256, H, Wd, device=dev)

        def gnet_step():
            plan = magnet_b200.MatchingPlan(g.ref_feat, g.nghbr_feat, g.nghbr_gmms, g.nghbr_poses, is_valid_d,
                                            {"intM": intM_d, "unit_ray_array_2D": rays_d}, thres=inp.thres)
            return magnet_b200.matching_loop(plan, g.ref_gmms, x_d3, head if split else head.gnet, N_ITER, karr,
                                             variant=variant)[-1]

        res = {}
        with torch.no_grad():
            for split in (False, True):
                for _ in range(3):
                    gnet_step()
                kg = max(3, K // 10)
                res[split] = timed(gnet_step, kg) / kg
        ms_g = res[True]
        with_gnet = {"value": world * B * 1e3 / ms_g, "unit": "frames/s", "ms_per_step": ms_g,
                     "reference_dataflow_ms_per_step": res[False],
                     "note": "same loop + G-Net conv head (cuDNN, fp32) on a random 256-ch D-Net feature; headline = "
                             "x_d3 half of the first conv hoisted out of the loop (no per-iteration cat), "
                             "reference_dataflow = cat([cost, x_d3]) every iteration as MAGNET.py:167"}

    # ---- e2e: drop-in API, pinned host buffers, H2D + D2H inside the timed region ---------------------------
    # Every step copies ALL of its inputs host -> device and its result device -> host.  The copies of step s+1 run
    # on a second stream into the other of two device buffer sets while step s computes (what a serving loop does);
    # the host "reads" result s-1 (waits for its D2H event) before it enqueues step s+1.
    names = ("ref_feat", "nghbr_feat", "ref_gmms", "nghbr_gmms", "nghbr_poses")
    host = {k: getattr(inp, k).contiguous().pin_memory() for k in names}
    dbuf = [{k: torch.empty_like(host[k], device=dev) for k in names} for _ in range(2)]
    out_host = [torch.empty(B, 2, H, Wd).pin_memory() for _ in range(2)]
    h2d = sum(t.numel() * t.element_size() for t in host.values())
    d2h = out_host[0].numel() * out_host[0].element_size()
    copy_stream = torch.cuda.Stream(device=dev)
    ev_ready = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    ev_done = [torch.cuda.Event() for _ in range(2)]
    e2e_variant = _lib.VARIANT_AUTO if variant == _lib.VARIANT_CELLS_NOREUSE else variant
    state = {"s": 0}

    def enqueue_h2d(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[i])                     # previous user of this buffer set is done
            for k in names:
                dbuf[i][k].copy_(host[k], non_blocking=True)
            ev_ready[i].record(copy_stream)

    def e2e_compute(i):
        cur = torch.cuda.current_stream()
        cur.wait_event(ev_ready[i])
        d = dbuf[i]
        R, t = d["nghbr_poses"][:, :, :3, :3], d["nghbr_poses"][:, :, :3, 3]
        pred = d["ref_gmms"]
        for _ in range(N_ITER):
            dvol = ops.sample_depths(pred, karr)
            magnet_b200.est_costvolume_CW(dvol, d["ref_feat"], d["nghbr_feat"], d["ref_gmms"], d["nghbr_gmms"],
                                          R, t, inp.is_valid, inp.cam_intrins, inp.thres, variant=e2e_variant)
            pred = ops.gaussian_update(raw, pred)
        out_host[i].copy_(pred, non_blocking=True)
        ev_done[i].record(cur)
        ev_free[i].record(cur)

    def e2e_step():
        s = state["s"]
        i = s & 1
        if s == 0:
            enqueue_h2d(0)                                         # prologue of the pipeline
        enqueue_h2d(i ^ 1)                                         # inputs of step s+1 (copied every step)
        e2e_compute(i)
        if s > 0:
            ev_done[i ^ 1].synchronize()                           # the caller reads result s-1 on the host
        state["s"] = s + 1

    def e2e_run(steps):
        """steps e2e steps incl. the drain of the last result; one extra H2D is in flight at the end."""
        for _ in range(steps):
            e2e_step()
        ev_done[(state["s"] - 1) & 1].synchronize()

    with torch.no_grad():
        for e in ev_free:
            e.record()
        e2e_run(3)
        torch.cuda.synchronize()
        # K steps per timed region (the same K as the device-timed arm); regions are repeated until at least 0.5 s of e2e
        # work AND at least 5 regions have been timed, the MEDIAN region is reported (max over ranks per region)
        ke = K
        regions = []
        total_ms = 0.0
        while (total_ms < 500.0 or len(regions) < 5) and len(regions) < 50:
            md.barrier()
            torch.cuda.synchronize()
            t_s, t_e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_s.record()
            e2e_run(ke)
            torch.cuda.synchronize()                               # includes the copy stream
            t_e.record()
            torch.cuda.synchronize()
            md.barrier()
            ms_r = md.max_over_ranks(t_s.elapsed_time(t_e), device=dev)
            regions.append(ms_r / ke)
            total_ms += ms_r
        regions.sort()
        ms_e = regions[len(regions) // 2]
    e2e = {"value": world * B * 1e3 / ms_e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "ms_per_step": ms_e, "api": "sample_depths + est_costvolume_CW (drop-in, d_volume mode) + gaussian_update",
           "steps": ke, "regions": len(regions), "min_ms_per_step": regions[0], "max_ms_per_step": regions[-1],
           "pipeline": "double-buffered: H2D of step s+1 on a copy stream overlaps the kernels of step s"}

    if rank != 0:
        md.shutdown()
        return
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    peak, peak_src = measured_peak()
    abytes = algorithmic_bytes(B, V, D, C, HW, fused=True)
    achieved = abytes / (kern_ms * 1e-3) / 1e9
    info_variant = _lib.VARIANT_MMA if split else (_lib.VARIANT_CELLS if variant in (_lib.VARIANT_CELLS_NOREUSE, _lib.VARIANT_AUTO) else variant)
    grid, block, smem = ops.cost_launch_info(B, V, D, C, H, Wd, variant=info_variant)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(args.config, kind), "kernel": "cost_mma_kernel<GAUSS,CW> (SPLIT16 planes, tcgen05.mma + TMA windows)" if split else {_lib.VARIANT_DIRECT: "cost_direct_kernel<CW>", _lib.VARIANT_CELLS: "cost_cells_kernel<64,GAUSS,CW> (TILED32 gather)",
                           _lib.VARIANT_CELLS_NOREUSE: "cost_cells_kernel<64,GAUSS,CW,noreuse>",
                           _lib.VARIANT_TMA: "cost_tma_kernel<64,GAUSS,CW> (PIXC layout, TMA-staged window)"}.get(
                               variant, "cost_cells_kernel<64,GAUSS,CW> (TILED32 gather)"),
                "kernel_ms_how": "CUDA events around every cost-kernel launch of %d eager steps run right after the "
                                 "graph-replayed timed region (same kernels, arguments and buffers; a 0.15 ms spin kernel "
                                 "at the start of each instrumented step lets the host enqueue ahead, so the intervals "
                                 "hold device time only)" % min(K, 50),
                "kernel_ms": kern_ms, "kernel_ms_max_over_ranks": max(per_rank["kernel_ms"]),
                "algorithmic_bytes_per_launch": abytes, "peak_source": peak_src,
                "launch": {"grid": grid, "block": block, "smem_bytes": smem}}
    # ---- reference-CUDA baseline (north_star / BASELINE.md §2): the reference's operator sequence (repeat,
    # grid_sample, mul, sum ... — ATen port, bit-identical to the reference on CPU) on the same B200, same inputs
    reference_cuda = None
    if world == 1 and not args.no_cpu_baseline:
        ref_cost_fn, ref_kind, _ = reference_ops()
        torch.backends.cuda.matmul.allow_tf32 = False
        dvol_ref = ops.sample_depths(g.ref_gmms, karr)
        cam_dev = {"intM": intM_d, "unit_ray_array_2D": rays_d}

        def ref_call():
            return ref_cost_fn(dvol_ref, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms, g.R, g.t,
                               inp.is_valid, cam_dev, inp.thres)

        with torch.no_grad():
            ref_out = ref_call()
            ours_out = magnet_b200.est_costvolume_CW(dvol_ref, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms, g.R,
                                                     g.t, inp.is_valid, inp.cam_intrins, inp.thres)
            scale = float(ref_out.abs().max())
            frac_diff = float(((ours_out - ref_out).abs() > 1e-4 * scale).float().mean())
            torch.cuda.synchronize()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            for _ in range(3):
                ref_call()
            r1.record()
            torch.cuda.synchronize()
            o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            o0.record()
            for _ in range(10):
                magnet_b200.est_costvolume_CW(dvol_ref, g.ref_feat, g.nghbr_feat, g.ref_gmms, g.nghbr_gmms, g.R, g.t,
                                              inp.is_valid, inp.cam_intrins, inp.thres)
            o1.record()
            torch.cuda.synchronize()
        ms_ref = r0.elapsed_time(r1) / 3
        reference_cuda = {"ms_per_cost_volume": ms_ref, "frames_per_s_cost_only": B * 1e3 / (N_ITER * ms_ref),
                          "ours_ms_per_cost_volume_drop_in": o0.elapsed_time(o1) / 10,
                          "frac_elements_beyond_1e-4": frac_diff, "kind": ref_kind,
                          "note": "est_costvolume_CW of the reference on CUDA tensors (stock ATen "
                                  "grid_sample / repeat / elementwise kernels), same B=%d batch; frames/s counts %d such "
                                  "calls per frame and nothing else" % (B, N_ITER)}
        del ref_out, ours_out
        torch.cuda.empty_cache()

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        if full_affinity is not None:
            os.sched_setaffinity(0, full_affinity)                   # the CPU arm may use every host core again
        fps, info = cpu_reference_frames(args.config, steps=8, warmup=1, budget_s=20.0)
        cpu_baseline = {"value": fps, "unit": "frames/s", "cores": info["cores"], "kind": info["kind"], "sample": info["sample"]}
    line = {
        "metric": METRIC, "value": frames_per_s, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOADS[args.config], "frames_per_step_per_gpu": B, "n_iter": N_ITER, "views": V,
                   "hypotheses": D, "channels": C, "grid": [H, Wd], "depth": inp.meta["depth"], "variant": args.variant,
                   "cache": "inputs_larger_than_l2 (%.0f MB resident per step vs 126 MB L2)" % ((abytes + 4 * V * B * C * HW) / 1e6),
                   "step": "repack + camera table + %d x (fused cost kernel + update kernel), one CUDA graph per rank, "
                           "K replays timed" % N_ITER},
        "clocks": own_clock,
        "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
        "reference_cuda": reference_cuda, "with_gnet": with_gnet, "repeats": repeats, "per_rank": per_rank,
        "gpu_launches_how": "%d kernels per step (counted by the library on an eager step) x %d graph replays" % (
            launches_per_step, K),
    }
    print(json.dumps(line), flush=True)
    md.shutdown()


if __name__ == "__main__":
    main()
