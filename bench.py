#!/usr/bin/env python
"""bench.py -- headline benchmark of the g4d hot path (BASELINE.json: render FPS & train-step ms @300k Gaussians,
1352x1014, HBM GB/s vs roofline), one JSON line on stdout.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA path through the public API)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU implementation of the path
    python bench.py --workload C1|C2|C3|C4                   # other BASELINE.json configs (default C3, the metric's)
    python bench.py --dump-outputs DIR ...                   # also write the outputs of the last timed step (DIR/*.npy)

A "step" is one pass of the hot path over one BATCH of synthetic views: `--views-per-step` (default 32) fused
deform + rasterize FORWARDS of the workload, back to back -- so that `--steps 20` times >= 0.5 s of device work instead of
20 ms.  Views / timestamps are sharded over ranks with no data-path collective (weak scaling, SURVEY 8e); the per-step
NCCL gradient all-reduce only exists in the training step, reported in `train_step` (B=2 views fwd+bwd + fused
L1 loss + flat-bucket all-reduce + Adam).

Timing: one CUDA-event pair per step on the launching stream, W warm-up steps (same code path and the same output
bindings as the timed steps), an L2 flush (512 MiB write) between steps outside the event pairs -- inside a step every
view moves ~0.3 GB (instance lists + images), more than the 126 MB L2, so consecutive views evict one another --
barrier + synchronize on both sides of the timed region, MAX over ranks.
`value` = inputs resident in HBM; `e2e` = the same steps through the public `render()` with the camera arriving from host
memory and every rendered image copied to pinned host memory (double-buffered, on a copy stream, inside the step's event
pair: reference render.py:59-60 semantics).
"""
from __future__ import annotations

import argparse
import gc
import importlib
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

UNIT = "frames/s"
NETS = {   # C (channels), L (levels), Wd, heads (k outputs) per reference config (SURVEY 8a)
    "dnerf": dict(C=32, L=2, Wd=64, heads=(3, 3, 4)),
    "hypernerf": dict(C=16, L=3, Wd=128, heads=(3, 3, 4)),
    "dynerf": dict(C=16, L=2, Wd=128, heads=(3, 3, 4, 1, 48)),
}
WORKLOAD_TEXT = {
    "C1": "C1: D-NeRF bouncingballs shape, 70k Gaussians, 800x800, dnerf net (C=32,L=2,T=75,Wd=64,3 heads)",
    "C2": "C2: HyperNeRF vrig-broom shape, 200k Gaussians, 536x960, hypernerf net (C=16,L=3,T=100,Wd=128,3 heads)",
    "C3": "C3: 300k Gaussians, 1352x1014, dynerf net (C=16,L=2,T=150,Wd=128,5 heads), sh_degree 3, 300 timestamps, "
          "views sharded over ranks",
    "C4": "C4: stress, 2M Gaussians, 64 cams 1920x1080, dynerf net, views sharded over ranks",
}


def metric_name(wl):
    w = importlib.import_module("4dgaussians_b200.synth").WORKLOADS[wl]
    return "render FPS @%dk gauss %dx%d (fused deform+rasterize forward); train-step ms in `train_step`" % (
        w["n"] // 1000, w["width"], w["height"])


def _peaks_json():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def _hbm_peak():
    j = _peaks_json()
    if "hbm_gbs" in j:
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def mlp_flops_per_gaussian(net):
    c = NETS[net]
    F, Wd, h = c["C"] * c["L"], c["Wd"], len(c["heads"])
    return 2.0 * (F * Wd + h * Wd * Wd + Wd * sum(c["heads"]))


def _tensor_roofline(net, n, geom_ms):
    """The geometry kernel is bound by the tensor pipe + its epilogues, not by HBM: report it against the measured dense
    BF16 peak too.  Algorithmic FLOPs = 2 * (F*Wd + h*Wd^2 + Wd*sum(k)) per Gaussian (SURVEY 8d)."""
    j = _peaks_json()
    if "bf16_tflops_sustained" in j:
        peak, src = float(j["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    else:
        peak, src = 2250.0, "fallback (nominal dense bf16 2.25 PFLOP/s)"
    flops = mlp_flops_per_gaussian(net) * n
    ach = flops / (geom_ms * 1e-3) / 1e12 if geom_ms > 0 else 0.0
    return {"bound": "tensor", "kernel": "deform_features + deform_f16_kernel (stage `geom`: HexPlane gather, then the fused "
                                         "deform MLP + activations + projection + SH colour on tcgen05)", "achieved": ach, "peak": peak,
            "unit": "TFLOP/s", "frac": ach / peak if peak else None, "peak_source": src, "algorithmic_flops": flops,
            "kernel_ms": geom_ms,
            "note": "fp32-accurate FP16x2 operands: every algorithmic MAC is 3 tensor-core MACs at the f16 rate, so the ceiling "
                    "of this scheme is peak/3 (frac 0.333) -- 0.28 with the measured 76-cycle 128x128x16 dispatch; net_width 64 "
                    "(dnerf) runs the FP32 FFMA kernel"}


def _blend_roofline(pairs, blend_ms, sm_count):
    """Blend is FP32-ALU / MUFU bound (SURVEY 7): (pixel, instance) evaluations per second against the SM peaks.
    pairs = sum over pixels of the index of the last instance the pixel had to look at (n_contrib) = the evaluations the
    reference algorithm performs; 27 flop + 1 ex2 each (dx,dy; quadratic form; exp; alpha clamp/tests; T update; 4 FMA)."""
    j = _peaks_json()
    mhz = float(j.get("sm_max_mhz", 1965.0))
    fp32 = sm_count * 128 * 2 * mhz * 1e6           # flop/s
    mufu = sm_count * 16 * mhz * 1e6                # ex2/s
    peak_pairs = min(fp32 / 27.0, mufu)
    ach = pairs / (blend_ms * 1e-3) if blend_ms > 0 else 0.0
    return {"bound": "fp32 alu / mufu", "kernel": "blend_forward_kernel", "achieved": ach / 1e9, "peak": peak_pairs / 1e9,
            "unit": "G(pixel x instance)/s", "frac": ach / peak_pairs if peak_pairs else None, "pairs_per_view": pairs,
            "kernel_ms": blend_ms, "fp32_bound_gpairs": fp32 / 27.0 / 1e9, "mufu_bound_gpairs": mufu / 1e9,
            "note": "27 flop + 1 MUFU.EX2 per evaluated pair; peaks = %d SMs x 128 FP32 lanes x 2 / x 16 MUFU lanes at %.0f MHz"
                    % (sm_count, mhz)}


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region.  In-process NVML (three light queries every 200 ms from a thread;
    ctypes drops the GIL during the calls); falls back to a low-rate `nvidia-smi -lms` subprocess when pynvml is unusable."""
    Q = "index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index: int):
        self.index, self.sm, self.mx, self.reasons, self.proc, self.nvml, self._stop = index, [], [], set(), None, None, False
        self.source = None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        return pynvml, h

    def start(self):
        try:
            self.nvml, self.handle = self._nvml_handle()
            self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM)
            self.source = "nvml"
            threading.Thread(target=self._poll_nvml, daemon=True).start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi -lms 100"
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        while not self._stop:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)))
                try:
                    r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    r = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                for name, bit in self.BITS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.2)       # NVML queries occasionally stall the driver for milliseconds: keep them rare

    def _pump(self):
        for line in self.proc.stdout:
            c = [x.strip() for x in line.split(",")]
            if len(c) >= 7 and c[1].replace(".", "").isdigit():
                self.sm.append(float(c[1])); self.mx.append(float(c[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)

    def mark(self):
        """start of the timed region: earlier samples (NVML warm-up, GPU idle) are dropped"""
        self.sm, self.mx, self.reasons = [], [], set()

    def stop(self):
        self._stop = True
        if self.proc is not None:
            self.proc.terminate()
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock source (pynvml / nvidia-smi unavailable or disabled)"]}
        sm_sorted = sorted(self.sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []      # under load = upper half of the samples
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": self.source}


def build_scene(workload, seed=0):
    g4d = importlib.import_module("4dgaussians_b200")
    synth = importlib.import_module("4dgaussians_b200.synth")
    w = synth.WORKLOADS[workload]
    scene = synth.make_scene(w["n"], seed=seed, scale_mean=w["scale_mean"])
    torch.manual_seed(seed)
    mod = g4d.deform_network(synth.hidden_args(w["net"]))
    synth.perturb_deformation(mod, seed)
    mod.deformation_net.set_aabb(scene["aabb"][0].tolist(), scene["aabb"][1].tolist())
    return g4d, synth, w, scene, mod


def algorithmic_bytes(n, H, W, R, param_bytes):
    """SURVEY 8d B_fwd per view and its per-stage split."""
    geom = n * 236 + n * 4 + param_bytes           # SoA read once + radii + planes/MLP read once
    binning = R * (8 + 4) * 2                      # one (key,id) record written then read
    blend = R * 44 + H * W * 16                    # per-instance fetch + colour/depth write
    return {"geom": geom, "binning": binning, "blend": blend, "total": geom + binning + blend}


class Pipe:
    convert_SHs_python = False
    compute_cov3D_python = False
    debug = False


def _max_over_ranks(dist, dev, x):
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the g4d path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        # keep stdout to the one JSON line: NCCL prints its version banner to stdout at levels VERSION and WARN
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    wl = args.workload
    g4d, synth, w, scene, mod = build_scene(wl)
    lib = g4d._lib
    mod = mod.to(dev)
    pc = synth.SyntheticGaussianModel(scene, mod, device=dev, sh_degree=3, requires_grad=False)
    K, Wm, V = args.steps, args.warmup, args.views_per_step
    ncams = 64 if wl == "C4" else 300
    cams_all = synth.orbit_cameras(ncams, w["width"], w["height"], radius=w["radius"], focal=w["focal"], timestamps=300)

    def cam_of(step, v):   # global view index -> this rank's camera (round robin over ranks)
        return cams_all[((step * V + v) * world + rank) % len(cams_all)]
    bg = torch.tensor(w["bg"], dtype=torch.float32, device=dev)
    ws = lib.Workspace.get(local)
    # per-stage CUDA events (ten cudaEventRecord per view, each a break in the programmatically dependent launch chain) are
    # recorded for ONE view of every timed step (the last) and for the untimed per-stage pass below, not for every view
    ws.set_option(lib.OPT_STAGE_TIMING, 0)
    ws.set_option(lib.OPT_SYNC_MODE, 1 if args.host_sync else 0)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    H, Wd = w["height"], w["width"]
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ------------------------------------------------------------------ resident arm (`value`)
    def resident_step(step, kept=None):
        out = None
        if kept is not None:
            kept.clear()      # the previous step's outputs go back to the allocator before this step allocates its own
        for v in range(V):
            if v == V - 1:
                ws.set_option(lib.OPT_STAGE_TIMING, 1)
            out = g4d.render(cam_of(step, v), pc, Pipe, bg)      # same binding in warm-up and timed steps
            if kept is not None:
                kept.append(out)
        ws.set_option(lib.OPT_STAGE_TIMING, 0)
        return out

    # --dump-outputs: every step (warm-up included, so that the allocator is warm) keeps its views' outputs until the next
    kept = [] if args.dump_outputs else None

    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    sampler = ClockSampler(local)
    if rank == 0 and not os.environ.get("G4D_BENCH_NO_SAMPLER"):
        sampler.start()          # NVML initialisation / first queries happen during the warm-up, not in the timed region
    with torch.no_grad():
        for i in range(Wm):
            flush.fill_(i & 0xFF)
            out = resident_step(i, kept)
        gc.collect(); gc.disable()     # a host hiccup shows up 1:1 in a ~1 ms view
        barrier()
        # ranks leave the collective barrier at different times and an idle B200 drops its clocks within milliseconds:
        # one more untimed step, then the synchronize that brackets the timed region
        out = resident_step(Wm, kept)
        torch.cuda.synchronize(dev)
        sampler.mark()
        t_wall0 = time.perf_counter()
        for i in range(K):
            flush.fill_(i & 0xFF)
            ev[i][0].record()
            out = resident_step(Wm + i, kept)
            ev[i][1].record()
        barrier()
        t_wall = time.perf_counter() - t_wall0
        gc.enable()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    if kept is not None:
        if rank == 0:
            dump_outputs(args.dump_outputs, kept)
        kept = None
    # the stage events of the last view of the last timed step (same context: no-grad renders release it at once)
    in_region_stage_ms = ws._free_contexts[-1].stage_times() if ws._free_contexts else {}
    total_ms = _max_over_ranks(dist, dev, sum(step_ms))
    value = world * K * V / (total_ms / 1e3)

    # ------------------------------------------------------------------ host enqueue time per view (is the loop host bound?)
    with torch.no_grad():
        torch.cuda.synchronize(dev)
        t_h0 = time.perf_counter()
        resident_step(Wm)
        t_h1 = time.perf_counter()
        torch.cuda.synchronize(dev)
        t_h2 = time.perf_counter()
    host_enqueue_ms = (t_h1 - t_h0) / V * 1e3
    host_total_ms = (t_h2 - t_h0) / V * 1e3

    # ------------------------------------------------------------------ per-stage device times, R, blend work (untimed pass)
    stage_acc, Rs, vis, pairs = {}, [], [], []
    ws.set_option(lib.OPT_STAGE_TIMING, 1)
    with torch.no_grad():
        for i in range(min(V, 8)):
            g4d.render(cam_of(Wm, i), pc, Pipe, bg)
            torch.cuda.synchronize(dev)
            fn_ctx = ws._free_contexts[-1] if ws._free_contexts else None
            if fn_ctx is not None:
                for k_, v_ in fn_ctx.stage_times().items():
                    stage_acc[k_] = stage_acc.get(k_, 0.0) + v_
                s_ = fn_ctx.stats()
                Rs.append(int(s_.num_rendered)); vis.append(int(s_.num_visible))
                if i < 2:
                    pairs.append(float(fn_ctx.read("n_contrib").astype(np.float64).sum()))

    ws.set_option(lib.OPT_STAGE_TIMING, 0)

    # ------------------------------------------------------------------ e2e arm: host camera in, image out to pinned host
    pinned = [torch.empty(3, H, Wd, dtype=torch.float32).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream(dev)
    main_stream = torch.cuda.current_stream(dev)
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    done = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_step(step):
        for v in range(V):
            out = g4d.render(cam_of(step, v), pc, Pipe, bg)      # camera matrices are HOST tensors -> kernel params
            img = out["render"]
            rendered = torch.cuda.Event(); rendered.record(main_stream)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(rendered)
                pinned[v & 1].copy_(img, non_blocking=True)      # (stream order: this buffer's previous copy has completed)
                img.record_stream(copy_stream)
                done[v & 1].record(copy_stream)
        main_stream.wait_event(done[0]); main_stream.wait_event(done[1])   # the step ends when its last image is on the host

    with torch.no_grad():
        e2e_step(0)
        barrier()
        e2e_step(1)
        torch.cuda.synchronize(dev)
        for i in range(K):
            flush.fill_(i & 0xFF)
            ev2[i][0].record()
            e2e_step(Wm + i)
            ev2[i][1].record()
        barrier()
    e2e_steps = [a.elapsed_time(b) for a, b in ev2]
    e2e_ms = _max_over_ranks(dist, dev, sum(e2e_steps))
    e2e_value = world * K * V / (e2e_ms / 1e3)
    cam_bytes = 4 * (16 + 16 + 3 + 3 + 4) + 16

    # ------------------------------------------------------------------ frame 0 of this workload against the CPU oracle (untimed)
    parity = None
    if rank == 0 and not args.no_parity_check:
        parity = parity_check(g4d, synth, wl, w, scene, mod, pc, cams_all[0], dev)

    # ------------------------------------------------------------------ training step (B=2 views, fwd+bwd, all-reduce, Adam)
    train = None
    if not args.no_train:
        train = run_train_steps(g4d, synth, lib, w, scene, mod, dev, dist, world, rank, K, 5, flush)
    clocks = sampler.stop() if rank == 0 else None     # sampled from the start of the timed region to the end of the train steps

    eager = None
    if rank == 0 and world == 1 and not args.no_eager_baseline:
        eager = gpu_eager_baseline(g4d, synth, w, scene, mod, dev)

    if rank == 0:
        peak, peak_src = _hbm_peak()
        R = float(np.mean(Rs)) if Rs else 0.0
        pbytes = sum(p.numel() * 4 for p in mod.flat_parameters())
        ab = algorithmic_bytes(w["n"], H, Wd, R, pbytes)
        stages = {k_: v_ / max(1, len(Rs)) for k_, v_ in stage_acc.items()}
        fwd_stages = {k_: stages.get(k_, 0.0) for k_ in ("prep", "geom", "scan", "emit", "sort", "ranges", "blend")}
        bin_ms = sum(fwd_stages[k_] for k_ in ("scan", "emit", "sort", "ranges"))
        dom = max(("geom", "blend", "binning"), key=lambda k_: bin_ms if k_ == "binning" else fwd_stages.get(k_, 0.0))
        dom_bytes = ab[dom]
        dom_ms = bin_ms if dom == "binning" else fwd_stages[dom]
        achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        traffic, traffic_src = None, None
        try:     # dram bytes per launch of the dominant kernel from the committed ncu --set full capture of this workload
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if tj.get("workload", "C3") == wl and dom in tj["per_stage"]:
                traffic, traffic_src = float(tj["per_stage"][dom]), tj["source"]
        except Exception:
            pass
        ms_per_view = total_ms / (K * V)
        srt = sorted(step_ms)
        # headline roofline = the geometry kernel (the one VERDICT.md r1 names).  It does 780 algorithmic flop per byte of its
        # SURVEY-8d traffic, far above the machine balance (1442 TFLOP/s / 6.5 TB/s = 222 flop/B): its roof is the tensor pipe,
        # so `bound` is "tensor"; the HBM view of the same stage is kept next to it (geom_hbm_*), DRAM traffic from ncu.
        geom_ms = fwd_stages.get("geom", 0.0)
        if NETS[w["net"]]["Wd"] == 128 and geom_ms > 0:
            roofline_main = _tensor_roofline(w["net"], w["n"], geom_ms)
            gt = None
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
                if tj.get("workload", "C3") == wl:
                    gt = float(tj["per_stage"]["geom"])
            except Exception:
                pass
            roofline_main.update({"traffic": gt, "traffic_unit": "bytes of DRAM per launch pair (ncu --set full, cold caches)",
                                  "geom_hbm_algorithmic_bytes": ab["geom"],
                                  "geom_hbm_achieved_gbs": ab["geom"] / (geom_ms * 1e-3) / 1e9,
                                  "geom_hbm_frac": ab["geom"] / (geom_ms * 1e-3) / 1e9 / peak if peak else None})
        else:
            roofline_main = {"bound": "hbm", "kernel": "deform_kernel (FP32 FFMA, net_width 64)" if dom == "geom" else dom,
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                             "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes": dom_bytes, "kernel_ms": dom_ms}
        line = {
            "metric": metric_name(wl), "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_TEXT[wl], "views_per_step": V, "n_gaussians": w["n"], "width": Wd, "height": H,
                       "focal_px": w["focal"], "orbit_radius": w["radius"], "scale_mean": w["scale_mean"],
                       "tile_instances_R": R, "visible_gaussians": float(np.mean(vis)) if vis else None,
                       "l2": "flushed between timed steps (512 MiB write, outside the event pairs); inside a step each view "
                             "moves ~%.2f GB > 126 MB L2" % (ab["total"] / 1e9),
                       "binning": "host sync on R (exact sizing)" if args.host_sync else
                                  "device-side R, capacity-bounded, no host sync (overflow-checked)",
                       "mlp": "tcgen05 FP16x2 forward (hi+lo operands, 3 products, fp32-accurate), BF16x2 tcgen05 backward" if NETS[w["net"]]["Wd"] == 128
                              else "FP32 FFMA (net_width 64)",
                       "launch": "programmatic dependent launch between the kernels of a view" if os.environ.get("G4D_PDL", "1") != "0"
                                 else "ordinary stream order (G4D_PDL=0)",
                       "parallelism": "scene replicated, views sharded (dp%d)" % world},
            "ms_per_view": ms_per_view,
            "host_enqueue_ms_per_view": host_enqueue_ms, "host_enqueue_note": "wall time per view of ENQUEUEING one step (no "
            "synchronisation) vs %.3f ms until the GPU has finished it; the asynchronous instance-count read-backs bound the host's "
            "run-ahead to two views, so a GPU-bound loop shows the GPU's time here (the Python side itself costs ~0.25 ms per view: "
            "tools/host_profile.py)" % host_total_ms,
            "step_ms_stats": {"mean": float(np.mean(step_ms)), "median": float(np.median(step_ms)), "min": srt[0], "max": srt[-1]},
            "step_ms": [round(x, 3) for x in step_ms],
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": cam_bytes * V, "d2h_bytes_per_step": 3 * H * Wd * 4 * V,
                    "step_ms_median": float(np.median(e2e_steps)),
                    "how": "public render() per view, camera from host memory, every image copied to pinned host memory "
                           "(double-buffered, copy stream) inside the step's event pair; the step ends when its last image "
                           "has landed"},
            "gpu_launches": launches_per_view(w["net"]) * K * V,
            "gpu_launches_note": "own kernels per view (fused forward): " + ", ".join(LAUNCH_LIST[0 if NETS[w["net"]]["Wd"] == 128 else 1]),
            "clocks": clocks,
            "roofline": roofline_main,
            "roofline_hbm": {"bound": "hbm", "kernel": {"geom": "deform_features + deform_f16_kernel (fused deform+activate+project, tcgen05)"
                                                        if NETS[w["net"]]["Wd"] == 128 else "deform_kernel (FFMA)",
                                                        "blend": "blend_forward_kernel", "binning": "bin_sort + bin_place + bin_fix"}[dom],
                             "what": "the longest stage of the forward against the HBM roof (SURVEY 8d bytes of that stage)",
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                             "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes": dom_bytes,
                             "kernel_ms": dom_ms},
            "roofline_path": {"what": "whole fused forward, B_fwd of SURVEY 8d", "algorithmic_bytes": ab["total"],
                              "achieved": ab["total"] / (ms_per_view * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                              "frac": ab["total"] / (ms_per_view * 1e-3) / 1e9 / peak},
            "roofline_blend": _blend_roofline(float(np.mean(pairs)) if pairs else 0.0, fwd_stages.get("blend", 0.0), sm_count),
            "stage_ms": stages, "stage_ms_note": "CUDA events on the launching stream around every stage, mean over 8 views rendered right "
            "after the timed region (one view per synchronize); `stage_ms_in_timed_region` = the same events for the last view of the "
            "last timed step (events are recorded for one view per timed step only: they break the dependent-launch chain)",
            "stage_ms_in_timed_region": in_region_stage_ms, "binning_ms": bin_ms, "train_step": train, "wall_s_timed_region": t_wall,
            "parity_check": parity, "gpu_eager_baseline": eager,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_reference_arm(wl, steps=2, warmup=1)["cpu_baseline"]
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


DUMP_BYTES = 60 * 10 ** 6      # data of the --dump-outputs files; with their headers they stay under 64 MB


def dump_outputs(path, outs):
    """Writes what render() returned for each view of the last timed step as PATH/<key>.npy, float32, views stacked on the
    first axis.  When the step's outputs exceed DUMP_BYTES, every key keeps the same fraction of each view's elements, at
    positions drawn with a fixed seed: (views, sampled elements), the same positions in every view and in every run."""
    os.makedirs(path, exist_ok=True)
    keys = sorted(outs[0])
    per_view = {k: outs[0][k].numel() for k in keys}
    frac = min(1.0, DUMP_BYTES / (4.0 * len(outs) * sum(per_view.values())))
    for k in keys:
        n = per_view[k]
        m = max(1, int(n * frac))
        if m < n:
            idx = np.sort(np.random.default_rng(0).choice(n, m, replace=False))
            idx = torch.from_numpy(idx).to(outs[0][k].device)
            arr = torch.stack([o[k].reshape(-1)[idx] for o in outs])
        else:
            arr = torch.stack([o[k] for o in outs])
        np.save(os.path.join(path, k + ".npy"), arr.float().cpu().numpy())


LAUNCH_LIST = (["pack_camera", "collapse_time_rows", "deform_features", "deform_f16_kernel", "bin_sort (cooperative)",
                "bin_place", "bin_fix", "blend_forward"],
               ["pack_camera", "collapse_time_rows", "deform_kernel", "bin_sort (cooperative)", "bin_place", "bin_fix", "blend_forward"])


def launches_per_view(net):
    return len(LAUNCH_LIST[0 if NETS[net]["Wd"] == 128 else 1])


def parity_check(g4d, synth, wl, w, scene, mod, pc, cam, dev):
    """Frame 0 of the benched workload, outside every timed region: the CUDA path against the CPU oracle (deformation
    restatement pinned to the reference module + C rasterizer port).  oracle/ is the checker here, never the thing timed."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from util_scene import oracle_params_from_module, oracle_render
        t0 = time.perf_counter()
        bg = torch.tensor(w["bg"], dtype=torch.float32, device=dev)
        with torch.no_grad():
            out = g4d.render(cam, pc, Pipe, bg)
            cfg, prm = oracle_params_from_module(mod)
            for t_ in prm.leaves():
                t_.requires_grad_(False)
            color, depth, radii, _, _ = oracle_render(cfg, prm, scene, cam, cam.time, w["bg"], sh_degree=3)
        err = (out["render"].cpu() - color).abs()
        derr = (out["depth"].cpu() - depth).abs()
        return {"frame": 0, "against": "oracle (CPU)", "image_linf": float(err.max()), "image_median_err": float(err.median()),
                "frac_pixels_gt_1e-4": float((err > 1e-4).float().mean()), "depth_linf": float(derr.max()),
                "radii_mismatch_frac": float((out["radii"].cpu() != radii).float().mean()),
                "ok": bool(float((err > 1e-4).float().mean()) <= 1e-3 and float(err.max()) <= 1e-2),
                "seconds": time.perf_counter() - t0}
    except Exception as e:       # the checker must never take the measurement down
        return {"error": "%s: %s" % (type(e).__name__, e)}


def gpu_eager_baseline(g4d, synth, w, scene, mod, dev):
    """BASELINE.md 3.2: what the fused kernel replaces in train.py -- the reference's own deform_network module running
    eager on this GPU (ATen grid_sample + cuBLAS SGEMM launches), CUDA events, same N / weights / inputs.  The reference
    rasterizer cannot run here (its source is absent), so this covers the deformation half only; our deform-only entry
    point (drop-in deform_network.forward, MODE 0) is timed beside it on the same tensors."""
    try:
        from oracle import deform_ref as dr
        from oracle.ref_loader import reference_available, load_reference_deform_network, reference_origin
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from util_scene import oracle_params_from_module
        if not reference_available():
            return {"unavailable": "reference module not present (oracle/_ref not materialised)"}
        cfg, prm = oracle_params_from_module(mod)
        ref = load_reference_deform_network(cfg)
        sd = ref.state_dict(); sd.update(dr.params_to_state_dict(prm)); ref.load_state_dict(sd)
        ref = ref.to(dev)
        n = w["n"]
        ins = [scene[k].to(dev) for k in ("xyz", "scaling", "rotation", "opacity")]
        shs = torch.cat([scene["features_dc"], scene["features_rest"]], dim=1).to(dev)
        tt = torch.tensor(0.37, device=dev).repeat(n, 1)

        def timeit(fn, iters=10, warm=3):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize(dev)
            evs = []
            for _ in range(iters):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); fn(); b.record(); evs.append((a, b))
            torch.cuda.synchronize(dev)
            return float(np.median([a.elapsed_time(b) for a, b in evs]))

        def ref_fwd():
            with torch.no_grad():
                return ref(*ins, shs, tt)

        def our_fwd():
            with torch.no_grad():
                return mod(*ins, shs, tt)

        leaves = [x.clone().requires_grad_(True) for x in ins + [shs]]

        def ref_fwdbwd():
            outs = ref(*leaves, tt)
            sum(o.sum() for o in outs).backward()

        def our_fwdbwd():
            outs = mod(*leaves, tt)
            sum(o.sum() for o in outs).backward()
        with torch.no_grad():
            err = max(float((a - b).abs().max()) for a, b in zip(ref_fwd(), our_fwd()))
        res = {"what": "reference scene.deformation.deform_network eager on this GPU (deformation half only)",
               "module_from": reference_origin(), "n": n,
               "reference_eager_fwd_ms": timeit(ref_fwd), "g4d_deform_fwd_ms": timeit(our_fwd),
               "reference_eager_fwd_bwd_ms": timeit(ref_fwdbwd, iters=5, warm=2), "g4d_deform_fwd_bwd_ms": timeit(our_fwdbwd, iters=5, warm=2),
               "max_abs_output_diff": err}
        res["fwd_speedup"] = res["reference_eager_fwd_ms"] / res["g4d_deform_fwd_ms"]
        res["fwd_bwd_speedup"] = res["reference_eager_fwd_bwd_ms"] / res["g4d_deform_fwd_bwd_ms"]
        return res
    except Exception as e:
        return {"error": "%s: %s" % (type(e).__name__, e)}


def run_train_steps(g4d, synth, lib, w, scene, mod, dev, dist, world, rank, steps, warmup, flush):
    """Full train step per rank through the data-parallel harness (4dgaussians_b200/train_dp.py, the shape of
    train.py:180-226,259-292): B=2 views (cook_spinach batch size) fused fwd + bwd, fused L1 loss kernel against a resident
    target, HexPlane regulariser kernel, densification statistics, the flat gradient buffer all-reduced in 4 slices
    pipelined with ONE-launch Adam slices.  Returns ms per step (max over ranks)."""
    td = importlib.import_module("4dgaussians_b200.train_dp")
    gs = td.GaussianSet(scene, mod, device=dev, sh_degree=3)
    tr = td.DPTrainer(gs, td.default_opt(), dist=dist, world_size=world, rank=rank, cameras_extent=2.6, seed=0)
    B = 2
    cams = synth.orbit_cameras(64, w["width"], w["height"], radius=w["radius"], focal=w["focal"], timestamps=300)
    bg = torch.tensor(w["bg"], dtype=torch.float32, device=dev)
    target = torch.rand(3, w["height"], w["width"], device=dev)
    evs = []
    wsp = lib.Workspace.get(dev.index)
    wsp.set_option(lib.OPT_STAGE_TIMING, 0)
    for it in range(steps + warmup):
        flush.fill_(it & 0xFF)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if it == warmup:
            torch.cuda.synchronize(dev)
            if dist is not None:
                dist.barrier()
        a.record()
        mine = [cams[((it * B + v) * world + rank) % len(cams)] for v in range(B)]
        tr.step(mine, [target] * B, bg, Pipe)
        b.record()
        if it >= warmup:
            evs.append((a, b))
    torch.cuda.synchronize(dev)
    ms = _max_over_ranks(dist, dev, sum(x.elapsed_time(y) for x, y in evs) / len(evs))
    # one more (untimed) step with the per-stage events on: stage times of its last view
    wsp.set_option(lib.OPT_STAGE_TIMING, 1)
    it = steps + warmup
    tr.step([cams[((it * B + v) * world + rank) % len(cams)] for v in range(B)], [target] * B, bg, Pipe)
    torch.cuda.synchronize(dev)
    wsp.set_option(lib.OPT_STAGE_TIMING, 0)
    ctx = wsp._free_contexts
    st = ctx[-1].stage_times() if ctx else {}
    numel = tr.state.numel
    mod.fused_grad_accumulation = False
    for p in mod.parameters():
        p.grad = None
    return {"ms_per_step": ms, "step_ms": [round(x.elapsed_time(y), 3) for x, y in evs],
            "views_per_step_per_gpu": B, "global_batch": B * world,
            "arithmetic": "forward MLP FP16x2 operands, 3 products (fp32-accurate); backward MLP BF16 hi+lo, 3 products (~16 mantissa bits) vs the "
                          "reference's fp32 SGEMM; everything else fp32",
            "includes": "DPTrainer.step: 2x fused fwd+bwd (network gradients accumulated straight into the flat buffer), fused L1 "
                        "loss + gradient kernels, HexPlane regulariser kernel, densification statistics, all-reduce of the flat "
                        "gradient buffer (%d floats, 4 pipelined slices), one-launch Adam per slice" % numel,
            "last_view_stage_ms": st}


# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_arm(workload: str, steps: int, warmup: int):
    """The reference's CPU implementation of the path on the host cores: deformation = the reference's OWN PyTorch module
    (imported from /root/reference in the build container, from the unmodified copies in oracle/_ref on the GPU box);
    rasterizer = oracle C port with OpenMP (the reference rasterizer's source is absent).  One step = one full view of
    the workload; the torch thread count is the best of a small sweep (reported)."""
    from oracle import deform_ref as dr
    from oracle import raster_ref as rr
    from oracle.ref_loader import reference_available, load_reference_deform_network, reference_origin
    g4d, synth, w, scene, mod = build_scene(workload)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from util_scene import cam_tuple, oracle_params_from_module
    cores = os.cpu_count() or 1
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    cfg, prm = oracle_params_from_module(mod)
    for t_ in prm.leaves():
        t_.requires_grad_(False)
    kind, origin, ref_net = "port", "oracle/deform_ref.py (restatement)", None
    if reference_available():
        ref_net = load_reference_deform_network(cfg)
        sd = ref_net.state_dict(); sd.update(dr.params_to_state_dict(prm)); ref_net.load_state_dict(sd)
        kind, origin = "reference(deform)+port(rasterizer)", reference_origin()
    cams = synth.orbit_cameras(max(8, steps + warmup), w["width"], w["height"], radius=w["radius"], focal=w["focal"], timestamps=300)
    shs = torch.cat([scene["features_dc"], scene["features_rest"]], dim=1)
    n = w["n"]

    def deform(cam):
        with torch.no_grad():
            if ref_net is not None:
                pts, sc, rot, op, sh = ref_net(scene["xyz"], scene["scaling"], scene["rotation"], scene["opacity"], shs,
                                               torch.tensor(cam.time).repeat(n, 1))
            else:
                pts, sc, rot, op, sh = dr.deform_forward(cfg, prm, scene["xyz"], scene["scaling"], scene["rotation"],
                                                         scene["opacity"], shs, cam.time)
            s, r, o = dr.activate(sc, rot, op)
        return pts, s, r, o, sh
    # thread sweep for the PyTorch-CPU deformation (element-wise ATen kernels stop scaling well before 128 threads)
    sweep = {}
    for th in sorted({min(cores, x) for x in (8, 16, 32, 64, cores)}):
        torch.set_num_threads(th)
        deform(cams[0])
        t0 = time.perf_counter(); deform(cams[0]); sweep[th] = time.perf_counter() - t0
    best = min(sweep, key=sweep.get)
    torch.set_num_threads(best)
    times, t_def, t_ras = [], [], []
    rr.lib()
    for i in range(steps + warmup):
        cam = cams[i % len(cams)]
        t0 = time.perf_counter()
        pts, s, r, o, sh = deform(cam)
        t1 = time.perf_counter()
        rc, _ = cam_tuple(cam, w["bg"], sh_degree=3)
        rr.rasterize_forward(rc, pts.numpy(), s.numpy(), r.numpy(), o.numpy(), sh.numpy())
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt); t_def.append(t1 - t0); t_ras.append(dt - (t1 - t0))
    ms = 1e3 * float(np.mean(times))
    fps = 1e3 / ms
    cb = {"value": fps, "unit": UNIT, "cores": cores, "kind": kind, "deform_module_from": origin,
          "torch_threads": best, "torch_thread_sweep_s_per_view": {str(k): round(v, 3) for k, v in sweep.items()},
          "sample": "%d full %s view(s) (%dk Gaussians, %dx%d): PyTorch-CPU deformation (%.2f s/view, %d threads) + OpenMP C "
                    "rasterizer port (%.2f s/view, %d threads), forward" % (len(times), workload, n // 1000, w["width"], w["height"],
                                                                            float(np.mean(t_def)), best, float(np.mean(t_ras)), cores)}
    line = {"impl": "reference", "metric": metric_name(workload), "value": fps, "unit": UNIT, "n_gpus": 1, "steps": steps,
            "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": WORKLOAD_TEXT[workload], "views_per_step": 1, "host": "CPU, %d cores" % cores},
            "cpu_baseline": cb, "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    return line


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # one step = one full view (~1-2 s of CPU work)
    line = cpu_reference_arm(args.workload, steps=args.steps, warmup=min(args.warmup, 2))
    line["n_gpus"] = args.gpus
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="g4d", choices=["g4d", "reference"])
    ap.add_argument("--workload", default="C3", choices=["C1", "C2", "C3", "C4"])
    ap.add_argument("--views-per-step", dest="views_per_step", type=int, default=32)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--host-sync", dest="host_sync", action="store_true",
                    help="size the instance buffer exactly with one host read of R per forward (the reference's behaviour) "
                         "instead of the default capacity-bounded device-side binning")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write what render() returned for each view of the last timed step (rank 0's "
                         "views) to DIR/<key>.npy as float32; a fixed, seeded sample of every output when all of them would "
                         "exceed 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
