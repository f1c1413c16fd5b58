#!/usr/bin/env python
"""bench.py - depth-maps/s of the MVSFormer++ depth-inference hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA library behind the reference seams)
  python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the reference's algorithm on the host cores

A step = one pass of the hot path (FMT -> 4-stage cascade: warp + group-correlation + visibility aggregation ->
cost regularisation -> soft-argmax) over one batch of synthetic reference views; the workload is BASELINE.json
configs[1] (DTU test config: V=5, numdepth 192, 1152x1536, ndepths 32/16/8/4), one depth map per GPU per step
(weak scaling: reference views shard embarrassingly; NCCL only gathers the depth maps).
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "dtu": dict(name="DTU test config: V=5 views, numdepth=192 (425..931mm), 1152x1536, ndepths [32,16,8,4], "
                     "feature pyramids C=[64,32,16,8] (BASELINE.json configs[1])", V=5, H=1152, W=1536, numdepth=192),
    "tt": dict(name="Tanks&Temples intermediate: V=10 views, numdepth=256 (425..1101mm), 1088x1920 (1080 rows padded to a "
                    "multiple of 64 as the reference's loader does), ndepths [32,16,8,4] (BASELINE.json configs[3])",
               V=10, H=1088, W=1920, numdepth=256, interval=2.65),
    "small": dict(name="plumbing: V=3, numdepth=48, 128x192", V=3, H=128, W=192, numdepth=48),
}
TMP = [5.0, 5.0, 5.0, 1.0]


def algorithmic_bytes(V, H, W, feat_chs=(64, 32, 16, 8), ndepths=(32, 16, 8, 4), G=8):
    """SURVEY.md §8(d): 4*[V*C*HW + D*HW + G*D*HW] per stage (features once, hypotheses once, volume once)."""
    out = []
    for c, d, sc in zip(feat_chs, ndepths, (8, 4, 2, 1)):
        hw = (H // sc) * (W // sc)
        out.append(4 * (V * c * hw + d * hw + G * d * hw))
    return out


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                   capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(o[0]))
                self.max_mhz = float(o[1])
                for n, v in zip(names, o[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def bind_to_gpu_numa_node(dev_index):
    """Pins this rank's host threads to the CPUs of its GPU's NUMA node (sysfs: the PCI device's numa_node and that node's
    cpulist), BEFORE the pinned staging buffers are allocated, so that first-touch places them on the local node: 8 ranks
    uploading 531 MB per step from two sockets otherwise cross the inter-socket link.  Returns a description or None."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(dev_index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"gpu": dev_index, "pci": bdf, "numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None


def make_inputs(wl, seed, jitter=0.0):
    from mvsformerplusplus_b200 import synth
    feats = synth.make_features(wl["V"], wl["H"], wl["W"], seed=seed, smooth=False)
    proj = synth.make_proj_matrices(wl["V"], wl["H"], wl["W"], jitter=jitter)
    dv = synth.make_depth_values(wl["numdepth"], 425.0, wl.get("interval", 2.65 * 192 / wl["numdepth"]))
    return feats, proj, dv


def dump_outputs(outs, directory):
    """--dump-outputs: writes {name: tensor} as DIR/<name>.npy in float32.  The final maps are written whole up to
    3 Mi values (one DTU or T&T depth map per GPU), every other array up to 512 Ki values; a larger array is written as a
    fixed, seeded sample of that many values (flattened) under <name>_sample.npy.  At most 2 x 12 + 12 x 2 = 48 MB."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    for name, t in outs.items():
        cap = (3 << 20) if name in ("refined_depth", "photometric_confidence") else (1 << 19)
        v = t.detach().float()
        if v.numel() > cap:
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            v = v.reshape(-1)[idx.to(v.device)]
            name += "_sample"
        np.save(os.path.join(directory, name + ".npy"), v.cpu().numpy().astype(np.float32))


def make_net(seed=7):
    import torch
    from mvsformerplusplus_b200 import synth
    from mvsformerplusplus_b200.config import default_args
    from mvsformerplusplus_b200.hotpath import HotPathNet
    torch.manual_seed(0)
    net = HotPathNet(default_args()).eval()
    sd = synth.randomize_state_dict(net, seed=seed)
    return net, sd


# ======================================================================================================
def cpu_reference_pass(wl, threads, seed=1234):
    """One pass of the hot path on the host cores, fp32.  Returns (seconds, kind):
    kind "reference" - the reference's OWN modules (models/FMT.py, models/cost_volume.py, models/module.py ... imported
                       from oracle/_ref, the build-time copy made by oracle/build_ref.py) through the glue of
                       DINOv2_mvsformer_model.py:117-179, with this repo's seeded weights loaded by state dict;
    kind "port"      - the oracle port with the reference's ATen kernels (F.grid_sample + SDPA), when oracle/_ref is absent."""
    import torch
    from mvsformerplusplus_b200 import synth
    from mvsformerplusplus_b200.config import default_args
    torch.set_num_threads(threads)
    feats, proj, dv = make_inputs(wl, seed)
    from oracle import ref_hotpath as RH  # bench.py's CPU legs are allowed oracle users (checker / baseline only)
    if RH.reference_root() is not None:
        R = RH.import_reference()
        args = default_args()
        torch.manual_seed(0)
        model = RH.RefHotPath(R, args).eval()
        synth.randomize_state_dict(model, seed=7)   # same seeded weights as make_net()
        t0 = time.perf_counter()
        RH.reference_hotpath(R, model, args, feats, proj, dv, TMP, capture=False)
        return time.perf_counter() - t0, "reference"
    from oracle import hotpath as O
    O.USE_ATEN_KERNELS = True
    net, sd = make_net()
    t0 = time.perf_counter()
    with torch.no_grad():
        O.hotpath_forward(feats, proj, dv, sd, default_args(), tmp=TMP)
    return time.perf_counter() - t0, "port"


def cpu_threads():
    """Host threads of the CPU arm: measured on the 2 x 32-core GPU box, the ATen kernels peak at 32 threads (12.5 s per
    depth map; 64: 14.6 s; all 128 hyper-threads: 170 s)."""
    return max(1, min(32, os.cpu_count() or 1))


def run_reference_arm(a, wl, rank, world):
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    threads = cpu_threads()
    times, kind = [], "port"
    for i in range(a.warmup + a.steps):
        dt, kind = cpu_reference_pass(wl, threads)
        if i >= a.warmup:
            times.append(dt)
    ms = 1000.0 * sum(times) / len(times)
    val = 1000.0 / ms
    what = ("the reference's own modules (oracle/_ref copy of models/), glue of DINOv2_mvsformer_model.py:117-179" if kind == "reference"
            else "oracle port calling the reference's ATen kernels")
    sample = f"1 full depth map (whole workload, fp32, {what}) per step"
    line = {"impl": "reference", "metric": "depth-maps/sec (hot path: FMT + 4-stage cascade)", "value": val, "unit": "depth-maps/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "host_threads": threads},
            "cpu_baseline": {"value": val, "unit": "depth-maps/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "depth-maps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ======================================================================================================
def run_ours(a, wl, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from mvsformerplusplus_b200 import _lib

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device - the B200 hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None   # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    net, _ = make_net()
    net = net.to(dev)
    B = a.batch
    # reference views (items) are dealt round-robin to the ranks (sharding.shard_items, SURVEY.md 8e); every item has its own
    # seed and jittered camera ring (SURVEY.md 8d config 3)
    from mvsformerplusplus_b200 import sharding
    n_items = B * world
    my_items = sharding.shard_items(n_items, rank, world)
    host_inputs = []
    for it in my_items:
        feats, proj, dv = make_inputs(wl, 1234 + it, jitter=0.02 * (it % 5))
        host_inputs.append(({k: v.pin_memory() for k, v in feats.items()}, {k: v.pin_memory() for k, v in proj.items()},
                            dv.pin_memory()))
    dev_inputs = [({k: v.to(dev) for k, v in f.items()}, {k: v.to(dev) for k, v in p.items()}, d.to(dev))
                  for f, p, d in host_inputs]
    h2d = sum(sum(v.numel() * 4 for v in f.values()) + sum(v.numel() * 4 for v in p.values()) + d.numel() * 4
              for f, p, d in host_inputs)
    H, W = wl["H"], wl["W"]
    local_buf = torch.empty((B, 2, H, W), device=dev)
    host_out = torch.empty((B, 2, H, W)).pin_memory()
    gather_ws = {}

    # Reference views are independent: with --streams 2 consecutive steps run on alternating compute streams ("lanes"), two
    # depth maps are in flight per GPU and the latency-bound kernels of one overlap the other's (tools/two_stream_probe.py).
    # Off by default (see --streams).  Every step still does all of its work; a lane's buffers are reused, stream-ordered.
    n_lanes = max(1, a.streams)
    lanes = [torch.cuda.Stream(device=dev) for _ in range(n_lanes)] if n_lanes > 1 else [torch.cuda.current_stream(dev)]
    lane_bufs = [local_buf] + [torch.empty_like(local_buf) for _ in range(n_lanes - 1)]
    lane_gathered = [torch.cuda.Event() for _ in range(n_lanes)]
    step_no = [0]
    last_outs = [None] * len(dev_inputs)   # --dump-outputs: what the latest step's forward calls returned

    def step_resident():
        k = step_no[0] % n_lanes
        step_no[0] += 1
        lane, buf = lanes[k], lane_bufs[k]
        with torch.cuda.stream(lane):
            lane.wait_event(lane_gathered[k])           # the gather of this lane's previous step has read `buf`
            for b, (f, p, d) in enumerate(dev_inputs):
                out = net.forward_features(f, p, d, TMP)
                buf[b, 0].copy_(out["refined_depth"][0])
                buf[b, 1].copy_(out["photometric_confidence"][0])
                if a.dump_outputs:
                    last_outs[b] = out
        # the only collective on the path: gather of the depth / confidence maps in item order (SURVEY.md 8e), issued on the
        # main stream in step order on every rank (after the lane's kernels; the other lane keeps running)
        if world > 1:
            main = torch.cuda.current_stream(dev)
            if n_lanes > 1:
                main.wait_stream(lane)
            sharding.gather_maps(buf, n_items, workspace=gather_ws)
            lane_gathered[k].record(main)

    # end to end through the package's host-side API: every step uploads its pinned host batch (copy stream, three device
    # slots: the upload of the next batches overlaps the kernels of the current one) and reads the depth + confidence maps back
    from mvsformerplusplus_b200.streaming import PrefetchingRunner
    runner = PrefetchingRunner(net, dev, slots=3 if n_lanes == 1 else 2 + n_lanes, lanes=n_lanes)

    def step_e2e():
        n = len(host_inputs)
        for b in range(n):
            out = runner.run(host_inputs[b], next_batch=host_inputs[(b + 1) % n], tmp=TMP)
            local_buf[b, 0].copy_(out["refined_depth"][0])
            local_buf[b, 1].copy_(out["photometric_confidence"][0])
        host_out.copy_(local_buf, non_blocking=True)
        sharding.gather_maps(local_buf, n_items, workspace=gather_ws)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        main = torch.cuda.current_stream(dev)
        for lane in lanes:
            if lane is not main:
                lane.wait_event(e0)
        for _ in range(steps):
            fn()
        for lane in list(lanes) + list(runner.lanes):
            if lane is not main:
                main.wait_stream(lane)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    _lib.launch_count(reset=True)
    ms_step = timed(step_resident, a.steps, max(a.warmup, 3))
    launches = _lib.launch_count(reset=True) // (a.steps + max(a.warmup, 3))
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:   # rank 0's reference views, in item order
        outs = {k: torch.stack([o[k][0] for o in last_outs]) for k in ("refined_depth", "photometric_confidence")}
        for s in range(1, 5):
            for k in ("depth", "photometric_confidence", "prob_volume"):
                outs[f"stage{s}_{k}"] = torch.stack([o[f"stage{s}"][k][0] for o in last_outs])
        dump_outputs(outs, a.dump_outputs)
    last_outs[:] = [None] * len(last_outs)   # released before the end-to-end timing
    ms_e2e = timed(step_e2e, a.steps, max(a.warmup, 3))
    d2h = host_out.numel() * 4

    # ---- per-entry-point device time (CUDA events on the launching stream) for the roofline of the fused
    #      warp + group-correlation kernels (pass A entropy + pass B aggregation, all 4 stages)
    line_extra = {}
    if rank == 0:
        f, p, d = dev_inputs[0]
        reps = 3
        _lib.ktimer_enable(True)
        with _lib.profile_calls() as prof:
            for _ in range(reps):
                net.forward_features(f, p, d, TMP)
        summ = prof.summary()
        att_ms, att_n = _lib.ktimer_read("attention_tc")
        _lib.ktimer_enable(False)
        per_map = {k: v["ms"] / reps for k, v in summ.items()}
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        peaks = json.load(open(peaks_path)) if os.path.exists(peaks_path) else {}
        # dominant kernel of the step: stage-1 softmax attention (tcgen05), one launch per transformer layer.
        # algorithmic FLOPs per launch = 2 GEMMs x 2 N^2 hd per head (the 3 split-precision products are overhead)
        n_tok = (net.ndepths[0] // 2) * (H // 8 // 4) * (W // 8 // 4)   # stage 1: D x H/8 x W/8, down_rate (2,4,4)
        att_flops = 4.0 * n_tok * n_tok * 16 * 4
        att_launch_ms = att_ms / max(att_n, 1)
        tf_peak = peaks.get("bf16_tflops_sustained", 1480.0)
        tf_which = ("measured (MEASURED_PEAKS.json bf16_tflops_sustained: the kernel runs inside a long step)"
                    if peaks else "fallback (B200_PROFILING.md)")
        achieved_tf = att_flops / 1e12 / (att_launch_ms / 1e3) if att_launch_ms > 0 else 0.0
        traffic = traffic_wc = None   # dram bytes of the same kernels from the committed ncu capture (profiles/)
        tpath = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
        if os.path.exists(tpath) and wl is WORKLOADS["dtu"]:
            tj = json.load(open(tpath))
            traffic = tj.get("attention_fa_kernel", {}).get("dram_bytes_per_launch")
            traffic_wc = tj.get("warp_corr_entropy_store + corr_aggregate (8 launches / depth map)", {}).get("dram_bytes_per_depth_map")
        line_extra["roofline"] = {"bound": "tensor", "kernel": "attention_fa_kernel (stage-1 transformer regulariser, 1 launch / layer)",
                                  "achieved": achieved_tf, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved_tf / tf_peak,
                                  "traffic": traffic, "peak_source": tf_which, "algorithmic_flops_per_launch": att_flops,
                                  "launch_ms": att_launch_ms, "launches_per_depth_map": att_n // reps,
                                  "share_of_step": att_ms / reps / ms_step if ms_step > 0 else None,
                                  "note": "bound by the XU pipe (ncu: 83.7 % busy): 3.06e9 exp2 per launch at 16 / clk / SM = 0.66 ms, plus the "
                                          "mbarrier handshake latency between the MMA and softmax warps (DESIGN.md 4); "
                                          "Q/K/V are fp16 hi+lo (3 products for the scores), the probabilities fp16"}
        # the fused warp + group-correlation kernels are the HBM-roofline kernels of the path (8 launches / depth map)
        t_wc = sum(per_map.get(k, 0.0) for k in ("mvsf_warp_corr_entropy", "mvsf_warp_corr_aggregate",
                                                  "mvsf_warp_corr_entropy_store", "mvsf_corr_aggregate"))
        alg = algorithmic_bytes(wl["V"], H, W)
        if peaks:
            peak, which = peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, which = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
        achieved = sum(alg) / 1e9 / (t_wc / 1e3) if t_wc > 0 else 0.0
        line_extra["roofline_hbm"] = {"bound": "hbm", "kernel": "warp_corr_entropy_store + corr_aggregate (8 launches / depth map)",
                                      "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                                      "traffic": traffic_wc, "peak_source": which, "algorithmic_bytes_per_depth_map": sum(alg),
                                      "kernel_ms_per_depth_map": t_wc,
                                      "note": "algorithmic bytes = features + hypotheses + volume; traffic = measured DRAM bytes of the pass-A / "
                                              "pass-B launches of one depth map (profiles/r2_ncu_traffic.json; stage 4 pass A = selection kernel + "
                                              "TMA pipeline kernel + the L1 kernel's skipped launch): the per-view group correlations spilled "
                                              "between the two passes are implementation traffic.  The 4-corner fp32 gather is bound by the SM "
                                              "load path (3.6 GB per stage and pass at 128 B/clk/SM): ceiling ~0.22 of the HBM roofline"}
        line_extra["kernel_ms_per_depth_map"] = {k.replace("mvsf_", ""): round(v, 4) for k, v in sorted(per_map.items())}

    if rank == 0:
        cpu = None
        if not a.no_cpu_baseline and world == 1:
            threads = cpu_threads()
            cpu_reference_pass(wl, threads)             # warm-up pass (allocator, thread pools), like the reference arm
            dt, kind = cpu_reference_pass(wl, threads)
            cpu = {"value": 1.0 / dt, "unit": "depth-maps/s", "cores": threads, "kind": kind,
                   "sample": "1 full depth map of the same workload (second of two passes, fp32; " +
                             ("the reference's own modules from oracle/_ref)" if kind == "reference" else
                              "oracle port calling the reference's ATen kernels F.grid_sample + SDPA)")}
        maps = B * world
        line = {"metric": "depth-maps/sec (hot path: FMT + 4-stage cascade)", "value": maps * 1000.0 / ms_step,
                "unit": "depth-maps/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": wl["name"], "ref_views_per_gpu_per_step": B, "parallelism": f"shard{world}",
                           "l2": "inputs_larger_than_l2 (531 MB feature pyramids per depth map)",
                           "precision": "fp32-class parity mode: tcgen05 GEMMs / attention scores / 3-D and 2-D convolutions on fp16 hi+lo "
                                        "split operands (22-bit mantissa, fp32 accumulate), attention probabilities fp16, "
                                        "everything else fp32 SIMT",
                           "e2e_pipeline": "pinned host batch (allocated on the GPU's NUMA node) -> copy stream -> device slots; "
                                           "upload of batch i+1 overlaps the kernels of batch i; depth+confidence read back every step; "
                                           "consecutive steps alternate between `compute_streams` streams (two depth maps in flight)",
                           "numa_binding": numa,
                           "compute_streams": n_lanes if n_lanes > 1 else 1},
                "e2e": {"value": maps * 1000.0 / ms_e2e, "unit": "depth-maps/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e},
                "gpu_launches": launches * a.steps, "gpu_launches_per_step": launches, "clocks": clocks,
                "cpu_baseline": cpu}
        line.update(line_extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_dsweep(a):
    """BASELINE.json configs[4] / SURVEY.md 8(d) config 5: kernel-level sweep of the fused warp + group-correlation
    kernels (pass A entropy + pass B aggregation; the vis CNN between them is timed separately) at the full-resolution
    stage geometry C = G = 8, 1152x1536, V = 5, with D in {48, 96, 192, 384} plane-sweep hypotheses spanning 425..931 mm
    uniformly in inverse depth.  Prints achieved algorithmic GB/s per D."""
    import ctypes
    import torch
    from mvsformerplusplus_b200 import _lib, packing, synth
    from mvsformerplusplus_b200.params import build_hotpath_params
    from mvsformerplusplus_b200.config import default_args
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    L = _lib.lib()
    V, C, G, H, W = 5, 8, 8, 1152, 1536
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    st = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator().manual_seed(1234)
    feat = torch.randn(V, H, W, C, generator=g).to(dev)
    pm = synth.make_proj_matrices(V, H, W)["stage4"][0].to(dev)
    homs, kinv = torch.empty((V - 1) * 12, device=dev), torch.empty(9, device=dev)
    _lib.check(L.mvsf_compose_geometry(P(pm), V, P(homs), P(kinv), st()), "compose_geometry")
    torch.manual_seed(0)
    sd = synth.randomize_state_dict(build_hotpath_params(default_args()).eval(), seed=7)
    wts = packing.pack_vis(sd, "fusions.3.vis.").to(dev)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = json.load(open(peaks_path))["hbm_gbs"] if os.path.exists(peaks_path) else 6650.0
    rows = []
    for D in (48, 96, 192, 384):
        k = torch.arange(D, dtype=torch.float32, device=dev) / (D - 1)
        inv = 1.0 / 931.15 + (1.0 / 425.0 - 1.0 / 931.15) * k
        depth = (1.0 / inv).view(D, 1, 1).expand(D, H, W).contiguous()
        ent = torch.empty(V - 1, H, W, device=dev)
        vis = torch.empty(V - 1, H, W, device=dev)
        vol = torch.empty(D, H, W, G, device=dev)

        def pass_a():
            _lib.check(L.mvsf_warp_corr_entropy(P(feat), P(homs), P(depth), P(ent), V, C, G, D, H, W, st()), "warp_corr_entropy")

        def pass_b():
            _lib.check(L.mvsf_warp_corr_aggregate(P(feat), P(homs), P(depth), P(vis), P(vol), V, C, G, D, H, W, st()), "warp_corr_aggregate")

        pass_a()
        _lib.check(L.mvsf_vis_cnn(P(ent), P(wts), P(vis), V - 1, H, W, st()), "vis_cnn")
        pass_b()
        torch.cuda.synchronize()
        reps = a.steps
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ta = tb = 0.0
        for _ in range(reps):
            ev[0].record(); pass_a(); ev[1].record(); pass_b(); ev[2].record()
            torch.cuda.synchronize()
            ta += ev[0].elapsed_time(ev[1]); tb += ev[1].elapsed_time(ev[2])
        ta, tb = ta / reps, tb / reps
        alg = 4 * (V * C * H * W + D * H * W + G * D * H * W)
        rows.append({"D": D, "pass_a_ms": round(ta, 4), "pass_b_ms": round(tb, 4), "algorithmic_bytes": alg,
                     "achieved_gbs": alg / 1e9 / ((ta + tb) / 1e3), "frac": alg / 1e9 / ((ta + tb) / 1e3) / peak})
        del depth, vol
    best = max(r["achieved_gbs"] for r in rows)
    line = {"metric": "warp+corr HBM GB/s vs D (C=G=8, 1152x1536, V=5; BASELINE.json configs[4])", "value": best, "unit": "GB/s",
            "n_gpus": 1, "steps": a.steps, "warmup": 1, "higher_is_better": True, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "dsweep: plane-sweep hypotheses uniform in inverse depth over 425..931 mm, two-gather plan "
                                   "(pass A entropy + pass B aggregation), inputs larger than L2 (283 MB of features)"},
            "roofline": {"bound": "hbm", "peak": peak, "unit": "GB/s", "achieved": best, "frac": best / peak, "traffic": None},
            "sweep": rows, "gpu_launches": 2 * len(rows) * a.steps}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="dtu", choices=sorted(WORKLOADS) + ["dsweep"])
    ap.add_argument("--batch", type=int, default=1, help="reference views per GPU per step")
    ap.add_argument("--streams", type=int, default=1,
                    help="compute streams per GPU: consecutive steps alternate between them.  EXPERIMENTAL above 1: two depth maps in "
                         "flight measured +8.7 %% (79.8 maps/s) but the attention kernel deadlocks once in a few hundred launches when "
                         "kernels of another stream run next to it (DESIGN.md 5); the bounded waits turn that into a CUDA error")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (final depth and confidence maps, "
                         "per-stage depth, confidence and probability volume of rank 0's reference views) as DIR/<name>.npy; "
                         "inputs and weights are seeded, so two builds run with the same arguments can be compared")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.workload == "dsweep"):
        ap.error("--dump-outputs needs --impl ours and a depth-map workload")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.workload == "dsweep":
        if rank == 0 and a.impl == "ours":
            run_dsweep(a)
        return
    wl = WORKLOADS[a.workload]
    if a.impl == "reference":
        a.warmup = min(a.warmup, 1)   # each pass is ~15-60 s of host work
        run_reference_arm(a, wl, rank, world)
        return
    run_ours(a, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
