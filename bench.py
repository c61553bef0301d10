#!/usr/bin/env python
"""Benchmark of the DD3D inference hot path (contract: see the task statement / DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload v2_99|dla34|nusc_v2_99]
                    [--batch B] [--dtype bf16|fp16] [--input mapped|raw] [--sweep 8,16,32,64] [--dump-outputs DIR]

A step = one DD3D.forward over one batch of synthetic images per GPU:
  v2_99 (default, the config BASELINE.json's metric is quoted on): V2-99 DD3D, 32 x 900x1600 per GPU;
  dla34: DLA-34 DD3D, 8 x 384x1280 per GPU (BASELINE.json configs[1]; its result rides in the default line as "secondary").
`value` = images/s with inputs resident in HBM (CUDA events, max over ranks); `e2e` = the same through the host-buffer
C-ABI call (pinned H2D of the uint8 images + D2H of the detections inside the timed region).
Weak scaling: every rank runs its own batch (images are independent, reference tridet/data/build.py:78-93); for N > 1 every
step ends with ONE NCCL all-gather of the packed [dets | counts | flags] buffer (dd3d_allgather through the C ABI; replaces
detectron2 comm.gather, kitti_3d_evaluator.py:152-164) issued on a side stream, so the exchange of step k overlaps the
forward of step k+1 and no host synchronisation happens inside the timed region.
`--impl reference` times the CPU oracle port of the reference forward (the reference itself cannot travel to the GPU box:
it needs detectron2/pytorch3d, not installable offline) on rank 0 with all host threads, following BASELINE.md 3
(batch = min(B, 8) images per forward, bounded so that the run ends within minutes).
`--sweep` (BASELINE.json configs[4]): per-GPU batch sweep; prints one JSON line per batch size.
`--dump-outputs DIR` (rank 0): the detections of the last timed step of every workload the run times, one float .npy per
Instances field (see dump_detections), so that two builds can be compared output for output on identical seeded inputs.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (arch, dataset, per-GPU batch, H, W, focal, conv GFLOP / image from BASELINE.md)
    "v2_99": ("v2_99", "nuscenes", 32, 900, 1600, 1266.4, 3066.0),
    "dla34": ("dla34", "kitti_3d", 8, 384, 1280, 721.5, 220.8),
    # NuscenesDD3D (configs/experiments/dd3d_nusc_v99.yaml): 5 samples x 6 cameras per GPU, attr/speed heads and the
    # cross-camera sample aggregation inside the step
    "nusc_v2_99": ("v2_99", "nuscenes", 30, 900, 1600, 1266.4, 3066.0),
}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(tflops=p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1400.0)), gbs=p.get("hbm_gbs", 6650.0),
                    source="measured (MEASURED_PEAKS.json: bf16_tflops_sustained / hbm_gbs)")
    return dict(tflops=1400.0, gbs=6650.0, source="fallback (B200_PROFILING.md: 1.4 PFLOP/s sustained, 6.65 TB/s)")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower() == "active" for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def usable_cpus():
    """Host threads this process can really use: affinity mask capped by the cgroup CPU quota (a container that
    reports 128 CPUs but is throttled to a few cores runs 10x slower when oversubscribed)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    n = min(n, max(1, int(float(parts[0]) / float(parts[1]) + 0.5)))
            else:
                q = int(parts[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                        n = min(n, max(1, int(q / int(f.read()) + 0.5)))
            break
        except Exception:  # noqa: BLE001
            continue
    return n


def pick_threads():
    """Fastest thread count for a representative conv among {usable, usable/2, ..., 4} (measured, ~1 s)."""
    import torch
    import torch.nn.functional as F
    cands, n = [], usable_cpus()
    while n >= 4:
        cands.append(n)
        n //= 2
    cands = cands or [usable_cpus()]
    x, w = torch.randn(1, 128, 120, 200), torch.randn(128, 128, 3, 3)
    best, best_t = cands[0], None
    for c in cands:  # largest first; a smaller count must be clearly (>15 %) faster to win
        torch.set_num_threads(c)
        F.conv2d(x, w, padding=1)
        dt = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            F.conv2d(x, w, padding=1)
            dt = min(dt, time.perf_counter() - t0)
        if best_t is None or dt < 0.85 * best_t:
            best, best_t = c, dt
    return best


DUMP_BUDGET = {"bytes": 64 << 20}  # all arrays of one --dump-outputs run together


def dump_detections(dirname, prefix, out, counts, glob=None):
    """Writes one step's packed [B][cap] dd3d_det buffer as the Instances fields a caller receives (DD3DB200._wrap), each
    padded to [B, cap, ...] with zeros past counts[b], float32 (float64 for the integer fields and counts).  If the arrays
    of all B images do not fit what is left of DUMP_BUDGET, only those of the first images that fit are written."""
    import numpy as np
    import torch
    out, counts = out.cpu(), counts.cpu()
    B, cap = out.shape[:2]
    words = out.clone()
    words[torch.arange(cap)[None, :] >= counts[:, None].long()] = 0
    f, i = words, words.view(torch.int32)
    fields = {"pred_boxes": f[..., 0:4], "scores": f[..., 4], "scores_3d": f[..., 5], "pred_classes": i[..., 6].double(),
              "fpn_levels": i[..., 7].double(), "quat": f[..., 8:12], "proj_ctr": f[..., 12:14], "depth": f[..., 14],
              "size": f[..., 15:18], "locations": f[..., 18:20]}
    if glob is not None:  # NuscenesDD3D
        g = glob.cpu().clone()
        g[torch.arange(cap)[None, :] >= counts[:, None].long()] = 0
        fields.update(pred_attributes=i[..., 21].double(), pred_speeds=f[..., 22], pred_boxes3d_global=g)
    per_image = sum(v[0].numel() * v.element_size() for v in fields.values()) + 8
    n = min(B, DUMP_BUDGET["bytes"] // per_image)
    assert n > 0, "--dump-outputs: 64 MB budget exhausted"
    DUMP_BUDGET["bytes"] -= n * per_image
    fields["counts"] = counts.double()
    os.makedirs(dirname, exist_ok=True)
    for name, v in fields.items():
        np.save(os.path.join(dirname, f"{prefix}{name}.npy"), v[:n].contiguous().numpy())


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:  # noqa: BLE001
        pass
    return "unknown CPU"


def cpu_oracle_rate(workload, forwards, warm=1, budget_s=150.0):
    """images/s of the CPU oracle port (fp32, all usable host threads), BASELINE.md 3: forwards of min(B, 8) images, the
    batch bounded so that warm + forwards passes fit `budget_s` seconds (CPU throughput is flat in the batch size).
    Returns (images/s of the best forward, mean images/s, threads, per-forward seconds, images per forward)."""
    import torch
    from dd3d_b200.config import get_cfg
    from dd3d_b200.synthetic import make_inputs, make_state_dict
    from oracle.dd3d_oracle import DD3DOracle
    arch, ds, B, H, W, focal, _ = WORKLOADS[workload]
    nusc = workload.startswith("nusc")
    torch.set_num_threads(pick_threads())
    cfg = get_cfg(arch, ds, meta_arch="NuscenesDD3D" if nusc else "DD3D")
    orc = DD3DOracle(cfg, make_state_dict(cfg))
    t0 = time.perf_counter()
    orc.forward(make_inputs(1, H, W, focal, seed_base=1), do_postprocess=not nusc)  # warm-up (also sizes the batch)
    t1 = time.perf_counter() - t0
    b = max(1, min(B, 8, int(budget_s / max(t1, 1e-3) / max(forwards + max(warm - 1, 0), 1))))
    times = []
    for i in range(max(warm - 1, 0) + forwards):
        inp = make_inputs(b, H, W, focal, seed_base=1 + i * b)
        t0 = time.perf_counter()
        orc.forward(inp, do_postprocess=not nusc)  # single images of a sample: no cross-camera aggregation
        dt = time.perf_counter() - t0
        if i >= max(warm - 1, 0):
            times.append(dt)
    return b / min(times), b * len(times) / sum(times), torch.get_num_threads(), times, b


def run_reference(args, rank):
    if rank != 0:
        return
    import torch
    arch, ds, B, H, W, focal, _ = WORKLOADS[args.workload]
    best, mean, cores, times, b = cpu_oracle_rate(args.workload, args.steps, warm=max(args.warmup, 1))
    sample = (f"{args.steps} forwards of {b} image(s) ({H}x{W}; BASELINE.md 3 asks for min(B, 8) = {min(B, 8)} per forward, "
              f"bounded here to fit a few minutes -- CPU throughput is flat in the batch size) of the fp32 CPU oracle port "
              f"after {max(args.warmup, 1)} warm-up forward(s); {cpu_model()}, {cores} threads, torch {torch.__version__}; "
              f"value = mean over the timed forwards, best forward {best:.3f} images/s")
    line = {
        "impl": "reference", "metric": "images/sec", "value": mean, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{arch} DD3D, {H}x{W}, {b} image(s) per step (bounded sample of the batch-{B} workload)"},
        "cpu_baseline": {"value": mean, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": mean, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_workload(args, workload, batch, rank, local_rank, world, gatherer_cache, with_cpu=True, steps=None, warmup=None,
                 dump_prefix=""):
    """Times one workload on this rank's GPU; returns the JSON line (dict).  All ranks must call it together."""
    import torch
    import torch.distributed as dist
    from dd3d_b200 import lib
    from dd3d_b200.config import get_cfg
    from dd3d_b200.gather import DetectionGatherer, PackedDetections, split_gathered
    from dd3d_b200.meta_arch import DD3DB200, NuscenesDD3DB200, group_indices
    from dd3d_b200.synthetic import make_inputs, make_nusc_inputs, make_state_dict

    steps = steps or args.steps
    warmup = warmup or args.warmup
    arch, ds, B, H, W, focal, gflop_img = WORKLOADS[workload]
    nusc = workload.startswith("nusc")
    if batch:
        B = batch
    assert not nusc or B % 6 == 0, "NuscenesDD3D batches are whole 6-camera samples"
    dev = torch.device("cuda", local_rank)

    cfg = get_cfg(arch, ds, meta_arch="NuscenesDD3D" if nusc else "DD3D", act_dtype=args.dtype)
    model = (NuscenesDD3DB200 if nusc else DD3DB200)(cfg).to(dev)
    model.load_state_dict(make_state_dict(cfg))
    if nusc:
        inputs = make_nusc_inputs(B // 6, H, W, focal, seed_base=1 + rank * B)
    else:
        inputs = make_inputs(B, H, W, focal, seed_base=1 + rank * B)
    batch_t, K, sizes, shape, is_u8 = model._gather_inputs(inputs, dev)
    raw_mode = args.input == "raw"
    assert not (raw_mode and nusc), "--input raw is wired for the DD3D workloads"
    if raw_mode:  # the mapped tensors stand in for the files: HWC raw images at the dataset resolution
        min_size, max_size = int(cfg.INPUT.RESIZE.MIN_SIZE_TEST), int(cfg.INPUT.RESIZE.MAX_SIZE_TEST)
        nh, nw = C.c_int32(), C.c_int32()
        lib.check(lib.load().dd3d_resize_shape(H, W, min_size, max_size, C.byref(nh), C.byref(nw)))
        shape = (B, nh.value, nw.value)
        h_raw = batch_t.permute(0, 2, 3, 1).contiguous().pin_memory()
        d_raw = h_raw.to(dev)
        raw_sizes = torch.tensor([[H, W]] * B, dtype=torch.int32)
        h_K_scaled = torch.empty((B, 9), dtype=torch.float32)
    model._plan(*shape)
    L, handle = lib.load(), model._handle
    cap = model._desc.out_cap
    dtype_code = lib.IMG_U8 if is_u8 else lib.IMG_F32

    d_batch, d_K, d_sizes = batch_t.to(dev), K.to(dev), sizes.to(dev)
    # two packed [dets | counts | flags] buffers: step k writes slot k & 1 while the all-gather of step k-1 still reads the other
    packed = [PackedDetections(B, cap, dev) for _ in range(2)]
    h_batch, h_K, h_sizes = batch_t.pin_memory(), K.pin_memory(), sizes.pin_memory()
    h_out = [torch.zeros((B, cap, lib.DET_WORDS), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_cnt = [torch.zeros((B, ), dtype=torch.int32).pin_memory() for _ in range(2)]
    stream = torch.cuda.current_stream(dev)
    sp = C.c_void_p(stream.cuda_stream)
    gat = None
    done = [None, None]  # event of the last gather that read packed[slot]
    if world > 1:
        key = (B, cap)
        if key not in gatherer_cache:
            gatherer_cache[key] = DetectionGatherer(B, cap, dev)
        gat = gatherer_cache[key]
        recv = [gat.new_recv() for _ in range(2)]

    if nusc:  # sample aggregation operands (nuscenes_dd3d.py:449-463)
        groups = group_indices([x["sample_token"] for x in inputs], 6)
        d_poses = model._gather_poses(inputs).to(dev)
        d_group = torch.tensor(groups, dtype=torch.int32, device=dev)
        d_glob = torch.zeros((B, cap, 10), dtype=torch.float32, device=dev)
        h_glob = torch.zeros((B, cap, 10), dtype=torch.float32).pin_memory()
        d_scr = torch.empty(int(L.dd3d_op_sample_aggregate_scratch_bytes(B, cap)), dtype=torch.uint8, device=dev)
        d_flags = torch.zeros(1, dtype=torch.int32, device=dev)

    state = {"k": 0}

    def begin_slot():
        slot = state["k"] & 1
        state["k"] += 1
        if gat is not None and done[slot] is not None:
            stream.wait_event(done[slot])  # device-side: the gather that still reads this slot must have finished
        return slot

    def end_slot(slot):
        pk = packed[slot]
        lib.check(L.dd3d_copy_flags(handle, C.c_void_p(pk.flags.data_ptr()), sp), handle)
        if gat is not None:  # ONE collective per step, on the side stream, overlapping the next step's forward
            done[slot] = gat.gather_async(pk, recv[slot], stream)

    def drain():
        if gat is not None:
            for ev in done:
                if ev is not None:
                    stream.wait_event(ev)

    def step_device():
        slot = begin_slot()
        pk = packed[slot]
        if raw_mode:
            lib.check(L.dd3d_forward_raw(handle, C.c_void_p(d_raw.data_ptr()), H, W, C.c_void_p(raw_sizes.data_ptr()),
                                         C.c_void_p(h_K.data_ptr()), min_size, max_size, C.c_void_p(pk.out.data_ptr()),
                                         C.c_void_p(pk.counts.data_ptr()), C.c_void_p(h_K_scaled.data_ptr()), None, sp), handle)
        else:
            lib.check(L.dd3d_forward(handle, C.c_void_p(d_batch.data_ptr()), dtype_code, C.c_void_p(d_K.data_ptr()),
                                     C.c_void_p(d_sizes.data_ptr()), C.c_void_p(pk.out.data_ptr()),
                                     C.c_void_p(pk.counts.data_ptr()), sp), handle)
        if nusc:
            lib.check(L.dd3d_op_sample_aggregate(
                C.c_void_p(pk.out.data_ptr()), C.c_void_p(pk.counts.data_ptr()), C.c_void_p(d_K.data_ptr()),
                C.c_void_p(d_poses.data_ptr()), C.c_void_p(d_group.data_ptr()), max(groups) + 1,
                C.c_void_p(d_glob.data_ptr()), C.c_void_p(d_scr.data_ptr()), C.c_void_p(d_flags.data_ptr()), B, cap,
                float(model.bev_nms_iou_thresh), int(model.max_num_dets_per_sample), sp), handle)
        end_slot(slot)
        return slot

    def step_host_explicit():  # H2D / D2H around the device step (NuscenesDD3D: the aggregation needs all cameras on the device)
        if raw_mode:
            d_raw.copy_(h_raw, non_blocking=True)
        else:
            d_batch.copy_(h_batch, non_blocking=True)
            d_K.copy_(h_K, non_blocking=True)
            d_sizes.copy_(h_sizes, non_blocking=True)
        slot = step_device()
        h_out[slot].copy_(packed[slot].out, non_blocking=True)
        h_cnt[slot].copy_(packed[slot].counts, non_blocking=True)
        if nusc:
            h_glob.copy_(d_glob, non_blocking=True)
        stream.synchronize()

    def step_host():
        if nusc or raw_mode:
            return step_host_explicit()
        slot = begin_slot()
        lib.check(L.dd3d_forward_host(handle, C.c_void_p(h_batch.data_ptr()), dtype_code, C.c_void_p(h_K.data_ptr()),
                                      C.c_void_p(h_sizes.data_ptr()), C.c_void_p(h_out[slot].data_ptr()),
                                      C.c_void_p(h_cnt[slot].data_ptr()), sp), handle)
        if gat is not None:  # whole-batch eval: this rank's detections go back into the packed device buffer and are gathered
            packed[slot].out.copy_(h_out[slot], non_blocking=True)
            packed[slot].counts.copy_(h_cnt[slot], non_blocking=True)
        end_slot(slot)

    def submit(slot):
        lib.check(L.dd3d_submit_host(handle, slot, C.c_void_p(h_batch.data_ptr()), dtype_code, C.c_void_p(h_K.data_ptr()),
                                     C.c_void_p(h_sizes.data_ptr()), C.c_void_p(h_out[slot].data_ptr()),
                                     C.c_void_p(h_cnt[slot].data_ptr()), sp), handle)

    def run_host_pipelined(n):
        """n end-to-end steps through dd3d_submit_host / dd3d_wait_host: every step copies its batch H2D and its
        detections D2H; the H2D of step k+1 (copy stream) overlaps the kernels of step k."""
        submit(0)
        for k in range(n):
            if k + 1 < n:
                submit((k + 1) & 1)
            lib.check(L.dd3d_wait_host(handle, k & 1), handle)
            if gat is not None:
                slot = k & 1
                if done[slot] is not None:
                    stream.wait_event(done[slot])
                packed[slot].out.copy_(h_out[slot], non_blocking=True)
                packed[slot].counts.copy_(h_cnt[slot], non_blocking=True)
                end_slot(slot)

    rank_ms = {}

    def finish_timing(e0, e1, tag):
        ms_local = e0.elapsed_time(e1)
        if world > 1:
            ms = torch.tensor([ms_local], dtype=torch.float64, device=dev)
            allr = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(allr, ms)
            vals = sorted(float(t.item()) for t in allr)
            rank_ms[tag] = {"min": vals[0] / steps, "median": statistics.median(vals) / steps, "max": vals[-1] / steps}
            return vals[-1]
        return ms_local

    def timed_pipelined():
        run_host_pipelined(warmup)
        drain()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run_host_pipelined(steps)
        drain()
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        return finish_timing(e0, e1, "e2e_pipelined")

    def timed(fn, tag, sampler=None):
        for _ in range(warmup):
            fn()
        drain()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        drain()  # the timed region ends when the last all-gather has delivered
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        clocks = sampler.stop() if sampler else None
        return finish_timing(e0, e1, tag), clocks

    ms_dev, clocks = timed(step_device, "value", ClockSampler(local_rank))
    if args.dump_outputs and rank == 0:  # before the e2e legs below reuse the buffers
        last = (state["k"] - 1) & 1
        dump_detections(args.dump_outputs, dump_prefix, packed[last].out, packed[last].counts, d_glob if nusc else None)
    ms_host, _ = timed(step_host, "e2e_serial")
    ms_host_serial = ms_host
    if not nusc and not raw_mode:  # double-buffered host path (H2D of the next step overlaps this step's kernels)
        ms_host = min(ms_host, timed_pipelined())
    torch.cuda.synchronize(dev)
    flags = int(packed[0].flags.item()) | int(packed[1].flags.item())
    assert flags == 0 and model.overflow_flags() == 0, "detection buffers overflowed"
    assert not nusc or int(d_flags.item()) == 0, "sample aggregation overflowed"
    n_det = int(h_cnt[0].sum())
    gathered_ok = None
    if gat is not None:  # the gathered buffer really holds every rank's detections
        last = (state["k"] - 1) & 1
        g_out, g_cnt, g_flags = split_gathered(recv[last], world, B, cap)
        mine = slice(rank * B, (rank + 1) * B)
        gathered_ok = bool(torch.equal(g_cnt[mine], packed[last].counts) and torch.equal(g_out[mine], packed[last].out) and
                           int(g_flags.sum()) == 0)

    # live per-kernel timing (CUDA events on the launch stream around every op of the step)
    model.set_profile(True)
    acc = None
    reps = max(1, min(3, steps))
    for _ in range(reps):
        step_device()
        prof = model.get_profile()
        if acc is None:
            acc = prof
        else:
            for k in acc:
                acc[k]["ms"] += prof[k]["ms"]
    model.set_profile(False)
    drain()
    torch.cuda.synchronize(dev)
    for k in acc:
        acc[k]["ms"] /= reps
    peaks = load_peaks()
    conv = acc["conv_igemm"]
    conv_tflops = conv["flops"] / (conv["ms"] * 1e-3) / 1e12 if conv["ms"] > 0 else 0.0
    step_ms = sum(v["ms"] for v in acc.values())
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "conv_igemm_traffic.json")
    if os.path.exists(tpath) and args.dtype == "bf16" and not batch:
        with open(tpath) as f:
            tj = json.load(f)
        traffic = tj.get(workload)
        traffic_src = tj.get("source", "ncu dram__bytes_read.sum + dram__bytes_write.sum over the conv launches of one step")

    images = world * B * steps
    value = images / (ms_dev * 1e-3)
    e2e = images / (ms_host * 1e-3)
    line = {
        "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms_dev / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {
            "workload": f"{arch} {'NuscenesDD3D' if nusc else 'DD3D'} {args.dtype}, batch {B} per GPU, {H}x{W} "
                        f"(padded to /{model.backbone.size_divisibility})" +
                        (f", raw HWC input resized on the GPU to {shape[1]}x{shape[2]}" if raw_mode else ""),
            "global_batch": world * B, "parallelism": f"dp{world}",
            "l2": "inputs (%.0f MB uint8) and activations (GBs) exceed the 126 MB L2; no explicit flush" %
                  (batch_t.numel() / 1e6),
            "collective": ("1 ncclAllGather per step of the packed [dets | counts | flags] buffer (%d B per rank) through "
                           "dd3d_allgather, on a side stream (overlaps the next forward; no host sync in the timed region)"
                           % packed[0].nbytes) if world > 1 else "none",
            "detections_per_step": n_det,
        },
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "images/s", "ms_per_step": ms_host / steps,
                "path": "dd3d_submit_host / dd3d_wait_host (double-buffered: H2D of step k+1 overlaps the kernels of step "
                        "k; every step still copies its inputs H2D and its detections D2H inside the timed region)"
                        if ms_host < ms_host_serial else "dd3d_forward_host (serial H2D -> kernels -> D2H)",
                "serial_ms_per_step": ms_host_serial / steps,
                "h2d_bytes_per_step": int(h_batch.numel() * h_batch.element_size() + h_K.numel() * 4 + h_sizes.numel() * 4),
                "d2h_bytes_per_step": int(h_out[0].numel() * 4 + h_cnt[0].numel() * 4 + (h_glob.numel() * 4 if nusc else 0))},
        "gpu_launches": (model.launches_per_forward() + (2 if nusc else 0)) * steps,
        "roofline": {
            "kernel": "conv_igemm_kernel (tcgen05 implicit GEMM, %d launches/step)" % conv["launches"],
            "bound": "tensor", "achieved": conv_tflops, "peak": peaks["tflops"], "unit": "TFLOP/s",
            "frac": conv_tflops / peaks["tflops"], "traffic": traffic,
            "traffic_source": ("static: " + traffic_src) if traffic is not None else "not captured for this configuration",
            "peak_source": peaks["source"],
            "algorithmic_flops_per_step": conv["flops"], "kernel_ms_per_step": conv["ms"],
            "share_of_step": conv["ms"] / step_ms if step_ms else None,
        },
        "kernels_ms_per_step": {k: round(v["ms"], 4) for k, v in acc.items()},
        "kernels_gbs": {k: round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) for k, v in acc.items()
                        if v["bytes"] and v["ms"] > 0},
    }
    if world > 1:
        line["rank_ms_per_step"] = rank_ms
        line["gathered_ok"] = gathered_ok
    if rank == 0 and world == 1 and with_cpu and args.cpu_images > 0:
        best, mean, cores, times, b = cpu_oracle_rate(workload, 1, warm=1, budget_s=30.0)
        line["cpu_baseline"] = {"value": mean, "unit": "images/s", "cores": cores, "kind": "port",
                                "sample": f"one forward of {b} image(s) {H}x{W} (BASELINE.md 3: min(B, 8) = {min(B, 8)} per "
                                          f"forward, bounded to ~30 s; CPU throughput is flat in the batch size) of the fp32 "
                                          f"CPU oracle port after a 1-image warm-up; {cpu_model()}, {cores} threads, torch "
                                          f"{torch.__version__}"}
    model._release()
    del model
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="v2_99", choices=list(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"],
                    help="16-bit storage type of activations / weights (fp16: BASELINE.json configs[4], the reference's "
                         "mixed-precision type); accumulation, head maps, decode and NMS are fp32 either way")
    ap.add_argument("--sweep", default="", help="comma list of per-GPU batch sizes: one JSON line per size (configs[4])")
    ap.add_argument("--cpu-images", type=int, default=2, help="0 disables the cpu_baseline leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the DLA-34 (configs[1]) leg of the default run")
    ap.add_argument("--input", default="mapped", choices=["mapped", "raw"],
                    help="raw: steps start from raw HWC uint8 dataset images (dd3d_forward_raw: ResizeShortestEdge to "
                         "INPUT.RESIZE.MIN_SIZE_TEST + intrinsics rescale on the GPU); not the BASELINE configuration")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the detections of the last timed step as DIR/<field>.npy (the DLA-34 leg of the default "
                         "run: secondary_<field>; --sweep: batch<B>_<field>)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout for the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    gatherers = {}
    if args.sweep:
        for b in [int(v) for v in args.sweep.split(",")]:
            line = run_workload(args, args.workload, b, rank, local_rank, world, gatherers, with_cpu=False,
                                dump_prefix=f"batch{b}_")
            if rank == 0:
                print(json.dumps(line), flush=True)
    else:
        line = run_workload(args, args.workload, args.batch, rank, local_rank, world, gatherers)
        default_run = (args.workload == "v2_99" and not args.batch and args.dtype == "bf16" and args.input == "mapped")
        if default_run and world == 1 and not args.no_secondary:
            # BASELINE.json configs[1] (DLA-34 bf16, batch 8, 384x1280) measured in the same process, so that a single
            # `bench.py` run records it too
            sec = run_workload(args, "dla34", 0, rank, local_rank, world, gatherers, with_cpu=False,
                               warmup=max(args.warmup, 5), dump_prefix="secondary_")
            line["secondary"] = {k: sec[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "dtype", "config",
                                                      "clocks", "e2e", "gpu_launches", "roofline", "kernels_ms_per_step")}
        if rank == 0:
            print(json.dumps(line), flush=True)
    for g in gatherers.values():
        g.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
