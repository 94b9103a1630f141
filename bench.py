#!/usr/bin/env python
"""bench.py -- frames/s of the ProPainter inference hot path on B200 (contract in the task statement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c2|c1|c3|c4|c5] [--no-cpu-baseline]
                  [--no-gpu-reference] [--no-strong] [--shard] [--dump-outputs DIR]

A "step" is one full pass of stages 1-4 (RAFT flow -> flow completion -> image propagation ->
sliding-window generator + compositing) over one synthetic clip.  N=1 workload = BASELINE.json
configs[1]: 80 frames, 432x240, object-removal mask, fp32, neighbor_length=10, ref_stride=10,
subvideo_length=80, raft_iter=20, random-init weights.
  value : frames/s with the uint8 clip + masks already resident in HBM
  e2e   : frames/s through ProPainterPipeline.__call__ with pinned HOST buffers: H2D of the clip
          and masks and D2H of the composited uint8 video inside the timed region
N>1: one clip per rank (clips are independent units; weak scaling, no data-path collective) -> `value`; in addition the
`strong` block times ONE 300-frame 1280x720 clip (BASELINE.json configs[3]) time-sharded over the N ranks by
propainter_b200/dist.py (point-to-point halo exchange over NCCL), at every N including 1, so that strong scaling
of the long-clip configuration can be read off the per-N lines.
--impl reference: the oracle (CPU restatement of the reference's PyTorch path) on the host cores
over a bounded sample of the same workload.
--dump-outputs DIR: after the timed steps, rank 0 writes the composited video its last timed step returned (see
dump_outputs); inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.
Two runs of one build (C2, one B200 at 1000 W) differed by one level in 0.2 % of the sampled values: compare with a
tolerance of one level.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "inpainted frames/sec at 432x240x80f"
WORKLOADS = {
    "c2": dict(T=80, H=240, W=432, mask="ellipse", raft_iter=20,
               name="C2: 80-frame 432x240 object-removal, neighbor_length=10 ref_stride=10 subvideo_length=80, fp32"),
    "c1": dict(T=8, H=128, W=128, mask="square", raft_iter=20, name="C1: 8-frame 128x128 square mask, fp32"),
    "c3": dict(T=80, H=240, W=432, mask="border", raft_iter=20,
               name="C3: 80-frame 432x240 video completion (25% border mask), fp32 storage"),
    "c4": dict(T=300, H=720, W=1280, mask="ellipse", raft_iter=20,
               name="C4: 300-frame 1280x720 object-removal, subvideo_length=80 ref_stride=10, fp32 storage"),
    "c5": dict(T=1000, H=1080, W=1920, mask="border", raft_iter=20,
               name="C5: 1000-frame 1920x1080 completion, subvideo_length=80, fp32 storage"),
}
STRONG_WORKLOAD = "c4"     # the long clip of BASELINE.json configs[3] that `strong` shards over the ranks
CPU_SAMPLE_FRAMES = 6      # bounded sample of the same workload for the CPU arm (full clip ~ 10 min of CPU)
DUMP_SAMPLE = 4 << 20      # --dump-outputs: elements kept of a larger output (4 B value + 8 B index each: 48 MiB)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons}


def _usable_cores():
    """Physical cores this process may use: min(affinity mask, cgroup CPU quota, physical cores in /proc/cpuinfo).
    One thread per hyper-thread sibling made the oracle 19x slower than one per core on the GPU box (128 vs 64 threads)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    try:
        cores, phys, core = set(), None, None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip() and phys is not None and core is not None:
                cores.add((phys, core))
                phys = core = None
        if cores:
            n = min(n, len(cores))
    except OSError:
        pass
    return max(1, n)


def _host_threads(torch):
    """Every usable physical core for the CPU arm whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1)."""
    n = _usable_cores()
    torch.set_num_threads(n)
    return n


def _seeded_state_dicts():
    from propainter_b200 import schemas
    from propainter_b200._params import ParamNet
    return {"raft": ParamNet(schemas.raft_schema(), seed=1).state_dict(), "rfc": ParamNet(schemas.rfc_schema(), seed=2).state_dict(),
            "gen": ParamNet(schemas.generator_schema(), seed=3).state_dict()}


def run_reference(args, wl, budget_s=240.0):
    """CPU arm: the oracle (restatement of the reference's PyTorch path, pinned by tests/golden) on ALL host cores over a
    bounded sample of the workload clip: its first T_s frames through the full 4-stage pipeline.  T_s is sized from one
    untimed calibration step so that warm-up + K timed steps stay within ~`budget_s` seconds (also under torchrun, where
    rank 0 alone runs and the other ranks exit)."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pipeline_ref
    from propainter_b200 import synth
    cores = _host_threads(torch)
    sds = _seeded_state_dicts()

    def step(T):
        u8, fm, md = synth.make_clip(T, wl["H"], wl["W"], mask=wl["mask"], seed=0)
        t0 = time.perf_counter()
        pipeline_ref.run_pipeline(sds, u8, fm, md, raft_iter=wl["raft_iter"])
        return time.perf_counter() - t0

    t_cal = step(2)                                                     # calibration (also warms the thread pool / allocator)
    n_steps = args.warmup + args.steps
    per_frame = t_cal / 2.0
    T = int(max(2, min(CPU_SAMPLE_FRAMES, wl["T"], budget_s / max(n_steps * per_frame, 1e-9))))
    times = []
    for i in range(n_steps):
        dt = step(T)
        if i >= args.warmup:
            times.append(dt)
    tot = sum(times)
    val = T * len(times) / tot
    sample = (f"first {T} frames of the workload clip ({wl['H']}x{wl['W']}), full 4-stage pipeline, raft_iter={wl['raft_iter']}, "
              f"{cores} host threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": wl["name"], "sample": sample},
        "cpu_baseline": {"value": val, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def _reference_cuda_setup(wl, dev):
    """The reference's PyTorch-CUDA execution plan: the oracle's functional restatement of the reference modules (pinned
    against the reference's own outputs, tests/golden) run on the GPU with stock torch / torchvision kernels --
    torchvision.ops.deform_conv2d for the deformable convs, per-window .cpu() compositing, torch defaults (cuDNN TF32 on,
    matmul TF32 off, cudnn.benchmark off).  None of propainter_b200's kernels are on this path."""
    import torch
    import torchvision
    from oracle import flowcomp_ref, generator_ref
    from propainter_b200 import synth

    def tv_deform(x, offset, mask, weight, bias):
        return torchvision.ops.deform_conv2d(x, offset, weight, bias, 1, 1, 1, mask)
    flowcomp_ref.deform_conv3x3 = tv_deform
    generator_ref.deform_conv3x3 = tv_deform
    u8, fm, md = synth.make_clip(wl["T"], wl["H"], wl["W"], mask=wl["mask"], seed=0)
    sds = {k: {n: v.to(dev) for n, v in sd.items()} for k, sd in _seeded_state_dicts().items()}
    return sds, u8, fm.to(dev), md.to(dev)


def gpu_reference(wl, dev, steps=2, warmup=1):
    """`gpu_reference` block of the bench line: frames/s of the reference's PyTorch-CUDA plan on this GPU for the same
    clip, (a) as the reference runs it, with torch.cuda.empty_cache() after every stage chunk / window
    (inference_propainter.py:323,360,395,452), and (b) without those calls (BASELINE.md section 2)."""
    import torch
    from oracle import pipeline_ref
    sds, u8, fm, md = _reference_cuda_setup(wl, dev)
    out = {}
    for key, ec in (("with_empty_cache", True), ("no_empty_cache", False)):
        times = []
        for i in range(warmup + steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pipeline_ref.run_pipeline(sds, u8, fm, md, raft_iter=wl["raft_iter"], empty_cache=ec)
            torch.cuda.synchronize()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        out[key] = {"value": wl["T"] * len(times) / sum(times), "ms_per_step": 1e3 * sum(times) / len(times)}
    out.update({"unit": "frames/s", "steps": steps, "warmup": warmup,
                "what": "oracle restatement of the reference modules on cuda:0 with stock torch/torchvision kernels (torch defaults)"})
    return out


def run_reference_cuda(args, wl):
    """Informational arm (not part of the driver contract): the denominator of north_star's ">= 10x the reference
    PyTorch-CUDA path" target at --steps / --warmup of your choice.  The normal bench line carries the same measurement
    as its `gpu_reference` block."""
    import torch
    if int(os.environ.get("RANK", "0")) != 0:
        return
    r = gpu_reference(wl, torch.device("cuda:0"), steps=args.steps, warmup=args.warmup)
    print(json.dumps({"impl": "reference-cuda", "metric": METRIC, "value": r["no_empty_cache"]["value"], "unit": "frames/s",
                      "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["no_empty_cache"]["ms_per_step"],
                      "higher_is_better": True, "dtype": "f32 (torch defaults: cuDNN TF32 on, matmul TF32 off)",
                      "data": "synthetic", "config": {"workload": wl["name"]}, "gpu_reference": r}))


def cpu_baseline(wl):
    import torch
    from oracle import pipeline_ref
    from propainter_b200 import synth
    cores = _host_threads(torch)
    T = min(CPU_SAMPLE_FRAMES, wl["T"])
    u8, fm, md = synth.make_clip(T, wl["H"], wl["W"], mask=wl["mask"], seed=0)
    sds = _seeded_state_dicts()
    t0 = time.perf_counter()
    pipeline_ref.run_pipeline(sds, u8, fm, md, raft_iter=wl["raft_iter"])
    dt = time.perf_counter() - t0
    return {"value": T / dt, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"first {T} frames of the workload clip, full 4-stage pipeline once ({dt:.1f} s), {cores} host threads"}


def dump_outputs(out_dir, comp):
    """The composited uint8 video [T,H,W,3] as float32 <out_dir>/comp.npy.  A video of more than DUMP_SAMPLE elements is
    written as a fixed sample: its values at DUMP_SAMPLE flat indices drawn once with seed 0, in ascending order, and those
    indices as float64 comp_index.npy."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    if comp.numel() > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(comp.numel(), DUMP_SAMPLE, replace=False))
        np.save(os.path.join(out_dir, "comp_index.npy"), idx.astype(np.float64))
        comp = comp.reshape(-1)[torch.from_numpy(idx).to(comp.device)]
    np.save(os.path.join(out_dir, "comp.npy"), comp.cpu().numpy().astype(np.float32))


def _time_kernel(torch, fn, reps=10):
    """CUDA events on the launch stream (= torch's current stream, which ops.* launch on), L2 flushed between reps."""
    flush = torch.empty(64 * 1024 * 1024, device="cuda")
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.mean(ts)


def roofline_probe(torch, pipe, wl):
    """Live roofline of our dominant kernels at the workload's shapes (DESIGN.md §4/§5).

    Primary entry = the tensor-core kernel the north star names (sparse window attention, tcgen05/TMEM); the
    `others` list carries the HBM-bound RAFT lookup and the deformable alignment.  ncu DRAM traffic figures
    (`traffic`, bytes per launch) come from the committed capture profiles/r2_ncu_kernels.csv (dram__bytes_read.sum +
    dram__bytes_write.sum of one `ncu --set full` pass over profiles/ncu_targets.py at these shapes; the lookup figure is the
    22-pair capture scaled to the batch; they cannot be measured outside a profiler and are only attached at the C2 shapes)."""
    from propainter_b200 import ops
    from propainter_b200.window_index import padded_grid, token_grid, window_key_table
    c2 = (wl["H"], wl["W"]) == (240, 432)
    ncu = (lambda mb: int(mb * 1e6)) if c2 else (lambda mb: None)
    hbm, bf16, src = peaks()
    tf32_peak = bf16 / 2.0                                          # tcgen05 kind::tf32 runs at half the bf16 rate
    dev = pipe.device
    # ---- sparse window attention: one transformer layer of a full generator window (t = 18 frames)
    t, C = 18, 512
    fh, fw = token_grid((wl["H"] // 4, wl["W"] // 4))
    H2, W2 = padded_grid(fh, fw)
    nwin = (H2 // 5) * (W2 // 9)
    qkv = torch.randn(t, H2 * W2, 3 * C, device=dev)
    pool = torch.randn(t, (H2 // 4) * (W2 // 4), 2 * C, device=dev)
    ktab = torch.from_numpy(window_key_table(H2, W2)).to(dev)
    flags = torch.zeros(nwin, dtype=torch.int32, device=dev)
    nmask = max(1, round(nwin * 5 / 16))                           # the C2 ellipse masks ~5 of 16 windows
    flags[:nmask] = 1
    nkf = len(range(0, t, 2))
    nkeys = nkf * (ktab.shape[1] + pool.shape[1])
    flops = nmask * 4 * 2 * 2 * (t * 45) * nkeys * 128             # QK^T + PV of the masked windows (SURVEY.md §8d)
    ms = _time_kernel(torch, lambda: ops.sparse_window_attn(qkv, pool, ktab, flags, t, H2 * W2, 0, 2))
    ach = flops / (ms * 1e-3) / 1e12
    primary = {"kernel": "k_sparse_attn_umma (+ unmasked-window kernel)", "bound": "tensor", "achieved": ach, "peak": tf32_peak,
               "unit": "TFLOP/s", "frac": ach / tf32_peak, "traffic": ncu(29.62 + 0.21), "peak_source": src + " bf16_tflops / 2 (TF32)",
               "launch_ms": ms, "algorithmic_flops": flops, "masked_windows": f"{nmask} of {nwin}"}
    # ---- RAFT correlation lookup, one refinement step of the whole clip
    h, w = wl["H"] // 8, wl["W"] // 8
    B = min(2 * (wl["T"] - 1), 158)
    fmap = torch.randn(B // 2 + 1, h * w, 256, device=dev)
    a = torch.arange(B // 2, device=dev, dtype=torch.int32)
    levels = ops.corr_alloc(B, h, w, dev)
    ops.corr_build(fmap, torch.cat([a, a + 1]), torch.cat([a + 1, a]), levels, h, w)
    ys, xs = torch.meshgrid(torch.arange(h, device=dev), torch.arange(w, device=dev), indexing="ij")
    coords = (torch.stack([xs, ys], -1).float()[None] + torch.randn(B, h, w, 2, device=dev) * 3).contiguous()
    out = torch.empty(B, h, w, 324, device=dev)
    ms_l = _time_kernel(torch, lambda: ops.corr_lookup(levels, coords, out))
    npx = h * w
    alg = B * (npx * 4 * 100 * 4 + npx * 324 * 4 + npx * 8)        # unique 10x10 patches at 4 levels + 324-ch output + coords
    ach_l = alg / (ms_l * 1e-3) / 1e9
    # ---- deformable alignment, one generator propagation step: sampling kernel + tcgen05 GEMM over the sampled columns
    Hh, Ww = wl["H"] // 4, wl["W"] // 4
    x, o = torch.randn(1, Hh, Ww, 128, device=dev), torch.randn(1, Hh, Ww, 432, device=dev)
    fl = torch.randn(1, Hh, Ww, 2, device=dev)
    wd = ops.pack_deform_weight_umma(torch.randn(128, 128, 3, 3, device=dev) * 0.03)
    bvec, dout = torch.randn(128, device=dev), torch.empty(1, Hh, Ww, 128, device=dev)
    cols = torch.empty(1, Hh, Ww, 9 * 128, device=dev)
    ms_g = _time_kernel(torch, lambda: ops.deform_gather(x, o, fl, 3.0, cols))
    ms_m = _time_kernel(torch, lambda: ops.conv_umma([cols], wd, 1, 1, 128, bias=bvec, out=dout))
    fl_d = Hh * Ww * 9 * 128 * 128 * 2
    # ---- the tcgen05 conv kernel on one 3x3 128->128 conv of a generator propagation step (bias + LeakyReLU + residual fused)
    xc = torch.randn(1, Hh, Ww, 128, device=dev)
    wc = ops.pack_conv_weight(torch.randn(128, 128, 3, 3, device=dev) * 0.03)
    rc, oc = torch.randn(1, Hh, Ww, 128, device=dev), torch.empty(1, Hh, Ww, 128, device=dev)
    ms_c = _time_kernel(torch, lambda: ops.conv_umma([xc], wc, 3, 3, 128, bias=bvec, act="leaky", slope=0.1, res=rc, out=oc))
    fl_c = Hh * Ww * 9 * 128 * 128 * 2
    primary["others"] = [
        {"key": "corr_lookup", "kernel": "k_corr_lookup_tma", "bound": "hbm", "achieved": ach_l, "peak": hbm, "unit": "GB/s", "frac": ach_l / hbm,
         "traffic": ncu((107.34 + 18.49) * B / 22.0), "launch_ms": ms_l, "algorithmic_bytes": alg},
        {"key": "deform", "kernel": "k_deform_gather + k_conv_umma (1x1 over the sampled columns)", "bound": "tensor",
         "achieved": fl_d / ((ms_g + ms_m) * 1e-3) / 1e12, "peak": tf32_peak, "unit": "TFLOP/s",
         "frac": fl_d / ((ms_g + ms_m) * 1e-3) / 1e12 / tf32_peak, "traffic": ncu(14.60 + 0.03 + 30.52 + 0.02), "launch_ms": ms_g + ms_m, "gather_ms": ms_g, "gemm_ms": ms_m,
         "algorithmic_flops": fl_d, "note": "two launches; the gather is L2-bandwidth bound (119 MB of corner reads per step)"},
        {"key": "conv", "kernel": "k_conv_umma 3x3 128->128 on the 60x108 map", "bound": "tensor", "achieved": fl_c / (ms_c * 1e-3) / 1e12,
         "peak": tf32_peak, "unit": "TFLOP/s", "frac": fl_c / (ms_c * 1e-3) / 1e12 / tf32_peak, "traffic": ncu(10.61), "launch_ms": ms_c,
         "algorithmic_flops": fl_c, "note": "single launch incl. launch latency; 112 CTAs on 148 SMs; tf32 operands from shared memory"}]
    return primary


def strong_block(torch, dist, pipe, dev, rank, world, steps=1, warmup=1):
    """One long clip (STRONG_WORKLOAD) cooperatively: every rank holds the uint8 clip + masks, computes its shard of every
    stage and exchanges halos point to point; device-timed, max over ranks.  world == 1: the plain single-GPU pipeline."""
    from propainter_b200 import synth
    from propainter_b200.inference_propainter import InferenceConfig
    wl = WORKLOADS[STRONG_WORKLOAD]
    u8_np, fm, md = synth.make_clip(wl["T"], wl["H"], wl["W"], mask=wl["mask"], seed=0)
    u8, fm, md = torch.from_numpy(u8_np).to(dev), fm.to(dev), md.to(dev)
    cfg = InferenceConfig(raft_iter=wl["raft_iter"])
    if world > 1:
        from propainter_b200.dist import ShardedProPainter
        runner = ShardedProPainter(pipe)
        step = lambda: runner(u8, fm, md, cfg)
    else:
        runner = None
        step = lambda: pipe(u8, fm, md, cfg)
    for _ in range(warmup):
        step()
    total = 0.0
    for _ in range(steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    t = torch.tensor([total], device=dev, dtype=torch.float64)
    sent = torch.tensor([sum(runner.last_bytes.values()) if runner else 0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(sent, op=dist.ReduceOp.SUM)
    out = {"workload": wl["name"], "scaling": "strong", "n_gpus": world, "steps": steps, "warmup": warmup,
           "value": wl["T"] * steps / (t.item() * 1e-3), "unit": "frames/s", "ms_per_clip": t.item() / steps,
           "p2p_bytes_per_clip": sent.item(), "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9,
           "exchange": "batched point-to-point (NCCL send/recv) of raw / completed flows, propagated frames, encoder features of "
                       "neighbour + reference frames, uint8 seam frames; no collective on the data path"}
    if runner is not None and rank == 0:
        out["p2p_bytes_rank0_by_stage"] = dict(runner.last_bytes)
    return out


def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        g.build()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        dist.barrier()
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    from propainter_b200 import ops, synth
    from propainter_b200.inference_propainter import InferenceConfig, ProPainterPipeline

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    shard = bool(args.shard) and world > 1
    u8_np, fm, md = synth.make_clip(wl["T"], wl["H"], wl["W"], mask=wl["mask"], seed=0 if shard else rank)
    u8_host = torch.from_numpy(u8_np).pin_memory()
    fm_host, md_host = fm.pin_memory(), md.pin_memory()
    out_host = torch.empty_like(u8_host).pin_memory()
    pipe = ProPainterPipeline(device=dev)
    cfg = InferenceConfig(raft_iter=wl["raft_iter"])
    if args.windows_in_flight:
        cfg.windows_in_flight = args.windows_in_flight
    u8_dev, fm_dev, md_dev = u8_host.to(dev), fm_host.to(dev), md_host.to(dev)
    flush = torch.empty(64 * 1024 * 1024, device=dev)          # 256 MiB > 126 MB L2

    runner = pipe
    if shard:                                                  # one clip time-sharded over the ranks (propainter_b200/dist.py)
        from propainter_b200.dist import ShardedProPainter
        runner = ShardedProPainter(pipe)

    last = {}                                                  # the latest resident step's result, for --dump-outputs

    def step_resident():
        r = runner(u8_dev, fm_dev, md_dev, cfg)
        last["comp"] = r[0] if shard else r
        return last["comp"]

    def dump_last():
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, last["comp"])

    def step_e2e():
        r = runner(u8_host, fm_host, md_host, cfg)             # H2D inside
        if shard:                                              # every rank reads back the frames whose final value it holds
            comp, ids = r
            out_host[:comp.shape[0]].copy_(comp, non_blocking=True)
            return comp
        out_host.copy_(r, non_blocking=True)                   # D2H of the result
        return r

    def timed(fn, steps, warmup, sample_clocks=False):
        for _ in range(warmup):
            fn()
        barrier()
        sampler = ClockSampler(local) if sample_clocks else None
        if sampler:
            sampler.start()
        l0 = ops.LAUNCHES
        total = 0.0
        ranged = sample_clocks and os.environ.get("PP_PROFILE_RANGE")     # ncu --profile-from-start off: timed steps only
        if ranged:
            torch.cuda.profiler.start()
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            total += e0.elapsed_time(e1)
        if ranged:
            torch.cuda.profiler.stop()
        barrier()
        clocks = sampler.stop() if sampler else None
        t = torch.tensor([total], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), ops.LAUNCHES - l0, clocks

    nfl = max(1, int(args.clips_in_flight)) if not shard else 1
    single = None
    if nfl > 1:
        # F independent engine replicas (same weights) on F streams: clip i+1's throughput-bound stages (RAFT, encoder, transformer)
        # fill the SMs that clip i's latency-bound recurrent scans leave idle.  Every step is still one full pass over one clip.
        pipes = [pipe] + [ProPainterPipeline(device=dev) for _ in range(nfl - 1)]
        streams = [torch.cuda.Stream(device=dev) for _ in range(nfl)]
        outs = [out_host] + [torch.empty_like(u8_host).pin_memory() for _ in range(nfl - 1)]

        def timed_pipelined(e2e, steps, warmup):
            def one(i):
                k = i % nfl
                if e2e:
                    outs[k].copy_(pipes[k](u8_host, fm_host, md_host, cfg), non_blocking=True)
                else:
                    last["comp"] = pipes[k](u8_dev, fm_dev, md_dev, cfg)
            main = torch.cuda.current_stream()
            for st in streams:
                st.wait_stream(main)
            for i in range(max(warmup, nfl)):                   # warm up on the streams the timed loop uses: the caching allocator
                with torch.cuda.stream(streams[i % nfl]):        # keeps one pool per stream, a first use would cudaMalloc inside the timing
                    one(i)
            for st in streams:
                main.wait_stream(st)
            barrier()
            sampler = ClockSampler(local) if not e2e else None
            if sampler:
                sampler.start()
            l0 = ops.LAUNCHES
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for st in streams:
                st.wait_stream(main)
            for i in range(steps):
                with torch.cuda.stream(streams[i % nfl]):
                    flush.zero_()
                    one(i)
            for st in streams:
                main.wait_stream(st)
            e1.record()
            torch.cuda.synchronize()
            barrier()
            clocks = sampler.stop() if sampler else None
            t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item(), ops.LAUNCHES - l0, clocks

        ms_one, _, _ = timed(step_resident, min(args.steps, 3), args.warmup)          # latency of one clip alone, for the record
        single = {"ms_per_clip": ms_one / min(args.steps, 3), "frames_per_s": wl["T"] * min(args.steps, 3) / (ms_one * 1e-3)}
        ms_total, launches, clocks = timed_pipelined(False, args.steps, args.warmup)
        dump_last()
        ms_e2e, _, _ = timed_pipelined(True, args.steps, 1)
    else:
        ms_total, launches, clocks = timed(step_resident, args.steps, args.warmup, True)
        dump_last()
        ms_e2e, _, _ = timed(step_e2e, args.steps, 1)
    strong = None
    frames_total = wl["T"] * (1 if shard else world) * args.steps
    if rank == 0:
        line = {
            "metric": METRIC, "value": frames_total / (ms_total * 1e-3), "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong" if shard else "weak", "vs_baseline": None, "dtype": "f32 (TF32 tensor-core products, fp32 accumulate)",
            "data": "synthetic",
            "config": {"workload": wl["name"], "frames_per_step_per_gpu": wl["T"], "parallelism": (f"one clip time-sharded x{world} (NCCL broadcast of stage 1-3 results + seam send/recv)" if shard
                                       else f"clip-parallel x{world} (independent clips, no data-path collective)"),
                       "weights": "random-init (seeded)", "l2": "256 MiB flush between timed steps",
                       "clips_in_flight": nfl},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": frames_total / (ms_e2e * 1e-3), "unit": "frames/s",
                    "h2d_bytes_per_step": u8_host.numel() + 4 * (fm_host.numel() + md_host.numel()),
                    "d2h_bytes_per_step": out_host.numel()},
        }
        from propainter_b200 import autotune
        plans = {}
        for k, v in autotune.choices().items():                    # which measured plan each step replays (stderr, not the line)
            plans.setdefault(f"{k[0]}[{v}]", []).append(str(k[1:3]))
        print("autotune plans:", {k: (len(v), v[:4]) for k, v in plans.items()}, file=sys.stderr)
        print("graph-timed plan candidates (ms):", {f"{k[0][0]}{k[0][1:]}#{k[1]}": round(v, 3) for k, v in autotune._timings.items()}, file=sys.stderr)
        try:
            line["roofline"] = roofline_probe(torch, pipe, wl)
            for o in line["roofline"].pop("others", []):           # flat top-level copies (nested lists get dropped by parsers)
                line["roofline_" + o.pop("key")] = o
        except Exception as exc:                                   # never lose the headline line to the probe
            line["roofline"] = {"error": repr(exc)}
        if single is not None:
            line["single_clip"] = single
        if world == 1 and not args.no_gpu_reference:
            try:                                                   # the >= 10x target's denominator, same box, same clip
                torch.cuda.empty_cache()
                line["gpu_reference"] = gpu_reference(wl, dev)
                line["gpu_reference"]["speedup_e2e"] = line["e2e"]["value"] / line["gpu_reference"]["no_empty_cache"]["value"]
            except Exception as exc:
                line["gpu_reference"] = {"error": repr(exc)}
    if not args.no_strong and not shard and args.workload == "c2":
        # last GPU block: its engine (own graph caches) is dropped afterwards.  Every rank takes part.
        try:
            import gc
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats(dev)
            spipe = ProPainterPipeline(device=dev)
            strong = strong_block(torch, dist, spipe, dev, rank, world)
            del spipe
            gc.collect()
            torch.cuda.empty_cache()
        except Exception as exc:                                   # never lose the headline line to the extra block
            strong = {"error": repr(exc)}
            if world > 1:
                raise
    if rank == 0:
        if strong is not None:
            line["strong"] = strong
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(wl)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the `strong` block (one 300-frame 720p clip sharded over the ranks)")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the gpu_reference block (reference PyTorch-CUDA plan, ~10 s)")
    ap.add_argument("--windows-in-flight", type=int, default=0, help="override InferenceConfig.windows_in_flight")
    ap.add_argument("--clips-in-flight", type=int, default=1,
                    help="engine replicas per GPU working on consecutive clips concurrently (each step is still one full clip)")
    ap.add_argument("--shard", action="store_true", help="N>1: cooperate on ONE clip (strong scaling) instead of one clip per rank")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the composited video of the last timed step under DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    elif args.impl == "reference-cuda":
        run_reference_cuda(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
