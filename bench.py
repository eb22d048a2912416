#!/usr/bin/env python
"""bench.py -- scenes/sec of the NeRF-RPN hot path (BASELINE.json config 2: ResNet50-3D + FPN + anchor head, 160x256x256 RGB-sigma
grids, 13 anchors/location, top-2500 per level, NMS 0.3) plus, in the same JSON line, the legs that explain it.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

One "step" = `scenes_per_step` scenes per rank through backbone -> FPN -> head -> decode / top-k -> NMS -> proposals (weak scaling:
scenes are independent, no collective on the inference path; SURVEY.md 8e).  ONE JSON line (contract in the task statement):
  value          whole-job scenes/s, inputs resident in HBM, device-timed, max over ranks
  e2e            the same metric through the public pipeline with pinned HOST grids (H2D + D2H inside the timed region); `forward_api`
                 inside it = NeRFRegionProposalNetwork.forward itself with the reference's own methodology (run_rpn.py:594-617)
  roofline       dominant kernel (tcgen05 implicit-GEMM conv, one RPN-head layer over P2..P5) timed live with CUDA events
  variants       other loads on the same box: seed-0 weights (round-1 line), rotated boxes (--rotated_bbox: polygon-clip NMS), one scene per
                 launch, bf16 (BASELINE's dtype, 8e-3 feature parity)
  train          BASELINE config 4: one training step (forward + losses + backward + clip + AdamW) per rank on one 160x256x256 scene with
                 rotated boxes, the flat gradient bucket all-reduced over NCCL and overlapped with the backward pass
  reference_gpu  the INCUMBENT: the unmodified reference (oracle/_ref: cuDNN + ATen + Python NMS + its own K1) on this GPU (rank 0, N = 1)
  cpu_baseline   the reference on this box's host cores (N = 1): its own modules when oracle/_ref is staged, else the oracle's port

`--impl reference` times the reference on the host CPU only: the unmodified reference modules from oracle/_ref when staged
(cpu_baseline.kind "reference"), else the fp32 port oracle/net.py ("port").
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIMS = (160, 256, 256)
ANCHOR_SIZES = ((8,), (16,), (32,), (64,),)
ASPECT = (((1., 1., 1.), (1., 1., 2.), (1., 2., 2.), (1., 1., 3.), (1., 3., 3.)),) * 4
SPREAD = 30.0                     # cls_logits.weight multiplier of the score-spread variant (SURVEY.md 8d: seed-0 init gives ~0.5 everywhere)
WORKLOAD = ("ResNet50-3D+FPN+anchor-head(AABB) 160x256x256x4 RGBsigma, 13 anchors/loc, pre/post-NMS top 2500, NMS 0.3, "
            f"reference init seed 0 with cls_logits.weight x{SPREAD:g} (spread objectness)")
FLOPS_PER_SCENE = 3.913e12        # SURVEY.md 8(d): conv FLOPs (2*MAC) of the reference's layers


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=None, choices=["bf16", "fp16", "fp16_w2"],
                    help="numeric mode (nerf_rpn_b200/precision.py); default fp16_w2 = the mode that meets north_star's <= 1e-3 on feature maps")
    ap.add_argument("--input-layout", default="dataset", choices=["dataset", "ncdhw", "dataset_u8"],
                    help="input grids: the dataset's fp32 channels-last view (default), contiguous fp32 (4,W,L,H), or the raw uint8 "
                         "channels-last view (uint8 npz files; normalised on the device instead of by datasets.py:59-61 on the host)")
    ap.add_argument("--skip-cpu-baseline", action="store_true", help="exploration runs only: omit the CPU timing")
    ap.add_argument("--skip-extras", action="store_true", help="exploration runs only: omit variants / train / reference_gpu legs")
    ap.add_argument("--scenes-per-step", type=int, default=int(os.environ.get("NRPN_SCENES_PER_STEP", "4")),
                    help="scenes per rank per step (one engine launch); weights are read once per step")
    ap.add_argument("--cpu-train-baseline", action="store_true", help=argparse.SUPPRESS)       # child process of --mode train
    ap.add_argument("--mode", default="infer", choices=["infer", "train"],
                    help="infer (default): the headline; train: BASELINE config 4's training step as the line's value (the default line carries it under `train`)")
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 5],
                    help="BASELINE.json configuration: 2 = the headline (default); 1 = VGG19 + anchor head on a 32^3 grid; 3 = Swin-S + FCOS (OBB) on "
                         "200x200x130; 5 = oriented IoU + NMS sweep 1k..1M boxes")
    ap.add_argument("--weights", default="spread", choices=["spread", "seed0"], help="headline weights: spread objectness (default) or plain seed-0 init")
    ap.add_argument("--rotated", action="store_true", help="headline with --rotated_bbox (8 deltas, OBB decode, polygon-clip NMS)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of the default run (config 2 inference), write the last step's proposals, scores and levels of every "
                         "scene as DIR/<name>.npy (float32), so that two builds can be compared output for output on the same seeded inputs; the other "
                         "configurations and modes are comparison legs of their own and are not dumped")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.mode != "infer" or args.config != 2):
        ap.error("--dump-outputs applies to the headline run (--impl b200 --mode infer --config 2)")
    return args


def dump_outputs(path, plan, prefix=""):
    """What a caller of the engine receives from the last timed step: per scene, the proposals (count x 6 or 7), their objectness scores and
    pyramid levels, as float32 .npy files (4 scenes x 2 500 proposals: well under 1 MB)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    count = plan.out_count.cpu()
    boxes, scores, levels = plan.out_boxes.cpu(), plan.out_scores.cpu(), plan.out_levels.cpu()
    for b in range(count.numel()):
        k = int(count[b])
        for name, t in (("boxes", boxes), ("scores", scores), ("levels", levels)):
            np.save(os.path.join(path, f"{prefix}scene{b}_{name}.npy"), t[b, :k].float().numpy())


def synth_scene(i, layout="ncdhw"):
    """Scene i of SURVEY.md 8(d): U[0,1) RGB + alpha, channels-last on disk like the real npz -> (4,W,L,H) fp32.
    layout "dataset": the (4,W,L,H) VIEW of the (W,L,H,4) array, exactly what datasets.py:55-56 hands to the model;
    layout "ncdhw": the same values as a contiguous (4,W,L,H) tensor (what the reference's torch.stack makes of it)."""
    import torch
    g = torch.Generator().manual_seed(1000 + i)
    grid = torch.rand(*DIMS, 4, generator=g)
    return grid.permute(3, 0, 1, 2) if layout == "dataset" else grid.permute(3, 0, 1, 2).contiguous()


def planted_boxes(i, n_gt=16, rotated=True):
    """Ground truth of scene i for the training leg: n_gt cuboids, sizes U[8,64], yaw U[-pi/2, pi/2) (SURVEY.md 8d)."""
    import math
    import torch
    g = torch.Generator().manual_seed(5000 + i)
    d = torch.tensor(DIMS, dtype=torch.float32)
    size = torch.rand(n_gt, 3, generator=g) * 56.0 + 8.0
    ctr = torch.rand(n_gt, 3, generator=g) * (d - 16.0) + 8.0
    if rotated:
        return torch.cat([ctr, size, (torch.rand(n_gt, 1, generator=g) - 0.5) * math.pi], 1)
    return torch.cat([ctr - size / 2, ctr + size / 2], 1)


def build_modules(rotated=False, spread=SPREAD):
    import torch
    from nerf_rpn_b200.model.anchor import AnchorGenerator3D, RPNHead
    from nerf_rpn_b200.model.feature_extractor import Bottleneck, ResNet_FPN_256
    torch.manual_seed(0)
    backbone = ResNet_FPN_256(Bottleneck, [3, 4, 6, 3], input_dim=4, is_max_pool=True)
    ag = AnchorGenerator3D(ANCHOR_SIZES, ASPECT)
    head = RPNHead(256, ag.num_anchors_per_location()[0], 4, rotate=rotated)
    if spread:
        with torch.no_grad():
            head.cls_logits.weight.mul_(spread)
    return backbone, ag, head


def build_model(rotated=False, spread=SPREAD, precision=None):
    from nerf_rpn_b200.model.nerf_rpn import NeRFRegionProposalNetwork
    backbone, ag, head = build_modules(rotated, spread)
    return NeRFRegionProposalNetwork(backbone, ag, head, rpn_pre_nms_top_n_test=2500, rpn_post_nms_top_n_test=2500, rpn_nms_thresh=0.3,
                                     rpn_score_thresh=0.0, rpn_fg_iou_thresh=0.35, rpn_bg_iou_thresh=0.2, rotated_bbox=rotated, precision=precision)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
        except OSError:
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for k, nm in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ the reference on the host CPU
_CPU = {}


def _cpu_state():
    """The reference on the host: its own modules (oracle/_ref, eval mode, AABB head: no native op on that path) when staged, else the
    oracle's fp32 port.  Same seed-0 + spread weights and scene as the B200 arm."""
    if _CPU:
        return _CPU
    import torch
    backbone, ag, head = build_modules()
    _CPU["scene"] = synth_scene(0)
    _CPU["kind"] = "port"
    _CPU["sd"] = {k: v.detach() for k, v in backbone.state_dict().items()}
    _CPU["hsd"] = {k: v.detach() for k, v in head.state_dict().items()}
    _CPU["cells"] = ag.cell_anchors_np()
    try:
        from oracle import ref_gpu
        if ref_gpu.available():
            sys.path.insert(0, os.path.join(ROOT, "tools", "ref_stub"))      # import-time stand-in for the native op; the AABB path never calls it
            try:
                ref = ref_gpu.load(need_k1=False)
            finally:
                sys.path.remove(os.path.join(ROOT, "tools", "ref_stub"))
            m = ref_gpu.build_reference_model(rotated=False, seed=0, spread=SPREAD).eval()
            _CPU["model"], _CPU["kind"] = m, "reference"
    except Exception as e:                                                   # noqa: BLE001 -- fall back to the port, say why
        _CPU["why_port"] = repr(e)
    return _CPU


def cpu_run(x_extent, n_threads, repeats=1, y_extent=None):
    """Time the reference on an (x_extent x y_extent x 256) block of the scene (x_extent*y_extent/(160*256) of a scene). Seconds per run."""
    import torch
    torch.set_num_threads(n_threads)
    st = _cpu_state()
    y_extent = DIMS[1] if y_extent is None else y_extent
    x = st["scene"][:, :x_extent, :y_extent].contiguous()
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        with torch.no_grad():
            if st["kind"] == "reference":
                st["model"]([x.clone()])
            else:
                from oracle import net as onet
                onet.full_forward(st["sd"], st["hsd"], x[None], st["cells"], False)
        times.append(time.perf_counter() - t0)
    return times


def best_cpu_threads():
    """Intra-op thread count that makes the CPU run fastest on this host: all cores is NOT it on a 128-thread box (measured on the B200 host:
    full scene 4.2 s with 32 threads vs 33 s with 128 -- profiles/r01_cpu_port_threads.txt). Sweeps {all, 64, 32, 16, 8} on a small block."""
    cores = os.cpu_count() or 1
    # more than 64 intra-op threads only ever lost on the B200 host (128 threads: 45 s per block vs 0.5 s with 16): not swept
    cands = sorted({c for c in (min(cores, 64), 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    cpu_run(32, min(cands), y_extent=64)                       # library warm-up (oneDNN JIT, thread pool), not timed
    sweep = {}
    for th in cands:
        sweep[th] = min(cpu_run(32, th, y_extent=128, repeats=2))
    best = min(sweep, key=sweep.get)
    return best, {k: round(v, 2) for k, v in sweep.items()}


def _cpu_desc(cores, sweep):
    import torch
    st = _cpu_state()
    what = ("the UNMODIFIED reference modules (oracle/_ref: NeRFRegionProposalNetwork.forward incl. its Python NMS loop) on the host CPU"
            if st["kind"] == "reference" else "oracle/net.py fp32 port of the reference")
    return f"{what}, torch {torch.__version__}, {cores} of {os.cpu_count()} threads = the fastest of the sweep {sweep}"


def run_reference(args):
    """--impl reference: the reference on the host cores; each step = a bounded block of the workload, sized so that the whole
    (warmup + steps) run stays within a few minutes whatever K is."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores, sweep = best_cpu_threads()
    torch.set_num_threads(cores)
    per_full = cpu_run(160, cores)[0]                          # one full scene with the chosen thread count
    budget = 150.0
    frac = budget / (per_full * (args.steps + args.warmup))
    cands = sorted(((ex * ey) / float(DIMS[0] * DIMS[1]), ex, ey) for ex in (32, 64, 96, 128, 160) for ey in (64, 128, 256))
    pick = cands[0]
    for c in cands:
        if c[0] <= frac:
            pick = c
    share, ex, ey = pick
    for _ in range(args.warmup):
        cpu_run(ex, cores, y_extent=ey)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_run(ex, cores, y_extent=ey)
    dt = time.perf_counter() - t0
    value = args.steps * share / dt
    sample = f"{ex}x{ey}x{DIMS[2]} block per step = {share:.3f} scene; full scene {per_full:.2f} s ({_cpu_desc(cores, sweep)})"
    out = {"impl": "reference", "metric": "scenes/sec", "value": value, "unit": "scenes/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD, "sample": sample},
           "cpu_baseline": {"value": value, "unit": "scenes/s", "cores": cores, "kind": _cpu_state()["kind"], "sample": sample},
           "e2e": {"value": value, "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    _emit(out)


# ------------------------------------------------------------------------------------------------ B200 arm
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json)"
    return 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


def time_dominant_kernel(plan, reps=10):
    """CUDA-event time of the dominant kernel: the first RPN-head layer (3^3 256->256 + ReLU over P2..P5 in one launch)."""
    import torch
    f = plan.head_launches[0]
    f(); torch.cuda.synchronize()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    times = []
    for _ in range(reps):
        flush.zero_()                       # evict L2 between repetitions
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); f(); b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    vox = plan.n * sum(d[0] * d[1] * d[2] for d in plan.feat_dims)
    flops = 2.0 * vox * 256 * 256 * 27
    return statistics.mean(times), min(times), flops


def device_throughput(model, dev_batches, K, W, barrier, sampler=None):
    """K engine steps over resident input batches; returns (ms, plan, proposals of the last scene).  `sampler`: clock sampler started
    right before the timed region (after the warm-up), so that its median is the clock UNDER LOAD."""
    import torch
    eng = model.engine()
    with torch.no_grad():
        for i in range(max(W, 4)):                            # >= 4: both buffer parities warmed and captured
            plan = eng.forward_device(dev_batches[i % len(dev_batches)])
        barrier()
        if sampler is not None:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            plan = eng.forward_device(dev_batches[i % len(dev_batches)])
        torch.cuda.current_stream().wait_event(plan.done)     # the last scene's post-processing (side stream)
        e1.record()
        barrier()
    return e0.elapsed_time(e1), plan, int(plan.out_count[0].item())


def train_leg(rank, local, world, barrier, steps=8, warm=4):       # warm-up covers the two eager steps + the graph capture of the launch lists
    """BASELINE config 4: ResNet50-FPN + anchor head, --rotated_bbox, one 160x256x256 scene per rank per step, data parallel: forward,
    target assignment + sampling + losses, backward (dgrad / wgrad on tcgen05), NCCL all-reduce of the flat gradient bucket overlapped
    with the backward pass, clip_grad_norm_(0.1) + AdamW.  bf16 activations / gradients, fp32 master weights and accumulation."""
    import torch
    import torch.distributed as dist
    model = build_model(rotated=True, spread=0.0).cuda().train()
    eng = model.train_engine(precision="bf16", lr=1e-4, weight_decay=0.01, clip_grad_norm=0.1, reg_loss_weight=5.0,
                             process_group=dist.group.WORLD if world > 1 else None)
    grids = [synth_scene(rank * 1000 + i, "dataset").permute(1, 2, 3, 0).contiguous().cuda().permute(3, 0, 1, 2)[None] for i in range(2)]
    gts = [[planted_boxes(rank * 1000 + i).cuda()] for i in range(2)]
    for i in range(warm):
        eng.train_step(grids[i % 2], gts[i % 2])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        losses = eng.train_step(grids[i % 2], gts[i % 2])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    plan = eng.plan(1, DIMS)
    out = {"metric": "training scenes/sec", "value": world * steps / (ms * 1e-3), "unit": "scenes/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warm,
           "scaling": "weak", "dtype": "bf16 activations / gradients, fp32 master weights + accumulation",
           "config": "ResNet50-3D+FPN+anchor head --rotated_bbox, 1 scene (160x256x256) per rank per step, 16 planted OBBs, sample 256 anchors, "
                     "smooth-L1 + BCE, clip 0.1, AdamW (BASELINE config 4)",
           "collective": (f"NCCL all-reduce (sum) of the flat fp32 gradient bucket, {eng.n_params} parameters = {eng.n_params * 4 / 1e6:.0f} MB per step, "
                          f"{getattr(plan, 'allreduce_calls', 0)} chunks launched as the backward pass finalises them (head -> FPN -> stages -> stem)")
                         if world > 1 else "none at N = 1 (the all-reduce is skipped)",
           "losses_last_step": [round(v, 5) for v in losses.tolist()], "params": eng.n_params}
    del eng, model
    torch.cuda.empty_cache()
    return out


def forward_api_leg(model, host_grid, reps=100, warm=10):
    """NeRFRegionProposalNetwork.forward through the reference's own benchmark methodology (run_rpn.py:594-617: eval mode, warm-up, CUDA events
    around model([grid]), synchronize per repetition), one scene per call, grid copied from pinned host memory inside the timed region like
    run_rpn.py:473 (`item.cuda()`), proposals copied back like :507."""
    import torch
    times = []
    with torch.no_grad():
        for i in range(warm + reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            x = host_grid.cuda(non_blocking=True)
            (feats, props, lv), _, scores = model([x])
            _ = props[0].cpu()
            b.record()
            torch.cuda.synchronize()
            if i >= warm:
                times.append(a.elapsed_time(b))
    return {"ms_per_scene": statistics.mean(times), "std_ms": statistics.pstdev(times), "scenes_per_s": 1000.0 / statistics.mean(times), "reps": reps,
            "warmup": warm, "api": "NeRFRegionProposalNetwork.forward([grid]) (features returned as fp32 NCDHW views), run_rpn.py:594-617 methodology",
            "h2d_bytes_per_step": host_grid.numel() * host_grid.element_size(), "d2h_bytes_per_step": int(props[0].numel() * 4)}


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device -- the B200 arm has no CPU fallback (use --impl reference for the CPU reference)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    from nerf_rpn_b200 import precision as nprec
    from nerf_rpn_b200.runtime import ScenePipeline
    args.precision = nprec.resolve(args.precision)
    spread = SPREAD if args.weights == "spread" else 0.0
    model = build_model(rotated=args.rotated, spread=spread, precision=args.precision).cuda().eval()
    eng = model.engine()
    B = max(1, args.scenes_per_step)
    n_pool = 4                                             # 4 x 168 MB of distinct inputs (> 126 MB L2)
    if args.input_layout == "dataset_u8":   # raw uint8 (W,L,H,4) arrays as stored in uint8 npz files
        host = [(synth_scene(rank * 1000 + i, "dataset").permute(1, 2, 3, 0) * 255.0).round().to(torch.uint8).contiguous().pin_memory()
                .permute(3, 0, 1, 2) for i in range(n_pool)]
    elif args.input_layout == "dataset":    # pinned (W,L,H,4) arrays, handed over as (4,W,L,H) views like the reference's dataset does
        host = [synth_scene(rank * 1000 + i, "dataset").permute(1, 2, 3, 0).contiguous().pin_memory().permute(3, 0, 1, 2) for i in range(n_pool)]
    else:
        host = [synth_scene(rank * 1000 + i).pin_memory() for i in range(n_pool)]
    hdev = [h.cuda() for h in host]

    def batches(b):
        if args.input_layout in ("dataset", "dataset_u8"):      # keep the (B,X,Y,Z,4) memory order: logical (B,4,X,Y,Z) views
            return [torch.stack([hdev[(i + k) % n_pool].permute(1, 2, 3, 0) for k in range(b)], 0).permute(0, 4, 1, 2, 3) for i in range(n_pool)]
        return [torch.stack([hdev[(i + k) % n_pool] for k in range(b)], 0) for i in range(n_pool)]
    dev = batches(B)
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (headline)
    sampler = ClockSampler(local)
    ms, plan, count = device_throughput(model, dev, K, W, barrier, sampler if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:                                  # before the pipeline below reuses the plan's output buffers
        dump_outputs(args.dump_outputs, plan, f"rank{rank}_" if world > 1 else "")

    # ---- end to end through the streaming pipeline (pinned host grids in, proposals out on the host)
    with torch.no_grad():
        pipe = ScenePipeline(model, DIMS, batch=B)
        pipe.run([host[i % n_pool] for i in range(W * B)], collect=True)
        barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e2.record()
        res = pipe.run([host[i % n_pool] for i in range(K * B)], collect=True)
        e3.record()
        barrier()
        wall_ms = 1000.0 * (time.perf_counter() - t0)
        ms_e2e = max(e2.elapsed_time(e3), wall_ms)         # host-side collection included
        assert len(res) == K * B
    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()

    launches_per_step = plan.num_launches() if rank == 0 else 0
    torch.cuda.synchronize()
    roofline = None
    fwd_api = None
    if rank == 0:
        k_mean, k_min, k_flops = time_dominant_kernel(plan)
        burst, sustained, how = measured_peaks()
        achieved = k_flops / (k_mean * 1e-3) / 1e12
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "r02_ncu_full_summary.json")) as f:
                for row in json.load(f):
                    if row.get("capture") == "head":
                        traffic = (row["dram_read_B"] + row["dram_write_B"]) * B
        except (OSError, ValueError, KeyError):
            traffic = None
        roofline = {"bound": "tensor", "kernel": "conv3d_igemm_kernel<256,4> (RPN head layer, 3x3x3 256->256 + bias + ReLU over P2..P5)",
                    "achieved": achieved, "peak": burst, "unit": "TFLOP/s", "frac": achieved / burst, "traffic": traffic,
                    "traffic_source": "profiles/r02_ncu_full_summary.json (dram__bytes_read.sum + dram__bytes_write.sum of an ncu --set full capture, 1 scene/launch) x scenes per launch; a profile number, not measured in this run",
                    "peak_source": how + ", burst figure (kernel timed alone, L2 flushed between launches)",
                    "launch_ms": k_mean, "flops_per_launch": k_flops,
                    "whole_step_frac_of_sustained": (FLOPS_PER_SCENE * world * K * B / (ms * 1e-3) / 1e12) / (sustained * world)}
        if world == 1 and not args.skip_extras:
            fwd_api = forward_api_leg(model, host[0])
    del pipe
    value = world * K * B / (ms * 1e-3)

    # ---- other loads on the same box (device-resident, same method)
    variants = {}
    train = None
    ref_gpu_out = None
    if not args.skip_extras:
        del model, eng, plan
        torch.cuda.empty_cache()
        Kv = max(8, K // 4)
        specs = [("seed0_weights", dict(rotated=False, spread=0.0, precision=args.precision), B),
                 ("rotated_bbox", dict(rotated=True, spread=SPREAD, precision=args.precision), B),
                 ("one_scene_per_step", dict(rotated=False, spread=SPREAD, precision=args.precision), 1),
                 ("bf16", dict(rotated=False, spread=SPREAD, precision="bf16"), B)]
        for name, kw, b in specs:
            m = build_model(**kw).cuda().eval()
            vms, vplan, vcount = device_throughput(m, dev if b == B else batches(b), Kv, W, barrier)
            tt = torch.tensor([vms], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            variants[name] = {"value": world * Kv * b / (float(tt.item()) * 1e-3), "unit": "scenes/s", "ms_per_step": float(tt.item()) / Kv, "scenes_per_step_per_gpu": b,
                              "steps": Kv, "proposals_last_scene": vcount, "precision": kw["precision"]}
            del m, vplan
            torch.cuda.empty_cache()
        train = train_leg(rank, local, world, barrier)
        if rank == 0 and world == 1:
            try:
                from oracle import incumbent
                ref_gpu_out = {"tf32_default": incumbent.time_reference_gpu(DIMS, rotated=False, spread=SPREAD, tf32=True, warmup=1, reps=3, budget_s=25.0),
                               "fp32": incumbent.time_reference_gpu(DIMS, rotated=False, spread=SPREAD, tf32=False, warmup=1, reps=2, budget_s=15.0)}
            except Exception as e:                           # noqa: BLE001
                ref_gpu_out = {"unavailable": repr(e)}

    out = None
    if rank == 0:
        cores = os.cpu_count() or 1
        sweep = {}
        torch.cuda.empty_cache()
        if args.skip_cpu_baseline or world > 1:            # the CPU baseline is timed on rank 0 of the single-GPU run only
            cpu_t, cpu_sample, cpu_kind = float("nan"), "not timed in this run (N > 1 or --skip-cpu-baseline)", "port"
        else:
            cores, sweep = best_cpu_threads()              # all 128 hardware threads are 8x SLOWER than 32 on the B200 host
            cpu_t = statistics.mean(cpu_run(160, cores, repeats=2))
            cpu_kind = _cpu_state()["kind"]
            cpu_sample = f"2 full scenes 160x256x256, mean ({_cpu_desc(cores, sweep)})"
        out = {"metric": "scenes/sec", "value": value, "unit": "scenes/s", "n_gpus": world, "steps": K, "warmup": W,
               "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": nprec.bench_dtype(args.precision),
               "data": "synthetic",
               "config": {"workload": WORKLOAD if (args.weights == "spread" and not args.rotated) else WORKLOAD + f" [weights={args.weights}, rotated={args.rotated}]",
                          "precision": args.precision, "feature_map_parity": "<= 1e-3 norm-wise vs the reference's fp32 on this GPU at 160x256x256 "
                          "(tests/test_gpu_reference.py)" if args.precision == "fp16_w2" else "see DESIGN.md section 4",
                          "scenes_per_step_per_gpu": B, "parallelism": f"dp{world} (scenes shard over ranks, no collective on the inference path)",
                          "l2": "4 distinct 168 MB input grids per rank cycled (> 126 MB L2); activations stream ~1.5 GB/scene",
                          "proposals_last_scene": count,
                          "input_layout": {"dataset": "fp32 (4,W,L,H) views of (W,L,H,4) arrays, as datasets.py:55-56 yields",
                                           "dataset_u8": "raw uint8 (4,W,L,H) views of (W,L,H,4) arrays, normalised on the device",
                                           "ncdhw": "fp32 contiguous (4,W,L,H)"}[args.input_layout]},
               "clocks": clocks,
               "e2e": {"value": world * K * B / (ms_e2e * 1e-3), "unit": "scenes/s", "h2d_bytes_per_step": int(4 * DIMS[0] * DIMS[1] * DIMS[2] * host[0].element_size() * B),
                       "d2h_bytes_per_step": int((2500 * (7 if args.rotated else 6) + 2 * 2500 + 1) * 4 * B), "ms_per_step": ms_e2e / K,
                       "api": "nerf_rpn_b200.runtime.ScenePipeline.run (pinned host grids -> host proposals)", "forward_api": fwd_api},
               "gpu_launches": launches_per_step * K,
               "roofline": roofline,
               "variants": variants,
               "train": train,
               "reference_gpu": ref_gpu_out,
               "cpu_baseline": {"value": (1.0 / cpu_t) if cpu_t == cpu_t else None, "unit": "scenes/s", "cores": cores, "kind": cpu_kind, "sample": cpu_sample}}
        _emit(out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


# ------------------------------------------------------------------------------------------------ the other BASELINE.json configurations
def _cfg_dist():
    import torch
    import torch.distributed as dist
    rank, local, world = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device -- the B200 arm has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return rank, local, world, barrier, max_over_ranks


def _cfg_reference_cpu(cfg, dims, budget_s=25.0):
    """The reference's own modules on the host cores for config 1 / 3 (network + its post-processing for the AABB anchor head; network only for
    the OBB FCOS head, whose Python NMS needs the reference's CUDA op)."""
    import argparse
    import torch
    from oracle import ref_gpu
    stub = os.path.join(ROOT, "tools", "ref_stub")
    sys.path.insert(0, stub)
    try:
        ref = ref_gpu.load(need_k1=False)
    finally:
        sys.path.remove(stub)
    torch.manual_seed(0)
    threads = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(threads)
    if cfg == 1:
        bb = ref.feature_extractor.VGG_FPN("EF", 4, True, 32)
        ag = ref.anchor.AnchorGenerator3D(ref_gpu.ANCHOR_SIZES, ref_gpu.ASPECT)
        m = ref.nerf_rpn.NeRFRegionProposalNetwork(bb, ag, ref.anchor.RPNHead(256, 13, 4), rpn_pre_nms_top_n_test=2500, rpn_post_nms_top_n_test=2500,
                                                   rpn_nms_thresh=0.3).eval()
        x = torch.rand(4, *dims)
        run = lambda: m([x.clone()])
        what, frac = "NeRFRegionProposalNetwork.forward of the UNMODIFIED reference (oracle/_ref), one 32^3 scene", 1.0
    else:
        bb = ref.feature_extractor.SwinTransformer_FPN(patch_size=[4, 4, 4], embed_dim=96, depths=[2, 2, 18, 2], num_heads=[3, 6, 12, 24],
                                                       window_size=[4, 4, 4], stochastic_depth_prob=0.0, expand_dim=True).eval()
        fa = argparse.Namespace(num_convs=4, norm_reg_targets=True, centerness_on_reg=True, rotated_bbox=True, pre_nms_thresh=0.0, pre_nms_top_n=2500,
                                nms_thresh=0.3, fpn_post_nms_top_n=2500, min_size=0.0)
        head = ref.fcos.FCOSHead(256, fa.num_convs, [4, 8, 16, 32], norm_reg_targets=True, centerness_on_reg=True, use_obb=True).eval()
        sub = (104, 104, 64)
        x = torch.rand(1, 4, *sub)
        run = lambda: head(list(bb(x)))
        frac = (sub[0] * sub[1] * sub[2]) / float(dims[0] * dims[1] * dims[2])
        what = (f"backbone + FPN + FCOS head of the UNMODIFIED reference (oracle/_ref) on a {sub[0]}x{sub[1]}x{sub[2]} block = {frac:.3f} scene "
                "(no post-processing: its Python OBB NMS needs the reference's CUDA op)")
    with torch.no_grad():
        run()
        times, t_all = [], time.perf_counter()
        while len(times) < 3 and time.perf_counter() - t_all < budget_s:
            t0 = time.perf_counter(); run(); times.append(time.perf_counter() - t0)
    sec = statistics.mean(times) / frac
    return {"value": 1.0 / sec, "unit": "scenes/s", "cores": threads, "kind": "reference", "sample": f"{what}; {len(times)} runs, {threads} threads"}


def run_config(args):
    """`--config 1|3|5`: the other BASELINE.json configurations with the same JSON contract (value device-resident, e2e through the public API with
    host buffers, roofline, cpu_baseline)."""
    import numpy as np
    import torch
    rank, local, world, barrier, max_over_ranks = _cfg_dist()
    from nerf_rpn_b200 import precision as nprec
    K, W = args.steps, max(args.warmup, 3)
    burst, sustained, how = measured_peaks()
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            hbm = float(json.load(f).get("hbm_gbs", 6570.0))
    except (OSError, ValueError):
        hbm = 6570.0
    sampler = ClockSampler(local)
    if args.config in (1, 3):
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_configs
        name = {1: "config1_vgg19_anchor_32", 3: "config3_swin_s_fcos_200x200x130"}[args.config]
        model, dims = bench_configs.build(name)
        model.precision = nprec.resolve(args.precision)
        model = model.cuda().eval()
        eng = model.engine()
        g = torch.Generator().manual_seed(1000 + rank)
        host = [torch.rand(*dims, 4, generator=g).pin_memory().permute(3, 0, 1, 2) for _ in range(3)]       # dataset views of (W,L,H,4) arrays
        xs = [h.cuda().contiguous()[None] for h in host]
        with torch.no_grad():
            for i in range(max(W, 4)):
                plan = eng.forward_device(xs[i % 3])
            barrier()
            if rank == 0:
                sampler.start()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(K):
                plan = eng.forward_device(xs[i % 3])
            torch.cuda.current_stream().wait_event(plan.done)
            b.record()
            barrier()
            clocks = sampler.stop() if rank == 0 else None
            ms = max_over_ranks(a.elapsed_time(b))
            for i in range(W):
                model([host[i % 3].cuda(non_blocking=True)])
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            d2h = 0
            for i in range(K):
                out = model([host[i % 3].cuda(non_blocking=True)])
                props = out[0][1][0] if args.config == 1 else out[0][0]
                d2h = props.cpu().numel() * 4
            b.record()
            barrier()
            ms_e2e = max_over_ranks(a.elapsed_time(b))
        flops = float(plan.algorithmic_flops)
        tf = flops * K / (ms * 1e-3) / 1e12
        out = None
        if rank == 0:
            try:
                cpu = _cfg_reference_cpu(args.config, dims)
            except Exception as e:                                        # noqa: BLE001
                cpu = {"value": None, "unit": "scenes/s", "cores": 0, "kind": "reference", "sample": "unavailable: " + repr(e)}
            out = {"metric": "scenes/sec", "value": world * K / (ms * 1e-3), "unit": "scenes/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
                   "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": nprec.bench_dtype(model.precision), "data": "synthetic",
                   "config": {"workload": {1: "BASELINE config 1: VGG19-3D + FPN + anchor head (AABB), one 32x32x32 RGBsigma grid",
                                           3: "BASELINE config 3: Swin-S 3D window attention + FPN + FCOS head (OBB), 200x200x130 RGBsigma grid"}[args.config],
                              "precision": model.precision, "scenes_per_step_per_gpu": 1, "parallelism": f"dp{world} (independent scenes per rank)",
                              "l2": "3 distinct input grids cycled" + ("; the 32^3 working set is L2-resident by nature of the configuration" if args.config == 1 else
                                                                       " (3 x 83 MB) and ~1 GB of activations per scene stream through the 126 MB L2"),
                              "proposals_last_scene": int(plan.out_count[0].item())},
                   "clocks": clocks,
                   "e2e": {"value": world * K / (ms_e2e * 1e-3), "unit": "scenes/s", "ms_per_step": ms_e2e / K, "h2d_bytes_per_step": int(host[0].numel() * 4),
                           "d2h_bytes_per_step": int(d2h), "api": type(model).__name__ + ".forward([grid]) with the grid copied from pinned host memory and the proposals read back"},
                   "gpu_launches": plan.num_launches() * K,
                   "roofline": {"bound": "tensor", "kernel": "whole step (all tcgen05 implicit-GEMM / attention launches of one scene)", "achieved": tf, "peak": sustained,
                                "unit": "TFLOP/s", "frac": tf / sustained, "traffic": None, "flops_per_step": flops,
                                "peak_source": how + ", sustained figure (kernels timed inside a long step)",
                                "note": "config 1 is launch-latency bound: 32^3 voxels keep a fraction of the 148 SMs busy" if args.config == 1 else
                                        "per-kernel rows in profiles/r01_ncu_per_kernel_config3.md"},
                   "cpu_baseline": cpu}
    else:
        # ---- config 5: oriented 3-D IoU + NMS, n = 1k .. 1M boxes of one scene (tools/nms_sweep.py distribution), threshold 0.3
        from nerf_rpn_b200 import ops
        from nerf_rpn_b200._lib import lib as _nlib

        def make(n, seed):
            g = torch.Generator().manual_seed(seed)
            c = torch.rand(n, 3, generator=g) * torch.tensor([256.0, 256.0, 160.0])
            s = torch.rand(n, 3, generator=g) * 44 + 4
            th = (torch.rand(n, 1, generator=g) - 0.5) * math.pi
            return torch.cat([c, s, th], 1).contiguous(), torch.rand(n, generator=g)
        sweep = []
        top = None
        for mode, n in [(0, v) for v in (1000, 4000, 16000, 64000, 256000)] + [(3, 64000), (3, 256000), (3, 1000000), (0, 1000000)]:   # headline last
            ops.set_nms_cull_mode(mode)
            sets = [make(n, 10 * rank + k) for k in range(2)]                     # 2 x 32 MB at 1 M; the sort / grid scratch is ~0.5 GB: not L2-resident
            dev = [(b.cuda(), s.cuda()) for b, s in sets]
            pin = [(b.pin_memory(), s.pin_memory()) for b, s in sets]
            reps = K                                                              # --steps timed repetitions at every size
            for i in range(W):
                keep, nk = ops.nms_device(dev[i % 2][0], dev[i % 2][1], None, 0.3)
            barrier()
            if rank == 0 and n == 1000000 and mode == 0:
                sampler.start()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            lc0 = int(_nlib().nrpn_launch_count())
            a.record()
            for i in range(reps):
                keep, nk = ops.nms_device(dev[i % 2][0], dev[i % 2][1], None, 0.3)
            b.record()
            barrier()
            launches = int(_nlib().nrpn_launch_count()) - lc0
            if rank == 0 and n == 1000000 and mode == 0:
                clocks = sampler.stop()
            ms = max_over_ranks(a.elapsed_time(b)) / reps
            kept = int(nk.item())
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(reps):
                bx, sc = pin[i % 2][0].cuda(non_blocking=True), pin[i % 2][1].cuda(non_blocking=True)
                keep, nk = ops.nms_device(bx, sc, None, 0.3)
                host_keep = keep[: int(nk.item())].cpu()
            b.record()
            barrier()
            ms_e2e = max_over_ranks(a.elapsed_time(b)) / reps
            row = {"cull_mode": mode, "n": n, "kept": kept, "ms": ms, "boxes_per_s": world * n / (ms * 1e-3), "gb_per_s": (32.0 * n + 8.0 * kept) / (ms * 1e-3) / 1e9,
                   "e2e_ms": ms_e2e, "e2e_boxes_per_s": world * n / (ms_e2e * 1e-3), "reps": reps}
            sweep.append(row)
            top = row
            del dev, pin, sets
            torch.cuda.empty_cache()
        out = None
        if rank == 0:
            from oracle import box as obox
            nb = 12000
            bb, ss = make(nb, 0)
            t0 = time.perf_counter()
            obox.nms(bb.numpy(), ss.numpy(), 0.3)
            cpu_s = time.perf_counter() - t0
            out = {"metric": "boxes/sec (oriented 3-D IoU + greedy NMS, 1M proposals of one scene)", "value": top["boxes_per_s"], "unit": "boxes/s", "n_gpus": world,
                   "steps": top["reps"], "warmup": W, "ms_per_step": top["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                   "data": "synthetic",
                   "config": {"workload": "BASELINE config 5: rotated 3-D OBB IoU + NMS sweep, 1k .. 1M proposals per scene (centres U[0,256)^2 x [0,160), sizes U[4,48], "
                                          "theta U[-pi/2,pi/2), scores U[0,1), threshold 0.3, one group); headline = the 1M point in cull mode 0 (exact-zero culls only: the keep set is "
                                          "provably the reference's); cull_mode 3 rows = opt-in geometric ratio culls (include/nerf_rpn_b200.h)", "sweep": sweep,
                              "parallelism": f"dp{world} (independent scenes per rank)", "l2": "two input sets alternate; ~0.5 GB of sort / cell-list scratch per call"},
                   "clocks": clocks,
                   "e2e": {"value": top["e2e_boxes_per_s"], "unit": "boxes/s", "ms_per_step": top["e2e_ms"], "h2d_bytes_per_step": 32 * top["n"],
                           "d2h_bytes_per_step": 8 * top["kept"] + 4, "api": "nerf_rpn_b200.ops.nms_device (the kernel behind model.utils.nms / batched_nms) with pinned host boxes in, kept indices out"},
                   "gpu_launches": None,
                   "roofline": {"bound": "hbm", "kernel": "whole NMS call (sort, cell lists, cross / adjacency passes, rounds, compaction)",
                                "achieved": top["gb_per_s"], "peak": hbm, "unit": "GB/s", "frac": top["gb_per_s"] / hbm, "traffic": None,
                                "algorithmic_bytes": "32 B per input box + 8 B per kept index (SURVEY 8d)",
                                "note": "greedy NMS is bound by the pair tests (cull arithmetic + polygon clips) and their dependency chain, not by HBM: the fraction is "
                                        "reported because the contract asks for it; the per-kernel split is in profiles/"},
                   "cpu_baseline": {"value": nb / cpu_s, "unit": "boxes/s", "cores": 1, "kind": "port",
                                    "sample": f"oracle/box.py nms (C restatement of utils.py:215-265 + cal_iou_3d) on {nb} boxes of the same distribution: {cpu_s:.1f} s; "
                                              "the cost grows ~ n x kept, so boxes/s at 1M would be far lower"}}
            out["gpu_launches"] = launches                                       # launch checks inside the timed region of the 1M point
    if rank == 0:
        _emit(out)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return out


def _train_reference_cpu(budget_s=40.0):
    """The reference's own training step (model.train(): forward with targets, loss.backward()) on the host cores, on a 40x64x64 block (1/64 of a
    scene) with 4 planted boxes -- a full scene's fp32 autograd graph needs ~100 GB."""
    import torch
    from oracle import ref_gpu
    stub = os.path.join(ROOT, "tools", "ref_stub")
    sys.path.insert(0, stub)
    try:
        ref_gpu.load(need_k1=False)
    finally:
        sys.path.remove(stub)
    threads = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(threads)
    m = ref_gpu.build_reference_model(rotated=True, seed=0).train()
    sub = (40, 64, 64)
    g = torch.Generator().manual_seed(3)
    x = torch.rand(4, *sub, generator=g)
    ctr = torch.rand(4, 3, generator=g) * torch.tensor(sub, dtype=torch.float32) * 0.6 + torch.tensor(sub, dtype=torch.float32) * 0.2
    gt = torch.cat([ctr, torch.rand(4, 3, generator=g) * 10 + 6, (torch.rand(4, 1, generator=g) - 0.5) * math.pi], 1)

    def step():
        m.zero_grad(set_to_none=True)
        _, losses, _ = m([x.clone()], [gt.clone()])
        (losses["loss_objectness"] + 5.0 * losses["loss_rpn_box_reg"]).backward()
    step()
    times, t_all = [], time.perf_counter()
    while len(times) < 3 and time.perf_counter() - t_all < budget_s:
        t0 = time.perf_counter(); step(); times.append(time.perf_counter() - t0)
    frac = (sub[0] * sub[1] * sub[2]) / float(DIMS[0] * DIMS[1] * DIMS[2])
    sec = statistics.mean(times) / frac
    return {"value": 1.0 / sec, "unit": "scenes/s", "cores": threads, "kind": "reference",
            "sample": f"forward + loss + backward of the UNMODIFIED reference (oracle/_ref, fp32 autograd) on a {sub[0]}x{sub[1]}x{sub[2]} block = 1/64 scene, "
                      f"scaled by voxels; {len(times)} runs, {threads} threads; no optimiser step"}


def run_train(args):
    """`--mode train`: BASELINE config 4 (ResNet50-FPN + anchor head --rotated_bbox, one 160x256x256 scene per rank and step, data parallel with ONE NCCL
    all-reduce of the flat gradient bucket overlapped with the backward pass) as the headline value."""
    import torch
    import torch.distributed as dist
    rank, local, world, barrier, max_over_ranks = _cfg_dist()
    K, W = args.steps, max(args.warmup, 4)             # two eager steps, the graph capture, one replay
    burst, sustained, how = measured_peaks()
    model = build_model(rotated=True, spread=0.0).cuda().train()
    eng = model.train_engine(precision="bf16", lr=1e-4, weight_decay=0.01, clip_grad_norm=0.1, reg_loss_weight=5.0,
                             process_group=dist.group.WORLD if world > 1 else None)
    host = [synth_scene(rank * 1000 + i, "dataset").permute(1, 2, 3, 0).contiguous().pin_memory().permute(3, 0, 1, 2) for i in range(2)]
    grids = [h.cuda()[None] for h in host]
    gts = [[planted_boxes(rank * 1000 + i).cuda()] for i in range(2)]
    gts_host = [planted_boxes(rank * 1000 + i).pin_memory() for i in range(2)]
    for i in range(W):
        eng.train_step(grids[i % 2], gts[i % 2])
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        losses = eng.train_step(grids[i % 2], gts[i % 2])
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = max_over_ranks(e0.elapsed_time(e1))
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for i in range(K):
        x = host[i % 2].cuda(non_blocking=True)[None]
        t = [gts_host[i % 2].cuda(non_blocking=True)]
        host_losses = eng.train_step(x, t).cpu()
    e3.record()
    barrier()
    ms_e2e = max_over_ranks(e2.elapsed_time(e3))
    plan = eng.plan(1, DIMS)
    out = None
    if rank == 0:
        try:
            if args.skip_cpu_baseline or world > 1:
                cpu = {"value": None, "unit": "scenes/s", "cores": 0, "kind": "reference", "sample": "not timed (N > 1 or --skip-cpu-baseline)"}
            else:       # in a child process without a visible GPU: the reference's OBB code hard-codes `.cuda()` (utils.py:412) and would mix devices
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-train-baseline"], capture_output=True, text=True, timeout=600,
                                   env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
                if r.returncode != 0:
                    raise RuntimeError(r.stderr[-300:])
                cpu = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:                                        # noqa: BLE001
            cpu = {"value": None, "unit": "scenes/s", "cores": 0, "kind": "reference", "sample": "unavailable: " + repr(e)}
        tf = 3.0 * FLOPS_PER_SCENE * K / (ms * 1e-3) / 1e12          # forward + data gradient + weight gradient
        out = {"metric": "training scenes/sec", "value": world * K / (ms * 1e-3), "unit": "scenes/s", "n_gpus": world, "steps": K, "warmup": W,
               "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "bf16 (activations / gradients; fp32 master weights, accumulation, optimiser state)", "data": "synthetic",
               "config": {"workload": "BASELINE config 4: ResNet50-3D+FPN+anchor head --rotated_bbox, one 160x256x256x4 scene per rank per step, 16 planted OBBs, "
                                      "256 sampled anchors, BCE + smooth-L1 (x5), clip_grad_norm 0.1, AdamW lr 1e-4 wd 0.01",
                          "scenes_per_step_per_gpu": 1, "parallelism": f"dp{world}",
                          "collective": (f"one NCCL all-reduce (sum) of the flat fp32 gradient bucket per step: {eng.n_params} parameters = {eng.n_params * 4 / 1e6:.0f} MB, "
                                         f"in {getattr(plan, 'allreduce_calls', 0)} ranges launched on a communication stream as the backward pass finalises them")
                                        if world > 1 else "none at N = 1 (the all-reduce is skipped)",
                          "l2": "two 168 MB input grids alternate; ~6 GB of activations / gradients stream per step",
                          "losses_last_step": [round(v, 5) for v in losses.tolist()]},
               "clocks": clocks,
               "e2e": {"value": world * K / (ms_e2e * 1e-3), "unit": "scenes/s", "ms_per_step": ms_e2e / K,
                       "h2d_bytes_per_step": int(host[0].numel() * 4 + gts_host[0].numel() * 4), "d2h_bytes_per_step": int(host_losses.numel() * 4),
                       "api": "RPNTrainEngine.train_step (model.train_engine()): pinned host grid + boxes in, the two losses read back every step"},
               "gpu_launches": None,
               "roofline": {"bound": "tensor", "kernel": "whole training step (forward + dgrad + wgrad = 3 x the forward's convolution FLOPs)", "achieved": tf,
                            "peak": sustained, "unit": "TFLOP/s", "frac": tf / sustained, "traffic": None, "flops_per_step": 3.0 * FLOPS_PER_SCENE,
                            "peak_source": how + ", sustained figure", "note": "per-kernel split: profiles/r02_train_step_kernels.md"},
               "cpu_baseline": cpu}
        _emit(out)
    del eng, model
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


_RESULT_FD = None


def _emit(obj):
    """The one JSON line, on the process's ORIGINAL stdout."""
    line = json.dumps(obj) + "\n"
    if _RESULT_FD is None:
        sys.stdout.write(line)
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, line.encode())


def main():
    global _RESULT_FD
    # stdout carries the JSON line and nothing else: native libraries write banners to fd 1 (NCCL prints its version there when NCCL_DEBUG is
    # set), so fd 1 is pointed at stderr for the run and the result goes to a private duplicate of the original.
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    if args.cpu_train_baseline:
        _emit(_train_reference_cpu())
    elif args.impl == "reference":
        run_reference(args)
    elif args.mode == "train":
        run_train(args)
    elif args.config != 2:
        run_config(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
