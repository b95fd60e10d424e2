#!/usr/bin/env python
"""bench.py — images/sec of the Uformer-B 256x256 forward (BASELINE.json configs[1]) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--mode fwd|train] [--dump-outputs DIR]

`--mode train` (not the default; BASELINE configs[2]) times the data-parallel training step instead: batch 8 per GPU,
native forward + recompute backward + NCCL bucketed gradient all-reduce + native AdamW (uformer_b200.training).

A "step" is one forward of a batch of 32 synthetic 256x256x3 images through the native engine
(bf16 activations, fp32 accumulate).  Weights: Uformer-B architecture, seeded synthetic init
(tests/paramgen.py).  N>1 (torchrun): independent replicas, one per GPU, no data-path collective
(inference shards by image); value = images of all ranks / max-over-ranks device time.

Timing: per-step CUDA events on the launching stream; an L2 flush (256 MB memset) runs between
timed steps outside the event brackets; W>=3 warm-up steps.  `e2e` repeats the measurement through
the public API with pinned HOST input, H2D copy and D2H of the restored image inside the timed region.
`roofline` is the dominant kernel class (largest share of step time), timed live with CUDA events
in an extra instrumented step.  `cpu_baseline` / `--impl reference` time the CPU oracle port of the
reference forward (oracle/lewin_oracle.py; the reference itself is Python and cannot travel to the
GPU box) on the host cores, on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step of rank 0 computed as DIR/<name>.npy (float32): the restored images
(`restored`, fwd) or the loss (`loss`, train).  Inputs and weights are seeded, so two builds run with the same arguments can be
compared output for output.  An output over the 64 MB budget is replaced by a fixed, seeded sample of its elements.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

UFORMER_B = dict(img_size=256, embed_dim=32, win_size=8, token_projection="linear", token_mlp="leff",
                 depths=[1, 2, 8, 8, 2, 8, 8, 2, 1], modulator=True, dd_in=3)       # utils/model_utils.py:76-78
GFLOP_PER_IMG = 173.1          # BASELINE.md §2 (2 x 86.57 GMAC)
DUMP_BYTES = 64 << 20          # --dump-outputs budget over all arrays


def note(msg):
    """progress line on stderr (stdout carries only the JSON line)"""
    print(f"[bench {time.strftime('%X')}] {msg}", file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons, samples=len(sm))


def dump_outputs(outdir, arrays):
    """Each tensor of `arrays` -> outdir/<name>.npy as float32; one larger than its share of DUMP_BYTES becomes the same
    seeded random sample of its elements (sorted flat indices) on every run."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    cap = DUMP_BYTES // 4 // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() > cap:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(outdir, name + ".npy"), a.numpy())
    note(f"outputs of the last timed step written to {outdir}: {', '.join(arrays)}")


def build_engine(device, seed=1234):
    import uformer_b200
    from paramgen import randomize_state
    net = uformer_b200.Uformer(**UFORMER_B)
    net.load_state_dict(randomize_state(net.state_dict(), seed), strict=True)
    return net.to(device).eval()


def _cpu_forward_fn(n_images):
    """Closure running the CPU oracle port (library-op formulation, fp32) of the Uformer-B forward."""
    from oracle import lewin_oracle as O
    from paramgen import randomize_state
    import uformer_b200
    O.FAST = True
    st = randomize_state(uformer_b200.Uformer(**UFORMER_B).state_dict(), 1234)
    torch.manual_seed(1234)
    x = torch.rand(n_images, 3, 256, 256)

    def fwd():
        with torch.no_grad():
            return O.uformer_forward(x, st, 256, 32, UFORMER_B["depths"])
    return fwd


def _pick_threads(fwd):
    """torch's CPU ops do not scale to 128 threads on these shapes; pick the best of a few counts
    (one forward each) so the baseline uses the host as well as it can."""
    best, best_t = None, None
    ncpu = os.cpu_count() or 8
    for th in sorted({min(ncpu, c) for c in (16, 32, 64)}):
        torch.set_num_threads(th)
        fwd()
        t0 = time.perf_counter()
        fwd()
        dt = time.perf_counter() - t0
        note(f"cpu port: {th} threads -> {dt:.2f}s per forward")
        if best is None or dt < best:
            best, best_t = dt, th
    torch.set_num_threads(best_t)
    return best_t


def cpu_oracle_rate(n_images, iters=2):
    """images/sec of the CPU oracle port on `n_images` 256x256 images (bounded sample)."""
    fwd = _cpu_forward_fn(n_images)
    threads = _pick_threads(fwd)
    t0 = time.perf_counter()
    for _ in range(iters):
        fwd()
    dt = (time.perf_counter() - t0) / iters
    return n_images / dt, threads, dt


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    nimg = 4                         # bounded sample of the batch-32 step
    fwd = _cpu_forward_fn(nimg)
    threads = _pick_threads(fwd)     # doubles as warm-up
    steps, warm = args.steps, 1
    t0 = time.perf_counter()
    for _ in range(steps):
        fwd()
    dt = (time.perf_counter() - t0) / steps
    v = nimg / dt
    sample = (f"{nimg} images of the batch-32 step per timed step (fp32 oracle port of model.py's forward, torch CPU ops, "
              f"{threads} of {os.cpu_count()} host threads = best of 16/32/64)")
    # same metric / unit / config as the GPU arm (the workload is the batch-32 step; each timed step runs a bounded sample of it)
    print(json.dumps({
        "impl": "reference", "metric": "images/sec Uformer-B 256x256 fwd", "value": v, "unit": "img/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic",
        "config": {"workload": "Uformer-B 256x256 inference fwd, batch 32 per GPU (BASELINE configs[1])", "global_batch": 32 * max(1, args.gpus),
                   "per_gpu_batch": 32, "sample_images_per_step": nimg, "implementation": "CPU port of the reference forward (oracle/)"},
        "cpu_baseline": {"value": v, "unit": "img/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


TRAIN_GFLOP_PER_IMG = 3 * GFLOP_PER_IMG      # fwd + bwd (2x fwd); the recompute in backward is overhead, not counted


def run_reference_train(args, rank):
    """CPU arm of --mode train: fwd + bwd + AdamW of the oracle port (torch autograd over its library-op formulation)."""
    if rank != 0:
        return
    from oracle import lewin_oracle as O
    from paramgen import randomize_state
    import uformer_b200
    O.FAST = True
    st = randomize_state(uformer_b200.Uformer(**UFORMER_B).state_dict(), 1234)
    params = {k: v.clone().requires_grad_(True) for k, v in st.items() if torch.is_floating_point(v)}
    full = dict(st)
    full.update(params)
    opt = torch.optim.AdamW(list(params.values()), lr=2e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.02)
    nimg = 1
    torch.manual_seed(1234)
    clean = torch.rand(nimg, 3, 256, 256)
    noisy = (clean + 0.1 * torch.randn_like(clean)).clamp(0, 1)
    threads = min(os.cpu_count() or 8, 32)
    torch.set_num_threads(threads)

    def step():
        opt.zero_grad()
        out = O.uformer_forward(noisy, full, 256, 32, UFORMER_B["depths"])
        torch.sqrt((out - clean) ** 2 + 1e-6).mean().backward()
        opt.step()
    step()
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    v = nimg / dt
    sample = f"{nimg} image of the batch-8 step per timed step (fp32 oracle port + torch autograd + torch AdamW, {threads} host threads)"
    print(json.dumps({
        "impl": "reference", "metric": "images/sec Uformer-B 256x256 train step", "value": v, "unit": "img/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": 1, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic",
        "config": {"workload": "Uformer-B 256x256 training step (BASELINE configs[2]), CPU port of the reference", "global_batch": nimg},
        "cpu_baseline": {"value": v, "unit": "img/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


def run_train(args, rank, world, local):
    """BASELINE configs[2]: Uformer-B 256x256 training step, bf16, batch 8 per GPU, gradient all-reduce over NCCL."""
    import torch.distributed as dist
    import uformer_b200
    from uformer_b200 import ops
    from uformer_b200.training import TrainStep
    from paramgen import randomize_state
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warm = max(args.warmup, 3)
    B = args.batch or 8
    net = uformer_b200.Uformer(**UFORMER_B, drop_path_rate=0.1)                  # the reference's default (model.py:1075)
    net.load_state_dict(randomize_state(net.state_dict(), 1234), strict=True)    # same weights on every rank
    net = net.to(dev)
    step = TrainStep(net, lr=2e-4, weight_decay=0.02)
    torch.manual_seed(1234 + rank)                                               # every rank draws its own shard
    clean_h = torch.rand(B, 3, 256, 256).pin_memory()
    noisy_h = (clean_h + 0.1 * torch.randn_like(clean_h)).clamp(0, 1).pin_memory()
    clean_d, noisy_d = clean_h.to(dev), noisy_h.to(dev)
    loss_h = torch.zeros(1).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """(total device ms over `steps` steps, max over ranks; what the last step returned)"""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for s, e in evs:
            flush.zero_()
            s.record()
            out = fn()
            e.record()
        barrier()
        t = torch.tensor([sum(s.elapsed_time(e) for s, e in evs)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), out

    def step_dev():
        return step(noisy_d, clean_d)

    def step_e2e():
        x = noisy_h.to(dev, non_blocking=True)
        t = clean_h.to(dev, non_blocking=True)
        loss_h.copy_(step(x, t).view(1), non_blocking=True)

    note("train: engine + arena built; warm-up")
    for _ in range(warm):
        step_dev()
    torch.cuda.synchronize()
    ops.LAUNCH_COUNT = 0
    step_dev()
    launches_per_step = ops.LAUNCH_COUNT                      # forward kernels + charbonnier + adamw (all go through ops)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms, loss = timed(step_dev, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss})
    e2e_ms, _ = timed(step_e2e, args.steps)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    value = world * B * args.steps / (total_ms / 1e3)
    e2e_val = world * B * args.steps / (e2e_ms / 1e3)
    ach = TRAIN_GFLOP_PER_IMG * value / world / 1e3
    print(json.dumps({
        "metric": "images/sec Uformer-B 256x256 train step", "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "Uformer-B 256x256 training step: fwd + bwd + AdamW, Charbonnier loss, batch 8 per GPU (BASELINE configs[2])",
                   "global_batch": B * world, "per_gpu_batch": B, "parallelism": f"dp{world} (NCCL bucketed gradient all-reduce, overlapped)",
                   "l2": "256MB flush between timed steps", "drop_path_rate": 0.1,
                   "backward": "recompute-from-block-input; restated torch statements under bf16 autocast (cuBLAS/ATen), not yet native"},
        "e2e": {"value": e2e_val, "unit": "img/s", "h2d_bytes_per_step": 2 * clean_h.numel() * 4, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches_per_step * args.steps, "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "whole training step", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                     "frac": ach / peaks["tf_sustained"], "peak_source": peaks["src"] + " sustained", "traffic": None,
                     "flops_per_image": TRAIN_GFLOP_PER_IMG * 1e9}}))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--batch", type=int, default=None, help="images per GPU per step (default: 32 for fwd, 8 for train)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mode", default="fwd", choices=["fwd", "train"])
    ap.add_argument("--size", type=int, default=256, choices=[256, 512],
                    help="image side: 256 (BASELINE configs[1], the headline) or 512 (configs[3]: the model built for 256 run on "
                         "512x512 images in one whole-image forward, default batch 8)")
    ap.add_argument("--residual", default=None, choices=["auto", "fp32", "bf16"],
                    help="residual-stream precision between the kernels of a stage (default: the engine's default, fp32)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy, float32, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the native engine's outputs (--impl ours)")
    if args.residual:
        os.environ["UFORMER_B200_RESIDUAL"] = args.residual
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))

    lib = os.path.join(ROOT, "uformer_b200", "lib", "liblewin_b200.so")
    if args.impl != "reference" and not os.path.isfile(lib):
        if local == 0:                       # the .so is git-ignored: build it in-tree if this checkout lacks it
            note("native library missing; building it (nvcc, ~30 s)")
            import __graft_entry__
            __graft_entry__.build()
        else:
            while not os.path.isfile(lib):
                time.sleep(1.0)
            time.sleep(2.0)
    if args.impl == "reference":
        if args.mode == "train":
            run_reference_train(args, rank)
        else:
            run_reference_arm(args, rank, world)
        return
    if args.mode == "train":
        run_train(args, rank, world, local)
        return

    import torch.distributed as dist
    from uformer_b200 import ops
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warm = max(args.warmup, 3)
    S = args.size
    B = args.batch or (32 if S == 256 else 8)
    net = build_engine(dev)
    torch.manual_seed(1234 + rank)
    x_host = torch.rand(B, 3, S, S).pin_memory()
    x_dev = x_host.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """(total device ms over `steps` steps, max over ranks; what the last step returned)"""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for s, e in evs:
            flush.zero_()                    # L2 flush, outside the event bracket
            s.record()
            out = fn()
            e.record()
        barrier()
        ms = sum(s.elapsed_time(e) for s, e in evs)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), out

    # device-resident leg: the forward captured once into a CUDA graph (uformer_b200.GraphedForward) and replayed;
    # falls back to eager launches if capture is unavailable
    graphed = None
    try:
        import uformer_b200
        graphed = uformer_b200.GraphedForward(net, x_dev)
    except Exception as exc:                                   # pragma: no cover
        note(f"CUDA graph capture unavailable ({exc}); timing eager launches")

    def step_dev():
        return graphed(graphed.x) if graphed is not None else net(x_dev)

    # ---- e2e: the same forward through the public API with HOST buffers.  Every step copies its input from pinned
    # host memory and its restored image back to pinned host memory inside the timed region; copies run on two copy
    # streams so step i+1's upload and step i-1's download overlap step i's compute (double-buffered).
    main_s = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    xd = [torch.empty_like(x_dev) for _ in range(2)]
    yh = [torch.empty(B, 3, S, S).pin_memory() for _ in range(2)]
    ev_h2d = [torch.cuda.Event() for _ in range(2)]
    ev_comp = [torch.cuda.Event() for _ in range(2)]
    ev_d2h = [torch.cuda.Event() for _ in range(2)]

    def run_e2e(steps):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(main_s)
        for i in range(steps):
            b = i & 1
            with torch.cuda.stream(s_in):
                if i >= 2:
                    s_in.wait_event(ev_comp[b])              # xd[b] is free once step i-2 finished computing
                else:
                    s_in.wait_event(t0)
                xd[b].copy_(x_host, non_blocking=True)
                ev_h2d[b].record(s_in)
            main_s.wait_event(ev_h2d[b])
            y = net(xd[b])
            ev_comp[b].record(main_s)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_comp[b])
                if i >= 2:
                    s_out.wait_event(ev_d2h[b])
                yh[b].copy_(y, non_blocking=True)
                y.record_stream(s_out)
                ev_d2h[b].record(s_out)
        for b in range(min(2, steps)):
            main_s.wait_event(ev_d2h[b])
        t1.record(main_s)
        barrier()
        t = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    note("engine built; warm-up")
    for _ in range(warm):
        step_dev()
    torch.cuda.synchronize()
    note("timing device-resident steps")
    ops.LAUNCH_COUNT = 0
    with torch.no_grad():
        net(x_dev)                                              # one eager forward: counts the native launches of a step
    launches_per_step = ops.LAUNCH_COUNT
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms, restored = timed(step_dev, args.steps)
    launches = launches_per_step * args.steps                  # the graph replays exactly these launches every step
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"restored": restored})   # before later forwards can reuse any buffer
    note(f"device-resident: {total_ms / args.steps:.2f} ms/step; timing e2e (host buffers)")
    run_e2e(2)
    e2e_ms = run_e2e(args.steps)

    # ---- instrumented step: per-kernel-class device time (CUDA events around every launch) ----
    prof = None
    if rank == 0:
        ops.PROFILE = []
        with torch.no_grad():
            net(x_dev)
        torch.cuda.synchronize()
        rec, ops.PROFILE = ops.PROFILE, None
        agg = {}
        for label, flops, s, e in rec:
            a = agg.setdefault(label, [0.0, 0, 0.0])
            a[0] += s.elapsed_time(e); a[1] += 1; a[2] += flops
        prof = agg

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    gflop_img = GFLOP_PER_IMG * (S / 256) ** 2            # every op of the forward is linear in the pixel count
    ms_step = total_ms / args.steps
    value = world * B * args.steps / (total_ms / 1e3)
    e2e_val = world * B * args.steps / (e2e_ms / 1e3)
    # dominant kernel class by device time
    tot_prof = sum(v[0] for v in prof.values())
    dom = max(prof.items(), key=lambda kv: kv[1][0])
    dname, (dms, dcount, dflops) = dom
    ach = dflops / dcount / (dms / dcount * 1e-3) / 1e12
    # DRAM traffic of the dominant kernel: from the committed ncu table (tools/kernel_metrics.py), only while it describes THESE
    # kernel sources (sha256 of csrc/ + the header recorded next to the numbers); otherwise null rather than a stale figure
    traffic, traffic_src, tensor_pct = None, None, None
    tpath = os.path.join(ROOT, "profiles", "r02_kernel_metrics.json")
    if os.path.isfile(tpath):
        from uformer_b200 import _lib as _ulib
        tj = json.load(open(tpath))
        if tj.get("csrc_sha256_16") == _ulib.csrc_hash() and dname in tj["dram_bytes_per_launch"]:
            traffic, traffic_src = tj["dram_bytes_per_launch"][dname], "profiles/r02_kernel_metrics.json (ncu, same kernel sources)"
            tensor_pct = tj.get("tensor_pipe_pct", {}).get(dname)
        else:
            traffic_src = "profiles/r02_kernel_metrics.json is for other kernel sources: dropped"
    roofline = {"bound": "tensor", "kernel": dname, "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                "frac": ach / peaks["tf_sustained"], "peak_source": peaks["src"] + " sustained (kernel timed inside a long step)",
                "traffic": traffic, "traffic_source": traffic_src, "tensor_pipe_pct_ncu": tensor_pct, "share_of_step": dms / tot_prof, "launches_per_step": dcount,
                "avg_launch_ms": dms / dcount,
                "model": {"achieved": gflop_img * value / world / 1e3, "unit": "TFLOP/s",
                          "frac": gflop_img * value / world / 1e3 / peaks["tf_sustained"]},
                "by_kernel_ms": {k: round(v[0], 3) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}}
    line = {
        "metric": f"images/sec Uformer-B {S}x{S} fwd", "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": (f"Uformer-B 256x256 inference fwd, batch {B} per GPU (BASELINE configs[1])" if S == 256 else
                                f"Uformer-B (built for 256x256) on {S}x{S} images, one whole-image forward each, batch {B} per GPU (BASELINE configs[3])"),
                   "global_batch": B * world,
                   "per_gpu_batch": B, "parallelism": f"replicas x{world} (no collective)", "l2": "256MB flush between timed steps",
                   "weights": "synthetic seeded init of the Uformer-B architecture",
                   "cuda_graph": graphed is not None,
                   "residual_stream": os.environ.get("UFORMER_B200_RESIDUAL", "auto") + " (fp32 between the kernels of the >=4-block stages, bf16 elsewhere; bf16 operands, fp32 accumulate)"},
        "e2e": {"value": e2e_val, "unit": "img/s", "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": yh[0].numel() * 4, "pipelined": "2 copy streams, double-buffered",
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline}
    if not args.no_cpu_baseline and world == 1 and S == 256:
        note("cpu baseline (oracle port on host cores)")
        v, threads, dt = cpu_oracle_rate(4, iters=2)
        line["cpu_baseline"] = {"value": v, "unit": "img/s", "cores": threads, "kind": "port",
                                "sample": f"4 images x 2 iterations of the same forward (fp32 oracle port, {dt:.2f}s per iteration, "
                                          f"best of 16/32/64 threads on {os.cpu_count()} cpus)"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
