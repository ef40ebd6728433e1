#!/usr/bin/env python
"""Benchmark of the allRank hot path on B200: slates/sec of a full training step
(scorer forward + listwise loss + backward + Adam) on synthetic MSLR-WEB30K-shaped slates.

    python bench.py --gpus 1 --steps 20 --warmup 5                  # this repo's CUDA path
    python bench.py --impl reference --steps 5 --warmup 3           # the reference's eager CPU path (oracle port)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line (rank 0).  Contract: see the task statement; fields are documented in DESIGN.md section 6.
Workloads (BASELINE.json configs):
    cfg2  Transformer(N=2,h=4,d=128,d_ff=512) + approxNDCGLoss, S=240, F=136      <- the metric's configuration
    cfg3  Transformer(N=4,h=8,d=256,d_ff=1024) + lambdaLoss(ndcgLoss2PP), S=240
    cfg4  Transformer(N=2,h=4,d=128,d_ff=512) + neuralNDCG, S=120
    cfg5  Transformer(N=4,h=8,d=256,d_ff=1024) + listMLE, S=240
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg2": dict(N=2, h=4, d=128, dff=512, S=240, loss="approxNDCGLoss", loss_args={"alpha": 1.0}),
    "cfg3": dict(N=4, h=8, d=256, dff=1024, S=240, loss="lambdaLoss",
                 loss_args={"weighing_scheme": "ndcgLoss2PP_scheme", "k": None, "mu": 10.0, "sigma": 1.0}),
    "cfg4": dict(N=2, h=4, d=128, dff=512, S=120, loss="neuralNDCG",
                 loss_args={"temperature": 1.0, "k": None, "powered_relevancies": True}),
    "cfg5": dict(N=4, h=8, d=256, dff=1024, S=240, loss="listMLE", loss_args={}),
}
F = 136
PAD = -1


def flops_per_slate_step(w):
    """Algorithmic FLOPs of one training step per slate (SURVEY.md 8d): 3 x forward."""
    S, d, dff, N = w["S"], w["d"], w["dff"], w["N"]
    fwd = 2 * S * F * d + N * (8 * S * d * d + 4 * S * S * d + 4 * S * d * dff) + 2 * S * d
    return 3 * fwd


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"],
                    bf16_tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx = max(mx, float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return None
        busy = [v for v in sm if v > 0.5 * mx] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------ CPU arm
def reference_available():
    return os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "allrank", "main.py"))


def cpu_reference_steps(w, batch, steps, warmup, threads):
    """The reference's own eager PyTorch path on the host cores, one step = train_utils.loss_batch
    (allrank/training/train_utils.py:18-29: forward, loss, backward, Adam step, loss.item()).
    kind "reference": the UNMODIFIED package installed in baseline/_ref (oracle/install_reference.py) -- its make_model,
    its loss function, its loss_batch; kind "port": the oracle restatement (only when baseline/_ref is absent).
    Must run in a process where CUDA is hidden: the reference hard-wires cuda:0 whenever a GPU is visible
    (allrank/models/model_utils.py:13-18)."""
    from allrank_b200.synth import make_slates
    torch.manual_seed(42)
    x, y, idx = make_slates(batch, w["S"], F, seed=1234)
    if reference_available():
        from oracle.install_reference import import_path
        sys.path[:0] = import_path()
        import allrank.models.losses as ref_losses
        from allrank.config import TransformerConfig
        from allrank.models.model import make_model as ref_make_model
        from allrank.training.train_utils import loss_batch
        from functools import partial
        model = ref_make_model(fc_model={"sizes": [w["d"]], "input_norm": False, "activation": None, "dropout": 0.0},
                               transformer=TransformerConfig(N=w["N"], d_ff=w["dff"], h=w["h"],
                                                             positional_encoding=None, dropout=0.0),
                               post_model={"d_output": 1, "output_activation": None}, n_features=F).train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        loss_fn = partial(getattr(ref_losses, w["loss"]), **w["loss_args"])
        kind = "reference"

        def one_step():
            t0 = time.perf_counter()
            loss_batch(model, loss_fn, x, y, idx, None, opt)
            return time.perf_counter() - t0
    else:
        from oracle import losses_ref
        from oracle.scorer_ref import make_ref_model
        model = make_ref_model(F, [w["d"]], w["N"], w["h"], w["dff"]).train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        loss_fn = losses_ref.LOSSES[w["loss"]]
        kind = "port"

        def one_step():
            t0 = time.perf_counter()
            loss = loss_fn(model(x, y == PAD, idx), y, **w["loss_args"])
            loss.backward()
            opt.step()
            opt.zero_grad()
            _ = loss.item()
            return time.perf_counter() - t0

    # "all the host threads it can use": intra-op thread counts above the box's real core budget make eager
    # PyTorch slower, so pick the fastest of a few candidates (one untimed + one timed step each) -- the
    # baseline reported is the best the host achieves.
    best, best_t = threads, None
    for cand in sorted({c for c in (8, 16, 32, 64, threads) if c <= threads}):
        torch.set_num_threads(cand)
        one_step()
        t = one_step()
        if best_t is None or t < best_t:
            best, best_t = cand, t
    torch.set_num_threads(best)
    times = [one_step() for _ in range(warmup + steps)][warmup:]
    total = sum(times)
    return batch * steps / total, 1e3 * total / steps, best, kind


def run_reference(args, w):
    rank, _, world = dist_env()
    if rank != 0:
        return
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    batch = args.ref_batch
    sps, ms, used, kind = cpu_reference_steps(w, batch, args.steps, args.warmup, threads)
    what = "the unmodified allRank package (baseline/_ref): make_model + loss + train_utils.loss_batch" \
        if kind == "reference" else "oracle port of the reference (baseline/_ref absent)"
    sample = (f"{batch} slates/step x {args.steps} steps (S={w['S']}, F={F}), {what}, eager PyTorch fp32 on the host, "
              f"{used} intra-op threads (fastest of 8..{threads} on a {threads}-thread host)")
    out = {
        "impl": "reference", "metric": "slates/sec", "value": sps, "unit": "slates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, w, batch),
        "cpu_baseline": {"value": sps, "unit": "slates/s", "cores": used, "kind": kind, "sample": sample},
        "e2e": {"value": sps, "unit": "slates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def run_reference_gpu(args, w):
    """Optional, stricter bar (SURVEY.md 8d): the UNMODIFIED reference (baseline/_ref) in eager PyTorch on the same
    B200 -- its make_model, its loss, train_utils.loss_batch, torch.optim.Adam, fp32 (torch's default matmul precision),
    inputs resident on the device.  One JSON line with impl "reference-gpu"."""
    rank, local_rank, world = dist_env()
    if rank != 0:
        return
    if not reference_available():
        print(json.dumps({"impl": "reference-gpu", "unavailable": "baseline/_ref is not installed"}), flush=True)
        return
    from oracle.install_reference import import_path
    sys.path[:0] = import_path()
    import allrank.models.losses as ref_losses
    from allrank.config import TransformerConfig
    from allrank.models.model import make_model as ref_make_model
    from allrank.training.train_utils import loss_batch
    from allrank_b200.synth import make_slates
    from functools import partial
    dev = torch.device("cuda", 0)
    torch.manual_seed(42)
    B = args.batch
    model = ref_make_model(fc_model={"sizes": [w["d"]], "input_norm": False, "activation": None, "dropout": 0.0},
                           transformer=TransformerConfig(N=w["N"], d_ff=w["dff"], h=w["h"], positional_encoding=None,
                                                         dropout=0.0),
                           post_model={"d_output": 1, "output_activation": None}, n_features=F).to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    loss_fn = partial(getattr(ref_losses, w["loss"]), **w["loss_args"])
    x, y, idx = make_slates(B, w["S"], F, seed=1234)
    x, y, idx = x.to(dev), y.to(dev), idx.to(dev)
    for _ in range(args.warmup):
        loss_batch(model, loss_fn, x, y, idx, None, opt)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss_batch(model, loss_fn, x, y, idx, None, opt)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    print(json.dumps({"impl": "reference-gpu", "metric": "slates/sec", "value": B / ms * 1e3, "unit": "slates/s",
                      "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                      "higher_is_better": True, "dtype": "f32", "data": "synthetic",
                      "config": workload_config(args, w, B),
                      "note": "unmodified allRank (baseline/_ref) in eager PyTorch on cuda:0; loss.item() every step "
                              "(train_utils.loss_batch)"}), flush=True)


def cpu_baseline_subprocess(args, w, steps=3, warmup=1):
    """The CPU leg of the default run: the reference arm in a child process with CUDA hidden, bounded to a few steps."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONDONTWRITEBYTECODE="1")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload, "--steps",
           str(steps), "--warmup", str(warmup), "--ref-batch", str(args.ref_batch), "--allow-short-warmup"]
    t0 = time.time()
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        return {"value": None, "unit": "slates/s", "cores": 0, "kind": "unavailable", "sample": r.stderr[-300:]}
    cb = json.loads(lines[-1])["cpu_baseline"]
    cb["sample"] += f"; {steps} timed steps after {warmup} warm-up, {time.time() - t0:.1f}s of CPU work"
    return cb


def workload_config(args, w, batch, live_frac=1.0):
    # bytes one step touches: ~20 MB of activations per slate for cfg2 (profiles/README.md), inputs batch*S*F*4;
    # live_frac: the share of the B * S rows the encoder runs over (packed rows, include/allrank_b200.h)
    act_mb = live_frac * batch * w["S"] * (w["N"] * (10 * w["d"] + 2 * w["dff"]) + w["d"]) * 4 * 2 / 1e6
    return {"workload": f"{args.workload}: Transformer(N={w['N']},h={w['h']},d_model={w['d']},d_ff={w['dff']}) + "
                        f"{w['loss']}, slate_len={w['S']}, {F} features, full training step (fwd+loss+bwd+Adam)",
            "batch_per_gpu": batch, "slate_len": w["S"], "n_features": F, "loss": w["loss"],
            "optimizer": "Adam(lr=1e-3)",
            "rows": (f"packed: the encoder runs over the {100 * live_frac:.0f} % of the B*S rows below the slate extents "
                     "(synthetic MSLR lengths N(120, 60) clipped to [1, slate_len]; padded items score 0)"
                     if live_frac < 1.0 else "dense: all B*S rows"),
            "l2": f"no explicit flush: one step streams ~{act_mb:.0f} MB of activations (+ {batch * w['S'] * F * 4 / 1e6:.0f} MB "
                  "of inputs) through the 126 MB L2, so every kernel's inputs come from HBM"
                  + ("" if act_mb > 252 else " -- EXCEPT at this small batch, where parts stay L2-resident between kernels")}


# ------------------------------------------------------------------------------------------------ GPU arm
def kernel_table(lib, psteps, peaks, dtype):
    """Per-kernel roofline from the library's per-launch CUDA-event timings (arb_prof_report): for each distinct
    kernel (GEMMs are named by shape) the algorithmic FLOPs and HBM bytes of its launches in one step, its device time,
    and the fraction of the roof that binds it -- the larger of flops / tensor peak and bytes / HBM copy peak, both
    from MEASURED_PEAKS.json."""
    lib.arb_prof_report.restype = ctypes.c_int64
    lib.arb_prof_report.argtypes = [ctypes.c_char_p, ctypes.c_int64]
    need = int(lib.arb_prof_report(None, 0))
    buf = ctypes.create_string_buffer(need + 64)
    lib.arb_prof_report(buf, need + 64)
    tf32_peak, bf16_peak = peaks["bf16_tflops_sustained"] * 0.5, peaks["bf16_tflops_sustained"]      # TFLOP/s
    rows = []
    for line in buf.value.decode().splitlines():
        name, cls, n, ms, work, nbytes = line.split("\t")
        cls, n, ms, work, nbytes = int(cls), int(n), float(ms), float(work), float(nbytes)
        if ms <= 0:
            continue
        flops = work if cls == 0 else 0.0
        nbytes = nbytes if cls == 0 else work          # non-GEMM classes state their algorithmic bytes as `work`
        tensor_peak = bf16_peak if "_bf16" in name else tf32_peak     # kind::f16 products vs kind::tf32 products
        t_tensor = flops / (tensor_peak * 1e12) * 1e3
        t_hbm = nbytes / (peaks["hbm_gbs"] * 1e9) * 1e3
        bound = "tensor" if t_tensor >= t_hbm else "hbm"
        rows.append({"kernel": name, "launches_per_step": n / psteps, "us_per_step": round(1e3 * ms / psteps, 2),
                     "flops_per_step": flops / psteps, "bytes_per_step": nbytes / psteps,
                     "tflops": round(flops / (ms * 1e-3) / 1e12, 2), "gbs": round(nbytes / (ms * 1e-3) / 1e9, 1),
                     "bound": bound, "frac": round(max(t_tensor, t_hbm) / ms, 4),
                     "tensor_frac": round(t_tensor / ms, 4), "hbm_frac": round(t_hbm / ms, 4), "tensor_peak": tensor_peak})
    rows.sort(key=lambda r: -r["us_per_step"])
    return rows, (bf16_peak if dtype == "bf16" else tf32_peak)


def run_b200(args, w):
    rank, local_rank, world = dist_env()
    import torch.distributed as dist
    from allrank_b200 import _lib, losses
    from allrank_b200.ddp import FlatDDP, loss_weight
    from allrank_b200.model import make_model
    from allrank_b200.optim import FlatAdam
    from allrank_b200.synth import make_slates

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (allrank_b200 has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.scaling == "strong":                 # fixed GLOBAL batch (SURVEY.md 8e: 512), split over the ranks
        if args.global_batch % world:
            raise SystemExit("--global-batch must be divisible by the number of GPUs")
        B = args.global_batch // world
    else:
        B = args.batch
    S = w["S"]
    torch.manual_seed(42)
    model = make_model(fc_model={"sizes": [w["d"]], "input_norm": False, "activation": None, "dropout": 0.0},
                       transformer={"N": w["N"], "d_ff": w["dff"], "h": w["h"], "positional_encoding": None,
                                    "dropout": 0.0},
                       post_model={"d_output": 1, "output_activation": None}, n_features=F,
                       compute_dtype=args.dtype).to(dev).train()
    loss_fn = getattr(losses, w["loss"])
    # two different pinned host batches, alternated by the end-to-end loop
    hosts = []
    for k in range(2):
        xh, yh, _ = make_slates(B, S, F, seed=1234 + rank + 1000 * k)
        hosts.append((xh.pin_memory(), yh.pin_memory()))
    x_host, y_host = hosts[0]
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)
    # share of the rows the encoder runs over when the library packs them (reported in `config`; host arithmetic only)
    live_frac = 1.0
    if _lib.lib().arb_get_pack_rows():
        ext = torch.where(y_host != PAD, torch.arange(1, S + 1)[None, :], torch.zeros(1, S, dtype=torch.long)).max(1).values
        live_frac = float(((ext + 15) // 16 * 16).clamp(max=(S + 15) // 16 * 16).sum()) / float(B * S)
    model._ensure_packed(dev)
    if args.optimizer == "torch":                # the optimiser allrank/main.py:82 instantiates from its config
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    else:
        opt = FlatAdam(model, lr=1e-3, capturable=args.cuda_graph)
    ddp = FlatDDP(model) if world > 1 else None
    mode = "sum" if w["loss"] == "lambdaLoss" else ("weighted" if w["loss"].startswith("neuralNDCG") else "mean")
    if ddp:
        ddp.average = mode != "sum"              # lambdaLoss(reduction="sum") gradients are summed across ranks

    kept = {}

    def step(x, y, keep=False):
        mask = y == PAD                                    # train_utils.py:19
        scores = model(x, mask, None)
        if keep:                                           # --dump-outputs: the scores of the last timed step
            kept["scores"] = scores.detach().clone()
        loss = loss_fn(scores, y, **w["loss_args"])
        loss.backward()
        scale = 1.0
        if ddp:
            if mode == "weighted":               # neuralNDCG: all-reduce numerator and count (neuralNDCG.py:62-69)
                ddp.reduce_gradients(local_weight=loss_weight(w["loss"], y))
            else:
                scale = ddp.reduce_gradients(fold_average_into_optimizer=args.optimizer == "flat")
        if args.optimizer == "flat":
            opt.step(grad_scale=scale)
        else:
            opt.step()
        opt.zero_grad()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    if world > 1:                     # broadcast rank-0 weights before the first step
        ddp.sync_parameters()
    for _ in range(args.warmup):
        step(x_dev, y_dev)
    gstep = None
    if args.cuda_graph:
        if world > 1 or args.optimizer != "flat":
            raise SystemExit("bench.py: --cuda-graph needs one GPU and the flat optimiser")
        from allrank_b200.graph import GraphedTrainStep
        gstep = GraphedTrainStep(model, loss_fn, opt, x_dev, y_dev, loss_kwargs=w["loss_args"])
        l_before = _lib.launch_count()
        step(x_dev, y_dev)                                   # (one eager step: the launches a replay stands for)
        launches_per_replay = _lib.launch_count() - l_before
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()

    # ---- (1) device-resident: inputs already in HBM
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = gstep.replay() if gstep else step(x_dev, y_dev, keep=args.dump_outputs and i == args.steps - 1)
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = launches_per_replay * args.steps if gstep else _lib.launch_count() - l0
    final_loss = loss.item()
    if args.dump_outputs and rank == 0:                    # before the steps below move the parameters on
        kept.update(loss=loss.detach().reshape(1), parameters=model.flat_parameters)
        kept = {k: v.float().cpu().numpy() for k, v in kept.items()}

    # ---- (2) end to end: every step's inputs come from pinned host memory (H2D inside the timed region, issued on
    #      a copy stream one step ahead, the way a training loop with a prefetching loader runs) and the loss is
    #      read back to the host every step (train_utils.loss_batch returns loss.item(), train_utils.py:29)
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)

    def prefetch(k):
        xh, yh = hosts[k & 1]
        with torch.cuda.stream(copy_stream):
            xb = xh.to(dev, non_blocking=True)
            yb = yh.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return xb, yb, ev

    def e2e_loop(n):
        nxt = prefetch(0)
        for i in range(n):
            xb, yb, ev = nxt
            main_stream.wait_event(ev)
            xb.record_stream(main_stream)
            yb.record_stream(main_stream)
            if i + 1 < n:
                nxt = prefetch(i + 1)
            _ = (gstep(xb, yb) if gstep else step(xb, yb)).item()

    e2e_loop(2)
    barrier()
    e0.record()
    e2e_loop(args.steps)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler else None

    # ---- (3) the gradient all-reduce alone (N > 1): the flat bucket, CUDA events, max over ranks
    allreduce_us = None
    if world > 1:
        g = model.flat_gradients
        for _ in range(5):
            dist.all_reduce(g)
        barrier()
        e0.record()
        for _ in range(20):
            dist.all_reduce(g)
        e1.record()
        barrier()
        allreduce_us = 1e3 * max_over_ranks(e0.elapsed_time(e1)) / 20
        g.zero_()

    # ---- (4) per-launch device timing of every kernel (roofline), a few extra steps
    lib = _lib.lib()
    lib.arb_prof_enable.argtypes = [ctypes.c_int32]
    if rank == 0:
        lib.arb_prof_enable(1)
    psteps = 3
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for _ in range(psteps):          # every rank runs these steps (they contain the gradient all-reduce)
        step(x_dev, y_dev)
    pe1.record()
    torch.cuda.synchronize()
    kernels, tensor_peak, step_ms_profiled = [], 0.0, 0.0
    peaks = measured_peaks()
    if rank == 0:
        kernels, tensor_peak = kernel_table(lib, psteps, peaks, args.dtype)
        step_ms_profiled = pe0.elapsed_time(pe1) / psteps
        lib.arb_prof_enable(0)
    if world > 1:
        dist.barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    slates = B * world * args.steps
    value = slates / (ms_total / 1e3)
    e2e_value = slates / (ms_e2e / 1e3)
    top = kernels[0] if kernels else None
    kernel_ms = sum(k["us_per_step"] for k in kernels) / 1e3
    step_flops = flops_per_slate_step(w) * B
    out = {
        "metric": "slates/sec", "value": value, "unit": "slates/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": args.scaling,
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": dict(workload_config(args, w, B, live_frac), global_batch=B * world, cuda_graph=bool(args.cuda_graph),
                       optimizer=("Adam(lr=1e-3), " + ("allrank_b200.optim.FlatAdam (one launch)" if args.optimizer == "flat"
                                                       else "torch.optim.Adam over the module's parameters")),
                       parallelism=f"dp{world}: one process per GPU, one NCCL all-reduce of the flat gradient per step"),
        "e2e": {"value": e2e_value, "unit": "slates/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(x_host.numel() * 4 + y_host.numel() * 4), "d2h_bytes_per_step": 4,
                "note": "two pinned host batches alternate; H2D one step ahead on a copy stream; loss.item() every step"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "final_loss": final_loss,
    }
    if allreduce_us is not None:
        out["allreduce"] = {"us": allreduce_us, "bytes": int(model.flat_gradients.numel() * 4),
                            "note": "flat gradient bucket alone, NCCL, CUDA events, max over ranks; issued after the "
                                    "backward on the compute stream"}
    if top:
        unit = "TFLOP/s" if top["bound"] == "tensor" else "GB/s"
        out["roofline"] = {
            "bound": top["bound"], "kernel": top["kernel"],
            "achieved": top["tflops"] if top["bound"] == "tensor" else top["gbs"],
            "peak": top["tensor_peak"] if top["bound"] == "tensor" else peaks["hbm_gbs"], "unit": unit, "frac": top["frac"],
            "traffic": measured_traffic(args, B, top["kernel"]),
            "us_per_step": top["us_per_step"], "launches_per_step": top["launches_per_step"],
            "share_of_step": round(top["us_per_step"] / 1e3 / step_ms_profiled, 4) if step_ms_profiled else None,
            "peak_source": f"{peaks['source']} (MEASURED_PEAKS.json): tensor = bf16_tflops_sustained "
                           f"{peaks['bf16_tflops_sustained']} for kind::f16 (bf16) products, half of it for kind::tf32 "
                           "products (tf32 issues at half the bf16 rate)" +
                           f", HBM = copy {peaks['hbm_gbs']} GB/s",
            "definition": "dominant kernel = largest device time per step; achieved = algorithmic flops (or bytes) of its "
                          "launches / their CUDA-event time, measured live; frac against the roof that binds that kernel",
            # model_tflops counts the NOMINAL model (all B * S items, padding included -- what the dense reference
            # computes); real_item_tflops the flops the kernels' own accounting attributes to the items below the slate
            # extents (packed rows / padding-tile skip), i.e. what is actually needed
            "whole_step": {"model_tflops": round(step_flops * world / (ms_total / args.steps * 1e-3) / 1e12, 2),
                           "frac_of_tensor_peak": round(step_flops / (ms_total / args.steps * 1e-3) / 1e12 / tensor_peak, 4),
                           "real_item_tflops": round(sum(k["flops_per_step"] for k in kernels) /
                                                     (ms_total / args.steps * 1e-3) / 1e12, 2) if kernels else None,
                           "algorithmic_gbs": round(sum(k["bytes_per_step"] for k in kernels) /
                                                    (kernel_ms * 1e-3) / 1e9, 1) if kernel_ms else None,
                           "kernel_ms_per_step": round(kernel_ms, 3), "step_ms_profiled": round(step_ms_profiled, 3)},
            "kernels": kernels,
        }
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_subprocess(args, w)
    if args.dump_outputs:
        out["dumped"] = dump_outputs(args.dump_outputs, kept)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_MAX_ELEMENTS = 4 << 20     # per array: 16 MB of float32, so that a dump stays within 64 MB


def dump_outputs(path, arrays):
    """Write each array as <path>/<name>.npy (float32).  An array longer than DUMP_MAX_ELEMENTS is replaced by the
    same fixed, seeded sample of its flattened entries in every run, so that two builds compare entry for entry."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    written = {}
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.size > DUMP_MAX_ELEMENTS:
            pick = np.sort(np.random.RandomState(0).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))
            a = a.reshape(-1)[pick]
        np.save(os.path.join(path, name + ".npy"), a)
        written[name] = list(a.shape)
    return written


def measured_traffic(args, batch, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed ncu capture of
    this exact workload / batch (profiles/r2_dram_traffic.json: {workload: {batch: {kernel: bytes}}}), else null."""
    path = os.path.join(ROOT, "profiles", "r2_dram_traffic.json")
    try:
        with open(path) as f:
            cap = json.load(f)
        per_kernel = cap[args.workload][str(int(batch))]
        for name, val in per_kernel.items():
            if kernel.startswith(name):
                return val
    except (OSError, ValueError, TypeError, KeyError):
        pass
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-gpu"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", default="tf32", choices=["tf32", "bf16"],
                    help="arithmetic of the encoder's tensor-core products (LTRModel.compute_dtype); fp32 elsewhere")
    ap.add_argument("--batch", type=int, default=4096,
                    help="slates per step per GPU (saturating batch; 64 = allRank's default batch_size, see profiles/)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch slates per GPU; strong: --global-batch slates split over the GPUs")
    ap.add_argument("--global-batch", type=int, default=512, help="global batch of --scaling strong (SURVEY.md 8e)")
    ap.add_argument("--optimizer", default="flat", choices=["flat", "torch"],
                    help="flat: allrank_b200.optim.FlatAdam; torch: torch.optim.Adam (what allrank/main.py:82 builds)")
    ap.add_argument("--ref-batch", type=int, default=64, help="slates per CPU step (reference default batch_size)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="replay the training step as one CUDA graph (allrank_b200.graph.GraphedTrainStep; one GPU, "
                         "flat optimiser): for small batches, where the host's launch path sets the pace")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last one computed -- the scores, the loss and the "
                         "updated parameters (no scores with --cuda-graph) -- as DIR/<name>.npy (float32); inputs are "
                         "seeded, so runs compare")
    ap.add_argument("--allow-short-warmup", action="store_true", help="(internal: the bounded CPU leg)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and not args.allow_short_warmup:
        args.warmup = 3
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""      # the reference hard-wires cuda:0 when it sees a GPU
        run_reference(args, w)
    elif args.impl == "reference-gpu":
        run_reference_gpu(args, w)
    else:
        run_b200(args, w)


if __name__ == "__main__":
    main()
