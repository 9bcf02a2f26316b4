#!/usr/bin/env python
"""Headline benchmark: MaxViT grid fields/sec of the 12hr MetNet3 model (BASELINE.json configs[1]:
inference, bf16, batch 64 synthetic CMAQ grids = 768 fields per step per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]

* a "step" = one forward of `MetNet3` over one batch of B=64 synthetic CMAQ tensors (64*12 = 768 grid fields)
* `value`  = fields/s with the inputs already resident in HBM (CUDA events, max over ranks)
* `e2e`    = same metric through the package's public streaming API (`HostPipeline`) with HOST (pinned) inputs: every step's
             H2D of x/timestamps and D2H of the predictions happen inside the timed region, overlapped with the kernels of
             the neighbouring steps on a side stream
* `roofline` = the dominant kernel (3x3-conv implicit GEMM + LN epilogue, tcgen05), from CUDA events recorded
             around its launches inside the timed region; algorithmic FLOPs = 2*84*70*128*1152 per field per launch
* `cpu_baseline` = the CPU oracle port of the reference (oracle/, plain PyTorch fp32) on the host cores, B=1
* `--impl reference` times that same CPU port as the reference arm (the Python reference cannot travel to the box)
* `gpu_eager_baseline` = the same oracle port run as plain PyTorch eager (cuDNN / cuBLAS / ATen) on cuda:0 -- SURVEY 2.1's
             "bar on the box" -- in fp32 with TF32 off and under bf16 autocast, at the largest batch it is run at (stated)
* `train`  = BASELINE configs[2]: the training step (train-mode forward, Focal-R, backward, NCCL gradient all-reduce, fused
             AdamW), with its own roofline block for the kernel with the largest share of the step
* `--config 3|4` = BASELINE configs[3] (512x512 domain, MaxViT depth 2) / configs[4] (512 channels, 32 x 64 heads, depth 4)
* `--dump-outputs DIR` = rank 0 writes the predictions of the last timed inference step as DIR/prediction.npy (float32), so
             that two builds can be compared output for output on identical seeded inputs
N>1: one process per GPU (torchrun), batch-sharded, no data-path collective (inference) -> weak scaling.
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

import torch  # noqa: E402

METRIC, UNIT = "grid_fields_per_sec", "fields/s"
CONV_FLOPS_PER_FIELD = 2.0 * 84 * 70 * 128 * 1152          # algorithmic: unpadded-frame pixels x Cout x 9*Cin x 2
ATTN_FLOPS_PER_FIELD = 2.0125e9                             # SURVEY 8d: qkv 1.2505 + QK^T 0.1726 + PV 0.1726 + out 0.4168 GF, 53-token count
FWD_GFLOP_PER_FIELD_REF = 25.864                            # SURVEY F8 (reference graph, no lead-time dedup)
FWD_GFLOP_PER_FIELD_EXEC = 17.516                           # with the stem computed once per sample (H5)
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, **arrays):
    """write each array as DIRECTORY/<name>.npy in float32.  When the arrays exceed DUMP_LIMIT_BYTES in all, each is replaced
    by a fixed strided sample of its flattened values (the same elements on every run with the same arguments)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    total = sum(a.numel() for a in arrays.values())
    stride = -(-total * 4 // (DUMP_LIMIT_BYTES - 4096 * len(arrays)))      # 4 KB per file for the .npy header
    for name, a in arrays.items():
        a = a.detach().float().cpu()
        if stride > 1:
            a = a.flatten()[::stride]
        np.save(os.path.join(directory, f"{name}.npy"), a.numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def cpu_port_forward_time(batch=1, repeats=3, threads=None):
    """time the CPU oracle port of the reference forward (fp32, eval) -> (best seconds, threads)"""
    from oracle import synth
    from oracle.metnet3_oracle import metnet3_forward
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    cfg = synth.CFG_12HR
    sd = synth.make_state_dict(synth.metnet3_spec(cfg), seed=0)
    x, ts, _ = synth.make_inputs(cfg, batch, seed=1234)
    best = float("inf")
    with torch.no_grad():
        metnet3_forward(x, ts, sd, cfg)                      # warm-up
        for _ in range(repeats):
            t0 = time.perf_counter()
            metnet3_forward(x, ts, sd, cfg)
            best = min(best, time.perf_counter() - t0)
    return best, threads


def gpu_eager_forward_time(dev, batch=16, repeats=3):
    """SURVEY 2.1 / BASELINE.md 4: "PyTorch eager (cuDNN / cuBLAS / ATen) running the reference module" on the same GPU.  The
    reference itself cannot travel to the box, so this runs the oracle port (pinned to the reference by tests/golden) with
    its tensors on the device -- the same ATen call sequence as the reference module.  Three settings: fp32 with TF32 disabled
    (the strict-parity setting), fp32 with TF32 allowed, and bf16 autocast."""
    from oracle import synth
    from oracle.metnet3_oracle import metnet3_forward
    cfg = synth.CFG_12HR
    sd = {k: v.to(dev) for k, v in synth.make_state_dict(synth.metnet3_spec(cfg), seed=0).items()}
    out = {"batch": batch, "fields_per_step": batch * cfg.L, "unit": UNIT, "kind": "oracle port on cuda (PyTorch eager)"}
    x, ts, _ = synth.make_inputs(cfg, batch, seed=1234)
    x, ts = x.to(dev), ts.to(dev)
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    for name in ("fp32_tf32_off", "fp32_tf32_on", "bf16_autocast"):
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = name == "fp32_tf32_on"
        try:
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=name == "bf16_autocast"):
                metnet3_forward(x, ts, sd, cfg)
                torch.cuda.synchronize()
                best = float("inf")
                for _ in range(repeats):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    metnet3_forward(x, ts, sd, cfg)
                    e1.record()
                    torch.cuda.synchronize()
                    best = min(best, e0.elapsed_time(e1))
            out[name] = {"value": batch * cfg.L / (best * 1e-3), "ms_per_step": best}
        except Exception as e:                              # OOM or an op the port cannot run on the device: report, do not fail
            out[name] = {"value": None, "error": f"{type(e).__name__}: {str(e)[:120]}"}
            torch.cuda.empty_cache()
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    del sd, x
    torch.cuda.empty_cache()
    return out


def run_reference(args, rank, world):
    """reference arm: the reference's CPU implementation of the path (oracle port) on the host cores"""
    if rank != 0:
        return
    from oracle import synth
    from oracle.metnet3_oracle import metnet3_forward
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    cfg = synth.CFG_12HR
    sd = synth.make_state_dict(synth.metnet3_spec(cfg), seed=0)
    bs = 1                                                   # bounded sample: one CMAQ tensor (12 fields) per step
    x, ts, _ = synth.make_inputs(cfg, bs, seed=1234)
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 2))):
            metnet3_forward(x, ts, sd, cfg)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            y = metnet3_forward(x, ts, sd, cfg)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, prediction=y)
    value = bs * cfg.L * args.steps / dt
    sample = f"B={bs} synthetic CMAQ tensor (12 fields) per step, fp32, eval, {threads} torch CPU threads"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "12hr MetNet3/MaxViT forward (BASELINE configs[1] model), bounded CPU sample", "batch": bs,
                   "fields_per_step": bs * cfg.L},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


ATTN_BWD_FLOPS_PER_FIELD = 2.0 * 2.0125e9                  # backward of one attention = 2x its forward FLOPs (dX and dW of every contraction)


def run_train(args, cfg, dev, rank, world, barrier, max_over_ranks):
    """BASELINE configs[2]: training step (train-mode forward, Focal-R, hand-written backward, gradient all-reduce over
    NCCL overlapped with backward when world > 1, fused AdamW), batch-sharded data parallel, weak scaling."""
    import torch.distributed as dist
    from oracle import synth
    from vit_grid_model_b200 import MetNet3, DataParallel, FlatAdamW, focal_r_loss, _lib
    Bt, L = args.train_batch, cfg.L
    model = MetNet3(**cfg.metnet3_kwargs())                     # reference defaults, incl. attention dropout 0.1
    model.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=0), strict=True)
    model = model.to(dev).train().set_precision("bf16")
    net = DataParallel(model) if world > 1 else model
    opt = FlatAdamW(model, lr=1e-5)
    x, ts, target = synth.make_inputs(cfg, Bt, seed=4321 + rank)
    x, ts, target = x.to(dev), ts.to(dev), target.to(dev)

    def step():
        opt.zero_grad()
        loss = focal_r_loss(net(x, timestamps=ts), target)
        loss.backward()
        opt.step()
        return loss

    for _ in range(max(5, args.warmup)):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = _lib.launch_count()
    steps = args.steps
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    barrier()
    launches = int((_lib.launch_count() - l0) // steps)
    ms = max_over_ranks(e0.elapsed_time(e1))
    # per-entry-point CUDA events on a few extra steps OUTSIDE the timed region (the host enqueues a step in about half its
    # device time; two event records per launch would eat into that margin)
    _lib.TRACE = []
    tsteps = 3
    for _ in range(tsteps):
        step()
    torch.cuda.synchronize()
    trace, _lib.TRACE = _lib.TRACE, None
    per = {}
    for name, tag, a, b in trace:
        key = name if name not in ("vg_gemm_fwd", "vg_wgrad") else f"{name}[{tag}]"
        per.setdefault(key, []).append(a.elapsed_time(b))
    tot = sum(sum(v) for v in per.values())
    if args.trace and rank == 0:
        print(f"# ---- training step, {Bt * L} fields: {ms / steps:.2f} ms/step, kernels {tot / tsteps:.2f} ms", file=sys.stderr)
        for name, v in sorted(per.items(), key=lambda kv: -sum(kv[1]))[:40]:
            print(f"# {name:60s} calls/step {len(v) // tsteps:3d}  ms/step {sum(v) / tsteps:9.3f}  {100 * sum(v) / tot:5.1f}%", file=sys.stderr)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    top = sorted(per.items(), key=lambda kv: -sum(kv[1]))[:6]
    breakdown = [{"entry": k, "ms_per_step": sum(v) / tsteps, "share": sum(v) / tot} for k, v in top]
    roof = None
    bwd = per.get("vg_attn_bwd_fused") or per.get("vg_attn_core_bwd")
    if bwd:
        name = "vg_attn_bwd_fused" if "vg_attn_bwd_fused" in per else "vg_attn_core_bwd"
        avg = sum(bwd) / len(bwd)
        # the fused backward covers the whole attention (projections included); the un-fused core only QK^T / PV and their gradients
        flops = ATTN_BWD_FLOPS_PER_FIELD if name == "vg_attn_bwd_fused" else 4.0 * 2 * 0.1726e9
        ach = flops * Bt * L / (avg * 1e-3) / 1e12
        roof = {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                "avg_launch_ms": avg, "launches_per_step": len(bwd) // tsteps, "share_of_step": sum(bwd) / tot, "traffic": None}
    n_params = sum(p.numel() for p in model.parameters())
    value = world * Bt * L * steps / (ms * 1e-3)
    return {"metric": "train_grid_fields_per_sec", "value": value, "unit": UNIT,
            "ms_per_step": ms / steps, "steps": steps, "warmup": max(5, args.warmup), "batch_per_gpu": Bt, "fields_per_step": world * Bt * L,
            "loss": float(loss.item()), "gpu_launches": launches,
            "parallelism": f"data parallel x{world}: per-rank batch shards, gradient all-reduce ({n_params * 4 / 1e6:.1f} MB fp32, "
                           f"6 sections, NCCL on a side stream overlapped with backward)" if world > 1 else "single GPU",
            "optimizer": "fused AdamW (one kernel over the flat parameter buffer)", "dropout": model.dropout,
            "gflop_per_field_fwd_bwd": 3 * FWD_GFLOP_PER_FIELD_EXEC,
            "model_tflops": value / world * 3 * FWD_GFLOP_PER_FIELD_EXEC / 1e3, "frac_of_bf16_peak": value / world * 3 * FWD_GFLOP_PER_FIELD_EXEC / 1e3 / peak_tf,
            "roofline": roof, "breakdown": breakdown}


def run_other_config(args, dev, rank, world):
    """BASELINE configs[3] / configs[4] as bench lines (same JSON contract; `config.workload` names the configuration)."""
    import torch.distributed as dist
    from oracle import synth
    from vit_grid_model_b200 import MetNet3, DataParallel, FlatAdamW, focal_r_loss, _lib
    if args.config == 3:
        cfg = synth.GridConfig(H=512, W=512, vit_depth=2)
        B = 1 if args.batch == 64 else args.batch
        workload = ("BASELINE configs[3]: enlarged 512x512 domain (518x518 padded, 1,369 windows per field, grid-partition stride 37), "
                    "MaxViT depth 2, bf16")
        gf_ref = 25.864 * (518 * 518) / (84 * 70) + 4.424 * (259 * 259) / (42 * 35)      # conv part scales with pixels, + one more MaxViT layer
    else:
        cfg = synth.GridConfig(dim=512, heads=32, dim_head=64, vit_depth=4)
        B = 8 if args.batch == 64 else args.batch
        workload = "BASELINE configs[4]: MetNet-3-style backbone, 512 channels, 32 heads x dim_head 64, MaxViT depth 4, 82x67 domain"
        gf_ref = 370.9
    L = cfg.L
    W = max(3, args.warmup)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    model = MetNet3(**cfg.metnet3_kwargs())
    model.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=0), strict=True)
    model = model.to(dev).eval()                               # the constructor's default precision for this width
    if args.config == 3:
        model.set_precision("bf16")
    precision = model.precision
    x, ts, target = synth.make_inputs(cfg, B, seed=1234 + rank)
    x_host, ts_host = x.pin_memory(), ts.pin_memory()
    x, ts, target = x.to(dev), ts.to(dev), target.to(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        for _ in range(W):
            y = model(x, timestamps=ts)               # held like in the timed loop: the allocator sees the same pattern
        barrier()
        l0 = _lib.launch_count()
        with ClockSampler(dev.index or 0) as clk:
            e0.record()
            for _ in range(args.steps):
                y = model(x, timestamps=ts)
            e1.record()
            barrier()
        launches = (_lib.launch_count() - l0) // args.steps
        ms = max_over_ranks(e0.elapsed_time(e1))
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, prediction=y)
        del y
        # end to end: pinned host tensor in, pinned host predictions out, synchronously per step (tiny batches: no pipelining)
        y_host = torch.empty(B, L, cfg.H, cfg.W, dtype=torch.float32).pin_memory()
        barrier()
        e0.record()
        for _ in range(args.steps):
            y_host.copy_(model(x_host.to(dev, non_blocking=True), timestamps=ts_host.to(dev, non_blocking=True)), non_blocking=True)
        e1.record()
        barrier()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    fields = world * B * L * args.steps
    value = fields / (ms * 1e-3)
    # per-entry-point CUDA events on two extra steps outside the timed region: breakdown + roofline of the dominant entry
    breakdown, roof = None, None
    if rank == 0:
        import re
        _lib.TRACE = []
        with torch.no_grad():
            for _ in range(2):
                model(x, timestamps=ts)
        torch.cuda.synchronize()
        trace, _lib.TRACE = _lib.TRACE, None
        per = {}
        for name, tag, a, b in trace:
            per.setdefault(f"{name}[{tag}]" if name == "vg_gemm_fwd" else name, []).append(a.elapsed_time(b))
        tot = sum(sum(v) for v in per.values())
        top = sorted(per.items(), key=lambda kv: -sum(kv[1]))
        breakdown = [{"entry": k, "launches_per_step": len(v) // 2, "ms_per_step": sum(v) / 2, "share": sum(v) / tot} for k, v in top[:8]]
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        name, v = top[0]
        avg = sum(v) / len(v)
        mt = re.search(r"M=(\d+) K=(\d+)x(\d+) N=(\d+) (\S+)( 3xTF32)?", name)
        if mt:                                                  # a GEMM: 2 M K N; a 3xTF32 product executes three times its algorithmic FLOPs
            Mg, taps, Kg, Ng = (int(mt.group(i)) for i in (1, 2, 3, 4))
            split, tf32 = mt.group(6) is not None, mt.group(5) == "tf32"
            algo = 2.0 * Mg * taps * Kg * Ng / (3 if split else 1)
            pk = peak_tf / 2 if tf32 else peak_tf
            roof = {"kernel": f"gemm_tc_kernel via {name}", "bound": "tensor", "achieved": algo / (avg * 1e-3) / 1e12, "peak": pk, "unit": "TFLOP/s",
                    "frac": algo / (avg * 1e-3) / 1e12 / pk, "executed_tflops": algo * (3 if split else 1) / (avg * 1e-3) / 1e12,
                    "avg_launch_ms": avg, "launches_per_step": len(v) // 2, "share_of_step": sum(v) / tot, "traffic": None,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" + (" / 2 (kind::tf32 runs at half the bf16 rate)" if tf32 else "")
                                   + ("; achieved counts the fp32 product's FLOPs, the 3xTF32 split executes three times as many" if split else "")}
        elif name.startswith("vg_conv3x3_ln"):
            C = cfg.dim
            algo = 2.0 * min(B * L, model.max_fields[model.compute_dtype]) * (cfg.H + (14 - cfg.H) % 14) * (cfg.W + (14 - cfg.W) % 14) * 9 * C * C
            tf32 = model.conv_tf32
            pk = peak_tf / 2 if tf32 else peak_tf
            roof = {"kernel": name, "bound": "tensor", "achieved": algo / (avg * 1e-3) / 1e12, "peak": pk, "unit": "TFLOP/s",
                    "frac": algo / (avg * 1e-3) / 1e12 / pk, "avg_launch_ms": avg, "launches_per_step": len(v) // 2, "share_of_step": sum(v) / tot,
                    "traffic": None, "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" + (" / 2 (kind::tf32)" if tf32 else ""),
                    "note": "algorithmic FLOPs of the padded frame (multiple of 14 in both directions) of the fields one launch covers"}
    opt_in = None
    if precision != "bf16":
        # the reduced-precision mode of a wide network is opt-in: it misses the 1e-2 tolerance at this depth (DESIGN.md 2)
        model.set_precision("bf16")
        with torch.no_grad():
            for _ in range(W):
                model(x, timestamps=ts)
            barrier()
            e0.record()
            for _ in range(args.steps):
                model(x, timestamps=ts)
            e1.record()
            barrier()
        ms16 = max_over_ranks(e0.elapsed_time(e1))
        opt_in = {"precision": "bf16 (opt-in; 3.6e-2 vs the oracle at this depth: outside the 1e-2 tolerance)", "value": fields / (ms16 * 1e-3),
                  "ms_per_step": ms16 / args.steps, "model_tflops_reference_graph": fields / (ms16 * 1e-3) / world * gf_ref / 1e3}
        model.set_precision(precision)
    train = None
    if not args.no_train:
        try:
            model.train()
            net = DataParallel(model) if world > 1 else model
            opt = FlatAdamW(model, lr=1e-5)

            def step():
                opt.zero_grad()
                loss = focal_r_loss(net(x, timestamps=ts), target)
                loss.backward()
                opt.step()
                return loss

            for _ in range(3):
                step()
            barrier()
            steps = args.steps
            e0.record()
            for _ in range(steps):
                loss = step()
            e1.record()
            barrier()
            tms = max_over_ranks(e0.elapsed_time(e1))
            train = {"metric": "train_grid_fields_per_sec", "value": world * B * L * steps / (tms * 1e-3), "unit": UNIT,
                     "ms_per_step": tms / steps, "steps": steps, "fields_per_step": world * B * L, "loss": float(loss.item()),
                     "max_memory_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
        except NotImplementedError as e:
            train = {"unavailable": str(e)}
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": precision,
            "data": "synthetic", "reduced_precision_opt_in": opt_in,
            "config": {"workload": workload, "batch_per_gpu": B, "fields_per_step": world * B * L,
                       "input_shape": [B, cfg.T, cfg.C, cfg.H, cfg.W], "gflop_per_field_reference_graph": gf_ref,
                       "l2": "activations of one step exceed the 126 MB L2", "parallelism": f"batch-sharded x{world}"},
            "clocks": clk.summary(),
            "e2e": {"value": fields / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": x_host.numel() * 4 + ts_host.numel() * 4, "d2h_bytes_per_step": y_host.numel() * 4},
            "gpu_launches": int(launches), "roofline": roof, "breakdown": breakdown,
            "model_tflops_reference_graph": value / world * gf_ref / 1e3,
            "max_memory_gb": torch.cuda.max_memory_allocated() / 2 ** 30,
            "train": train,
        }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every leg")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="CMAQ samples per GPU per step (x12 lead times = fields)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step measurement (BASELINE configs[2])")
    ap.add_argument("--train-batch", type=int, default=16, help="CMAQ samples per GPU per training step")
    ap.add_argument("--trace", action="store_true", help="print a per-entry-point time breakdown (rank 0)")
    ap.add_argument("--config", type=int, default=1, choices=[1, 3, 4],
                    help="BASELINE.json configs index: 1 = the headline (12hr model, B=64 inference + the configs[2] training step); "
                         "3 = 512x512 domain, MaxViT depth 2 (inference + training step); 4 = 512 channels, 32 x 64 heads, depth 4")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the PyTorch-eager-on-GPU comparator")
    ap.add_argument("--e2e-input", default="bf16", choices=["bf16", "fp32"],
                    help="host format of the e2e leg's inputs: bf16 = batches packed by pipeline.pack_host (bit-identical "
                         "predictions, half the H2D bytes); fp32 = the reference's tensor; the other one is reported beside it")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the predictions of the last timed step to DIR/prediction.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from oracle import synth                                  # synthetic weights / inputs only (no oracle compute here)
    from vit_grid_model_b200 import MetNet3, _lib

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(3, args.warmup)

    if args.config != 1:
        run_other_config(args, dev, rank, world)
        if world > 1:
            dist.destroy_process_group()
        return

    cfg = synth.CFG_12HR
    B, L = args.batch, cfg.L
    model = MetNet3(**cfg.metnet3_kwargs())
    model.load_state_dict(synth.make_state_dict(synth.metnet3_spec(cfg), seed=0), strict=True)
    model = model.to(dev).eval().set_precision(args.precision)
    x, ts, _ = synth.make_inputs(cfg, B, seed=1234 + rank)    # every rank has its own shard of CMAQ time steps
    x_host, ts_host = x.pin_memory(), ts.pin_memory()
    x_dev, ts_dev = x_host.to(dev), ts_host.to(dev)
    y_host = torch.empty(B, L, cfg.H, cfg.W, dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def step_resident():
        return model(x_dev, timestamps=ts_dev)

    with torch.no_grad():
        # ---------------- device-resident throughput
        for _ in range(W):
            y = step_resident()                       # held like in the timed loop: the allocator sees the same pattern
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = _lib.launch_count()
        _lib.TRACE = []
        with ClockSampler(local) as clk:
            e0.record()
            for _ in range(args.steps):
                y = step_resident()
            e1.record()
            barrier()
        trace, _lib.TRACE = _lib.TRACE, None
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, prediction=y)
        del y
        launches = (_lib.launch_count() - launches0) // args.steps
        ms_total = max_over_ranks(e0.elapsed_time(e1))
        # ---------------- end to end (host buffers in, host predictions out) through the package's streaming API:
        # every step's inputs come from pinned host memory and its predictions land in pinned host memory inside the timed
        # region; HostPipeline overlaps those copies with the kernels of the neighbouring steps (side stream + events)
        from vit_grid_model_b200 import HostPipeline, pack_host
        pipe = HostPipeline(model)
        y_hosts = [torch.empty(B, L, cfg.H, cfg.W, dtype=torch.float32).pin_memory() for _ in range(2)]
        x_packed = pack_host(x, cfg.pm25_mean, cfg.pm25_std)          # data-loader side, outside the timed region (stated in config)

        def e2e_run(x_in):
            for _ in pipe.run((x_in, ts_host, y_hosts[i % 2]) for i in range(2)):
                pass
            barrier()
            e0.record()
            n_out = 0
            for _ in pipe.run((x_in, ts_host, y_hosts[i % 2]) for i in range(args.steps)):
                n_out += 1
            e1.record()
            barrier()
            assert n_out == args.steps
            return max_over_ranks(e0.elapsed_time(e1))

        ms_e2e_fp32 = e2e_run(x_host)
        y_ref = y_hosts[(args.steps - 1) % 2].clone()
        ms_e2e_bf16 = e2e_run(x_packed)
        packed_identical = bool(torch.equal(y_ref, y_hosts[(args.steps - 1) % 2]))
        ms_e2e = ms_e2e_bf16 if args.e2e_input == "bf16" else ms_e2e_fp32

    train = None
    if not args.no_train and args.precision == "bf16":
        train = run_train(args, cfg, dev, rank, world, barrier, max_over_ranks)

    fields = world * B * L * args.steps
    value = fields / (ms_total * 1e-3)
    e2e_value = fields / (ms_e2e * 1e-3)

    # ---------------- per-entry-point breakdown + roofline of the dominant kernel (events from the timed region)
    per = {}
    for name, tag, a, b in trace:
        per.setdefault(name, []).append(a.elapsed_time(b))
        if name == "vg_conv3x3_ln_fwd":
            per.setdefault(f"  conv[{tag}]", []).append(a.elapsed_time(b))
        if name == "vg_gemm_fwd":
            per.setdefault(f"  gemm[{tag}]", []).append(a.elapsed_time(b))
    conv_ms = per.get("vg_conv3x3_ln_fwd", [])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)     # sustained: the kernel is timed inside a long step
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    traffic, traffic_all = None, {}
    try:
        traffic_all = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        traffic = traffic_all.get("conv3x3_ln_dram_bytes_per_launch")
    except Exception:
        pass
    roofline, kernels = None, []
    if conv_ms and args.precision == "bf16":
        avg_ms = sum(conv_ms) / len(conv_ms)
        achieved = CONV_FLOPS_PER_FIELD * B * L / (avg_ms * 1e-3) / 1e12
        kernels.append({"kernel": "conv_halo_kernel (3x3 conv 128->128 implicit GEMM, tcgen05 kind::f16, + ChanLN/FiLM/ReLU/residual epilogue)",
                        "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                        "traffic": traffic, "launches_per_step": len(conv_ms) // args.steps, "avg_launch_ms": avg_ms,
                        "peak_source": peak_src, "share_of_step": sum(conv_ms) / ms_total,
                        "algorithmic_gflop_per_field_per_launch": CONV_FLOPS_PER_FIELD / 1e9,
                        "variants": {k.strip()[5:-1]: {"launches_per_step": len(v) // args.steps, "avg_launch_ms": sum(v) / len(v),
                                                       "frac": CONV_FLOPS_PER_FIELD * B * L / (sum(v) / len(v) * 1e-3) / 1e12 / peak_tf,
                                                       "traffic": (traffic_all.get("conv_variants") or {}).get(k.strip()[5:-1])}
                                     for k, v in per.items() if k.startswith("  conv[")}})
    attn_ms = (per.get("vg_attn_fused2_fwd") or per.get("vg_attn_fused_fwd", []))
    if attn_ms and args.precision == "bf16":
        avg_ms = sum(attn_ms) / len(attn_ms)
        achieved = ATTN_FLOPS_PER_FIELD * B * L / (avg_ms * 1e-3) / 1e12
        attn_traffic = None
        try:
            attn_traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get("attn_fused_dram_bytes_per_launch")
        except Exception:
            pass
        kernels.append({"kernel": "attn_fused2_kernel (window / grid attention in one kernel, in place on the residual stream: partition = TMA tensor maps, "
                                  "residual add = TMA reduce-store; tcgen05 kind::f16 QKV projection, QK^T and PV on fp16 / bf16 operands, kind::tf32 out-projection; "
                                  "X, P, O operands in TMEM; two compute groups on alternate heads, three MMA issuers)",
                        "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                        "traffic": attn_traffic, "launches_per_step": len(attn_ms) // args.steps, "avg_launch_ms": avg_ms,
                        "peak_source": peak_src + "; 21 % of this kernel's FLOPs (the out-projection) run as kind::tf32 (half the bf16 rate)",
                        "share_of_step": sum(attn_ms) / ms_total,
                        "algorithmic_gflop_per_field_per_launch": ATTN_FLOPS_PER_FIELD / 1e9})
    kernels.sort(key=lambda k: -k["share_of_step"])
    # HBM-bound kernels of the step against the measured copy bandwidth: algorithmic bytes (the tensors each kernel must read
    # and write once, in their storage types) / launch time.  The two GELU kernels are issue-bound, not bandwidth-bound; they are
    # listed with the same yardstick so that nothing hides.
    peak_bw = peaks.get("hbm_gbs", 6560.0)
    F, PXB, PXN, LOWP = B * L, B * 85 * 71 + 71, B * L * 85 * 71 + 71, B * L * 42 * 35
    bw_spec = [
        ("vg_prepare_fwd", None, "prepare (PM2.5 standardise, pad, NCHW fp32 -> channels-last bf16)", x_host.numel() * 4 + PXB * 640 * 2),
        ("vg_stem_finish_fwd", None, "stem finish (+time terms, ChanLN, FiLM, ReLU per lead time; bf16 + fp32 skip out)", PXB * 128 * 4 * 2 + PXN * 128 * (2 + 4)),
        ("vg_pool2_fwd", None, "2x2 max-pool bf16 -> fp32", PXN * 128 * 2 + LOWP * 128 * 4),
        ("vg_gemm_fwd", "K=1x128 N=512", "MBConv expand 1x1 + BN + GELU (tf32 MMA, fp16 out; GELU issue-bound)", LOWP * 128 * 4 + LOWP * 512 * 2),
        ("vg_dw3x3_fwd", None, "MBConv depthwise 3x3 + BN + GELU (fp16 in / out; GELU + stencil issue-bound)", LOWP * 512 * 2 * 2),
        ("vg_gemm_fwd", "K=1x512 N=128", "MBConv project 1x1 + BN (fp16 operands, SE gate folded into per-field weights)", LOWP * 512 * 2 + LOWP * 128 * 4),
        ("vg_convT2_fwd", None, "ConvTranspose 2x2 as GEMM + depth-to-space (bf16 + fp32 skip out)", LOWP * 128 * 4 + PXN * 128 * (2 + 4)),
    ]
    bandwidth = []
    if args.precision == "bf16":
        for entry, tagpat, label, nbytes in bw_spec:
            ms_list = [a.elapsed_time(b) for name, tag, a, b in trace if name == entry and (tagpat is None or tagpat in tag)]
            if ms_list:
                avg = sum(ms_list) / len(ms_list)
                gbs = nbytes / (avg * 1e-3) / 1e9
                bandwidth.append({"kernel": label, "entry": entry, "avg_launch_ms": avg, "algorithmic_bytes": nbytes, "achieved_gbs": gbs,
                                  "peak_gbs": peak_bw, "frac": gbs / peak_bw, "share_of_step": sum(ms_list) / ms_total})
    if kernels:
        roofline = dict(kernels[0])                           # the dominant kernel of the step
        roofline["other_kernels"] = kernels[1:]
        roofline["bandwidth_kernels"] = bandwidth

    if rank == 0:
        if args.trace:
            tot = sum(sum(v) for k, v in per.items() if not k.startswith("  "))
            for name, v in sorted(per.items(), key=lambda kv: -sum(kv[1])):
                print(f"# {name:24s} calls/step {len(v) // args.steps:3d}  ms/step {sum(v) / args.steps:9.3f}  {100 * sum(v) / tot:5.1f}%", file=sys.stderr)
        cpu = eager = None
        if world == 1 and not args.no_cpu_baseline:
            # BASELINE.md 3: all host cores, and the reference's own setting of 4 threads (evaluation_vit.py:3-5)
            allc = os.cpu_count() or 1
            sec, threads = cpu_port_forward_time(batch=1, repeats=3, threads=allc)
            sec4, _ = cpu_port_forward_time(batch=1, repeats=2, threads=min(4, allc))
            cpu = {"value": L / sec, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": f"oracle port of the reference forward, B=1 (12 fields), fp32 eval, best of 3 after 1 warm-up, {threads} torch threads, {sec:.3f} s/forward",
                   "threads_4": {"value": L / sec4, "cores": min(4, allc), "seconds_per_forward": sec4,
                                 "note": "the reference pins OMP/MKL/OPENBLAS threads to 4 (evaluation_vit.py:3-5)"}}
        if world == 1 and not args.no_eager_baseline:
            eager = gpu_eager_forward_time(dev, batch=16)
            for k in ("fp32_tf32_off", "fp32_tf32_on", "bf16_autocast"):
                if eager.get(k, {}).get("value"):
                    eager[k]["speedup_of_this_repo"] = value / eager[k]["value"]
        h2d = {"bf16": x_packed.numel() * 2 + ts_host.numel() * 4, "fp32": x_host.numel() * 4 + ts_host.numel() * 4}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": "BASELINE configs[1]: 12hr MetNet3/MaxViT inference, batch 64 synthetic CMAQ grids per GPU (768 fields/step/GPU)",
                       "batch_per_gpu": B, "fields_per_step": world * B * L, "input_shape": [B, cfg.T, cfg.C, cfg.H, cfg.W],
                       "l2": "inputs (844 MB) and every activation exceed the 126 MB L2", "parallelism": f"batch-sharded x{world}, no collective",
                       "e2e_input": f"{args.e2e_input}: " + ("pinned bf16 batches packed once by pipeline.pack_host outside the timed region (the data-loader "
                                    "side; PM2.5 channels standardised in fp32 before the rounding, predictions bit-identical to the fp32 tensor: "
                                    f"checked in this run = {packed_identical})" if args.e2e_input == "bf16" else "the reference's pinned fp32 tensor"),
                       "gflop_per_field_reference_graph": FWD_GFLOP_PER_FIELD_REF, "gflop_per_field_executed": FWD_GFLOP_PER_FIELD_EXEC,
                       "lead_time_dedup": True},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": h2d[args.e2e_input], "d2h_bytes_per_step": y_host.numel() * 4,
                    "frac_of_device_resident": e2e_value / value,
                    "fp32_host_input": {"value": fields / (ms_e2e_fp32 * 1e-3), "ms_per_step": ms_e2e_fp32 / args.steps, "h2d_bytes_per_step": h2d["fp32"]},
                    "bf16_host_input": {"value": fields / (ms_e2e_bf16 * 1e-3), "ms_per_step": ms_e2e_bf16 / args.steps, "h2d_bytes_per_step": h2d["bf16"],
                                        "bit_identical_to_fp32_input": packed_identical}},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "gpu_eager_baseline": eager,
            "model_tflops_executed": value * FWD_GFLOP_PER_FIELD_EXEC / 1e3,
            "train": train,
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
