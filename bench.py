#!/usr/bin/env python
"""bench.py -- headline measurement of the AdaIN-VC hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--c-in 80] [--batch 256] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A "step" is one full Solver train step (forward + backward + grad-norm clip + Adam/amsgrad)
on one batch of 256 synthetic 80-mel x 128-frame segments per GPU (BASELINE.json config 3;
weak scaling, config 4, for N > 1).  Prints ONE JSON line (rank 0).

  value   : segments/s with inputs resident in HBM (CUDA-graph replay of the fused step),
            K steps timed with CUDA events between barriers, max over ranks.
  e2e     : the same metric through the public API ``Solver.ae_step`` with pinned HOST
            batches: per step one H2D copy of the batch and a D2H read of the losses.
  roofline: the dominant kernel (fused conv block 128->128, k=5, T=128, IN+ReLU, B=256),
            timed alone with CUDA events on rotating >L2 buffers.
  cpu_baseline / --impl reference: the CPU oracle port of the reference path
            (oracle/ae_oracle.py, torch CPU fp32, all host threads) on a bounded sample.

--dump-outputs DIR: after the timed steps, the parameters and the optimizer state are put back to what they
were before the first step, and one more step runs through the timed path (the captured graph, called through
Solver.ae_step on the first host batch).  That step's losses and the gradient it computed are written as
DIR/<name>.npy.  Weights, batch and noise are seeded, so this step has the same inputs on every run (for a
given --c-in, --batch and number of GPUs), and its outputs differ between runs only by the rounding of the
reductions that add with atomics (bias and weight gradients, loss sums).  On a B200 (1000 W power limit),
runs at --steps 20 and 3 agreed to 1.1e-7 relative L2 on the gradient and 4e-7 relative on the losses.
The chained timed steps are not what is dumped: every Adam step carries that rounding into the next, and a
weight whose gradient is analytically zero (a bias in front of an InstanceNorm) moves by +-lr in the direction
of its rounding noise, so after the timed steps two runs of one build are far apart.  For the same reason the
updated parameters are not dumped.
"""
from __future__ import annotations

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

# torchrun exports OMP_NUM_THREADS=1 to every rank; rank 0 also runs the CPU legs (cpu_baseline,
# --impl reference), which must be free to use the host's cores: clear it BEFORE torch loads.
if os.environ.get("RANK", "0") == "0":
    for _v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.pop(_v, None)

import torch  # noqa: E402

METRIC = "mel-segments/sec (80x128) train step"
UNIT = "segments/s"
SEG_T = 128


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--c-in", type=int, default=80)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--skip-extras", action="store_true", help="skip the extra configurations (fp32 path, c_in=512, inference) of the N=1 line")
    ap.add_argument("--windows", type=int, default=3, help="timed windows of --steps steps each; the median window is reported")
    ap.add_argument("--e2e-api", choices=["ae_step", "run_steps"], default="run_steps",
                    help="public call timed by the e2e arm: Solver.run_steps (the loop body of Solver.train: pinned host batch "
                         "copied per step, losses read per step, copy/read pipelined one step deep; default), or Solver.ae_step "
                         "per pinned host batch (the reference's blocking call)")
    ap.add_argument("--workload", default="train", choices=["train", "inference"],
                    help="train: BASELINE config 3/4 (default, the headline metric); inference: config 5, 64 (src,tgt) pairs of 80x512")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, run one step from the initial parameters and optimizer state through the timed path "
                         "and write its losses and gradient as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl, args.workload) != ("b200", "train"):
        ap.error("--dump-outputs writes the outputs of the training step of --impl b200 --workload train")
    return args


def config_for(c_in, batch):
    from adaptive_voice_conversion_b200.config import default_config
    cfg = default_config(c_in)
    cfg["data_loader"]["batch_size"] = batch
    return cfg


def workload_config(args, world):
    """`config` of the JSON line -- the same dict on the product arm and on the reference arm."""
    B = args.batch
    return {"workload": f"Solver.ae_step fwd+bwd+clip+Adam(amsgrad), batch {B}/GPU of {args.c_in}-mel x 128-frame segments (BASELINE config 3/4)",
            "global_batch": B * world, "per_gpu_batch": B, "c_in": args.c_in, "parallelism": f"dp{world}",
            # timing rule: inputs / working set larger than L2 (a property of the workload, the same on both arms)
            "l2": "per-step working set (~1.5 GB saved activations at batch 256) >> 126 MB L2; no explicit flush"}


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region.  NVML in-process (about a
    thousand samples per second); falls back to polling nvidia-smi (a few samples per second)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.sm, self.power, self.mask, self.sm_max, self.how = [], [], 0, None, "nvidia-smi"
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml, self.how = pynvml, "nvml"
        except Exception:
            self.nvml = None
        self.th = threading.Thread(target=self.run_nvml if self.nvml else self.run_smi, daemon=True)

    def run_nvml(self):
        n = self.nvml
        reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self.stop.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.power.append(n.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                if reasons is not None:
                    self.mask |= int(reasons(self.h))
            except Exception:
                pass
            self.stop.wait(0.002)

    def run_smi(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.02)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=3)

    def summary(self):
        if self.nvml:
            if not self.sm:
                return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": [], "samples": 0, "how": self.how}
            sm = sorted(self.sm)
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.sm_max, "power_w_max": max(self.power) if self.power else None,
                    "reasons": [name for name, bit in self.REASONS if self.mask & bit], "samples": len(sm), "how": self.how}
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "how": self.how}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max((float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()), default=None),
                "reasons": reasons, "samples": len(self.rows), "how": self.how}


# ----------------------------------------------------------------------------- CPU arm
def cpu_reference_rate(c_in, batch, steps, warmup):
    """The reference path on the host cores: oracle port of Solver.ae_step (fwd+bwd+clip+Adam,
    stock torch CPU kernels).  "All the host threads it can use": the thread count is chosen by
    a short sweep (oversubscribing a many-core host makes oneDNN slower, not faster)."""
    import oracle.ae_oracle as orc
    cfg = orc.default_config(c_in)
    stepper = orc.TorchOptimStep(orc.init_state(cfg, seed=0), cfg)
    g = torch.Generator().manual_seed(1)
    x = torch.randn((batch, c_in, SEG_T), generator=g)
    eps = torch.randn((batch, 128, SEG_T // 8), generator=g)
    ncpu = os.cpu_count() or 1
    cands = sorted({n for n in (ncpu, ncpu // 2, ncpu // 4, 32, 16, 8) if 1 <= n <= ncpu}, reverse=True)
    xs, es = x[: max(8, batch // 8)], eps[: max(8, batch // 8)]
    best_n, best_t = cands[0], float("inf")
    for n in cands:
        torch.set_num_threads(n)
        stepper.step(xs, es, 1.0)
        t0 = time.perf_counter()
        stepper.step(xs, es, 1.0)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best_n, best_t = n, dt
    torch.set_num_threads(best_n)
    for _ in range(warmup):
        stepper.step(x, eps, 1.0)
    t0 = time.perf_counter()
    for _ in range(steps):
        stepper.step(x, eps, 1.0)
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps, best_n


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_b = args.batch          # the product arm's per-GPU batch: same config on both arms
    steps, warmup = max(1, min(args.steps, 20)), max(1, min(args.warmup, 2))
    rate, spt, cores = cpu_reference_rate(args.c_in, sample_b, steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": spt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic N(0,1) segments, random-init weights (seed 0)",
        "config": workload_config(args, max(1, args.gpus)),   # identical to the product arm's
        "run": {"executed_on": "host CPU (reference arm: the oracle port of the reference's Solver.ae_step)"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{steps} steps of one GPU's batch ({sample_b} segments) after {warmup} warm-up (oracle port of the reference Solver.ae_step, torch CPU fp32, best of a thread sweep: {cores} of {os.cpu_count()} threads)"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- roofline leg
def dominant_kernel_roofline(dev, batch):
    """Fused conv block 128->128, k=5, T=128, InstanceNorm+ReLU, save_c on (training form)."""
    from adaptive_voice_conversion_b200.engine import A4, Engine
    from adaptive_voice_conversion_b200 import _lib as L
    eng = Engine(config_for(80, batch), dev)
    Cc, T, K = 128, SEG_T, 5
    w = torch.randn(Cc, Cc, K, device=dev) * 0.04
    P = {"r.weight": w, "r.bias": torch.zeros(Cc, device=dev)}
    eng.conv_names = lambda: ["r"]
    eng.pack_weights(P, need_dgrad=False)
    nbuf = 10  # 10 x 16.8 MB inputs > 126 MB L2
    xs = [A4.empty(batch, Cc, T, dev) for _ in range(nbuf)]
    for a in xs:
        a.t.normal_()
    # the kernel is shorter than a Python launch: time a CUDA graph of `reps` back-to-back launches
    # (rotating >L2 inputs) with events on the launching stream
    reps = 20
    side = torch.cuda.Stream(dev)

    def timed():
        for i in range(3):
            eng.conv(P, "r", xs[i % nbuf], norm=True, relu=True, train=True)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        keep = []
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                for i in range(reps):
                    keep.append(eng.conv(P, "r", xs[i % nbuf], norm=True, relu=True, train=True))
            graph.replay()
            side.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(side)
            for _ in range(3):
                graph.replay()
            e1.record(side)
            side.synchronize()
        return e0.elapsed_time(e1) / (3 * reps)

    # the block as the FIRST conv of a ConvBlock pair sees it: fp32 residual-stream input, rounded to TF32 while staged
    avg_ms = timed()
    # ... and as the SECOND conv sees it: input already TF32-exact (written by a rounding producer), no rounding pass
    avg_ms_pre = None
    if eng.precision == "tf32":
        for a in xs:
            a.tf32 = True
        avg_ms_pre = timed()
    flops = 2.0 * Cc * Cc * K * T * batch
    alg_bytes = (Cc * T * batch * 4) * 3 + w.numel() * 4  # read x, write c (saved for bwd) and y, read weights
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    peak_hbm = float(peaks.get("hbm_gbs", 6650.0))
    src = ("measured (MEASURED_PEAKS.json: hbm_gbs copy bandwidth; bf16_tflops burst for the tensor keys)" if peaks
           else "fallback 6.65 TB/s / 1.59 PFLOP/s (B200_PROFILING.md)")
    tf = flops / (avg_ms * 1e-3) / 1e12
    gbs = alg_bytes / (avg_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None   # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full capture
    if eng.precision == "tf32":
        for name in ("r2_ncu_full_conv_block_tc.json", "r1_ncu_full_conv_block_tc.json"):
            try:
                m = json.load(open(os.path.join(ROOT, "profiles", name)))
                scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
                traffic = sum(float(m[k][0]) * scale[m[k][1]] for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
                traffic_src = "profiles/" + name
                break
            except Exception:
                continue
    # Governing roofline: at the TF32 tensor rate (half the bf16 rate) this block needs ~4.7 us of tensor time
    # but ~7.7 us of HBM time for its algorithmic bytes (x in once, c and y out once, weights) -> HBM-bound.
    return {"bound": "hbm", "achieved": gbs, "peak": peak_hbm, "unit": "GB/s", "frac": gbs / peak_hbm, "traffic": traffic,
            "traffic_source": traffic_src,
            "kernel": ("conv_block_tc2_kernel (persistent tcgen05 TF32: fused reflect-pad conv k5 128->128 + InstanceNorm + ReLU, saves c)" if eng.precision == "tf32"
                       else "conv_block_fwd_kernel<5,1,128,128> (same block, fp32 FFMA path)"),
            "shape": f"B={batch}, 128->128, k=5, T={T}",
            "avg_launch_ms": avg_ms, "avg_launch_ms_prerounded_input": avg_ms_pre,
            "input": "fp32 (the residual stream: rounded to TF32 while staged); avg_launch_ms_prerounded_input = the same launch on a TF32-exact input "
                     "(the second conv of every block), not used for frac",
            "alg_bytes_per_launch": alg_bytes, "alg_flops_per_launch": flops,
            "alg_bytes_note": "read x 16.8 MB + write c (saved for backward) 16.8 MB + write y 16.8 MB + weights 0.33 MB",
            "tensor_tflops": tf, "tensor_frac_of_bf16_peak": tf / peak_tf, "tensor_frac_of_tf32_rate": tf / (0.5 * peak_tf),
            "peak_source": src, "precision": eng.precision,
            "timing": "CUDA graph of 20 back-to-back launches on rotating >L2 inputs (10 x 16.8 MB), CUDA events on the launching stream"}


# ----------------------------------------------------------------------------- main arm
def run_b200(args):
    import types
    from adaptive_voice_conversion_b200 import _lib as L
    from adaptive_voice_conversion_b200.solver import Solver
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    L.load(build_if_missing=False)

    cfg = config_for(args.c_in, args.batch)
    sargs = types.SimpleNamespace(data_dir="synthetic", train_set="", train_index_file="", logdir="/tmp/avc_log", load_model=False,
                                  load_opt=False, store_model_path=None, load_model_path=None, summary_steps=10 ** 9,
                                  save_steps=10 ** 9, tag="bench", iters=0)
    import contextlib, io
    torch.manual_seed(0)   # the initial weights and the reparameterisation noise: the same on every run
    with contextlib.redirect_stdout(io.StringIO()):
        solver = Solver(cfg, sargs)
    tr = solver.trainer
    B, K, W = args.batch, args.steps, max(args.warmup, 3)
    host_batches = solver.train_loader.batches          # pinned host N(0,1) batches (seed 1+rank)
    x_dev = host_batches[0].to(dev)
    opt = solver.opt
    step_state = [opt.flat_p, opt.flat_m, opt.flat_v, opt.flat_vmax, opt.step_dev]   # what a step reads and updates
    initial_state = [t.clone() for t in step_state] if args.dump_outputs else None

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident arm: NWIN windows of exactly K steps, each bracketed by barrier + synchronize; the
    # reported window is the MEDIAN one (a single 0.1 s window is at the mercy of one straggler rank)
    tr.auto_graph = False            # the capture below is explicit; --no-graph (profiling runs) stays eager
    if not args.no_graph:
        tr.capture(x_dev, warmup=2)
    for _ in range(W):
        tr.step(x_dev, 1.0)
    launches_per_step = tr.launches_per_step
    NWIN = max(1, args.windows)

    def timed_windows(run_k):
        out = []
        for _ in range(NWIN):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            meta_ = run_k()
            e1.record()
            barrier()
            t = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)   # max over ranks, per window
            out.append(float(t[0]))
        return out, meta_

    def run_resident():
        for _ in range(K):
            tr.step(x_dev, 1.0)

    def run_e2e():
        if args.e2e_api == "run_steps":
            return solver.run_steps(K, lambda_of=lambda it: 1.0)
        for i in range(K):
            m = solver.ae_step(host_batches[i % len(host_batches)], 1.0)
        return m

    with ClockSampler(local) as clk:
        win, _ = timed_windows(run_resident)
        # ---- end-to-end arm through the public API, host batches
        if args.e2e_api == "run_steps":
            solver.run_steps(2, lambda_of=lambda it: 1.0)
        else:
            for i in range(2):
                solver.ae_step(host_batches[i % len(host_batches)], 1.0)
        win_e2e, meta = timed_windows(run_e2e)
    ms, ms_e2e = sorted(win)[len(win) // 2], sorted(win_e2e)[len(win_e2e) // 2]
    finite = all(map(lambda v: v == v and abs(v) != float("inf"), meta.values()))
    precision = tr.eng.precision
    if args.dump_outputs:   # every rank takes the step (it all-reduces); rank 0 writes it
        for t, t0 in zip(step_state, initial_state):
            t.copy_(t0)
        tr.eng.pack_weights(tr.P, need_dgrad=True)
        torch.manual_seed(0)   # its noise, whatever --steps and --warmup ran before
        losses = solver.ae_step(host_batches[0], 1.0)
        if rank == 0:
            dump_outputs(args.dump_outputs, losses, opt.flat_g)

    if rank == 0:
        value = B * world * K / (ms * 1e-3)
        e2e = B * world * K / (ms_e2e * 1e-3)
        roof = dominant_kernel_roofline(dev, B)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            # arithmetic type of the conv path: tcgen05 kind::tf32 (TF32 operands, fp32 accumulate) or exact fp32 FFMA
            "dtype": "tf32" if precision == "tf32" else "f32",
            "data": "synthetic N(0,1) segments, random-init weights",
            "config": workload_config(args, world),   # identical on the reference arm
            "run": {"executed_on": "B200", "cuda_graph": not args.no_graph,
                    "streams": ("3 (speaker-encoder branch beside the content-encoder branch, forward and backward; the decoder's weight "
                                "gradients on a third, lower-priority stream)") if os.environ.get("AVC_OVERLAP", "1") == "1" else "1"},
            "timing": {"windows": NWIN, "steps_per_window": K, "reported": "median window",
                       "window_ms": win, "e2e_window_ms": win_e2e},
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e / K, "h2d_bytes_per_step": B * args.c_in * SEG_T * 4, "d2h_bytes_per_step": 16,
                    "api": ("Solver.ae_step(pinned host batch, lambda_kl) -> {'loss_rec','loss_kl','grad_norm'}" if args.e2e_api == "ae_step" else
                            "Solver.run_steps(K) (= the loop of Solver.train): every step copies its own pinned host batch to the device and reads its own 16-byte loss report; the copy of batch i+1 and the read of step i-1 overlap step i")},
            "gpu_launches": int(launches_per_step) * K,
            "launches_per_step": int(launches_per_step),
            "clocks": clk.summary(),
            "roofline": roof,
            "last_losses": meta, "losses_finite": finite,
            "build": L.load().avc_build_info().decode(),
        }
    del solver, tr
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    if world == 1 and not args.skip_extras:
        line["extras"] = extra_lines(args, dev)
    if world == 1 and not args.skip_cpu:   # cpu_baseline: rank 0 at N=1 only (no rank spins on a barrier meanwhile)
        rate, spt, cores = cpu_reference_rate(args.c_in, B, 3, 1)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"3 steps of batch {B} after 1 warm-up (oracle port of the reference Solver.ae_step, torch CPU fp32, best of a thread sweep: {cores} of {os.cpu_count()} threads), {spt:.2f} s/step"}
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, losses, flat_g):
    """What the dumped step computed, as out_dir/<name>.npy: the losses Solver.ae_step returns (float64
    scalars) and the step's gradient (float32, flattened in model.parameters() order).  Gradient elements
    beyond the dump's 64 MB are replaced by a fixed, seeded sample of them, in index order."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, value in losses.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.float64(value))
    g = flat_g.detach().cpu()
    keep = (DUMP_BYTES - 4096) // 4
    if g.numel() > keep:
        g = g[torch.randperm(g.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values]
    np.save(os.path.join(out_dir, "gradients.npy"), g.numpy())


def _quick_train_rate(c_in, batch, dev, steps, precision=None):
    """seg/s of the graph-replayed step for one more configuration (device-resident, CUDA events)."""
    import types, contextlib, io
    from adaptive_voice_conversion_b200.solver import Solver
    old = os.environ.get("AVC_PRECISION")
    if precision:
        os.environ["AVC_PRECISION"] = precision
    try:
        sargs = types.SimpleNamespace(data_dir="synthetic", train_set="", train_index_file="", logdir="/tmp/avc_log", load_model=False,
                                      load_opt=False, store_model_path=None, load_model_path=None, summary_steps=10 ** 9,
                                      save_steps=10 ** 9, tag="bench", iters=0)
        with contextlib.redirect_stdout(io.StringIO()):
            solver = Solver(config_for(c_in, batch), sargs)
        tr = solver.trainer
        x = solver.train_loader.batches[0].to(dev)
        tr.capture(x, warmup=2)
        for _ in range(3):
            tr.step(x, 1.0)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            tr.step(x, 1.0)
        e1.record()
        torch.cuda.synchronize(dev)
        tr.losses()
        ms = e0.elapsed_time(e1) / steps
        return {"value": batch / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "precision": tr.eng.precision,
                "launches_per_step": int(tr.launches_per_step)}
    finally:
        if precision:
            if old is None:
                os.environ.pop("AVC_PRECISION", None)
            else:
                os.environ["AVC_PRECISION"] = old


def extra_lines(args, dev):
    """Other configurations, measured in the same run (N=1): the exact-fp32 path, the shipped config.yaml
    (c_in=512) and BASELINE config 5 (inference).  Each is a short device-resident measurement."""
    out = {}
    legs = (("train_fp32_path", lambda: _quick_train_rate(args.c_in, args.batch, dev, 5, "fp32")),
            ("train_c_in_512", lambda: _quick_train_rate(512, args.batch, dev, 10)),
            ("inference_config5", lambda: inference_rates(args.c_in, 10, 3, skip_cpu=True)))
    for name, fn in legs:
        try:
            out[name] = fn()
        except Exception as e:   # an extra must never take the headline line down
            out[name] = {"error": repr(e)[:200]}
        torch.cuda.empty_cache()
    return out


def inference_rates(c_in, K, W, skip_cpu=False):
    """BASELINE config 5: one-shot VC on 64 synthetic (src, tgt) 80-mel utterance pairs of 512
    frames through Inferencer.inference_batch; utterances/s, device-resident and e2e (host pairs)."""
    import types
    from adaptive_voice_conversion_b200.inference import Inferencer
    dev = torch.device("cuda", 0)
    cfg = config_for(c_in, 64)
    inf = Inferencer(cfg, types.SimpleNamespace(attr=None, model=None, source=None, target=None, output=None, sample_rate=24000))
    g = torch.Generator().manual_seed(3)
    xs = torch.randn((64, c_in, 512), generator=g).pin_memory()
    xc = torch.randn((64, c_in, 512), generator=g).pin_memory()
    xd, cd = xs.to(dev), xc.to(dev)
    for _ in range(W):
        out = inf.inference_batch(xd, cd)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        out = inf.inference_batch(xd, cd)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    host = torch.empty((64, c_in, 512), dtype=torch.float32).pin_memory()
    for _ in range(K):   # every step: pinned host pairs -> device, convert, converted mels -> pinned host memory, wait for them
        host.copy_(inf.inference_batch(xs.to(dev, non_blocking=True), xc.to(dev, non_blocking=True)), non_blocking=True)
        torch.cuda.current_stream().synchronize()
    f1.record()
    torch.cuda.synchronize()
    ms2 = f0.elapsed_time(f1)
    inf.model.engine(dev).check_tc_status()
    precision = inf.model.engine(dev).precision
    line = {"metric": "inference utts/sec (one-shot VC, 80-mel x 512-frame pairs)", "value": 64 * K / (ms * 1e-3), "unit": "utterances/s",
            "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "tf32" if precision == "tf32" else "f32", "data": "synthetic N(0,1) mels, random-init weights",
            "config": {"workload": "AE.inference, 64 (src,tgt) pairs of 80x512 (BASELINE config 5)", "global_batch": 64},
            "e2e": {"value": 64 * K / (ms2 * 1e-3), "unit": "utterances/s", "h2d_bytes_per_step": 2 * xs.numel() * 4, "d2h_bytes_per_step": host.numel() * 4},
            "precision": precision}
    if not skip_cpu:
        import oracle.ae_oracle as orc
        torch.set_num_threads(min(16, os.cpu_count() or 1))
        sd = orc.init_state(cfg, seed=0)
        with torch.no_grad():
            orc.ae_inference(sd, cfg, xs[:8], xc[:8])
            t0 = time.perf_counter()
            orc.ae_inference(sd, cfg, xs, xc)
            dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": 64 / dt, "unit": "utterances/s", "cores": min(16, os.cpu_count() or 1), "kind": "port",
                                "sample": "one batched pass over the 64 pairs (oracle port, torch CPU fp32)"}
    return line


def run_inference(args):
    print(json.dumps(inference_rates(args.c_in, args.steps, max(args.warmup, 3), args.skip_cpu)), flush=True)


def main():
    args = parse()
    if args.workload == "inference" and args.impl != "reference":
        return run_inference(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
