"""Cost of the spectral-normalised decoder (Decoder.sn: True) on the training step.

    python tools/bench_sn.py [--batch 256] [--c-in 80 512] [--steps 20] [--windows 3] [--out profiles/r3_bench_sn.json]

For every c_in it builds the same model twice (sn off / on), records both steps into CUDA graphs and then
ALTERNATES timed windows of `steps` replays between the two (off, on, off, on, ...), so that both arms see the
same clocks and neighbours; each arm reports the median window.  It also times the two spectral-norm kernels
alone (CUDA events around a CUDA graph of 50 back-to-back launches, median of 5) and reports the launches per
step of both arms, and the card's name and power limit.  Synthetic N(0,1) segments, device-resident batch.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import oracle.ae_oracle as orc  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"nvidia_smi": q, "torch_name": torch.cuda.get_device_name(0)}


def make_solver(c_in, batch, sn):
    from adaptive_voice_conversion_b200.solver import Solver
    cfg = orc.default_config(c_in)
    cfg["Decoder"]["sn"] = sn
    cfg["data_loader"]["batch_size"] = batch
    args = types.SimpleNamespace(data_dir="synthetic", train_set="", train_index_file="", logdir="/tmp/avc_log", load_model=False,
                                 load_opt=False, store_model_path=None, load_model_path=None, summary_steps=10 ** 9,
                                 save_steps=10 ** 9, tag="bench", iters=0)
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        solver = Solver(cfg, args)
    tr = solver.trainer
    tr.auto_graph = False
    x = solver.train_loader.batches[0].to(tr.dev)
    tr.capture(x, warmup=2)          # two eager steps (they set launches_per_step), then the recording
    for _ in range(3):
        tr.step(x, 1.0)
    torch.cuda.synchronize()
    return solver, x


def window(solver, x, steps):
    tr = solver.trainer
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        tr.step(x, 1.0)
    e1.record()
    torch.cuda.synchronize()
    tr.losses()
    return e0.elapsed_time(e1) / steps


def kernel_times(model, dev, reps=50, trials=5):
    """us per launch of avc_spectral_norm_fwd (update=1) and avc_spectral_norm_bwd over the model's 26 layers."""
    from adaptive_voice_conversion_b200 import _lib as L
    lib = L.load()
    n = len(model.sn_layers())
    params = dict(model.named_parameters())
    G = {l + ".weight": torch.randn_like(params[l + ".weight_orig"]) * 1e-3 for l in model.sn_layers()}
    fwd_tab, bwd_tab = model.sn_table(dev), model.sn_table(dev, G)
    out = {}
    for name, call in (("spectral_norm_fwd", lambda s: lib.avc_spectral_norm_fwd(fwd_tab.data_ptr(), n, 1, s)),
                       ("spectral_norm_bwd", lambda s: lib.avc_spectral_norm_bwd(bwd_tab.data_ptr(), n, s))):
        st = torch.cuda.Stream(dev)
        with torch.cuda.stream(st):
            call(st.cuda_stream)         # warm-up outside the capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            for _ in range(reps):
                L.check(call(st.cuda_stream), name)
        ts = []
        for _ in range(trials):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3 / reps)
        out[name + "_us"] = sorted(ts)[len(ts) // 2]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--c-in", type=int, nargs="+", default=[80, 512])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bench_sn.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sn.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"card": card(), "batch": a.batch, "steps_per_window": a.steps, "windows": a.windows,
           "precision": os.environ.get("AVC_PRECISION", "tf32"), "configs": {}}
    for c_in in a.c_in:
        arms = {sn: make_solver(c_in, a.batch, sn) for sn in (False, True)}
        ms = {False: [], True: []}
        for _ in range(a.windows):
            for sn in (False, True):
                ms[sn].append(window(*arms[sn], a.steps))
        row = {}
        for sn, tag in ((False, "sn_off"), (True, "sn_on")):
            med = sorted(ms[sn])[len(ms[sn]) // 2]
            row[tag] = {"ms_per_step": med, "seg_per_s": a.batch / (med * 1e-3), "windows_ms": ms[sn],
                        "launches_per_step": int(arms[sn][0].trainer.launches_per_step)}
        row["overhead_pct"] = 100.0 * (row["sn_on"]["ms_per_step"] / row["sn_off"]["ms_per_step"] - 1.0)
        row["kernels"] = kernel_times(arms[True][0].model, dev)
        res["configs"][f"c{c_in}"] = row
        print(json.dumps({f"c{c_in}": row}), flush=True)
        del arms
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
