"""CPU: host-side logic that does not need a device."""
import pytest
import torch

import oracle.ae_oracle as orc


def test_conv_geometry_matches_torch():
    from adaptive_voice_conversion_b200.engine import conv_geometry
    for K in range(1, 9):
        for stride in (1, 2):
            for T in (8, 16, 37, 128, 301):
                pl, pr, Tout = conv_geometry(K, stride, T)
                w = torch.zeros(1, 1, K)
                y = orc.reflect_conv1d(torch.zeros(1, 1, T), w, None, stride)
                assert Tout == y.shape[-1] and pl + pr == K - 1


def test_model_state_dict_matches_reference_inventory():
    from adaptive_voice_conversion_b200.model import AE
    for c_in in (80, 512):
        cfg = orc.default_config(c_in)
        m = AE(cfg)
        sd = m.state_dict()
        assert [(k, tuple(v.shape)) for k, v in sd.items()] == [(k, tuple(s)) for k, s in orc.param_shapes(cfg)]


def test_no_cpu_fallback():
    from adaptive_voice_conversion_b200 import _lib as L
    from adaptive_voice_conversion_b200.model import AE
    m = AE(orc.default_config(80))
    with pytest.raises(L.AvcError):
        m(torch.zeros(1, 80, 128))
    with pytest.raises(L.AvcError):
        m.inference(torch.zeros(1, 80, 128), torch.zeros(1, 80, 128))
    if not torch.cuda.is_available():
        from adaptive_voice_conversion_b200.engine import Engine
        with pytest.raises(L.AvcError):
            Engine(orc.default_config(80), torch.device("cpu"))


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under the package may reference it."""
    import os
    from conftest import ROOT
    pkg = os.path.join(ROOT, "adaptive_voice_conversion_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_collate_and_synthetic_loader():
    import numpy as np
    from adaptive_voice_conversion_b200.data_utils import CollateFn, SyntheticSegments
    items = [np.arange(128 * 80, dtype=np.float32).reshape(128, 80) for _ in range(3)]
    out = CollateFn(1)(items)
    assert out.shape == (3, 80, 128) and float(out[0, 5, 7]) == 7 * 80 + 5
    it = iter(SyntheticSegments(4, 80, 128, seed=3))
    a, b = next(it), next(it)
    assert a.shape == (4, 80, 128) and not torch.equal(a, b)


def test_bench_reference_arm_schema():
    """`bench.py --impl reference` (the CPU oracle port timed on the host) prints ONE JSON line
    with the contract's keys; runs without a GPU."""
    import json, subprocess, sys, os
    from conftest import ROOT
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, env=dict(os.environ, OMP_NUM_THREADS="8"))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    # same workload as the product arm's default line: batch 256 per GPU, c_in 80 (not a smaller sample batch)
    import argparse, importlib.util
    spec = importlib.util.spec_from_file_location("avc_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    want = bench.workload_config(argparse.Namespace(batch=256, c_in=80), 1)
    assert d["config"] == want      # the very dict the product arm prints (arm-specific facts live under "run")


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: one float64 .npy per loss, the gradient in float32, and a fixed sample of
    the gradient when it exceeds the dump's size limit."""
    import importlib.util, os, sys
    import numpy as np
    from conftest import ROOT
    spec = importlib.util.spec_from_file_location("avc_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.randn(1000)
    losses = {"loss_rec": 1.5, "loss_kl": 0.25, "grad_norm": 3.0}
    bench.dump_outputs(str(tmp_path / "a"), losses, g)
    for k, v in losses.items():
        a = np.load(tmp_path / "a" / f"{k}.npy")
        assert a.dtype == np.float64 and float(a) == v
    a = np.load(tmp_path / "a" / "gradients.npy")
    assert a.dtype == np.float32 and np.array_equal(a, g.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 4 * 100)
    bench.dump_outputs(str(tmp_path / "b"), losses, g)
    bench.dump_outputs(str(tmp_path / "c"), losses, g)
    b, c = np.load(tmp_path / "b" / "gradients.npy"), np.load(tmp_path / "c" / "gradients.npy")
    assert b.shape == (100,) and np.array_equal(b, c) and np.isin(b, a).all()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--dump-outputs", str(tmp_path)])
    with pytest.raises(SystemExit):
        bench.parse()


def test_cli_flags_match_reference_names():
    """main.py keeps the reference's flag names (main.py:9-22 of the reference)."""
    import importlib.util, os
    from conftest import ROOT
    spec = importlib.util.spec_from_file_location("avc_main", os.path.join(ROOT, "main.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    a = m.parse_args(["-c", "x.yaml", "-d", "dd", "-train_set", "tr", "-train_index_file", "i.json", "-logdir", "l", "--load_model",
                      "-store_model_path", "s", "-load_model_path", "p", "-summary_steps", "7", "-save_steps", "9", "-t", "tag", "-iters", "3"])
    assert (a.config, a.data_dir, a.train_set, a.train_index_file, a.load_model, a.load_opt, a.summary_steps, a.iters, a.tag) == \
           ("x.yaml", "dd", "tr", "i.json", True, False, 7, 3, "tag")
