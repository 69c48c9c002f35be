"""CPU: the spectral-normalised decoder (Decoder.sn: True).  AE builds with the reference's parameter / state_dict
inventory, and the CPU restatement (oracle/sn_oracle.py) reproduces the fixtures written by the unmodified reference
with sn: True (oracle/make_golden_sn.py): outputs, sigma, the u / v trajectory and gradients."""
import ctypes
import os
import subprocess
import tempfile

import pytest
import torch

import oracle.ae_oracle as orc
import oracle.sn_oracle as sno
from oracle.make_golden import reference_eps
from conftest import ROOT


def load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), weights_only=False)


def rel(a, b):
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def x_of(fx):
    return torch.randn(fx["x_shape"], generator=torch.Generator().manual_seed(fx["x_seed"]))


def eps_of(rec):
    """The reference's N(0,1) draw of a step, regenerated from its seed (the fixtures do not store it)."""
    return reference_eps(rec["eps_shape"], rec["eps_seed"])


@pytest.mark.parametrize("name", ["train_c80_sn_b4.pt", "train_c512_sn_b2.pt"])
def test_ae_inventory_matches_reference(golden_dir, name):
    from adaptive_voice_conversion_b200.model import AE
    fx = load(golden_dir, name)
    cfg = sno.sn_config(fx["c_in"])
    model = AE(cfg)
    assert [n for n, _ in model.named_parameters()] == fx["names"]
    sd = model.state_dict()
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == fx["state_keys"]
    assert len(sd) == 218 and len(fx["names"]) == 166
    # (the reference's parameter-less act / dropout / norm modules have metadata entries of their own)
    sn_meta = {k: dict(v) for k, v in sd._metadata.items() if "spectral_norm" in v}
    assert sn_meta == {k: v for k, v in fx["metadata"].items() if "spectral_norm" in v}
    assert len(sn_meta) == 26 and all(v["spectral_norm"] == {"weight.version": 1} for v in sn_meta.values())
    assert model.sn_layers() == sno.sn_layers(cfg) and len(model.sn_layers()) == 26
    # the oracle's inventory, and its state loads strict
    assert [n for n, _ in sno.param_shapes(cfg)] == fx["names"]
    assert [(k, tuple(s)) for k, s in sno.state_shapes(cfg)] == fx["state_keys"]
    model.load_state_dict(sno.init_state(cfg, seed=0), strict=True)
    model.load_state_dict(sd, strict=True)   # and our own state_dict round-trips


def test_sn_false_is_unchanged():
    from adaptive_voice_conversion_b200.model import AE
    cfg = orc.default_config(80)
    model = AE(cfg)
    assert not model.sn and model.sn_layers() == []
    assert [(k, tuple(v.shape)) for k, v in model.state_dict().items()] == [(k, tuple(s)) for k, s in orc.param_shapes(cfg)]


def test_sn_item_layout_matches_header():
    from adaptive_voice_conversion_b200 import _lib as L
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "avc_b200.h"\nint main(){printf("%zu %zu\\n", sizeof(avc_sn_item), offsetof(avc_sn_item, rows));return 0;}\n'
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "s.c")
        open(c, "w").write(prog)
        exe = os.path.join(td, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        size, off = [int(v) for v in subprocess.check_output([exe]).split()]
    assert (size, off) == (ctypes.sizeof(L.SnItem), L.SnItem.rows.offset)


def test_oracle_train_steps(golden_dir):
    fx = load(golden_dir, "train_c80_sn_b4.pt")
    cfg = sno.sn_config(fx["c_in"])
    sd = sno.init_state(cfg, seed=0)
    x = x_of(fx)
    st = orc.AdamState(sno.params_of(sd))
    for i, rec in enumerate(fx["steps"]):
        tol = 2e-4 if i == 0 else 3e-2    # Adam drift of two fp32 implementations, as in test_oracle_golden.py
        res = sno.ae_train_step(sd, st, cfg, x, eps_of(rec), fx["lambda_kl"])
        o = res["outs"]
        for k in ("mu", "log_sigma", "emb", "dec"):    # (after the first step: the first sample's only)
            a = o[k][:rec[k].shape[0]]
            assert rel(a, rec[k]) < tol, (i, k, rel(a, rec[k]))
        assert abs(res["loss_rec"] - float(rec["loss_rec"])) / float(rec["loss_rec"]) < tol / 10
        assert abs(res["grad_norm"] - float(rec["grad_norm"])) / float(rec["grad_norm"]) < tol
        assert torch.allclose(o["sigma"], rec["sigma"], rtol=1e-5 if i == 0 else 1e-3)
        gl2 = torch.stack([res["grads"][k].norm() for k in fx["names"]])
        assert torch.allclose(gl2, rec["grad_l2"], rtol=50 * tol, atol=1e-5)
        if i == 0:
            for k, g in rec["grad_small"].items():
                assert rel(res["grads"][k], g) < 5e-3 or float(g.abs().max()) < 1e-5, k
        pl2 = torch.stack([sd[k].norm() for k in fx["names"]])
        assert torch.allclose(pl2, rec["param_l2_after"], rtol=1e-5 if i == 0 else 2e-3)
        if i + 1 in fx["uv"]:
            for layer, (u, v) in fx["uv"][i + 1].items():
                t = 1e-5 if i == 0 else 1e-3
                assert rel(sd[layer + ".weight_u"], u) < t and rel(sd[layer + ".weight_v"], v) < t, (i, layer)


def test_oracle_train_step_c512(golden_dir):
    fx = load(golden_dir, "train_c512_sn_b2.pt")
    cfg = sno.sn_config(fx["c_in"])
    sd = sno.init_state(cfg, seed=0)
    rec = fx["steps"][0]
    res = sno.ae_train_step(sd, orc.AdamState(sno.params_of(sd)), cfg, x_of(fx), eps_of(rec), fx["lambda_kl"])
    assert rel(res["outs"]["dec"], rec["dec"]) < 2e-4
    assert abs(res["grad_norm"] - float(rec["grad_norm"])) / float(rec["grad_norm"]) < 2e-4
    assert torch.allclose(res["outs"]["sigma"], rec["sigma"], rtol=1e-5)
    for layer, (u, v) in fx["uv"][1].items():
        assert rel(sd[layer + ".weight_u"], u) < 1e-5 and rel(sd[layer + ".weight_v"], v) < 1e-5, layer


def test_oracle_inference_eval_mode(golden_dir):
    fx = load(golden_dir, "infer_c80_sn.pt")
    cfg = sno.sn_config(fx["c_in"])
    sd = sno.init_state(cfg, seed=0)
    before = {k: v.clone() for k, v in sd.items()}
    with torch.no_grad():
        dec, sig = sno.ae_inference(sd, cfg, fx["x"], fx["x_cond"])
    assert rel(dec, fx["dec"]) < 2e-4
    assert torch.allclose(sig, fx["sigma"], rtol=1e-6)
    assert all(torch.equal(sd[k], before[k]) for k in sd)     # eval mode writes nothing
