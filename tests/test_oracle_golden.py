"""The CPU oracle (oracle/ae_oracle.py) against the fixtures generated from the unmodified
reference (oracle/make_golden.py).  This is what pins the oracle: every later GPU parity
test compares the CUDA path with this oracle and with the same fixtures."""
import os

import pytest
import torch

import oracle.ae_oracle as orc


def load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), weights_only=False)


def rel(a, b):
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def test_state_dict_inventory():
    cfg = orc.default_config(80)
    shapes = orc.param_shapes(cfg)
    assert len(shapes) == 166                       # SURVEY.md section 8b: 166 tensors, no buffers
    assert sum(torch.Size(s).numel() for _, s in shapes) == 4892880
    assert sum(torch.Size(s).numel() for _, s in orc.param_shapes(orc.default_config(512))) == 9040512


def test_helpers(golden_dir):
    fx = load(golden_dir, "helpers.pt")
    x = fx["x"]
    for key, stride in (("pad_conv_k1", 1), ("pad_conv_k2", 1), ("pad_conv_k5", 1), ("pad_conv_k8", 1), ("pad_conv_k5_s2", 2)):
        g = fx[key]
        assert rel(orc.reflect_conv1d(x, g["w"], g["b"], stride), g["y"]) < 1e-6, key
    assert torch.equal(orc.pixel_shuffle_1d(x, 2), fx["pixel_shuffle"])
    assert torch.equal(torch.nn.functional.interpolate(x, scale_factor=2, mode="nearest"), fx["upsample"])
    assert rel(orc.adain(x, fx["cond"]), fx["append_cond"]) < 1e-6
    assert rel(orc.instance_norm(x), fx["instance_norm"]) < 1e-5


@pytest.mark.parametrize("name", ["train_c80_b1.pt", "train_c80_b4.pt", "train_c512_b2.pt"])
def test_train_steps(golden_dir, name):
    fx = load(golden_dir, name)
    cfg = orc.default_config(fx["c_in"])
    sd = orc.init_state(cfg, seed=0)
    chk = torch.tensor([float(sum(v.double().sum() for v in sd.values())),
                        float(sum(v.double().abs().sum() for v in sd.values()))])
    assert torch.allclose(chk, fx["state_checksum"], rtol=1e-6), "seeded init differs from the fixture's"
    assert list(sd) == fx["names"]
    st = orc.AdamState(sd)
    # Adam's first steps move every element by ~lr*sign(g): elements whose gradient is
    # rounding noise (e.g. biases feeding an InstanceNorm, analytically zero) take a
    # +-lr step in a noise-determined direction, so trajectories of two fp32
    # implementations drift apart after the first step.  Step 0 is checked tightly, later
    # steps loosely (they still catch optimizer-state bugs: wrong bias correction or
    # amsgrad max shows up as O(1) relative error in param_l2_after).
    for i, rec in enumerate(fx["steps"]):
        tol = 2e-4 if i == 0 else 3e-2
        res = orc.ae_train_step(sd, st, cfg, fx["x"], rec["eps"], fx["lambda_kl"])
        o = res["outs"]
        for k in ("mu", "log_sigma", "emb", "dec"):
            assert rel(o[k], rec[k]) < tol, (name, i, k, rel(o[k], rec[k]))
        assert abs(res["loss_rec"] - float(rec["loss_rec"])) / float(rec["loss_rec"]) < tol / 10
        assert abs(res["loss_kl"] - float(rec["loss_kl"])) / float(rec["loss_kl"]) < tol / 10
        assert abs(res["grad_norm"] - float(rec["grad_norm"])) / float(rec["grad_norm"]) < tol
        gl2 = torch.stack([res["grads"][k].norm() for k in fx["names"]])
        assert torch.allclose(gl2, rec["grad_l2"], rtol=50 * tol, atol=1e-5)
        if i == 0:
            for k, g in rec["grad_small"].items():
                assert rel(res["grads"][k], g) < 5e-3 or float(g.abs().max()) < 1e-5, (name, k)
        pl2 = torch.stack([sd[k].norm() for k in fx["names"]])
        assert torch.allclose(pl2, rec["param_l2_after"], rtol=1e-5 if i == 0 else 2e-3)
        if i == 0:
            for k, p in rec["param_small_after"].items():
                g = rec["grad_small"][k]
                sel = g.abs() > 1e-5          # skip noise-gradient elements (see above)
                assert ((sd[k] - p).abs() * sel).max() < 1e-4, (name, k)


@pytest.mark.parametrize("name", ["infer_c80.pt", "infer_c80_t512.pt"])
def test_inference(golden_dir, name):
    fx = load(golden_dir, name)
    cfg = orc.default_config(fx["c_in"])
    sd = orc.init_state(cfg, seed=0)
    with torch.no_grad():
        dec = orc.ae_inference(sd, cfg, fx["x"], fx["x_cond"])
        emb = orc.speaker_encoder(sd, fx["x_cond"], cfg["SpeakerEncoder"]["subsample"])
    assert dec.shape == fx["dec"].shape
    assert rel(dec, fx["dec"]) < 2e-4
    assert rel(emb, fx["emb"]) < 2e-4


def test_live_reference_matches_fixture(golden_dir):
    """A forward pass of the unmodified reference, recorded by oracle/make_golden.py, against the
    training fixture made from the same seeds (guards the fixture generator itself) and against
    the oracle fed the noise the reference draws after seeding torch's generator."""
    from oracle.make_golden import reference_eps
    ref = load(golden_dir, "reference_fwd_c80_b1.pt")
    fx = load(golden_dir, "train_c80_b1.pt")
    assert torch.equal(ref["x"], fx["x"])
    assert rel(ref["dec"], fx["steps"][0]["dec"]) < 1e-5
    cfg = orc.default_config(80)
    eps = reference_eps(ref["log_sigma"].shape, ref["eps_seed"])
    with torch.no_grad():
        mu, ls, emb, dec = orc.ae_forward(orc.init_state(cfg, seed=0), cfg, ref["x"], eps)
    for k, v in (("mu", mu), ("log_sigma", ls), ("emb", emb), ("dec", dec)):
        assert rel(v, ref[k]) < 2e-4, (k, rel(v, ref[k]))


def test_torch_optim_step_agrees_with_restated_adam(golden_dir):
    """The two CPU step drivers of the oracle (hand-restated clip+Adam vs stock torch.optim)
    agree on the first step."""
    fx = load(golden_dir, "train_c80_b1.pt")
    cfg = orc.default_config(80)
    sd = orc.init_state(cfg, seed=0)
    stepper = orc.TorchOptimStep(sd, cfg)
    eps = fx["steps"][0]["eps"]
    m = stepper.step(fx["x"], eps, fx["lambda_kl"])
    res = orc.ae_train_step(sd, orc.AdamState(sd), cfg, fx["x"], eps, fx["lambda_kl"])
    assert abs(m["grad_norm"] - res["grad_norm"]) / res["grad_norm"] < 1e-5
    worst = max(float((stepper.params[k].detach() - sd[k]).abs().max()) for k in sd)
    assert worst < 1e-6
