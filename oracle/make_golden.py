"""Generate tests/golden/*.pt by running the UNMODIFIED reference (/root/reference/model.py).

TEST INFRASTRUCTURE.  Runs only in the authoring container (the GPU box has no
/root/reference); the fixtures it writes are committed.  Usage:

    python oracle/make_golden.py            # writes tests/golden/

The reference cannot be imported as-is: utils.py:3-4 imports tensorboardX and
editdistance, which are not installed, so empty stand-in modules are registered first.
Nothing is written into /root/reference and no reference source is copied.

Weights come from ``oracle.ae_oracle.init_state(config, seed)`` (portable, seeded) and are
loaded into the reference ``AE`` with ``load_state_dict`` -- this also proves the 166
state_dict names/shapes of ``param_shapes`` match the reference exactly (strict load).
``eps`` is injected by seeding torch's global generator right before ``AE.forward``: with
dropout p=0 the ``normal_()`` at model.py:383 is the first draw after the seed.
"""
from __future__ import annotations

import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = "/root/reference"


def import_reference():
    tb = types.ModuleType("tensorboardX")
    tb.SummaryWriter = type("SummaryWriter", (), {"__init__": lambda self, *a, **k: None})
    sys.modules.setdefault("tensorboardX", tb)
    sys.modules.setdefault("editdistance", types.ModuleType("editdistance"))
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import model as ref_model  # noqa: E402  (the reference's model.py)
    return ref_model


def randn(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


def run_ae(ref_model, config, sd, x, eps_seed):
    ae = ref_model.AE(config)
    ae.load_state_dict(sd, strict=True)
    torch.manual_seed(eps_seed)
    mu, ls, emb, dec = ae(x)
    return ae, mu, ls, emb, dec


def reference_eps(shape, eps_seed):
    torch.manual_seed(eps_seed)
    return torch.empty(shape).normal_(0, 1)


SMALL_GRADS = [
    "speaker_encoder.conv_bank.0.bias", "speaker_encoder.in_conv_layer.bias",
    "speaker_encoder.second_conv_layers.1.bias", "speaker_encoder.first_dense_layers.0.weight",
    "speaker_encoder.output_layer.weight", "content_encoder.conv_bank.7.bias",
    "content_encoder.first_conv_layers.0.bias", "content_encoder.mean_layer.weight",
    "content_encoder.std_layer.bias", "decoder.in_conv_layer.weight",
    "decoder.second_conv_layers.0.bias", "decoder.second_conv_layers.1.bias",
    "decoder.conv_affine_layers.0.weight", "decoder.conv_affine_layers.11.bias",
    "decoder.out_conv_layer.weight", "decoder.out_conv_layer.bias",
]


def make_train_fixture(ref_model, c_in, batch, T, n_steps, name):
    import oracle.ae_oracle as orc
    config = orc.default_config(c_in)
    sd = orc.init_state(config, seed=0)
    x = randn((batch, c_in, T), seed=1)
    ae = ref_model.AE(config)
    ae.load_state_dict(sd, strict=True)
    o = config["optimizer"]
    opt = torch.optim.Adam(ae.parameters(), lr=o["lr"], betas=(o["beta1"], o["beta2"]),
                           amsgrad=o["amsgrad"], weight_decay=o["weight_decay"])
    fx = {"c_in": c_in, "x": x, "lambda_kl": 0.37, "steps": []}
    fx["state_checksum"] = torch.tensor([float(sum(v.double().sum() for v in sd.values())),
                                         float(sum(v.double().abs().sum() for v in sd.values()))])
    for step in range(n_steps):
        eps_seed = 100 + step
        torch.manual_seed(eps_seed)
        # the ae_step body of solver.py:82-93 driven through the reference's own modules
        mu, ls, emb, dec = ae(x)
        loss_rec = torch.nn.L1Loss()(dec, x)
        loss_kl = 0.5 * torch.mean(torch.exp(ls) + mu ** 2 - 1 - ls)
        loss = config["lambda"]["lambda_rec"] * loss_rec + fx["lambda_kl"] * loss_kl
        opt.zero_grad()
        loss.backward()
        grads = {k: (p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p))
                 for k, p in ae.named_parameters()}
        gnorm = torch.nn.utils.clip_grad_norm_(ae.parameters(), max_norm=o["grad_norm"])
        opt.step()
        rec = {
            "eps": reference_eps(ls.shape, eps_seed),
            "mu": mu.detach().clone(), "log_sigma": ls.detach().clone(),
            "emb": emb.detach().clone(), "dec": dec.detach().clone(),
            "loss_rec": loss_rec.detach().clone(), "loss_kl": loss_kl.detach().clone(),
            "grad_norm": torch.as_tensor(float(gnorm)),
            "grad_l2": torch.stack([grads[k].norm() for k in grads]),
            "grad_small": {k: grads[k] for k in SMALL_GRADS},
            "param_l2_after": torch.stack([p.detach().norm() for p in ae.parameters()]),
            "param_small_after": {k: dict(ae.named_parameters())[k].detach().clone() for k in SMALL_GRADS},
        }
        fx["steps"].append(rec)
    fx["names"] = [k for k, _ in ae.named_parameters()]
    torch.save(fx, os.path.join(ROOT, "tests", "golden", name))
    print(name, "loss_rec", float(fx["steps"][0]["loss_rec"]), "loss_kl", float(fx["steps"][0]["loss_kl"]),
          "gnorm", float(fx["steps"][0]["grad_norm"]))


def make_infer_fixture(ref_model, c_in, batch, T, T_cond, name):
    import oracle.ae_oracle as orc
    config = orc.default_config(c_in)
    sd = orc.init_state(config, seed=0)
    ae = ref_model.AE(config)
    ae.load_state_dict(sd, strict=True)
    x = randn((batch, c_in, T), seed=3)
    xc = randn((batch, c_in, T_cond), seed=4)
    with torch.no_grad():
        dec = ae.inference(x, xc)
        emb = ae.get_speaker_embeddings(xc)
    torch.save({"c_in": c_in, "x": x, "x_cond": xc, "dec": dec, "emb": emb},
               os.path.join(ROOT, "tests", "golden", name))
    print(name, tuple(dec.shape))


def make_reference_forward_fixture(ref_model, name):
    """One forward pass of the reference AE, recorded with the seeds of train_c80_b1.pt's first step, so that
    the suite can check that fixture and the oracle against the reference without the reference itself."""
    import oracle.ae_oracle as orc
    config = orc.default_config(80)
    x = randn((1, 80, 128), seed=1)
    with torch.no_grad():
        _, mu, ls, emb, dec = run_ae(ref_model, config, orc.init_state(config, seed=0), x, eps_seed=100)
    torch.save({"x": x, "eps_seed": 100, "mu": mu, "log_sigma": ls, "emb": emb, "dec": dec},
               os.path.join(ROOT, "tests", "golden", name))
    print(name, tuple(dec.shape))


def make_helper_fixture(ref_model, name):
    """Known answers for the small helpers of model.py:21-32, 52-63, 77-83."""
    x = randn((2, 8, 11), seed=5)
    fx = {"x": x}
    for k in (1, 2, 5, 8):
        conv = torch.nn.Conv1d(8, 4, kernel_size=k)
        g = torch.Generator().manual_seed(10 + k)
        with torch.no_grad():
            conv.weight.copy_(torch.randn(conv.weight.shape, generator=g))
            conv.bias.copy_(torch.randn(conv.bias.shape, generator=g))
        fx[f"pad_conv_k{k}"] = {"w": conv.weight.detach().clone(), "b": conv.bias.detach().clone(),
                                "y": ref_model.pad_layer(x, conv).detach().clone()}
    conv = torch.nn.Conv1d(8, 4, kernel_size=5, stride=2)
    fx["pad_conv_k5_s2"] = {"w": conv.weight.detach().clone(), "b": conv.bias.detach().clone(),
                            "y": ref_model.pad_layer(x, conv).detach().clone()}
    fx["pixel_shuffle"] = ref_model.pixel_shuffle_1d(x, 2)
    fx["upsample"] = ref_model.upsample(x, 2)
    cond = randn((2, 16), seed=6)
    fx["cond"] = cond
    fx["append_cond"] = ref_model.append_cond(x, cond)
    fx["instance_norm"] = torch.nn.InstanceNorm1d(8, affine=False)(x)
    fx["avg_pool_ceil"] = torch.nn.functional.avg_pool1d(x, kernel_size=2, ceil_mode=True)
    torch.save(fx, os.path.join(ROOT, "tests", "golden", name))
    print(name)


def main():
    ref_model = import_reference()
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)
    make_helper_fixture(ref_model, "helpers.pt")
    make_train_fixture(ref_model, 80, 1, 128, 1, "train_c80_b1.pt")      # BASELINE config 1
    make_train_fixture(ref_model, 80, 4, 128, 3, "train_c80_b4.pt")      # 3 Adam steps
    make_train_fixture(ref_model, 512, 2, 128, 1, "train_c512_b2.pt")    # shipped config.yaml
    make_infer_fixture(ref_model, 80, 2, 301, 173, "infer_c80.pt")       # odd lengths, T_cond != T
    make_infer_fixture(ref_model, 80, 1, 512, 512, "infer_c80_t512.pt")  # BASELINE config 5 shape
    make_reference_forward_fixture(ref_model, "reference_fwd_c80_b1.pt")


if __name__ == "__main__":
    main()
