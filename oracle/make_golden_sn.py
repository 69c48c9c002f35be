"""Generate the spectral-norm fixtures (tests/golden/*_sn_*.pt) by running the UNMODIFIED reference with
``Decoder.sn: True``.

TEST INFRASTRUCTURE, like oracle/make_golden.py (whose stand-ins for the reference's unused imports it
reuses); the fixtures it writes are committed.  Usage:

    python oracle/make_golden_sn.py            # writes tests/golden/{train_c80_sn_b4,train_c512_sn_b2,infer_c80_sn}.pt

The initial state comes from ``oracle.sn_oracle.init_state`` and is loaded into the reference ``AE`` with
``load_state_dict(strict=True)``, which also proves the inventory (166 parameters + 52 buffers).  sigma of
a layer is read back as the reference's hook computes it, ``dot(u, mv(weight_orig, v))`` from the
buffers it has just updated.
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.make_golden import import_reference, randn, reference_eps  # noqa: E402

# Kept under 1 MB each: eps is not stored (reference_eps(eps_shape, eps_seed) regenerates it bit for bit, as x
# is regenerated from x_seed); the gradients below are stored for the first step only, and only those of at most
# SN_GRAD_MAX elements (every tensor's gradient L2 is stored for every step); steps after the first keep the outputs of
# the first sample only (they are compared loosely anyway: Adam drift).
SN_GRAD_MAX = 16384
SN_GRADS = [
    "decoder.in_conv_layer.bias", "decoder.second_conv_layers.0.bias", "decoder.conv_affine_layers.11.bias",
    "decoder.out_conv_layer.weight_orig", "decoder.out_conv_layer.bias", "content_encoder.std_layer.bias",
    "speaker_encoder.output_layer.bias",
]


def sigmas(ae, layers):
    mods = dict(ae.named_modules())
    out = []
    with torch.no_grad():
        for n in layers:
            m = mods[n]
            w = m.weight_orig
            out.append(torch.dot(m.weight_u, torch.mv(w.reshape(w.shape[0], -1), m.weight_v)))
    return torch.stack(out)


def uv(ae, layers):
    mods = dict(ae.named_modules())
    return {n: (mods[n].weight_u.detach().clone(), mods[n].weight_v.detach().clone()) for n in layers}


def inventory(ae):
    sd = ae.state_dict()
    meta = {k: dict(v) for k, v in sd._metadata.items() if k.startswith("decoder")}
    return {"names": [k for k, _ in ae.named_parameters()],
            "state_keys": [(k, tuple(v.shape)) for k, v in sd.items()],
            "metadata": meta}


def make_train_fixture(ref_model, c_in, batch, T, n_steps, name):
    import oracle.sn_oracle as sno
    config = sno.sn_config(c_in)
    layers = sno.sn_layers(config)
    sd = sno.init_state(config, seed=0)
    x = randn((batch, c_in, T), seed=1)
    ae = ref_model.AE(config)
    ae.load_state_dict(sd, strict=True)
    ae.train()
    o = config["optimizer"]
    opt = torch.optim.Adam(ae.parameters(), lr=o["lr"], betas=(o["beta1"], o["beta2"]),
                           amsgrad=o["amsgrad"], weight_decay=o["weight_decay"])
    # x is not stored (it is as large as dec): randn(shape, seed=x_seed) regenerates it bit for bit
    fx = {"c_in": c_in, "x_shape": tuple(x.shape), "x_seed": 1, "lambda_kl": 0.37, "steps": [], "uv": {}, **inventory(ae)}
    for step in range(n_steps):
        eps_seed = 100 + step
        torch.manual_seed(eps_seed)
        mu, ls, emb, dec = ae(x)      # the power iteration runs here, once
        sig = sigmas(ae, layers)
        loss_rec = torch.nn.L1Loss()(dec, x)
        loss_kl = 0.5 * torch.mean(torch.exp(ls) + mu ** 2 - 1 - ls)
        loss = config["lambda"]["lambda_rec"] * loss_rec + fx["lambda_kl"] * loss_kl
        opt.zero_grad()
        loss.backward()
        grads = {k: (p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p))
                 for k, p in ae.named_parameters()}
        gnorm = torch.nn.utils.clip_grad_norm_(ae.parameters(), max_norm=o["grad_norm"])
        opt.step()
        keep = slice(None) if step == 0 else slice(0, 1)
        rec = {
            "eps_shape": tuple(ls.shape), "eps_seed": eps_seed,
            "mu": mu.detach()[keep].clone(), "log_sigma": ls.detach()[keep].clone(),
            "emb": emb.detach()[keep].clone(), "dec": dec.detach()[keep].clone(),
            "loss_rec": loss_rec.detach().clone(), "loss_kl": loss_kl.detach().clone(),
            "grad_norm": torch.as_tensor(float(gnorm)),
            "grad_l2": torch.stack([grads[k].norm() for k in grads]),
            "param_l2_after": torch.stack([p.detach().norm() for p in ae.parameters()]),
            "sigma": sig,
        }
        if step == 0:
            rec["grad_small"] = {k: grads[k] for k in SN_GRADS if grads[k].numel() <= SN_GRAD_MAX}
        fx["steps"].append(rec)
        if step in (0, n_steps - 1):
            fx["uv"][step + 1] = uv(ae, layers)
    torch.save(fx, os.path.join(ROOT, "tests", "golden", name))
    print(name, "loss_rec", float(fx["steps"][0]["loss_rec"]), "gnorm", float(fx["steps"][0]["grad_norm"]),
          "sigma[0]", float(fx["steps"][0]["sigma"][0]))


def make_infer_fixture(ref_model, c_in, batch, T, T_cond, name):
    import oracle.sn_oracle as sno
    config = sno.sn_config(c_in)
    ae = ref_model.AE(config)
    ae.load_state_dict(sno.init_state(config, seed=0), strict=True)
    ae.eval()
    x = randn((batch, c_in, T), seed=3)
    xc = randn((batch, c_in, T_cond), seed=4)
    with torch.no_grad():
        dec = ae.inference(x, xc)
    torch.save({"c_in": c_in, "x": x, "x_cond": xc, "dec": dec, "sigma": sigmas(ae, sno.sn_layers(config))},
               os.path.join(ROOT, "tests", "golden", name))
    print(name, tuple(dec.shape))


def main():
    ref_model = import_reference()
    torch.set_num_threads(os.cpu_count() or 1)
    make_train_fixture(ref_model, 80, 4, 128, 3, "train_c80_sn_b4.pt")
    make_train_fixture(ref_model, 512, 2, 128, 1, "train_c512_sn_b2.pt")
    make_infer_fixture(ref_model, 80, 2, 301, 173, "infer_c80_sn.pt")


if __name__ == "__main__":
    main()
