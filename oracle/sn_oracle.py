"""CPU oracle of the spectral-normalised decoder (``Decoder.sn: True``) -- TEST INFRASTRUCTURE ONLY.

A restatement of what the reference gets from wrapping every decoder layer in
``torch.nn.utils.spectral_norm`` (model.py:334-344): dim=0, one power iteration per training
forward, eps=1e-12.  It builds on ``oracle.ae_oracle`` (whose functions are unchanged): the
spectral-normalised layers are turned into plain ``.weight`` entries W/sigma and handed to the
existing functional model, so autograd differentiates sigma while u and v stay constants.

State dicts here carry the reference's inventory: per decoder layer ``bias``, ``weight_orig``
(parameters, in that order) and the ``weight_u`` / ``weight_v`` buffers.
"""
from __future__ import annotations

from typing import Dict, List, Tuple

import torch
import torch.nn.functional as F

from . import ae_oracle as orc

Tensor = torch.Tensor
State = Dict[str, Tensor]

SN_EPS = 1e-12


def sn_config(c_in: int = 80) -> dict:
    cfg = orc.default_config(c_in)
    cfg["Decoder"]["sn"] = True
    return cfg


def sn_layers(config: dict) -> List[str]:
    """The 26 spectral-normalised layers in registration order (every decoder layer)."""
    return [n[:-len(".weight")] for n, _ in orc.param_shapes(config) if n.startswith("decoder.") and n.endswith(".weight")]


def param_shapes(config: dict) -> List[Tuple[str, tuple]]:
    """Parameters in registration order (= .opt layout): a spectral-normalised layer registers bias, then weight_orig."""
    out = []
    layers = set(sn_layers(config))
    shapes = orc.param_shapes(config)
    i = 0
    while i < len(shapes):
        name, shp = shapes[i]
        layer = name[:-len(".weight")] if name.endswith(".weight") else None
        if layer in layers:
            out.append(shapes[i + 1])                       # bias
            out.append((layer + ".weight_orig", shp))
            i += 2
        else:
            out.append((name, shp))
            i += 1
    return out


def state_shapes(config: dict) -> List[Tuple[str, tuple]]:
    """AE.state_dict() keys and shapes in order: per spectral-normalised layer bias, weight_orig, weight_u, weight_v."""
    out = []
    for name, shp in param_shapes(config):
        out.append((name, shp))
        if name.endswith(".weight_orig"):
            layer = name[:-len(".weight_orig")]
            rows = shp[0]
            cols = 1
            for s in shp[1:]:
                cols *= s
            out += [(layer + ".weight_u", (rows,)), (layer + ".weight_v", (cols,))]
    return out


def init_state(config: dict, seed: int = 0) -> State:
    """weight_orig takes the values ``ae_oracle.init_state`` gives weight (biases and the encoders likewise); u and v
    are normalised normals from a generator seeded with seed + 1000."""
    base = orc.init_state(config, seed)
    g = torch.Generator().manual_seed(seed + 1000)
    sd = {}
    for name, shp in state_shapes(config):
        if name.endswith(".weight_orig"):
            sd[name] = base[name[:-len("_orig")]]
        elif name.endswith((".weight_u", ".weight_v")):
            sd[name] = F.normalize(torch.randn(shp, generator=g), dim=0, eps=SN_EPS)
        else:
            sd[name] = base[name]
    return sd


def spectral_normalize(sd: State, config: dict, update: bool) -> Tuple[State, Tensor]:
    """torch's SpectralNorm.compute_weight for every decoder layer.  update (module.training): one power iteration,
    ``v = normalize(W^T u)``, ``u = normalize(W v)``, written into sd's weight_u / weight_v; then
    ``sigma = u . (W v)``.  Returns (the state with ``.weight`` = weight_orig / sigma for the spectral-normalised
    layers, the 26 sigmas).  sigma is differentiable in weight_orig; u and v are constants."""
    out = {k: v for k, v in sd.items() if not k.endswith((".weight_orig", ".weight_u", ".weight_v"))}
    sigmas = []
    for layer in sn_layers(config):
        w = sd[layer + ".weight_orig"]
        wm = w.reshape(w.shape[0], -1)
        u, v = sd[layer + ".weight_u"], sd[layer + ".weight_v"]
        if update:
            with torch.no_grad():
                v_new = F.normalize(torch.mv(wm.t(), u), dim=0, eps=SN_EPS)
                u_new = F.normalize(torch.mv(wm, v_new), dim=0, eps=SN_EPS)
                u.copy_(u_new)
                v.copy_(v_new)
        sigma = torch.dot(u.detach(), torch.mv(wm, v.detach()))
        out[layer + ".weight"] = w / sigma
        sigmas.append(sigma)
    return out, torch.stack(sigmas)


def ae_forward(sd: State, config: dict, x: Tensor, eps: Tensor, update: bool = True):
    """AE.forward in training mode (update=True) with the N(0,1) draw injected -> (mu, log_sigma, emb, dec, sigmas)."""
    eff, sig = spectral_normalize(sd, config, update)
    return (*orc.ae_forward(eff, config, x, eps), sig)


def ae_inference(sd: State, config: dict, x: Tensor, x_cond: Tensor, update: bool = False) -> Tuple[Tensor, Tensor]:
    """AE.inference (eval mode by default: sigma from the stored u, v) -> (dec, sigmas)."""
    eff, sig = spectral_normalize(sd, config, update)
    return orc.ae_inference(eff, config, x, x_cond), sig


def params_of(sd: State) -> State:
    """The parameters of a state (the buffers weight_u / weight_v dropped)."""
    return {k: v for k, v in sd.items() if not k.endswith((".weight_u", ".weight_v"))}


def ae_loss_and_grads(sd: State, config: dict, x: Tensor, eps: Tensor, lambda_kl: float, update: bool = True):
    """solver.py:83-90 with spectral norm: one power iteration (update; u, v of ``sd`` are overwritten), then the loss
    and d(loss)/d(param) for every parameter (weight_orig, not the buffers)."""
    leaves = {k: (v.detach().clone().requires_grad_(True) if k in params_of(sd) else v) for k, v in sd.items()}
    mu, log_sigma, emb, dec, sig = ae_forward(leaves, config, x, eps, update)
    loss_rec, loss_kl = orc.ae_losses(x, mu, log_sigma, dec)
    loss = config["lambda"]["lambda_rec"] * loss_rec + lambda_kl * loss_kl
    names = list(params_of(sd))
    grads = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
    gd = {k: (g if g is not None else torch.zeros_like(sd[k])) for k, g in zip(names, grads)}
    outs = dict(mu=mu.detach(), log_sigma=log_sigma.detach(), emb=emb.detach(), dec=dec.detach(),
                loss_rec=loss_rec.detach(), loss_kl=loss_kl.detach(), sigma=sig.detach())
    return outs, gd


def ae_train_step(sd: State, st: orc.AdamState, config: dict, x: Tensor, eps: Tensor, lambda_kl: float) -> dict:
    """Solver.ae_step with spectral norm on CPU: the power iteration at the start of the forward, then clip + Adam on
    the parameters.  Mutates sd (parameters and u / v) and st (an AdamState over ``params_of(sd)``)."""
    outs, grads = ae_loss_and_grads(sd, config, x, eps, lambda_kl, update=True)
    p = params_of(sd)
    gnorm = orc.clip_and_adam(p, grads, st, config["optimizer"])
    return {"loss_rec": float(outs["loss_rec"]), "loss_kl": float(outs["loss_kl"]), "grad_norm": gnorm,
            "outs": outs, "grads": grads}
