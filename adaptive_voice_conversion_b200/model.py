"""Reference-shaped model API on top of the sm_100a kernels.

Drop-in for the reference's ``model.py`` classes used by its Solver / Inferencer
(model.py:209-395 of jjery2243542/adaptive_voice_conversion):

  * ``AE(config)`` with ``forward(x) -> (mu, log_sigma, emb, dec)``, ``inference(x, x_cond)``
    and ``get_speaker_embeddings(x)``;
  * identical constructor kwargs (the keys of config.yaml) and an identical ``state_dict``:
    166 fp32 tensors named ``speaker_encoder.conv_bank.0.weight`` ... with nn.Conv1d
    ``[Cout, Cin, k]`` / nn.Linear ``[out, in]`` shapes, so reference checkpoints load both
    ways.  nn.Conv1d / nn.Linear modules are kept purely as *parameter containers* (names,
    shapes, default init); their ``forward`` is never called.

The arithmetic runs in ``engine.Engine`` (hand-written CUDA through the C ABI); autograd
sees three custom Functions (speaker encoder, content encoder, reparam+decoder) whose
backward passes are hand-sequenced kernels as well.  There is no CPU path: calling the
model on CPU tensors raises.
"""
from __future__ import annotations

import os

from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import _lib as L
from .engine import A4, Engine


def _bank_kernel_sizes(bank_size: int, bank_scale: int) -> List[int]:
    return list(range(bank_scale, bank_size + 1, bank_scale))


class _ParamStack(nn.Module):
    """Base: a bag of nn.Conv1d / nn.Linear parameter holders registered under the
    reference's attribute names."""

    def _convs(self, attr: str, specs):
        setattr(self, attr, nn.ModuleList([nn.Conv1d(ci, co, kernel_size=k, stride=s) for (ci, co, k, s) in specs]))

    def _linears(self, attr: str, specs):
        setattr(self, attr, nn.ModuleList([nn.Linear(i, o) for (i, o) in specs]))

    def forward(self, *a, **k):  # pragma: no cover
        raise L.AvcError("sub-stacks are parameter containers; call AE.forward / AE.inference / AE.get_speaker_embeddings")


class SpeakerEncoder(_ParamStack):
    """Parameters of the reference SpeakerEncoder (model.py:209-235)."""

    def __init__(self, c_in, c_h, c_out, kernel_size, bank_size, bank_scale, c_bank, n_conv_blocks,
                 n_dense_blocks, subsample, act, dropout_rate):
        super().__init__()
        ks = _bank_kernel_sizes(bank_size, bank_scale)
        self._convs("conv_bank", [(c_in, c_bank, k, 1) for k in ks])
        self.in_conv_layer = nn.Conv1d(c_bank * len(ks) + c_in, c_h, kernel_size=1)
        self._convs("first_conv_layers", [(c_h, c_h, kernel_size, 1)] * n_conv_blocks)
        self._convs("second_conv_layers", [(c_h, c_h, kernel_size, s) for s, _ in zip(subsample, range(n_conv_blocks))])
        self._linears("first_dense_layers", [(c_h, c_h)] * n_dense_blocks)
        self._linears("second_dense_layers", [(c_h, c_h)] * n_dense_blocks)
        self.output_layer = nn.Linear(c_h, c_out)


class ContentEncoder(_ParamStack):
    """Parameters of the reference ContentEncoder (model.py:279-299)."""

    def __init__(self, c_in, c_h, c_out, kernel_size, bank_size, bank_scale, c_bank, n_conv_blocks, subsample,
                 act, dropout_rate):
        super().__init__()
        ks = _bank_kernel_sizes(bank_size, bank_scale)
        self._convs("conv_bank", [(c_in, c_bank, k, 1) for k in ks])
        self.in_conv_layer = nn.Conv1d(c_bank * len(ks) + c_in, c_h, kernel_size=1)
        self._convs("first_conv_layers", [(c_h, c_h, kernel_size, 1)] * n_conv_blocks)
        self._convs("second_conv_layers", [(c_h, c_h, kernel_size, s) for s, _ in zip(subsample, range(n_conv_blocks))])
        self.mean_layer = nn.Conv1d(c_h, c_out, kernel_size=1)
        self.std_layer = nn.Conv1d(c_h, c_out, kernel_size=1)


class Decoder(_ParamStack):
    """Parameters of the reference Decoder (model.py:325-345).  With ``sn`` every layer is registered through
    ``torch.nn.utils.spectral_norm`` like the reference's: parameters ``bias``, ``weight_orig`` and buffers
    ``weight_u``, ``weight_v`` per layer, and the ``spectral_norm`` state_dict metadata.  torch's forward hook
    never runs (the containers are not called) and the plain ``weight`` attribute it leaves behind is never
    read: the effective weights W/sigma are computed by ``AE`` (csrc/spectral_norm.cu)."""

    def __init__(self, c_in, c_cond, c_h, c_out, kernel_size, n_conv_blocks, upsample, act, sn, dropout_rate):
        super().__init__()
        f = nn.utils.spectral_norm if sn else (lambda m: m)
        self.in_conv_layer = f(nn.Conv1d(c_in, c_h, kernel_size=1))
        self.first_conv_layers = nn.ModuleList([f(nn.Conv1d(c_h, c_h, kernel_size=kernel_size)) for _ in range(n_conv_blocks)])
        self.second_conv_layers = nn.ModuleList([f(nn.Conv1d(c_h, c_h * up, kernel_size=kernel_size))
                                                 for _, up in zip(range(n_conv_blocks), upsample)])
        self.conv_affine_layers = nn.ModuleList([f(nn.Linear(c_cond, c_h * 2)) for _ in range(2 * n_conv_blocks)])
        self.out_conv_layer = f(nn.Conv1d(c_h, c_out, kernel_size=1))


def _check_input(x: torch.Tensor, what: str) -> torch.Tensor:
    if not x.is_cuda:
        raise L.AvcError(f"{what}: tensor is on {x.device}; this implementation has no CPU path (move it to a B200)")
    if x.dtype != torch.float32 or x.dim() != 3:
        raise L.AvcError(f"{what}: expected float32 [B, C, T], got {x.dtype} {tuple(x.shape)}")
    return x.contiguous()


class _StackFn(torch.autograd.Function):
    """Common plumbing: params arrive as *args so autograd tracks them; gradients are
    produced into one zeroed flat buffer and returned as views."""

    @staticmethod
    def _begin(ctx, model, prefix, params, train):
        names = model._names_by_prefix[prefix]
        P = dict(zip(names, params))
        eng = model.engine(params[0].device)
        if prefix == "decoder." and model.sn:
            model.spectral_norm_fwd(params[0].device, update=model.training)
            P, _ = model.sn_views(P)
        eng.pack_weights(P, need_dgrad=train, prefixes=(prefix,))
        ctx.model, ctx.prefix, ctx.P, ctx.train = model, prefix, P, train
        return eng, P

    @staticmethod
    def _grads(ctx, eng):
        names = ctx.model._names_by_prefix[ctx.prefix]
        sizes = [ctx.P[n].numel() for n in names]
        flat = eng.zeros(sum(sizes))
        G, off = {}, 0
        for n, s in zip(names, sizes):
            G[n] = flat[off:off + s].view(ctx.P[n].shape)
            off += s
        return G, names


class _SpeakerFn(_StackFn):
    @staticmethod
    def forward(ctx, model, x, *params):
        train = any(ctx.needs_input_grad)  # grad mode is off inside Function.forward
        eng, P = _StackFn._begin(ctx, model, "speaker_encoder.", params, train)
        emb, ctx.saved = eng.speaker_fwd(P, x, train)
        return emb

    @staticmethod
    def backward(ctx, demb):
        eng = ctx.model.engine(demb.device)
        G, names = _StackFn._grads(ctx, eng)
        eng.speaker_bwd(ctx.P, G, ctx.saved, demb.contiguous())
        ctx.saved = None
        return (None, None, *[G[n] for n in names])


class _ContentFn(_StackFn):
    @staticmethod
    def forward(ctx, model, x, *params):
        train = any(ctx.needs_input_grad)  # grad mode is off inside Function.forward
        eng, P = _StackFn._begin(ctx, model, "content_encoder.", params, train)
        mu4, ls4, ctx.saved = eng.content_fwd(P, x, train)
        mu, ls, _ = eng.reparam_fwd(mu4, ls4, None)
        ctx.ls4 = ls4 if train else None
        return mu, ls

    @staticmethod
    def backward(ctx, dmu, dls):
        eng = ctx.model.engine(dmu.device)
        G, names = _StackFn._grads(ctx, eng)
        dmu4, dls4 = eng.reparam_bwd(None, ctx.ls4, None, dmu.contiguous(), dls.contiguous())
        eng.content_bwd(ctx.P, G, ctx.saved, dmu4, dls4)
        ctx.saved = None
        return (None, None, *[G[n] for n in names])


class _DecoderFn(_StackFn):
    """z = mu + exp(log_sigma/2)*eps (model.py:383-384; eps None -> z = mu) then Decoder."""

    @staticmethod
    def forward(ctx, model, mu, log_sigma, eps, emb, *params):
        train = any(ctx.needs_input_grad)
        eng, P = _StackFn._begin(ctx, model, "decoder.", params, train)
        B, Cc, T = mu.shape
        mu4, ls4 = A4.empty(B, Cc, T, mu.device), A4.empty(B, Cc, T, mu.device)
        eng.pack_a4(mu.contiguous(), mu4)
        eng.pack_a4(log_sigma.contiguous(), ls4)
        eps = None if eps is None else eps.contiguous()
        _, _, z4 = eng.reparam_fwd(mu4, ls4, eps, want_planar=False)
        dec4, ctx.saved = eng.decoder_fwd(P, z4, emb.contiguous(), train)
        ctx.ls4, ctx.eps = (ls4, eps) if train else (None, None)
        return eng.unpack_a4(dec4)

    @staticmethod
    def backward(ctx, ddec):
        model = ctx.model
        eng = model.engine(ddec.device)
        G, names = _StackFn._grads(ctx, eng)
        B, Cc, T = ddec.shape
        ddec4 = A4.empty(B, Cc, T, ddec.device)
        eng.pack_a4(ddec.contiguous(), ddec4)
        if model.sn:
            _, Gk = model.sn_views(ctx.P, G)
            dz4, demb = eng.decoder_bwd(ctx.P, Gk, ctx.saved, ddec4)
            model.spectral_norm_bwd(Gk)
        else:
            dz4, demb = eng.decoder_bwd(ctx.P, G, ctx.saved, ddec4)
        dmu4, dls4 = eng.reparam_bwd(dz4, ctx.ls4, ctx.eps, None, None)
        dmu, dls = eng.unpack_a4(dmu4), eng.unpack_a4(dls4)
        ctx.saved = None
        return (None, dmu, dls, None, demb, *[G[n] for n in names])


class AE(nn.Module):
    """The auto-encoder of the reference (model.py:373-395), B200-native."""

    def __init__(self, config: dict):
        super().__init__()
        self.config = {k: dict(v) if isinstance(v, dict) else v for k, v in config.items()}
        self.speaker_encoder = SpeakerEncoder(**config["SpeakerEncoder"])
        self.content_encoder = ContentEncoder(**config["ContentEncoder"])
        self.decoder = Decoder(**config["Decoder"])
        self.sn = bool(config["Decoder"].get("sn", False))
        self._sn_dev: Dict[str, dict] = {}
        self._engines: Dict[str, Engine] = {}
        self._names_by_prefix = {}
        self._flat: Optional[torch.Tensor] = None
        self._index_names()

    # ---- parameter bookkeeping
    def _index_names(self):
        names = [n for n, _ in self.named_parameters()]
        for prefix in ("speaker_encoder.", "content_encoder.", "decoder."):
            self._names_by_prefix[prefix] = [n for n in names if n.startswith(prefix)]

    def _params(self, prefix: str):
        d = dict(self.named_parameters())
        return [d[n] for n in self._names_by_prefix[prefix]]

    def engine(self, device) -> Engine:
        key = str(torch.device(device))
        if key not in self._engines:
            self._engines[key] = Engine(self.config, torch.device(device))
        return self._engines[key]

    def flatten_parameters(self) -> torch.Tensor:
        """Re-home every parameter as a view of one flat fp32 buffer (registration order) so
        the optimizer and the gradient all-reduce are single launches over one buffer."""
        params = list(self.parameters())
        dev = params[0].device
        flat = torch.empty(sum(p.numel() for p in params), dtype=torch.float32, device=dev)
        off = 0
        for p in params:
            n = p.numel()
            flat[off:off + n].copy_(p.data.reshape(-1))
            p.data = flat[off:off + n].view(p.shape)
            off += n
        self._flat = flat
        return flat

    # ---- spectral normalisation of the decoder (sn: True)
    def sn_layers(self) -> List[str]:
        """The spectral-normalised layers ("decoder.in_conv_layer", ...) in registration order; [] without sn."""
        if not self.sn:
            return []
        return [n[:-len(".weight_orig")] for n, _ in self.named_parameters() if n.endswith(".weight_orig")]

    def _sn_state(self, device) -> dict:
        """Per device: one buffer holding every layer's effective weight W/sigma and the sigma vector.  Allocated once
        and never moved -- CUDA graphs and the engine's weight-pack tables hold their addresses."""
        key = str(torch.device(device))
        st = self._sn_dev.get(key)
        if st is None:
            params = dict(self.named_parameters())
            layers = self.sn_layers()
            shapes = [params[n + ".weight_orig"].shape for n in layers]
            w = torch.zeros(sum(s.numel() for s in shapes), dtype=torch.float32, device=device)
            views, off = {}, 0
            for n, shp in zip(layers, shapes):
                views[n] = w[off:off + shp.numel()].view(shp)
                off += shp.numel()
            st = self._sn_dev[key] = dict(w_sn=w, views=views, sigma=torch.zeros(len(layers), dtype=torch.float32, device=device),
                                          tables={})
        return st

    def sn_views(self, P: Dict[str, torch.Tensor], G: Optional[Dict[str, torch.Tensor]] = None):
        """The engine's view of the decoder's parameters: ``P["decoder.X.weight"]`` is the effective weight W/sigma
        and ``G["decoder.X.weight"]`` aliases the gradient slot of ``decoder.X.weight_orig``.  The kernels then
        write dL/d(W/sigma) there, which ``spectral_norm_bwd`` turns into dL/dweight_orig in place.  The other
        entries are passed through; returns new dicts (P, G)."""
        layers = self.sn_layers()
        st = self._sn_state(P[layers[0] + ".weight_orig"].device)
        P = dict(P, **{n + ".weight": st["views"][n] for n in layers})
        if G is not None:
            G = dict(G, **{n + ".weight": G[n + ".weight_orig"] for n in layers})
        return P, G

    def sigma(self, device) -> torch.Tensor:
        """The 26 sigmas of the last spectral-norm forward on `device` (sn_layers() order)."""
        return self._sn_state(device)["sigma"]

    def sn_table(self, device, G=None) -> torch.Tensor:
        """Device item table of avc_spectral_norm_fwd / _bwd (the gradient slots of G for the backward), cached
        until an address changes.  Building it is a host-to-device copy: a CUDA-graph capture needs it built
        before (FusedTrainer.capture does; Inferencer runs an eager call first)."""
        st = self._sn_state(device)
        params, bufs = dict(self.named_parameters()), dict(self.named_buffers())
        layers = self.sn_layers()
        rows = []
        for i, n in enumerate(layers):
            w = params[n + ".weight_orig"]
            rows.append((w.data_ptr(), st["views"][n].data_ptr(), bufs[n + ".weight_u"].data_ptr(), bufs[n + ".weight_v"].data_ptr(),
                         st["sigma"].data_ptr() + 4 * i, 0 if G is None else G[n + ".weight"].data_ptr(),
                         w.shape[0], w.numel() // w.shape[0]))
        key = tuple(rows)
        hit = st["tables"].get(G is None)
        if hit is None or hit[0] != key:
            items = (L.SnItem * len(rows))()
            for it, r in zip(items, rows):
                it.w_orig, it.w_sn, it.u, it.v, it.sigma, it.grad, it.rows, it.cols = r
            hit = st["tables"][G is None] = (key, torch.frombuffer(bytearray(bytes(items)), dtype=torch.uint8).to(device))
        return hit[1]

    def spectral_norm_fwd(self, device, update: bool):
        """W/sigma of every decoder layer into the effective-weight buffer (one launch).  update (module.training in
        the reference): one power iteration first, u and v overwritten; otherwise sigma from the stored u, v."""
        lib = L.load()
        st = torch.cuda.current_stream(device).cuda_stream
        L.check(lib.avc_spectral_norm_fwd(self.sn_table(device).data_ptr(), len(self.sn_layers()), int(bool(update)), st),
                "spectral_norm_fwd")

    def spectral_norm_bwd(self, G):
        """dL/d(W/sigma) -> dL/dweight_orig in place in G's slots (G as mapped by sn_views; one launch)."""
        lib = L.load()
        device = G[self.sn_layers()[0] + ".weight"].device
        st = torch.cuda.current_stream(device).cuda_stream
        L.check(lib.avc_spectral_norm_bwd(self.sn_table(device, G).data_ptr(), len(self.sn_layers()), st), "spectral_norm_bwd")

    # ---- the reference API
    def forward(self, x: torch.Tensor, *, eps: Optional[torch.Tensor] = None):
        """AE.forward (model.py:380-385).  ``eps`` (keyword-only extension) injects the
        N(0,1) draw for parity tests; by default it is drawn from the device generator."""
        x = _check_input(x, "AE.forward(x)")
        emb = _SpeakerFn.apply(self, x, *self._params("speaker_encoder."))
        mu, log_sigma = _ContentFn.apply(self, x, *self._params("content_encoder."))
        if eps is None:
            eps = torch.randn_like(log_sigma)
        dec = _DecoderFn.apply(self, mu, log_sigma, eps, emb, *self._params("decoder."))
        return mu, log_sigma, emb, dec

    def inference(self, x: torch.Tensor, x_cond: torch.Tensor):
        """AE.inference (model.py:387-391): content mean of x, speaker of x_cond."""
        x = _check_input(x, "AE.inference(x)")
        x_cond = _check_input(x_cond, "AE.inference(x_cond)")
        with torch.no_grad():
            side = self._side_stream(x.device)
            if side is None:
                emb = _SpeakerFn.apply(self, x_cond, *self._params("speaker_encoder."))
                mu, log_sigma = _ContentFn.apply(self, x, *self._params("content_encoder."))
                return _DecoderFn.apply(self, mu, log_sigma, None, emb, *self._params("decoder."))
            # the speaker encoder (on x_cond) and the content encoder (on x) are independent until the decoder: the
            # speaker branch runs on a second stream (fork / join), as in the fused train step (trainer.py)
            main = torch.cuda.current_stream(x.device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                emb = _SpeakerFn.apply(self, x_cond, *self._params("speaker_encoder."))
            mu, log_sigma = _ContentFn.apply(self, x, *self._params("content_encoder."))
            main.wait_stream(side)
            if not torch.cuda.is_current_stream_capturing():
                emb.record_stream(main)   # allocated on the side stream, read by the decoder on this one
            return _DecoderFn.apply(self, mu, log_sigma, None, emb, *self._params("decoder."))

    def _side_stream(self, dev):
        if os.environ.get("AVC_OVERLAP", "1") != "1":
            return None
        st = getattr(self, "_side_streams", None)
        if st is None:
            st = self._side_streams = {}
        if dev not in st:
            st[dev] = torch.cuda.Stream(dev)
        return st[dev]

    def get_speaker_embeddings(self, x: torch.Tensor):
        """AE.get_speaker_embeddings (model.py:393-395)."""
        x = _check_input(x, "AE.get_speaker_embeddings(x)")
        return _SpeakerFn.apply(self, x, *self._params("speaker_encoder."))
