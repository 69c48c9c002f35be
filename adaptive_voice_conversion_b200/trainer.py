"""The fused training step: forward, losses, hand-written backward, gradient all-reduce,
clip + Adam -- the body of ``Solver.ae_step`` (solver.py:81-97) without autograd.

Data parallelism (SURVEY.md section 8e): one process per GPU, parameters and Adam state
replicated, each rank steps on its own segments, ONE NCCL all-reduce(SUM) of the flat
gradient buffer per iteration; the 1/world scale is folded into the clip/Adam kernel so
the order backward -> all-reduce -> global-norm clip -> Adam matches a single-process
step on the concatenated batch.

The speaker encoder and the content encoder are independent until the decoder (model.py:381-385), and so
are their backward passes after it: ``_fwd_bwd`` runs the speaker branch on a second stream (fork / join with
events, also inside the captured graph), so the two chains of ~100 dependent launches each fill each other's
launch-boundary bubbles and the SMs the small-T layers leave idle (AVC_OVERLAP=0: one stream).

``capture()`` records the step once into CUDA graphs (static shapes) and ``step()`` replays
them: one graph for the whole step in a single process; with N > 1 graph A = zero-grad +
forward + loss + backward, graph B = norm + Adam + weight re-pack, and the all-reduce runs
between them.
"""
from __future__ import annotations

import os
from typing import Dict, Optional

import torch

from . import _lib as L
from .engine import A4, Engine
from .optim import FusedAdam


class FusedTrainer:
    def __init__(self, model, opt: FusedAdam, config: dict, process_group=None):
        self.model, self.opt, self.cfg = model, opt, config
        self.dev = opt.flat_p.device
        self.eng: Engine = model.engine(self.dev)
        self.lib = L.load()
        self.P: Dict[str, torch.Tensor] = dict(model.named_parameters())
        self.G: Dict[str, torch.Tensor] = opt.named_grad_views(model)
        if model.sn:   # the kernels read W/sigma and write its gradient into the weight_orig slots (model.AE.sn_views)
            self.P, self.G = model.sn_views(self.P, self.G)
        self.pg = process_group
        self.world = opt.world_size
        # one 16-byte report block so that reading a step's scalars is ONE device->host copy:
        # [sum|dec-x|, sum KL terms, sum g^2, tcgen05 status word]
        self.report = torch.zeros(4, dtype=torch.float32, device=self.dev)
        self.sums = self.report[0:2]
        opt.sqnorm = self.report[2:3]
        self.eng.tc_status = self.report[3:4].view(torch.int32)
        self.n_rec = 1
        self.n_lat = 1
        self._graphs = None
        self._graph_training = None   # the model.training a captured graph was recorded for (the power iteration runs only in training)
        self._static = None
        # the third consecutive step on the same batch shape (no injected eps) is recorded into CUDA graphs and every
        # later one replays them: a plain `Solver.train` loop gets the graph path without calling capture() (AVC_GRAPH=0: eager)
        self.auto_graph = os.environ.get("AVC_GRAPH", "1") == "1"
        self._eager_shape, self._eager_n = None, 0
        self.launches_per_step = 0
        self.eng.pack_weights(self.P, need_dgrad=True)
        self.eng.prepare_tables(self.P, self.G)   # before any CUDA-graph capture
        self.eng.prepare_wgrad_acc(self.P, self.G)
        self.overlap = os.environ.get("AVC_OVERLAP", "1") == "1"
        # Conv weight gradients are leaves of the backward pass: they can fork onto their own (lower-priority) stream
        # while the dgrad / norm-backward chain continues.  Measured (B=256): forking the DECODER's weight gradients
        # only -- the phase in which ONE chain is active and SMs idle -- 60.1k -> 62.4k seg/s (AVC_WGRAD_STREAM=2,
        # default); forking all of them 60.6k (=1): during the encoders' backward two chains are already active, and a
        # weight-gradient kernel holds 128 SMs for ~20 us (one ~190 KB CTA per SM, like the conv kernel), so whenever it
        # grabs them inside a bubble the next critical-path conv waits for it; =0: all in line.  The chains are captured
        # on high-priority streams, the weight gradients on a normal-priority one.
        self._wg_mode = os.environ.get("AVC_WGRAD_STREAM", "2")   # "1": every conv weight gradient, "2": the decoder's only
        wg = self._wg_mode in ("1", "2") and self.overlap
        self._side = torch.cuda.Stream(self.dev, priority=-1 if wg else 0) if self.overlap else None
        self._wgs = torch.cuda.Stream(self.dev, priority=0) if wg else None
        self._cap = torch.cuda.Stream(self.dev, priority=-1) if wg else None   # capture stream of the graphs
        self._lambda_kl = None
        self._hp_key = None
        self._static_eps = None
        self._host_ring = None
        opt.sync_hparams(lambda_rec=float(config["lambda"]["lambda_rec"]), lambda_kl=float(config["lambda"]["lambda_kl"]))

    # ------------------------------------------------------------------ pieces
    def _fwd_bwd(self, x: torch.Tensor, eps: Optional[torch.Tensor]):
        eng, P, G = self.eng, self.P, self.G
        main, side = torch.cuda.current_stream(self.dev), self._side
        self.opt.zero_grad()
        if self.model.sn:
            # W/sigma (+ the power iteration in training mode) before any decoder kernel, then the step's one re-pack of
            # the whole model (with sn it moves here from the end of the previous step, _update: a separate decoder
            # pack would bump the pack version and make the lazily packed stride-2 encoder layers re-pack every step)
            self.model.spectral_norm_fwd(self.dev, update=self.model.training)
            eng.pack_weights(P, need_dgrad=True)
        # ---- forward: speaker branch || content branch (both only read x), joined in front of the decoder
        if side is not None:
            side.wait_stream(main)
            with torch.cuda.stream(side):
                emb, cs = eng.speaker_fwd(P, x, True)
                aff = eng.decoder_affine_fwd(P, emb, True)   # the AdaIN rows need the speaker embedding only
        else:
            emb, cs = eng.speaker_fwd(P, x, True)
            aff = None
        mu4, ls4, ce = eng.content_fwd(P, x, True)
        if eps is None:
            eps = torch.randn((mu4.B, mu4.C, mu4.T), dtype=torch.float32, device=self.dev)
        mu, ls, z4 = eng.reparam_fwd(mu4, ls4, eps)
        if side is not None:
            main.wait_stream(side)
        dec4, cd = eng.decoder_fwd(P, z4, emb, True, affine=aff)
        dec = eng.unpack_a4(dec4)
        ddec, dmu, dls = torch.empty_like(dec), torch.empty_like(mu), torch.empty_like(ls)
        self.n_rec, self.n_lat = dec.numel(), mu.numel()
        L.check(self.lib.avc_vae_loss(dec.data_ptr(), x.data_ptr(), dec.numel(), mu.data_ptr(), ls.data_ptr(), mu.numel(),
                                      self.opt.hp.data_ptr(), self.sums.data_ptr(), ddec.data_ptr(), dmu.data_ptr(),
                                      dls.data_ptr(), eng.stream), "vae_loss")
        ddec4 = A4.empty(dec4.B, dec4.C, dec4.T, self.dev)
        eng.pack_a4(ddec, ddec4)
        eng.wgrad_stream = self._wgs
        try:
            return self._bwd(x, eps, mu, ls, emb, dec, ls4, dmu, dls, cs, ce, cd, ddec4)
        finally:
            eng.wgrad_stream = None
            eng._wg_keep.clear()

    def _bwd(self, x, eps, mu, ls, emb, dec, ls4, dmu, dls, cs, ce, cd, ddec4):
        eng, P, G = self.eng, self.P, self.G
        main, side = torch.cuda.current_stream(self.dev), self._side
        # the affine-layer gradients and demb fork onto the side stream after the decoder's block loop, beside its in_conv
        dz4, demb = eng.decoder_bwd(P, G, cd, ddec4, affine_stream=side)
        if self._wg_mode == "2":
            eng.wgrad_stream = None      # only the decoder's weight gradients fork (one chain active: idle SMs to fill)
            if self._wgs is not None:
                with torch.cuda.stream(self._wgs):
                    eng.flush_wgrad(decoder_only=True)   # ... and are folded into the gradient buffer there, behind them
        # ---- backward: the two encoders again in parallel (disjoint parameters, disjoint gradient buffers); the speaker
        # branch follows demb on the side stream without waiting for the rest of the main chain
        if side is not None:
            with torch.cuda.stream(side):
                eng.speaker_bwd(P, G, cs, demb)
        dmu4, dls4 = eng.reparam_bwd(dz4, ls4, eps, dmu, dls)
        eng.content_bwd(P, G, ce, dmu4, dls4)
        if side is not None:
            main.wait_stream(side)
        else:
            eng.speaker_bwd(P, G, cs, demb)
        # (every tensor the side stream touched -- x, emb, demb, cs -- is a local that lives until this function
        # returns, i.e. until after the join: the caching allocator cannot hand its memory to the other stream early)
        eng.wgrad_stream = self._wgs
        eng.join_wgrad()    # the forked weight gradients (of both branches) before their accumulators are flushed
        eng.flush_wgrad()   # no-op unless weight gradients were accumulated in place (AVC_WGRAD_ACC=1)
        if self.model.sn:   # every decoder weight gradient is final here (flushes and both streams joined)
            self.model.spectral_norm_bwd(G)
        return mu, ls, emb, dec

    def _allreduce(self):
        if self.world > 1:
            torch.distributed.all_reduce(self.opt.flat_g, op=torch.distributed.ReduceOp.SUM, group=self.pg)

    def _update(self):
        self.opt.step()
        if not self.model.sn:    # with sn the next step packs, from W/sigma (_fwd_bwd)
            self.eng.pack_weights(self.P, need_dgrad=True)

    def set_lambda_kl(self, lambda_kl: float):
        """Push lambda_kl and the optimizer's param_group hyper-parameters (an lr scheduler may have changed
        them) to the device vector the kernels read -- only when something changed."""
        g = self.opt.param_groups[0]
        key = (float(lambda_kl), g["lr"], tuple(g["betas"]), g["eps"], g["weight_decay"], bool(g["amsgrad"]))
        if key != self._hp_key:
            self._hp_key = key
            self._lambda_kl = lambda_kl
            self.opt.sync_hparams(lambda_kl=float(lambda_kl))

    # ------------------------------------------------------------------ public
    def step(self, x: torch.Tensor, lambda_kl: float, eps: Optional[torch.Tensor] = None, return_outputs=False):
        """One optimizer step on device batch x [B, c_in, T].  Enqueues work only; read
        ``losses()`` to synchronise."""
        if not x.is_cuda or x.dtype != torch.float32:
            raise L.AvcError("FusedTrainer.step: x must be a float32 CUDA tensor")
        x = x.contiguous()
        self.set_lambda_kl(lambda_kl)
        if self._graphs is not None and self._graph_training != self.model.training:
            self._graphs = None      # recorded for the other mode: record again
        replay = self._graphs is not None and tuple(x.shape) == tuple(self._static.shape) and not return_outputs
        if replay and (eps is None) == (self._static_eps is None):
            if x.data_ptr() != self._static.data_ptr():
                self._static.copy_(x, non_blocking=True)
            if eps is not None and eps.data_ptr() != self._static_eps.data_ptr():
                self._static_eps.copy_(eps, non_blocking=True)
            self._replay()
            return None
        if self.auto_graph and self._graphs is None and eps is None and not return_outputs:
            shp = tuple(x.shape)
            self._eager_n = self._eager_n + 1 if shp == self._eager_shape else 1
            self._eager_shape = shp
            if self._eager_n > 2:          # two eager steps of this shape are behind us (allocator, tables, packs warm)
                self.capture(x, warmup=0)  # records only; `_static` is a copy of x
                self._replay()             # ... and this is the step itself
                return None
        n0 = L.launch_count()
        outs = self._fwd_bwd(x, eps)
        self._allreduce()
        self._update()
        self.launches_per_step = L.launch_count() - n0
        return outs if return_outputs else None

    def _replay(self):
        self._graphs[0].replay()
        if self._graphs[1] is not None:   # N > 1: the NCCL all-reduce sits between the two graphs
            self._allreduce()
            self._graphs[1].replay()

    def capture(self, x_example: torch.Tensor, warmup: int = 2, eps_example: Optional[torch.Tensor] = None):
        """Capture the step for x_example's shape into CUDA graphs.  Runs `warmup` real
        (eager) steps first -- they DO update the parameters.  With eps_example the graph reads the
        reparameterisation noise from a static buffer that step(x, lambda_kl, eps=...) refills (parity
        tests inject eps); without it eps is drawn inside the graph from torch's device generator.
        (capture_error_mode="thread_local": a DataLoader's pin-memory thread may allocate pinned memory while this
        thread records.)"""
        lam = self._lambda_kl if self._lambda_kl is not None else float(self.cfg["lambda"]["lambda_kl"])
        self.eng.prepare_tables(self.P, self.G)
        self.eng.prepare_wgrad_acc(self.P, self.G)
        if self.model.sn:    # the spectral-norm item tables as well (host-to-device copies)
            self.model.sn_table(self.dev)
            self.model.sn_table(self.dev, self.G)
        self._graphs = None
        self._static = x_example.contiguous().clone()
        self._static_eps = None if eps_example is None else eps_example.contiguous().clone()
        for _ in range(warmup):
            self.step(self._static, lam, eps=self._static_eps)
        torch.cuda.synchronize(self.dev)
        self._graph_training = self.model.training
        ga = torch.cuda.CUDAGraph()
        pool = torch.cuda.graph_pool_handle()
        if self.world == 1:    # one process: the whole step (zero-grad .. weight re-pack) is ONE graph
            with torch.cuda.graph(ga, pool=pool, stream=self._cap, capture_error_mode="thread_local"):
                self._fwd_bwd(self._static, self._static_eps)
                self._update()
            self._graphs = (ga, None)
            return self._static
        gb = torch.cuda.CUDAGraph()
        with torch.cuda.graph(ga, pool=pool, stream=self._cap, capture_error_mode="thread_local"):
            self._fwd_bwd(self._static, self._static_eps)
        with torch.cuda.graph(gb, pool=pool, stream=self._cap, capture_error_mode="thread_local"):
            self._update()
        self._graphs = (ga, gb)
        return self._static

    def _decode_report(self, r):
        import struct
        status = struct.unpack("<i", struct.pack("<f", r[3]))[0]
        if status != 0:              # a tcgen05 pipeline barrier time-out must not go unnoticed
            raise L.AvcError(f"tcgen05 conv pipeline barrier timed out (code {status})")
        return r[0] / self.n_rec, 0.5 * r[1] / self.n_lat, (r[2] ** 0.5) / self.world

    def losses(self):
        """(loss_rec, loss_kl, grad_norm) as Python floats -- synchronises."""
        return self._decode_report(self.report.tolist())     # the only synchronisation of a step

    def losses_async(self):
        """Enqueue the 16-byte device->host read of this step's report block behind the step and return a
        handle; ``handle()`` waits for THAT copy only (not for work enqueued later) and returns
        (loss_rec, loss_kl, grad_norm).  Lets a training loop enqueue step i+1 before it reads step i."""
        if self._host_ring is None:
            self._host_ring = [torch.zeros(4, dtype=torch.float32).pin_memory() for _ in range(4)]
            self._ring_i = 0
        slot = self._host_ring[self._ring_i % len(self._host_ring)]
        self._ring_i += 1
        slot.copy_(self.report, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))

        def get():
            ev.synchronize()
            return self._decode_report(slot.tolist())
        return get
