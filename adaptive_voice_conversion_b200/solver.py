"""Solver with the reference's surface (solver.py:16-118): ``Solver(config, args)``,
``train(n)``, ``ae_step(data, lambda_kl) -> {'loss_rec','loss_kl','grad_norm'}``,
``save_model`` / ``load_model`` / ``save_config`` / ``build_model`` / ``get_data_loaders``.

What changed underneath: the model is the B200-native ``AE``; one optimizer step is
``FusedTrainer.step`` (hand-written forward+backward kernels, a single NCCL all-reduce of
the flat gradient when launched with torchrun, fused clip+Adam(amsgrad)); checkpoints stay
``<path>.ckpt`` (model state_dict) + ``<path>.opt`` (torch.optim.Adam state_dict format),
written by rank 0 only.  ``args.data_dir == 'synthetic'`` trains on N(0,1) segments.
"""
from __future__ import annotations

import json
import os

import torch
import yaml

from .data_utils import PickleDataset, SyntheticSegments, get_data_loader
from .model import AE
from .optim import FusedAdam
from .trainer import FusedTrainer
from .utils import Logger, cc, infinite_iter, local_device


def _dist_info():
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        return torch.distributed.get_rank(), torch.distributed.get_world_size()
    return 0, 1


class Solver(object):
    def __init__(self, config, args):
        self.config = config
        self.args = args
        self.rank, self.world = _dist_info()
        if self.rank == 0:
            print(config)
            print(args)
        self.logger = Logger(getattr(args, "logdir", "log/")) if self.rank == 0 else None
        self.iteration = 0   # optimizer steps done so far (checkpointed: the KL-annealing position survives a resume)
        self.get_data_loaders()
        self.build_model()
        if self.rank == 0 and getattr(args, "store_model_path", None):
            self.save_config()
        if getattr(args, "load_model", False):
            self.load_model()

    # ---- checkpoints (solver.py:39-55)
    def save_model(self, iteration):
        """<path>.ckpt / <path>.opt exactly as the reference writes them (solver.py:39-43) plus <path>.iter:
        the number of steps done.  The reference drops `iteration`, so a resumed run restarts its KL
        annealing from zero (solver.py:100-104); here load_model restores it."""
        if self.rank != 0:
            return
        torch.save(self.model.state_dict(), f"{self.args.store_model_path}.ckpt")
        torch.save(self.opt.state_dict(), f"{self.args.store_model_path}.opt")
        with open(f"{self.args.store_model_path}.iter", "w") as f:
            json.dump({"iteration": int(iteration) + 1}, f)

    def save_config(self):
        with open(f"{self.args.store_model_path}.config.yaml", "w") as f:
            yaml.dump(self.config, f)
        with open(f"{self.args.store_model_path}.args.yaml", "w") as f:
            yaml.dump(vars(self.args), f)

    def load_model(self):
        if self.rank == 0:
            print(f"Load model from {self.args.load_model_path}")
        dev = local_device()
        self.model.load_state_dict(torch.load(f"{self.args.load_model_path}.ckpt", map_location=dev))
        opt_path = f"{self.args.load_model_path}.opt"
        if os.path.exists(opt_path):
            self.opt.load_state_dict(torch.load(opt_path, map_location=dev))
        it_path = f"{self.args.load_model_path}.iter"
        if os.path.exists(it_path):    # absent for checkpoints written by the reference: start at 0 like it does
            with open(it_path) as f:
                self.iteration = int(json.load(f)["iteration"])
        self.trainer.eng.pack_weights(self.trainer.P, need_dgrad=True)

    # ---- data (solver.py:57-68)
    def get_data_loaders(self):
        dl = self.config["data_loader"]
        data_dir = getattr(self.args, "data_dir", "synthetic")
        if data_dir in (None, "synthetic"):
            n_mels = self.config["ContentEncoder"]["c_in"] // dl["frame_size"]
            self.train_dataset = None
            self.train_loader = SyntheticSegments(dl["batch_size"], n_mels * dl["frame_size"], dl["segment_size"] // dl["frame_size"],
                                                  seed=1 + self.rank)
        else:
            self.train_dataset = PickleDataset(os.path.join(data_dir, f"{self.args.train_set}.pkl"),
                                               os.path.join(data_dir, self.args.train_index_file),
                                               segment_size=dl["segment_size"])
            self.train_loader = get_data_loader(self.train_dataset, frame_size=dl["frame_size"], batch_size=dl["batch_size"],
                                                shuffle=dl["shuffle"], num_workers=4, drop_last=False)
        self.train_iter = infinite_iter(self.train_loader)

    # ---- model + optimizer (solver.py:70-79)
    def build_model(self):
        self.model = cc(AE(self.config))
        if self.world > 1:  # replicas start identical: broadcast rank 0's init (and the spectral-norm u, v buffers)
            for t in list(self.model.parameters()) + list(self.model.buffers()):
                torch.distributed.broadcast(t.data, src=0)
        self.model.flatten_parameters()
        o = self.config["optimizer"]
        self.opt = FusedAdam(self.model, lr=o["lr"], betas=(o["beta1"], o["beta2"]), amsgrad=o["amsgrad"],
                             weight_decay=o["weight_decay"], max_norm=o["grad_norm"], world_size=self.world)
        self.trainer = FusedTrainer(self.model, self.opt, self.config)
        if self.rank == 0:
            print(self.model)
            print(self.opt)

    # ---- one step (solver.py:81-97)
    def ae_step(self, data, lambda_kl, eps=None):
        x = data.to(local_device(), non_blocking=True)
        self.trainer.step(x, lambda_kl, eps=eps)
        loss_rec, loss_kl, grad_norm = self.trainer.losses()
        return {"loss_rec": loss_rec, "loss_kl": loss_kl, "grad_norm": grad_norm}

    # ---- the training loop's data path (replaces the reference's per-step `.to(device)` + `.item()` stalls,
    # solver.py:82-97): the host-to-device copy of batch i+1 runs on a copy stream while step i computes, and
    # step i's losses are read (16 bytes, pinned) only after step i+1 has been enqueued, so the GPU never waits
    # for the host.  Every step still copies its own batch and reports its own losses.  AVC_PIPELINE=0 selects
    # the plain loop (ae_step per batch).
    def _prefetch(self, batch):
        dev = local_device()
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(dev)
        with torch.cuda.stream(self._copy_stream):
            x = batch.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
        return x, ev

    def run_steps(self, n_iterations, lambda_of=None, on_step=None):
        """n optimizer steps on the training iterator; returns the last step's losses.
        lambda_of(iteration) -> lambda_kl (default: the configured constant); on_step(iteration, meta,
        lambda_kl) is called for every step (one step late when pipelined).  `iteration` counts from
        self.iteration (0, or the checkpointed position after load_model)."""
        lam0 = self.config["lambda"]["lambda_kl"]
        pipelined = os.environ.get("AVC_PIPELINE", "1") == "1"
        meta = None
        if not pipelined:
            for iteration in range(self.iteration, self.iteration + n_iterations):
                lambda_kl = lam0 if lambda_of is None else lambda_of(iteration)
                meta = self.ae_step(next(self.train_iter), lambda_kl)
                self.iteration = iteration + 1
                if on_step is not None:
                    on_step(iteration, meta, lambda_kl)
            return meta

        def finish(p):
            it_, lam_, get = p
            loss_rec, loss_kl, grad_norm = get()
            m = {"loss_rec": loss_rec, "loss_kl": loss_kl, "grad_norm": grad_norm}
            self.iteration = it_ + 1
            if on_step is not None:
                on_step(it_, m, lam_)
            return m

        start, end = self.iteration, self.iteration + n_iterations
        nxt = self._prefetch(next(self.train_iter)) if n_iterations > 0 else None
        pending = None
        for iteration in range(start, end):
            lambda_kl = lam0 if lambda_of is None else lambda_of(iteration)
            x, ev = nxt
            cur = torch.cuda.current_stream(x.device)
            cur.wait_event(ev)
            x.record_stream(cur)
            self.trainer.step(x, lambda_kl)
            get = self.trainer.losses_async()
            if iteration + 1 < end:
                nxt = self._prefetch(next(self.train_iter))     # overlaps with this step
            if pending is not None:
                meta = finish(pending)                          # step i-1's losses, read while step i runs
            pending = (iteration, lambda_kl, get)
        if pending is not None:
            meta = finish(pending)
        return meta

    # ---- loop (solver.py:99-118)
    def train(self, n_iterations):
        lam = self.config["lambda"]["lambda_kl"]
        anneal = self.config["annealing_iters"]
        last = self.iteration + n_iterations

        def on_step(iteration, meta, lambda_kl):
            if self.rank != 0:
                return
            if iteration % self.args.summary_steps == 0:
                self.logger.scalars_summary(f"{self.args.tag}/ae_train", meta, iteration)
            print(f"AE:[{iteration + 1}/{last}], loss_rec={meta['loss_rec']:.2f}, "
                  f"loss_kl={meta['loss_kl']:.2f}, lambda={lambda_kl:.1e}     ", end="\r")
            if (iteration + 1) % self.args.save_steps == 0 or iteration + 1 == last:
                self.save_model(iteration=iteration)
                print()

        self.run_steps(n_iterations, lambda_of=lambda it: lam if it >= anneal else lam * (it + 1) / anneal, on_step=on_step)
