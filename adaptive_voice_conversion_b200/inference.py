"""Inferencer with the reference's surface (inference.py:24-93).

The model call (``AE.inference``) is the B200 path.  The wav <-> mel DSP of the reference
(librosa STFT / Griffin-Lim in preprocess/tacotron/utils.py) is out of scope (SURVEY.md
section 2 rows 8, 12) and its dependencies are not in this image: ``inference_from_path``
uses a caller-supplied ``vocoder`` object with ``get_spectrograms(path)`` /
``melspectrogram2wav(mel)`` and raises a clear error without one.  ``inference_batch`` is
the batched entry point BASELINE config 5 measures.
"""
from __future__ import annotations

import os
import pickle

import torch
import torch.nn.functional as F

from .model import AE
from .utils import cc, local_device


class Inferencer(object):
    def __init__(self, config, args, vocoder=None):
        self.config = config
        self.args = args
        self.vocoder = vocoder
        self.build_model()
        if getattr(args, "model", None):
            self.load_model()
        self.attr = None
        if getattr(args, "attr", None):
            with open(args.attr, "rb") as f:
                self.attr = pickle.load(f)

    def load_model(self):
        print(f"Load model from {self.args.model}")
        self.model.load_state_dict(torch.load(f"{self.args.model}", map_location=local_device()))

    def build_model(self):
        self.model = cc(AE(self.config))
        self.model.eval()

    def utt_make_frames(self, x):
        """[T, n_mels] -> [1, n_mels*frame_size, T/frame_size] (inference.py:54-60)."""
        frame_size = self.config["data_loader"]["frame_size"]
        remains = x.size(0) % frame_size
        if remains != 0:
            x = F.pad(x, (0, remains))
        return x.view(1, x.size(0) // frame_size, frame_size * x.size(1)).transpose(1, 2).contiguous()

    def denormalize(self, x):
        return x * self.attr["std"] + self.attr["mean"]

    def normalize(self, x):
        return (x - self.attr["mean"]) / self.attr["std"]

    @torch.no_grad()
    def inference_batch(self, x, x_cond):
        """x [B, n_mels, T], x_cond [B, n_mels, T_c] device tensors -> dec [B, n_mels, 8*ceil(T/8)].

        One conversion is ~150 dependent kernel launches of a few microseconds each -- issued one by one from Python
        the GPU waits for the host.  The call is therefore captured ONCE per (shape, parameter version) into a CUDA
        graph (the speaker / content branches on two streams, model.AE.inference) and replayed on static input
        buffers; at most 8 shapes (serving buckets) are kept.  AVC_INFER_GRAPH=0: plain eager calls."""
        if os.environ.get("AVC_INFER_GRAPH", "1") != "1" or not x.is_cuda:
            return self.model.inference(x, x_cond)
        key = (tuple(x.shape), tuple(x_cond.shape), str(x.device), self._param_version())
        graphs = self.__dict__.setdefault("_graphs", {})
        g = graphs.get(key)
        if g is None:
            if len(graphs) >= 8:
                graphs.clear()
            sx, sc = x.contiguous().clone(), x_cond.contiguous().clone()
            self.model.inference(sx, sc)          # eager once: weight packs, allocator warm-up, argument checks
            torch.cuda.synchronize(x.device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                out = self.model.inference(sx, sc)
            g = graphs[key] = (graph, sx, sc, out)
        graph, sx, sc, out = g
        sx.copy_(x, non_blocking=True)
        sc.copy_(x_cond, non_blocking=True)
        graph.replay()
        return out.clone()

    def _param_version(self):
        # in-place updates (optimizer steps, load_state_dict) bump a tensor's version counter: a captured graph reads
        # the weight packs of the version it was captured with (and, with sn, the u / v buffers sigma is computed from)
        return sum(int(t._version) for t in list(self.model.parameters()) + list(self.model.buffers()))

    @torch.no_grad()
    def inference_ragged(self, xs, x_conds):
        """Batched one-shot conversion of utterance pairs of DIFFERENT lengths (the serving form of the loop around
        inference.py:62-70).  xs[i]: [T_i, n_mels], x_conds[i]: [Tc_i, n_mels] normalised mels on the device.
        Pairs are bucketed by their exact (T_i, Tc_i): every bucket is one batched AE.inference call, so each
        utterance gets bit-for-bit the result of converting it alone (InstanceNorm statistics are per sample and
        no padded frame ever enters them -- no masking needed).  Returns the list of [8*ceil(T_i/8), n_mels] mels
        in the input order (device tensors, normalised domain)."""
        if len(xs) != len(x_conds):
            raise ValueError("inference_ragged: xs and x_conds must have the same length")
        buckets = {}
        for i, (x, c) in enumerate(zip(xs, x_conds)):
            buckets.setdefault((int(x.shape[0]), int(c.shape[0])), []).append(i)
        out = [None] * len(xs)
        for (_, _), idx in sorted(buckets.items()):
            xb = torch.cat([self.utt_make_frames(xs[i]) for i in idx], dim=0)
            cb = torch.cat([self.utt_make_frames(x_conds[i]) for i in idx], dim=0)
            dec = self.inference_batch(xb, cb)               # [n, n_mels, 8*ceil(T/8)]
            for j, i in enumerate(idx):
                out[i] = dec[j].transpose(0, 1)
        self.model.engine(xs[0].device).check_tc_status()
        return out

    @torch.no_grad()
    def inference_one_utterance(self, x, x_cond):
        """x, x_cond: [T, n_mels] normalised mels on the device (inference.py:62-70)."""
        dec = self.model.inference(self.utt_make_frames(x), self.utt_make_frames(x_cond))
        dec = dec.transpose(1, 2).squeeze(0).detach().cpu().numpy()
        self.model.engine(x.device).check_tc_status()
        if self.attr is not None:
            dec = self.denormalize(dec)
        wav = self.vocoder.melspectrogram2wav(dec) if self.vocoder is not None else None
        return wav, dec

    def write_wav_to_file(self, wav_data, output_path):
        from scipy.io.wavfile import write
        write(output_path, rate=self.args.sample_rate, data=wav_data)

    def inference_from_path(self):
        if self.vocoder is None:
            raise RuntimeError("inference_from_path needs a vocoder with get_spectrograms/melspectrogram2wav "
                               "(the reference's librosa/Griffin-Lim DSP is outside this hot-path build)")
        src_mel, _ = self.vocoder.get_spectrograms(self.args.source)
        tar_mel, _ = self.vocoder.get_spectrograms(self.args.target)
        dev = local_device()
        src = torch.from_numpy(self.normalize(src_mel)).float().to(dev)
        tar = torch.from_numpy(self.normalize(tar_mel)).float().to(dev)
        wav, _ = self.inference_one_utterance(src, tar)
        self.write_wav_to_file(wav, self.args.output)
