"""Host-side sequencing of the sm_100a kernels for the AdaIN-VC stacks.

This is the layer between the reference-shaped Python API (model.AE, solver.Solver) and
the C ABI (include/avc_b200.h).  It mirrors, launch by launch, what the reference's
SpeakerEncoder / ContentEncoder / Decoder ``forward`` methods do with torch.nn modules
(model.py:265-277, 301-323, 347-371) and what autograd does for them in
``loss.backward()`` (solver.py:90) -- but every arithmetic op is one of our kernels, and
the backward is written out by hand (no autograd inside).

Tensors inside the engine are "A4" activations ([B][C/4][T][4], see avc_b200.h); PyTorch
only provides device memory (torch.empty) and the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional

import torch

from . import _lib as L

IN_EPS = 1e-5


class A4:
    """A [B][C/4][T][4] fp32 activation, possibly a channel sub-range of a wider buffer."""
    __slots__ = ("t", "ptr", "B", "C", "T", "bstride", "tf32")

    def __init__(self, t, ptr, B, C, T, bstride, tf32=False):
        self.t, self.ptr, self.B, self.C, self.T, self.bstride = t, ptr, B, C, T, bstride
        self.tf32 = tf32   # every value is TF32-exact (written by a rounding producer)

    @staticmethod
    def empty(B, C, T, device):
        assert C % 4 == 0, f"A4 layout needs C % 4 == 0, got {C}"
        t = torch.empty((B, C // 4, T, 4), dtype=torch.float32, device=device)
        return A4(t, t.data_ptr(), B, C, T, C * T)

    def channels(self, c0, c1):
        assert c0 % 4 == 0 and c1 % 4 == 0
        return A4(self.t, self.ptr + (c0 // 4) * self.T * 16, self.B, c1 - c0, self.T, self.bstride, self.tf32)

    def to_planar(self):  # test/debug helper (torch ops, not on the product path)
        v = self.t if self.t.shape[1] * 4 == self.C else None
        assert v is not None, "to_planar only on whole tensors"
        return v.permute(0, 1, 3, 2).reshape(self.B, self.C, self.T).contiguous()


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def conv_geometry(K: int, stride: int, Tin: int):
    pl = K // 2
    pr = K // 2 - 1 if K % 2 == 0 else K // 2
    Tout = (Tin + pl + pr - K) // stride + 1
    return pl, pr, Tout


class Engine:
    """Launch sequencer for one AE configuration on one device."""

    def __init__(self, config: dict, device: torch.device):
        self.cfg = config
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise L.AvcError("adaptive_voice_conversion_b200 runs on CUDA (sm_100a) only; there is no CPU path")
        self.lib = L.load()
        self.packed: Dict[str, Dict[str, torch.Tensor]] = {}
        self.debug = None  # optional callback(name, stage, obj) for tools/diag_*.py
        # "tf32": conv blocks / data gradients on the tcgen05 tensor cores (TF32 inputs rounded
        # to nearest, fp32 accumulate); "fp32": the exact FFMA kernels.  AVC_PRECISION overrides.
        self.precision = os.environ.get("AVC_PRECISION", "tf32")
        if self.precision not in ("tf32", "fp32"):
            raise L.AvcError("AVC_PRECISION must be 'tf32' or 'fp32'")
        self.tc_status = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self._packed_key = None
        self._init_options()
        se, ce, de = config["SpeakerEncoder"], config["ContentEncoder"], config["Decoder"]
        for c in (se, ce):
            if c.get("act", "relu") != "relu" or c.get("dropout_rate", 0) != 0:
                raise L.AvcError("only act='relu', dropout_rate=0 (the reference config.yaml) are implemented")
        if de.get("act", "relu") != "relu" or de.get("dropout_rate", 0) != 0:
            raise L.AvcError("Decoder: only act='relu', dropout_rate=0 are implemented")
        for up in de["upsample"]:
            if up not in (1, 2):
                raise L.AvcError("Decoder.upsample entries must be 1 or 2")
        for c in (se, ce):
            for s in c["subsample"]:
                if s not in (1, 2):
                    raise L.AvcError("subsample entries must be 1 or 2")

    def _init_options(self):
        """Path switches (environment defaults, see README): every one can also be set on the instance."""
        # opt-in: the speaker dense stack as one kernel per direction and the 12 AdaIN affine layers
        # as one launch each (csrc/dense_fused.cu); off = one launch per nn.Linear
        self.fused_dense = os.environ.get("AVC_FUSED_DENSE", "1" if L.DEFAULT_FUSED_DENSE else "0") == "1"
        self._ptr_tables: Dict[tuple, tuple] = {}
        # opt-in: conv weight gradients accumulate in place (vector atomics) and are folded into the
        # nn.Conv1d gradients by ONE flush launch per backward pass; only on buffers registered with
        # prepare_wgrad_acc (the trainer's persistent flat gradient)
        self.wgrad_acc = os.environ.get("AVC_WGRAD_ACC", "1" if L.DEFAULT_WGRAD_ACC else "0") == "1"
        # opt-in: stride-1 data-gradient convs apply the reflect-padding / residual adjoint in their own
        # epilogue (AVC_F_FOLD) instead of a separate avc_fold_add_fwd pass
        self.fold_fused = os.environ.get("AVC_FOLD_FUSED", "1" if L.DEFAULT_FOLD_FUSED else "0") == "1"
        self._wg_acc = None
        self.wgrad_stream = None     # set by FusedTrainer around a step: weight gradients fork onto this stream
        self._wg_keep = []
        self.tc_conv_v2 = bool(self.lib.avc_get_option(b"tc_conv_v2"))
        # the data-gradient conv of a block also runs the upstream block's norm backward (AVC_F_NORMBWD); off = one
        # avc_norm_bwd launch per block
        self.norm_bwd_fused = os.environ.get("AVC_NORM_BWD_FUSED", "1" if L.DEFAULT_NORM_BWD_FUSED else "0") == "1"
        # diagnostic (tools/diag_tf32.py, tests/test_gpu_tf32_accuracy.py): forward conv blocks on the exact-fp32 FFMA
        # kernels while the backward stays on the tensor cores -- separates "TF32 forward flips ReLU masks" from
        # "TF32 backward kernels are inaccurate" in the gradient-parity numbers
        self.fwd_fp32 = os.environ.get("AVC_FWD_FP32", "0") == "1"

    # ------------------------------------------------------------------ utilities
    @property
    def stream(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def _ck(self, rc, what):
        if rc != 0:
            raise L.AvcError(f"{what}: rc={rc}: {L.last_error()}")

    def empty(self, *shape):
        return torch.empty(shape, dtype=torch.float32, device=self.dev)

    def check_tc_status(self):
        """Synchronises; raises if a tcgen05 pipeline barrier ever timed out."""
        code = int(self.tc_status.item())
        if code != 0:
            raise L.AvcError(f"tcgen05 conv pipeline barrier timed out (code {code})")

    def zeros(self, *shape):
        t = self.empty(*shape)
        self._ck(self.lib.avc_fill_zero(t.data_ptr(), t.numel() * 4, self.stream), "fill_zero")
        return t

    def _ptr_table(self, key, tensors) -> torch.Tensor:
        """Device-resident table of the tensors' addresses (int64), cached until one of them moves."""
        ptrs = tuple(t.data_ptr() for t in tensors)
        hit = self._ptr_tables.get(key)
        if hit is None or hit[0] != ptrs:
            hit = (ptrs, torch.tensor(ptrs, dtype=torch.int64).to(self.dev))
            self._ptr_tables[key] = hit
        return hit[1]

    def _dense_names(self, enc="speaker_encoder"):
        nd = self.cfg["SpeakerEncoder"]["n_dense_blocks"]
        return ([f"{enc}.first_dense_layers.{l}" for l in range(nd)] + [f"{enc}.second_dense_layers.{l}" for l in range(nd)]
                + [f"{enc}.output_layer"])

    def _affine_names(self, dn="decoder"):
        return [f"{dn}.conv_affine_layers.{i}" for i in range(2 * self.cfg["Decoder"]["n_conv_blocks"])]

    def _param_table(self, kind: str, names, D: Dict[str, torch.Tensor]) -> torch.Tensor:
        return self._ptr_table((kind, names[0]), [D[n + sfx] for n in names for sfx in (".weight", ".bias")])

    def _bank_bias_table(self, enc, nb, G):
        """Device table of the nb conv-bank bias-gradient pointers (avc_bias_grad_groups); None when the bank's
        biases are not all in G (a partial parameter set in tests)."""
        names = [f"{enc}.conv_bank.{i}.bias" for i in range(nb)]
        if not all(n in G for n in names):
            return None
        return self._ptr_table(("bank_bias", enc), [G[n] for n in names])

    def prepare_tables(self, P, G=None):
        """Build the device pointer tables of the fused dense paths NOW (a host-to-device copy):
        they must exist before a CUDA-graph capture, which cannot contain that copy."""
        if G is not None:
            for enc, key in (("speaker_encoder", "SpeakerEncoder"), ("content_encoder", "ContentEncoder")):
                c = self.cfg[key]
                self._bank_bias_table(enc, len(range(c["bank_scale"], c["bank_size"] + 1, c["bank_scale"])), G)
        if not self.fused_dense:
            return
        for names in (self._dense_names(), self._affine_names()):
            if all(n + ".weight" in P for n in names):
                self._param_table("params", names, P)
                if G is not None:
                    self._param_table("grads", names, G)

    def pack_a4(self, planar: torch.Tensor, dst: A4):
        B, Cc, T = planar.shape
        assert planar.is_contiguous() and planar.dtype == torch.float32
        rnd = 1 if (self.precision == "tf32" and not self.fwd_fp32) else 0
        self._ck(self.lib.avc_pack_a4(planar.data_ptr(), dst.ptr, dst.bstride, B, Cc, T, rnd, self.stream), "pack_a4")
        if rnd and dst.bstride == dst.C * dst.T:
            dst.tf32 = True

    def unpack_a4(self, src: A4, planar: Optional[torch.Tensor] = None) -> torch.Tensor:
        if planar is None:
            planar = self.empty(src.B, src.C, src.T)
        self._ck(self.lib.avc_unpack_a4(src.ptr, src.bstride, planar.data_ptr(), src.B, src.C, src.T, self.stream), "unpack_a4")
        return planar

    # ------------------------------------------------------------------ weights
    def conv_names(self) -> List[str]:
        se, ce, de = self.cfg["SpeakerEncoder"], self.cfg["ContentEncoder"], self.cfg["Decoder"]
        names = []
        for enc, c in (("speaker_encoder", se), ("content_encoder", ce)):
            nb = len(range(c["bank_scale"], c["bank_size"] + 1, c["bank_scale"]))
            names += [f"{enc}.conv_bank.{i}" for i in range(nb)]
            names.append(f"{enc}.in_conv_layer")
            names += [f"{enc}.first_conv_layers.{l}" for l in range(c["n_conv_blocks"])]
            names += [f"{enc}.second_conv_layers.{l}" for l in range(c["n_conv_blocks"])]
        names += ["content_encoder.mean_layer", "content_encoder.std_layer", "decoder.in_conv_layer"]
        names += [f"decoder.first_conv_layers.{l}" for l in range(de["n_conv_blocks"])]
        names += [f"decoder.second_conv_layers.{l}" for l in range(de["n_conv_blocks"])]
        names.append("decoder.out_conv_layer")
        return names

    def _stride2_names(self):
        names = set()
        for enc, key in (("speaker_encoder", "SpeakerEncoder"), ("content_encoder", "ContentEncoder")):
            c = self.cfg[key]
            for l, s_ in enumerate(c["subsample"][: c["n_conv_blocks"]]):
                if s_ > 1:
                    names.add(f"{enc}.second_conv_layers.{l}")
        return names

    def pack_weights(self, P: Dict[str, torch.Tensor], need_dgrad: bool, prefixes=None):
        """nn.Conv1d weights -> kernel operand layouts, ONE launch for the whole model
        (re-run whenever parameters change).  tf32: tensor-core packs for every layer, FFMA
        packs only for the layers that stay on the FFMA kernels (stride-2 convs); other FFMA
        packs are produced lazily by _ensure_simt_pack (long-sequence inference)."""
        names = [n for n in self.conv_names() if prefixes is None or n.startswith(prefixes)]
        key = (tuple(names), bool(need_dgrad), self.precision,
               tuple((P[n + ".weight"].data_ptr(), tuple(P[n + ".weight"].shape)) for n in names))
        self._pack_version = getattr(self, "_pack_version", 0) + 1
        tables = self.__dict__.setdefault("_pack_tables", {})
        if key in tables:   # still pointing at live buffers? (tests pop / replace entries of self.packed)
            for (nm, k), ptr in tables[key][3].items():
                if nm not in self.packed or k not in self.packed[nm] or self.packed[nm][k].data_ptr() != ptr:
                    del tables[key]
                    break
        if key not in tables:
            s2 = self._stride2_names()
            used = {}
            items = (L.PackItem * len(names))()
            max_elems = 1
            for i, name in enumerate(names):
                w = P[name + ".weight"]
                Cout, Cin, K = w.shape
                slot = self.packed.setdefault(name, {})
                want_dgrad = need_dgrad and ".conv_bank." not in name  # the bank's input (x) needs no gradient
                simt = self.precision == "fp32" or name in s2
                it = items[i]
                it.w, it.Cout, it.Cin, it.K = w.data_ptr(), Cout, Cin, K
                max_elems = max(max_elems, w.numel())

                def buf(k, n):
                    if k not in slot or slot[k].numel() != n:
                        slot[k] = self.empty(n)   # (tables that pointed at a replaced buffer fail the liveness check above)
                    used[(name, k)] = slot[k].data_ptr()
                    return slot[k].data_ptr()
                if simt:
                    it.simt_fwd = buf("fwd", w.numel())
                    if want_dgrad:
                        it.simt_dgrad = buf("dgrad", w.numel())
                if self.precision == "tf32":
                    if Cin % 16 == 0:
                        n = int(self.lib.avc_tc_packed_floats(Cout, Cin, K))
                        it.tc_fwd = buf("fwd_tc", n)
                        max_elems = max(max_elems, n)
                    if want_dgrad and Cout % 16 == 0:
                        n = int(self.lib.avc_tc_packed_floats(Cin, Cout, K))
                        it.tc_dgrad = buf("dgrad_tc", n)
                        max_elems = max(max_elems, n)
                        if name in s2:   # transposed stride-2 conv = two stride-1 convs over even / odd taps
                            it.tc_dgrad_even = buf("dgrad_tc_even", int(self.lib.avc_tc_packed_floats(Cin, Cout, (K + 1) // 2)))
                            it.tc_dgrad_odd = buf("dgrad_tc_odd", int(self.lib.avc_tc_packed_floats(Cin, Cout, K // 2)))
            raw = torch.frombuffer(bytearray(bytes(items)), dtype=torch.uint8).to(self.dev)
            tables[key] = (raw, len(names), max_elems, used)
        raw, n, max_elems, _ = tables[key]
        self._ck(self.lib.avc_pack_conv_weights_batch(raw.data_ptr(), n, max_elems, self.stream), "pack_weights_batch")
        for name in names:
            slot = self.packed[name]
            for k in ("fwd", "dgrad"):
                if k in slot:
                    slot[k + "_ver"] = self._pack_version if (self.precision == "fp32" or name in self._stride2_names()) else slot.get(k + "_ver", -1)

    def _ensure_simt_pack(self, P, name, key):
        """FFMA-layout pack of one layer on demand (shapes the tensor-core path does not cover)."""
        slot = self.packed.setdefault(name, {})
        if slot.get(key + "_ver", -1) == getattr(self, "_pack_version", 0) and key in slot:
            return
        w = P[name + ".weight"]
        Cout, Cin, K = w.shape
        if key not in slot or slot[key].numel() != w.numel():
            slot[key] = self.empty(w.numel())
        mode = L.PACK_FWD if key == "fwd" else L.PACK_DGRAD
        self._ck(self.lib.avc_pack_conv_weight(w.data_ptr(), slot[key].data_ptr(), Cout, Cin, K, mode, self.stream), "pack_w")
        slot[key + "_ver"] = getattr(self, "_pack_version", 0)

    # ------------------------------------------------------------------ one conv block
    def conv(self, P, name, xin: A4, *, stride=1, shuffle=False, norm=False, cond=None, relu=False,
             res: Optional[A4] = None, res_mode=L.RES_NONE, out: Optional[A4] = None, train=False, round_out=False):
        """One fused conv block.  round_out (tf32 mode only): round the block output to TF32 -- set ONLY when
        every consumer of `out` is a tensor-core conv operand (the first conv of a block, the bank convs), so
        that the consumer can skip its rounding pass.  The residual stream, the mean/std heads and out_conv
        stay full fp32 like the reference's activations (cuDNN-TF32 rounds matmul inputs only)."""
        w = P[name + ".weight"]
        Cout, Cin, K = w.shape
        assert Cin == xin.C, (name, Cin, xin.C)
        pl, pr, Tout = conv_geometry(K, stride, xin.T)
        B = xin.B
        Cn, Tn = (Cout // 2, Tout * 2) if shuffle else (Cout, Tout)
        if out is None:
            out = A4.empty(B, Cn, Tn, self.dev)
        assert (out.C, out.T) == (Cn, Tn)
        need_c = train and (norm or relu)
        # tcgen05 path: one tile per sample up to 256 columns (fused block).  Longer samples (inference) are
        # time-tiled by the persistent kernel: fused when the block has no whole-sample statistics, otherwise
        # as a plain conv whose raw output avc_norm_apply_fwd finishes (shuffle / InstanceNorm / AdaIN / residual)
        tc_ok = (self.precision == "tf32" and not self.fwd_fp32 and Cin % 16 == 0 and not (stride == 2 and shuffle)
                 and "fwd_tc" in self.packed[name])
        use_tc = tc_ok and (Tout * stride <= 256 or (self.tc_conv_v2 and not norm and not shuffle))
        tc_split = tc_ok and not use_tc and self.tc_conv_v2 and norm
        fused = use_tc or (not tc_split and ((not norm) or (Tout <= 128) or (Tout <= 256 and K in (1, 5))))
        c = A4.empty(B, Cout, Tout, self.dev) if (need_c or not fused) else None
        stats = self.empty(B, Cn, 2) if norm else None
        d = L.ConvDesc()
        d.B, d.Cin, d.Cout, d.K, d.stride = B, Cin, Cout, K, stride
        d.pad_left, d.pad_mode, d.in_ups, d.Tin, d.Tout = pl, L.PAD_REFLECT, 1, xin.T, Tout
        d.in_, d.in_bstride = xin.ptr, xin.bstride
        if not (use_tc or tc_split):
            self._ensure_simt_pack(P, name, "fwd")
            d.w_packed = self.packed[name]["fwd"].data_ptr()
        d.w_ld = Cout
        d.bias = P[name + ".bias"].data_ptr()
        d.eps = IN_EPS
        if self.precision == "tf32" and not self.fwd_fp32:
            d.flags = (L.F_ROUND_OUT if round_out else 0) | (L.F_IN_TF32 if xin.tf32 else 0)
            if round_out and out.bstride == out.C * out.T:
                out.tf32 = True
        if fused:
            self._fill_epilogue(d, out, shuffle, norm, relu, cond, res, res_mode, stats)
            d.save_c = c.ptr if c is not None else None
            if use_tc:
                d.w_tc = self.packed[name]["fwd_tc"].data_ptr()
                self._ck(self.lib.avc_conv_block_tc(C.byref(d), self.tc_status.data_ptr(), self.stream), f"conv_block_tc[{name}]")
            else:
                self._ck(self.lib.avc_conv_block_fwd(C.byref(d), self.stream), f"conv_block_fwd[{name}]")
        else:
            d.out, d.out_bstride = c.ptr, c.bstride
            if tc_split:
                flags = int(d.flags)
                d.flags = flags & ~L.F_ROUND_OUT     # the raw conv output feeds the statistics: keep it fp32
                d.w_tc = self.packed[name]["fwd_tc"].data_ptr()
                self._ck(self.lib.avc_conv_block_tc(C.byref(d), self.tc_status.data_ptr(), self.stream), f"conv_tc_plain[{name}]")
                d.flags = flags
            else:
                self._ck(self.lib.avc_conv_block_fwd(C.byref(d), self.stream), f"conv_block_fwd[{name}]")
            self._fill_epilogue(d, out, shuffle, norm, relu, cond, res, res_mode, stats)
            d.save_c = c.ptr
            self._ck(self.lib.avc_norm_apply_fwd(C.byref(d), self.stream), f"norm_apply_fwd[{name}]")
            if not need_c:
                c = None
        rec = None
        if train:
            rec = dict(name=name, xin=xin, c=c, stats=stats, cond=cond, out=out, stride=stride, shuffle=shuffle,
                       norm=norm, relu=relu, K=K, Cin=Cin, Cout=Cout, Tout=Tout, pl=pl, pr=pr)
        return out, rec

    def prepare_wgrad_acc(self, P, G):
        """Register the persistent gradient buffers G for in-place accumulation: one zeroed arena
        with a [K][Cin/4][coutp][4] region per conv layer and the device item table of the flush
        kernel.  Must run before a CUDA-graph capture (it copies the table to the device)."""
        if not self.wgrad_acc or self.precision != "tf32":
            self._wg_acc = None
            return
        names = [n for n in self.conv_names() if n + ".weight" in P and n + ".weight" in G]
        key = tuple((G[n + ".weight"].data_ptr(), tuple(P[n + ".weight"].shape)) for n in names)
        if self._wg_acc is not None and self._wg_acc["key"] == key:
            return
        offs, total, max_units, rows = {}, 0, 1, []
        for n in names:
            Cout, Cin, K = P[n + ".weight"].shape
            nf = int(self.lib.avc_wgrad_acc_floats(Cout, Cin, K))
            if nf <= 0 or Cout % 4 != 0:
                continue
            offs[n] = total
            rows.append((n, total, Cout, Cin, K))
            total += nf
            max_units = max(max_units, nf // 4)
        if not rows:
            self._wg_acc = None
            return
        arena = self.zeros(total)
        items = (L.WgradAccItem * len(rows))()
        dw_ptr = {}
        for it, (n, off, Cout, Cin, K) in zip(items, rows):
            it.acc, it.dw = arena.data_ptr() + 4 * off, G[n + ".weight"].data_ptr()
            it.Cout, it.Cin, it.K = Cout, Cin, K
            dw_ptr[n] = it.dw
        raw = torch.frombuffer(bytearray(bytes(items)), dtype=torch.uint8).to(self.dev)
        n_dec = sum(1 for r in rows if r[0].startswith("decoder."))
        if n_dec and not all(r[0].startswith("decoder.") for r in rows[len(rows) - n_dec:]):
            n_dec = 0   # (conv_names lists the decoder last; anything else: no partial flush)
        self._wg_acc = dict(key=key, arena=arena, offs=offs, dw_ptr=dw_ptr, items=raw, n=len(rows), max_units=max_units, dirty=False,
                            n_dec=n_dec, dec_done=False)

    def flush_wgrad(self, decoder_only=False):
        """Fold the accumulated conv weight gradients into the registered gradient buffers.  decoder_only: just the
        decoder's layers (the last rows of the item table) -- they are final as soon as the decoder's backward is, so
        the trainer folds them on the weight-gradient stream while the encoders' backward runs; the closing call then
        covers the remaining rows."""
        acc = self._wg_acc
        if acc is None or not acc["dirty"]:
            return
        n, nd = acc["n"], acc["n_dec"]
        item = C.sizeof(L.WgradAccItem)
        if decoder_only:
            if nd > 0 and not acc["dec_done"]:
                self._ck(self.lib.avc_wgrad_acc_flush(acc["items"].data_ptr() + (n - nd) * item, nd, acc["max_units"], self.stream), "wgrad_acc_flush[decoder]")
                acc["dec_done"] = True
            return
        rows = n - nd if acc["dec_done"] else n
        if rows > 0:
            self._ck(self.lib.avc_wgrad_acc_flush(acc["items"].data_ptr(), rows, acc["max_units"], self.stream), "wgrad_acc_flush")
        acc["dirty"], acc["dec_done"] = False, False

    def wgrad(self, wd, name, keep=()):
        """dW += conv weight gradient; tensor cores when the shape allows, FFMA otherwise.
        A weight gradient is a LEAF of the backward pass (nothing downstream reads it before the optimizer), so
        with ``wgrad_stream`` set (FusedTrainer does, around its step) it is forked onto that stream behind the
        caller's current stream and the dgrad / norm-backward chain continues without it; ``join_wgrad()`` joins.
        `keep`: the tensors the launch reads -- held until the join so that the caching allocator cannot hand their
        memory to the launching stream while the forked kernel still reads them."""
        ws = self.wgrad_stream
        if ws is not None:
            ws.wait_stream(torch.cuda.current_stream(self.dev))
            self._wg_keep.extend(keep)
            with torch.cuda.stream(ws):
                self._wgrad_launch(wd, name)
            return
        self._wgrad_launch(wd, name)

    def join_wgrad(self):
        """The current stream waits for every forked weight gradient; releases the tensors held for them."""
        if self.wgrad_stream is not None:
            torch.cuda.current_stream(self.dev).wait_stream(self.wgrad_stream)
        self._wg_keep.clear()

    def _wgrad_launch(self, wd, name):
        if self.precision == "tf32":
            n = int(self.lib.avc_wgrad_tc_scratch_floats(C.byref(wd)))
            acc = self._wg_acc
            if n > 0 and acc is not None and acc["dw_ptr"].get(name) == wd.dw:
                ptr = acc["arena"].data_ptr() + 4 * acc["offs"][name]
                self._ck(self.lib.avc_conv_wgrad_tc_acc(C.byref(wd), ptr, self.tc_status.data_ptr(), self.stream), f"conv_wgrad_tc_acc[{name}]")
                acc["dirty"] = True
                return
            if n > 0:
                scratch = self.empty(n)
                self._ck(self.lib.avc_conv_wgrad_tc(C.byref(wd), scratch.data_ptr(), self.tc_status.data_ptr(), self.stream), f"conv_wgrad_tc[{name}]")
                return
        self._ck(self.lib.avc_conv_wgrad(C.byref(wd), self.stream), f"conv_wgrad[{name}]")

    @staticmethod
    def _fill_epilogue(d, out, shuffle, norm, relu, cond, res, res_mode, stats):
        d.out, d.out_bstride = out.ptr, out.bstride
        d.shuffle, d.norm, d.relu = int(shuffle), int(norm), int(relu)
        if cond is not None:
            d.cond, d.cond_bstride = cond.data_ptr(), cond.stride(0)
        if res is not None:
            d.res, d.res_bstride, d.res_mode, d.res_T = res.ptr, res.bstride, res_mode, res.T
        d.stats = _ptr(stats)

    def _can_fuse_norm_bwd(self, rec, up, Cdx) -> bool:
        """May the data-gradient conv of `rec` run the InstanceNorm/AdaIN/ReLU backward of the upstream block `up`
        in its own epilogue (AVC_F_NORMBWD)?  Needs the persistent kernel's fold path and matching shapes."""
        if not (self.norm_bwd_fused and self.fold_fused and self.tc_conv_v2 and self.precision == "tf32") or up is None:
            return False
        xin, K, pl, pr = rec["xin"], rec["K"], rec["pl"], rec["pr"]
        Lp = xin.T + pl + pr
        if not (rec["stride"] == 1 and K > 1 and rec["Cout"] % 16 == 0 and Lp <= 144 and "dgrad_tc" in self.packed[rec["name"]]
                and xin.T >= 2 * pl + 1 and xin.T >= pr + 2):
            return False
        return (not up["shuffle"] and up["c"] is not None and (up["norm"] or up["relu"]) and up["Cout"] == Cdx and Cdx <= 128
                and up["Tout"] == xin.T)

    def conv_bwd(self, P, G, rec, dy: Optional[A4], *, need_dx=True, dres: Optional[A4] = None, dres_mode=L.RES_NONE,
                 dcond: Optional[torch.Tensor] = None, mask: Optional[A4] = None, dx_channels=None,
                 dc_pre: Optional[A4] = None, fuse_up: Optional[dict] = None) -> Optional[A4]:
        """Backward of one conv block.  dy: grad w.r.t. the block output *before* the residual
        add.  Returns grad w.r.t. the block input (+ adjoint of the residual branch `dres`).

        dc_pre: the gradient w.r.t. this block's raw conv output, already produced by the downstream block's fused
        epilogue (then dy is ignored).  fuse_up = {"rec": upstream block, "dcond": its AdaIN-row gradient or None,
        "need_dx": bool}: if eligible, this block's data-gradient conv also runs the upstream block's norm backward;
        fuse_up["dc"] then holds the upstream dc (pass it as dc_pre to the upstream conv_bwd) and the return value is
        None unless need_dx."""
        name, xin, B = rec["name"], rec["xin"], rec["xin"].B
        K, Cin, Cout, Tout, stride = rec["K"], rec["Cin"], rec["Cout"], rec["Tout"], rec["stride"]
        st = self.stream
        gb = G[name + ".bias"]
        if fuse_up is not None:
            fuse_up["dc"] = None
        if dc_pre is not None:
            dc = dc_pre
        elif rec["norm"] or rec["relu"]:
            dc = A4.empty(B, Cout, Tout, self.dev)
            d = L.ConvDesc()
            d.B, d.Cin, d.Cout, d.K, d.stride, d.Tin, d.Tout = B, Cin, Cout, K, stride, xin.T, Tout
            d.in_ups = 1
            d.shuffle, d.norm, d.relu, d.eps = int(rec["shuffle"]), int(rec["norm"]), int(rec["relu"]), IN_EPS
            d.save_c, d.stats = rec["c"].ptr, _ptr(rec["stats"])
            if rec["cond"] is not None:
                d.cond, d.cond_bstride = rec["cond"].data_ptr(), rec["cond"].stride(0)
                d.dcond, d.dcond_bstride = dcond.data_ptr(), dcond.stride(0)
            d.dy, d.dy_bstride = dy.ptr, dy.bstride
            # the bias of a conv that feeds an InstanceNorm has an identically zero gradient (the norm removes the
            # per-channel mean); autograd returns ~1e-9 rounding noise there, we leave the zeroed buffer untouched
            # (not with pixel shuffle: there two conv rows with different biases share one normalised channel)
            d.dc, d.dbias = dc.ptr, (None if (rec["norm"] and not rec["shuffle"]) else gb.data_ptr())
            if self.precision == "tf32":
                d.flags = L.F_ROUND_OUT
                dc.tf32 = True
            self._ck(self.lib.avc_norm_bwd(C.byref(d), st), f"norm_bwd[{name}]")
            if self.debug:
                self.debug(name, "dc", dc)
        else:
            dc = dy
            self._ck(self.lib.avc_bias_grad(dc.ptr, dc.bstride, gb.data_ptr(), B, Cout, Tout, st), f"bias_grad[{name}]")
        wd = L.WgradDesc()
        wd.B, wd.Cin, wd.Cout, wd.K, wd.stride, wd.pad_left, wd.Tin, wd.Tout = B, Cin, Cout, K, stride, rec["pl"], xin.T, Tout
        wd.x, wd.x_bstride, wd.dc, wd.dc_bstride = xin.ptr, xin.bstride, dc.ptr, dc.bstride
        wd.dw = G[name + ".weight"].data_ptr()
        self.wgrad(wd, name, keep=(xin.t, dc.t))
        if self.debug:
            self.debug(name, "dw", G[name + ".weight"])
        if not need_dx:
            return None
        # data gradient: full transposed conv (zero pad) then fold the reflect halo back
        Cdx = Cin if dx_channels is None else dx_channels
        Lp = xin.T + rec["pl"] + rec["pr"]
        direct = (K == 1 and stride == 1 and dres is None)
        dx = A4.empty(B, Cdx, xin.T, self.dev)
        dxp = dx if direct else A4.empty(B, Cdx, Lp, self.dev)
        d = L.ConvDesc()
        d.B, d.Cin, d.Cout, d.K, d.stride = B, Cout, Cdx, K, 1
        d.pad_left, d.pad_mode, d.in_ups, d.Tin, d.Tout = K - 1, L.PAD_ZERO, stride, Tout, Lp
        d.in_, d.in_bstride = dc.ptr, dc.bstride
        d.w_ld = Cin
        d.out, d.out_bstride = dxp.ptr, dxp.bstride
        d.eps = IN_EPS
        if self.precision == "tf32" and dc.tf32:
            d.flags = L.F_IN_TF32
        if mask is not None:
            assert direct
            d.mask, d.mask_bstride = mask.ptr, mask.bstride
        if (self.precision == "tf32" and stride == 2 and K == 5 and Cout % 16 == 0 and Lp <= 512 and "dgrad_tc_even" in self.packed[name]):
            # dxp[2v]   = sum_{jj<3} Wd[2jj]   dc[v + jj - 2]   (taps 0,2,4; pad_left 2)
            # dxp[2v+1] = sum_{jj<2} Wd[2jj+1] dc[v + jj - 1]   (taps 1,3;   pad_left 1)
            for par, kk, pl_, key in ((0, 3, 2, "dgrad_tc_even"), (1, 2, 1, "dgrad_tc_odd")):
                d.K, d.pad_left, d.in_ups = kk, pl_, 1
                d.Tout = (Lp + 1 - par) // 2
                d.out_tstride, d.out_toff, d.out_T = 2, par, Lp
                d.w_tc = self.packed[name][key].data_ptr()
                self._ck(self.lib.avc_conv_block_tc(C.byref(d), self.tc_status.data_ptr(), st), f"conv_dgrad_tc_s2[{name}]")
        elif (self.precision == "tf32" and stride == 1 and Cout % 16 == 0 and Lp <= 256 and "dgrad_tc" in self.packed[name]):
            d.w_tc = self.packed[name]["dgrad_tc"].data_ptr()
            if self.fold_fused and not direct and xin.T >= 2 * rec["pl"] + 1 and xin.T >= rec["pr"] + 2:
                # the data-gradient conv folds the reflect halo and the residual adjoint in its own epilogue
                d.out, d.out_bstride, d.out_T = dx.ptr, dx.bstride, xin.T
                d.flags = int(d.flags) | L.F_FOLD | (rec["pl"] << 8) | (rec["pr"] << 16)
                if dres is not None:
                    d.res, d.res_bstride, d.res_mode, d.res_T = dres.ptr, dres.bstride, dres_mode, dres.T
                up = fuse_up["rec"] if fuse_up is not None else None
                if up is not None and mask is None and self._can_fuse_norm_bwd(rec, up, Cdx):
                    # ... and the upstream block's InstanceNorm / AdaIN / ReLU backward (avc_norm_bwd's job)
                    dc_up = A4.empty(B, Cdx, xin.T, self.dev)
                    dc_up.tf32 = True
                    d.flags = int(d.flags) | L.F_NORMBWD | L.F_ROUND_OUT
                    d.norm, d.relu, d.eps = int(up["norm"]), int(up["relu"]), IN_EPS
                    d.save_c, d.stats = up["c"].ptr, _ptr(up["stats"])
                    if up["cond"] is not None:
                        d.cond, d.cond_bstride = up["cond"].data_ptr(), up["cond"].stride(0)
                        d.dcond, d.dcond_bstride = fuse_up["dcond"].data_ptr(), fuse_up["dcond"].stride(0)
                    d.dc = dc_up.ptr
                    d.dbias = None if up["norm"] else G[up["name"] + ".bias"].data_ptr()
                    if not fuse_up.get("need_dx", True):
                        d.out = None
                    self._ck(self.lib.avc_conv_block_tc(C.byref(d), self.tc_status.data_ptr(), st), f"conv_dgrad_tc_fold_normbwd[{name}]")
                    fuse_up["dc"] = dc_up
                    if self.debug:
                        self.debug(up["name"], "dc", dc_up)
                    return dx if fuse_up.get("need_dx", True) else None
                self._ck(self.lib.avc_conv_block_tc(C.byref(d), self.tc_status.data_ptr(), st), f"conv_dgrad_tc_fold[{name}]")
                if self.debug:
                    self.debug(name, "dx", dx)
                return dx
            self._ck(self.lib.avc_conv_block_tc(C.byref(d), self.tc_status.data_ptr(), st), f"conv_dgrad_tc[{name}]")
        else:
            self._ensure_simt_pack(P, name, "dgrad")
            d.w_packed = self.packed[name]["dgrad"].data_ptr()
            self._ck(self.lib.avc_conv_block_fwd(C.byref(d), st), f"conv_dgrad[{name}]")
        if direct:
            return dx
        f = L.FoldDesc()
        f.B, f.C, f.Tin, f.pad_left, f.pad_right = B, Cdx, xin.T, rec["pl"], rec["pr"]
        f.dxp = dxp.ptr
        if dres is not None:
            f.dres, f.dres_bstride, f.res_mode, f.res_T = dres.ptr, dres.bstride, dres_mode, dres.T
        f.dx, f.dx_bstride = dx.ptr, dx.bstride
        self._ck(self.lib.avc_fold_add_fwd(C.byref(f), st), f"fold_add[{name}]")
        if self.debug:
            self.debug(name, "dxp", dxp)
            self.debug(name, "dx", dx)
        return dx

    # ------------------------------------------------------------------ linear layers
    def linear(self, P, name, x: torch.Tensor, *, relu=False, res=None, out=None, train=False):
        w = P[name + ".weight"]
        N, K = w.shape
        B = x.shape[0]
        if out is None:
            out = self.empty(B, N)
        y_act = self.empty(B, N) if (train and relu) else None
        d = L.LinearDesc()
        d.B, d.N, d.K, d.relu = B, N, K, int(relu)
        d.x, d.x_bstride = x.data_ptr(), x.stride(0)
        d.w, d.bias = w.data_ptr(), P[name + ".bias"].data_ptr()
        d.res, d.y_act = _ptr(res), _ptr(y_act)
        d.out, d.out_bstride = out.data_ptr(), out.stride(0)
        self._ck(self.lib.avc_linear_fwd(C.byref(d), self.stream), f"linear_fwd[{name}]")
        rec = dict(name=name, x=x, y_act=y_act, relu=relu, N=N, K=K) if train else None
        return out, rec

    def linear_bwd(self, P, G, rec, dy: torch.Tensor, *, dx_add=None, need_dx=True):
        name = rec["name"]
        B = rec["x"].shape[0]
        d = L.LinearDesc()
        d.B, d.N, d.K, d.relu = B, rec["N"], rec["K"], int(rec["relu"])
        d.x, d.x_bstride = rec["x"].data_ptr(), rec["x"].stride(0)
        d.w = P[name + ".weight"].data_ptr()
        d.y_act = _ptr(rec["y_act"])
        d.dy, d.dy_bstride = dy.data_ptr(), dy.stride(0)
        dx = self.empty(B, rec["K"]) if need_dx else None
        d.dx, d.dx_add = _ptr(dx), _ptr(dx_add)
        d.dw, d.db = G[name + ".weight"].data_ptr(), G[name + ".bias"].data_ptr()
        self._ck(self.lib.avc_linear_bwd(C.byref(d), self.stream), f"linear_bwd[{name}]")
        return dx

    # ------------------------------------------------------------------ encoders
    def _bank_and_in_conv(self, P, enc, c, x_planar: torch.Tensor, norm: bool, train: bool, ctx: dict):
        """conv_bank + in_conv_layer (model.py:85-91, 266-269 / 302-307).  The concat is never
        assembled by a copy: every bank conv writes its channel range of one A4 buffer and
        x itself is packed straight into the last c_in channels."""
        B, c_in, T = x_planar.shape
        ks = list(range(c["bank_scale"], c["bank_size"] + 1, c["bank_scale"]))
        c_bank = c["c_bank"]
        ctot = c_bank * len(ks) + c_in
        cat = A4.empty(B, ctot, T, self.dev)
        x4 = cat.channels(c_bank * len(ks), ctot)
        self.pack_a4(x_planar, x4)
        recs = []
        for i, _k in enumerate(ks):
            _, r = self.conv(P, f"{enc}.conv_bank.{i}", x4, relu=True, out=cat.channels(i * c_bank, (i + 1) * c_bank), train=False,
                             round_out=True)   # the concat is read by in_conv (and its weight gradient) only
            recs.append(r)
        # every writer of `cat` (pack_a4 and the bank convs' epilogues) rounds to TF32 in tf32 mode
        cat.tf32 = self.precision == "tf32" and not self.fwd_fp32
        out, rec_in = self.conv(P, f"{enc}.in_conv_layer", cat, norm=norm, relu=True, train=train)
        if train:
            ctx["cat"], ctx["x4"], ctx["in"] = cat, x4, rec_in
            ctx["n_bank"], ctx["c_bank"] = len(ks), c_bank
        return out

    def _enc_blocks(self, P, enc, c, out: A4, norm: bool, train: bool, ctx: dict):
        blocks = []
        for l, s in enumerate(c["subsample"][: c["n_conv_blocks"]]):
            y, r1 = self.conv(P, f"{enc}.first_conv_layers.{l}", out, norm=norm, relu=True, train=train, round_out=True)
            new, r2 = self.conv(P, f"{enc}.second_conv_layers.{l}", y, stride=s, norm=norm, relu=True, res=out,
                                res_mode=L.RES_POOL if s > 1 else L.RES_SAME, train=train)
            blocks.append((r1, r2, s, out))
            out = new
        if train:
            ctx["blocks"] = blocks
        return out

    def speaker_fwd(self, P, x_planar: torch.Tensor, train: bool):
        """SpeakerEncoder.forward (model.py:265-277) -> emb [B, c_out]."""
        c = self.cfg["SpeakerEncoder"]
        enc = "speaker_encoder"
        ctx: dict = {}
        out = self._bank_and_in_conv(P, enc, c, x_planar, norm=False, train=train, ctx=ctx)
        out = self._enc_blocks(P, enc, c, out, norm=False, train=train, ctx=ctx)
        B = out.B
        pooled = self.empty(B, out.C)
        self._ck(self.lib.avc_time_mean_fwd(out.ptr, out.bstride, pooled.data_ptr(), B, out.C, out.T, self.stream), "time_mean_fwd")
        nd = c["n_dense_blocks"]
        if self.fused_dense and out.C == 128 and c["c_out"] == 128:
            names = self._dense_names(enc)
            tab = self._param_table("params", names, P)
            save = self.empty(3 * nd + 1, B, 128) if train else None
            emb = self.empty(B, 128)
            d = L.DenseStackDesc()
            d.B, d.C, d.c_out, d.n_blocks = B, 128, 128, nd
            d.params, d.x, d.save, d.out = tab.data_ptr(), pooled.data_ptr(), _ptr(save), emb.data_ptr()
            self._ck(self.lib.avc_dense_stack_fwd(C.byref(d), self.stream), "dense_stack_fwd")
            if train:
                ctx.update(dense_fused=dict(save=save, tab=tab, names=names, pooled=pooled), last=out)
            return emb, ctx
        h = pooled
        dense = []
        for l in range(nd):
            y, r1 = self.linear(P, f"{enc}.first_dense_layers.{l}", h, relu=True, train=train)
            h, r2 = self.linear(P, f"{enc}.second_dense_layers.{l}", y, relu=True, res=h, train=train)
            dense.append((r1, r2))
        emb, r_out = self.linear(P, f"{enc}.output_layer", h, train=train)
        if train:
            ctx.update(dense=dense, out_rec=r_out, last=out)
        return emb, ctx

    def speaker_bwd(self, P, G, ctx, demb: torch.Tensor):
        c = self.cfg["SpeakerEncoder"]
        last = ctx["last"]
        if "dense_fused" in ctx:
            f = ctx["dense_fused"]
            nd, B = c["n_dense_blocks"], last.B
            gsave, dh = self.empty(2 * nd + 1, B, 128), self.empty(B, 128)
            demb = demb.contiguous()
            d = L.DenseStackDesc()
            d.B, d.C, d.c_out, d.n_blocks = B, 128, 128, nd
            d.params, d.save, d.dout = f["tab"].data_ptr(), f["save"].data_ptr(), demb.data_ptr()
            d.gsave, d.dx = gsave.data_ptr(), dh.data_ptr()
            self._ck(self.lib.avc_dense_stack_bwd(C.byref(d), self.stream), "dense_stack_bwd")
            # weight gradients of the 2n+1 layers in one launch: (gsave plane, save plane) per layer
            gtab = self._param_table("grads", f["names"], G)
            plane = B * 128
            slots = [(l, l) for l in range(nd)] + [(nd + l, nd + 1 + l) for l in range(nd)] + [(2 * nd, nd)]
            bd = L.LinearBatchDesc()
            bd.L, bd.B, bd.N, bd.K = len(slots), B, 128, 128
            bd.grads, bd.x, bd.x_bstride, bd.y, bd.y_bstride = gtab.data_ptr(), f["save"].data_ptr(), 128, gsave.data_ptr(), 128
            for i, (gs, xs) in enumerate(slots):
                bd.y_off[i], bd.x_off[i] = gs * plane, xs * plane
            self._ck(self.lib.avc_linear_batch_dw(C.byref(bd), self.stream), "linear_batch_dw[dense]")
        else:
            dh = self.linear_bwd(P, G, ctx["out_rec"], demb)
            for r1, r2 in reversed(ctx["dense"]):
                dy = self.linear_bwd(P, G, r2, dh)                 # through second layer (+ReLU mask)
                dh = self.linear_bwd(P, G, r1, dy, dx_add=dh)       # through first layer, + identity branch
        dout = A4.empty(last.B, last.C, last.T, self.dev)
        self._ck(self.lib.avc_time_mean_bwd(dh.data_ptr(), dout.ptr, dout.bstride, last.B, last.C, last.T, self.stream), "time_mean_bwd")
        self._enc_bwd(P, G, "speaker_encoder", c, ctx, dout)

    def content_fwd(self, P, x_planar: torch.Tensor, train: bool):
        """ContentEncoder.forward (model.py:301-323) -> (mu4, ls4) A4 [B, c_out, T/8]."""
        c = self.cfg["ContentEncoder"]
        enc = "content_encoder"
        ctx: dict = {}
        out = self._bank_and_in_conv(P, enc, c, x_planar, norm=True, train=train, ctx=ctx)
        out = self._enc_blocks(P, enc, c, out, norm=True, train=train, ctx=ctx)
        mu4, r_mu = self.conv(P, f"{enc}.mean_layer", out, train=train)
        ls4, r_ls = self.conv(P, f"{enc}.std_layer", out, train=train)
        if train:
            ctx.update(mu_rec=r_mu, ls_rec=r_ls)
        return mu4, ls4, ctx

    def content_bwd(self, P, G, ctx, dmu4: A4, dls4: A4):
        c = self.cfg["ContentEncoder"]
        d1 = self.conv_bwd(P, G, ctx["mu_rec"], dmu4)
        d2 = self.conv_bwd(P, G, ctx["ls_rec"], dls4)
        dout = self._add(d1, d2)
        self._enc_bwd(P, G, "content_encoder", c, ctx, dout)

    def _add(self, a: A4, b: A4) -> A4:
        """a + b via the fold kernel (pad 0, residual SAME)."""
        out = A4.empty(a.B, a.C, a.T, self.dev)
        f = L.FoldDesc()
        f.B, f.C, f.Tin, f.pad_left, f.pad_right = a.B, a.C, a.T, 0, 0
        f.dxp = a.ptr
        assert a.bstride == a.C * a.T
        f.dres, f.dres_bstride, f.res_mode, f.res_T = b.ptr, b.bstride, L.RES_SAME, b.T
        f.dx, f.dx_bstride = out.ptr, out.bstride
        self._ck(self.lib.avc_fold_add_fwd(C.byref(f), self.stream), "add")
        return out

    def _enc_bwd(self, P, G, enc, c, ctx, dout: A4):
        blocks = ctx["blocks"]
        dc2 = None    # dc of the current block's second conv when the downstream data-gradient conv already produced it
        for l in reversed(range(len(blocks))):
            r1, r2, s, _blk_in = blocks[l]
            f1 = dict(rec=r1, dcond=None, need_dx=False)           # r2's data gradient feeds r1's norm backward only
            dy1 = self.conv_bwd(P, G, r2, dout, dc_pre=dc2, fuse_up=f1)
            up = blocks[l - 1][1] if l > 0 else ctx["in"]           # whose output gradient r1's data gradient produces
            f2 = dict(rec=up, dcond=None, need_dx=l > 0)            # ... needed again as the residual adjoint of block l-1
            dout = self.conv_bwd(P, G, r1, dy1, dc_pre=f1["dc"], dres=dout, dres_mode=L.RES_POOL if s > 1 else L.RES_SAME, fuse_up=f2)
            dc2 = f2["dc"]
        # in_conv: dgrad only towards the bank outputs (x needs no grad), ReLU mask fused
        cat, nb, cb = ctx["cat"], ctx["n_bank"], ctx["c_bank"]
        bank_out = cat.channels(0, nb * cb)
        dbank = self.conv_bwd(P, G, ctx["in"], dout, dc_pre=dc2, mask=bank_out, dx_channels=nb * cb)
        x4 = ctx["x4"]
        st = self.stream
        # bias gradients of the whole bank in one launch (the bank outputs all have x's length: K//2 + (K-1)//2 padding)
        btab = self._bank_bias_table(enc, nb, G)
        if btab is not None:
            self._ck(self.lib.avc_bias_grad_groups(dbank.ptr, dbank.bstride, btab.data_ptr(), cb, x4.B, nb * cb, x4.T, st), "bias_grad_groups")
        for i in range(nb):
            name = f"{enc}.conv_bank.{i}"
            w = P[name + ".weight"]
            Cout, Cin, K = w.shape
            pl, pr, Tout = conv_geometry(K, 1, x4.T)
            dci = dbank.channels(i * cb, (i + 1) * cb)
            if btab is None:
                self._ck(self.lib.avc_bias_grad(dci.ptr, dci.bstride, G[name + ".bias"].data_ptr(), x4.B, Cout, Tout, st), "bias_grad")
            wd = L.WgradDesc()
            wd.B, wd.Cin, wd.Cout, wd.K, wd.stride, wd.pad_left, wd.Tin, wd.Tout = x4.B, Cin, Cout, K, 1, pl, x4.T, Tout
            wd.x, wd.x_bstride, wd.dc, wd.dc_bstride = x4.ptr, x4.bstride, dci.ptr, dci.bstride
            wd.dw = G[name + ".weight"].data_ptr()
            self.wgrad(wd, name, keep=(x4.t, dbank.t))

    # ------------------------------------------------------------------ reparameterisation
    def reparam_fwd(self, mu4: A4, ls4: A4, eps: Optional[torch.Tensor], want_planar=True):
        B, Cc, T = mu4.B, mu4.C, mu4.T
        z4 = A4.empty(B, Cc, T, self.dev)
        mu = self.empty(B, Cc, T) if want_planar else None
        ls = self.empty(B, Cc, T) if want_planar else None
        self._ck(self.lib.avc_reparam_fwd(mu4.ptr, ls4.ptr, _ptr(eps), _ptr(mu), _ptr(ls), z4.ptr, B, Cc, T, self.stream), "reparam_fwd")
        return mu, ls, z4

    def reparam_bwd(self, dz4: Optional[A4], ls4: A4, eps, dmu_ext, dls_ext):
        B, Cc, T = ls4.B, ls4.C, ls4.T
        dmu4, dls4 = A4.empty(B, Cc, T, self.dev), A4.empty(B, Cc, T, self.dev)
        self._ck(self.lib.avc_reparam_bwd(None if dz4 is None else dz4.ptr, ls4.ptr, _ptr(eps), _ptr(dmu_ext), _ptr(dls_ext),
                                          dmu4.ptr, dls4.ptr, B, Cc, T, self.stream), "reparam_bwd")
        return dmu4, dls4

    # ------------------------------------------------------------------ decoder
    def decoder_affine_fwd(self, P, emb: torch.Tensor, train: bool):
        """The 2*n AdaIN rows (beta|gamma) of every decoder block: conv_affine_layers (model.py:342-343, used :356,:363).
        They read the speaker embedding only, so a caller that runs the speaker encoder on its own stream computes
        them there (trainer.py) and hands the result to decoder_fwd.  -> (conds [B, 2n, 2*c_h], aff)"""
        c = self.cfg["Decoder"]
        dn = "decoder"
        nblk = c["n_conv_blocks"]
        ch2 = 2 * c["c_h"]
        B = emb.shape[0]
        conds = self.empty(B, 2 * nblk, ch2)
        aff = []
        naff = 2 * nblk
        fused_aff = self.fused_dense and naff <= L.LINEAR_BATCH_MAX and emb.is_contiguous()
        if fused_aff:
            anames = self._affine_names(dn)
            tab = self._param_table("params", anames, P)
            bd = L.LinearBatchDesc()
            bd.L, bd.B, bd.N, bd.K = naff, B, ch2, emb.shape[1]
            bd.params, bd.x, bd.x_bstride = tab.data_ptr(), emb.data_ptr(), emb.stride(0)
            bd.out, bd.y_bstride = conds.data_ptr(), naff * ch2
            for i in range(naff):
                bd.x_off[i], bd.y_off[i] = 0, i * ch2
            self._ck(self.lib.avc_linear_batch_fwd(C.byref(bd), self.stream), "linear_batch_fwd[affine]")
            aff = dict(tab=tab, names=anames)
        else:
            for i in range(naff):
                _, r = self.linear(P, f"{dn}.conv_affine_layers.{i}", emb, out=conds[:, i], train=train)
                aff.append(r)
        return conds, aff

    def decoder_fwd(self, P, z4: A4, emb: torch.Tensor, train: bool, affine=None):
        """Decoder.forward (model.py:347-371) -> dec4 A4 [B, c_out, 8*T].  affine: the result of decoder_affine_fwd
        when the caller already computed it (on the speaker branch's stream)."""
        c = self.cfg["Decoder"]
        dn = "decoder"
        ctx: dict = {}
        out, r_in = self.conv(P, f"{dn}.in_conv_layer", z4, norm=True, relu=True, train=train)
        nblk = c["n_conv_blocks"]
        conds, aff = affine if affine is not None else self.decoder_affine_fwd(P, emb, train)
        blocks = []
        for l, up in enumerate(c["upsample"][:nblk]):
            y, r1 = self.conv(P, f"{dn}.first_conv_layers.{l}", out, norm=True, cond=conds[:, 2 * l], relu=True, train=train,
                              round_out=True)
            new, r2 = self.conv(P, f"{dn}.second_conv_layers.{l}", y, shuffle=(up > 1), norm=True, cond=conds[:, 2 * l + 1],
                                relu=True, res=out, res_mode=L.RES_UP if up > 1 else L.RES_SAME, train=train)
            blocks.append((r1, r2, up))
            out = new
        dec4, r_out = self.conv(P, f"{dn}.out_conv_layer", out, train=train)
        if train:
            ctx.update(in_rec=r_in, aff=aff, blocks=blocks, out_rec=r_out, conds=conds, emb=emb)
        return dec4, ctx

    def decoder_bwd(self, P, G, ctx, ddec4: A4, need_dz=True, affine_stream=None):
        """Returns (dz4, demb).  affine_stream: the gradients of the AdaIN affine layers (and demb, which only the
        speaker encoder's backward needs) are complete after the block loop; with a stream given they fork onto it
        there, beside the in_conv data gradient -- demb is then produced ON that stream (the caller continues the
        speaker branch on it) and the tensors the forked launches read stay alive in ctx."""
        c = self.cfg["Decoder"]
        nblk = c["n_conv_blocks"]
        dout = self.conv_bwd(P, G, ctx["out_rec"], ddec4)
        dconds = self.empty(*ctx["conds"].shape)
        blocks = ctx["blocks"]
        dc2 = None
        for l in reversed(range(nblk)):
            r1, r2, up = blocks[l]
            f1 = dict(rec=r1, dcond=dconds[:, 2 * l], need_dx=False)
            dy1 = self.conv_bwd(P, G, r2, dout, dcond=dconds[:, 2 * l + 1], dc_pre=dc2, fuse_up=f1)
            if l > 0:
                f2 = dict(rec=blocks[l - 1][1], dcond=dconds[:, 2 * l - 1], need_dx=True)
            else:
                f2 = dict(rec=ctx["in_rec"], dcond=None, need_dx=False)
            dout = self.conv_bwd(P, G, r1, dy1, dc_pre=f1["dc"], dres=dout, dres_mode=L.RES_UP if up > 1 else L.RES_SAME,
                                 dcond=dconds[:, 2 * l], fuse_up=f2)
            dc2 = f2["dc"]
        if affine_stream is not None:
            affine_stream.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(affine_stream):
                demb = self._decoder_affine_bwd(P, G, ctx, dconds)
            ctx["_keep_bwd"] = (dconds,)
            dz4 = self.conv_bwd(P, G, ctx["in_rec"], dout, dc_pre=dc2, need_dx=need_dz)
            return dz4, demb
        dz4 = self.conv_bwd(P, G, ctx["in_rec"], dout, dc_pre=dc2, need_dx=need_dz)
        return dz4, self._decoder_affine_bwd(P, G, ctx, dconds)

    def _decoder_affine_bwd(self, P, G, ctx, dconds):
        demb = None
        aff = ctx["aff"]
        if isinstance(aff, dict):   # the 2n affine layers in three launches
            emb = ctx["emb"]
            naff, B, ch2, K = len(aff["names"]), emb.shape[0], dconds.shape[2], emb.shape[1]
            gtab = self._param_table("grads", aff["names"], G)
            part, demb = self.empty(naff, B, K), self.empty(B, K)
            bd = L.LinearBatchDesc()
            bd.L, bd.B, bd.N, bd.K = naff, B, ch2, K
            bd.params, bd.grads = aff["tab"].data_ptr(), gtab.data_ptr()
            bd.x, bd.x_bstride = emb.data_ptr(), emb.stride(0)
            bd.y, bd.y_bstride = dconds.data_ptr(), naff * ch2
            for i in range(naff):
                bd.x_off[i], bd.y_off[i] = 0, i * ch2
            bd.part, bd.dx = part.data_ptr(), demb.data_ptr()
            self._ck(self.lib.avc_linear_batch_dx(C.byref(bd), self.stream), "linear_batch_dx[affine]")
            self._ck(self.lib.avc_linear_batch_dw(C.byref(bd), self.stream), "linear_batch_dw[affine]")
        else:
            for i, r in enumerate(aff):
                demb = self.linear_bwd(P, G, r, dconds[:, i], dx_add=demb)
        return demb
