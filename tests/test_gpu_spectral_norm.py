"""GPU: the spectral-normalised decoder (Decoder.sn: True).

* the two kernels of csrc/spectral_norm.cu against float64 torch on random tables (odd shapes included);
* AE / Solver / Inferencer with sn against the fixtures written by the unmodified reference with sn: True
  (oracle/make_golden_sn.py): outputs, losses, gradients, sigma and the u / v trajectory;
* graph replay == eager, checkpoints, and a two-rank step.
"""
import os
import socket
import subprocess
import sys
import types

import pytest
import torch

import oracle.ae_oracle as orc
import oracle.sn_oracle as sno
from oracle.make_golden import reference_eps

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
REL = 1e-3
SHAPES = [(80, 128), (512, 128), (256, 640), (128, 640), (7, 13), (1, 1), (33, 1000), (1000, 3), (2, 4097)]


@pytest.fixture(params=["fp32", "tf32"])
def precision(request, monkeypatch):
    monkeypatch.setenv("AVC_PRECISION", request.param)
    return request.param


def tol(precision, fp32, tf32):
    return fp32 if precision == "fp32" else tf32


def relerr(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def rel_l2(a, b):
    a, b = a.detach().double().cpu().flatten(), b.detach().double().cpu().flatten()
    return float((a - b).norm() / (b.norm() + 1e-30))


def load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), weights_only=False)


def x_of(fx):
    return torch.randn(fx["x_shape"], generator=torch.Generator().manual_seed(fx["x_seed"]))


def eps_of(rec):
    """The reference's N(0,1) draw of a step, regenerated from its seed (the fixtures do not store it)."""
    return reference_eps(rec["eps_shape"], rec["eps_seed"])


# --------------------------------------------------------------------------- kernels
class _Table:
    def __init__(self, shapes, seed):
        g = torch.Generator().manual_seed(seed)
        self.layers = []
        for r, c in shapes:
            w = torch.randn((r, c), generator=g) / c ** 0.5
            u = torch.nn.functional.normalize(torch.randn(r, generator=g), dim=0, eps=1e-12)
            v = torch.nn.functional.normalize(torch.randn(c, generator=g), dim=0, eps=1e-12)
            self.layers.append(dict(w=w.cuda(), u=u.cuda(), v=v.cuda(), w_sn=torch.full((r, c), float("nan")).cuda(),
                                    grad=torch.randn((r, c), generator=g).cuda()))
        self.sigma = torch.full((len(shapes),), float("nan")).cuda()

    def items(self, with_grad=False):
        from adaptive_voice_conversion_b200 import _lib as L
        items = (L.SnItem * len(self.layers))()
        for i, (it, l) in enumerate(zip(items, self.layers)):
            it.w_orig, it.w_sn, it.u, it.v = l["w"].data_ptr(), l["w_sn"].data_ptr(), l["u"].data_ptr(), l["v"].data_ptr()
            it.sigma = self.sigma.data_ptr() + 4 * i
            it.grad = l["grad"].data_ptr() if with_grad else None
            it.rows, it.cols = l["w"].shape
        return torch.frombuffer(bytearray(bytes(items)), dtype=torch.uint8).cuda()

    def fwd(self, update):
        from adaptive_voice_conversion_b200 import _lib as L
        tab = self.items()
        L.check(L.load().avc_spectral_norm_fwd(tab.data_ptr(), len(self.layers), int(update),
                                               torch.cuda.current_stream().cuda_stream), "sn_fwd")
        torch.cuda.synchronize()

    def bwd(self):
        from adaptive_voice_conversion_b200 import _lib as L
        tab = self.items(with_grad=True)
        L.check(L.load().avc_spectral_norm_bwd(tab.data_ptr(), len(self.layers), torch.cuda.current_stream().cuda_stream), "sn_bwd")
        torch.cuda.synchronize()


def _ref64(w, u, v, update):
    w, u, v = w.double().cpu(), u.double().cpu(), v.double().cpu()
    if update:
        v = torch.nn.functional.normalize(w.t() @ u, dim=0, eps=1e-12)
        u = torch.nn.functional.normalize(w @ v, dim=0, eps=1e-12)
    sigma = torch.dot(u, w @ v)
    return u, v, sigma, w / sigma


@pytest.mark.parametrize("update", [1, 0])
def test_kernel_fwd_vs_float64(update):
    t = _Table(SHAPES, seed=3)
    if not update:
        # eval mode reads u, v that training left behind; random ones can make u . (W v) a cancellation near zero
        t.fwd(1)
    before = [(l["u"].clone(), l["v"].clone()) for l in t.layers]
    t.fwd(update)
    for i, (l, (u0, v0)) in enumerate(zip(t.layers, before)):
        u, v, sigma, wsn = _ref64(l["w"], u0, v0, update)
        assert abs(float(t.sigma[i]) - float(sigma)) / abs(float(sigma)) < 1e-6, (SHAPES[i], float(t.sigma[i]), float(sigma))
        assert relerr(l["w_sn"], wsn) < 1e-6, SHAPES[i]
        if update:
            assert relerr(l["u"], u) < 1e-6 and relerr(l["v"], v) < 1e-6, SHAPES[i]
        else:
            assert torch.equal(l["u"], u0) and torch.equal(l["v"], v0), SHAPES[i]


def test_kernels_are_bitwise_deterministic():
    outs = []
    for _ in range(2):
        t = _Table(SHAPES, seed=4)
        t.fwd(1)
        t.fwd(1)
        t.bwd()
        outs.append([torch.cat([l[k].flatten() for k in ("u", "v", "w_sn", "grad")]).cpu() for l in t.layers] + [t.sigma.cpu()])
    assert all(torch.equal(a, b) for a, b in zip(*outs))


def test_kernel_bwd_vs_autograd():
    t = _Table(SHAPES, seed=5)
    t.fwd(1)
    dw = [l["grad"].clone() for l in t.layers]
    t.bwd()
    for l, g in zip(t.layers, dw):
        w = l["w"].double().cpu().requires_grad_(True)
        u, v = l["u"].double().cpu(), l["v"].double().cpu()     # constants: the vectors the forward left behind
        wsn = w / torch.dot(u, w @ v)
        (wsn * g.double().cpu()).sum().backward()
        assert rel_l2(l["grad"], w.grad) < 1e-5, tuple(w.shape)


# --------------------------------------------------------------------------- models vs the reference
def make_model(c_in):
    from adaptive_voice_conversion_b200.model import AE
    cfg = sno.sn_config(c_in)
    m = AE(cfg)
    m.load_state_dict(sno.init_state(cfg, seed=0), strict=True)
    return m.cuda(), cfg


def assert_uv(model, uv, t, what=""):
    bufs = dict(model.named_buffers())
    for layer, (u, v) in uv.items():
        assert relerr(bufs[layer + ".weight_u"], u) < t and relerr(bufs[layer + ".weight_v"], v) < t, (what, layer)


@pytest.mark.parametrize("name", ["train_c80_sn_b4.pt", "train_c512_sn_b2.pt"])
def test_forward_backward_vs_reference_fixture(golden_dir, name, precision):
    """AE.forward in training mode (one power iteration) + loss.backward() through the autograd path."""
    fx = load(golden_dir, name)
    rec = fx["steps"][0]
    model, cfg = make_model(fx["c_in"])
    x = x_of(fx).cuda()
    mu, ls, emb, dec = model(x, eps=eps_of(rec).cuda())
    for k, v in (("mu", mu), ("log_sigma", ls), ("emb", emb), ("dec", dec)):
        assert relerr(v, rec[k]) < tol(precision, REL, 8e-3), (k, relerr(v, rec[k]))
    # the iteration reads fp32 weight_orig: TF32 does not enter
    assert relerr(model.sigma(x.device), rec["sigma"]) < 1e-5
    assert_uv(model, fx["uv"][1], 1e-5)
    loss_rec = torch.nn.L1Loss()(dec, x)
    loss_kl = 0.5 * torch.mean(torch.exp(ls) + mu ** 2 - 1 - ls)
    assert abs(float(loss_rec) - float(rec["loss_rec"])) / float(rec["loss_rec"]) < REL
    loss = cfg["lambda"]["lambda_rec"] * loss_rec + fx["lambda_kl"] * loss_kl
    loss.backward()
    grads = {k: p.grad for k, p in model.named_parameters()}
    gl2 = torch.stack([grads[k].norm() for k in fx["names"]]).cpu()
    assert torch.allclose(gl2, rec["grad_l2"], rtol=tol(precision, 3e-2, 2e-1), atol=1e-5)
    for k, g in rec["grad_small"].items():
        if float(g.norm()) > 1e-4:
            assert rel_l2(grads[k], g) < tol(precision, 5e-2, 3e-1), (k, rel_l2(grads[k], g))
    total = torch.sqrt(sum((g.double() ** 2).sum() for g in grads.values()))
    assert abs(float(total) - float(rec["grad_norm"])) / float(rec["grad_norm"]) < tol(precision, 5e-3, 3e-2)
    model.engine(x.device).check_tc_status()


def _solver_args(tmp_path, name="model"):
    return types.SimpleNamespace(data_dir="synthetic", train_set="train", train_index_file="", logdir=str(tmp_path / "log"),
                                 load_model=False, load_opt=False, store_model_path=str(tmp_path / name),
                                 load_model_path=str(tmp_path / name), summary_steps=1, save_steps=1000, tag="t", iters=0)


def _solver(tmp_path, c_in, batch, name="model"):
    import contextlib, io
    from adaptive_voice_conversion_b200.solver import Solver
    cfg = sno.sn_config(c_in)
    cfg["data_loader"]["batch_size"] = batch
    with contextlib.redirect_stdout(io.StringIO()):
        solver = Solver(cfg, _solver_args(tmp_path, name))
    solver.model.load_state_dict(sno.init_state(cfg, seed=0), strict=True)
    return solver, cfg


def test_solver_steps_vs_reference_fixture(tmp_path, golden_dir, precision):
    """Solver.ae_step over the fixture's 3 Adam steps: losses, grad_norm, per-tensor gradients, sigma, u, v and the
    post-step weights."""
    fx = load(golden_dir, "train_c80_sn_b4.pt")
    solver, cfg = _solver(tmp_path, 80, 4)
    x = x_of(fx)
    for i, rec in enumerate(fx["steps"]):
        meta = solver.ae_step(x, fx["lambda_kl"], eps=eps_of(rec).cuda())
        t_ = REL if i == 0 else 2e-2          # Adam drift after step 1 (tests/test_gpu_model.py)
        assert abs(meta["loss_rec"] - float(rec["loss_rec"])) / float(rec["loss_rec"]) < t_, (i, meta)
        assert abs(meta["loss_kl"] - float(rec["loss_kl"])) / float(rec["loss_kl"]) < t_, (i, meta)
        assert abs(meta["grad_norm"] - float(rec["grad_norm"])) / float(rec["grad_norm"]) < tol(precision, 10 * t_, 5e-2), (i, meta)
        assert relerr(solver.model.sigma(solver.trainer.dev), rec["sigma"]) < (1e-5 if i == 0 else t_), i
        G = solver.trainer.G
        gl2 = torch.stack([G[k].norm() for k in fx["names"]]).cpu()
        assert torch.allclose(gl2, rec["grad_l2"], rtol=tol(precision, 3e-2, 2e-1) if i == 0 else 3e-1, atol=1e-5), i
        if i == 0:
            for k, g in rec["grad_small"].items():
                if float(g.norm()) > 1e-4:
                    assert rel_l2(G[k], g) < tol(precision, 5e-2, 3e-1), (k, rel_l2(G[k], g))
        p = dict(solver.model.named_parameters())
        pl2 = torch.stack([p[k].detach().norm() for k in fx["names"]]).cpu()
        assert torch.allclose(pl2, rec["param_l2_after"], rtol=tol(precision, 1e-4, 2e-3) if i == 0 else 3e-3), i
        if i + 1 in fx["uv"]:
            assert_uv(solver.model, fx["uv"][i + 1], 1e-5 if i == 0 else t_, i)
    solver.trainer.eng.check_tc_status()


def test_solver_step_b256_vs_oracle(tmp_path):
    """Full size: one Solver.ae_step at batch 256 against the oracle's step on the same x / eps."""
    B = 256
    solver, cfg = _solver(tmp_path, 80, B)
    sd = sno.init_state(cfg, seed=0)
    st = orc.AdamState(sno.params_of(sd))
    x = torch.randn((B, 80, 128), generator=torch.Generator().manual_seed(1))
    eps = torch.randn((B, 128, 16), generator=torch.Generator().manual_seed(2))
    res = sno.ae_train_step(sd, st, cfg, x, eps, 1.0)
    meta = solver.ae_step(x, 1.0, eps=eps.cuda())
    prec = solver.trainer.eng.precision
    assert abs(meta["loss_rec"] - res["loss_rec"]) / res["loss_rec"] < REL
    assert abs(meta["loss_kl"] - res["loss_kl"]) / res["loss_kl"] < REL
    assert abs(meta["grad_norm"] - res["grad_norm"]) / res["grad_norm"] < tol(prec, 1e-2, 3e-2)
    assert relerr(solver.model.sigma(solver.trainer.dev), res["outs"]["sigma"]) < 1e-5
    G = solver.trainer.G
    num = den = 0.0
    for k, r in res["grads"].items():
        num += float((G[k].double().cpu() - r.double()).pow(2).sum())
        den += float(r.double().pow(2).sum())
    assert (num / den) ** 0.5 < tol(prec, 1e-2, 1e-1)
    bufs = dict(solver.model.named_buffers())
    for k in bufs:
        assert relerr(bufs[k], sd[k]) < 1e-5, k
    after = dict(solver.model.named_parameters())
    lr = cfg["optimizer"]["lr"]
    for k in res["grads"]:
        assert float((after[k].detach().cpu() - sd[k]).abs().max()) <= 2.05 * lr, k
    solver.trainer.eng.check_tc_status()


def test_inference_eval_mode_vs_reference_fixture(golden_dir, precision):
    """Eval mode: sigma from the stored u, v (nothing written), AE.inference and Inferencer.inference_batch."""
    from adaptive_voice_conversion_b200.inference import Inferencer
    fx = load(golden_dir, "infer_c80_sn.pt")
    model, cfg = make_model(fx["c_in"])
    model.eval()
    before = {k: v.clone() for k, v in model.named_buffers()}
    x, xc = fx["x"].cuda(), fx["x_cond"].cuda()
    dec = model.inference(x, xc)
    assert dec.shape == fx["dec"].shape
    assert relerr(dec, fx["dec"]) < tol(precision, REL, 8e-3)
    # (1/sigma > 1 scales up every decoder layer, and with it the TF32 rounding of the stack: 5e-3, not 3e-3)
    assert rel_l2(dec, fx["dec"]) < tol(precision, 1e-4, 5e-3)
    assert relerr(model.sigma(x.device), fx["sigma"]) < 1e-6
    assert all(torch.equal(v, before[k]) for k, v in model.named_buffers())
    args = types.SimpleNamespace(attr=None, model=None, source=None, target=None, output=None, sample_rate=24000)
    inf = Inferencer(cfg, args)
    inf.model.load_state_dict(sno.init_state(cfg, seed=0), strict=True)
    out = inf.inference_batch(x, xc)       # captures a graph
    out2 = inf.inference_batch(x, xc)      # replays it
    assert relerr(out, dec) < 1e-6 and torch.equal(out2, out)
    # a load that changes only u / v invalidates the captured graph
    sd = sno.init_state(cfg, seed=7)
    sd = {k: (sd[k] if k.endswith((".weight_u", ".weight_v")) else v) for k, v in sno.init_state(cfg, seed=0).items()}
    inf.model.load_state_dict(sd, strict=True)
    out3 = inf.inference_batch(x, xc)
    with torch.no_grad():
        ref3, _ = sno.ae_inference(sd, cfg, fx["x"], fx["x_cond"])
    assert relerr(out3, ref3) < tol(precision, REL, 8e-3)
    assert not torch.equal(out3, dec)


def test_train_mode_inference_iterates(golden_dir):
    """AE.inference in training mode runs the power iteration, like the reference's."""
    fx = load(golden_dir, "infer_c80_sn.pt")
    model, cfg = make_model(fx["c_in"])
    model.train()
    sd = sno.init_state(cfg, seed=0)
    with torch.no_grad():
        ref, sig = sno.ae_inference(sd, cfg, fx["x"], fx["x_cond"], update=True)
        dec = model.inference(fx["x"].cuda(), fx["x_cond"].cuda())
    assert relerr(dec, ref) < 8e-3
    assert relerr(model.sigma(dec.device), sig) < 1e-5
    bufs = dict(model.named_buffers())
    assert all(relerr(bufs[k], sd[k]) < 1e-5 for k in bufs)


# --------------------------------------------------------------------------- graph, checkpoints, DP
def test_graph_step_matches_eager(tmp_path):
    outs = []
    for use_graph in (False, True):
        solver, cfg = _solver(tmp_path, 80, 4)
        xs = [torch.randn((4, 80, 128), generator=torch.Generator().manual_seed(10 + i)).cuda() for i in range(3)]
        es = [torch.randn((4, 128, 16), generator=torch.Generator().manual_seed(20 + i)).cuda() for i in range(3)]
        if use_graph:
            solver.trainer.capture(xs[0], warmup=0, eps_example=es[0])
        rec = []
        for i in range(3):
            solver.trainer.step(xs[i], 1.0, eps=es[i])
            bufs = torch.cat([b.detach().flatten() for b in solver.model.buffers()]).cpu()
            rec.append(solver.trainer.losses() + (solver.opt.flat_g.detach().cpu().clone(), solver.opt.flat_p.detach().cpu().clone(), bufs))
        if use_graph:
            assert solver.trainer._graphs is not None
        outs.append(rec)
    for i, ((l0, k0, n0, g0, p0, b0), (l1, k1, n1, g1, p1, b1)) in enumerate(zip(*outs)):
        lt, gt = (1e-5, 1e-4) if i == 0 else (2e-3, 3e-1)
        assert abs(l0 - l1) / l0 < lt and abs(k0 - k1) / k0 < lt and abs(n0 - n1) / n0 < gt, (i, l0, l1, n0, n1)
        assert rel_l2(g1, g0) < gt and rel_l2(p1, p0) < (1e-3 if i == 0 else 5e-3), i
        if i == 0:   # the first iteration reads identical weights: the deterministic kernel gives identical vectors
            assert torch.equal(b0, b1)
        else:        # u / v follow weights that drift like p0 / p1 above
            assert rel_l2(b1, b0) < 5e-3, (i, rel_l2(b1, b0))


def test_graph_recaptures_on_mode_change(tmp_path):
    solver, cfg = _solver(tmp_path, 80, 4)
    x = torch.randn((4, 80, 128), generator=torch.Generator().manual_seed(1)).cuda()
    e = torch.randn((4, 128, 16), generator=torch.Generator().manual_seed(2)).cuda()
    solver.trainer.capture(x, warmup=0, eps_example=e)
    solver.trainer.step(x, 1.0, eps=e)
    solver.model.eval()
    u = [b.clone() for b in solver.model.buffers()]
    solver.trainer.step(x, 1.0, eps=e)        # eval mode: no power iteration, u / v untouched
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(u, solver.model.buffers()))
    solver.model.train()
    solver.trainer.step(x, 1.0, eps=e)
    torch.cuda.synchronize()
    assert not all(torch.equal(a, b) for a, b in zip(u, solver.model.buffers()))


def test_checkpoint_resume_continues_identically(tmp_path):
    """Save after 2 steps, load into a fresh Solver: its state (incl. u / v and the Adam moments) equals the saved
    one, and the next step of both lands on the same losses, sigma and u / v."""
    x = torch.randn((4, 80, 128), generator=torch.Generator().manual_seed(1))
    es = [torch.randn((4, 128, 16), generator=torch.Generator().manual_seed(30 + i)).cuda() for i in range(3)]
    s1, cfg = _solver(tmp_path, 80, 4, "a")
    for i in range(2):
        s1.ae_step(x, 1.0, eps=es[i])
    s1.save_model(1)
    ck = torch.load(str(tmp_path / "a.ckpt"), map_location="cpu")
    assert [(k, tuple(v.shape)) for k, v in ck.items()] == [(k, tuple(s)) for k, s in sno.state_shapes(cfg)]
    args = _solver_args(tmp_path, "a")
    args.load_model = True
    import contextlib, io
    from adaptive_voice_conversion_b200.solver import Solver
    with contextlib.redirect_stdout(io.StringIO()):
        s2 = Solver(cfg, args)
    for k, v in s2.model.state_dict().items():
        assert torch.equal(v.cpu(), ck[k]), k
    assert torch.equal(s2.opt.flat_m, s1.opt.flat_m) and torch.equal(s2.opt.flat_vmax, s1.opt.flat_vmax)
    m1 = s1.ae_step(x, 1.0, eps=es[2])
    m2 = s2.ae_step(x, 1.0, eps=es[2])
    for k in ("loss_rec", "loss_kl"):
        assert abs(m1[k] - m2[k]) / m1[k] < 1e-6, (k, m1, m2)
    assert torch.equal(s1.model.sigma(s1.trainer.dev), s2.model.sigma(s2.trainer.dev))
    assert all(torch.equal(a, b) for a, b in zip(s1.model.buffers(), s2.model.buffers()))


def test_stock_adam_opt_file_loads(tmp_path):
    """A .opt written by torch.optim.Adam over the reference's parameter order (bias before weight_orig) loads, and
    its moments land in the right slots of the flat buffers."""
    solver, cfg = _solver(tmp_path, 80, 4)
    sd = sno.init_state(cfg, seed=0)
    params = [torch.nn.Parameter(v.clone()) for v in sno.params_of(sd).values()]
    ref = torch.optim.Adam(params, lr=5e-4, amsgrad=True, weight_decay=1e-4)
    g = torch.Generator().manual_seed(9)
    for p in params:
        p.grad = torch.randn(p.shape, generator=g)
    ref.step()
    torch.save(ref.state_dict(), str(tmp_path / "ref.opt"))
    torch.save({**{k: p.detach() for k, p in zip(sno.params_of(sd), params)},
                **{k: v for k, v in sd.items() if k.endswith((".weight_u", ".weight_v"))}}, str(tmp_path / "ref.ckpt"))
    solver.args.load_model_path = str(tmp_path / "ref")
    solver.load_model()
    names = [n for n, _ in solver.model.named_parameters()]
    assert names == list(sno.params_of(sd))
    for i, (n, p) in enumerate(solver.model.named_parameters()):
        st = solver.opt.state[p]
        assert torch.equal(st["exp_avg"].cpu(), ref.state[params[i]]["exp_avg"]), n
        assert torch.equal(st["max_exp_avg_sq"].cpu(), ref.state[params[i]]["max_exp_avg_sq"]), n
    assert float(solver.opt.step_dev.item()) == 1.0
    meta = solver.ae_step(torch.randn((4, 80, 128)), 1.0)
    assert meta["loss_rec"] == meta["loss_rec"]      # trains on from the loaded state (finite)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_two_rank_step_equals_single_process_step(tmp_path):
    per_rank = 4
    ngpu = torch.cuda.device_count()
    backend = "nccl" if ngpu >= 2 else "gloo"
    port = _free_port()
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", LOCAL_RANK=str(rank if ngpu >= 2 else 0),
                   MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(HERE, "_dp_sn_worker.py"), str(tmp_path), backend, str(per_rank)],
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = []
    for p in procs:
        try:
            outs.append(p.communicate(timeout=600)[0])
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o[-3000:]
    r0 = torch.load(str(tmp_path / "rank0.pt"))
    r1 = torch.load(str(tmp_path / "rank1.pt"))
    assert all(torch.equal(r0["init"][k], r1["init"][k]) for k in r0["init"])    # parameters AND u / v broadcast
    # the single process on the concatenated batch, from the same initial state
    solver, cfg = _solver(tmp_path, 80, 2 * per_rank, "single")
    solver.model.load_state_dict(r0["init"], strict=True)
    x = torch.randn((2 * per_rank, 80, 128), generator=torch.Generator().manual_seed(1)).cuda()
    for it in range(2):
        eps = torch.randn((2 * per_rank, 128, 16), generator=torch.Generator().manual_seed(50 + it)).cuda()
        solver.trainer.step(x, 0.37, eps=eps)
        _, _, gn = solver.trainer.losses()
        a, b = r0["steps"][it], r1["steps"][it]
        assert torch.equal(a["flat_g"], b["flat_g"]) and torch.equal(a["flat_p"], b["flat_p"])
        assert all(torch.equal(a["bufs"][k], b["bufs"][k]) for k in a["bufs"])   # u / v bit-identical across ranks
        gt = 2e-4 if it == 0 else 1e-1
        assert rel_l2(0.5 * a["flat_g"], solver.opt.flat_g) < gt, it
        assert abs(a["grad_norm"] - gn) / gn < gt
        bufs = dict(solver.model.named_buffers())
        for k, v in a["bufs"].items():
            assert relerr(v, bufs[k]) < (1e-6 if it == 0 else 1e-3), (it, k)
