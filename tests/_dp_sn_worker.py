"""Worker of tests/test_gpu_spectral_norm.py: one rank of a data-parallel step of the spectral-normalised model
(RANK / WORLD_SIZE / LOCAL_RANK / MASTER_* in the environment).  Each rank seeds torch differently before building
its Solver, so the replicas only agree if Solver.build_model broadcasts parameters AND the u / v buffers."""
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import oracle.sn_oracle as sno  # noqa: E402


def main():
    out_dir, backend, per_rank = sys.argv[1], sys.argv[2], int(sys.argv[3])
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if backend == "nccl":
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist.init_process_group("gloo")
    from adaptive_voice_conversion_b200.solver import Solver
    cfg = sno.sn_config(80)
    cfg["data_loader"]["batch_size"] = per_rank
    args = types.SimpleNamespace(data_dir="synthetic", train_set="train", train_index_file="", logdir=os.path.join(out_dir, "log"),
                                 load_model=False, load_opt=False, store_model_path=os.path.join(out_dir, "model"),
                                 load_model_path=os.path.join(out_dir, "model"), summary_steps=1, save_steps=10 ** 9, tag="t", iters=0)
    torch.manual_seed(1234 + rank)      # different initial weights and u / v on every rank before the broadcast
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        solver = Solver(cfg, args)
    init = {k: v.detach().cpu().clone() for k, v in solver.model.state_dict().items()}
    n = per_rank * world
    x = torch.randn((n, 80, 128), generator=torch.Generator().manual_seed(1))
    sl = slice(rank * per_rank, (rank + 1) * per_rank)
    tr = solver.trainer
    recs = []
    for it in range(2):
        eps = torch.randn((n, 128, 16), generator=torch.Generator().manual_seed(50 + it))
        tr.step(x[sl].to(dev), 0.37, eps=eps[sl].to(dev))
        lr_, lk_, gn_ = tr.losses()
        bufs = {k: v.detach().cpu().clone() for k, v in solver.model.named_buffers()}
        recs.append(dict(loss_rec=lr_, loss_kl=lk_, grad_norm=gn_, flat_g=tr.opt.flat_g.detach().cpu().clone(),
                         flat_p=tr.opt.flat_p.detach().cpu().clone(), bufs=bufs))
    torch.save({"init": init, "steps": recs}, os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
