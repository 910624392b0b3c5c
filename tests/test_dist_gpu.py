"""2-rank NCCL parity of the multi-GPU path (SURVEY.md 8e: "centers after one step must equal the single-process result
on the concatenated batch"): the packed center all-reduce of losses._reduce_and_update and the gradient AVG all-reduce
of engine.SelfDistillStep.reduce_gradients, on CUDA through NCCL, against the SAME CUDA path run in one process on the
concatenated batch.  Skipped on a 1-GPU box (the CPU gloo test tests/test_dist_cpu.py covers the host logic there)."""
import os
import socket
import tempfile

import pytest
import torch

from helpers import load_golden, rel

pytestmark = pytest.mark.gpu


def _build(G, device):
    from esvit_b200 import engine
    D = G["dense"]
    meta = D["meta"]
    sp = meta["spec"]
    spec = dict(embed_dim=sp["embed_dim"], depths=list(sp["depths"]), num_heads=list(sp["num_heads"]),
                window_size=sp["window_size"], drop_path_rate=0.0)
    hp = meta["hp"]
    step, student, teacher, loss = engine.make_step(
        out_dim=meta["out_dim"], ncrops=meta["ncrops"], dense=True, device=device, lr=hp["lr"],
        weight_decay=hp["weight_decay"], clip_grad=hp["clip_grad"], freeze_last_layer=hp["freeze_last_layer"],
        img_size=sp["img_size"], head_kwargs=meta["head"], spec=spec, teacher_temp=hp["teacher_temp"])
    student.load_state_dict(D["state_dict"])
    teacher.load_state_dict(D["state_dict"])
    return step, student, teacher, loss


def _fwd_bwd(step, student, teacher, loss, crops):
    """the step body up to (and including) the gradient reduction, without the optimiser sweep"""
    from esvit_b200 import ops
    with torch.no_grad():
        t = teacher(crops[:2])
    s = student(crops)
    l = loss(s, t, 0, None)
    for p in student.parameters():
        p.grad = None
    ops.begin_step(l.device)
    try:
        l.backward()
    finally:
        ops.end_step()
    step.reduce_gradients()
    torch.cuda.synchronize()
    return float(l)


def _worker(rank, world, port, path):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        G = load_golden()
        step, student, teacher, loss = _build(G, dev)
        assert step.grad_allreduce, "make_step must enable the gradient all-reduce when a process group of size > 1 exists"
        crops = [c[rank:rank + 1].to(dev) for c in G["dense"]["crops"]]  # this rank's shard of the batch (B = 1)
        l = _fwd_bwd(step, student, teacher, loss, crops)
        want = torch.load(path, map_location="cpu", weights_only=False)
        # centers: SUM all-reduce / (rows * world) == column mean over the concatenated batch
        for name in ("center", "center_grid"):
            r = rel(getattr(loss, name), want[name])
            assert r < 1e-5, (name, r)
        # gradients: AVG over ranks of per-rank means == gradient of the mean over the concatenated batch
        bad = {}
        for n, p in student.named_parameters():
            if n not in want["grads"]:
                assert p.grad is None, n
                continue
            r = rel(p.grad, want["grads"][n])
            if r >= 2e-2 and float(want["grads"][n].norm()) > 1e-7:
                bad[n] = r
        assert not bad, bad
        # and the two ranks hold IDENTICAL reduced gradients / centers
        flat = torch.cat([p.grad.reshape(-1) for p in student.parameters() if p.grad is not None] + [loss.center.view(-1)])
        other = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(other, flat)
        assert torch.equal(other[0], other[1])
        lt = torch.tensor([l], device=dev, dtype=torch.float64)
        dist.all_reduce(lt)
        assert abs(float(lt) / world - want["loss"]) < 2e-3 * abs(want["loss"]), (float(lt) / world, want["loss"])
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_centers_and_gradients_equal_single_process():
    import torch.multiprocessing as mp
    G = load_golden()
    step, student, teacher, loss = _build(G, "cuda:0")
    crops = [c.cuda() for c in G["dense"]["crops"]]  # the concatenated batch (B = 2)
    l = _fwd_bwd(step, student, teacher, loss, crops)
    want = {"loss": l, "center": loss.center.detach().cpu(), "center_grid": loss.center_grid.detach().cpu(),
            "grads": {n: p.grad.detach().cpu() for n, p in student.named_parameters() if p.grad is not None}}
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "want.pt")
        torch.save(want, path)
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        mp.spawn(_worker, args=(2, port, path), nprocs=2, join=True)
