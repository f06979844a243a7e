"""Two-GPU check (NCCL) of the sharded all-pairs matrix's backward: a row-local InfoNCE loss on each rank's row block
of aas_matrix_sharded(..., gather_to_all=False), backward on both ranks.  The forward block is bitwise the rows of the
single-GPU matrix, and every rank's gradients are bitwise those of one device's ops.aas_matrix_bwd (separate self
buffers, dk_self + dk per image).  Skipped on boxes with fewer than two GPUs."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n_images, ret):
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch.distributed as dist

    from diffsim_b200 import ops, scoring, synth

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        m = synth.SynthModel(2, 4, 256, 64, seed=2334)
        images, _ = synth.make_styles(m, (n_images + 1) // 2, 2, torch.float16, seed=8)
        images = images[:n_images]
        r0, r1 = scoring.row_block(n_images, rank, world)
        local = scoring.QKVCache.from_images(images[r0:r1], dev)
        leaves = [t.detach().requires_grad_() for t in (local.q, local.k, local.v)]
        block = scoring.aas_matrix_sharded(scoring.QKVCache(*leaves), "cosine", gather_to_all=False)
        block.retain_grad()
        targets = torch.arange(r0, r1, device=dev)
        torch.nn.functional.cross_entropy(block / 0.05, targets, reduction="sum").backward()
        torch.cuda.synchronize()
        mine = [t.detach().cpu() for t in (block, block.grad, leaves[0].grad, leaves[1].grad, leaves[2].grad)]
        parts = [None] * world
        dist.all_gather_object(parts, mine)
        if rank == 0:
            block_all, d_all, dq, dk, dv = (torch.cat([p[i] for p in parts]).to(dev) for i in range(5))
            whole = scoring.QKVCache.from_images(images, dev)
            with torch.no_grad():
                ref_dm = ops.aas_matrix(whole.q, whole.k, whole.v, whole.k, whole.v, "cosine")
            grads = [torch.zeros(t.shape, dtype=torch.float32, device=dev)   # separate self buffers
                     for t in (whole.q, whole.k, whole.v, whole.k, whole.v)]
            rq, rks, rvs, rk, rv = ops.aas_matrix_bwd(whole.q, whole.k, whole.v, whole.k, whole.v, d_all, "cosine",
                                                      grads=grads)
            ret["block_equal"] = bool(torch.equal(block_all, ref_dm))
            ret["dq_equal"] = bool(torch.equal(dq, rq.half()))
            ret["dk_equal"] = bool(torch.equal(dk, (rks + rk).half()))
            ret["dv_equal"] = bool(torch.equal(dv, (rvs + rv).half()))
            ret["nonzero"] = all(float(t.float().abs().sum()) > 0 for t in (dq, dk, dv))
    finally:
        dist.barrier()
        dist.destroy_process_group()


@pytest.mark.parametrize("n_images", [8, 7])
def test_sharded_matrix_backward_on_two_gpus(n_images):
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import torch.multiprocessing as mp

    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), n_images, ret), nprocs=2, join=True)
    assert ret["block_equal"], "forward block"
    assert ret["nonzero"]
    assert ret["dq_equal"] and ret["dk_equal"] and ret["dv_equal"], dict(ret)
