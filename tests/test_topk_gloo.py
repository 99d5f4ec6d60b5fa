"""Host logic of ``bulk.topk_sharded`` on CPU: world-size-2 gloo run with a ``torch.sort``-based top-k in place of the CUDA
kernel, equal to the single-process result (values bit for bit, indices exactly)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from sidekit_b200 import bulk


def _data(n_q, n_g, d=16):
    # small integers: every dot product is exact whatever the summation order, and there are many equal scores
    g = torch.Generator().manual_seed(5)
    return (torch.randint(-3, 4, (n_q, d), generator=g).float(), torch.randint(-3, 4, (n_g, d), generator=g).float())


def _topk_torch(queries, gallery, k, passes):
    s = queries @ gallery.T
    v, i = torch.sort(s, dim=1, descending=True, stable=True)
    return v[:, :k].contiguous(), i[:, :k].contiguous()


def _worker(rank, world, port, q, n_q, n_g, k):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    Q, G = _data(n_q, n_g)
    v, i = bulk.topk_sharded(Q, G, k, passes=3, topk_fn=_topk_torch)
    q.put((rank, v.numpy(), i.numpy()))
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("n_q,n_g,k", [(37, 50, 7), (1, 20, 3)])
def test_topk_sharded_world2_equals_single_process(n_q, n_g, k):
    Q, G = _data(n_q, n_g)
    ref_v, ref_i = _topk_torch(Q, G, k, 3)
    single_v, single_i = bulk.topk_sharded(Q, G, k, passes=3, topk_fn=_topk_torch)
    assert torch.equal(single_v, ref_v) and torch.equal(single_i, ref_i)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, n_q, n_g, k)) for r in range(2)]
    for p in procs:
        p.start()
    res = {r: (v, i) for r, v, i in (q.get(timeout=120) for _ in range(2))}
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for r in range(2):
        v, i = res[r]
        assert v.dtype == ref_v.numpy().dtype and i.dtype == ref_i.numpy().dtype
        assert (v.view("int32") == ref_v.numpy().view("int32")).all()           # bit for bit
        assert (i == ref_i.numpy()).all()


def test_topk_sharded_needs_a_fixed_pass_count():
    Q, G = _data(4, 5)
    with pytest.raises(ValueError, match="fixed pass count"):
        bulk.topk_sharded(Q, G, 2, passes=0, topk_fn=_topk_torch)
