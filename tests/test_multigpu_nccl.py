"""2-GPU NCCL run of the row-sharded all-pairs DGG path against the unsharded single-GPU result
(skipped on a machine with fewer than two GPUs)."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from dgg_b200 import functional as K
        from dgg_b200 import sharding as S

        n, d, kc, seed = 1500, 64, 16, 77
        gen = torch.Generator().manual_seed(1)
        z0 = torch.softmax(torch.randn(n, d, generator=gen), -1)
        w = torch.randn(n, kc, generator=gen)
        rb, cnt, _ = S.row_block(n, world, rank)
        zl = z0[rb:rb + cnt].cuda().requires_grad_(True)
        t = torch.tensor([2.0], device="cuda", requires_grad=True)
        idx, y = S.sharded_allpairs_topk(zl, t, n, kc, seed=seed, noise_scale=0.3)
        (y * w[rb:rb + cnt].cuda()).sum().backward()
        S.all_reduce_grads([t])
        # unsharded reference on this rank's own GPU
        zf = z0.cuda().requires_grad_(True)
        tf = torch.tensor([2.0], device="cuda", requires_grad=True)
        idx_f, y_f = K.allpairs_topk(zf, tf, None, kc, 3, seed=seed, noise_scale=0.3)
        (y_f * w.cuda()).sum().backward()
        assert torch.equal(idx, idx_f[rb:rb + cnt]) and torch.equal(y, y_f[rb:rb + cnt])
        torch.testing.assert_close(zl.grad, zf.grad[rb:rb + cnt], rtol=1e-4, atol=1e-6)
        torch.testing.assert_close(t.grad, tf.grad, rtol=1e-4, atol=1e-5)
        ret[rank] = True
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_allpairs_matches_unsharded():
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, 29900 + os.getpid() % 90, ret), nprocs=world, join=True)
    assert all(ret.get(r) for r in range(world))
