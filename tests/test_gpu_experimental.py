"""Opt-in paths that have NOT run end to end on a GPU yet (DESIGN.md section 6): ahead-of-time id
grouping (B200REC_GROUP_AHEAD) and the fused FM-gradient push of the sharded path
(B200REC_FUSED_PUSH; its kernel is tested on one GPU with virtual peers in
tests/test_gpu_shard_kernels.py, the exchange across GPUs is not).  Both must reproduce the default
path bit for bit:
the same kernels compute the same values, only the stream / the number of launches differs.

    B200REC_TEST_EXPERIMENTAL=1 python -m pytest tests/test_gpu_experimental.py -m gpu -q
"""
import os

import numpy as np
import pytest
import torch

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(os.environ.get("B200REC_TEST_EXPERIMENTAL") != "1",
                                 reason="not yet validated on a GPU: opt in with "
                                        "B200REC_TEST_EXPERIMENTAL=1")]


def _deepfm_step(ahead: bool):
    from paddlerec_b200 import ops
    from paddlerec_b200.rank.deepfm import net
    from paddlerec_b200 import functional as BF
    ops.set_group_ahead(ahead)
    try:
        dev = torch.device("cuda", 0)
        torch.manual_seed(7)
        V, D, B = 5000, 16, 2048
        model = net.DeepFMLayer(V, D, 13, 26, [64, 64], device=dev)
        g = torch.Generator().manual_seed(11)
        ids = torch.randint(0, V, (B, 26), generator=g).to(dev)
        dense = torch.rand(B, 13, generator=g).to(dev)
        label = (torch.rand(B, 1, generator=g) < 0.3).float().to(dev)
        out = []
        for _ in range(3):        # several steps: buffers allocated on the side stream get recycled
            for p in model.parameters():
                p.grad = None
                if hasattr(p, "grad_rows"):
                    p.grad_rows = None
            pred = model(ids, dense)
            BF.log_loss(pred, label).mean().backward()
            torch.cuda.synchronize()
            res = {"pred": pred.detach().cpu().numpy()}
            for k, p in model.named_parameters():
                sr = getattr(p, "grad_rows", None)
                if sr is not None:
                    res["g:" + k] = sr.to_dense().cpu().numpy()
                elif p.grad is not None:
                    res["g:" + k] = p.grad.cpu().numpy()
            out.append(res)
        return out
    finally:
        ops.set_group_ahead(False)


def test_group_ahead_is_bit_identical():
    serial = _deepfm_step(False)
    ahead = _deepfm_step(True)
    for a, b in zip(serial, ahead):
        assert a.keys() == b.keys()
        for k in a:
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)


def _fused_push_worker(rank, world, port, out_dir, fused):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["B200REC_P2P"] = "1"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        from paddlerec_b200 import functional as BF
        from paddlerec_b200 import sharded
        from tests.test_sharded_cpu import D, Dn, F, FC, V, _full_problem, _NoStep
        sharded.FUSED_PUSH = bool(fused)
        dev = torch.device("cuda", rank)
        B = 48
        p, ids, dense, label = _full_problem(B)
        torch.manual_seed(100 + rank)
        model = sharded.ShardedDeepFMLayer(V, D, Dn, F, FC, rank, world, device=dev)
        with torch.no_grad():
            sd = model.state_dict()
            for k, v in p.items():
                sd[k].copy_(v[rank::world] if k.startswith("fm.embedding") else v)
        per = B // world
        sl = slice(rank * per, (rank + 1) * per)
        pred = model(ids[sl].to(dev), dense[sl].to(dev))
        loss = BF.log_loss(pred, label[sl].to(dev)).mean()
        opt = sharded.DistributedOptimizer(_NoStep(), model, world)
        opt.scale_loss(loss).backward()
        opt.step()
        dW, dW1 = model.fm.table_grad_dense()
        np.savez(os.path.join(out_dir, "fp%d_%d.npz" % (int(fused), rank)),
                 dW=dW.cpu().numpy(), dW1=dW1.cpu().numpy(),
                 dense_w=model.fm.dense_w.grad.cpu().numpy())
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_fused_fm_grads_push_matches_two_kernel_path(world, tmp_path):
    import torch.multiprocessing as mp
    from tests.test_sharded_cpu import _free_port
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    for fused in (0, 1):
        mp.spawn(_fused_push_worker, args=(world, _free_port(), str(tmp_path), fused), nprocs=world,
                 join=True)
    for rank in range(world):
        a = np.load(os.path.join(str(tmp_path), "fp0_%d.npz" % rank))
        b = np.load(os.path.join(str(tmp_path), "fp1_%d.npz" % rank))
        for k in a.files:
            # same per-slot values, same owner-side merge order -> identical bits
            np.testing.assert_array_equal(a[k], b[k], err_msg="%s rank %d" % (k, rank))
