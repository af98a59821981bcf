"""N>1 path on CPU: world_size=2 over gloo.  The sharded DeepFM (row-cyclic tables, all-to-all of
ids/rows/grads, all-reduced dense grads) must reproduce the single-process oracle on the global
batch: predictions, dense gradients, and each rank's shard of the table gradients."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import nets
from tests import cpu_kernels

V, D, Dn, F, FC, B = 53, 8, 13, 26, [16, 8], 12


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _full_problem(B=B):
    g = torch.Generator().manual_seed(2468)
    p = {"fm.embedding.weight": torch.randn(V, D, generator=g) * 0.1,
         "fm.embedding_one.weight": torch.randn(V, 1, generator=g) * 0.1,
         "fm.dense_w": torch.randn(1, Dn, D, generator=g) * 0.1,
         "fm.dense_w_one": torch.randn(Dn, generator=g) * 0.1}
    sizes = [(F + Dn) * D] + FC + [1]
    for i in range(len(sizes) - 1):
        p["dnn.linear_%d.weight" % i] = torch.randn(sizes[i], sizes[i + 1], generator=g) / sizes[i] ** 0.5
        p["dnn.linear_%d.bias" % i] = torch.randn(sizes[i + 1], generator=g) * 0.01
    p["fm.embedding.weight"][0] = 0
    p["fm.embedding_one.weight"][0] = 0
    ids = torch.randint(0, V, (B, F), generator=g)
    ids[0, :3] = 0
    ids[5, 2] = V + 3     # out-of-range id: zeros, no gradient
    dense = torch.rand(B, Dn, generator=g)
    label = (torch.rand(B, 1, generator=g) < 0.4).float()
    return p, ids, dense, label


def _batch_for(world):
    return B if B % world == 0 else 2 * world


def _worker(rank, world, port, out_dir, fused=True):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from paddlerec_b200 import functional as BF
        from paddlerec_b200 import sharded
        B = _batch_for(world)
        p, ids, dense, label = _full_problem(B)
        torch.manual_seed(100 + rank)   # different init per rank: broadcast must fix the tower
        model = sharded.ShardedDeepFMLayer(V, D, Dn, F, FC, rank, world, device="cpu",
                                           kernels=cpu_kernels, fused_table=fused)
        with torch.no_grad():
            sd = model.state_dict()
            for k, v in p.items():
                if k in ("fm.embedding.weight", "fm.embedding_one.weight"):
                    sd[k].copy_(v[rank::world])
                else:
                    sd[k].copy_(v)
        per = B // world
        sl = slice(rank * per, (rank + 1) * per)
        pred = model(ids[sl], dense[sl])
        loss = BF.log_loss(pred, label[sl]).mean()
        opt = sharded.DistributedOptimizer(_NoStep(), model, world)
        opt.scale_loss(loss).backward()
        opt.step()   # all-reduce of the dense grads only
        res = {"pred": pred.detach().numpy(),
               "dW": model.fm.table_grad_dense()[0].numpy(),
               "dW1": model.fm.table_grad_dense()[1].numpy()}
        for k, v in model.named_parameters():
            if v.grad is not None:
                res["g:" + k] = v.grad.numpy()
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **res)
    finally:
        dist.destroy_process_group()


class _NoStep:
    def step(self):
        pass

    def clear_grad(self):
        pass


@pytest.mark.parametrize("world,fused", [(2, True), (2, False), (8, True)])
def test_sharded_deepfm_matches_oracle(world, fused, tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(world, port, str(tmp_path), fused), nprocs=world, join=True)
    B = _batch_for(world)
    p, ids, dense, label = _full_problem(B)
    pp = {k: v.double().requires_grad_(True) for k, v in p.items()}
    ids_ok = ids.clone()
    ids_ok[ids_ok >= V] = 0
    pred = nets.deepfm_forward(pp, [ids_ok[:, i:i + 1] for i in range(F)], dense.double(), len(FC))
    loss = nets.log_loss(pred, label.double()).mean()
    loss.backward()
    per = B // world
    for rank in range(world):
        r = np.load(os.path.join(str(tmp_path), "rank%d.npz" % rank))
        np.testing.assert_allclose(r["pred"], pred.detach().numpy()[rank * per:(rank + 1) * per],
                                   rtol=2e-5, atol=1e-6)
        np.testing.assert_allclose(r["dW"], pp["fm.embedding.weight"].grad.numpy()[rank::world],
                                   rtol=2e-4, atol=1e-7)
        np.testing.assert_allclose(r["dW1"], pp["fm.embedding_one.weight"].grad.numpy()[rank::world],
                                   rtol=2e-4, atol=1e-7)
        for k in pp:
            if k.startswith("fm.embedding"):
                continue
            np.testing.assert_allclose(r["g:" + k], pp[k].grad.numpy(), rtol=2e-4, atol=1e-7,
                                       err_msg=k)


def test_shard_rows_partition():
    from paddlerec_b200.sharded import shard_rows
    for V_ in (1, 7, 8, 9, 100000001):
        for w in (1, 2, 4, 8):
            assert sum(shard_rows(V_, r, w) for r in range(w)) == V_


def _dcn_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from paddlerec_b200 import functional as BF
        from paddlerec_b200 import nn as bnn
        from paddlerec_b200 import sharded
        from paddlerec_b200.rank.wide_deep import net
        from tests.util import load_golden
        g = load_golden("wide_deep")
        Vg, Dg = g["param"]["embedding.weight"].shape
        fc = [g["param"]["linear_%d.weight" % i].shape[1] for i in range(2)]
        torch.manual_seed(7 + rank)
        model = net.WideDeepLayer(Vg, Dg, 13, 26, fc, device="cpu")
        with torch.no_grad():
            for k, v in model.state_dict().items():
                v.copy_(torch.tensor(g["param"][k], dtype=torch.float32))
        # the plain gather of bnn.Embedding is CUDA-only; the sharded lookup takes the stand-in
        sharded.shard_embeddings(model, rank, world, kernels=cpu_kernels)
        ids = torch.tensor(g["in"]["ids"])
        dense = torch.tensor(g["in"]["dense"], dtype=torch.float32)
        label = torch.tensor(g["in"]["label"], dtype=torch.float32)
        Bg = ids.shape[0] // world * world
        per = Bg // world
        sl = slice(rank * per, (rank + 1) * per)
        pred = model(ids[sl], dense[sl])
        loss = BF.log_loss(pred, label[sl]).sum() / Bg       # global-batch mean
        loss.backward()
        np.savez(os.path.join(out_dir, "wd%d.npz" % rank), pred=pred.detach().numpy(),
                 dW=model.embedding.grad_rows.to_dense().numpy())
    finally:
        dist.destroy_process_group()


def test_shard_embeddings_generic_lookup(tmp_path):
    """shard_embeddings() on Wide&Deep: the generic sharded lookup (exchange + gather) must give the
    single-process predictions and table gradients (golden truncated to a multiple of world)."""
    from tests.util import load_golden, to_params, slots
    world = 2
    mp.spawn(_dcn_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    g = load_golden("wide_deep")
    p = to_params(g["param"])
    ids = torch.tensor(g["in"]["ids"])
    Bg = ids.shape[0] // world * world
    dense = torch.tensor(g["in"]["dense"], dtype=torch.float64)[:Bg]
    label = torch.tensor(g["in"]["label"], dtype=torch.float64)[:Bg]
    pred = nets.wide_deep_forward(p, slots(ids[:Bg]), dense, 2)
    nets.log_loss(pred, label).mean().backward()
    per = Bg // world
    for rank in range(world):
        r = np.load(os.path.join(str(tmp_path), "wd%d.npz" % rank))
        np.testing.assert_allclose(r["pred"], pred.detach().numpy()[rank * per:(rank + 1) * per],
                                   rtol=2e-5, atol=1e-6)
        np.testing.assert_allclose(r["dW"], p["embedding.weight"].grad.numpy()[rank::world],
                                   rtol=2e-4, atol=1e-7)


def _dlrm_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from paddlerec_b200 import functional as BF
        from paddlerec_b200 import ops, sharded
        from paddlerec_b200.rank.dlrm import net
        from tests.util import load_golden
        # K6 is CUDA-only: the stand-in takes its place for this choreography test
        ops.raw_dot_interact_fwd = cpu_kernels.raw_dot_interact_fwd
        ops.raw_dot_interact_bwd = cpu_kernels.raw_dot_interact_bwd
        g = load_golden("dlrm_pairs")
        Vg, Dg = g["param"]["embedding.weight"].shape
        model = net.DLRMLayer(13, [32, 16, 8], Vg, Dg, [32, 16, 2], 26, device="cpu")
        sd = model.state_dict()
        with torch.no_grad():
            for k, v in g["param"].items():
                if not (k.endswith("._mean") or k.endswith("._variance")):
                    sd[k].copy_(torch.tensor(v, dtype=torch.float32))
        sharded.shard_embeddings(model, rank, world, kernels=cpu_kernels)
        model.train()
        ids = torch.tensor(g["in"]["ids"])
        dense = torch.tensor(g["in"]["dense"], dtype=torch.float32)
        label = torch.tensor(g["in"]["label"])
        Bg = ids.shape[0] // world * world
        per = Bg // world
        sl = slice(rank * per, (rank + 1) * per)
        pred = model(ids[sl], dense[sl])
        loss = BF.softmax_cross_entropy(pred, label[sl]).sum() / Bg
        loss.backward()
        np.savez(os.path.join(out_dir, "dlrm%d.npz" % rank), pred=pred.detach().numpy(),
                 dW=model.embedding.grad_rows.to_dense().numpy(),
                 dtop=model.top_mlp.dense_0.weight.grad.numpy())
    finally:
        dist.destroy_process_group()


def test_sharded_dlrm_matches_per_rank_oracle(tmp_path):
    """DLRM on a row-sharded table (generic exchange + K6 stand-in).  BatchNorm normalises with each
    rank's LOCAL batch statistics — as the reference's collective mode does — so the oracle is run on
    each rank's slice; the table gradient of an owner is the sum of both ranks' contributions."""
    from tests.util import load_golden, to_params, slots
    world = 2
    mp.spawn(_dlrm_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    g = load_golden("dlrm_pairs")
    ids = torch.tensor(g["in"]["ids"])
    Bg = ids.shape[0] // world * world
    per = Bg // world
    dW = 0
    for rank in range(world):
        p = to_params({k: v for k, v in g["param"].items()
                       if not (k.endswith("._mean") or k.endswith("._variance"))})
        sl = slice(rank * per, (rank + 1) * per)
        pred = nets.dlrm_forward(p, slots(ids[sl]), torch.tensor(g["in"]["dense"])[sl], n_bot=3, n_top=3)
        lse = torch.logsumexp(pred, 1) - pred.gather(1, torch.tensor(g["in"]["label"])[sl]).squeeze(1)
        (lse.sum() / Bg).backward()
        r = np.load(os.path.join(str(tmp_path), "dlrm%d.npz" % rank))
        np.testing.assert_allclose(r["pred"], pred.detach().numpy(), rtol=2e-4, atol=2e-5)
        np.testing.assert_allclose(r["dtop"], p["top_mlp.dense_0.weight"].grad.numpy(), rtol=2e-3, atol=1e-6)
        dW = dW + p["embedding.weight"].grad.numpy()
    for rank in range(world):
        r = np.load(os.path.join(str(tmp_path), "dlrm%d.npz" % rank))
        np.testing.assert_allclose(r["dW"], dW[rank::world], rtol=2e-3, atol=1e-6)


def _clip_worker(rank, world, port, out_dir):
    """One SGD step with ClipGradByGlobalNorm under DistributedOptimizer on a row-sharded
    Wide&Deep: the clip scale must come from the GLOBAL gradient norm (dense + every shard)."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from paddlerec_b200 import functional as BF
        from paddlerec_b200 import ops, optim, sharded
        from paddlerec_b200.rank.wide_deep import net
        from tests.util import load_golden
        ops.raw_sparse_sgd = cpu_kernels.raw_sparse_sgd
        g = load_golden("wide_deep")
        Vg, Dg = g["param"]["embedding.weight"].shape
        fc = [g["param"]["linear_%d.weight" % i].shape[1] for i in range(2)]
        model = net.WideDeepLayer(Vg, Dg, 13, 26, fc, device="cpu")
        with torch.no_grad():
            for k, v in model.state_dict().items():
                v.copy_(torch.tensor(g["param"][k], dtype=torch.float32))
        sharded.shard_embeddings(model, rank, world, kernels=cpu_kernels)
        ids = torch.tensor(g["in"]["ids"])
        dense = torch.tensor(g["in"]["dense"], dtype=torch.float32)
        label = torch.tensor(g["in"]["label"], dtype=torch.float32)
        Bg = ids.shape[0] // world * world
        per = Bg // world
        sl = slice(rank * per, (rank + 1) * per)
        inner = optim.SGD(0.5, model.parameters(), grad_clip=optim.ClipGradByGlobalNorm(CLIP))
        opt = sharded.DistributedOptimizer(inner, model, world)
        pred = model(ids[sl], dense[sl])
        loss = BF.log_loss(pred, label[sl]).mean()
        opt.scale_loss(loss).backward()
        opt.step()
        out = {k: v.detach().numpy() for k, v in model.state_dict().items()}
        np.savez(os.path.join(out_dir, "clip%d.npz" % rank), **out)
    finally:
        dist.destroy_process_group()


CLIP = 0.02


def test_sharded_global_norm_clip_is_global(tmp_path):
    """ADVICE r1: the clip scale under sharding must use the norm over ALL shards (one scalar
    all-reduce), otherwise the replicated dense parameters diverge between ranks."""
    from tests.util import load_golden, to_params, slots
    world = 2
    mp.spawn(_clip_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    g = load_golden("wide_deep")
    p = to_params(g["param"])
    ids = torch.tensor(g["in"]["ids"])
    Bg = ids.shape[0] // world * world
    dense = torch.tensor(g["in"]["dense"], dtype=torch.float64)[:Bg]
    label = torch.tensor(g["in"]["label"], dtype=torch.float64)[:Bg]
    pred = nets.wide_deep_forward(p, slots(ids[:Bg]), dense, 2)
    nets.log_loss(pred, label).mean().backward()
    norm = float(sum((v.grad ** 2).sum() for v in p.values() if v.grad is not None) ** 0.5)
    assert norm > 2 * CLIP          # the clip is active, so a rank-local norm would show
    scale = CLIP / max(norm, CLIP)
    r = [np.load(os.path.join(str(tmp_path), "clip%d.npz" % k)) for k in range(world)]
    for k, v in p.items():
        want = (v.detach() - 0.5 * scale * v.grad).numpy()
        if k == "embedding.weight":
            for rank in range(world):
                np.testing.assert_allclose(r[rank][k], want[rank::world], rtol=1e-5, atol=1e-7)
        else:
            np.testing.assert_array_equal(r[0][k], r[1][k])          # replicas stay identical
            np.testing.assert_allclose(r[0][k], want, rtol=1e-5, atol=1e-7, err_msg=k)


def _exchange_blocks(blocks, recv_lens):
    """Variable-size all-to-all of int64 blocks (gloo has all_to_all_single only)."""
    out = torch.empty(sum(recv_lens), dtype=torch.int64)
    dist.all_to_all_single(out, torch.cat(blocks), recv_lens, [b.numel() for b in blocks])
    return list(out.split(recv_lens))


def _tables_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from paddlerec_b200 import sharded
        Vt, n = 1000, 517
        ex = sharded.ShardExchange(Vt, rank, world, kernels=cpu_kernels)
        ex.p2p_cols = 4          # forces the segment / destination tables of the peer-memory exchange
        g = torch.Generator().manual_seed(900 + rank)
        ids = torch.randint(0, Vt, (n,), generator=g)
        ids[:5] = torch.tensor([0, Vt + 3, -1, rank, Vt - 1])      # padding, out of range, edge rows
        send_ids, perm, inv_perm, both, tables = ex._bucketize_and_count(ids)
        counts, recv_counts = both[0], both[1]
        recv_ids = torch.empty(int(recv_counts.sum()), dtype=torch.int64)
        dist.all_to_all_single(recv_ids, send_ids, recv_counts.tolist(), counts.tolist())
        # --- what b200rec_shard_gather_push does: the owner stores row i of its segment for requester
        # r at row dst_pull[r] + i of r's buffer.  Row content here = the global id it stands for.
        rows = torch.where(recv_ids >= 0, recv_ids * world + rank, torch.full_like(recv_ids, -7))
        seg, dst = tables["recv_seg"], tables["dst_pull"]
        blocks = [torch.cat([dst[r:r + 1], rows[int(seg[r]):int(seg[r + 1])]]) for r in range(world)]
        got = _exchange_blocks(blocks, [1 + int(counts[o]) for o in range(world)])
        buf = torch.full((n,), -99, dtype=torch.int64)
        for o in range(world):
            d = int(got[o][0])
            buf[d:d + int(counts[o])] = got[o][1:]
        valid = (ids >= 0) & (ids < Vt)
        want = torch.where(valid, ids, torch.full_like(ids, -7))
        assert torch.equal(buf[perm], want), "pull tables"
        # --- b200rec_shard_push_rows: slot k of owner o's bucket goes to row dst_push[o] + k - send_seg[o]
        # of o's gradient buffer; the owner expects requester r's rows at recv_seg[r].
        sseg, dpush = tables["send_seg"], tables["dst_push"]
        payload = inv_perm.to(torch.int64) * world + rank          # (position, requester) tag per slot
        blocks = [torch.cat([dpush[o:o + 1], payload[int(sseg[o]):int(sseg[o + 1])]])
                  for o in range(world)]
        got = _exchange_blocks(blocks, [1 + int(recv_counts[r]) for r in range(world)])
        gbuf = torch.full((int(recv_counts.sum()),), -99, dtype=torch.int64)
        for r in range(world):
            d = int(got[r][0])
            assert d == int(seg[r]), "push destination != owner's receive segment"
            gbuf[d:d + int(recv_counts[r])] = got[r][1:]
        assert (gbuf >= 0).all()
        for r in range(world):      # every row of requester r's segment really came from r
            assert ((gbuf[int(seg[r]):int(seg[r + 1])] % world) == r).all()
        with open(os.path.join(out_dir, "ok%d" % rank), "w") as f:
            f.write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 8])
def test_peer_memory_exchange_tables(world, tmp_path):
    """The device tables that steer the peer-memory exchange (send_seg / recv_seg / dst_pull /
    dst_push of ShardExchange._bucketize_and_count), replayed with gloo: rows land where K1's `perm`
    expects them, gradient rows land in the owner's receive segments.  The kernels that consume
    these tables are tested on one GPU, from the same formulas, in tests/test_gpu_shard_kernels.py."""
    mp.spawn(_tables_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(os.path.join(str(tmp_path), "ok%d" % r)) for r in range(world))


class _HostPeer:
    """PeerBuffers made of shared-memory host tensors: every rank holds every rank's buffer, a store
    into `ptrs[r]` is a store into rank r's memory, the publishing barrier is a gloo barrier."""

    def __init__(self, bufs, rank, cap, cols, world):
        self.cap, self.cap_g, self.cols, self.world = cap, 2 * cap, cols, world
        self.rows, self.grads = bufs[rank][:cap], bufs[rank][cap:]
        self.rows_ptrs = [b[:cap] for b in bufs]
        self.grads_ptrs = [b[cap:] for b in bufs]

    def publish_rows(self):
        dist.barrier()

    def publish_grads(self):
        dist.barrier()


def _peer_worker(rank, world, port, out_dir, bufs, cap, fused_push):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from paddlerec_b200 import functional as BF
        from paddlerec_b200 import sharded
        sharded.FUSED_PUSH = bool(fused_push)
        B = _batch_for(world)
        p, ids, dense, label = _full_problem(B)
        torch.manual_seed(100 + rank)
        model = sharded.ShardedDeepFMLayer(V, D, Dn, F, FC, rank, world, device="cpu",
                                           kernels=cpu_kernels, fused_table=True)
        cols = model.fm._fused.grad_cols
        model.fm.exchange.inject_peer(_HostPeer(bufs, rank, cap, cols, world), cols)
        calls = {"gather_push": 0, "push_rows": 0, "fm_grads_push": 0}
        for name in calls:        # count what the exchange really called

            def counted(*a, _f=getattr(cpu_kernels, "raw_shard_" + name), _n=name, **kw):
                calls[_n] += 1
                return _f(*a, **kw)
            setattr(cpu_kernels, "raw_shard_" + name, counted)
        with torch.no_grad():
            sd = model.state_dict()
            for k, v in p.items():
                sd[k].copy_(v[rank::world] if k.startswith("fm.embedding") else v)
        per = B // world
        sl = slice(rank * per, (rank + 1) * per)
        res = {}
        for step in range(2):          # twice: the buffers are reused, stale rows must not leak
            for q in model.parameters():
                q.grad = None
            model.fm._fused.weight.grad_rows = None
            pred = model(ids[sl], dense[sl])
            loss = BF.log_loss(pred, label[sl]).mean()
            opt = sharded.DistributedOptimizer(_NoStep(), model, world)
            opt.scale_loss(loss).backward()
            opt.step()
            dist.barrier()
        want = {"gather_push": 2, "push_rows": 0 if fused_push else 2,
                "fm_grads_push": 2 if fused_push else 0}
        assert calls == want, calls          # the peer-memory path ran, not the all-to-all fallback
        res = {"pred": pred.detach().numpy(),
               "dW": model.fm.table_grad_dense()[0].numpy(),
               "dW1": model.fm.table_grad_dense()[1].numpy()}
        for k, v in model.named_parameters():
            if v.grad is not None:
                res["g:" + k] = v.grad.numpy()
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,fused_push", [(2, False), (2, True), (8, False), (8, True)])
def test_peer_memory_choreography_on_host_buffers(world, fused_push, tmp_path):
    """The peer-memory pull / push of ShardExchange (and, with fused_push, the one-kernel
    FM-gradient push) replayed on shared host tensors: same oracle, same tolerances as the all-to-all
    path.  Covers the host logic (tables, buffer offsets, barriers, zero-segment K2 call) with the
    torch stand-ins of tests/cpu_kernels.py.  The CUDA kernels themselves are compared with those
    stand-ins and with float64 references on one GPU, with virtual peers, by
    tests/test_gpu_shard_kernels.py; tests/test_sharded_gpu.py runs them across 2 or more GPUs."""
    B = _batch_for(world)
    cols = (D + 1 + 3) // 4 * 4
    cap = B // world * F + 8
    bufs = [torch.full((3 * cap, cols), float("nan")).share_memory_() for _ in range(world)]
    mp.spawn(_peer_worker, args=(world, _free_port(), str(tmp_path), bufs, cap, fused_push),
             nprocs=world, join=True)
    p, ids, dense, label = _full_problem(B)
    pp = {k: v.double().requires_grad_(True) for k, v in p.items()}
    ids_ok = ids.clone()
    ids_ok[ids_ok >= V] = 0
    pred = nets.deepfm_forward(pp, [ids_ok[:, i:i + 1] for i in range(F)], dense.double(), len(FC))
    nets.log_loss(pred, label.double()).mean().backward()
    per = B // world
    for rank in range(world):
        r = np.load(os.path.join(str(tmp_path), "rank%d.npz" % rank))
        np.testing.assert_allclose(r["pred"], pred.detach().numpy()[rank * per:(rank + 1) * per],
                                   rtol=2e-5, atol=1e-6)
        np.testing.assert_allclose(r["dW"], pp["fm.embedding.weight"].grad.numpy()[rank::world],
                                   rtol=2e-4, atol=1e-7)
        np.testing.assert_allclose(r["dW1"], pp["fm.embedding_one.weight"].grad.numpy()[rank::world],
                                   rtol=2e-4, atol=1e-7)
        for k in pp:
            if not k.startswith("fm.embedding"):
                np.testing.assert_allclose(r["g:" + k], pp[k].grad.numpy(), rtol=2e-4, atol=1e-7,
                                           err_msg=k)
