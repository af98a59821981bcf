"""Kernel-level parity of the peer-memory exchange kernels (csrc/shard.cuh) on ONE GPU.

The kernels take `world` raw destination base pointers and store through them with plain stores.
With `world` separate receive buffers on cuda:0 standing in for the peers' NVLink mappings they run
exactly as on a multi-GPU box, minus the transport, at any world up to kMaxPeers = 16.  One process,
one stream: the "ranks" are called one after another, with no barrier, no symmetric memory and no
collective.

Every receive buffer starts as NaN.  After each call the rows the call owns must hold the expected
values and every other element (guard rows, rows of other segments, columns past the row width) must
still be NaN: over NVLink a store outside its segment lands in a peer's memory, and the sentinel is
how a test on one device sees it.  Copies are compared bit for bit, arithmetic against float64.
"""
import ctypes
import types

import pytest
import torch

from paddlerec_b200 import _lib, ops, sharded
from tests import cpu_kernels
from tests.test_gpu_kernels import make_fm_inputs, oracle_fm
from tests.util import rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda"
NAN = float("nan")
GUARD = 3       # receive-buffer rows past the last segment: must never be written
HOT = 3         # local row requested many times


# ---- virtual-peer harness ---------------------------------------------------------------------
def nan_buffers(world, rows, ld):
    """`world` receive buffers on cuda:0 and their base pointers, typed like PeerBuffers.rows_ptrs."""
    bufs = [torch.full((rows, ld), NAN, device=DEV) for _ in range(world)]
    return bufs, (ctypes.c_uint64 * world)(*[b.data_ptr() for b in bufs])


def exchange_tables(counts):
    """Segment tables of the peer-memory exchange for counts[r][o] = ids requester r sends to owner
    o, by the formulas ShardExchange._bucketize_and_count evaluates with collectives:
        send_seg_r    = [0, cumsum(counts[r])]          requester r's bucket order, by owner
        recv_seg_o[r] = sum_{r' < r} counts[r'][o]      owner o's received list, by requester
        dst_pull_o[r] = send_seg_r[o]                   where o's rows for r go in r's row buffer
        dst_push_r[o] = recv_seg_o[r]                   where r's gradient rows go in o's buffer
    Host int64 tensors, one per rank."""
    world = counts.shape[0]
    zero = torch.zeros(1, dtype=torch.int64)
    send_seg = [torch.cat([zero, counts[r].cumsum(0)]) for r in range(world)]
    recv_seg = [torch.cat([zero, counts[:, o].cumsum(0)]) for o in range(world)]
    dst_pull = [torch.stack([send_seg[r][o] for r in range(world)]) for o in range(world)]
    dst_push = [torch.stack([recv_seg[o][r] for o in range(world)]) for r in range(world)]
    return send_seg, recv_seg, dst_pull, dst_push


def count_matrix(world, seed, hi=128):
    """Random counts with the edge cases of the segment search: empty first, middle and last
    segments at the owners and in the requesters' buckets, and a peer that asks for nothing."""
    if world == 1:
        # odd, so n * (chunks per row) never fills the last block of 1024 chunks
        return torch.tensor([[1537]])
    c = torch.randint(1, hi, (world, world), generator=torch.Generator().manual_seed(seed))
    c[0, 0] = 0                    # owner 0: empty first segment; requester 0: empty first bucket
    c[world - 1, world - 1] = 0    # the same, last
    if world > 2:
        c[world // 2, :] = 0       # asks for nothing: an empty middle segment at every owner
        c[0, world // 2] = 0       # requester 0: an empty middle bucket
    return c


def assert_same_bits(got, want, what):
    """Bit-for-bit equality (NaN sentinels and the sign of zero included)."""
    if got.device != want.device:
        got, want = got.cpu(), want.cpu()
    g = got.detach().contiguous().view(torch.int32)
    w = want.detach().contiguous().view(torch.int32)
    assert g.shape == w.shape, "%s: shape %s, want %s" % (what, tuple(g.shape), tuple(w.shape))
    bad = (g != w).nonzero()
    if bad.shape[0]:
        i = tuple(bad[0].tolist())
        raise AssertionError("%s: %d of %d elements differ, first at %s: got %r, want %r"
                             % (what, bad.shape[0], g.numel(), i, float(got[i]), float(want[i])))


def row_vec(D):
    """Floats per store of the gather / push kernels (pick_row_shape)."""
    return 4 if D % 4 == 0 else (2 if D % 2 == 0 else 1)


def recv_ids_for(n, V_loc, pad, g):
    """Local rows an owner received: uniform rows plus -1 (what bucketize sends for an id out of
    range), the local padding row, V_loc (one past the shard) and one hot row repeated many times."""
    ids = torch.randint(0, V_loc, (n,), generator=g)
    u = torch.rand(n, generator=g)
    ids[u < 0.05] = -1
    ids[(u >= 0.05) & (u < 0.10)] = V_loc
    ids[(u >= 0.10) & (u < 0.15)] = pad
    ids[u >= 0.75] = HOT
    k = min(n, 4)
    ids[:k] = torch.tensor([-1, V_loc, pad, HOT])[:k]
    return ids


def gathered(shard, ids, pad, D):
    """shard[ids, :D] with the padding row and out-of-range rows as +0.0."""
    ok = (ids >= 0) & (ids < shard.shape[0]) & (ids != pad)
    return torch.where(ok.unsqueeze(1), shard[ids.clamp(0, shard.shape[0] - 1), :D], 0.0)


# ---- B.1 / B.2: gather_push and push_rows -----------------------------------------------------
D_GRID = [1, 2, 3, 9, 12, 16, 20, 64, 128]      # VEC 1, 2 and 4; 128 = 32 chunks, the widest row
WORLDS = [1, 2, 3, 8, 16]


def run_gather_push(D, world, ldw, ld_dst, seed):
    g = torch.Generator().manual_seed(seed)
    counts = count_matrix(world, seed)
    send_seg, recv_seg, dst_pull, _ = exchange_tables(counts)
    n_req = counts.sum(1)                        # rows every requester receives
    cap = int(n_req.max()) + GUARD
    bufs, ptrs = nan_buffers(world, cap, ld_dst)
    want = [torch.full((cap, ld_dst), NAN) for _ in range(world)]
    stand_in = [torch.full((cap, ld_dst), NAN) for _ in range(world)]
    for o in range(world):
        V_loc = 300 + 17 * o
        pad = 7 if o % 2 == 0 else -1            # -1: no padding row on this rank
        shard = torch.randn(V_loc, ldw, generator=g)
        ids = recv_ids_for(int(recv_seg[o][-1]), V_loc, pad, g)
        ops.raw_shard_gather_push(shard.to(DEV), ids.to(DEV), pad, D, recv_seg[o].to(DEV),
                                  dst_pull[o].to(DEV), ptrs, ld_dst, world)
        rows = gathered(shard, ids, pad, D)
        for r in range(world):
            a, b, d = int(recv_seg[o][r]), int(recv_seg[o][r + 1]), int(dst_pull[o][r])
            want[r][d:d + b - a, :D] = rows[a:b]
        cpu_kernels.raw_shard_gather_push(shard, ids, pad, D, recv_seg[o], dst_pull[o], stand_in,
                                          ld_dst, world)
        for r in range(world):
            got = bufs[r].cpu()
            assert_same_bits(got, want[r], "owner %d -> requester %d" % (o, r))
            assert_same_bits(stand_in[r], got, "cpu_kernels stand-in, owner %d -> requester %d"
                             % (o, r))
    for r in range(world):           # the segments tile every requester's rows: no hole, no overlap
        assert not want[r][:int(n_req[r]), :D].isnan().any()


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("D", D_GRID)
def test_gather_push(D, world):
    run_gather_push(D, world, ldw=D, ld_dst=D + row_vec(D), seed=100 * D + world)


@pytest.mark.parametrize("world", [2, 8])
def test_gather_push_fused_slot_table(world):
    """What the DeepFM pull does: the first G = fused_grad_cols(D) columns of 32-float
    [emb | w1 | pad] slots, into rows of exactly G floats."""
    D = 16
    G = ops.fused_grad_cols(D)
    run_gather_push(G, world, ldw=ops.fused_slot(D), ld_dst=G, seed=7 + world)


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("D", D_GRID)
def test_push_rows(D, world):
    seed = 200 * D + world
    g = torch.Generator().manual_seed(seed)
    counts = count_matrix(world, seed)
    send_seg, recv_seg, _, dst_push = exchange_tables(counts)
    ld = ld_dst = D + row_vec(D)                 # only the first D columns of a row travel
    cap = int(counts.sum(0).max()) + GUARD
    bufs, ptrs = nan_buffers(world, cap, ld_dst)
    want = [torch.full((cap, ld_dst), NAN) for _ in range(world)]
    stand_in = [torch.full((cap, ld_dst), NAN) for _ in range(world)]
    for r in range(world):
        rows = torch.randn(int(send_seg[r][-1]), ld, generator=g)
        ops.raw_shard_push_rows(rows.to(DEV), D, send_seg[r].to(DEV), dst_push[r].to(DEV), ptrs,
                                ld_dst, world)
        for o in range(world):
            a, b, d = int(send_seg[r][o]), int(send_seg[r][o + 1]), int(dst_push[r][o])
            want[o][d:d + b - a, :D] = rows[a:b, :D]
        cpu_kernels.raw_shard_push_rows(rows, D, send_seg[r], dst_push[r], stand_in, ld_dst, world)
        for o in range(world):
            got = bufs[o].cpu()
            assert_same_bits(got, want[o], "requester %d -> owner %d" % (r, o))
            assert_same_bits(stand_in[o], got, "cpu_kernels stand-in, requester %d -> owner %d"
                             % (r, o))
    for o in range(world):
        assert not want[o][:int(counts[:, o].sum()), :D].isnan().any()


# ---- B.3: fm_grads_push -----------------------------------------------------------------------
FM_CASES = ([(D, ops.fused_grad_cols(D), world, B, with_dfeat)
             for D in (4, 8, 16, 64) for world in (1, 2, 8, 16) for B in (1, 7, 300)
             for with_dfeat in (False, True)]
            + [(16, 24, world, B, True) for world in (2, 16) for B in (7, 300)]    # G = D + 8
            # production shape (n = 1.7 M): the grid is capped at 32 blocks per SM, so the
            # grid-stride loop runs several times
            + [(16, 20, 8, 65536, True), (16, 20, 16, 65536, False), (64, 68, 2, 65536, True)])


@pytest.mark.parametrize("D,G,world,B,with_dfeat", FM_CASES)
def test_fm_grads_push(D, G, world, B, with_dfeat):
    F, Dn, V = 26, 13, 10000
    n = B * F
    seed = 1000 * D + 100 * world + B + G + int(with_dfeat)
    gd = torch.Generator(device=DEV).manual_seed(seed)
    ids = torch.randint(0, V, (B, F), generator=gd, device=DEV)
    ids[torch.rand(B, F, generator=gd, device=DEV) < 0.02] = V + 3    # out of range: owner 0
    feat = torch.randn(B, F + Dn, D, generator=gd, device=DEV)
    S = feat.sum(1)
    dfeat = torch.randn(B, F + Dn, D, generator=gd, device=DEV) if with_dfeat else None
    gy1 = torch.randn(B, generator=gd, device=DEV)
    gy2 = torch.randn(B, generator=gd, device=DEV)
    dense = torch.rand(B, Dn, generator=gd, device=DEV)
    _, _, inv_perm, counts_r = ops.raw_shard_bucketize(ids, world, V)
    # this requester is the last rank, so its rows land at non-zero offsets of the owners' buffers
    r = world - 1
    counts = torch.randint(0, 50, (world, world), generator=torch.Generator().manual_seed(seed))
    counts[r] = counts_r.cpu()
    send_seg, _, _, dst_push = exchange_tables(counts)
    seg, dst = send_seg[r].to(DEV), dst_push[r].to(DEV)
    ld_dst = G + 4                               # columns G.. of every row must stay NaN
    cap = int(counts.sum(0).max()) + GUARD
    fused, fused_ptrs = nan_buffers(world, cap, ld_dst)
    two, two_ptrs = nan_buffers(world, cap, ld_dst)
    ops.raw_shard_fm_grads_push(feat, S, dfeat, gy1, gy2, inv_perm, F, G, seg, dst, fused_ptrs,
                                ld_dst, world)

    # reference 1, bit for bit: the product's path without the flag, K2 with every slot its own
    # segment (ShardedFM.trivial_groups) followed by push_rows
    fm = types.SimpleNamespace(_trivial={})
    iota, num = sharded.ShardedFM.trivial_groups(fm, n, feat.device)
    dW, _, ddw, ddw1 = ops.raw_embed_fm_bwd(feat, S, dfeat, gy1, gy2, dense, iota, inv_perm, num, F,
                                            fused_cols=G)
    ops.raw_shard_push_rows(dW[:n], G, seg, dst, two_ptrs, ld_dst, world)
    for o in range(world):
        assert_same_bits(fused[o], two[o], "owner %d: fused push vs K2 + push_rows" % o)

    # reference 2: [g2*(S - feat) + dfeat | g1 | 0..] in float64, at 2e-6 of the row's scale
    p = inv_perm.long()
    b, f = p // F, p % F
    e, s, g2 = feat[b, f].double(), S[b].double(), gy2[b].double().unsqueeze(1)
    want = torch.zeros(n, G, dtype=torch.float64, device=DEV)
    want[:, :D] = g2 * (s - e)
    scale = g2.abs() * (s.abs() + e.abs())
    if dfeat is not None:
        dd = dfeat[b, f].double()
        want[:, :D] += dd
        scale += dd.abs()
    want[:, D] = gy1[b].double()
    row_scale = torch.maximum(scale.amax(1), gy1[b].double().abs())
    for o in range(world):
        a, c, d = int(send_seg[r][o]), int(send_seg[r][o + 1]), int(dst_push[r][o])
        got = fused[o][d:d + c - a]
        err = (got[:, :G].double() - want[a:c]).abs().amax(1) if c > a else row_scale[:0]
        assert bool((err <= 2e-6 * row_scale[a:c]).all()), \
            "owner %d: max error / row scale %.3g" % (o, float((err / row_scale[a:c]).max()))
        assert torch.equal(got[:, D], gy1[b[a:c]])          # g1: a copy
        assert not got[:, D + 1:G].any()                     # zero padding of the row
        outside = torch.ones_like(fused[o], dtype=torch.bool)
        outside[d:d + c - a, :G] = False
        assert bool(fused[o][outside].isnan().all()), "owner %d: store outside the segment" % o

    # the fused branch then runs K2 over zero segments for the dense-feature half only
    # (ShardedFM.zero_groups): its gradients must be the full call's, bit for bit
    zero = sharded.ShardedFM.zero_groups(fm, feat.device)
    _, _, ddw0, ddw10 = ops.raw_embed_fm_bwd(feat, S, dfeat, gy1, gy2, dense, iota, inv_perm, zero, F,
                                             fused_cols=G)
    assert_same_bits(ddw0, ddw, "ddense_w of the zero-segment K2 call")
    assert_same_bits(ddw10, ddw1, "ddense_w1 of the zero-segment K2 call")


# ---- C: the N>1 data path of the DeepFM FM block in one process --------------------------------
@pytest.mark.parametrize("world", [1, 2, 4, 8, 16])
@pytest.mark.parametrize("D", [16, 9])
def test_virtual_world_fm_block(D, world):
    """_ShardedEmbedFM forward and backward for `world` virtual ranks with the real kernels:
    bucketize, id exchange (torch.cat), gather_push into the requesters' row buffers, K1 over them;
    K2 + push_rows or the fused push into the owners' gradient buffers, owner-side group_ids +
    segment_reduce.  Two steps with different ids run through the same buffers.  D = 9 (G = 12)
    is a table the fused push does not take (D % 4 != 0): two-kernel path only."""
    F, Dn, V, Bg = 26, 13, 2000, 96
    G, slot = ops.fused_grad_cols(D), ops.fused_slot(D)
    Bp = Bg // world
    n = Bp * F
    paths = ["two_kernel", "fused"] if D % 4 == 0 else ["two_kernel"]
    _, _, W, W1, dense_w, dense_w1 = make_fm_inputs(Bg, F, Dn, D, V, seed=50 + D)
    Wf = torch.full((V, slot), 123.0)            # slot padding: travels with the rows, never read
    Wf[:, :D] = W
    Wf[:, D] = W1[:, 0]
    # row-cyclic shards; the padding id 0 is local row 0 of rank 0, no other rank has a padding row
    shards = [Wf[o::world].contiguous().to(DEV) for o in range(world)]
    pads = [0] + [-1] * (world - 1)
    V_loc = [sharded.shard_rows(V, o, world) for o in range(world)]
    assert [s.shape[0] for s in shards] == V_loc
    dw, dw1 = dense_w.reshape(Dn, D).to(DEV), dense_w1.to(DEV)
    rows_bufs, rows_ptrs = nan_buffers(world, n + GUARD, G)
    grad_bufs = {path: nan_buffers(world, Bg * F + GUARD, G) for path in paths}
    fm = types.SimpleNamespace(_trivial={})
    iota, num = sharded.ShardedFM.trivial_groups(fm, n, torch.device(DEV))
    zero = sharded.ShardedFM.zero_groups(fm, torch.device(DEV))

    for step in range(2):
        ids, dense, *_ = make_fm_inputs(Bg, F, Dn, D, V, seed=60 + 10 * step + D, zipf=True)
        ids[0, 3], ids[2, 4], ids[Bg - 1, 0] = V + 5, -7, V    # out of range, both signs
        gen = torch.Generator().manual_seed(70 + step)
        A = torch.randn(Bg, F + Dn, D, generator=gen)
        g1 = torch.randn(Bg, generator=gen)
        g2 = torch.randn(Bg, generator=gen)
        ids_d, dense_d, A_d, g1_d, g2_d = (t.to(DEV) for t in (ids, dense, A, g1, g2))
        sl = [slice(r * Bp, (r + 1) * Bp) for r in range(world)]

        # ---- forward: bucketize, id exchange, gather_push, K1 over the row buffers
        plan = [ops.raw_shard_bucketize(ids_d[sl[r]], world, V) for r in range(world)]
        counts = torch.stack([plan[r][3].cpu() for r in range(world)])
        send_seg, recv_seg, dst_pull, dst_push = exchange_tables(counts)
        recv_ids = [torch.cat([plan[r][0][int(send_seg[r][o]):int(send_seg[r][o + 1])]
                               for r in range(world)]) for o in range(world)]
        before = [b.cpu() for b in rows_bufs]
        for o in range(world):
            ops.raw_shard_gather_push(shards[o], recv_ids[o], pads[o], G, recv_seg[o].to(DEV),
                                      dst_pull[o].to(DEV), rows_ptrs, G, world)
        for r in range(world):
            gid = ids[sl[r]].reshape(-1)[plan[r][2].cpu().long()]    # global ids in bucket order
            want = before[r].clone()
            want[:n] = gathered(Wf, torch.where(gid == 0, -1, gid), -1, G)
            assert_same_bits(rows_bufs[r], want, "step %d: row buffer of rank %d" % (step, r))
        out = [ops.raw_embed_fm_fwd(rows_bufs[r][:n], None, plan[r][1].reshape(Bp, F),
                                    dense_d[sl[r]], dw, dw1, -1, D=D) for r in range(world)]
        # unsharded K1 on the global batch: the rows are copies and the per-sample reduction order
        # is the same, so the results are identical
        feat_g, y1_g, y2_g, _ = ops.raw_embed_fm_fwd(Wf.to(DEV), None, ids_d, dense_d, dw, dw1, 0,
                                                     D=D)
        ops.raw_oob_count()        # the global call counted the out-of-range ids: reset
        for k, ref in enumerate((feat_g, y1_g, y2_g)):
            assert torch.equal(torch.cat([o_[k] for o_ in out]), ref), \
                "step %d: forward output %d" % (step, k)

        # ---- backward, fp64 oracle on the global batch
        ids_ok = torch.where((ids >= 0) & (ids < V), ids, 0)
        p, y1, y2, feat = oracle_fm(ids_ok, dense, W, W1, dense_w, dense_w1)
        ((feat * A.double()).sum() + (y1.reshape(-1) * g1.double()).sum()
         + (y2.reshape(-1) * g2.double()).sum()).backward()
        gW, gW1 = p["fm.embedding.weight"].grad, p["fm.embedding_one.weight"].grad[:, 0]
        gdw, gdw1 = p["fm.dense_w"].grad[0], p["fm.dense_w_one"].grad
        for path in paths:
            bufs, ptrs = grad_bufs[path]
            before = [b.cpu() for b in bufs]
            ddw_sum = torch.zeros(Dn, D, dtype=torch.float64)
            ddw1_sum = torch.zeros(Dn, dtype=torch.float64)
            slot_rows = []
            for r in range(world):
                feat_r, _, _, S_r = out[r]
                args = (feat_r, S_r, A_d[sl[r]], g1_d[sl[r]], g2_d[sl[r]], dense_d[sl[r]], iota,
                        plan[r][2])
                seg, dst = send_seg[r].to(DEV), dst_push[r].to(DEV)
                if path == "fused":
                    ops.raw_shard_fm_grads_push(*args[:5], plan[r][2], F, G, seg, dst, ptrs, G,
                                                world)
                    _, _, ddw, ddw1 = ops.raw_embed_fm_bwd(*args, zero, F, fused_cols=G)
                else:
                    dW, _, ddw, ddw1 = ops.raw_embed_fm_bwd(*args, num, F, fused_cols=G)
                    ops.raw_shard_push_rows(dW[:n], G, seg, dst, ptrs, G, world)
                    slot_rows.append(dW[:n].cpu())
                ddw_sum += ddw.cpu().double()
                ddw1_sum += ddw1.cpu().double()
            for o in range(world):
                if path == "two_kernel":     # every requester's rows in its segment of the owner
                    want = before[o].clone()
                    for r in range(world):
                        a, b = int(recv_seg[o][r]), int(recv_seg[o][r + 1])
                        s0 = int(send_seg[r][o])
                        want[a:b] = slot_rows[r][s0:s0 + b - a]
                else:
                    want = grad_bufs["two_kernel"][0][o]
                assert_same_bits(bufs[o], want, "step %d, %s: gradient buffer of rank %d"
                                 % (step, path, o))
            assert rel_err(ddw_sum, gdw) < 3e-6 and rel_err(ddw1_sum, gdw1) < 3e-6

            # ---- owner side: merge the received rows by local row, compare with the oracle's shard
            for o in range(world):
                m = int(recv_seg[o][-1])
                grp = ops.raw_group_ids(recv_ids[o], max(V_loc[o], 1), pads[o])
                red = ops.raw_segment_reduce(bufs[o][:m], grp.seg_offsets, grp.sorted_pos, grp.num,
                                             grp.n)
                dense_g = ops.SelectedRows(grp.unique_ids, red, grp.num, V_loc[o]).to_dense().cpu()
                what = "step %d, %s, rank %d" % (step, path, o)
                assert rel_err(dense_g[:, :D], gW[o::world]) < 3e-6, what
                assert rel_err(dense_g[:, D], gW1[o::world]) < 3e-6, what
                assert not dense_g[:, D + 1:].any(), what
                if o == 0:
                    assert not dense_g[0].any(), what + ": the padding row got a gradient"


# ---- D: argument checks, all with n == 0 so that no kernel is launched ---------------------------
KINDS = ["gather_push", "push_rows", "fm_grads_push"]


def call_empty(kind, ptrs, world, D=16, seg=None, dst=None, recv_ids=None):
    F, Dn = 26, 13
    if seg is None:
        seg = torch.zeros(world + 1, dtype=torch.int64, device=DEV)
    if dst is None:
        dst = torch.zeros(world, dtype=torch.int64, device=DEV)
    if kind == "gather_push":
        if recv_ids is None:
            recv_ids = torch.zeros(0, dtype=torch.int64, device=DEV)
        ops.raw_shard_gather_push(torch.zeros(4, D, device=DEV), recv_ids, -1, D, seg, dst, ptrs, D,
                                  world)
    elif kind == "push_rows":
        ops.raw_shard_push_rows(torch.zeros(0, D, device=DEV), D, seg, dst, ptrs, D, world)
    else:
        G = ops.fused_grad_cols(D)
        ops.raw_shard_fm_grads_push(torch.zeros(0, F + Dn, D, device=DEV),
                                    torch.zeros(0, D, device=DEV), None,
                                    torch.zeros(0, device=DEV), torch.zeros(0, device=DEV),
                                    torch.zeros(0, dtype=torch.int32, device=DEV), F, G, seg, dst,
                                    ptrs, G, world)


@pytest.fixture(scope="module")
def recv_buffer():
    return torch.zeros(64, 64, device=DEV)


def ptrs_of(*addrs):
    return (ctypes.c_uint64 * len(addrs))(*addrs)


@pytest.mark.parametrize("kind", KINDS)
def test_rejects_null_peer_pointer(kind, recv_buffer):
    base = recv_buffer.data_ptr()
    with pytest.raises(_lib.B200RecError, match="receive buffer of rank 1 is NULL"):
        call_empty(kind, ptrs_of(base, 0, base), 3)


@pytest.mark.parametrize("kind,D,offset,align", [
    ("gather_push", 16, 8, 16), ("gather_push", 2, 4, 8), ("push_rows", 12, 4, 16),
    ("push_rows", 6, 4, 8), ("fm_grads_push", 16, 8, 16), ("fm_grads_push", 4, 4, 16)])
def test_rejects_misaligned_peer_pointer(kind, D, offset, align, recv_buffer):
    base = recv_buffer.data_ptr()
    with pytest.raises(_lib.B200RecError,
                       match="receive buffer of rank 2 is not %d-byte aligned" % align):
        call_empty(kind, ptrs_of(base, base, base + offset), 3, D=D)


@pytest.mark.parametrize("kind,D,offset", [("gather_push", 2, 8), ("gather_push", 1, 4),
                                           ("push_rows", 3, 4), ("push_rows", 16, 256)])
def test_accepts_pointer_aligned_to_the_store_width(kind, D, offset, recv_buffer):
    base = recv_buffer.data_ptr()
    call_empty(kind, ptrs_of(base + offset, base), 2, D=D)


@pytest.mark.parametrize("kind", KINDS)
def test_rejects_world_above_max_peers(kind, recv_buffer):
    with pytest.raises(_lib.B200RecError, match=r"world=17 \(max 16\)"):
        call_empty(kind, ptrs_of(*[recv_buffer.data_ptr()] * 17), 17)


@pytest.mark.parametrize("kind", ["gather_push", "push_rows"])
def test_rejects_rows_wider_than_32_chunks(kind, recv_buffer):
    with pytest.raises(_lib.B200RecError, match="unsupported D=33"):
        call_empty(kind, ptrs_of(recv_buffer.data_ptr()), 1, D=33)


@pytest.mark.parametrize("kind", KINDS)
def test_rejects_bad_segment_tables(kind, recv_buffer):
    ptrs = ptrs_of(*[recv_buffer.data_ptr()] * 4)
    i64 = dict(dtype=torch.int64, device=DEV)
    with pytest.raises(_lib.B200RecError, match="seg_dev must have world\\+1 = 5 entries"):
        call_empty(kind, ptrs, 4, seg=torch.zeros(4, **i64))
    with pytest.raises(_lib.B200RecError, match="dst_dev world = 4, got 5 and 5"):
        call_empty(kind, ptrs, 4, dst=torch.zeros(5, **i64))
    with pytest.raises(_lib.B200RecError, match="seg_dev must be torch.int64"):
        call_empty(kind, ptrs, 4, seg=torch.zeros(5, dtype=torch.int32, device=DEV))
    with pytest.raises(_lib.B200RecError, match="dst_dev must be a CUDA tensor"):
        call_empty(kind, ptrs, 4, dst=torch.zeros(4, dtype=torch.int64))
    with pytest.raises(_lib.B200RecError, match="3 peer pointers for world=4"):
        call_empty(kind, ptrs_of(*[recv_buffer.data_ptr()] * 3), 4)


def test_rejects_int32_recv_ids(recv_buffer):
    with pytest.raises(_lib.B200RecError, match="recv_ids must be torch.int64"):
        call_empty("gather_push", ptrs_of(recv_buffer.data_ptr()), 1,
                   recv_ids=torch.zeros(0, dtype=torch.int32, device=DEV))
