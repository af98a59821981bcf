"""Row-cyclic sharding of the embedding tables over the GPUs of one box, with an NCCL all-to-all on
the id -> owner and row -> requester exchanges (SURVEY.md §8e).

Behavioural spec in the reference: the PSGPU / HeterPS pull-push of the GPUBox trainer
(tools/static_gpubox_trainer.py:152-159 builds the per-GPU HBM tables, :244-259 runs
pull_sparse -> fwd/bwd -> push_sparse per batch; tools/run_gpubox.sh:7-45 launches it).  Here:

    owner(id) = id mod world,  local_row(id) = id div world        (padding id 0 lives on rank 0)
    forward   bucketize ids by owner  ->  all-to-all(counts)  ->  all-to-all(ids)
              owner: b200rec_gather on its shard  ->  all-to-all(rows) back
              requester: the SAME fused kernel as the single-GPU path (b200rec_embed_fm_fwd) over
              the received rows, indexed by the bucket permutation
    backward  requester: b200rec_embed_fm_bwd emits per-slot gradients in bucket order
              all-to-all(grads) to the owners  ->  owner: group_ids + segment_reduce on local rows
              -> SelectedRows on the local shard -> row-wise optimizer
    dense     parameters are replicated; their gradients are all-reduced in one flat bucket.

The collective plumbing is torch.distributed (NCCL on GPUs; gloo in the CPU unit tests, which
inject a torch stand-in for the kernel set — the product default `ops` has no CPU path).
"""
from __future__ import annotations

import contextlib
import math
import os
from dataclasses import dataclass
from typing import List, Optional

import torch
import torch.distributed as dist
import torch.nn as tnn

from . import nn as bnn
from . import ops as _cuda_ops
from . import optim


def _timed(name: str):
    """CUDA-event pair around a collective when bench.py collects per-kernel times (CUDA only)."""
    return _cuda_ops._Timed(name) if torch.cuda.is_available() else contextlib.nullcontext()


def shard_rows(V: int, rank: int, world: int) -> int:
    """Number of global ids with id % world == rank."""
    return (V - rank + world - 1) // world if V > rank else 0


@dataclass
class ExchangePlan:
    n: int
    perm: torch.Tensor        # int64 [n]: slot of each position in bucket order
    inv_perm: torch.Tensor    # int32 [n]
    send_splits: List[int]    # ids sent to each rank
    recv_splits: List[int]    # ids received from each rank
    recv_ids: torch.Tensor    # int64 [m]: local rows requested from this rank (owner view)
    owner_groups: object = None   # grouping of recv_ids by local row, if it was precomputed
    tables: object = None         # device segment tables of the peer-memory exchange (or None)


class _PendingPlan:
    """Bucketing + count exchange of a FUTURE batch, running on a side stream."""

    def __init__(self, ids, send_ids, perm, inv_perm, host_counts, event):
        self.ids, self.send_ids, self.perm, self.inv_perm = ids, send_ids, perm, inv_perm
        self.host_counts, self.event = host_counts, event


class PeerBuffers:
    """Receive buffers mapped by every rank (torch symmetric memory over NVLink): rows [cap, cols]
    for the pull, gradient rows [2*cap, cols] for the push, plus the device-side barrier that
    publishes the peers' stores.  With these the row / gradient exchange is done by OUR kernels
    (b200rec_shard_gather_push / _push_rows) storing into peer memory — no NCCL call on the data
    path, the owner-side gather and its transfer are one kernel."""

    def __init__(self, cap: int, cols: int, world: int, group, device):
        import ctypes

        import torch.distributed._symmetric_memory as symm_mem
        self.cap, self.cap_g, self.cols, self.world = cap, 2 * cap, cols, world
        self.buf = symm_mem.empty(self.cap + self.cap_g, cols, dtype=torch.float32, device=device)
        self.hdl = symm_mem.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.rows = self.buf[:cap]
        self.grads = self.buf[cap:]
        ptrs = list(self.hdl.buffer_ptrs)
        self.rows_ptrs = (ctypes.c_uint64 * world)(*ptrs)
        self.grads_ptrs = (ctypes.c_uint64 * world)(*[p + cap * cols * 4 for p in ptrs])

    def publish_rows(self):
        self.hdl.barrier(channel=0)

    def publish_grads(self):
        self.hdl.barrier(channel=1)


P2P_MAX_WORLD = 4
# b200rec_shard_fm_grads_push (K2's sparse half + the push as one kernel) stores the same bits as K2 +
# b200rec_shard_push_rows on one GPU with virtual peers (tests/test_gpu_shard_kernels.py), but the
# exchange with it has not run across GPUs yet -> opt-in only.
FUSED_PUSH = os.environ.get("B200REC_FUSED_PUSH", "0") == "1"


def p2p_enabled(world: int) -> bool:
    """Peer-memory exchange on/off.  B200REC_P2P=1 forces it on, =0 off; unset = on for up to
    P2P_MAX_WORLD ranks.  The limit is the largest world size the peer-memory path has completed
    tests + bench on (2 and 4 ranks, profiles/r2g_*, r2h_*, r2j_*); the one 8-rank bench attempt with
    it did not finish inside its 300 s limit and could not be diagnosed (DESIGN.md section 5), so
    more than 4 ranks use the NCCL all-to-all exchange, which is validated at 8
    (profiles/r2_sharded_parity_n8.log, profiles/r2k_cfg3_dcn_n8.jsonl)."""
    env = os.environ.get("B200REC_P2P", "auto")
    if env == "0":
        return False
    if env == "1":
        return True
    return world <= P2P_MAX_WORLD


class ShardExchange:
    """The all-to-all choreography; shared by every table that is looked up with the same ids.

    The split sizes of the id exchange must be known on the host.  `plan()` alone therefore costs a
    device->host sync per step, which also drains the launch queue (the CPU can no longer run
    ahead of the GPU).  `prefetch(ids_next)` removes it: bucketing, the count all-to-all and the
    D2H copy of the NEXT batch run on a side stream while the current step computes; by the time
    `plan(ids_next)` is called the counts are already on the host."""

    def __init__(self, V: int, rank: int, world: int, group=None, kernels=_cuda_ops,
                 owner_pad: Optional[int] = None):
        self.V, self.rank, self.world, self.group, self.k = V, rank, world, group, kernels
        self._pending = None
        self._side = None
        # local padding row of the tables behind this exchange (None = unknown): lets the prefetch
        # also run the OWNER-side grouping of the received ids (a CUB sort) off the critical path
        self.owner_pad = owner_pad
        # peer-memory exchange (set up lazily by enable_p2p on the first pull; None = NCCL path)
        self.p2p_cols = None
        self.peer = None
        self._p2p_failed = False
        self._peer_injected = False   # tests only: a host-memory stand-in for PeerBuffers (inject_peer)

    def _bucketize_and_count(self, ids):
        send_ids, perm, inv_perm, counts = self.k.raw_shard_bucketize(ids, self.world, self.V)
        if self.p2p_cols is None:
            recv_counts = torch.empty_like(counts)
            dist.all_to_all_single(recv_counts, counts, group=self.group)
            return send_ids, perm, inv_perm, torch.stack([counts, recv_counts]), None
        # peer-memory exchange: besides the counts every owner learns WHERE in the requester's row
        # buffer its rows go (the requester's bucket offset), and every requester where in the
        # owner's gradient buffer its rows go (the owner's receive offset).  All on the device.
        zero = torch.zeros(1, dtype=counts.dtype, device=counts.device)
        send_seg = torch.cat([zero, counts.cumsum(0)])
        got = torch.empty(self.world, 2, dtype=counts.dtype, device=counts.device)
        dist.all_to_all_single(got, torch.stack([counts, send_seg[:-1]], 1).contiguous(),
                               group=self.group)
        recv_counts, dst_pull = got[:, 0].contiguous(), got[:, 1].contiguous()
        recv_seg = torch.cat([zero, recv_counts.cumsum(0)])
        dst_push = torch.empty_like(counts)
        dist.all_to_all_single(dst_push, recv_seg[:-1].contiguous(), group=self.group)
        tables = {"send_seg": send_seg, "recv_seg": recv_seg, "dst_pull": dst_pull,
                  "dst_push": dst_push}
        return send_ids, perm, inv_perm, torch.stack([counts, recv_counts]), tables

    def prefetch(self, ids: torch.Tensor) -> None:
        """Start planning the exchange of a future batch (CUDA only; a no-op on CPU tensors)."""
        if not ids.is_cuda:
            return
        if self._side is None:
            self._side = torch.cuda.Stream(device=ids.device)
        flat = ids.reshape(-1)
        self._side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self._side):
            send_ids, perm, inv_perm, both, tables = self._bucketize_and_count(flat)
            host = torch.empty(both.shape, dtype=both.dtype, pin_memory=True)
            host.copy_(both, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._side)
        for t in (flat, send_ids, perm, inv_perm, both):
            t.record_stream(self._side)
        self._pending = _PendingPlan(ids, send_ids, perm, inv_perm, host, ev)
        self._pending.tables = tables

    def finish_prefetch(self) -> None:
        """Second half of the prefetch (call it later in the step, e.g. after backward was
        launched): once the counts are on the host, run the id all-to-all of the NEXT batch on the
        side stream too, so the next forward starts directly with the owner-side gather."""
        pend = self._pending
        if pend is None or getattr(pend, "recv_ids", None) is not None:
            return
        # Every rank must issue its collectives in the same order, so this must not depend on a
        # rank-local "is it ready yet" test: always wait for the counts (the GPU is busy with the
        # backward pass that was already enqueued, so the host wait costs no GPU time).
        pend.event.synchronize()
        send_splits, recv_splits = pend.host_counts[0].tolist(), pend.host_counts[1].tolist()
        with torch.cuda.stream(self._side):
            recv_ids = torch.empty(sum(recv_splits), dtype=torch.int64, device=pend.send_ids.device)
            dist.all_to_all_single(recv_ids, pend.send_ids, recv_splits, send_splits,
                                   group=self.group)
            groups = None
            if self.owner_pad is not None:
                # what owner_reduce() needs in the backward of the NEXT step: done here, on the side
                # stream, while the current backward runs (own scratch buffer: ws_tag)
                groups = self.k.raw_group_ids(recv_ids, max(shard_rows(self.V, self.rank, self.world), 1),
                                              self.owner_pad, ws_tag="group_side")
            ev = torch.cuda.Event()
            ev.record(self._side)
        recv_ids.record_stream(self._side)
        pend.recv_ids, pend.splits, pend.event2 = recv_ids, (send_splits, recv_splits), ev
        pend.groups = groups

    def plan(self, ids: torch.Tensor) -> ExchangePlan:
        pend, self._pending = self._pending, None
        flat = ids.reshape(-1)
        n = flat.numel()
        if pend is not None and pend.ids is ids:
            send_ids, perm, inv_perm = pend.send_ids, pend.perm, pend.inv_perm
            if getattr(pend, "recv_ids", None) is not None:       # fully prefetched
                torch.cuda.current_stream().wait_event(pend.event2)
                send_splits, recv_splits = pend.splits
                cur = torch.cuda.current_stream()
                for t in (pend.recv_ids, perm, inv_perm):
                    t.record_stream(cur)
                groups = getattr(pend, "groups", None)
                if groups is not None:
                    for t in (groups.unique_ids, groups.seg_offsets, groups.sorted_pos, groups.num):
                        t.record_stream(cur)
                tables = getattr(pend, "tables", None)
                if tables is not None:
                    for t in tables.values():
                        t.record_stream(cur)
                return ExchangePlan(n, perm, inv_perm, send_splits, recv_splits, pend.recv_ids,
                                    groups, tables)
            pend.event.synchronize()                              # normally long complete
            torch.cuda.current_stream().wait_event(pend.event)
            send_splits, recv_splits = pend.host_counts[0].tolist(), pend.host_counts[1].tolist()
            tables = getattr(pend, "tables", None)
        else:
            send_ids, perm, inv_perm, both, tables = self._bucketize_and_count(flat)
            both = both.cpu()                                     # host sync (no prefetch)
            send_splits, recv_splits = both[0].tolist(), both[1].tolist()
        recv_ids = torch.empty(sum(recv_splits), dtype=torch.int64, device=ids.device)
        dist.all_to_all_single(recv_ids, send_ids, recv_splits, send_splits, group=self.group)
        return ExchangePlan(n, perm, inv_perm, send_splits, recv_splits, recv_ids, None, tables)

    def enable_p2p(self, cols: int) -> None:
        """Ask for the peer-memory exchange of `cols`-wide rows (takes effect from the next
        bucketing on; the buffers are created collectively at the first pull)."""
        if self.world > 1 and p2p_enabled(self.world) and torch.cuda.is_available():
            self.p2p_cols = int(cols)

    def inject_peer(self, peer, cols: int) -> None:
        """TEST HOOK (tests/test_sharded_cpu.py): run the peer-memory choreography of pull / push on
        host tensors — `peer` quacks like PeerBuffers with shared-memory tensors instead of NVLink
        mappings and `kernels` are the torch stand-ins.  Never used by the product path."""
        self.peer, self.p2p_cols, self._peer_injected = peer, int(cols), True

    def _use_p2p(self, plan: ExchangePlan, cols: int, shard: torch.Tensor) -> bool:
        if self.p2p_cols is None or plan.tables is None or cols != self.p2p_cols or self._p2p_failed:
            return False
        if not (shard.is_cuda or self._peer_injected):
            return False
        if self.peer is None or plan.n > self.peer.cap:
            # collective: every rank sees the same plan.n (B per GPU is fixed) and gets here together
            cap = max(1024, int(plan.n * 1.25))
            try:
                self.peer = PeerBuffers(cap, cols, self.world, self.group, shard.device)
            except Exception as exc:   # no symmetric memory in this environment: NCCL path
                import warnings
                warnings.warn("peer-memory exchange unavailable (%r): using NCCL all-to-all" % (exc,))
                self._p2p_failed, self.peer = True, None
                return False
        if plan.recv_ids.numel() > self.peer.cap_g:
            # a rank-local fall-back would desynchronise the collectives: fail loudly instead
            raise RuntimeError(
                "peer-memory exchange: %d rows requested from this rank exceed the receive capacity "
                "%d (ids are too skewed for owner = id mod world); set B200REC_P2P=0"
                % (plan.recv_ids.numel(), self.peer.cap_g))
        return True

    def pull(self, plan: ExchangePlan, shard: torch.Tensor, local_pad: int,
             D: Optional[int] = None) -> torch.Tensor:
        """Owner-side gather of the first D columns (default: all) + rows back to the requesters:
        returns [n, D] in bucket order."""
        cols = D if D is not None else shard.shape[1]
        if self._use_p2p(plan, cols, shard):
            # ONE kernel gathers the requested rows and stores them into the requesters' buffers
            # over NVLink; the barrier publishes every rank's stores.
            self.k.raw_shard_gather_push(shard, plan.recv_ids, local_pad, cols,
                                         plan.tables["recv_seg"], plan.tables["dst_pull"],
                                         self.peer.rows_ptrs, self.peer.cols, self.world)
            with _timed("p2p_barrier"):
                self.peer.publish_rows()
            return self.peer.rows[:plan.n]
        rows_out = self.k.raw_gather(shard, plan.recv_ids, local_pad, D)
        rows_in = torch.empty(plan.n, rows_out.shape[-1], dtype=shard.dtype, device=shard.device)
        with _timed("nccl_a2a_rows"):
            dist.all_to_all_single(rows_in, rows_out, plan.send_splits, plan.recv_splits,
                                   group=self.group)
        return rows_in

    def push(self, plan: ExchangePlan, grads_bucket_order: torch.Tensor) -> torch.Tensor:
        """Per-slot gradients [n, D] (bucket order) -> owners: returns [m, D] aligned with
        plan.recv_ids."""
        D = grads_bucket_order.shape[1]
        if (self.peer is not None and plan.tables is not None and D == self.peer.cols and
                (grads_bucket_order.is_cuda or self._peer_injected)):
            self.k.raw_shard_push_rows(grads_bucket_order, D, plan.tables["send_seg"],
                                       plan.tables["dst_push"], self.peer.grads_ptrs,
                                       self.peer.cols, self.world)
            with _timed("p2p_barrier"):
                self.peer.publish_grads()
            return self.peer.grads[:plan.recv_ids.numel()]
        out = torch.empty(plan.recv_ids.numel(), D, dtype=grads_bucket_order.dtype,
                          device=grads_bucket_order.device)
        with _timed("nccl_a2a_grads"):
            dist.all_to_all_single(out, grads_bucket_order.contiguous(), plan.recv_splits,
                                   plan.send_splits, group=self.group)
        return out

    def push_fm_grads(self, plan: ExchangePlan, feat, S, dfeat, gy1, gy2, F: int, G: int):
        """DeepFM over peer memory: K2's sparse half and the push as ONE kernel (None if the
        peer-memory exchange is not active for this plan: caller falls back to K2 + push)."""
        D = feat.shape[2]
        if (not FUSED_PUSH or self.peer is None or plan.tables is None or G != self.peer.cols or
                not (feat.is_cuda or self._peer_injected) or D % 4 or G % 4):
            return None
        self.k.raw_shard_fm_grads_push(feat, S, dfeat, gy1, gy2, plan.inv_perm, F, G,
                                       plan.tables["send_seg"], plan.tables["dst_push"],
                                       self.peer.grads_ptrs, self.peer.cols, self.world)
        with _timed("p2p_barrier"):
            self.peer.publish_grads()
        return self.peer.grads[:plan.recv_ids.numel()]

    def owner_reduce(self, plan: ExchangePlan, grads: torch.Tensor, V_loc: int, local_pad: int):
        """Merge the received gradients by local row -> SelectedRows on the local shard."""
        groups = plan.owner_groups
        if groups is None or local_pad != self.owner_pad:
            groups = self.k.raw_group_ids(plan.recv_ids, max(V_loc, 1), local_pad)
        rows = self.k.raw_segment_reduce(grads.contiguous(), groups.seg_offsets, groups.sorted_pos,
                                         groups.num, groups.n)
        return self.k.SelectedRows(groups.unique_ids, rows, groups.num, V_loc)


class _ShardedLookup(torch.autograd.Function):
    """paddle.nn.Embedding forward/backward over a row-cyclically sharded table: the generic
    (non-FM) lookup used by DCN-V2 / Wide&Deep / DIN when their tables are sharded."""

    @staticmethod
    def forward(ctx, ids, emb, _hook):
        ex, k = emb.exchange, emb.exchange.k
        plan = ex.plan(ids)
        rows = ex.pull(plan, emb.weight, emb.pad)                  # [n, D] in bucket order
        out = k.raw_gather(rows, plan.perm, -1)                    # back to position order
        ctx.plan, ctx.emb = plan, emb
        return out.reshape(*ids.shape, rows.shape[1])

    @staticmethod
    def backward(ctx, dout):
        plan, emb = ctx.plan, ctx.emb
        ex, k = emb.exchange, emb.exchange.k
        D = dout.shape[-1]
        g = k.raw_gather(dout.reshape(-1, D).contiguous(), plan.inv_perm.to(torch.int64), -1)
        g = ex.push(plan, g)
        emb.accept(ex.owner_reduce(plan, g, emb.num_embeddings, emb.pad))
        return None, None, None


class ShardedEmbedding(bnn.Embedding):
    """The local shard ([ceil((V-rank)/world), D]) of a row-cyclically sharded table.  `forward`
    has paddle.nn.Embedding's signature; the all-to-all exchange happens inside."""

    def __init__(self, num_embeddings, embedding_dim, padding_idx, rank, world, init_std=None,
                 init="truncated_normal", device=None, group=None, kernels=_cuda_ops):
        local_pad = None
        if padding_idx is not None and padding_idx % world == rank:
            local_pad = padding_idx // world
        super().__init__(shard_rows(num_embeddings, rank, world), embedding_dim, local_pad,
                         init_std=init_std, init=init, device=device)
        self.global_rows, self.rank, self.world = num_embeddings, rank, world
        self.exchange = ShardExchange(num_embeddings, rank, world, group, kernels,
                                      owner_pad=(-1 if local_pad is None else local_pad))

    def forward(self, ids):
        return _ShardedLookup.apply(ids, self, bnn._autograd_hook(ids.device))


@torch.no_grad()
def shard_embeddings(model: tnn.Module, rank: int, world: int, group=None, min_rows: int = 0,
                     kernels=_cuda_ops) -> tnn.Module:
    """Replace every `bnn.Embedding` of `model` whose table has >= min_rows rows by the local
    shard of a row-cyclic ShardedEmbedding (rows rank, rank+world, ... of the original, so a
    replicated initialisation stays consistent), then broadcast the dense parameters.  This is how
    DCN-V2 (BASELINE config 3), Wide&Deep and large-vocabulary DIN run on N GPUs."""
    for parent in list(model.modules()):
        for name, child in list(parent.named_children()):
            if type(child) is bnn.Embedding and child.num_embeddings >= min_rows:
                sh = ShardedEmbedding(child.num_embeddings, child.embedding_dim, child.padding_idx,
                                      rank, world, init="empty", device=child.weight.device,
                                      group=group, kernels=kernels)
                sh.weight.copy_(child.weight[rank::world])
                setattr(parent, name, sh)
    sync_dense_parameters(model, group)
    return model


class _ShardedEmbedFM(torch.autograd.Function):
    """DeepFM's FM block over sharded tables: exchange + the single-GPU fused kernels."""

    @staticmethod
    def forward(ctx, ids, dense, dense_w, dense_w1, fm):
        k, ex = fm.k, fm.exchange
        B, F = ids.shape
        plan = ex.plan(ids)
        D = fm.sparse_feature_dim
        slot_ids = plan.perm.reshape(B, F)
        if fm.fused:   # ONE exchange of [emb | w1 | pad] rows instead of two
            tab = fm._fused
            rows = ex.pull(plan, tab.weight, tab.pad, tab.grad_cols)
            feat, y1, y2, S = k.raw_embed_fm_fwd(rows, None, slot_ids, dense,
                                                 dense_w.reshape(-1, D), dense_w1.reshape(-1), -1,
                                                 D=D)
        else:
            rows = ex.pull(plan, fm.embedding.weight, fm.embedding.pad)
            rows1 = ex.pull(plan, fm.embedding_one.weight, fm.embedding_one.pad)
            feat, y1, y2, S = k.raw_embed_fm_fwd(rows, rows1, slot_ids, dense,
                                                 dense_w.reshape(-1, D), dense_w1.reshape(-1), -1)
        ctx.save_for_backward(dense, feat, S)
        ctx.plan, ctx.fm, ctx.F = plan, fm, F
        ctx.dense_w_shape = dense_w.shape
        return feat, y1.unsqueeze(1), y2.unsqueeze(1)

    @staticmethod
    def backward(ctx, dfeat, dy1, dy2):
        dense, feat, S = ctx.saved_tensors
        fm, plan, F = ctx.fm, ctx.plan, ctx.F
        k, ex = fm.k, fm.exchange
        B = feat.shape[0]
        dev = feat.device
        gy1 = dy1.reshape(-1).contiguous() if dy1 is not None else torch.zeros(B, device=dev)
        gy2 = dy2.reshape(-1).contiguous() if dy2 is not None else torch.zeros(B, device=dev)
        if dfeat is not None:
            dfeat = dfeat.contiguous()
        n = plan.n
        iota, num = fm.trivial_groups(n, dev)
        # seg_offsets = iota, sorted_pos = inv_perm: row k of the output is the gradient of slot k
        if fm.fused:
            tab = fm._fused
            g = ex.push_fm_grads(plan, feat, S, dfeat, gy1, gy2, F, tab.grad_cols)
            if g is not None:
                # sparse half + push were one kernel; only the dense-feature gradients remain
                # (the segmented part of K2 sees zero segments)
                _, _, ddense_w, ddense_w1 = k.raw_embed_fm_bwd(feat, S, dfeat, gy1, gy2, dense, iota,
                                                               plan.inv_perm, fm.zero_groups(dev), F,
                                                               fused_cols=tab.grad_cols)
            else:
                dW, _, ddense_w, ddense_w1 = k.raw_embed_fm_bwd(feat, S, dfeat, gy1, gy2, dense,
                                                                iota, plan.inv_perm, num, F,
                                                                fused_cols=tab.grad_cols)
                g = ex.push(plan, dW[:n])
            tab.accept_fused(ex.owner_reduce(plan, g, tab.num_embeddings, tab.pad))
        else:
            dW, dW1, ddense_w, ddense_w1 = k.raw_embed_fm_bwd(feat, S, dfeat, gy1, gy2, dense, iota,
                                                              plan.inv_perm, num, F)
            g = ex.push(plan, dW[:n])
            g1 = ex.push(plan, dW1[:n].unsqueeze(1))
            emb, emb1 = fm.embedding, fm.embedding_one
            emb.accept(ex.owner_reduce(plan, g, emb.num_embeddings, emb.pad))
            emb1.accept(ex.owner_reduce(plan, g1, emb1.num_embeddings, emb1.pad))
        return None, None, ddense_w.reshape(ctx.dense_w_shape), ddense_w1, None


class ShardedFusedTable(bnn.FusedTable):
    """Local shard of a row-cyclically sharded FusedTable."""

    def __init__(self, num_embeddings, embedding_dim, padding_idx, rank, world, init_std=None,
                 device=None):
        local_pad = None
        if padding_idx is not None and padding_idx % world == rank:
            local_pad = padding_idx // world
        super().__init__(shard_rows(num_embeddings, rank, world), embedding_dim, local_pad,
                         init_std=init_std, device=device)
        self.global_rows, self.rank, self.world = num_embeddings, rank, world


class ShardedFM(bnn.FusedTableOwner):
    """FM of models/rank/deepfm/net.py:52-139 with both tables sharded (same state_dict names;
    `embedding*.weight` hold the LOCAL shard).  With `fused_table` (default when D+1 <= 32) the
    shard is a FusedTable and every exchange moves [emb | w1 | pad] rows in ONE all-to-all."""

    def __init__(self, sparse_feature_number, sparse_feature_dim, dense_feature_dim,
                 sparse_num_field, rank, world, group=None, device="cuda", kernels=_cuda_ops,
                 fused_table=None):
        super().__init__()
        self.k = kernels
        self.sparse_feature_number = sparse_feature_number
        self.sparse_feature_dim = sparse_feature_dim
        std = 0.1 / math.sqrt(float(sparse_feature_dim))
        self.fused = (sparse_feature_dim + 1 <= 32) if fused_table is None else bool(fused_table)
        if self.fused:
            self._fused = ShardedFusedTable(sparse_feature_number, sparse_feature_dim, 0, rank,
                                            world, init_std=std, device=device)
        else:
            self.embedding_one = ShardedEmbedding(sparse_feature_number, 1, 0, rank, world,
                                                  init_std=std, device=device)
            self.embedding = ShardedEmbedding(sparse_feature_number, sparse_feature_dim, 0, rank,
                                              world, init_std=std, device=device)
        self.dense_w_one = tnn.Parameter(torch.empty(dense_feature_dim, device=device))
        self.dense_w = tnn.Parameter(
            torch.empty(1, dense_feature_dim, sparse_feature_dim, device=device))
        tnn.init.trunc_normal_(self.dense_w_one, 0.0, std, -2 * std, 2 * std)
        tnn.init.trunc_normal_(self.dense_w, 0.0, std, -2 * std, 2 * std)
        self.exchange = ShardExchange(sparse_feature_number, rank, world, group, kernels,
                                      owner_pad=(0 if rank == 0 else -1))   # padding id 0 lives on rank 0
        if self.fused and kernels is _cuda_ops:
            self.exchange.enable_p2p(self._fused.grad_cols)
        self._trivial = {}

    def table_grad_dense(self):
        if self.fused:
            return self._fused.grad_dense()
        return (self.embedding.grad_rows.to_dense(), self.embedding_one.grad_rows.to_dense())

    def zero_groups(self, device):
        """num = {0, 0}: "no segments" (the fused push kernel already produced the sparse rows)."""
        key = ("zero", str(device))
        hit = self._trivial.get(key)
        if hit is None:
            hit = torch.zeros(2, dtype=torch.int32, device=device)
            self._trivial[key] = hit
        return hit

    def trivial_groups(self, n: int, device):
        """seg_offsets = 0..n and num = {n, n}: "every slot is its own segment" (cached per n so
        the backward issues no allocation / host->device copy for them)."""
        key = (n, str(device))
        hit = self._trivial.get(key)
        if hit is None:
            hit = (torch.arange(n + 1, dtype=torch.int32, device=device),
                   torch.full((2,), n, dtype=torch.int32, device=device))
            self._trivial[key] = hit
        return hit

    def forward(self, sparse_inputs, dense_inputs):
        ids = (torch.cat(list(sparse_inputs), dim=1) if isinstance(sparse_inputs, (list, tuple))
               else sparse_inputs)
        feat, y1, y2 = _ShardedEmbedFM.apply(ids, dense_inputs, self.dense_w, self.dense_w_one, self)
        return y1, y2, feat


class ShardedDeepFMLayer(tnn.Module):
    """DeepFMLayer (net.py:21-49) with sharded tables and a replicated tower."""

    def __init__(self, sparse_feature_number, sparse_feature_dim, dense_feature_dim,
                 sparse_num_field, layer_sizes, rank, world, group=None, device="cuda",
                 kernels=_cuda_ops, fused_table=None):
        super().__init__()
        from .rank.deepfm import net
        self.fm = ShardedFM(sparse_feature_number, sparse_feature_dim, dense_feature_dim,
                            sparse_num_field, rank, world, group, device, kernels, fused_table)
        self.dnn = net.DNN(sparse_feature_number, sparse_feature_dim, dense_feature_dim,
                           dense_feature_dim + sparse_num_field, layer_sizes, device=device)
        self.bias = tnn.Parameter(torch.zeros(1, device=device))
        self.world, self.group = world, group
        sync_dense_parameters(self, group)

    def forward(self, sparse_inputs, dense_inputs):
        y1, y2, feat = self.fm(sparse_inputs, dense_inputs)
        y_dnn = self.dnn(feat)
        if y_dnn.is_cuda and self.fm.k is _cuda_ops:
            return _cuda_ops.sum_sigmoid(y1, y2, y_dnn)
        return torch.sigmoid(y1 + y2 + y_dnn)

    def prefetch(self, next_sparse_inputs) -> None:
        """Hint: the ids of the NEXT batch (the very tensor that will be passed to forward)."""
        self.fm.exchange.prefetch(next_sparse_inputs)

    def finish_prefetch(self) -> None:
        self.fm.exchange.finish_prefetch()


def dense_parameters(model: tnn.Module) -> List[torch.Tensor]:
    return [p for p in model.parameters() if not getattr(p, "is_sparse_table", False)]


@torch.no_grad()
def sync_dense_parameters(model: tnn.Module, group=None) -> None:
    """Replicas must start identical: broadcast rank 0's dense parameters."""
    for p in dense_parameters(model):
        dist.broadcast(p.data, src=dist.get_global_rank(group, 0) if group is not None else 0,
                       group=group)


class DistributedOptimizer:
    """Wraps a paddlerec_b200.optim optimizer: all-reduces (SUM) the dense gradients in one flat
    bucket before the step.  Callers scale the local loss by 1/world (`scale_loss`) so that the
    summed dense gradients and the owner-summed table gradients both equal the gradient of the
    global-batch mean loss — what fleet.distributed_model does at tools/trainer.py:113-118."""

    def __init__(self, inner, model: tnn.Module, world: int, group=None):
        self.inner, self.world, self.group = inner, world, group
        self._dense = [p for p in dense_parameters(model) if p.requires_grad]
        self._side = None
        if world > 1 and hasattr(inner, "sparse_sq_reduce"):
            # ClipGradByGlobalNorm (DCN-V2): the table gradients live on their owners, so the
            # squared norm of that part is one scalar all-reduce; the dense part is identical on
            # every rank after the bucket all-reduce below.
            inner.sparse_sq_reduce = self._sum_over_ranks

    def _sum_over_ranks(self, t: torch.Tensor) -> torch.Tensor:
        t = t.clone()
        dist.all_reduce(t, group=self.group)
        return t

    def scale_loss(self, loss: torch.Tensor) -> torch.Tensor:
        return loss / self.world

    def clear_grad(self):
        self.inner.clear_grad()

    def _allreduce_dense(self):
        from . import tower
        tower.wait_pending()        # the tower's dW GEMMs may still run on their side stream
        grads = [p.grad for p in self._dense if p.grad is not None]
        if grads and self.world > 1:
            with _timed("nccl_allreduce_dense"):
                flat = torch.cat([g.reshape(-1) for g in grads])
                dist.all_reduce(flat, group=self.group)
                off = 0
                for g in grads:
                    g.copy_(flat[off:off + g.numel()].view_as(g))
                    off += g.numel()

    def step(self):
        inner = self.inner
        split = (hasattr(inner, "step_sparse") and getattr(inner, "_clip", None) is None
                 and self.world > 1 and self._dense and self._dense[0].is_cuda)
        if not split:       # clipping needs the reduced gradients first (global norm)
            self._allreduce_dense()
            inner.step()
            return
        # The dense all-reduce runs on a side stream while the row-wise table update (the large
        # part of the optimizer) runs on the main stream; they touch disjoint tensors.
        main = torch.cuda.current_stream()
        if self._side is None:
            self._side = torch.cuda.Stream()
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            self._allreduce_dense()
        inner.step_sparse()
        main.wait_stream(self._side)
        inner.step_dense()


def create_sharded_deepfm(config, device, rank, world, group=None, kernels=_cuda_ops):
    return ShardedDeepFMLayer(
        config.get("hyper_parameters.sparse_feature_number"),
        config.get("hyper_parameters.sparse_feature_dim"),
        config.get("hyper_parameters.dense_input_dim"),
        config.get("hyper_parameters.sparse_inputs_slots") - 1,
        config.get("hyper_parameters.fc_sizes"), rank, world, group, device, kernels)


def create_optimizer(model, config, world=None, group=None):
    lr = config.get("hyper_parameters.optimizer.learning_rate", 0.001)
    inner = optim.Adam(learning_rate=lr, parameters=model.parameters(), lazy_mode=True)
    world = world if world is not None else dist.get_world_size(group)
    return DistributedOptimizer(inner, model, world, group)
