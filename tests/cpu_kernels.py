"""A torch (CPU) stand-in for the kernel set that paddlerec_b200.sharded takes by injection.
TEST DOUBLE ONLY: it lets the world_size-2 gloo tests exercise the all-to-all choreography,
split bookkeeping and gradient routing on a box without a GPU.  The product default is
paddlerec_b200.ops (CUDA through the C ABI, no CPU path)."""
from dataclasses import dataclass

import torch


@dataclass
class IdGroups:
    unique_ids: torch.Tensor
    seg_offsets: torch.Tensor
    sorted_pos: torch.Tensor
    num: torch.Tensor
    n: int
    height: int


@dataclass
class SelectedRows:
    rows: torch.Tensor
    value: torch.Tensor
    num: torch.Tensor
    height: int
    ncols: int = None

    @property
    def cols(self):
        return self.value.shape[1] if self.ncols is None else self.ncols

    def to_dense(self):
        U = int(self.num[0])
        out = torch.zeros(self.height, self.cols)
        out[self.rows[:U]] += self.value[:U, :self.cols]
        return out


def raw_shard_bucketize(ids, world, V):
    ids = ids.reshape(-1)
    n = ids.numel()
    valid = (ids >= 0) & (ids < V)
    owner = torch.where(valid, ids % world, torch.zeros_like(ids))
    inv_perm = torch.sort(owner, stable=True).indices
    perm = torch.empty(n, dtype=torch.int64)
    perm[inv_perm] = torch.arange(n)
    local = torch.where(valid, ids // world, torch.full_like(ids, -1))
    counts = torch.bincount(owner, minlength=world).to(torch.int64)
    return local[inv_perm], perm, inv_perm.to(torch.int32), counts


def raw_gather(W, ids, pad, D=None):
    W = W if D is None else W[:, :D]
    ok = (ids >= 0) & (ids < W.shape[0]) & (ids != pad)
    # where, not a multiply by the mask: the kernels store +0.0 for these rows (x * 0 is -0.0 for
    # a negative x)
    return torch.where(ok.unsqueeze(-1), W[ids.clamp(0, max(W.shape[0] - 1, 0))], 0.0)


def raw_embed_fm_fwd(W, W1, ids, dense, dense_w, dense_w1, pad, want_S=True, D=None):
    if W1 is None:       # fused [emb | w1 | pad] rows
        W, W1 = W[:, :D], W[:, D]
    e = raw_gather(W, ids, pad)
    e1 = raw_gather(W1.reshape(-1, 1), ids, pad)
    feat = torch.cat([e, dense.unsqueeze(2) * dense_w.unsqueeze(0)], 1)
    y1 = e1.sum((1, 2)) + (dense * dense_w1).sum(1)
    S = feat.sum(1)
    y2 = 0.5 * (S.square() - feat.square().sum(1)).sum(1)
    return feat, y1, y2, S


def raw_group_ids(ids, V, pad):
    ids = ids.reshape(-1)
    n = ids.numel()
    keep = (ids >= 0) & (ids < V) & (ids != pad)
    key = torch.where(keep, ids, torch.full_like(ids, V))
    order = torch.sort(key, stable=True).indices
    kept = int(keep.sum())
    uniq, cnt = torch.unique_consecutive(key[order][:kept], return_counts=True)
    U = uniq.numel()
    seg = torch.zeros(n + 1, dtype=torch.int32)
    seg[1:U + 1] = torch.cumsum(cnt, 0).to(torch.int32)
    unique_ids = torch.zeros(max(n, 1), dtype=torch.int64)
    unique_ids[:U] = uniq
    return IdGroups(unique_ids, seg, order.to(torch.int32), torch.tensor([U, kept], dtype=torch.int32),
                    n, V)


def raw_segment_reduce(dOut, seg, pos, num, n):
    D = dOut.shape[-1]
    rows = torch.zeros(max(n, 1), D)
    for u in range(int(num[0])):
        rows[u] = dOut[pos[seg[u]:seg[u + 1]].long()].sum(0)
    return rows


def raw_embed_fm_bwd(feat, S, dfeat_dnn, gy1, gy2, dense, seg, pos, num, F, fused_cols=0):
    B, N, D = feat.shape
    dfeat = gy2.reshape(B, 1, 1) * (S.unsqueeze(1) - feat)
    if dfeat_dnn is not None:
        dfeat = dfeat + dfeat_dnn
    flat = dfeat[:, :F].reshape(B * F, D)
    g1 = gy1.reshape(B, 1).expand(B, F).reshape(B * F, 1)
    n = B * F
    dW = raw_segment_reduce(flat, seg, pos, num, n)
    dW1 = raw_segment_reduce(g1, seg, pos, num, n).reshape(-1)
    ddense_w = (dense.unsqueeze(2) * dfeat[:, F:]).sum(0)
    ddense_w1 = (gy1.reshape(B, 1) * dense).sum(0)
    if fused_cols:
        fusedW = torch.zeros(dW.shape[0], fused_cols)
        fusedW[:, :D] = dW
        fusedW[:, D] = dW1
        return fusedW, None, ddense_w, ddense_w1
    return dW, dW1, ddense_w, ddense_w1


def raw_dot_interact_fwd(T, self_interaction=False):
    from oracle import nets
    return nets.dot_interact(T, self_interaction)


def raw_dot_interact_bwd(T, dR, self_interaction=False):
    from oracle import nets
    with torch.enable_grad():
        Tq = T.detach().clone().requires_grad_(True)
        nets.dot_interact(Tq, self_interaction).backward(dR)
    return Tq.grad


# ---- row-wise optimizers / densify (stand-ins for b200rec_sparse_* and b200rec_rows_to_dense) -------
def _valid(sr):
    U = int(sr.num[0])
    return sr.rows[:U], sr.value[:U, :sr.cols]


def raw_rows_to_dense(sr, dW):
    rows, g = _valid(sr)
    dW[rows, :g.shape[1]] += g


def raw_sparse_sgd(W, sr, lr):
    rows, g = _valid(sr)
    W[rows, :g.shape[1]] -= lr * g


def raw_sparse_adam(W, m, v, sr, lr, beta1, beta2, eps, beta1_pow, beta2_pow):
    """Paddle's adam op on the touched rows: lr_t = lr*sqrt(1-b2^t)/(1-b1^t),
    w -= lr_t * m / (sqrt(v) + eps*sqrt(1-b2^t))."""
    rows, g = _valid(sr)
    C = g.shape[1]
    m[rows, :C] = beta1 * m[rows, :C] + (1 - beta1) * g
    v[rows, :C] = beta2 * v[rows, :C] + (1 - beta2) * g * g
    c2 = (1 - beta2_pow) ** 0.5
    W[rows, :C] -= lr * c2 / (1 - beta1_pow) * m[rows, :C] / (v[rows, :C].sqrt() + eps * c2)


KERNEL_NAMES = ("raw_gather", "raw_embed_fm_fwd", "raw_embed_fm_bwd", "raw_segment_reduce",
                "raw_rows_to_dense", "raw_sparse_sgd", "raw_sparse_adam", "raw_dot_interact_fwd",
                "raw_dot_interact_bwd", "raw_gather_pool_sum", "raw_cvm_fwd", "raw_cvm_bwd")


def install(monkeypatch, ops):
    """Patch the stand-ins over paddlerec_b200.ops for a CPU test of HOST logic (trainer / infer
    loops, checkpoints, readers).  Never used by the product or by the GPU parity tests."""
    import sys

    me = sys.modules[__name__]
    for name in KERNEL_NAMES:
        fn = getattr(me, name)
        if name == "raw_segment_reduce":
            def seg_reduce(dOut, seg, pos, num, n, row_of_pos=None):
                if row_of_pos is not None:      # pooled lookup: position p contributes dOut[bag(p)]
                    dOut = dOut[row_of_pos[:n].long()]
                return raw_segment_reduce(dOut, seg, pos, num, n)
            monkeypatch.setattr(ops, name, seg_reduce)
        else:
            monkeypatch.setattr(ops, name, fn)

    def group(ids, V, pad):
        g = raw_group_ids(ids, V, pad)
        return ops.IdGroups(g.unique_ids, g.seg_offsets, g.sorted_pos, g.num, g.n, V)

    monkeypatch.setattr(ops, "raw_group_ids", group)


# ---- LoD pooling + CVM stand-ins -------------------------------------------------------------------
def raw_gather_pool_sum(W, keys, offsets, padding_idx, D=None):
    W = W if D is None else W[:, :D]
    keys, offsets = keys.reshape(-1), offsets.reshape(-1)
    n_bags = offsets.numel() - 1
    lens = offsets[1:] - offsets[:-1]
    bag = torch.repeat_interleave(torch.arange(n_bags), lens)
    rows = raw_gather(W, keys, padding_idx)
    out = torch.zeros(n_bags, W.shape[1]).index_add(0, bag, rows)
    return out, bag.to(torch.int32)


def raw_cvm_fwd(x, use_cvm):
    from oracle import nets
    return nets.cvm(x, use_cvm)


def raw_cvm_bwd(dy, show_click, D, use_cvm):
    return torch.cat([show_click[:, :2], dy[:, 2:] if use_cvm else dy], 1)


# ---- peer-memory exchange stand-ins: `ptrs` is a list of every rank's receive buffer (host tensors
# in shared memory) instead of NVLink mappings; same argument order as ops.raw_shard_*.
def _peer_of(seg, k):
    return int(torch.searchsorted(seg[1:].contiguous(), torch.tensor(k), right=True))


def raw_shard_gather_push(shard, recv_ids, local_pad, cols, recv_seg, dst_pull, ptrs, ld_dst, world):
    rows = raw_gather(shard, recv_ids, local_pad, cols)
    for r in range(world):
        a, b = int(recv_seg[r]), int(recv_seg[r + 1])
        d = int(dst_pull[r])
        ptrs[r][d:d + (b - a), :cols] = rows[a:b]


def _store_rows(rows, D, send_seg, dst_push, ptrs, world):
    for o in range(world):
        a, b = int(send_seg[o]), int(send_seg[o + 1])
        d = int(dst_push[o])
        ptrs[o][d:d + (b - a), :D] = rows[a:b, :D]


def raw_shard_push_rows(rows, D, send_seg, dst_push, ptrs, ld_dst, world):
    _store_rows(rows, D, send_seg, dst_push, ptrs, world)


def raw_shard_fm_grads_push(feat, S, dfeat_dnn, gy1, gy2, inv_perm, F, G, send_seg, dst_push, ptrs,
                            ld_dst, world):
    """Slot k (position p = inv_perm[k] = b*F + f) gets [gy2[b]*(S[b]-feat[b,f]) + dfeat[b,f] | gy1[b] | 0]."""
    B, N, D = feat.shape
    p = inv_perm.to(torch.int64)
    b, f = p // F, p % F
    rows = torch.zeros(p.numel(), G, dtype=feat.dtype)
    rows[:, :D] = gy2[b].unsqueeze(1) * (S[b] - feat[b, f])
    if dfeat_dnn is not None:
        rows[:, :D] += dfeat_dnn[b, f]
    rows[:, D] = gy1[b]
    _store_rows(rows, G, send_seg, dst_push, ptrs, world)
