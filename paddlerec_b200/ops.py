"""Torch-facing wrappers of the C ABI (include/b200rec.h).

Two layers:
  * `raw_*`  — one function per C entry point; takes CUDA tensors, allocates outputs/workspace
               with torch's caching allocator (the "caller owns every buffer" side of the ABI) and
               enqueues on torch's current stream.
  * autograd.Function classes — what the net.py-shaped layers call.  The sparse-table gradients
    are not materialised as dense [V,D] tensors: backward stores a `SelectedRows` (Paddle's name
    for the rows/value pair that `Embedding(sparse=True)` produces) on the owning table object.

There is deliberately no CPU path: a CPU tensor raises.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import check, ptr


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _req(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.B200RecError(
            "%s must be a CUDA tensor: the b200rec hot path has no CPU fallback" % name)
    if t.dtype != dtype:
        raise _lib.B200RecError("%s must be %s, got %s" % (name, dtype, t.dtype))
    return t if t.is_contiguous() else t.contiguous()


# ---- accounting -------------------------------------------------------------------------------
# LAUNCHES counts OUR kernels (not CUB's, not torch's) enqueued through the C ABI; bench.py reports
# it as `gpu_launches`.  KERNELS_PER_CALL is the static number of our kernels each entry point runs.
LAUNCHES = 0
KERNELS_PER_CALL = {
    "embed_fm_fwd": 1, "group_ids": 3, "embed_fm_bwd": 5, "gather": 1, "segment_reduce": 3,
    "shard_gather_push": 1, "shard_push_rows": 1, "shard_fm_grads_push": 1, "rows_to_dense": 1, "sparse_sgd": 1, "sparse_adam": 1, "sparse_adagrad": 1, "cross_v2_fwd": 1,
    "cross_v2_bwd": 2, "shard_bucketize": 2, "tower_split": 1, "tower_relu_bwd_split": 2,
    "tower_prep_weight": 1, "tower_fold_dw": 1, "tc_split": 1, "tc_split_bwd": 2,
    "tc_prep_weight": 1, "tc_linear_fwd": 1, "tc_cross_fwd": 1, "tc_linear_bwd_dx": 1,
    "tc_linear_bwd_dx_db": 2, "tc_linear_bwd_dw": 2, "tc_head_fwd": 1, "tc_head_bwd": 2,
    "auc_update": 1, "sum_sigmoid_fwd": 1, "sum_sigmoid_bwd": 1, "log_loss_mean_fwd": 1, "log_loss_mean_bwd": 1, "din_attn_fwd": 2, "din_attn_bwd": 3, "gather_pool_sum": 2, "cvm_fwd": 1, "cvm_bwd": 1, "hash_keys": 1, "dot_interact_fwd": 1, "dot_interact_bwd": 1,
}
# When set to a list, (name, start_event, end_event) triples are appended around the raw_* calls
# (all of them, or only the names in EVENT_FILTER when that is a set) — bench.py's per-kernel times.
EVENTS = None
EVENT_FILTER = None


def _count(name: str) -> None:
    global LAUNCHES
    LAUNCHES += KERNELS_PER_CALL[name]


class _Timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        self.on = EVENTS is not None and (EVENT_FILTER is None or self.name in EVENT_FILTER)
        if self.on:
            self.start = torch.cuda.Event(enable_timing=True)
            self.end = torch.cuda.Event(enable_timing=True)
            self.start.record()
        return self

    def __exit__(self, *exc):
        if self.on and EVENTS is not None:
            self.end.record()
            EVENTS.append((self.name, self.start, self.end))
        return False


_ws_cache = {}


def workspace(nbytes: int, device, tag: str = "default") -> torch.Tensor:
    """A grow-only per-(device, tag) scratch buffer.  Safe because every consumer runs on the
    current stream in program order."""
    key = (device.index if device.index is not None else torch.cuda.current_device(), tag)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


# ------------------------------------------------------------------------------------------------
@dataclass
class IdGroups:
    """Output of b200rec_group_ids: positions grouped by distinct id."""
    unique_ids: torch.Tensor   # int64 [n]   (first num[0] valid)
    seg_offsets: torch.Tensor  # int32 [n+1]
    sorted_pos: torch.Tensor   # int32 [n]
    num: torch.Tensor          # int32 [2] on device: {#distinct, #kept}
    n: int
    height: int                # V


@dataclass
class SelectedRows:
    """rows/value pair: gradient of a [height, D] table restricted to the touched rows.
    Mirrors Paddle's SelectedRows (what paddle.nn.Embedding(sparse=True) hands the optimizer),
    already merged (each row appears once)."""
    rows: torch.Tensor    # int64 [n]  (first num[0] valid)
    value: torch.Tensor   # f32 [n, ld] (first num[0] rows valid; the rest is unspecified)
    num: torch.Tensor     # int32 [2] device
    height: int
    ncols: Optional[int] = None   # gradient columns (<= ld); None = all of value's columns

    @property
    def cols(self) -> int:
        return self.value.shape[1] if self.ncols is None else self.ncols

    def to_dense(self) -> torch.Tensor:
        out = torch.zeros(self.height, self.cols, dtype=torch.float32, device=self.value.device)
        raw_rows_to_dense(self, out)
        return out

    def count(self) -> int:
        return int(self.num[0].item())


def raw_oob_count(reset: bool = True) -> int:
    lib = _lib.load()
    out = ctypes.c_uint64(0)
    check(lib.b200rec_oob_count(ctypes.byref(out), int(reset), _stream()), "oob_count")
    return int(out.value)


def raw_embed_fm_fwd(W, W1, ids, dense, dense_w, dense_w1, padding_idx: int, want_S: bool = True,
                     D: Optional[int] = None):
    """W: [V, ldw] table.  W1: [V]/[V,1] first-order table, or None for the FUSED slot layout
    (row = [D emb | w1 | pad], so W1 = W + D with the same stride; `D` must then be given)."""
    lib = _lib.load()
    W = _req(W, torch.float32, "W")
    ids = _req(ids, torch.int64, "ids")
    dense = _req(dense, torch.float32, "dense")
    dense_w = _req(dense_w, torch.float32, "dense_w")
    dense_w1 = _req(dense_w1, torch.float32, "dense_w1")
    B, F = ids.shape
    Dn = dense.shape[1]
    V, ldw = W.shape
    if W1 is None:
        assert D is not None and D + 1 <= ldw, "fused layout needs D and a slot of >= D+1 floats"
        w1_ptr, ldw1 = ctypes.c_void_p(W.data_ptr() + 4 * D), ldw
    else:
        W1 = _req(W1, torch.float32, "W1")
        D = ldw if D is None else D
        assert W1.numel() == V
        w1_ptr, ldw1 = ptr(W1), 1
    assert dense.shape[0] == B and dense_w.numel() == Dn * D and dense_w1.numel() == Dn
    dev = W.device
    feat = torch.empty(B, F + Dn, D, dtype=torch.float32, device=dev)
    y1 = torch.empty(B, dtype=torch.float32, device=dev)
    y2 = torch.empty(B, dtype=torch.float32, device=dev)
    S = torch.empty(B, D, dtype=torch.float32, device=dev) if want_S else None
    with _Timed("embed_fm_fwd"):
        check(lib.b200rec_embed_fm_fwd(ptr(W), ldw, w1_ptr, ldw1, ptr(ids), ptr(dense), ptr(dense_w),
                                       ptr(dense_w1), ptr(feat), ptr(y1), ptr(y2), ptr(S), B, F, Dn,
                                       D, V, int(padding_idx), _stream()), "embed_fm_fwd")
    _count("embed_fm_fwd")
    return feat, y1, y2, S


def raw_group_ids(ids: torch.Tensor, V: int, padding_idx: int, ws_tag: str = "group") -> IdGroups:
    """ws_tag: a call enqueued on a SIDE stream must not share the scratch buffer of the calls on
    the main stream (the workspace cache is ordered by stream, not across streams)."""
    lib = _lib.load()
    ids = _req(ids, torch.int64, "ids").reshape(-1)
    n = ids.numel()
    dev = ids.device
    nbytes = ctypes.c_size_t(0)
    check(lib.b200rec_group_ids_workspace_bytes(n, V, ctypes.byref(nbytes)), "group_ids_ws")
    ws = workspace(nbytes.value, dev, ws_tag)
    unique_ids = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    seg_offsets = torch.empty(n + 1, dtype=torch.int32, device=dev)
    sorted_pos = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    num = torch.empty(2, dtype=torch.int32, device=dev)
    check(lib.b200rec_group_ids(ptr(ids), n, V, int(padding_idx), ptr(unique_ids), ptr(seg_offsets),
                                ptr(sorted_pos), ptr(num), ptr(ws), ws.numel(), _stream()),
          "group_ids")
    _count("group_ids")
    return IdGroups(unique_ids, seg_offsets, sorted_pos, num, n, V)


# The grouping (a radix sort + run-length pass over the ids) only depends on the ids, but its
# consumer is the BACKWARD kernel.  Started in the forward on a side stream it runs under the
# tower's tensor-bound GEMMs instead of serially in front of the segmented reduction
# (0.35 ms of a 1.6 ms DeepFM step when serial).  Opt-in (B200REC_GROUP_AHEAD=1 / set_group_ahead):
# written after the round's GPU budget ended, so it has not been run or timed on a GPU yet.
GROUP_AHEAD = os.environ.get("B200REC_GROUP_AHEAD", "0") == "1"
_group_streams: dict = {}


def set_group_ahead(on: bool) -> None:
    global GROUP_AHEAD
    GROUP_AHEAD = bool(on)


def group_ids_ahead(ids: torch.Tensor, V: int, padding_idx: int):
    """Enqueue b200rec_group_ids for `ids` on the grouping side stream; returns (IdGroups, event)
    or None when disabled.  `groups_ready` makes the current stream wait for it."""
    if not GROUP_AHEAD or not ids.is_cuda:
        return None
    dev = ids.device
    main = torch.cuda.current_stream(dev)
    side = _group_streams.get(dev.index)
    if side is None:
        side = _group_streams[dev.index] = torch.cuda.Stream(device=dev)
    side.wait_stream(main)                      # ids may have been produced / copied on `main`
    with torch.cuda.stream(side):
        groups = raw_group_ids(ids, V, padding_idx, ws_tag="group_ahead")
        ev = torch.cuda.Event()
        ev.record(side)
    for t in (groups.unique_ids, groups.seg_offsets, groups.sorted_pos, groups.num):
        t.record_stream(main)                   # allocated on `side`, consumed (and freed) on `main`
    ids.record_stream(side)
    return groups, ev


def groups_ready(ahead) -> IdGroups:
    groups, ev = ahead
    torch.cuda.current_stream(groups.num.device).wait_event(ev)
    return groups


def raw_embed_fm_bwd(feat, S, dfeat_dnn, gy1, gy2, dense, seg_offsets, sorted_pos, num, F: int,
                     fused_cols: int = 0):
    """Returns (dW_rows, dW1_rows, ddense_w [Dn,D], ddense_w1 [Dn]).
    fused_cols == 0: dW_rows [n,D], dW1_rows [n].
    fused_cols == G (>= D+1, multiple of 4): ONE buffer dW_rows [n,G] = [D | g1 | zeros], and
    dW1_rows is None."""
    lib = _lib.load()
    feat = _req(feat, torch.float32, "feat")
    S = _req(S, torch.float32, "S")
    if dfeat_dnn is not None:
        dfeat_dnn = _req(dfeat_dnn, torch.float32, "dfeat_dnn")
    gy1 = _req(gy1, torch.float32, "gy1").reshape(-1)
    gy2 = _req(gy2, torch.float32, "gy2").reshape(-1)
    dense = _req(dense, torch.float32, "dense")
    B, N, D = feat.shape
    Dn = N - F
    n = B * F
    dev = feat.device
    nbytes = ctypes.c_size_t(0)
    check(lib.b200rec_embed_fm_bwd_workspace_bytes(B, F, Dn, D, ctypes.byref(nbytes)), "fm_bwd_ws")
    ws = workspace(nbytes.value, dev, "fm_bwd")
    if fused_cols:
        assert fused_cols >= D + 1
        dW_rows = torch.empty(max(n, 1), fused_cols, dtype=torch.float32, device=dev)
        dW1_rows = None
        dw1_ptr = ctypes.c_void_p(dW_rows.data_ptr() + 4 * D)
        ld_dw, ld_dw1, zero_pad = fused_cols, fused_cols, fused_cols - D - 1
    else:
        dW_rows = torch.empty(max(n, 1), D, dtype=torch.float32, device=dev)
        dW1_rows = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
        dw1_ptr, ld_dw, ld_dw1, zero_pad = ptr(dW1_rows), D, 1, 0
    ddense_w = torch.empty(Dn, D, dtype=torch.float32, device=dev)
    ddense_w1 = torch.empty(Dn, dtype=torch.float32, device=dev)
    check(lib.b200rec_embed_fm_bwd(ptr(feat), ptr(S), ptr(dfeat_dnn), ptr(gy1), ptr(gy2),
                                   ptr(dense), ptr(seg_offsets), ptr(sorted_pos), ptr(num),
                                   ptr(dW_rows), ld_dw, dw1_ptr, ld_dw1, zero_pad, ptr(ddense_w),
                                   ptr(ddense_w1), B, F, Dn, D, ptr(ws), ws.numel(), _stream()),
          "embed_fm_bwd")
    _count("embed_fm_bwd")
    return dW_rows, dW1_rows, ddense_w, ddense_w1


def raw_gather(W: torch.Tensor, ids: torch.Tensor, padding_idx: int,
               D: Optional[int] = None) -> torch.Tensor:
    """out[..., :] = W[ids, :D]; W is [V, ldw] (D defaults to ldw)."""
    lib = _lib.load()
    W = _req(W, torch.float32, "W")
    ids = _req(ids, torch.int64, "ids")
    V, ldw = W.shape
    D = ldw if D is None else D
    n = ids.numel()
    out = torch.empty(*ids.shape, D, dtype=torch.float32, device=W.device)
    check(lib.b200rec_gather(ptr(W), ldw, ptr(ids), ptr(out), n, D, V, int(padding_idx), _stream()),
          "gather")
    _count("gather")
    return out


def raw_gather_pool_sum(W, keys, offsets, padding_idx: int, D: Optional[int] = None):
    """Sum-pooled lookup of variable-length key lists.  keys int64 [nnz], offsets int64
    [n_bags+1].  Returns (out [n_bags, D], bag_of_pos int32 [nnz])."""
    lib = _lib.load()
    W = _req(W, torch.float32, "W")
    keys = _req(keys, torch.int64, "keys").reshape(-1)
    offsets = _req(offsets, torch.int64, "offsets").reshape(-1)
    V, ldw = W.shape
    D = ldw if D is None else D
    n_bags = offsets.numel() - 1
    out = torch.empty(n_bags, D, dtype=torch.float32, device=W.device)
    bag_of_pos = torch.empty(max(keys.numel(), 1), dtype=torch.int32, device=W.device)
    check(lib.b200rec_gather_pool_sum(ptr(W), ldw, ptr(keys), ptr(offsets), ptr(out),
                                      ptr(bag_of_pos), n_bags, D, V, int(padding_idx), _stream()),
          "gather_pool_sum")
    _count("gather_pool_sum")
    return out, bag_of_pos


def raw_segment_reduce(dOut: torch.Tensor, groups_seg, groups_pos, num, n: int,
                       row_of_pos=None) -> torch.Tensor:
    lib = _lib.load()
    dOut = _req(dOut, torch.float32, "dOut")
    D = dOut.shape[-1]
    rows = torch.empty(max(n, 1), D, dtype=torch.float32, device=dOut.device)
    nbytes = ctypes.c_size_t(0)
    check(lib.b200rec_segment_reduce_workspace_bytes(n, D, ctypes.byref(nbytes)), "segment_reduce_ws")
    ws = workspace(nbytes.value, dOut.device, "segred")
    check(lib.b200rec_segment_reduce(ptr(dOut), ptr(row_of_pos), ptr(groups_seg), ptr(groups_pos),
                                     ptr(num), ptr(rows), n, D, ptr(ws), ws.numel(), _stream()),
          "segment_reduce")
    _count("segment_reduce")
    return rows


def merge_selected_rows(a: SelectedRows, b: SelectedRows) -> SelectedRows:
    """Paddle's merge-add of two SelectedRows gradients of the same table (a table looked up twice
    in one forward, or gradients accumulated over micro-batches): concatenate the valid rows and
    reduce duplicates with the same sorted segment reduce the backward uses (deterministic).
    Rare path: reads the two row counts on the host."""
    na, nb = a.count(), b.count()
    cols = min(a.cols, b.cols)
    rows = torch.cat([a.rows[:na], b.rows[:nb]])
    vals = torch.cat([a.value[:na, :cols], b.value[:nb, :cols]]).contiguous()
    groups = raw_group_ids(rows, a.height, -1)
    merged = raw_segment_reduce(vals, groups.seg_offsets, groups.sorted_pos, groups.num, groups.n)
    return SelectedRows(groups.unique_ids, merged, groups.num, a.height,
                        cols if a.ncols is not None else None)


def raw_rows_to_dense(sr: SelectedRows, dW: torch.Tensor) -> None:
    lib = _lib.load()
    dW = _req(dW, torch.float32, "dW")
    n, ld_rows = sr.value.shape
    check(lib.b200rec_rows_to_dense(ptr(sr.rows), ptr(sr.value), ld_rows, ptr(sr.num), ptr(dW),
                                    dW.shape[1], n, sr.cols, sr.height, _stream()), "rows_to_dense")
    _count("rows_to_dense")


def raw_sparse_sgd(W: torch.Tensor, sr: SelectedRows, lr: float) -> None:
    lib = _lib.load()
    n, ld_rows = sr.value.shape[0], sr.value.stride(0)     # column views of a table are allowed
    check(lib.b200rec_sparse_sgd(ptr(W), W.stride(0), ptr(sr.rows), ptr(sr.value), ld_rows,
                                 ptr(sr.num), n, sr.cols, sr.height, float(lr), _stream()),
          "sparse_sgd")
    _count("sparse_sgd")


def raw_sparse_adam(W, m, v, sr: SelectedRows, lr, beta1, beta2, eps, beta1_pow, beta2_pow) -> None:
    lib = _lib.load()
    n, ld_rows = sr.value.shape[0], sr.value.stride(0)
    check(lib.b200rec_sparse_adam(ptr(W), ptr(m), ptr(v), W.stride(0), ptr(sr.rows), ptr(sr.value),
                                  ld_rows, ptr(sr.num), n, sr.cols, sr.height, float(lr),
                                  float(beta1), float(beta2), float(eps), float(beta1_pow),
                                  float(beta2_pow), _stream()), "sparse_adam")
    _count("sparse_adam")


def raw_sparse_adagrad(W, g2sum, sr: SelectedRows, lr, initial_g2sum, lo, hi) -> None:
    lib = _lib.load()
    n, ld_rows = sr.value.shape[0], sr.value.stride(0)
    check(lib.b200rec_sparse_adagrad(ptr(W), ptr(g2sum), W.stride(0), ptr(sr.rows), ptr(sr.value),
                                     ld_rows, ptr(sr.num), n, sr.cols, sr.height, float(lr),
                                     float(initial_g2sum), float(lo), float(hi), _stream()),
          "sparse_adagrad")
    _count("sparse_adagrad")


def raw_cross_v2_fwd(x0, xl, xw, bias) -> torch.Tensor:
    lib = _lib.load()
    x0 = _req(x0, torch.float32, "x0")
    xl = _req(xl, torch.float32, "xl")
    xw = _req(xw, torch.float32, "xw")
    bias = _req(bias, torch.float32, "bias")
    B, C = x0.shape
    out = torch.empty_like(x0)
    check(lib.b200rec_cross_v2_fwd(ptr(x0), ptr(xl), ptr(xw), ptr(bias), ptr(out), B, C, _stream()),
          "cross_v2_fwd")
    _count("cross_v2_fwd")
    return out


def raw_cross_v2_bwd(dout, x0, xw, bias):
    """returns (dxw, dx0, dbias)."""
    lib = _lib.load()
    dout = _req(dout, torch.float32, "dout")
    B, C = dout.shape
    nbytes = ctypes.c_size_t(0)
    check(lib.b200rec_cross_bwd_workspace_bytes(B, C, ctypes.byref(nbytes)), "cross_ws")
    ws = workspace(nbytes.value, dout.device, "cross")
    dxw = torch.empty_like(dout)
    dx0 = torch.empty_like(dout)
    dbias = torch.empty(C, dtype=torch.float32, device=dout.device)
    check(lib.b200rec_cross_v2_bwd(ptr(dout), ptr(x0), ptr(xw), ptr(bias), ptr(dxw), ptr(dx0),
                                   ptr(dbias), B, C, ptr(ws), ws.numel(), _stream()), "cross_v2_bwd")
    _count("cross_v2_bwd")
    return dxw, dx0, dbias


def raw_shard_bucketize(ids: torch.Tensor, world: int, V: int):
    """Returns (send_ids [n], perm [n] i64, inv_perm [n] i32, counts [world] i64 device)."""
    lib = _lib.load()
    ids = _req(ids, torch.int64, "ids").reshape(-1)
    n = ids.numel()
    dev = ids.device
    nbytes = ctypes.c_size_t(0)
    check(lib.b200rec_shard_bucketize_workspace_bytes(n, world, ctypes.byref(nbytes)), "shard_ws")
    ws = workspace(nbytes.value, dev, "shard")
    send_ids = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    perm = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    inv_perm = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    counts = torch.empty(world, dtype=torch.int64, device=dev)
    check(lib.b200rec_shard_bucketize(ptr(ids), n, world, V, ptr(send_ids), ptr(perm),
                                      ptr(inv_perm), ptr(counts), ptr(ws), ws.numel(), _stream()),
          "shard_bucketize")
    _count("shard_bucketize")
    return send_ids[:n], perm[:n], inv_perm[:n], counts


def raw_tower_split(x: torch.Tensor, bias, relu: bool) -> torch.Tensor:
    """fp32 [M,K] -> bf16 [M,2K] = [hi | lo] of relu?(x + bias?)."""
    lib = _lib.load()
    x = _req(x, torch.float32, "x")
    M, K = x.shape
    out = torch.empty(M, 2 * K, dtype=torch.bfloat16, device=x.device)
    check(lib.b200rec_tower_split(ptr(x), ptr(bias), int(relu), ptr(out), M, K, _stream()),
          "tower_split")
    _count("tower_split")
    return out


def raw_tower_relu_bwd_split(dy: torch.Tensor, act):
    """Returns (dz bf16 [M,2N], dbias [N])."""
    lib = _lib.load()
    dy = _req(dy, torch.float32, "dy")
    M, N = dy.shape
    nbytes = ctypes.c_size_t(0)
    check(lib.b200rec_tower_bwd_workspace_bytes(M, N, ctypes.byref(nbytes)), "tower_ws")
    ws = workspace(nbytes.value, dy.device, "tower")
    dz = torch.empty(M, 2 * N, dtype=torch.bfloat16, device=dy.device)
    dbias = torch.empty(N, dtype=torch.float32, device=dy.device)
    check(lib.b200rec_tower_relu_bwd_split(ptr(dy), ptr(act), ptr(dz), ptr(dbias), M, N, ptr(ws),
                                           ws.numel(), _stream()), "tower_relu_bwd_split")
    _count("tower_relu_bwd_split")
    return dz, dbias


def raw_tower_prep_weight(W: torch.Tensor):
    """W fp32 [K,N] -> (W2r bf16 [2K,N], W2c bf16 [K,2N], Wlo bf16 [K,N])."""
    lib = _lib.load()
    W = _req(W, torch.float32, "W")
    K, N = W.shape
    W2r = torch.empty(2 * K, N, dtype=torch.bfloat16, device=W.device)
    W2c = torch.empty(K, 2 * N, dtype=torch.bfloat16, device=W.device)
    Wlo = torch.empty(K, N, dtype=torch.bfloat16, device=W.device)
    check(lib.b200rec_tower_prep_weight(ptr(W), ptr(W2r), ptr(W2c), ptr(Wlo), K, N, _stream()),
          "tower_prep_weight")
    _count("tower_prep_weight")
    return W2r, W2c, Wlo


def raw_tower_fold_dw(Mx: torch.Tensor, K: int, N: int) -> torch.Tensor:
    lib = _lib.load()
    Mx = _req(Mx, torch.float32, "Mx")
    dW = torch.empty(K, N, dtype=torch.float32, device=Mx.device)
    check(lib.b200rec_tower_fold_dw(ptr(Mx), ptr(dW), K, N, _stream()), "tower_fold_dw")
    _count("tower_fold_dw")
    return dW


# ---- sharded exchange over NVLink peer memory (csrc/shard.cuh) ----------------------------------
def _peer_tables(seg_dev: torch.Tensor, dst_dev: torch.Tensor, peer_ptrs, world: int):
    """The kernels read world+1 entries of seg_dev and world of dst_dev on the device and store
    through peer_ptrs[0..world): a short table would send rows to addresses read past its end."""
    seg_dev = _req(seg_dev, torch.int64, "seg_dev")
    dst_dev = _req(dst_dev, torch.int64, "dst_dev")
    if seg_dev.numel() != world + 1 or dst_dev.numel() != world:
        raise _lib.B200RecError(
            "shard exchange: seg_dev must have world+1 = %d entries and dst_dev world = %d, got %d "
            "and %d" % (world + 1, world, seg_dev.numel(), dst_dev.numel()))
    if len(peer_ptrs) < world:
        raise _lib.B200RecError("shard exchange: %d peer pointers for world=%d"
                                % (len(peer_ptrs), world))
    return seg_dev, dst_dev


def raw_shard_gather_push(shard: torch.Tensor, recv_ids: torch.Tensor, local_pad: int, D: int,
                          seg_dev: torch.Tensor, dst_dev: torch.Tensor, peer_ptrs, ld_dst: int,
                          world: int) -> None:
    """Owner side of the pull: the rows peer r asked for are gathered from `shard` and stored
    directly into r's receive buffer (peer_ptrs: ctypes uint64 array of mapped base pointers)."""
    lib = _lib.load()
    shard = _req(shard, torch.float32, "shard") if shard.is_contiguous() else shard
    recv_ids = _req(recv_ids, torch.int64, "recv_ids")
    seg_dev, dst_dev = _peer_tables(seg_dev, dst_dev, peer_ptrs, world)
    check(lib.b200rec_shard_gather_push(ptr(shard), shard.stride(0), D, shard.shape[0],
                                        int(local_pad), ptr(recv_ids), ptr(seg_dev), ptr(dst_dev),
                                        peer_ptrs, ld_dst, world, recv_ids.numel(), _stream()),
          "shard_gather_push")
    _count("shard_gather_push")


def raw_shard_fm_grads_push(feat, S, dfeat_dnn, gy1, gy2, inv_perm, F: int, G: int, seg_dev, dst_dev,
                            peer_ptrs, ld_dst: int, world: int) -> None:
    """Sparse half of the DeepFM FM backward fused with the gradient push (sharded path): the
    per-slot gradient rows go straight into the owners' receive buffers over NVLink."""
    lib = _lib.load()
    feat = _req(feat, torch.float32, "feat")
    S = _req(S, torch.float32, "S")
    if dfeat_dnn is not None:
        dfeat_dnn = _req(dfeat_dnn, torch.float32, "dfeat_dnn")
    B, N, D = feat.shape
    seg_dev, dst_dev = _peer_tables(seg_dev, dst_dev, peer_ptrs, world)
    check(lib.b200rec_shard_fm_grads_push(ptr(feat), ptr(S), ptr(dfeat_dnn),
                                          ptr(_req(gy1, torch.float32, "gy1")),
                                          ptr(_req(gy2, torch.float32, "gy2")),
                                          ptr(_req(inv_perm, torch.int32, "inv_perm")), ptr(seg_dev),
                                          ptr(dst_dev), peer_ptrs, ld_dst, world, B, F, N - F, D, G,
                                          _stream()), "shard_fm_grads_push")
    _count("shard_fm_grads_push")


def raw_shard_push_rows(rows: torch.Tensor, D: int, seg_dev: torch.Tensor, dst_dev: torch.Tensor,
                        peer_ptrs, ld_dst: int, world: int) -> None:
    """Requester side of the push: gradient rows in bucket order -> the owners' receive buffers."""
    lib = _lib.load()
    rows = _req(rows, torch.float32, "rows")
    seg_dev, dst_dev = _peer_tables(seg_dev, dst_dev, peer_ptrs, world)
    check(lib.b200rec_shard_push_rows(ptr(rows), rows.stride(0), D, ptr(seg_dev), ptr(dst_dev),
                                      peer_ptrs, ld_dst, world, rows.shape[0], _stream()),
          "shard_push_rows")
    _count("shard_push_rows")


# ---- tcgen05 tower GEMMs (csrc/tc_gemm.cuh) ---------------------------------------------------
def plane_ld(n: int, ones_col: bool = False) -> int:
    """Plane pitch of a logical width n (+1 with a ones column): the hi and lo planes must both be
    16-byte aligned."""
    return (int(n) + int(ones_col) + 7) // 8 * 8


def _planes(M: int, n: int, device, ones_col: bool = False) -> torch.Tensor:
    return torch.empty(M, 2 * plane_ld(n, ones_col), dtype=torch.bfloat16, device=device)


def raw_tc_split(x: torch.Tensor, bias=None, relu: bool = False,
                 ones_col: bool = False) -> torch.Tensor:
    """fp32 [M,K] -> planes [M, 2*ld] of relu?(x + bias?); ones_col: hi[:, K] = 1 (see
    raw_tc_linear_bwd_dw)."""
    lib = _lib.load()
    x = _req(x, torch.float32, "x")
    M, K = x.shape
    out = _planes(M, K, x.device, ones_col)
    check(lib.b200rec_tc_split(ptr(x), K, ptr(bias), int(relu), ptr(out), out.shape[1] // 2, M, K,
                               int(ones_col), _stream()), "tc_split")
    _count("tc_split")
    return out


def raw_tc_split_bwd(dy: torch.Tensor, mask_planes):
    """g = dy * (mask_hi > 0) -> (planes(g) [M, 2*ld(N)], dbias [N])."""
    lib = _lib.load()
    dy = _req(dy, torch.float32, "dy")
    M, N = dy.shape
    nbytes = ctypes.c_size_t(0)
    check(lib.b200rec_tower_bwd_workspace_bytes(M, N, ctypes.byref(nbytes)), "tower_ws")
    ws = workspace(nbytes.value, dy.device, "tower")
    g = _planes(M, N, dy.device)
    dbias = torch.empty(N, dtype=torch.float32, device=dy.device)
    ld_mask = mask_planes.shape[1] // 2 if mask_planes is not None else 0
    check(lib.b200rec_tc_split_bwd(ptr(dy), ptr(mask_planes), ld_mask, ptr(g), plane_ld(N),
                                   ptr(dbias), M, N, ptr(ws), ws.numel(), _stream()),
          "tc_split_bwd")
    _count("tc_split_bwd")
    return g, dbias


def raw_tc_prep_weight(W: torch.Tensor, want_w: bool = True, want_wt: bool = True):
    """W fp32 [K,N] -> (planes(W) [K, 2*ld(N)], planes(W^T) [N, 2*ld(K)])."""
    lib = _lib.load()
    W = _req(W, torch.float32, "W")
    K, N = W.shape
    Wp = _planes(K, N, W.device) if want_w else None
    WTp = _planes(N, K, W.device) if want_wt else None
    check(lib.b200rec_tc_prep_weight(ptr(W), K, N, ptr(Wp), plane_ld(N), ptr(WTp), plane_ld(K),
                                     _stream()), "tc_prep_weight")
    _count("tc_prep_weight")
    return Wp, WTp


def raw_tc_linear_fwd(a_planes: torch.Tensor, K: int, WTp: torch.Tensor, N: int, bias, relu: bool,
                      want_f32: bool, want_planes: bool, ones_col: bool = False):
    """y = a @ W + bias (ReLU optional) on the tcgen05 tensor cores.  Returns (y fp32 [M,N] | None,
    planes(y) [M, 2*ld] | None)."""
    lib = _lib.load()
    M = a_planes.shape[0]
    dev = a_planes.device
    y = torch.empty(M, N, dtype=torch.float32, device=dev) if want_f32 else None
    yp = _planes(M, N, dev, ones_col) if want_planes else None
    check(lib.b200rec_tc_linear_fwd(ptr(a_planes), a_planes.shape[1] // 2, ptr(WTp),
                                    WTp.shape[1] // 2, ptr(bias), int(relu), ptr(y), N, ptr(yp),
                                    yp.shape[1] // 2 if yp is not None else 0,
                                    int(ones_col and want_planes), M, N, K, _stream()),
          "tc_linear_fwd")
    _count("tc_linear_fwd")
    return y, yp


def raw_tc_cross_fwd(xl_planes, WTp, bias, x0, xl, want_planes: bool, want_u: bool = False,
                     ones_col: bool = False):
    """CrossNetV2 layer out = x0 * u + xl, u = xl @ W + b, with the Hadamard/residual epilogue fused
    into the tcgen05 GEMM.  Returns (out fp32 [M,C], planes(out) | None, u fp32 | None)."""
    lib = _lib.load()
    x0 = _req(x0, torch.float32, "x0")
    xl = _req(xl, torch.float32, "xl")
    M, C = x0.shape
    out = torch.empty(M, C, dtype=torch.float32, device=x0.device)
    u = torch.empty(M, C, dtype=torch.float32, device=x0.device) if want_u else None
    op = _planes(M, C, x0.device, ones_col) if want_planes else None
    check(lib.b200rec_tc_cross_fwd(ptr(xl_planes), xl_planes.shape[1] // 2, ptr(WTp),
                                   WTp.shape[1] // 2, ptr(bias), ptr(x0), ptr(xl), C, ptr(u),
                                   ptr(out), C, ptr(op), op.shape[1] // 2 if op is not None else 0,
                                   int(ones_col and want_planes), M, C, _stream()), "tc_cross_fwd")
    _count("tc_cross_fwd")
    return out, op, u


def _tc_bwd_ws(M: int, K: int, N: int, device, tag: str = "tc_bwd") -> torch.Tensor:
    nbytes = ctypes.c_size_t(0)
    lib = _lib.load()
    check(lib.b200rec_tc_linear_bwd_workspace_bytes(M, K, N, ctypes.byref(nbytes)),
          "tc_linear_bwd_ws")
    return workspace(nbytes.value, device, tag)


def raw_tc_linear_bwd_dx(g_planes, N: int, Wp, K: int, mask_planes, want_f32: bool,
                         want_planes: bool, want_dbias: bool, addend=None):
    """dx = g @ W^T with the ReLU mask of the layer input, the hi/lo split and the bias column-sum
    of the PREVIOUS layer fused into the epilogue.  Returns (dx fp32 | None, planes | None,
    dbias_prev [K] | None)."""
    lib = _lib.load()
    M = g_planes.shape[0]
    dev = g_planes.device
    dx = torch.empty(M, K, dtype=torch.float32, device=dev) if want_f32 else None
    dxp = _planes(M, K, dev) if want_planes else None
    db = torch.empty(K, dtype=torch.float32, device=dev) if want_dbias else None
    ws = _tc_bwd_ws(M, K, N, dev)
    ld_mask = mask_planes.shape[1] // 2 if mask_planes is not None else 0
    check(lib.b200rec_tc_linear_bwd_dx(ptr(g_planes), g_planes.shape[1] // 2, ptr(Wp),
                                       Wp.shape[1] // 2, ptr(mask_planes), ld_mask,
                                       ptr(_req(addend, torch.float32, "addend")
                                           if addend is not None else None), ptr(dx), K,
                                       ptr(dxp), plane_ld(K), ptr(db), M, K, N, ptr(ws), ws.numel(),
                                       _stream()), "tc_linear_bwd_dx")
    _count("tc_linear_bwd_dx_db" if want_dbias else "tc_linear_bwd_dx")
    return dx, dxp, db


def raw_tc_linear_bwd_dw(a_planes, K: int, g_planes, N: int, bias_row: bool = False,
                         ws_tag: str = "tc_bwd"):
    """dW [K,N] = a^T @ g (batch-split tcgen05 GEMM + fixed-order reduce).  With bias_row the
    operand `a` carries a column of ones at index K (ones_col of raw_tc_split / raw_tc_linear_fwd)
    and the result is (dW [K,N], dbias [N]) — the bias gradient is row K of the same GEMM."""
    lib = _lib.load()
    M = a_planes.shape[0]
    dev = a_planes.device
    if bias_row:
        K = K + 1
    dW = torch.empty(K, N, dtype=torch.float32, device=dev)
    ws = _tc_bwd_ws(M, K, N, dev, ws_tag)
    check(lib.b200rec_tc_linear_bwd_dw(ptr(a_planes), a_planes.shape[1] // 2, ptr(g_planes),
                                       g_planes.shape[1] // 2, ptr(dW), M, K, N, ptr(ws),
                                       ws.numel(), _stream()), "tc_linear_bwd_dw")
    _count("tc_linear_bwd_dw")
    if bias_row:
        return dW[:K - 1], dW[K - 1]
    return dW


def raw_tc_head_fwd(a_planes, K: int, w, bias) -> torch.Tensor:
    """y [M,1] = a @ w + bias for a width-1 last layer (w fp32 [K,1] or [K]): one streaming pass."""
    lib = _lib.load()
    M = a_planes.shape[0]
    y = torch.empty(M, 1, dtype=torch.float32, device=a_planes.device)
    check(lib.b200rec_tc_head_fwd(ptr(a_planes), a_planes.shape[1] // 2, K,
                                  ptr(_req(w.detach().reshape(-1), torch.float32, "w")), ptr(bias),
                                  ptr(y), M, _stream()), "tc_head_fwd")
    _count("tc_head_fwd")
    return y


def raw_tc_head_bwd(a_planes, K: int, w, dy):
    """Backward of the width-1 head: (planes(g) [M, 2*ld(K)] with g = dy * w^T masked by a_hi > 0,
    dW [K,1], db [1]) in one streaming pass + a fixed-order reduce."""
    lib = _lib.load()
    M = a_planes.shape[0]
    dev = a_planes.device
    g = _planes(M, K, dev)
    dW = torch.empty(K, 1, dtype=torch.float32, device=dev)
    db = torch.empty(1, dtype=torch.float32, device=dev)
    nbytes = ctypes.c_size_t(0)
    check(lib.b200rec_tc_head_bwd_workspace_bytes(K, ctypes.byref(nbytes)), "tc_head_bwd_ws")
    ws = workspace(nbytes.value, dev, "tc_head")
    check(lib.b200rec_tc_head_bwd(ptr(a_planes), a_planes.shape[1] // 2, K,
                                  ptr(_req(w.detach().reshape(-1), torch.float32, "w")),
                                  ptr(_req(dy.reshape(-1), torch.float32, "dy")), ptr(g),
                                  g.shape[1] // 2, ptr(dW), ptr(db), M, ptr(ws), ws.numel(),
                                  _stream()), "tc_head_bwd")
    _count("tc_head_bwd")
    return g, dW, db


# ---- CTR head: sigmoid of the summed logits, mean log-loss (csrc/ctr_head.cuh) ------------------
class _SumSigmoid(torch.autograd.Function):
    """pred = sigmoid(a + b + c): ONE kernel each way (the reference's add, add, sigmoid and their
    three backward kernels are pure launch latency at [B,1])."""

    @staticmethod
    def forward(ctx, a, b, c):
        lib = _lib.load()
        a, b, c = (None if t is None else _req(t.reshape(-1), torch.float32, "logit part")
                   for t in (a, b, c))
        pred = torch.empty_like(a)
        check(lib.b200rec_sum_sigmoid_fwd(ptr(a), ptr(b), ptr(c), ptr(pred), a.numel(), _stream()),
              "sum_sigmoid_fwd")
        _count("sum_sigmoid_fwd")
        ctx.save_for_backward(pred)
        return pred.reshape(-1, 1)

    @staticmethod
    def backward(ctx, dpred):
        lib = _lib.load()
        (pred,) = ctx.saved_tensors
        dpred = _req(dpred.reshape(-1), torch.float32, "dpred")
        dlogit = torch.empty_like(pred)
        check(lib.b200rec_sum_sigmoid_bwd(ptr(pred), ptr(dpred), ptr(dlogit), pred.numel(),
                                          _stream()), "sum_sigmoid_bwd")
        _count("sum_sigmoid_bwd")
        g = dlogit.reshape(-1, 1)
        return tuple(g if need else None for need in ctx.needs_input_grad)


def sum_sigmoid(a, b=None, c=None):
    """sigmoid(a + b + c) for [B,1] logit parts (b, c optional)."""
    return _SumSigmoid.apply(a, b, c)


_loss_ws = {}


class _LogLossMean(torch.autograd.Function):
    """mean(log_loss(pred, label, eps)) as one deterministic reduction kernel + one backward
    kernel (paddle.nn.functional.log_loss + paddle.mean, deepfm/dygraph_model.py:53-58)."""

    @staticmethod
    def forward(ctx, pred, label, eps):
        lib = _lib.load()
        p = _req(pred.reshape(-1), torch.float32, "pred")
        if label.dtype not in (torch.float32, torch.int64):
            label = label.to(torch.float32)
        y = label.reshape(-1).contiguous()
        key = p.device.index
        ws = _loss_ws.get(key)
        if ws is None:
            nbytes = ctypes.c_size_t(0)
            check(lib.b200rec_log_loss_workspace_bytes(ctypes.byref(nbytes)), "log_loss_ws")
            ws = torch.zeros(nbytes.value, dtype=torch.uint8, device=p.device)   # ticket starts at 0
            _loss_ws[key] = ws
        loss = torch.empty((), dtype=torch.float32, device=p.device)
        check(lib.b200rec_log_loss_mean_fwd(ptr(p), ptr(y), int(y.dtype == torch.int64), float(eps),
                                            ptr(loss), p.numel(), ptr(ws), ws.numel(), _stream()),
              "log_loss_mean_fwd")
        _count("log_loss_mean_fwd")
        ctx.save_for_backward(p, y)
        ctx.eps, ctx.shape = float(eps), pred.shape
        return loss

    @staticmethod
    def backward(ctx, dloss):
        lib = _lib.load()
        p, y = ctx.saved_tensors
        dloss = _req(dloss.reshape(1), torch.float32, "dloss")
        dpred = torch.empty_like(p)
        check(lib.b200rec_log_loss_mean_bwd(ptr(p), ptr(y), int(y.dtype == torch.int64), ctx.eps,
                                            ptr(dloss), ptr(dpred), p.numel(), _stream()),
              "log_loss_mean_bwd")
        _count("log_loss_mean_bwd")
        return dpred.reshape(ctx.shape), None, None


def log_loss_mean(pred, label, eps: float = 1e-4):
    return _LogLossMean.apply(pred, label, eps)


def raw_auc_update(pred: torch.Tensor, label: torch.Tensor, stat_pos: torch.Tensor,
                   stat_neg: torch.Tensor, num_thresholds: int) -> None:
    """paddle.metric.Auc.update as one kernel on the device-resident int64 histograms."""
    lib = _lib.load()
    p = _req(pred.reshape(-1), torch.float32, "pred")
    if label.dtype not in (torch.float32, torch.int64):
        label = label.to(torch.float32)
    y = label.reshape(-1).contiguous()
    check(lib.b200rec_auc_update(ptr(p), ptr(y), int(y.dtype == torch.int64), ptr(stat_pos),
                                 ptr(stat_neg), int(num_thresholds), p.numel(), _stream()),
          "auc_update")
    _count("auc_update")


def tc_debug(key: int, value: int) -> None:
    """Bring-up / tuning knobs of the tcgen05 GEMMs (0: force tile width BN; 0 = automatic)."""
    lib = _lib.load()
    check(lib.b200rec_tc_debug(key, value), "tc_debug")


def tc_timeout_word() -> int:
    """Non-zero if a pipeline watchdog of the tcgen05 kernels fired (which wait, see tc_gemm.cuh)."""
    lib = _lib.load()
    w = ctypes.c_uint(0)
    check(lib.b200rec_tc_timeout_word(ctypes.byref(w)), "tc_timeout_word")
    return int(w.value)


# ------------------------------------------------------------------------------------------------
# autograd glue
class _EmbedFM(torch.autograd.Function):
    """FM.forward of models/rank/deepfm/net.py:105-139 as one kernel (+ one in backward).

    `sink` receives the SelectedRows gradient(s): `sink.accept(sr_w, sr_w1)` for two separate
    tables, `sink.accept_fused(sr)` for the fused slot layout (W1 is None)."""

    @staticmethod
    def forward(ctx, W, W1, ids, dense, dense_w, dense_w1, padding_idx, sink, D):
        feat, y1, y2, S = raw_embed_fm_fwd(W, W1, ids, dense, dense_w.reshape(-1, D),
                                           dense_w1.reshape(-1), padding_idx, D=D)
        ctx.save_for_backward(ids, dense, feat, S)
        ctx.padding_idx = padding_idx
        ctx.sink = sink
        ctx.V = W.shape[0]
        ctx.ahead = (group_ids_ahead(ids, ctx.V, padding_idx)
                     if GROUP_AHEAD and any(ctx.needs_input_grad) else None)
        ctx.fused = W1 is None
        ctx.dense_w_shape = dense_w.shape
        ctx.mark_non_differentiable(S)
        return feat, y1.unsqueeze(1), y2.unsqueeze(1), S

    @staticmethod
    def backward(ctx, dfeat, dy1, dy2, _dS):
        ids, dense, feat, S = ctx.saved_tensors
        B, F = ids.shape
        D = feat.shape[2]
        dev = feat.device
        gy1 = dy1.reshape(-1).contiguous() if dy1 is not None else torch.zeros(B, device=dev)
        gy2 = dy2.reshape(-1).contiguous() if dy2 is not None else torch.zeros(B, device=dev)
        if dfeat is not None:
            dfeat = dfeat.contiguous()
        groups = (groups_ready(ctx.ahead) if ctx.ahead is not None
                  else ctx.sink.groups_for(ids, ctx.V, ctx.padding_idx))
        G = fused_grad_cols(D) if ctx.fused else 0
        dW_rows, dW1_rows, ddense_w, ddense_w1 = raw_embed_fm_bwd(
            feat, S, dfeat, gy1, gy2, dense, groups.seg_offsets, groups.sorted_pos, groups.num, F,
            fused_cols=G)
        if ctx.fused:
            ctx.sink.accept_fused(SelectedRows(groups.unique_ids, dW_rows, groups.num, ctx.V))
        else:
            ctx.sink.accept(SelectedRows(groups.unique_ids, dW_rows, groups.num, ctx.V),
                            SelectedRows(groups.unique_ids, dW1_rows.unsqueeze(1), groups.num, ctx.V))
        return (None, None, None, None, ddense_w.reshape(ctx.dense_w_shape), ddense_w1, None, None,
                None)


def fused_grad_cols(D: int) -> int:
    """Columns of a fused gradient row [D | g1 | pad]: D+1 rounded up to a multiple of 4."""
    return (D + 1 + 3) // 4 * 4


def fused_slot(D: int) -> int:
    """Floats per table row in the fused layout: 128-byte slots (32 floats)."""
    return (D + 1 + 31) // 32 * 32


class _Gather(torch.autograd.Function):
    """paddle.nn.Embedding forward/backward (lookup_table_v2 / _grad, sparse=True)."""

    @staticmethod
    def forward(ctx, W, ids, padding_idx, sink, _hook):
        out = raw_gather(W, ids, padding_idx)
        ctx.save_for_backward(ids)
        ctx.padding_idx = padding_idx
        ctx.sink = sink
        ctx.V = W.shape[0]
        ctx.ahead = (group_ids_ahead(ids, ctx.V, padding_idx)
                     if GROUP_AHEAD and any(ctx.needs_input_grad) else None)
        return out

    @staticmethod
    def backward(ctx, dout):
        (ids,) = ctx.saved_tensors
        dout = dout.contiguous()
        groups = (groups_ready(ctx.ahead) if ctx.ahead is not None
                  else raw_group_ids(ids, ctx.V, ctx.padding_idx))
        rows = raw_segment_reduce(dout.reshape(-1, dout.shape[-1]), groups.seg_offsets,
                                  groups.sorted_pos, groups.num, groups.n)
        ctx.sink.accept(SelectedRows(groups.unique_ids, rows, groups.num, ctx.V))
        return None, None, None, None, None


class _GatherPool(torch.autograd.Function):
    """sparse_embedding + sequence_pool(sum) over LoD key lists (slot_dnn/net.py:63-75)."""

    @staticmethod
    def forward(ctx, W, keys, offsets, padding_idx, sink, _hook):
        out, bag_of_pos = raw_gather_pool_sum(W, keys, offsets, padding_idx)
        ctx.save_for_backward(keys, bag_of_pos)
        ctx.padding_idx, ctx.sink, ctx.V = padding_idx, sink, W.shape[0]
        ctx.ahead = (group_ids_ahead(keys, ctx.V, padding_idx)
                     if GROUP_AHEAD and any(ctx.needs_input_grad) else None)
        return out

    @staticmethod
    def backward(ctx, dout):
        keys, bag_of_pos = ctx.saved_tensors
        groups = (groups_ready(ctx.ahead) if ctx.ahead is not None
                  else raw_group_ids(keys, ctx.V, ctx.padding_idx))
        rows = raw_segment_reduce(dout.contiguous(), groups.seg_offsets, groups.sorted_pos,
                                  groups.num, groups.n, row_of_pos=bag_of_pos)
        ctx.sink.accept(SelectedRows(groups.unique_ids, rows, groups.num, ctx.V))
        return None, None, None, None, None, None


def gather_pool_sum(W, keys, offsets, padding_idx, sink, hook):
    return _GatherPool.apply(W, keys, offsets, padding_idx, sink, hook)


def tc_backend() -> bool:
    """True when the hand-written tcgen05 GEMMs serve the 'bf16x3' matmuls (tower.BACKEND)."""
    from . import tower
    return tower.BACKEND == "tcgen05"


class _TcLinear(torch.autograd.Function):
    """y = x @ W (+ b) as ONE tcgen05 GEMM per direction (split precision): forward with the bias in
    the epilogue, dW as the batch-split MN-major GEMM (the bias gradient rides along as an extra
    output row when the input width is not a multiple of 128), dx as the K-major GEMM.  Used by
    every nn.Linear / split_mm of the package in 'bf16x3' precision."""

    @staticmethod
    def forward(ctx, x, W, b):
        K, N = W.shape
        ones = b is not None and K % 128 != 0
        xs = raw_tc_split(x, ones_col=ones)
        Wp, WTp = raw_tc_prep_weight(W, want_w=ctx.needs_input_grad[0])
        y, _ = raw_tc_linear_fwd(xs, K, WTp, N, b, False, True, False)
        ctx.xs, ctx.Wp, ctx.shape, ctx.ones, ctx.has_b = xs, Wp, (K, N), ones, b is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        K, N = ctx.shape
        gs, db = raw_tc_split_bwd(dy.contiguous(), None)
        if ctx.ones:
            dW, db = raw_tc_linear_bwd_dw(ctx.xs, K, gs, N, bias_row=True)
        else:
            dW = raw_tc_linear_bwd_dw(ctx.xs, K, gs, N)
        dx = None
        if ctx.needs_input_grad[0]:
            dx, _, _ = raw_tc_linear_bwd_dx(gs, N, ctx.Wp, K, None, True, False, False)
        ctx.xs = ctx.Wp = None
        return dx, dW, (db if ctx.has_b else None)


def tc_linear(x, W, b=None):
    lead = x.shape[:-1]
    y = _TcLinear.apply(x.reshape(-1, x.shape[-1]).contiguous(), W, b)
    return y.reshape(*lead, y.shape[-1])


class _CrossV2Tc(torch.autograd.Function):
    """One CrossNetV2 layer X_{i+1} = X_i + X_0 * (X_i W + b) (dcn_v2/net.py:222-226) on the tcgen05
    kernels: ONE GEMM whose epilogue applies bias, Hadamard and residual, saves u = X_i W + b for
    the backward and emits the next layer's hi/lo operand; backward = K3 (dxw, dx0) + the split +
    the dW GEMM + the dX GEMM with the residual gradient added in its epilogue."""

    @staticmethod
    def forward(ctx, x0, xl, W, bias, xl_planes):
        C = W.shape[0]
        ones = bias is not None and C % 128 != 0
        xs = xl_planes if xl_planes is not None else raw_tc_split(xl, ones_col=ones)
        Wp, WTp = raw_tc_prep_weight(W)
        out, outp, u = raw_tc_cross_fwd(xs, WTp, bias, x0, xl, True, want_u=True, ones_col=ones)
        ctx.save_for_backward(x0, u)
        ctx.xs, ctx.Wp, ctx.C, ctx.ones, ctx.has_b = xs, Wp, C, ones, bias is not None
        ctx.mark_non_differentiable(outp)   # handed to the next cross layer (no re-split)
        return out, outp

    @staticmethod
    def backward(ctx, dout, _dplanes):
        x0, u = ctx.saved_tensors
        C = ctx.C
        dout = dout.contiguous()
        zero_b = torch.zeros(C, dtype=torch.float32, device=dout.device)
        dxw, dx0, dbias = raw_cross_v2_bwd(dout, x0, u, zero_b)        # u already holds the bias
        gs, _ = raw_tc_split_bwd(dxw, None)
        if ctx.ones:
            dW, dbias = raw_tc_linear_bwd_dw(ctx.xs, C, gs, C, bias_row=True)
        else:
            dW = raw_tc_linear_bwd_dw(ctx.xs, C, gs, C)
        dxl, _, _ = raw_tc_linear_bwd_dx(gs, C, ctx.Wp, C, None, True, False, False, addend=dout)
        ctx.xs = ctx.Wp = None
        return dx0, dxl, dW, (dbias if ctx.has_b else None), None


class _CrossV2(torch.autograd.Function):
    """One CrossNetV2 layer: X_{i+1} = X_i + X_0 * (X_i W + b)   (dcn_v2/net.py:222-226).
    The contraction is a tensor-core library GEMM; in 'bf16x3' precision its operands go through the
    fused hi/lo split kernels of the tower (one pass per operand) and the backward dW uses the same
    [a_hi|a_lo]^T [g_hi|g_lo] fold; bias + Hadamard + residual (and their backward) are K3."""

    @staticmethod
    def forward(ctx, x0, xl, W, bias, mm, precision):
        ctx.split = precision == "bf16x3"
        if ctx.split:
            K, N = W.shape
            xs = raw_tower_split(xl, None, False)                    # [B, 2K] bf16
            W2r, W2c, Wlo = raw_tower_prep_weight(W)
            xw = torch.mm(xs, W2r, out_dtype=torch.float32)
            torch.addmm(xw, xs[:, :K], Wlo, out_dtype=torch.float32, out=xw)
            ctx.xs, ctx.wprep = xs, (W2c, Wlo)
        else:
            xw = mm(xl, W)
        out = raw_cross_v2_fwd(x0, xl, xw, bias)
        ctx.save_for_backward(x0, xl, xw, W, bias)
        ctx.mm = mm
        return out

    @staticmethod
    def backward(ctx, dout):
        x0, xl, xw, W, bias = ctx.saved_tensors
        dout = dout.contiguous()
        dxw, dx0, dbias = raw_cross_v2_bwd(dout, x0, xw, bias)
        if ctx.split:
            K, N = W.shape
            W2c, Wlo = ctx.wprep
            gs, _ = raw_tower_relu_bwd_split(dxw, None)               # [B, 2N] bf16 (no mask)
            dW = raw_tower_fold_dw(torch.mm(ctx.xs.t(), gs, out_dtype=torch.float32), K, N)
            dxl = torch.mm(gs, W2c.t(), out_dtype=torch.float32)
            torch.addmm(dxl, gs[:, :N], Wlo.t(), out_dtype=torch.float32, out=dxl)
            dxl += dout
            ctx.xs = ctx.wprep = None
        else:
            dxl = dout + ctx.mm(dxw, W.t())
            dW = ctx.mm(xl.t(), dxw)
        return dx0, dxl, dW, dbias, None, None


# ---- K6: DLRM dot interaction --------------------------------------------------------------------
def dot_interact_width(N: int, d: int, self_interaction: bool = False) -> int:
    return d + (N * (N + 1) // 2 if self_interaction else N * (N - 1) // 2)


def raw_dot_interact_fwd(T: torch.Tensor, self_interaction: bool = False) -> torch.Tensor:
    """T [B, N, d] (x is the last row) -> R [B, d + P] = [x | upper-triangle dots]."""
    lib = _lib.load()
    T = _req(T, torch.float32, "T")
    B, N, d = T.shape
    R = torch.empty(B, dot_interact_width(N, d, self_interaction), dtype=torch.float32,
                    device=T.device)
    check(lib.b200rec_dot_interact_fwd(ptr(T), ptr(R), B, N, d, int(bool(self_interaction)),
                                       _stream()), "dot_interact_fwd")
    _count("dot_interact_fwd")
    return R


def raw_dot_interact_bwd(T: torch.Tensor, dR: torch.Tensor, self_interaction: bool = False) -> torch.Tensor:
    lib = _lib.load()
    T = _req(T, torch.float32, "T")
    dR = _req(dR, torch.float32, "dR")
    B, N, d = T.shape
    if dR.shape != (B, dot_interact_width(N, d, self_interaction)):
        raise ValueError("dot_interact_bwd: dR has shape %s" % (tuple(dR.shape),))
    dT = torch.empty_like(T)
    check(lib.b200rec_dot_interact_bwd(ptr(T), ptr(dR), ptr(dT), B, N, d,
                                       int(bool(self_interaction)), _stream()), "dot_interact_bwd")
    _count("dot_interact_bwd")
    return dT


class _DotInteract(torch.autograd.Function):
    @staticmethod
    def forward(ctx, T, self_interaction):
        T = T.contiguous()
        ctx.save_for_backward(T)
        ctx.self_interaction = self_interaction
        return raw_dot_interact_fwd(T, self_interaction)

    @staticmethod
    def backward(ctx, dR):
        (T,) = ctx.saved_tensors
        return raw_dot_interact_bwd(T, dR.contiguous(), ctx.self_interaction), None


def dot_interact(T: torch.Tensor, self_interaction: bool = False) -> torch.Tensor:
    """DLRM's pairwise-dot feature interaction with the `concat([x, Zflat])` fused in
    (models/rank/dlrm/net.py:97-115); T = [26 embedding rows ..., x]."""
    return _DotInteract.apply(T, self_interaction)


# ---- uint64 feasigns -> rows ---------------------------------------------------------------------
def raw_hash_keys(keys: torch.Tensor, V: int, slot_of_key: Optional[torch.Tensor] = None,
                  reserve_zero: bool = True) -> torch.Tensor:
    """keys: uint64 (or int64 holding the same bits) feasigns, any shape -> int64 rows in [0, V) of
    the same shape; slot_of_key: int32 per key (salts the hash per slot) or None."""
    lib = _lib.load()
    if keys.dtype not in (torch.uint64, torch.int64):
        raise TypeError("hash_keys: keys must be uint64 or int64, got %s" % keys.dtype)
    if not keys.is_cuda:
        raise _lib.B200RecError("hash_keys: keys must be a CUDA tensor (no CPU fallback)")
    keys = keys.contiguous()
    if slot_of_key is not None:
        slot_of_key = _req(slot_of_key, torch.int32, "slot_of_key")
        if slot_of_key.numel() != keys.numel():
            raise ValueError("hash_keys: slot_of_key must have one entry per key")
    rows = torch.empty(keys.shape, dtype=torch.int64, device=keys.device)
    check(lib.b200rec_hash_keys(ptr(keys), ptr(slot_of_key), keys.numel(), int(V),
                                int(bool(reserve_zero)), ptr(rows), _stream()), "hash_keys")
    _count("hash_keys")
    return rows


hash_keys = raw_hash_keys


# ---- continuous_value_model ---------------------------------------------------------------------
def raw_cvm_fwd(x: torch.Tensor, use_cvm: bool) -> torch.Tensor:
    lib = _lib.load()
    x = _req(x, torch.float32, "x")
    N, W = x.shape
    D = W - 2
    y = torch.empty(N, W if use_cvm else D, dtype=torch.float32, device=x.device)
    check(lib.b200rec_cvm_fwd(ptr(x), ptr(y), N, D, int(use_cvm), _stream()), "cvm_fwd")
    _count("cvm_fwd")
    return y


def raw_cvm_bwd(dy: torch.Tensor, show_click: torch.Tensor, D: int, use_cvm: bool) -> torch.Tensor:
    lib = _lib.load()
    dy = _req(dy, torch.float32, "dy")
    show_click = _req(show_click, torch.float32, "show_click")
    N = dy.shape[0]
    dx = torch.empty(N, D + 2, dtype=torch.float32, device=dy.device)
    check(lib.b200rec_cvm_bwd(ptr(dy), ptr(show_click), ptr(dx), N, D, int(use_cvm), _stream()),
          "cvm_bwd")
    _count("cvm_bwd")
    return dx


class _CVM(torch.autograd.Function):
    """paddle.static.nn.continuous_value_model(input, cvm, use_cvm) — wide_deep/net.py:87-88."""

    @staticmethod
    def forward(ctx, x, show_click, use_cvm):
        ctx.save_for_backward(show_click)
        ctx.use_cvm, ctx.D = use_cvm, x.shape[1] - 2
        return raw_cvm_fwd(x, use_cvm)

    @staticmethod
    def backward(ctx, dy):
        (show_click,) = ctx.saved_tensors
        return raw_cvm_bwd(dy.contiguous(), show_click, ctx.D, ctx.use_cvm), None, None


def continuous_value_model(x, show_click, use_cvm):
    return _CVM.apply(x, show_click, use_cvm)


def fused_seqpool_cvm(W, keys, offsets, n_slots: int, show_click, use_cvm: bool, padding_idx, sink,
                      hook):
    """`fused_seqpool_cvm(embs, "sum", show_clk, use_cvm)` of the PS/GPUBox models
    (tools/utils/static_ps/model_util.py:411-415; slot_dnn/net.py:63-75 spells it as
    sequence_pool(sum) + continuous_value_model): for every (sample, slot) bag the rows of its
    variable-length key list are summed, then the two leading show/click columns are transformed
    (use_cvm) or dropped; backward writes `show_click` into those two gradient columns so the table
    accumulates the statistics.

    ALL slots go through ONE pooled gather and ONE CVM launch: `keys`/`offsets` hold the bags in
    sample-major order, bag b = n*n_slots + f — the layout dataio.parse_slot_text_lod emits.
    W: [V, D+2]; show_click: [B, 2].  Returns [B, n_slots, D+2 if use_cvm else D]."""
    n_bags = offsets.numel() - 1
    if n_bags % n_slots:
        raise ValueError("fused_seqpool_cvm: %d bags is not a multiple of n_slots=%d" % (n_bags, n_slots))
    B = n_bags // n_slots
    if show_click.shape != (B, 2):
        raise ValueError("fused_seqpool_cvm: show_click must be [%d, 2], got %s" % (B, tuple(show_click.shape)))
    pooled = gather_pool_sum(W, keys, offsets, padding_idx, sink, hook)            # [B*F, D+2]
    per_bag = show_click.to(torch.float32).repeat_interleave(n_slots, dim=0)         # [B*F, 2]
    out = continuous_value_model(pooled, per_bag, use_cvm)
    return out.reshape(B, n_slots, out.shape[1])


# ---- K4: DIN attention pooling ------------------------------------------------------------------
HAVE_DIN_ATTN = True


def raw_din_attn_fwd(hist, tseq, mask, W1, b1, W2, b2, W3, b3):
    """hist [B,L,E], tseq [B,E] (tiled target), mask int64 [B,L(,1)] or None.
    Returns (out [B,E], weights [B,L])."""
    lib = _lib.load()
    hist = _req(hist, torch.float32, "hist")
    tseq = _req(tseq, torch.float32, "tseq")
    B, L, E = hist.shape
    W1 = W1.detach()
    Wa, Wb, Wc, Wd = W1[0:E], W1[E:2 * E], W1[2 * E:3 * E], W1[3 * E:4 * E]
    Wac = (Wa + Wc).contiguous()
    Wd = Wd.contiguous()
    tb = torch.addmm(b1.detach(), tseq, Wb - Wc)            # [B,80]: the per-sample t-term
    if mask is not None:
        mask = _req(mask.reshape(B, L), torch.int64, "mask")
    dev = hist.device
    scores = torch.empty(B, L, dtype=torch.float32, device=dev)
    weights = torch.empty(B, L, dtype=torch.float32, device=dev)
    out = torch.empty(B, E, dtype=torch.float32, device=dev)
    check(lib.b200rec_din_attn_fwd(ptr(hist), ptr(tseq), ptr(tb), ptr(Wac), ptr(Wd),
                                   ptr(_req(W2.detach(), torch.float32, "W2")), ptr(b2.detach()),
                                   ptr(_req(W3.detach().reshape(-1), torch.float32, "W3")),
                                   ptr(b3.detach()), ptr(mask), ptr(scores), ptr(weights), ptr(out),
                                   B, L, E, float(E) ** -0.5, _stream()), "din_attn_fwd")
    _count("din_attn_fwd")
    return out, weights


def raw_din_attn_bwd(hist, tseq, W1, b1, W2, b2, W3, weights, dout):
    """Fused backward of the DIN attention pooling.  Returns
    (dhist, dtseq, dW1, db1, dW2, db2, dW3 [40,1], db3 [1])."""
    lib = _lib.load()
    hist = _req(hist, torch.float32, "hist")
    tseq = _req(tseq, torch.float32, "tseq")
    dout = _req(dout, torch.float32, "dout")
    weights = _req(weights, torch.float32, "weights")
    B, L, E = hist.shape
    W1 = W1.detach()
    Wa, Wb, Wc, Wd = W1[0:E], W1[E:2 * E], W1[2 * E:3 * E], W1[3 * E:4 * E]
    Wac, Wbc, Wd = (Wa + Wc).contiguous(), (Wb - Wc), Wd.contiguous()
    tb = torch.addmm(b1.detach(), tseq, Wbc)
    dev = hist.device
    f32 = dict(dtype=torch.float32, device=dev)
    da = torch.empty(B, L, **f32)
    dhist = torch.empty_like(hist)
    dtseq = torch.empty(B, E, **f32)
    dtb = torch.empty(B, 80, **f32)
    dWac, dWd = torch.empty(E, 80, **f32), torch.empty(E, 80, **f32)
    dW2, db2, dW3 = torch.empty(80, 40, **f32), torch.empty(40, **f32), torch.empty(40, **f32)
    nbytes = ctypes.c_size_t(0)
    check(lib.b200rec_din_attn_bwd_workspace_bytes(B, L, E, ctypes.byref(nbytes)), "din_bwd_ws")
    ws = workspace(nbytes.value, dev, "din_bwd")
    check(lib.b200rec_din_attn_bwd(ptr(hist), ptr(tseq), ptr(tb), ptr(Wac), ptr(Wd),
                                   ptr(_req(W2.detach(), torch.float32, "W2")), ptr(b2.detach()),
                                   ptr(_req(W3.detach().reshape(-1), torch.float32, "W3")),
                                   ptr(weights), ptr(dout), ptr(da), ptr(dhist), ptr(dtseq),
                                   ptr(dtb), ptr(dWac), ptr(dWd), ptr(dW2), ptr(db2), ptr(dW3), B, L,
                                   E, float(E) ** -0.5, ptr(ws), ws.numel(), _stream()),
          "din_attn_bwd")
    _count("din_attn_bwd")
    # the t-path: tb = t (Wb - Wc) + b1
    dtseq = torch.addmm(dtseq, dtb, Wbc.t())
    Gt = tseq.t() @ dtb
    dW1 = torch.cat([dWac, Gt, dWac - Gt, dWd], dim=0)
    return dhist, dtseq, dW1, dtb.sum(0), dW2, db2, dW3.reshape(-1, 1), da.sum().reshape(1)


def _din_attention_composite(hist, tseq, mask, W1, b1, W2, b2, W3, b3):
    """The reference's op sequence (din/net.py:155-173) in torch — used to differentiate."""
    E = hist.shape[2]
    t = tseq.unsqueeze(1).expand_as(hist)
    c = torch.cat([hist, t, hist - t, hist * t], dim=2)
    a = torch.sigmoid(c @ W1 + b1)
    a = torch.sigmoid(a @ W2 + b2)
    a = a @ W3 + b3
    if mask is not None:
        a = a + mask.reshape(a.shape).to(a.dtype)
    w = torch.softmax(a.transpose(1, 2) * (E ** -0.5), dim=-1)
    return torch.matmul(w, hist).reshape(-1, E)


FUSED_DIN_BACKWARD = True


class _DinAttn(torch.autograd.Function):
    """Forward and backward are the fused K4 kernels (only the softmax weights are saved; z1/z2
    are recomputed in backward).  With FUSED_DIN_BACKWARD = False the backward re-runs the
    reference's op sequence under autograd on chunks of samples (kept as a cross-check)."""

    CHUNK_BYTES = 256 << 20

    @staticmethod
    def forward(ctx, hist, tseq, mask, W1, b1, W2, b2, W3, b3):
        out, w = raw_din_attn_fwd(hist, tseq, mask, W1, b1, W2, b2, W3, b3)
        ctx.save_for_backward(hist, tseq, W1, b1, W2, b2, W3, b3, w)
        ctx.mask = mask
        return out

    @staticmethod
    def backward(ctx, dout):
        hist, tseq, W1, b1, W2, b2, W3, b3, w = ctx.saved_tensors
        if FUSED_DIN_BACKWARD:
            dhist, dtseq, dW1, db1, dW2, db2, dW3, db3 = raw_din_attn_bwd(
                hist, tseq, W1, b1, W2, b2, W3, w, dout.contiguous())
            return dhist, dtseq, None, dW1, db1, dW2, db2, dW3.reshape(W3.shape), db3
        B, L, E = hist.shape
        per_sample = L * 4 * E * 4 * 3
        chunk = max(1, min(B, _DinAttn.CHUNK_BYTES // max(per_sample, 1)))
        params = [p.detach().requires_grad_(True) for p in (W1, b1, W2, b2, W3, b3)]
        dhist = torch.empty_like(hist)
        dtseq = torch.empty_like(tseq)
        pgrads = [torch.zeros_like(p) for p in params]
        for s in range(0, B, chunk):
            e = min(B, s + chunk)
            h = hist[s:e].detach().requires_grad_(True)
            t = tseq[s:e].detach().requires_grad_(True)
            m = ctx.mask[s:e] if ctx.mask is not None else None
            with torch.enable_grad():
                o = _din_attention_composite(h, t, m, *params)
            gs = torch.autograd.grad(o, [h, t] + params, dout[s:e])
            dhist[s:e] = gs[0]
            dtseq[s:e] = gs[1]
            for acc, g in zip(pgrads, gs[2:]):
                acc += g
        return (dhist, dtseq, None, *pgrads)


def din_attention(hist, tseq, mask, W1, b1, W2, b2, W3, b3):
    return _DinAttn.apply(hist, tseq, mask, W1, b1, W2, b2, W3, b3)


class _SplitMM(torch.autograd.Function):
    """a @ W for fp32 operands on the bf16 tensor cores (hi/lo split, three products, fp32
    accumulate) with the fused split kernels — the GEMM building block of tower.py as a
    stand-alone autograd node (used by CrossNetMix's two large projections)."""

    @staticmethod
    def forward(ctx, a, W):
        K, N = W.shape
        a_s = raw_tower_split(a.contiguous(), None, False)
        W2r, W2c, Wlo = raw_tower_prep_weight(W)
        out = torch.mm(a_s, W2r, out_dtype=torch.float32)
        torch.addmm(out, a_s[:, :K], Wlo, out_dtype=torch.float32, out=out)
        ctx.a_s, ctx.wprep, ctx.shape = a_s, (W2c, Wlo), (K, N)
        return out

    @staticmethod
    def backward(ctx, dout):
        K, N = ctx.shape
        W2c, Wlo = ctx.wprep
        gs, _ = raw_tower_relu_bwd_split(dout.contiguous(), None)
        dW = raw_tower_fold_dw(torch.mm(ctx.a_s.t(), gs, out_dtype=torch.float32), K, N)
        da = torch.mm(gs, W2c.t(), out_dtype=torch.float32)
        torch.addmm(da, gs[:, :N], Wlo.t(), out_dtype=torch.float32, out=da)
        ctx.a_s = ctx.wprep = None
        return da, dW


class _CrossCombine(torch.autograd.Function):
    """out = xl + x0 * (xw + bias) with xw given (K3 epilogue as its own node)."""

    @staticmethod
    def forward(ctx, x0, xl, xw, bias):
        ctx.save_for_backward(x0, xw, bias)
        return raw_cross_v2_fwd(x0, xl, xw, bias)

    @staticmethod
    def backward(ctx, dout):
        x0, xw, bias = ctx.saved_tensors
        dout = dout.contiguous()
        dxw, dx0, dbias = raw_cross_v2_bwd(dout, x0, xw, bias)
        return dx0, dout, dxw, dbias


def split_mm(a, W):
    if tc_backend() and a.is_cuda:
        return tc_linear(a, W, None)
    return _SplitMM.apply(a, W)


def cross_combine(x0, xl, xw, bias):
    return _CrossCombine.apply(x0, xl, xw, bias)


def embed_fm(W, W1, ids, dense, dense_w, dense_w1, padding_idx, sink, D=None):
    D = W.shape[1] if D is None else D
    return _EmbedFM.apply(W, W1, ids, dense, dense_w, dense_w1, padding_idx, sink, D)


def gather(W, ids, padding_idx, sink, hook):
    return _Gather.apply(W, ids, padding_idx, sink, hook)


def cross_v2(x0, xl, W, bias, mm, precision="fp32", xl_planes=None):
    """-> (X_{i+1}, its hi/lo planes or None).  Pass the planes back as `xl_planes` of the next
    layer: on the tcgen05 back end the GEMM epilogue has already produced that operand."""
    if precision == "bf16x3" and x0.is_cuda and tc_backend():
        return _CrossV2Tc.apply(x0, xl, W, bias, xl_planes)
    return _CrossV2.apply(x0, xl, W, bias, mm, precision), None


# ---- per-kernel CUDA-event timing of every entry point (bench.py roofline_step) -----------------
def _wrap_timed(fn, name):
    import functools

    @functools.wraps(fn)
    def timed(*a, **k):
        if EVENTS is None:
            return fn(*a, **k)
        with _Timed(name):
            return fn(*a, **k)
    return timed


for _n in ("group_ids", "embed_fm_bwd", "gather", "gather_pool_sum", "segment_reduce", "sparse_sgd",
           "sparse_adam", "sparse_adagrad", "cross_v2_fwd", "cross_v2_bwd", "shard_bucketize",
           "shard_gather_push", "shard_push_rows", "shard_fm_grads_push",
           "tc_split", "tc_split_bwd", "tc_prep_weight", "tc_linear_fwd", "tc_cross_fwd",
           "tc_linear_bwd_dx", "tc_linear_bwd_dw", "tc_head_fwd", "tc_head_bwd", "din_attn_fwd", "din_attn_bwd", "tower_split",
           "tower_relu_bwd_split", "tower_prep_weight", "tower_fold_dw"):
    globals()["raw_" + _n] = _wrap_timed(globals()["raw_" + _n], _n)
del _n
