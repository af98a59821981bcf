#!/usr/bin/env python
"""bench.py — CTR training samples/s of DeepFM on a synthetic Criteo-shaped batch (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch: clear_grad -> DeepFMLayer.forward (fused
gather+FM kernel, MLP tower) -> log_loss -> backward (sort/segment-reduce scatter-add, fused FM
grad) -> optimizer step (lazy Adam on the touched rows, Adam on the dense parameters).

Workload (config.workload): DeepFM, 26 sparse + 13 dense slots, hashed vocab V=1e8, D=16,
B=65536 per GPU, fc [400,400,400], uniform hashed ids with 2 % padding, 8 rotating batches
(per-step working set: 164 MB feat + 6.4 GB table >> 126 MB L2, so no L2 flush is needed).
N>1: tables row-sharded (owner = id mod N), NCCL all-to-all of ids/rows/grads, dense grads
all-reduced; weak scaling (B per GPU fixed).

Printed JSON (one line, rank 0): see the contract in the task statement; extra keys `roofline`
(fused gather+FM forward kernel, algorithmic bytes / CUDA-event time inside the timed region
against MEASURED_PEAKS.json), `cpu_baseline` (oracle port timed on the host cores, N=1 only),
`e2e` (same metric through the public API — runner.DevicePrefetcher over pinned HOST batches +
DygraphModel.train_forward incl. its AUC update: H2D of every batch and D2H of the loss inside the
timed region), `roofline_step` (CUDA-event time of every kernel family of the step + the
composite bound of the whole step), `clocks`, `gpu_launches`; at N>1 also `parity` (step-0 loss
of the sharded model == the fp64 oracle on a slice of the global batch).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

F_SPARSE, N_DENSE = 26, 13


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=30)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--batch", type=int, default=65536, help="samples per GPU per step")
    p.add_argument("--vocab", type=int, default=100_000_000)
    p.add_argument("--dim", type=int, default=16)
    p.add_argument("--fc", type=str, default="400,400,400")
    p.add_argument("--precision", default="bf16x3", choices=["fp32", "tf32", "bf16x3"])
    p.add_argument("--dist", default="uniform", choices=["uniform", "zipf"])
    p.add_argument("--nbatches", type=int, default=8)
    p.add_argument("--cpu-batch", type=int, default=65536)
    p.add_argument("--cpu-steps", type=int, default=4)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--timeline", default="", help="write a CUPTI timeline of 3 steps (rank 0) "
                   "as <path>.json (chrome trace) and <path>.txt (per-stream summary) and exit")
    p.add_argument("--dump-outputs", default="", metavar="DIR",
                   help="after the timed steps write what the last one computed (rank 0) as "
                        "DIR/<name>.npy, so that two builds can be compared output for output")
    args = p.parse_args()
    if args.dump_outputs and args.impl != "b200":
        p.error("--dump-outputs applies to --impl b200")
    return args


def algorithmic_bytes_fwd(D, F=F_SPARSE, Dn=N_DENSE):
    """SURVEY.md §8(d): ids + dense + rows + first-order scalars + feat write + (y1,y2)."""
    return F * 8 + Dn * 4 + F * 4 * D + F * 4 + (F + Dn) * 4 * D + 8


def make_batches(n, B, V, dist, seed, pin):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        if dist == "zipf":
            r = torch.rand(B, F_SPARSE, generator=g, dtype=torch.float64)
            ids = (float(V) ** r).to(torch.int64).clamp_(1, V - 1)
        else:
            ids = torch.randint(1, V, (B, F_SPARSE), generator=g)
        ids[torch.rand(B, F_SPARSE, generator=g) < 0.02] = 0
        dense = torch.rand(B, N_DENSE, generator=g)
        dense[torch.rand(B, N_DENSE, generator=g) < 0.3] = 0.0
        label = (torch.rand(B, 1, generator=g) < 0.29).to(torch.int64)
        if pin:
            ids, dense, label = ids.pin_memory(), dense.pin_memory(), label.pin_memory()
        out.append((label, ids, dense))
    return out


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4)
                          if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# -------------------------------------------------------------------------------- reference arm
def run_reference(args, rank):
    """The reference's own CPU implementation of the path = the oracle port (Paddle is not
    installable here, see DESIGN.md), on all host threads, on a bounded sample of the workload."""
    if rank != 0:
        return
    V = args.vocab
    try:
        import psutil
        need = V * (args.dim + 1) * 4 * 3.2
        if psutil.virtual_memory().available < need * 1.3:
            V = max(1_000_001, int(psutil.virtual_memory().available / 1.3 / ((args.dim + 1) * 4 * 3.2)))
    except ImportError:
        pass
    K = max(1, min(args.steps, args.cpu_steps))
    W = 1
    value, cores, sec_per_step, loss = time_cpu_port(args, V, K)
    secs = sec_per_step * K
    sample = ("%d steps of B=%d (after warm-up + thread-count calibration: %d of %d host threads) of "
              "the same DeepFM step, V=%d, fp32, lazy Adam" % (K, args.cpu_batch, cores,
                                                            os.cpu_count() or 1, V))
    line = {
        "impl": "reference", "metric": "DeepFM Criteo-shape CTR training samples/sec",
        "value": value, "unit": "samples/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": secs / K * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "loss": loss,
    }
    print(json.dumps(line), flush=True)


def time_cpu_port(args, V, steps):
    """Times the CPU port with the thread count that serves it best: one calibration step at each
    of {all, 1/2, 1/4, 1/8 of the host threads}; torch's intra-op pool is not always fastest at 128
    threads on these op sizes.  Returns (samples/s, threads used, steps timed, last loss)."""
    from oracle.cpu_train import CpuDeepFM, time_steps

    total = os.cpu_count() or 1
    model = CpuDeepFM(V, args.dim, fc=[int(x) for x in args.fc.split(",")])
    B = args.cpu_batch
    batches = [(i, d, l.float()) for (l, i, d) in make_batches(2, B, V, args.dist, 12345, False)]
    torch.set_num_threads(total)
    time_steps(model, batches, 1, 0)                       # warm-up (page faults, allocator)
    best_t, best_s = total, None
    for t in sorted({total, max(1, total // 2), max(1, total // 4), max(1, total // 8)}, reverse=True):
        torch.set_num_threads(t)
        secs, _ = time_steps(model, batches, 1, 0)
        if best_s is None or secs < best_s:
            best_t, best_s = t, secs
    torch.set_num_threads(best_t)
    secs, loss = time_steps(model, batches, steps, 0)
    return B * steps / secs, best_t, secs / steps, loss


def exchange_name(world):
    """How table rows / gradients move at N>1 (mirrors paddlerec_b200.sharded.p2p_enabled)."""
    env = os.environ.get("B200REC_P2P", "auto")
    p2p = env == "1" or (env != "0" and world <= 4)
    return ("row / gradient exchange by our kernels storing into peer memory over NVLink, ids by "
            "NCCL all-to-all" if p2p else "NCCL all-to-all")


def workload_config(args, world):
    return {"workload": "DeepFM Criteo-shape: 26 sparse + 13 dense slots, hashed vocab %d, D=%d, "
                        "B=%d per GPU, fc [%s], %s ids (2%% padding)" %
                        (args.vocab, args.dim, args.batch, args.fc, args.dist),
            "global_batch": args.batch * world, "tower_matmul": args.precision,
            "optimizer": "Adam (lazy rows on the tables)",
            "parallelism": "single GPU" if world == 1 else
            "tables row-sharded (id mod %d) + %s; dense params data-parallel (NCCL all-reduce)" %
            (world, exchange_name(world)),
            "l2": "inputs larger than L2 (8 rotating batches; 164 MB feat + 6.4 GB table per step)"}


# ------------------------------------------------------------------------------------- our arm
def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist

    from paddlerec_b200 import nn as bnn
    from paddlerec_b200 import ops
    from paddlerec_b200.rank.deepfm.dygraph_model import DygraphModel

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bnn.set_matmul_precision(args.precision)
    from paddlerec_b200 import tower
    tower.set_overlap_dw(True)      # dW GEMMs on a side stream; the optimizers wait for them
    fc = [int(x) for x in args.fc.split(",")]
    config = {
        "hyper_parameters.sparse_feature_number": args.vocab,
        "hyper_parameters.sparse_feature_dim": args.dim,
        "hyper_parameters.fc_sizes": fc,
        "hyper_parameters.dense_input_dim": N_DENSE,
        "hyper_parameters.sparse_inputs_slots": F_SPARSE + 1,
        "hyper_parameters.optimizer.learning_rate": 1e-3,
    }
    torch.manual_seed(12345)
    dm = DygraphModel()
    dm.device = dev
    if world > 1:
        from paddlerec_b200 import sharded
        model = sharded.create_sharded_deepfm(config, dev, rank, world)
        optimizer = sharded.create_optimizer(model, config)
    else:
        model = dm.create_model(config)
        optimizer = dm.create_optimizer(model, config)
    model.train()

    host = make_batches(args.nbatches, args.batch, args.vocab, args.dist, 12345 + rank, pin=True)
    resident = [tuple(t.to(dev) for t in b) for b in host]
    label_f = [b[0].to(torch.float32) for b in resident]

    scale = optimizer.scale_loss if hasattr(optimizer, "scale_loss") else (lambda x: x)

    prefetch = getattr(model, "prefetch", None)
    finish_prefetch = getattr(model, "finish_prefetch", None)
    # detached: a reference to pred or loss would keep the step's autograd graph, and with it the
    # tower's activation planes, alive into the next step
    last = {} if args.dump_outputs else None

    def step_resident(i):
        label, ids, dense = resident[i % len(resident)]
        optimizer.clear_grad()
        pred = model(ids, dense)
        if prefetch is not None:   # plan the NEXT batch's exchange while this step computes
            prefetch(resident[(i + 1) % len(resident)][1])
        loss = dm.create_loss(pred, label_f[i % len(resident)])
        scale(loss).backward()
        if finish_prefetch is not None:
            finish_prefetch()
        optimizer.step()
        if last is not None:
            last["pred"], last["loss"], last["ids"] = pred.detach(), loss.detach(), ids
        return loss

    from paddlerec_b200 import runner
    metrics, _ = dm.create_metrics()
    state = {"pf": None}

    def host_stream():
        i = 0
        while True:
            yield host[i % len(host)]
            i += 1

    def step_e2e(i):
        """The public API with HOST batches: runner.DevicePrefetcher uploads batch i+1 from pinned
        memory on a copy stream while step i computes (one 17.6 MB H2D per step, inside the timed
        region); DygraphModel.train_forward = create_feeds + forward + loss + AUC update, as the
        reference's train_forward (deepfm/dygraph_model.py:75-87); the loss is read back every step."""
        if state["pf"] is None:
            state["pf"] = runner.DevicePrefetcher(host_stream(), dm, config)
        batch = next(state["pf"])
        optimizer.clear_grad()
        loss, _, _ = dm.train_forward(model, metrics, batch, config)
        if prefetch is not None:
            prefetch(state["pf"].peek()[1])
        scale(loss).backward()
        if finish_prefetch is not None:
            finish_prefetch()
        optimizer.step()
        return loss.item()  # D2H read of the step's result

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, collect_events=False, event_filter=None):
        for i in range(warmup):
            fn(i)
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        ops.EVENTS = [] if collect_events else None
        ops.EVENT_FILTER = event_filter
        n0 = ops.LAUNCHES
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = ops.LAUNCHES - n0
        events, ops.EVENTS = ops.EVENTS, None
        clocks = sampler.stop() if rank == 0 else None
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, events, clocks

    K, W = args.steps, max(args.warmup, 3)
    if args.timeline:
        timeline(args.timeline, step_resident, barrier, rank, W)
        return
    parity = parity_bit(args, model, dm, resident, label_f, rank, world, dev) if world > 1 else None
    ms, launches, events, clocks = timed(step_resident, K, W, collect_events=True,
                                         event_filter={"embed_fm_fwd"})
    if args.dump_outputs and rank == 0:   # before the passes below train the model further
        dump_outputs(args.dump_outputs, model, last, args, rank, world)
    value = args.batch * world * K / (ms / 1e3)
    k_ms = [s.elapsed_time(e) for (name, s, e) in events if name == "embed_fm_fwd"]
    kernel_ms = sum(k_ms) / max(len(k_ms), 1)
    ms_e2e, _, _, _ = timed(step_e2e, K, 3)
    e2e_value = args.batch * world * K / (ms_e2e / 1e3)
    # a third, short pass with an event pair around EVERY kernel family: the step's breakdown
    kb = min(K, 10)
    ms_b, _, ev_all, _ = timed(step_resident, kb, 2, collect_events=True)
    per = {}
    for name, s0, e0 in ev_all:
        per[name] = per.get(name, 0.0) + s0.elapsed_time(e0)
    per = {k: v / kb for k, v in per.items()}

    if rank != 0:
        return
    peak, peak_src = measured_peaks()
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(tpath) and args.dim == 16 and args.batch == 65536:
        with open(tpath) as fh:
            t = json.load(fh)
        traffic = t["dram_bytes_read_per_launch"] + t["dram_bytes_write_per_launch"]
    alg = algorithmic_bytes_fwd(args.dim) * args.batch
    achieved = alg / (kernel_ms / 1e3) / 1e9 if kernel_ms > 0 else 0.0
    line = {
        "metric": "DeepFM Criteo-shape CTR training samples/sec", "value": value,
        "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args, world),
        "roofline": {"kernel": "embed_fm_fwd_kernel (fused 26-slot gather + FM, forward)" +
                     ("" if world == 1 else
                      " over the RECEIVED rows (contiguous reads: the random gather is the owner-side "
                      "shard_gather_push / gather kernel, see roofline_step)"),
                     "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg, "kernel_ms": kernel_ms,
                     "kernel_share_of_step": kernel_ms / (ms / K), "traffic": traffic,
                     "traffic_source": "profiles/k1_traffic.json (ncu --set full, one launch)",
                     "frac_of_nominal_8TBs": achieved / 8000.0},
        "e2e": {"value": e2e_value, "unit": "samples/s", "ms_per_step": ms_e2e / K,
                "h2d_bytes_per_step": args.batch * (F_SPARSE * 8 + N_DENSE * 4 + 8),
                "d2h_bytes_per_step": 4},
        "gpu_launches": launches, "clocks": clocks,
        "roofline_step": roofline_step(args, per, ms / K, ms_b / kb, world),
    }
    if parity is not None:
        line["parity"] = parity
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline(args)
        except Exception as exc:  # the GPU numbers stand on their own
            line["cpu_baseline"] = {"error": repr(exc)}
    print(json.dumps(line), flush=True)


def timeline(path, step, barrier, rank, warmup):
    """CUPTI (torch.profiler) timeline of 3 resident steps: where the GPU idles and what runs on
    which stream.  nsys is not installed; this is the same data (kernel start/end per stream)."""
    from torch.profiler import ProfilerActivity, profile
    for i in range(warmup):
        step(i)
    barrier()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for i in range(3):
            step(warmup + i)
        barrier()
    if rank != 0:
        return
    prof.export_chrome_trace(path + ".json")
    ev = [e for e in json.load(open(path + ".json"))["traceEvents"]
          if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")]
    ev.sort(key=lambda e: e["ts"])
    t0, t1 = ev[0]["ts"], max(e["ts"] + e["dur"] for e in ev)
    streams = {}
    for e in ev:
        streams.setdefault(e["args"].get("stream", e.get("tid")), []).append(e)
    lines = ["3 steps: %.1f us wall on the GPU (%.1f us / step)" % (t1 - t0, (t1 - t0) / 3)]
    main = max(streams, key=lambda k: sum(x["dur"] for x in streams[k]))
    for k, v in sorted(streams.items(), key=lambda kv: -sum(x["dur"] for x in kv[1])):
        lines.append("stream %s: %d launches, busy %.1f us%s" % (
            k, len(v), sum(x["dur"] for x in v), "  <- main" if k == main else ""))
    # union of busy intervals over all streams -> idle time
    busy, cur_s, cur_e = 0.0, None, None
    for e in ev:
        s0, e0 = e["ts"], e["ts"] + e["dur"]
        if cur_e is None or s0 > cur_e:
            if cur_e is not None:
                busy += cur_e - cur_s
            cur_s, cur_e = s0, e0
        else:
            cur_e = max(cur_e, e0)
    busy += cur_e - cur_s
    lines.append("GPU busy (any stream) %.1f us = %.1f %%; idle %.1f us" % (
        busy, 100 * busy / (t1 - t0), (t1 - t0) - busy))
    lines.append("")
    lines.append("main stream, in order (start offset us, duration us, gap before us, name):")
    prev = None
    for e in streams[main]:
        gap = e["ts"] - prev if prev is not None else 0.0
        lines.append("%10.1f %9.1f %8.1f  %s" % (e["ts"] - t0, e["dur"], gap, e["name"][:90]))
        prev = e["ts"] + e["dur"]
    for k, v in streams.items():
        if k == main:
            continue
        lines.append("")
        lines.append("stream %s:" % k)
        for e in v:
            lines.append("%10.1f %9.1f           %s" % (e["ts"] - t0, e["dur"], e["name"][:90]))
    open(path + ".txt", "w").write("\n".join(lines) + "\n")
    print("\n".join(lines[:12]), flush=True)


DUMP_TABLE_ROWS = 1 << 16
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, model, last, args, rank, world):
    """The last timed step's prediction and loss and the parameters it left (state_dict names) as
    float32 `<name>.npy`.  A table of more than DUMP_TABLE_ROWS rows is written at a fixed, seeded
    sample of rows, half of them drawn from the ids that step looked up (so rows it updated) and
    half from all ids; `table_rows.npy` (float64) holds their global ids.  At N>1: rank 0's shard."""
    import numpy as np

    g = torch.Generator().manual_seed(2024)
    looked = last["ids"].reshape(-1).cpu()
    gid = torch.unique(torch.cat([
        looked[torch.randint(0, looked.numel(), (DUMP_TABLE_ROWS // 2,), generator=g)],
        torch.randint(0, args.vocab, (DUMP_TABLE_ROWS // 2,), generator=g)]))
    gid = gid[gid % world == rank]
    out = {"pred": last["pred"].reshape(-1), "loss": last["loss"].reshape(-1)}
    for name, t in model.state_dict().items():
        if t.dim() == 2 and t.shape[0] > DUMP_TABLE_ROWS:
            t = t[(gid // world).to(t.device)]
            out["table_rows"] = gid
        out[name] = t
    out = {k: v.detach().to("cpu", torch.float64 if k == "table_rows" else torch.float32).numpy()
           for k, v in out.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


def roofline_step(args, per_ms, step_ms, step_ms_with_events, world):
    """Where the step goes, and how far the WHOLE step is from its own bound.

    per_ms: CUDA-event time per step of every kernel family (event pairs around each C-ABI call;
    the calls of a family are summed).  Composite bound = tower GEMM flops at the measured
    SUSTAINED bf16 rate + the algorithmic HBM bytes of the memory-bound kernels at the measured
    copy bandwidth (SURVEY.md §8(d) per-sample figures; no overlap credit):
      tower   3 (bf16x3) x 3 (fwd, dX, dW) x 2 M sum(K N) flops
      K1      4532 B/sample at D=16 (ids + dense + rows + w1 + feat + y)
      K2      7696 B/sample (ids + dfeat + feat re-read + row RMW)
      Adam    distinct rows x 3 arrays (w, m, v) x G cols x 4 B x 2 (read + write)
      planes  every tower activation is written once and read by the next GEMM, the dW GEMM and the
              ReLU mask (4 B/element each way), dfeat fp32 out
    """
    D, B, F, Dn = args.dim, args.batch, F_SPARSE, N_DENSE
    fc = [int(x) for x in args.fc.split(",")]
    sizes = [(F + Dn) * D] + fc + [1]
    kn = sum(sizes[i] * sizes[i + 1] for i in range(len(sizes) - 1))
    flops = 3 * 3 * 2.0 * B * kn
    peaks = {}
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            peaks = json.load(fh)
    tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    G = (D + 1 + 3) // 4 * 4
    k1 = algorithmic_bytes_fwd(D) * B
    k2 = (F * 8 + (F + Dn) * 4 * D + F * 4 * D + F * 2 * 4 * D) * B
    adam = 0.98 * F * B * 3 * G * 4 * 2
    act = sum(sizes[:-1]) * 4 * B           # planes of every layer input (same bytes as fp32)
    planes = act * 3 + sizes[0] * 4 * B * 2  # written, read by fwd GEMM + dW GEMM (+mask) ; dfeat out/in
    hbm_bytes = k1 + k2 + adam + planes
    bound_ms = flops / (tf * 1e12) * 1e3 + hbm_bytes / (hbm * 1e9) * 1e3
    top = sorted(per_ms.items(), key=lambda kv: -kv[1])
    gemm_ms = sum(v for k, v in per_ms.items() if k in ("tc_linear_fwd", "tc_linear_bwd_dx",
                                                         "tc_linear_bwd_dw"))
    out = {
        "per_kernel_ms": {k: round(v, 4) for k, v in top},
        "sum_of_kernels_ms": round(sum(per_ms.values()), 4),
        "step_ms": round(step_ms, 4), "step_ms_with_events": round(step_ms_with_events, 4),
        "tower_gemm": {"ms": round(gemm_ms, 4), "flops": flops,
                       "achieved_tflops": round(flops / (gemm_ms / 1e3) / 1e12, 1) if gemm_ms else None,
                       "peak_tflops_sustained": tf,
                       "frac": round(flops / (gemm_ms / 1e3) / 1e12 / tf, 3) if gemm_ms else None,
                       "kernels": "tc_gemm_kmajor_kernel / tc_gemm_dw_kernel (tcgen05 + TMEM + TMA)"},
        "composite_bound": {"gemm_ms": round(flops / (tf * 1e12) * 1e3, 4),
                            "hbm_ms": round(hbm_bytes / (hbm * 1e9) * 1e3, 4),
                            "hbm_bytes": int(hbm_bytes), "bound_ms": round(bound_ms, 4),
                            "frac_of_step": round(bound_ms / step_ms, 3)},
    }
    if world > 1:
        out["note"] = ("N>1: embed_fm_fwd reads the RECEIVED rows (contiguous), the random gather is "
                       "the owner-side `gather`; exchange bytes per GPU per direction = "
                       "(N-1)/N * B*F*(8 + 4G) = %d" % int((world - 1) / world * B * F * (8 + 4 * G)))
    return out


def parity_bit(args, model, dm, resident, label_f, rank, world, dev):
    """N>1 correctness bit carried by the scaling run itself: the sharded model's step-0 loss on
    rank 0's first 4096 samples must equal the fp64 oracle evaluated on those samples with the
    touched rows fetched from their owners (a forward through the NCCL exchange, no optimizer)."""
    import torch.distributed as dist
    n = min(4096, args.batch)
    label, ids, dense = resident[0]
    with torch.no_grad():
        pred = model(ids, dense)          # collective: every rank runs its own batch
    loss_dev = float(dm.create_loss(pred[:n], label_f[0][:n]))
    # owners serve rank 0's rows: all-gather of the (small) id slice, each rank contributes its rows
    sl = ids[:n].contiguous()
    dist.broadcast(sl, src=0)
    flat = sl.reshape(-1)
    uniq = torch.unique(flat[flat != 0])
    mine = uniq[uniq % world == rank]
    tab = model.fm._fused
    rows = tab.weight[mine // world, :tab.embedding_dim + 1].contiguous()
    sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(sizes, torch.tensor([mine.numel()], device=dev))
    cap = int(max(int(t) for t in sizes))
    pad_ids = torch.zeros(cap, dtype=torch.int64, device=dev)
    pad_rows = torch.zeros(cap, rows.shape[1], device=dev)
    pad_ids[:mine.numel()], pad_rows[:mine.numel()] = mine, rows
    all_ids = [torch.empty_like(pad_ids) for _ in range(world)]
    all_rows = [torch.empty_like(pad_rows) for _ in range(world)]
    dist.all_gather(all_ids, pad_ids)
    dist.all_gather(all_rows, pad_rows)
    if rank != 0:
        return None
    from oracle import nets
    gid = torch.cat([a[:int(k)] for a, k in zip(all_ids, sizes)])
    grow = torch.cat([a[:int(k)] for a, k in zip(all_rows, sizes)])
    order = torch.argsort(gid)
    gid, grow = gid[order], grow[order]
    Dd = tab.embedding_dim
    remap = (torch.searchsorted(gid, sl.reshape(-1)).reshape(sl.shape) + 1) * (sl != 0)
    p = {"fm.embedding.weight": torch.cat([torch.zeros(1, Dd, device=dev), grow[:, :Dd]]),
         "fm.embedding_one.weight": torch.cat([torch.zeros(1, 1, device=dev), grow[:, Dd:Dd + 1]])}
    for k, v in model.state_dict().items():
        if not k.startswith("fm.embedding"):
            p[k] = v
    p = {k: v.detach().double().cpu() for k, v in p.items()}
    remap = remap.cpu()
    ref = nets.deepfm_forward(p, [remap[:, i:i + 1] for i in range(remap.shape[1])],
                              dense[:n].double().cpu(), len([int(x) for x in args.fc.split(",")]))
    loss_ref = float(nets.log_loss(ref, label_f[0][:n].double().cpu()).mean())
    err = float((pred[:n].double().cpu() - ref).abs().max())
    return {"samples": n, "loss": loss_dev, "oracle_loss": loss_ref,
            "max_abs_pred_err": err, "ok": bool(abs(loss_dev - loss_ref) < 1e-4 * abs(loss_ref)
                                                and err < 1e-4)}


def cpu_baseline(args):
    V = args.vocab
    note = ""
    try:
        import psutil
        need = V * (args.dim + 1) * 4 * 3.2
        avail = psutil.virtual_memory().available
        if avail < need * 1.3:
            V = max(1_000_001, int(avail / 1.3 / ((args.dim + 1) * 4 * 3.2)))
            note = " (V reduced from %d: host RAM)" % args.vocab
    except ImportError:
        pass
    value, cores, _, _ = time_cpu_port(args, V, args.cpu_steps)
    return {"value": value, "unit": "samples/s", "cores": cores, "kind": "port",
            "sample": "%d steps of B=%d after warm-up and thread-count calibration (%d of %d host "
                      "threads), same DeepFM step, V=%d%s, fp32, sparse grads + lazy Adam "
                      "(oracle/cpu_train.py)" % (args.cpu_steps, args.cpu_batch, cores,
                                                 os.cpu_count() or 1, V, note)}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        # a multi-rank job that stops making progress (a rank waiting in a collective its peers
        # never entered) would otherwise sit until the caller's limit with no trace: after
        # B200REC_BENCH_WATCHDOG_S seconds dump every thread's Python stack to stderr and exit.
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ.get("B200REC_BENCH_WATCHDOG_S", "420")),
                                          exit=True)
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    elif args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import faulthandler

            import torch.distributed as dist
            dist.destroy_process_group()
            faulthandler.cancel_dump_traceback_later()


if __name__ == "__main__":
    main()
