#!/usr/bin/env python
"""Benchmark of the gated-GCN hot path (BASELINE.json metric: fwd+bwd graphs/sec).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference ...                     # the reference algorithm on host cores
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed

One step = one pass of the hot path over one synthetic batch: gated GCN stack
forward + loss (CE + 0.01 xy + 0.01 kl, train.py:115-118) + backward + Adam step.
Workload at every N: config C2 of BASELINE.json per GPU (4096 trees <= 50 tokens,
D = 300, L = 2, bf16) -> weak scaling; for N > 1 each rank owns its own batch
and parameter gradients are all-reduced over NCCL every step.
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

GATE_W = KL_W = 0.01        # train.py:300-301
L2_BYTES = 126e6


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
def make_workload(cfg_name: str, rank: int, n_graphs=None):
    from ed_gated_gcn_b200 import synth
    c = dict(synth.CONFIGS[cfg_name])
    batch = synth.config_batch(cfg_name, n_graphs=n_graphs, seed_offset=rank)
    g = torch.Generator().manual_seed(synth.REFERENCE_SEED + rank)
    x = torch.randn(batch.n_rows, c["D"], generator=g)
    targets = torch.randint(0, c["C"], (batch.n_graphs,), generator=g)
    return c, batch, x, targets


def algorithmic_per_graph(c, batch):
    """SURVEY 8d: per token-row per layer fwd+bwd = 5*D*s + 32 bytes, 6*D^2 + 12*D flops."""
    s = 2 if c["dtype"] == "bf16" else 4
    rows_per_graph = batch.n_rows / batch.n_graphs
    return (5 * c["D"] * s + 32) * c["L"] * rows_per_graph, (6 * c["D"] ** 2 + 12 * c["D"]) * c["L"] * rows_per_graph


def algo_bytes_of_call(name, args):
    """Algorithmic HBM bytes of one C-ABI call (compulsory reads + writes of its row matrices)."""
    es = lambda d: 2 if d == 1 else 4
    if name == "edg_linear":      # A[M,K] read + C[M,Nout] write (+ weights, read once)
        _, adt, _, M, K, _, _, Nout, _, _, _, cdt, _, _ = args
        return M * K * es(adt) + M * Nout * es(cdt) + Nout * K * es(adt)
    if name == "edg_aggregate":   # x read + y write + 16 B/row of CSR (SURVEY 8d)
        _, xdt, _, _, ydt, _, N, D = args[:8]
        return N * D * (es(xdt) + es(ydt)) + 16 * N
    if name == "edg_wgrad":       # both row matrices read once
        _, _, K1, _, _, K2, dt, R = args[:8]
        return R * (K1 + K2) * es(dt)
    if name == "edg_gcn_layer":   # x read + y write + 16 B/row of graph structure + the weight slice (SURVEY 8d, fused form)
        _, _, N, K, _, _, Nout = args[:7]
        return N * K * 2 + N * Nout * 2 + 16 * N + Nout * K * 2
    if name == "edg_head_du":     # du written once; seven [B,D] fp32 side arrays
        N, B, D = args[9:12]
        return N * D * 2 + 7 * B * D * 4
    if name in ("edg_pool_fwd", "edg_scores_kl_fwd"):       # one read of the row matrix
        _, dt, _, _, B, D = args[:6]
        N = args[18] if name == "edg_scores_kl_fwd" else args[11]
        return N * D * es(dt)
    if name == "edg_head_bwd":    # h read, dh written
        _, dt, _, _, B, D = args[:6]
        return 2 * args[-2] * D * es(dt) if args[18] else args[-2] * D * es(dt)
    return None


def algo_flops_of_call(name, args):
    """Tensor-core flops of one C-ABI call (2 * M * N * K of its GEMM), None for the streaming kernels."""
    if name == "edg_linear":
        return 2 * args[3] * args[4] * args[7]
    if name == "edg_gcn_layer":
        return 2 * args[2] * args[3] * args[6]
    if name == "edg_wgrad":
        return 2 * args[7] * args[2] * args[5]
    return None


class KernelTimer:
    """CUDA-event timing of every C-ABI call (events recorded on the launching stream)."""

    def __init__(self):
        self.records = []

    def hook(self, name, args, fn):
        # no synchronisation here: the profiled step is enqueued while the GPU is still busy with a spin kernel
        # (see `preload`), so the host runs ahead and the interval between the two events is this call's kernel
        # time as it is inside the CUDA-graph replay, not launch latency on an idle GPU
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = fn(*args)
        b.record()
        self.records.append((name, args, a, b))
        return rc

    @staticmethod
    def preload(ms: float = 12.0):
        """Keep the GPU busy for ~ms so that the whole next step is enqueued before its first kernel starts."""
        torch.cuda.synchronize()
        torch.cuda._sleep(int(ms * 1e-3 * 1.9e9))

    def table(self, n_steps):
        torch.cuda.synchronize()
        agg = {}
        for name, args, a, b in self.records:
            key = name
            if name == "edg_linear":
                key = f"edg_linear[M={args[3]},K={args[4]},N={args[7]}]"
            elif name == "edg_aggregate":
                key = f"edg_aggregate[mode={args[10]}]"
            elif name == "edg_wgrad":
                key = f"edg_wgrad[R={args[7]}]"
            ms = a.elapsed_time(b)
            e = agg.setdefault(key, dict(ms=0.0, n=0, bytes=algo_bytes_of_call(name, args), flops=algo_flops_of_call(name, args),
                                         name=name))
            e["ms"] += ms
            e["n"] += 1
        for e in agg.values():
            e["ms_per_step"] = e["ms"] / n_steps
            e["us_per_launch"] = 1e3 * e["ms"] / e["n"]
            e["launches_per_step"] = e["n"] / n_steps
        return agg


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """Write every tensor as ``out_dir/<name>.npy`` in float32, at most DUMP_BYTES in all, so two builds can be compared
    output for output.  The smallest arrays are written whole; an array larger than its share of what is left keeps
    the first rows of a permutation seeded by its name, in ascending order, and their indices go to
    ``<name>.rows.npy`` (float64).  A smaller share keeps a subset of the rows a larger one keeps, so two dumps whose
    budgets split differently (one array more or less) still line up on the rows they share."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(((k, v.detach().float().cpu().numpy()) for k, v in arrays.items()), key=lambda kv: kv[1].nbytes)
    left = DUMP_BYTES - 2 * 256 * len(items)      # room for the .npy headers of each array and its row indices
    for i, (name, a) in enumerate(items):
        share = left // (len(items) - i)
        if a.nbytes > share:
            perm = np.random.default_rng(zlib.crc32(name.encode())).permutation(a.shape[0])
            rows = np.sort(perm[:max(1, share // (a.nbytes // a.shape[0] + 8))]).astype(np.float64)
            np.save(os.path.join(out_dir, name + ".rows.npy"), rows)
            a = a[rows.astype(np.int64)]
            left -= rows.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes


# ---------------------------------------------------------------------------------------------
def build_model(c, device, torch_head=False):
    import ed_gated_gcn_b200 as E
    torch.manual_seed(14181)
    stack = E.GatedGCNStack(c["D"], n_layers=c["L"], n_classes=c["C"], gate_arch="sig-2",
                            compute_dtype=c["dtype"]).to(device)
    # self.dense (bert_amir5.py:643): E.DenseHead is that nn.Linear run by the block's own kernels; --torch-head keeps
    # torch's nn.Linear + F.cross_entropy (cat, three cuBLAS GEMMs, four loss kernels) for comparison
    dense = (torch.nn.Linear if torch_head else E.DenseHead)(2 * c["D"], c["C"]).to(device)
    for p in list(stack.parameters()) + list(dense.parameters()):        # train.py:75-84
        if p.dim() > 1:
            torch.nn.init.xavier_uniform_(p)
        else:
            torch.nn.init.uniform_(p, -1.0 / p.shape[0] ** 0.5, 1.0 / p.shape[0] ** 0.5)
    return stack, dense


def run_b200(args):
    import torch.distributed as dist
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import _lib, ops, parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))

    c, batch, x_host, tgt_host = make_workload(args.config, rank)
    if args.dtype:                       # not the headline: the fp32-parity mode of the same step (DESIGN section 5)
        c["dtype"] = args.dtype
    cd = torch.bfloat16 if c["dtype"] == "bf16" else torch.float32
    if cd == torch.bfloat16:
        # the caller's own classifier head (self.dense, bert_amir5.py:643) is host torch: let cuBLAS use TF32
        # tensor cores for it in the bf16 configuration (the fp32 parity mode keeps full fp32)
        torch.backends.cuda.matmul.allow_tf32 = True
    stack, dense = build_model(c, dev, torch_head=args.torch_head)
    params = list(stack.parameters()) + list(dense.parameters())
    if world > 1:
        for p in params:
            dist.broadcast(p.data, 0)
    # train.py:239-243 trains with Adam: the same update rule as ONE launch of this package (edg_adam_multi);
    # --torch-adam keeps torch.optim.Adam(fused, capturable) for comparison
    if args.torch_adam:
        opt = torch.optim.Adam(params, lr=1e-3, fused=True, capturable=True)
    else:
        opt = E.FusedAdam(params, lr=1e-3)
    reducer = parallel.GradientAllReducer(params)
    if args.allreduce == "none" and not args.overlap_allreduce:
        reducer = lambda: None
    ar_mode = "layer" if args.overlap_allreduce else args.allreduce
    if world > 1 and ar_mode == "layer":
        stack.grad_ready_hook = reducer.hook          # per-layer all-reduce from inside the backward pass
    if world > 1 and ar_mode == "bucket":
        stack.grad_bucket_hook = reducer.bucket       # one flat all-reduce next to the input-gradient projection
    if args.torch_head:
        logits_fn = lambda a, p: dense(torch.cat([a, p], 1))
        ce_loss = torch.nn.functional.cross_entropy
    else:
        logits_fn = dense
        ce_loss = E.cross_entropy                     # nn.CrossEntropyLoss (train.py:96) in two launches
    # train.py:115-118: loss = CE + gate_weight * xy + kl_weight * kl
    if args.torch_head or os.environ.get("EDG_BENCH_TORCH_SUM") == "1":      # (env: same-box A/B of E.total_loss)
        combine = lambda ce, xy, kl: ce + GATE_W * xy + KL_W * kl
    else:
        combine = lambda ce, xy, kl: E.total_loss(ce, xy, kl, GATE_W, KL_W)
    head_params = list(dense.parameters())

    # ---- device-resident inputs (the `value` number)
    # the whole padded [N, pitch] allocation is the leaf: its gradient comes back dense, so autograd keeps
    # it without the strided copy a [:, :D] view would need
    x_dev = torch.zeros(batch.n_rows, ops.row_pitch(c["D"], cd), dtype=cd, device=dev)
    x_dev[:, :c["D"]].copy_(x_host)
    x_dev.requires_grad_(True)
    graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=dev)
    anchor = torch.from_numpy(batch.anchor).to(dev)
    dist_dev = E.tree_distance(graph, anchor)
    tgt = tgt_host.to(dev)

    # what the latest step computed; under a CUDA graph these are the buffers every replay rewrites.  The gradients are
    # taken here, not from p.grad later: the steps that follow the capture (zero_grad, the e2e graphs) rebind p.grad
    last = {}
    named = [("stack." + n, p) for n, p in stack.named_parameters()] + [("dense." + n, p) for n, p in dense.named_parameters()]

    def step_resident():
        opt.zero_grad(set_to_none=True)
        x_dev.grad = None
        out = stack(x_dev, graph, anchor, dist_dev, logits_fn, head_params=head_params)
        loss = combine(ce_loss(out.logits, tgt), out.xy, out.kl)
        loss.backward()
        reducer()
        opt.step()
        last.clear()
        last.update(loss=loss.detach(), logits=out.logits.detach(), xy=out.xy.detach(), kl=out.kl.detach(),
                    scores=out.scores.detach(), pooled=out.pooled.detach())
        last["x.grad"] = x_dev.grad[:, :c["D"]]
        last.update({"grad." + n: p.grad for n, p in named if p.grad is not None})
        return loss

    # ---- host-resident inputs through the public API (the `e2e` number)
    pin = lambda t: t.pin_memory()
    ld = ops.row_pitch(c["D"], cd)
    x_pin = torch.zeros(batch.n_rows, ld, dtype=cd).pin_memory()
    x_pin[:, :c["D"]].copy_(x_host)
    heads_pin, sp_pin = pin(torch.from_numpy(batch.heads)), pin(torch.from_numpy(batch.sent_ptr))
    anchor_pin, tgt_pin = pin(torch.from_numpy(batch.anchor)), pin(tgt_host)
    max_len = int(batch.lengths.max())
    h2d = sum(t.numel() * t.element_size() for t in (x_pin, heads_pin, sp_pin, anchor_pin, tgt_pin))
    loss_pin = torch.zeros((), dtype=torch.float32).pin_memory()

    def step_e2e_enqueue():
        opt.zero_grad(set_to_none=True)
        xb = x_pin.to(dev, non_blocking=True).requires_grad_(True)
        g = E.build_graph(heads_pin.to(dev, non_blocking=True), sp_pin.to(dev, non_blocking=True), max_len=max_len,
                          device=dev)
        an = anchor_pin.to(dev, non_blocking=True)
        tg = tgt_pin.to(dev, non_blocking=True)
        dd = E.tree_distance(g, an)
        out = stack(xb, g, an, dd, logits_fn, head_params=head_params)
        loss = combine(ce_loss(out.logits, tg), out.xy, out.kl)
        loss.backward()
        reducer()
        opt.step()
        loss_pin.copy_(loss.detach(), non_blocking=True)

    def step_e2e():
        step_e2e_enqueue()
        torch.cuda.current_stream().synchronize()                 # the caller reads the loss every step
        return loss_pin

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    from ed_gated_gcn_b200.runtime import GraphedStep
    run_resident, run_e2e = step_resident, step_e2e
    l0 = _lib.LAUNCHES["kernels"]
    step_resident()
    kernels_per_step = _lib.LAUNCHES["kernels"] - l0           # this package's kernels in one step
    if not args.no_graph:
        # whole step (fwd + loss + bwd + all-reduce + Adam) as one CUDA graph; the e2e graph also holds
        # the H2D copies from pinned memory, the CSR/distance kernels and the loss D2H copy
        g_res = GraphedStep(step_resident)
        run_resident = g_res
        opt.zero_grad(set_to_none=True)

        # e2e: two static input sets; batch i+1's H2D copies (pinned -> device, copy stream) overlap batch i's
        # graph (CSR + distance kernels + fwd + bwd + all-reduce + Adam + loss D2H); every step still copies its
        # own inputs inside the timed region and the host reads every step's loss
        from ed_gated_gcn_b200.runtime import DoubleBufferedStep
        sets = []
        for _k in range(2):
            sets.append(dict(x=torch.zeros(batch.n_rows, ld, dtype=cd, device=dev).requires_grad_(True),
                             heads=torch.zeros(batch.n_rows, dtype=torch.int32, device=dev),
                             sp=torch.zeros(batch.n_graphs + 1, dtype=torch.int32, device=dev),
                             anchor=torch.zeros(batch.n_graphs, dtype=torch.int32, device=dev),
                             tgt=torch.zeros(batch.n_graphs, dtype=torch.int64, device=dev)))

        def copy_in(k):
            st = sets[k]
            with torch.no_grad():
                st["x"].copy_(x_pin, non_blocking=True)
                st["heads"].copy_(heads_pin, non_blocking=True)
                st["sp"].copy_(sp_pin, non_blocking=True)
                st["anchor"].copy_(anchor_pin, non_blocking=True)
                st["tgt"].copy_(tgt_pin, non_blocking=True)

        def compute(k):
            st = sets[k]
            opt.zero_grad(set_to_none=True)
            st["x"].grad = None
            g = E.build_graph(st["heads"], st["sp"], max_len=max_len, device=dev)
            dd = E.tree_distance(g, st["anchor"])
            out = stack(st["x"], g, st["anchor"], dd, logits_fn, head_params=head_params)
            loss = combine(ce_loss(out.logits, st["tgt"]), out.xy, out.kl)
            loss.backward()
            reducer()
            opt.step()
            loss_pin.copy_(loss.detach(), non_blocking=True)
            return loss_pin

        pipe = DoubleBufferedStep(copy_in, compute)
        run_e2e = pipe.step
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total = timed(run_resident, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {**last, **{"param." + n: p for n, p in named}})    # params: after this step's Adam
    launches = kernels_per_step * args.steps
    loss_val = float(run_resident().item())
    ms_e2e = timed(run_e2e, args.steps, max(3, args.warmup // 2))
    clocks = sampler.stop() if rank == 0 else None          # sampled across both timed regions

    graphs_total = batch.n_graphs * world
    if world > 1:
        t = torch.tensor([batch.n_graphs], device=dev)
        dist.all_reduce(t)
        graphs_total = int(t.item())
    ms_step = ms_total / args.steps
    value = graphs_total / (ms_step * 1e-3)
    e2e_value = graphs_total / (ms_e2e / args.steps * 1e-3)

    # ---- per-kernel CUDA-event pass (rank 0): which kernel dominates, and its roofline
    roof = None
    ktable = {}
    nprof = 5
    kt = KernelTimer()
    torch.cuda.synchronize()
    if rank == 0:
        _lib.HOOK = kt.hook
    from ed_gated_gcn_b200 import gated as _gated
    overlap_was, _gated._OVERLAP = _gated._OVERLAP, False      # one stream: every interval is one kernel, undisturbed
    for _ in range(nprof):          # every rank runs these steps: they contain the gradient all-reduce
        if rank == 0:
            kt.preload()
        step_resident()
    _gated._OVERLAP = overlap_was
    _lib.HOOK = None
    torch.cuda.synchronize()
    if rank == 0:
        ktable = kt.table(nprof)
        peaks = load_peaks()
        # dominant kernel = largest time per step among the row-matrix kernels (those with defined algorithmic bytes)
        top_key, top = max(((k, v) for k, v in ktable.items() if v["bytes"]), key=lambda kv: kv[1]["ms_per_step"])
        achieved = None
        if top["bytes"]:
            achieved = top["bytes"] / (top["us_per_launch"] * 1e-6) / 1e9
        share = top["ms_per_step"] / sum(e["ms_per_step"] for e in ktable.values())
        traffic = None                  # DRAM bytes per launch of that kernel from the committed ncu --set full capture
        tpath = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
        if os.path.exists(tpath):
            t = json.load(open(tpath)).get(top_key)
            if t:
                traffic = t["dram_read_bytes"] + t["dram_write_bytes"]
        bpg, fpg = algorithmic_per_graph(c, batch)
        # which roofline binds this configuration (SURVEY 8d): bytes / HBM peak against flops / sustained tensor peak
        tensor_bound = fpg / (peaks["tf_sust"] * 1e12) > bpg / (peaks["hbm"] * 1e9)
        if tensor_bound and top.get("flops"):
            tf = top["flops"] / (top["us_per_launch"] * 1e-6) / 1e12
            roof = {"bound": "tensor", "kernel": top_key, "achieved": tf, "peak": peaks["tf_sust"], "unit": "TFLOP/s",
                    "frac": tf / peaks["tf_sust"], "traffic": traffic}
        else:
            roof = {"bound": "hbm", "kernel": top_key, "achieved": achieved, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": (achieved / peaks["hbm"]) if achieved else None, "traffic": traffic}
        roof.update({"peak_source": peaks["src"], "us_per_launch": top["us_per_launch"],
                     "launches_per_step": top["launches_per_step"], "share_of_kernel_time": share,
                     "algorithmic_bytes_per_launch": top["bytes"], "hbm_gbps": achieved,
                     "hbm_frac": (achieved / peaks["hbm"]) if achieved else None})
        # every row-streaming kernel against the HBM peak (algorithmic bytes / measured time)
        roof["row_kernels"] = {k: {"us": round(v["us_per_launch"], 1), "gbps": round(v["bytes"] / (v["us_per_launch"] * 1e-6) / 1e9),
                                   "hbm_frac": round(v["bytes"] / (v["us_per_launch"] * 1e-6) / 1e9 / peaks["hbm"], 3)}
                               for k, v in ktable.items() if v["bytes"]}
        roof["whole_step"] = {
            "algorithmic_bytes_per_graph": bpg, "algorithmic_flops_per_graph": fpg,
            "hbm_frac": bpg * (value / world) / (peaks["hbm"] * 1e9),
            "tensor_frac": fpg * (value / world) / (peaks["tf_sust"] * 1e12)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args.config, budget_s=args.cpu_seconds)

    if rank == 0:
        work_mb = 28 * batch.n_rows * ops.row_pitch(c["D"], cd) * (2 if cd == torch.bfloat16 else 4) / 1e6
        line = {
            "metric": "gated-GCN fwd+bwd graphs/sec", "value": value, "unit": "graphs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": c["dtype"], "data": "synthetic",
            "config": {"workload": f"{args.config}: {c['L']}-layer gated GCN, hidden {c['D']}, "
                                   f"{batch.n_graphs} synthetic dependency trees <= {c['n_max']} tokens per GPU "
                                   f"({batch.n_rows} rows), fwd+bwd + gate-diversity + importance-score loss + Adam",
                       "graphs_per_gpu": batch.n_graphs, "rows_per_gpu": batch.n_rows, "hidden": c["D"],
                       "layers": c["L"], "classes": c["C"], "parallelism": f"dp{world}",
                       "allreduce": (ar_mode if world > 1 else None),
                       "l2": f"no explicit flush: each step streams ~{work_mb:.0f} MB of distinct row matrices "
                             f"(> {L2_BYTES / 1e6:.0f} MB L2) so inputs are evicted between steps",
                       "loss": float(loss_val)},
            "e2e": {"value": e2e_value, "unit": "graphs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps,
                    "note": "pinned host inputs -> H2D (copy stream, double-buffered: batch i+1 copies while batch i "
                            "computes) -> heads->CSR + distance kernels -> fwd+bwd+Adam -> loss D2H + host sync every step; the host rows "
                            "are already bf16 with the padded pitch (a caller holding the reference's fp32 features pays a "
                            "cast or twice the bytes)"},
            "gpu_launches": int(launches),
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "kernels": {k: {"us_per_launch": round(v["us_per_launch"], 2), "launches_per_step": v["launches_per_step"],
                            "ms_per_step": round(v["ms_per_step"], 4)} for k, v in
                        sorted(ktable.items(), key=lambda kv: -kv[1]["ms_per_step"])},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # leave without tearing the NCCL communicator down: destroy_process_group() can block while CUDA graphs
        # that captured collectives are still alive, and there is nothing left to do
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


# ---------------------------------------------------------------------------------------------
def cpu_baseline(cfg_name: str, budget_s: float = 15.0, graphs: int = 256, as_line: bool = False, steps=None,
                 warmup=None):
    """The reference algorithm (oracle port: reference GraphConvolution x L + the BertAmir55 block,
    fp32, dense padded [B,T,T] adjacency exactly as the reference consumes it) on the host cores."""
    from oracle import ref_oracle as O
    from ed_gated_gcn_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    c = synth.CONFIGS[cfg_name]
    graphs = min(graphs, c["n_graphs"])                        # train.py:297 default batch_size 256
    batch = synth.config_batch(cfg_name, n_graphs=graphs)
    D, C, Lyr = c["D"], c["C"], c["L"]
    T = int(batch.lengths.max())
    g = torch.Generator().manual_seed(1)
    x = torch.randn(graphs, T, D, generator=g, requires_grad=True)
    adj = O.dense_batch_from_heads(batch.heads_list(), T)
    dist = torch.tensor([O.pad_distance(O.tree_distance_bfs(h, int(batch.anchor[b])), T, "max+1")
                         for b, h in enumerate(batch.heads_list())])
    anchor = torch.from_numpy(batch.anchor).long()
    targets = torch.randint(0, C, (graphs,), generator=g)
    mk = lambda *s: torch.nn.Parameter(torch.empty(*s))
    gcn_p = [(mk(D, D), mk(D)) for _ in range(Lyr)]
    gate_p = [[(mk(D, D), mk(D)), (mk(D, D), mk(D))] for _ in range(Lyr)]
    fc_w, fc_b, dw, db = mk(C, 2 * D), mk(C), mk(C, 2 * D), mk(C)
    params = [p for pair in gcn_p for p in pair] + [p for gp in gate_p for pair in gp for p in pair] + [fc_w, fc_b, dw, db]
    O.reference_init_(params, g)
    opt = torch.optim.Adam(params, lr=1e-3)

    def step():
        opt.zero_grad(set_to_none=True)
        x.grad = None
        out = O.gated_block_ref(x, adj, anchor, dist, gcn_p, gate_p, fc_w, fc_b,
                                lambda a, p: torch.cat([a, p], 1) @ dw.t() + db)
        loss = O.block_loss_ref(out, targets, GATE_W, KL_W)
        loss.backward()
        opt.step()
        return loss

    nw = 5 if warmup is None else warmup
    for _ in range(nw):
        step()
    times = []
    t_end = time.time() + budget_s
    n_max = steps if steps is not None else 10_000
    while len(times) < n_max and (steps is not None or time.time() < t_end or len(times) < 20):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    med = float(np.median(times))
    try:
        model = [l.split(":")[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")][0]
    except Exception:
        model = "unknown"
    res = {"value": graphs / med, "unit": "graphs/s", "cores": cores, "kind": "port",
           "sample": f"{cfg_name} shapes (D={D}, L={Lyr}, C={C}, trees <= {c['n_max']} tokens) at the reference's "
                     f"default batch of {graphs} graphs (train.py:297), fp32, dense [B,{T},{T}] adjacency, "
                     f"{len(times)} timed fwd+bwd+Adam steps after {nw} warm-up, median {med * 1e3:.2f} ms/step",
           "cpu_model": model, "ms_per_step": med * 1e3, "steps": len(times)}
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    res = cpu_baseline(args.config, steps=args.steps, warmup=args.warmup)
    from ed_gated_gcn_b200 import synth
    c = synth.CONFIGS[args.config]
    line = {"impl": "reference", "metric": "gated-GCN fwd+bwd graphs/sec", "value": res["value"], "unit": "graphs/s",
            "n_gpus": world, "steps": res["steps"], "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.config}: reference algorithm (oracle port) on host CPU; " + res["sample"]},
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "cpu_model")},
            "e2e": {"value": res["value"], "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dtype", default=None, choices=["bf16", "f32"],
                    help="override the configuration's compute mode (f32 = the 1e-5 parity mode; the headline is the config's own)")
    ap.add_argument("--overlap-allreduce", action="store_true",
                    help="all-reduce every gradient group from inside the backward pass (GradientAllReducer.hook) instead of "
                         "one coalesced in-place all-reduce after it")
    ap.add_argument("--allreduce", default=os.environ.get("EDG_BENCH_ALLREDUCE", "bucket"), choices=["flat", "layer", "bucket", "none"],
                    help="flat: one flat-bucket all-reduce after the backward pass; bucket: the same bucket packed inside the "
                         "backward pass as soon as the last parameter gradient exists, reduced next to the input-gradient "
                         "projection (GradientAllReducer.bucket); layer = --overlap-allreduce; none = NO all-reduce (diagnostic "
                         "only: what N processes cost without the collective; not a training step)")
    ap.add_argument("--torch-head", action="store_true",
                    help="torch nn.Linear + F.cross_entropy for the classifier head and the loss instead of E.DenseHead / E.cross_entropy")
    ap.add_argument("--torch-adam", action="store_true", help="torch.optim.Adam(fused, capturable) instead of edg_adam_multi")
    ap.add_argument("--no-graph", action="store_true", help="enqueue kernels from Python instead of replaying a CUDA graph")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (loss, logits, xy, kl, scores, "
                         "pooled, the input and parameter gradients, the updated parameters) as DIR/<name>.npy, float32, "
                         "<= 64 MB in all (larger arrays: a seeded sample of their rows, indices in DIR/<name>.rows.npy)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
