"""Micro-benchmark of the fused layer kernel (edg_gcn_layer) at config-C2 size against the unfused kernels it
replaces (aggregate + linear + pool).  Ring of 4 input sets (> L2), CUDA events around back-to-back launches.
Sweeps the bring-up switches EDG_FUSED_EPI_WARPS / EDG_FUSED_STAGES / EDG_FUSED_ROWS / EDG_FUSED_PF."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ed_gated_gcn_b200 as E
from ed_gated_gcn_b200 import ops, synth

cfg = os.environ.get("CFG", "C2")
dev = "cuda:0"
c = synth.CONFIGS[cfg]
batch = synth.config_batch(cfg)
D, B, N = c["D"], batch.n_graphs, batch.n_rows
cd = torch.bfloat16
graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=dev)
RING = 4
xs = [ops.alloc_rows(N, D, cd, dev, zero=True) for _ in range(RING)]
for t in xs:
    t.copy_(torch.randn(N, D, device=dev))
w = ops.alloc_rows(D, D, cd, dev, zero=True); w.copy_(torch.randn(D, D) / D ** 0.5)
bias = torch.randn(D, device=dev)
gates = torch.rand(1, B, D, device=dev)
pv = torch.randn(B, D, device=dev)
two = 2 * N * D * 2 + 16 * N


def bench(name, fn, nbytes=two, rounds=3):
    """RING * rounds launches captured into ONE CUDA graph and replayed: device time without host launch overhead."""
    for i in range(RING):
        fn(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    keep = []
    with torch.cuda.graph(g):
        for r in range(rounds):
            for i in range(RING):
                keep.append(fn(i))
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        g.replay()
    b.record(); torch.cuda.synchronize()
    us = a.elapsed_time(b) * 1e3 / (3 * rounds * RING)
    print(f"{name:58s} {us:8.1f} us {nbytes / us / 1e3:7.0f} GB/s ({nbytes / us / 1e3 / 6450.3:.2f} of 6450)", flush=True)
    return us


print(f"cfg {cfg}: N={N} D={D} B={B}; one row matrix = {N * xs[0].stride(0) * 2 / 1e6:.1f} MB")
bench("aggregate fwd (unfused)", lambda i: ops.aggregate(xs[i], graph, 0))
bench("linear (unfused)", lambda i: ops.linear(xs[i], w, bias))
bench("pool_fwd V=1 (unfused)", lambda i: ops.pool_fwd(xs[i], graph, gates), N * D * 2)
bench("torch copy (ref)", lambda i: xs[(i + 1) % RING].copy_(xs[i]), 2 * N * D * 2)

KEYS = ("EPI_WARPS", "STAGES", "ROWS", "PF", "DEBUG", "SLEEP", "BOXROWS")
sweeps = [dict(), dict(EPI_WARPS=12), dict(STAGES=3)]
only_plain = False
if len(sys.argv) > 1 and sys.argv[1] == "pipe":       # load-pipeline study: epilogue work switched off
    only_plain = True
    sweeps = [dict(DEBUG=d, PF=0, BOXROWS=b) for d in (3, 23, 23 + 64, 3 + 64) for b in (32, 64, 128)]
    sweeps += [dict(DEBUG=23 + 64, PF=0, STAGES=s) for s in (2, 3)] + [dict(DEBUG=0, PF=0, BOXROWS=b) for b in (32, 128)]
if len(sys.argv) > 1 and sys.argv[1] == "quick":      # one configuration taken from the environment (ncu runs)
    sweeps = [{k: int(os.environ["EDG_FUSED_" + k]) for k in KEYS if "EDG_FUSED_" + k in os.environ}]
for sw in sweeps:
    for k in KEYS:
        os.environ.pop("EDG_FUSED_" + k, None)
    for k, v in sw.items():
        os.environ["EDG_FUSED_" + k] = str(v)
    rows = ops.fused_tile_rows(D, D)
    graph.__dict__.pop("_plans", None)
    plan = graph.tile_plan(rows)
    nt = int(plan[1].item())
    tag = f"{sw} rows={rows} tiles={nt}"
    y, hmax, harg, _ = ops.gcn_layer(xs[0], w, bias, graph, 0, plan, rows, want_pool=True)
    pa = harg.clone()
    if only_plain:
        bench(f"fused fwd no pool     {tag}", lambda i: ops.gcn_layer(xs[i], w, bias, graph, 0, plan, rows))
        continue
    bench(f"fused fwd + pool      {tag}", lambda i: ops.gcn_layer(xs[i], w, bias, graph, 0, plan, rows, want_pool=True))
    bench(f"fused fwd no pool     {tag}", lambda i: ops.gcn_layer(xs[i], w, bias, graph, 0, plan, rows))
    bench(f"fused adjoint+colsum  {tag}", lambda i: ops.gcn_layer(xs[i], w, None, graph, 1, plan, rows, want_colsum=True))
    bench(f"fused adjoint+patch+cs{tag}", lambda i: ops.gcn_layer(xs[i], w, None, graph, 1, plan, rows, patch=(pv, pa), want_colsum=True))
