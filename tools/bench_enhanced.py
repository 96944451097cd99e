"""Cost of carrying dependency graphs that are not forests (enhanced dependencies) on the packed path, at the C2 shape
(4096 sentences of 5..50 tokens, D = 300, L = 2, bf16).  Prints one JSON line (and writes it to --out if given):

  - CUDA-event medians of the CSR build: build_graph on heads only, on heads + extra edges at two synthetic rates
    (synth.with_extra_edges), and graph_from_dense on the equivalent device-resident [4096, 50, 50] fp32 matrix;
  - host->device bytes per batch of the packed form and of the dense form, computed from shapes;
  - the captured C2 training step (bench.build_model; CSR build + distances + forward + backward + Adam in one CUDA
    graph, from device-resident inputs) on the tree batch and on the same batch with extra edges, with the fused
    layer plan asserted to be taken;
  - the card's name, power limit and max SM clock, read in the same run.

    python tools/bench_enhanced.py [--out profiles/r03_a_bench_enhanced.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch


def card(dev):
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        pl, sm = (v.strip() for v in q.strip().split(","))
        info.update(power_limit_w=float(pl), sm_max_mhz=float(sm))
    except Exception as e:                      # noqa: BLE001 -- report what could not be read
        info.update(power_limit_w=None, sm_max_mhz=None, nvidia_smi=str(e))
    return info


def median_ms(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def exact_max_sent_nnz(batch):
    """n_b + 2 (tree edges) + 2 E_b, maximised (synth trees have n_b - 1 edges; synth extras are distinct)."""
    n = batch.lengths.astype(np.int64)
    e = np.diff(batch.edge_ptr).astype(np.int64) if batch.extra_edges is not None else 0
    return int((n + 2 * np.maximum(n - 1, 0) + 2 * e).max())


def dense_of(batch, T):
    adj = np.zeros((batch.n_graphs, T, T), dtype=np.float32)
    adj[:, np.arange(T), np.arange(T)] = 1.0
    b = np.repeat(np.arange(batch.n_graphs), batch.lengths)
    i = np.arange(batch.n_rows) - batch.sent_ptr[b]
    kid = batch.heads >= 0
    adj[b[kid], i[kid], batch.heads[kid]] = adj[b[kid], batch.heads[kid], i[kid]] = 1.0
    if batch.extra_edges is not None and len(batch.extra_edges):
        eb = np.repeat(np.arange(batch.n_graphs), np.diff(batch.edge_ptr))
        x, y = batch.extra_edges[:, 0], batch.extra_edges[:, 1]
        adj[eb, x, y] = adj[eb, y, x] = 1.0
    return adj


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rates", default="0.05,0.2")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_enhanced.py measures on a CUDA device; none found")
    import bench
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import gated, synth
    from ed_gated_gcn_b200.runtime import GraphedStep

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"what": "enhanced-dependency graphs on the packed path, C2 shape", **card(dev)}
    c, tree, x_host, tgt_host = bench.make_workload("C2", 0)
    rates = [float(r) for r in args.rates.split(",")]
    batches = {"tree": tree}
    for r in rates:
        batches[f"extra_{r:g}"] = synth.with_extra_edges(tree, rate=r, seed=synth.REFERENCE_SEED + 7)
    T = int(tree.lengths.max())
    res.update(n_graphs=tree.n_graphs, n_rows=tree.n_rows, max_len=T)

    def dev_inputs(b):
        d = {k: torch.from_numpy(getattr(b, k)).to(dev) for k in ("heads", "sent_ptr", "anchor")}
        if b.extra_edges is not None:
            d["extra_edges"] = torch.from_numpy(b.extra_edges).to(dev)
            d["edge_ptr"] = torch.from_numpy(b.edge_ptr).to(dev)
        return d

    def build(b, d):
        if b.extra_edges is None:
            return E.build_graph(d["heads"], d["sent_ptr"], max_len=T)
        return E.build_graph(d["heads"], d["sent_ptr"], max_len=T, extra_edges=d["extra_edges"],
                             edge_ptr=d["edge_ptr"], max_sent_nnz=exact_max_sent_nnz(b))

    # ---- 1. the CSR build, and 2. the bytes a batch moves host->device
    csr, h2d = {}, {}
    for name, b in batches.items():
        d = dev_inputs(b)
        g = build(b, d)
        want = E.build_graph(d["heads"], d["sent_ptr"], extra_edges=d.get("extra_edges"), edge_ptr=d.get("edge_ptr"))
        assert g.max_sent_nnz in (None, want.max_sent_nnz), (g.max_sent_nnz, want.max_sent_nnz)
        csr[f"build_graph_{name}_ms"] = median_ms(lambda: build(b, d), args.iters, args.warmup)
        n_extra = 0 if b.extra_edges is None else len(b.extra_edges)
        csr[f"n_extra_edges_{name}"] = n_extra
        csr[f"max_sent_nnz_{name}"] = exact_max_sent_nnz(b) if b.extra_edges is not None else 3 * T - 2
        h2d[f"packed_{name}"] = 4 * (b.n_rows + b.n_graphs + 1) + (0 if b.extra_edges is None else 8 * n_extra + 4 * (b.n_graphs + 1))
        adj = torch.from_numpy(dense_of(b, T)).to(dev)
        dg = E.graph_from_dense(adj)
        assert dg.max_sent_nnz is not None
        if name in ("tree", f"extra_{rates[-1]:g}"):
            csr[f"graph_from_dense_{name}_ms"] = median_ms(lambda: E.graph_from_dense(adj), args.iters, args.warmup)
        del adj, dg
    h2d["dense_fp32_T50"] = 4 * tree.n_graphs * T * T
    h2d["dense_fp32_T100_reference_padding"] = 4 * tree.n_graphs * 100 * 100
    res["csr_build"] = csr
    res["h2d_bytes_per_batch_graph_only"] = h2d

    # ---- 3. the captured C2 training step
    stack, dense = bench.build_model(c, dev)
    params = list(stack.parameters()) + list(dense.parameters())
    opt = E.FusedAdam(params, lr=1e-3)
    from ed_gated_gcn_b200 import ops
    cd = torch.bfloat16
    x_dev = torch.zeros(tree.n_rows, ops.row_pitch(c["D"], cd), dtype=cd, device=dev)
    x_dev[:, :c["D"]].copy_(x_host)
    x_dev.requires_grad_(True)
    tgt = tgt_host.to(dev)
    head_params = list(dense.parameters())
    seen, orig = [], gated._fused_plan

    def spy(*a):
        seen.append(orig(*a))
        return seen[-1]
    gated._fused_plan = spy
    steps = {}
    for name in ["tree"] + [f"extra_{r:g}" for r in rates]:
        b = batches[name]
        d = dev_inputs(b)

        def step():
            opt.zero_grad(set_to_none=True)
            x_dev.grad = None
            g = build(b, d)
            dist = E.tree_distance(g, d["anchor"])
            out = stack(x_dev, g, d["anchor"], dist, dense, head_params=head_params)
            loss = E.total_loss(E.cross_entropy(out.logits, tgt), out.xy, out.kl, bench.GATE_W, bench.KL_W)
            loss.backward()
            opt.step()
            return loss

        seen.clear()
        gs = GraphedStep(step)
        assert seen and all(s is not None for s in seen), f"{name}: the fused layer plan was not taken"
        ms = [median_ms(gs, args.steps, 3) for _ in range(3)]
        steps[f"{name}_ms"] = float(np.median(ms))
        steps[f"{name}_ms_repeats"] = ms
        steps[f"{name}_loss"] = float(gs().item())
        opt.zero_grad(set_to_none=True)
        del gs
        torch.cuda.synchronize()
    gated._fused_plan = orig
    res["captured_c2_step"] = steps
    res["timing"] = (f"CUDA-event medians: CSR builds over {args.iters} calls after {args.warmup} warm-up calls; "
                     f"captured steps: median of 3 medians over {args.steps} replays each")
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
