"""Micro-benchmark of the block's head at config-C2 size (B = 4096, D = 300, C = 34, fp32 operands):
edg_block_head_fwd / _bwd / _wgrad in their three modes -- both heads (a DenseHead in the block), fc only (the logits
of a torch logits_fn as input) and dense only (a DenseHead called on its own).

Each direction is captured as a CUDA graph over a ring of input sets larger than L2 (so every replay reads HBM, as in
the training step), replayed many times between two CUDA events.  Prints microseconds per call of each direction.

    python tools/bench_block_head.py [--reps 200] [--ring 8]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--ring", type=int, default=8, help="input sets cycled through (8 x ~30 MB > the 126 MB L2)")
    args = ap.parse_args()
    from ed_gated_gcn_b200 import ops
    B, D, C = 4096, 300, 34
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(0)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    W, bias, Wf, bf = r(C, 2 * D) * 0.05, r(C), r(C, 2 * D) * 0.05, r(C)
    scale = torch.ones(1, device=dev)
    ring = [dict(a=r(B, D), hmax=r(B, D), gate=torch.rand(B, D, device=dev, generator=g), dv=r(B, D), dc=r(B),
                 g_lg=r(B, C)) for _ in range(args.ring)]

    def both_fwd(t):
        t["pooled"], t["lg"], t["v"], t["c"] = ops.block_head_fwd(t["a"], t["a"], t["hmax"], t["gate"], W, bias, Wf, bf)

    def both_bwd(t):
        t["dlg"], _, _ = ops.block_head_bwd(t["lg"], t["a"], t["a"], False, W, Wf, bf, t["dv"], t["dc"], scale,
                                            t["g_lg"], None)

    def both_wgrad(t):
        ops.block_head_wgrad(t["lg"], t["dlg"], t["a"], t["a"], t["pooled"], t["dv"], t["dc"], scale)

    def fc_fwd(t):
        ops.block_head_fwd(t["a"], t["a"], None, None, None, None, Wf, bf, logits=t["lg"])

    def fc_bwd(t):
        ops.block_head_bwd(t["lg"], t["a"], t["a"], False, None, Wf, bf, t["dv"], t["dc"], scale, t["g_lg"], None)

    def fc_wgrad(t):
        ops.block_head_wgrad(t["lg"], None, t["a"], t["a"], None, t["dv"], t["dc"], scale)

    def dense_fwd(t):
        ops.block_head_fwd(t["a"], None, t["pooled"], None, W, bias, None, None)

    def dense_bwd(t):
        ops.block_head_bwd(None, t["a"], None, False, W, None, None, g_logits=t["g_lg"])

    def dense_wgrad(t):
        ops.block_head_wgrad(None, t["g_lg"], t["a"], None, t["pooled"])

    def time_graph(fn):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for t in ring:                  # warm-up: module load, allocator
                fn(t)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for t in ring:
                fn(t)
        graph.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            graph.replay()
        e1.record()
        torch.cuda.synchronize()
        return 1e3 * e0.elapsed_time(e1) / (args.reps * len(ring))

    for t in ring:                          # forward outputs the other modes and the backward read
        both_fwd(t)
        both_bwd(t)
    res = {}
    modes = dict(both=(both_fwd, both_bwd, both_wgrad), fc_only=(fc_fwd, fc_bwd, fc_wgrad),
                 dense_only=(dense_fwd, dense_bwd, dense_wgrad))
    for name, (fwd, bwd, wg) in modes.items():
        res[name] = dict(fwd_us=time_graph(fwd), bwd_us=time_graph(bwd), wgrad_us=time_graph(wg))
    res["device"] = torch.cuda.get_device_name()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
