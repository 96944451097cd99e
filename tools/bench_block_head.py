"""Micro-benchmark of the block's head at config-C2 size (B = 4096, D = 300, C = 34, fp32 operands): the launch chain of
edg_dense_head_* + edg_fc_head_* (forward: memset + dense head, torch gate * hmax, fc head; backward: fc head parts=1 +
its reduction, dense head parts=1; parameter gradients: both parts=2 kernels + their two reductions) against
edg_block_head_fwd / _bwd / _wgrad (1 + 1 + 2 launches).

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

    def old_fwd(t):
        t["pooled"] = t["gate"] * t["hmax"]
        t["lg"] = ops.dense_head_fwd(t["a"], t["pooled"], W, bias)
        t["v"], t["c"] = ops.fc_head_fwd(t["lg"], Wf, bf, t["a"])

    def old_bwd(t):
        d_lg, da_fc, _, _ = ops.fc_head_bwd(t["lg"], Wf, bf, t["a"], t["dv"], t["dc"], scale, parts=1)
        ops.dense_head_bwd(t["g_lg"], t["a"], t["pooled"], W, parts=1, g2=d_lg, da_add=da_fc)
        t["d_lg"] = d_lg

    def old_wgrad(t):
        ops.fc_head_bwd(t["lg"], Wf, bf, t["a"], t["dv"], t["dc"], scale, parts=2)
        ops.dense_head_bwd(t["g_lg"], t["a"], t["pooled"], W, parts=2, g2=t["d_lg"])

    def new_fwd(t):
        t["pooled"], t["lg"], t["v"], t["c"] = ops.block_head_fwd(t["a"], t["a"], t["hmax"], t["gate"], W, bias, Wf, bf)

    def new_bwd(t):
        t["dlg"], _, _ = ops.block_head_bwd(t["lg"], t["a"], t["a"], False, W, Wf, bf, t["dv"], t["dc"], scale,
                                            t["g_lg"], None)

    def new_wgrad(t):
        ops.block_head_wgrad(t["lg"], t["dlg"], t["a"], t["a"], t["pooled"], t["dv"], t["dc"], scale)

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

    res = {}
    for name, (fwd, bwd, wg) in dict(chain=(old_fwd, old_bwd, old_wgrad), block=(new_fwd, new_bwd, new_wgrad)).items():
        for t in ring:                      # forward outputs the backward reads
            fwd(t)
            bwd(t)
        res[name] = dict(fwd_us=time_graph(fwd), bwd_us=time_graph(bwd), wgrad_us=time_graph(wg))
    res["device"] = torch.cuda.get_device_name()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
