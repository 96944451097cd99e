"""Bring-up: clock64 timelines of CTA 0 in edg_gcn_layer (EDG_FUSED_DEBUG bit 32): epilogue thread 0, the thread that
issues the aggregation product, lane 0 of the Adj builder."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["EDG_FUSED_DEBUG"] = str(32 | int(os.environ.get("DBG", "0")))
pool = len(sys.argv) > 1 and sys.argv[1] == "pool"
import ed_gated_gcn_b200 as E
from ed_gated_gcn_b200 import ops, synth, _lib as L
dev = "cuda:0"
batch = synth.config_batch("C2")
D, B, N = 300, batch.n_graphs, batch.n_rows
graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=dev)
x = ops.alloc_rows(N, D, torch.bfloat16, dev, zero=True); x.copy_(torch.randn(N, D, device=dev))
w = ops.alloc_rows(D, D, torch.bfloat16, dev, zero=True); w.copy_(torch.randn(D, D) / D ** 0.5)
bias = torch.randn(D, device=dev)
rows = ops.fused_tile_rows(D, D)
info, n_tiles = graph.tile_plan(rows)
y = ops.alloc_rows(N, D, torch.bfloat16, dev)
hmax = torch.empty(B, D, device=dev); harg = torch.empty(B, D, dtype=torch.int32, device=dev)
ws = torch.zeros(3 * 160, dtype=torch.int64, device=dev)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
for rep in range(3):
    flush.zero_(); ws.zero_()
    L.call("edg_gcn_layer", L.ptr(x), ops.ld(x), N, D, L.ptr(w), ops.ld(w), D, L.ptr(bias), 0, L.ptr(graph.row_ptr),
           L.ptr(graph.col), L.ptr(graph.sent_ptr), L.ptr(info), L.ptr(n_tiles), rows, L.ptr(y), ops.ld(y),
           L.ptr(hmax) if pool else None, L.ptr(harg) if pool else None, D, None, None, 0, None, 0, L.ptr(ws), ws.numel() * 8,
           L.stream())
    torch.cuda.synchronize()
t = ws.cpu().view(3, 160).tolist()
t0 = min(v for r in t for v in r if v)
def show(name, row, per, labels):
    row = [v - t0 for v in row if v]
    print(name)
    for k in range(0, len(row) - per + 1, per):
        seg = row[k:k + per]
        print("  tile %2d @%7d  " % (k // per, seg[0]) + "  ".join("%s %5d" % (labels[j], seg[j + 1] - seg[j]) for j in range(per - 1)))
show("epilogue thread 0", t[0], 10, ["wait_meta", "wait_U", "phaseA", "wait_Y", "phaseC", "bar1", "phaseD", "bar2", "table"])
show("aggregation MMA issuer", t[1], 4, ["wait_adj", "wait_S", "issue"])
show("Adj builder", t[2], 5, ["wait_meta_free", "meta+wait_adj_free", "clear", "set"])
