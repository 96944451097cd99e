"""Run the same step twice (fresh allocations polluted in between) and compare bit for bit."""
import os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import ed_gated_gcn_b200 as E
from ed_gated_gcn_b200 import synth
dev = "cuda:0"
def run(dtype, D, Lyr, B, lo, hi, seed, dense_head=False):
    torch.manual_seed(seed)
    batch = synth.make_batch(B, lo, hi, seed=seed)
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=5, compute_dtype=dtype).to(dev)
    dense = (E.DenseHead if dense_head else torch.nn.Linear)(2 * D, 5).to(dev)
    # E.DenseHead: the head runs on the block's own kernels (edg_block_head_*); nn.Linear: torch autograd inside the node
    logits_fn = dense if dense_head else (lambda a, p: dense(torch.cat([a, p], 1)))
    graph = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(batch.sent_ptr), device=dev)
    anchor = torch.from_numpy(batch.anchor).to(dev)
    dist = E.tree_distance(graph, anchor)
    xp = torch.randn(batch.n_rows, D)
    res = []
    for rep in range(3):
        junk = torch.full((64 << 20,), float("nan"), device=dev); del junk       # poison the allocator's free blocks
        for p in list(stack.parameters()) + list(dense.parameters()):
            p.grad = None
        x = xp.to(dev).requires_grad_(True)
        out = stack(x, graph, anchor, dist, logits_fn, head_params=list(dense.parameters()))
        loss = torch.nn.functional.cross_entropy(out.logits, (torch.arange(B) % 5).to(dev)) + 0.01 * out.xy + 0.01 * out.kl
        loss.backward()
        torch.cuda.synchronize()
        d = {"loss": loss.detach().clone(), "scores": out.scores.detach().clone(), "dx": x.grad.clone()}
        for n, p in list(stack.named_parameters()) + [("dense.w", dense.weight), ("dense.b", dense.bias)]:
            d[n] = p.grad.clone()
        res.append(d)
    bad = []
    for k in res[0]:
        for r in res[1:]:
            if not torch.equal(res[0][k], r[k]):
                nan = bool(torch.isnan(r[k]).any() or torch.isnan(res[0][k]).any())
                bad.append((k, (res[0][k].float() - r[k].float()).abs().max().item(), nan))
                break
    print(dtype, D, Lyr, B, "DenseHead" if dense_head else "torch head", "mismatches:", bad if bad else "none (bitwise identical)")
for dtype in (torch.float32, torch.bfloat16):
    for dense_head in (False, True):
        run(dtype, 300, 2, 32, 5, 50, 1, dense_head)
        run(dtype, 32, 1, 5, 2, 9, 2, dense_head)
    run(dtype, 64, 3, 9, 1, 20, 3)
    run(dtype, 128, 4, 6, 30, 90, 4)
