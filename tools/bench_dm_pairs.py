"""BertDM's tail on grouped (sentence, trigger) pairs against the expanded batch, on the all-candidates workload.

The LitBank reader makes one example per token of a sentence.  With C2's sentence lengths (U{5..50}), every token a
candidate and ``--sentences 149`` (about 4,200 pairs), BertDM's word rows (D = 768, bertdm.py:190, bf16) enter the
tail of bertdm.py:174-193 -- left/right pooling around the trigger, the trigger row, ``self.dense`` -- in two arms that
compute the same thing, alternating:

  grouped   : the word rows hold every sentence once; ``lr_pool(..., pairs=)`` + trigger rows + cat + head
  expanded  : each sentence's rows copied once per pair (the copy is part of the step), then the per-sentence
              ``lr_pool`` + trigger-row gather + cat + head

The head is a torch ``nn.Linear(3D, 34)`` in fp32 in both arms, followed by cross-entropy.  Each arm is timed as a
captured forward + backward (gradient down to the word rows), as a captured ``no_grad`` forward, and with the pooling
kernels alone (``pool_fwd_ms``: the forward; ``pool_fwd_bwd_ms``: forward + backward of the pool on the arm's own rows),
with CUDA events over ``--steps`` replays after ``--warmup``, ``--rounds`` times.  Reported: ms per call for every
round, pairs/s from the best round, host-to-device bytes per batch if the arm's rows (bf16) and integer arrays were
shipped from the host, and the card name and power limit read in the same run.  One JSON line to stdout and, with
``--out``, to that file.

    python tools/bench_dm_pairs.py --sentences 149 --steps 200 --warmup 20 --rounds 5 --out profiles/r07_a_bench_dm_pairs.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sentences", type=int, default=149)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=14181)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    from ed_gated_gcn_b200.runtime import GraphedStep
    from bench_pairs import card
    dev = torch.device("cuda", torch.cuda.current_device())
    D, C = 768, 34
    cd = torch.bfloat16
    batch = synth.make_batch(args.sentences, 5, 50, seed=args.seed)
    pp, an = synth.candidate_pairs(batch)
    P, S, N = len(an), batch.n_graphs, batch.n_rows
    sp = batch.sent_ptr
    owner = np.repeat(np.arange(S), np.diff(pp))
    rows = torch.from_numpy(np.concatenate([np.arange(sp[s], sp[s + 1]) for s in owner])).to(dev)
    e_sp = np.zeros(P + 1, dtype=np.int32)
    e_sp[1:] = np.cumsum(batch.lengths[owner])
    max_len = int(batch.lengths.max())

    torch.manual_seed(args.seed)
    head = torch.nn.Linear(3 * D, C).to(dev)
    words = torch.randn(N, D, generator=torch.Generator().manual_seed(args.seed + 1)).to(cd).to(dev).requires_grad_(True)
    tgt = (torch.arange(P) % C).to(dev)
    gg = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(sp), max_len=max_len, device=dev)
    pairs = E.pairs_from_ptr(gg, torch.from_numpy(pp), torch.from_numpy(an))
    trig_g = (pairs.pair_start + pairs.anchor).long()
    e_heads = np.concatenate([batch.heads[sp[s]:sp[s + 1]] for s in owner]).astype(np.int32)
    ge = E.build_graph(torch.from_numpy(e_heads), torch.from_numpy(e_sp), max_len=max_len, device=dev)
    ane = torch.from_numpy(an).to(dev)
    trig_e = (ge.sent_ptr[:-1] + ane).long()

    def grouped():
        pooled = E.lr_pool(words, gg, pairs.anchor, pairs=pairs)
        return head(torch.cat([words[trig_g].float(), pooled], 1))

    def expanded():
        xe = words[rows]                                   # each sentence's rows once per pair
        pooled = E.lr_pool(xe, ge, ane)
        return head(torch.cat([xe[trig_e].float(), pooled], 1))

    # the two arms compute the same dense input (bit for bit) and the same word-row gradient up to summation order
    with torch.no_grad():
        lg, le = grouped(), expanded()
    same_logits = bool(torch.equal(lg, le))
    grads = []
    for fn in (grouped, expanded):
        words.grad = None
        torch.nn.functional.cross_entropy(fn(), tgt).backward()
        grads.append(words.grad.float().clone())
    max_rel_dwords = float((grads[0] - grads[1]).abs().max() / grads[1].abs().max())

    def train(fn):
        def step():
            for p in head.parameters():
                p.grad = None
            words.grad = None
            loss = torch.nn.functional.cross_entropy(fn(), tgt)
            loss.backward()
            return loss
        return step

    def fwd(fn):
        def step():
            with torch.no_grad():
                return fn()
        return step

    # the pooling kernels alone, each arm on its own rows (the expanded rows copied once, outside the timing)
    xe_static = words.detach()[rows].clone().requires_grad_(True)
    xg_static = words.detach().clone().requires_grad_(True)
    probe = torch.randn(P, 2 * D, generator=torch.Generator().manual_seed(args.seed + 2)).to(dev)
    pool_fns = {"grouped": lambda: E.lr_pool(xg_static, gg, pairs.anchor, pairs=pairs),
                "expanded": lambda: E.lr_pool(xe_static, ge, ane)}

    def pool_fwd_bwd(fn, x):
        def step():
            x.grad = None
            out = fn()
            out.backward(probe)
            return out
        return step

    runs = {"grouped": dict(train=train(grouped), fwd=fwd(grouped), pool_fwd=fwd(pool_fns["grouped"]),
                            pool_fwd_bwd=pool_fwd_bwd(pool_fns["grouped"], xg_static)),
            "expanded": dict(train=train(expanded), fwd=fwd(expanded), pool_fwd=fwd(pool_fns["expanded"]),
                             pool_fwd_bwd=pool_fwd_bwd(pool_fns["expanded"], xe_static))}
    graphs = {a: {k: GraphedStep(f) for k, f in r.items()} for a, r in runs.items()}

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    kinds = ("train", "fwd", "pool_fwd", "pool_fwd_bwd")
    ms = {a: {k: [] for k in kinds} for a in graphs}
    for _ in range(args.rounds):                         # alternate the arms inside one process
        for a in graphs:
            for k in kinds:
                ms[a][k].append(timed(graphs[a][k]))
    name, pl = card()
    n_exp = int(rows.numel())
    h2d = {"grouped": N * D * 2 + 4 * (2 * (S + 1) + P) + 8 * P,
           "expanded": n_exp * D * 2 + 4 * ((P + 1) + P) + 8 * P}
    res = {"tool": "bench_dm_pairs", "gpu": name, "power_limit": pl, "sentences": S, "pairs": P, "sentence_rows": N,
           "expanded_rows": n_exp, "D": D, "dtype": "bf16", "head": "torch nn.Linear(3D, 34) fp32 + cross_entropy",
           "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
           "logits_grouped_equal_expanded": same_logits, "max_rel_dwords_grouped_vs_expanded": max_rel_dwords, "arms": {}}
    for a in graphs:
        best = {k: min(v) for k, v in ms[a].items()}
        res["arms"][a] = {**{f"{k}_ms": v for k, v in ms[a].items()},
                          "train_pairs_per_s": P / (best["train"] * 1e-3), "fwd_pairs_per_s": P / (best["fwd"] * 1e-3),
                          "h2d_bytes_per_batch": int(h2d[a])}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
