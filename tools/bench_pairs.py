"""Grouped (sentence, trigger) pairs against the expanded batch on the all-candidates workload.

The LitBank reader makes one example per token of a sentence.  With C2's sentence lengths (U{5..50}, D = 300, L = 2,
34 classes, bf16) and every token a candidate, ``--sentences 149`` gives about 4,100 pairs, the size of a C2 batch.
Two arms run the same call, alternating:

  grouped   : x holds every sentence once, ``GatedGCNStack(..., pairs=)``
  expanded  : each sentence's rows copied once per pair, the existing per-pair path

Each arm is timed as a captured training step (forward + loss + backward in one CUDA graph) and as a ``no_grad``
forward, with CUDA events over ``--steps`` calls after ``--warmup``.  Reported: pairs/s, ms per call, host-to-device
bytes per batch (the x rows in bf16 plus the integer arrays each arm needs), and the card name and power limit read in
the same run.  Writes one JSON line to stdout and, with ``--out``, to that file.

``--dropout P`` runs both arms in train() mode with gate dropout P (the reference trainer's default is 0.25): the
grouped arm with ``pair_dropout=True`` (per-pair masked passes over the sentence rows), the expanded arm on the existing
path (masked copies of the expanded rows).  Both arms draw their masks from the same seed, so they compute the same
result.

``--fc-sigmoid`` runs BertAmir54's block in both arms (``fc_sigmoid=True``; the grouped arm with
``pair_fc_sigmoid=True``, which forms every pair's sigmoid rows inside the per-pair kernels).  ``--hidden`` sets D
(BertAmir54's LSTM output is 256 wide).

    python tools/bench_pairs.py --sentences 149 --steps 100 --warmup 10 --rounds 3 --out profiles/r04_a_bench_pairs.json
    python tools/bench_pairs.py --dropout 0.25 --out profiles/r05_a_bench_pairs_dropout.json
    python tools/bench_pairs.py --fc-sigmoid --hidden 256 --out profiles/r08_a_bench_pairs_fc_sigmoid.json
    python tools/bench_pairs.py --fc-sigmoid --hidden 256 --dropout 0.25 --out profiles/r08_b_bench_pairs_fc_sigmoid_dropout.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                 # the number is reported as unknown rather than guessed
        pl = f"unknown ({type(e).__name__})"
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sentences", type=int, default=149)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=14181)
    ap.add_argument("--dropout", type=float, default=0.0)
    ap.add_argument("--fc-sigmoid", action="store_true")
    ap.add_argument("--hidden", type=int, default=300)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    from ed_gated_gcn_b200.runtime import GraphedStep
    dev = torch.device("cuda", torch.cuda.current_device())
    D, Lyr, C = args.hidden, 2, 34
    cd = torch.bfloat16
    batch = synth.make_batch(args.sentences, 5, 50, seed=args.seed)
    pp, an = synth.candidate_pairs(batch)
    P = len(an)
    sp = batch.sent_ptr
    owner = np.repeat(np.arange(batch.n_graphs), np.diff(pp))
    rows = torch.from_numpy(np.concatenate([np.arange(sp[s], sp[s + 1]) for s in owner]))
    e_heads = np.concatenate([batch.heads[sp[s]:sp[s + 1]] for s in owner]).astype(np.int32)
    e_sp = np.zeros(P + 1, dtype=np.int32)
    e_sp[1:] = np.cumsum(batch.lengths[owner])

    torch.manual_seed(args.seed)
    stack = E.GatedGCNStack(D, n_layers=Lyr, n_classes=C, compute_dtype=cd, dropout=args.dropout,
                            pair_dropout=args.dropout > 0, fc_sigmoid=args.fc_sigmoid,
                            pair_fc_sigmoid=args.fc_sigmoid).to(dev)
    head = E.DenseHead(2 * D, C).to(dev)
    x_host = torch.randn(batch.n_rows, D, generator=torch.Generator().manual_seed(args.seed + 1)).to(cd)
    tgt = (torch.arange(P) % C).to(dev)
    max_len = int(batch.lengths.max())

    arms = {}
    # grouped: sentence rows once, pair map built on the device without a host read
    xg = x_host.to(dev).requires_grad_(True)
    gg = E.build_graph(torch.from_numpy(batch.heads), torch.from_numpy(sp), max_len=max_len, device=dev)
    pairs = E.pairs_from_ptr(gg, torch.from_numpy(pp), torch.from_numpy(an))
    ang = torch.from_numpy(an).to(dev)
    dg = E.tree_distance(gg, ang, pairs=pairs)
    arms["grouped"] = dict(x=xg, g=gg, an=ang, d=dg, pairs=pairs,
                           h2d=batch.n_rows * D * 2 + 4 * (batch.n_rows + (batch.n_graphs + 1) * 2 + P) + 8 * P)
    # expanded: today's path, each sentence copied per pair
    xe = x_host[rows].to(dev).requires_grad_(True)
    ge = E.build_graph(torch.from_numpy(e_heads), torch.from_numpy(e_sp), max_len=max_len, device=dev)
    ane = torch.from_numpy(an).to(dev)
    de = E.tree_distance(ge, ane)
    arms["expanded"] = dict(x=xe, g=ge, an=ane, d=de, pairs=None,
                            h2d=len(rows) * D * 2 + 4 * (len(rows) + (P + 1) + P) + 8 * P)

    def train_step(a):
        def fn():
            for p in list(stack.parameters()) + list(head.parameters()):
                p.grad = None
            a["x"].grad = None
            out = stack(a["x"], a["g"], a["an"], a["d"], head, pairs=a["pairs"])
            loss = E.total_loss(E.cross_entropy(out.logits, tgt), out.xy, out.kl, 0.01, 0.01)
            loss.backward()
            return loss
        return fn

    def fwd_step(a):
        def fn():
            with torch.no_grad():
                return stack(a["x"], a["g"], a["an"], a["d"], head, pairs=a["pairs"]).logits
        return fn

    # same results: the grouped arm must reproduce the expanded one
    torch.manual_seed(args.seed + 2)                   # the same dropout seed for both arms
    lg = fwd_step(arms["grouped"])().float()
    torch.manual_seed(args.seed + 2)
    le = fwd_step(arms["expanded"])().float()
    max_rel_logits = float((lg - le).abs().max() / le.abs().max())

    runs = {name: dict(train=GraphedStep(train_step(a)), fwd=GraphedStep(fwd_step(a))) for name, a in arms.items()}

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

    ms = {name: {"train": [], "fwd": []} for name in arms}
    for _ in range(args.rounds):                       # alternate the arms inside one process
        for name in arms:
            for kind in ("train", "fwd"):
                ms[name][kind].append(timed(runs[name][kind]))
    name, pl = card()
    res = {"tool": "bench_pairs", "gpu": name, "power_limit": pl, "sentences": batch.n_graphs, "pairs": P,
           "sentence_rows": batch.n_rows, "expanded_rows": int(len(rows)), "D": D, "L": Lyr, "dtype": "bf16",
           "dropout": args.dropout, "fc_sigmoid": args.fc_sigmoid,
           "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds, "max_rel_logits_grouped_vs_expanded":
           max_rel_logits, "arms": {}}
    for n in arms:
        tr, fw = min(ms[n]["train"]), min(ms[n]["fwd"])
        res["arms"][n] = {"train_ms": ms[n]["train"], "fwd_ms": ms[n]["fwd"], "train_pairs_per_s": P / (tr * 1e-3),
                          "fwd_pairs_per_s": P / (fw * 1e-3), "h2d_bytes_per_batch": int(arms[n]["h2d"])}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
