"""CPU-only checks: the C-ABI library loads and exports every symbol include/edgcn.h
declares, the ctypes table mirrors the header, the host logic (sharding, drop-in module
surface, synthetic generator) and the 2-rank gloo gradient averaging."""
import ctypes
import os
import re
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT


def _declared():
    src = open(os.path.join(ROOT, "include", "edgcn.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(edg_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from ed_gated_gcn_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "build libedgcn.so first (__graft_entry__.build())"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), n
    assert set(names) == set(_lib.SIGNATURES), set(names) ^ set(_lib.SIGNATURES)


def test_version_and_error_strings_without_gpu():
    from ed_gated_gcn_b200 import _lib
    lib = _lib.load()
    assert lib.edg_version() == 4
    assert b"aligned" in lib.edg_strerror(-2)
    assert lib.edg_strerror(0) == b"ok"


def test_prototype_arity_matches_header():
    from ed_gated_gcn_b200 import _lib
    src = open(os.path.join(ROOT, "include", "edgcn.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    for name, (_, args) in _lib.SIGNATURES.items():
        m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", src, flags=re.S)
        assert m, name
        inner = m.group(1).strip()
        n = 0 if inner in ("", "void") else len(inner.split(","))
        assert n == len(args), (name, n, len(args))


def test_no_cpu_fallback():
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200._lib import EdgError
    with pytest.raises(EdgError):
        E.GraphConvolution(4, 4)(torch.zeros(1, 3, 4), torch.eye(3)[None])
    with pytest.raises(EdgError):
        E.build_graph(torch.tensor([-1, 0]), torch.tensor([0, 2]))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "ed-gated-gcn_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dp, f)).read()
                assert "ref_oracle" not in text and "from oracle" not in text and "import oracle" not in text, f


def test_drop_in_surface():
    import ed_gated_gcn_b200 as E
    layer = E.GraphConvolution(6, 4, object())              # third positional arg `opt`, gcn.py:14
    assert layer.weight.shape == (6, 4) and layer.bias.shape == (4,)
    assert E.GraphConvolution(6, 4, None, bias=False).bias is None
    stack = E.GatedGCNStack(8, 2, 3)
    want = {"gc1.weight", "gc1.bias", "gc2.weight", "gc2.bias", "fc.0.weight", "fc.0.bias"} | \
        {f"gate{g}.{i}.{k}" for g in (1, 2) for i in (1, 3) for k in ("weight", "bias")}
    assert set(stack.state_dict()) == want                  # the keys of BertAmir55, bert_amir5.py:559-572


def test_synthetic_trees_are_trees():
    from ed_gated_gcn_b200 import synth
    for skew in (False, True):
        b = synth.make_batch(50, 1, 80, seed=1, skewed=skew)
        for h in b.heads_list():
            n = len(h)
            assert (h == -1).sum() == 1
            seen = set()
            for i in range(n):                              # every token reaches the root: no cycles
                j, steps = i, 0
                while h[j] >= 0:
                    j = h[j]; steps += 1
                    assert steps <= n
        assert (b.anchor < b.lengths).all() and (b.anchor >= 0).all()
    hub = synth.make_batch(4, 400, 512, seed=2, skewed=True)
    for h in hub.heads_list():
        assert np.bincount(h[h >= 0]).max() > len(h) // 4      # config 4: a hub of degree ~ n/2


def test_shards_are_balanced_and_disjoint():
    from ed_gated_gcn_b200 import parallel, synth
    b = synth.make_batch(4096, 5, 50, seed=3)
    b.lengths.sort()                                        # the reference sorts by length (data_utils.py:341-346)
    parts = [parallel.shard_graphs(b.lengths, 8, r) for r in range(8)]
    allidx = np.concatenate(parts)
    assert len(np.unique(allidx)) == 4096
    toks = [int(b.lengths[p].sum()) for p in parts]
    assert all(len(p) == 512 for p in parts)
    assert max(toks) - min(toks) <= 50 * 2
    sub, idx = parallel.shard_tree_batch(synth.make_batch(10, 2, 9, seed=4), 2, 1)
    assert sub.n_graphs == 5 and sub.n_rows == int(sub.lengths.sum())


WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from ed_gated_gcn_b200 import parallel, synth
from oracle import ref_oracle as O
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
batch = synth.make_batch(8, 3, 9, seed=6)
D = 8
g = torch.Generator().manual_seed(0)
w = torch.randn(D, D, generator=g); b = torch.randn(D, generator=g)
x = torch.randn(batch.n_rows, D, generator=g)
def loss_of(bt, rows, W, Bv):
    tot = 0.0
    off = 0
    for h in bt.heads_list():
        n = len(h)
        adj = torch.from_numpy(O.dense_adjacency_from_heads(h, n)).float()[None]
        y = O.gcn_layer_ref(rows[off:off + n][None], adj, W, Bv)
        tot = tot + y.max(1)[0].sum()
        off += n
    return tot / bt.n_graphs
# single-process answer
W = w.clone().requires_grad_(True); Bv = b.clone().requires_grad_(True)
loss_of(batch, x, W, Bv).backward()
# this rank's shard
sub, idx = parallel.shard_tree_batch(batch, world, rank)
rows = torch.cat([x[batch.sent_ptr[i]:batch.sent_ptr[i + 1]] for i in idx])
Wl = torch.nn.Parameter(w.clone()); Bl = torch.nn.Parameter(b.clone())
loss_of(sub, rows, Wl, Bl).backward()
red = parallel.GradientAllReducer([Wl, Bl])
red.hook([Wl.grad])          # what a backward pass does as soon as a layer's gradient exists (overlapped reduction) ...
red()                        # ... and the rest (here: the bias) after backward; then wait for everything
ok = torch.allclose(Wl.grad, W.grad, atol=1e-6) and torch.allclose(Bl.grad, Bv.grad, atol=1e-6)
# a second step must start clean (no gradient skipped because of the first step's bookkeeping)
Wl.grad = None; Bl.grad = None
loss_of(sub, rows, Wl, Bl).backward()
red()
ok = ok and torch.allclose(Wl.grad, W.grad, atol=1e-6) and torch.allclose(Bl.grad, Bv.grad, atol=1e-6)
# third variant: a backward pass hands ALL its gradients over at once (GradientAllReducer.bucket) and returns the views
# of the reduced flat buffer to autograd -- emulated here by installing the views as .grad
Wl.grad = None; Bl.grad = None
loss_of(sub, rows, Wl, Bl).backward()
gW, gB = Wl.grad, Bl.grad
keep = red.bucket([gW, None, gB])          # .grad already populated: the bucket must refuse (autograd would accumulate)
ok = ok and keep[0] is gW and keep[2] is gB
Wl.grad = None; Bl.grad = None             # inside a real backward pass nothing is installed yet
out = red.bucket([gW, None, gB])
ok = ok and out[1] is None and out[0].shape == gW.shape and out[0].data_ptr() != gW.data_ptr()
Wl.grad, Bl.grad = out[0], out[2]
red()                        # nothing left to announce: only waits (and applies the gloo scale)
ok = ok and red.n_late == 0
ok = ok and torch.allclose(Wl.grad, W.grad, atol=1e-6) and torch.allclose(Bl.grad, Bv.grad, atol=1e-6)
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 3)
'''


def test_two_rank_gloo_gradient_average_equals_single_process(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script), ROOT], env=env))
    codes = [p.wait(timeout=240) for p in procs]
    assert codes == [0, 0]


def _reference_items(batch, pieces, ori_ml=60, bert_ml=90):
    """Per-sentence item dicts shaped like the reference datasets build them (data_utils.py:362-379, 438-490)."""
    from oracle import ref_oracle as O
    items = []
    for b, h in enumerate(batch.heads_list()):
        n = len(h)
        adj = O.dense_adjacency_from_heads(h, ori_ml)
        dist = O.pad_distance(O.tree_distance_bfs(h, int(batch.anchor[b])), ori_ml, "max+1")
        items.append({"dependency_graph": adj.tolist(), "anchor_index": int(batch.anchor[b]), "sentence_length": n,
                      "dist_to_target": dist, "transform": O.wordpiece_transform_ref(pieces[b], ori_ml, bert_ml),
                      "cls_text_sep_length": sum(pieces[b]) + 2, "polarity": b % 3})
    return items


def test_packed_wire_format_from_reference_items():
    """collate_packed (SURVEY 8f N3) over reference-format items: the heads it extracts give the same CSR as
    the dense matrix, distances / segments survive, and the payload is ~16 B/token instead of ~90 KB/sentence."""
    import ed_gated_gcn_b200 as E
    from ed_gated_gcn_b200 import synth
    from oracle import ref_oracle as O
    batch = synth.make_batch(12, 1, 40, seed=21)
    rng = np.random.default_rng(5)
    pieces = [rng.integers(1, 4, size=int(n)).tolist() for n in batch.lengths]
    items = _reference_items(batch, pieces)
    pb = E.collate_packed(items)
    assert pb.n_graphs == 12 and pb.n_rows == batch.n_rows and pb.max_len == int(batch.lengths.max())
    assert np.array_equal(pb.sent_ptr.numpy(), batch.sent_ptr) and np.array_equal(pb.anchor.numpy(), batch.anchor)
    for b, h in enumerate(batch.heads_list()):
        lo, hi = batch.sent_ptr[b], batch.sent_ptr[b + 1]
        got = pb.heads[lo:hi].numpy()
        n = len(h)
        # any orientation of the same undirected tree yields the same symmetric pattern
        assert np.array_equal(O.dense_adjacency_from_heads(got, n), O.dense_adjacency_from_heads(h, n))
        assert pb.dist[lo:hi].tolist() == O.tree_distance_bfs(h, int(batch.anchor[b]))
        # segments: word i = pieces [1 + sum(pieces[:i]), +pieces[i]) of the sentence's own [CLS] .. [SEP] rows
        start = pb.seg_start[lo:hi].numpy() - int(pb.piece_ptr[b])
        assert start.tolist() == (1 + np.concatenate([[0], np.cumsum(pieces[b])[:-1]])).tolist()
        assert pb.seg_len[lo:hi].tolist() == pieces[b]
    assert int(pb.piece_ptr[-1]) == sum(sum(p) + 2 for p in pieces)
    dense_bytes = 12 * (60 * 60 * 4 + 60 * 90 * 4 + 60 * 8)
    assert pb.nbytes() < dense_bytes / 50
    with pytest.raises(ValueError):
        cyc = np.eye(4, dtype=np.int64)
        for i, j in ((0, 1), (1, 2), (2, 0)):
            cyc[i, j] = cyc[j, i] = 1
        E.heads_from_adjacency(cyc, 4)


def test_segments_from_dense_transform_host_logic():
    from ed_gated_gcn_b200 import segment
    from ed_gated_gcn_b200._lib import EdgError
    from oracle import ref_oracle as O
    t = torch.tensor([O.wordpiece_transform_ref([2, 1, 3], 5, 9), O.wordpiece_transform_ref([1], 5, 9)])
    s, n = segment.segments_from_transform(t)
    assert n.view(2, 5).tolist() == [[2, 1, 3, 0, 0], [1, 0, 0, 0, 0]]
    assert s.view(2, 5)[0, :3].tolist() == [1, 3, 4] and int(s.view(2, 5)[1, 0]) == 9 + 1
    bad = t.clone(); bad[0, 0, 5] = 0.5                       # not a contiguous run of 1/len
    with pytest.raises(EdgError):
        segment.segments_from_transform(bad)


def test_heads_from_adjacency_forest_and_singletons():
    """A forest (several components, as CoreNLP emits for fragments) and one-token sentences orient cleanly;
    the packed batch tolerates missing optional fields."""
    import ed_gated_gcn_b200 as E
    from oracle import ref_oracle as O
    heads = np.array([-1, 0, 0, -1, 3, -1], dtype=np.int32)            # three components: {0,1,2}, {3,4}, {5}
    adj = O.dense_adjacency_from_heads(heads, 9)                        # padded to 9 like the [100,100] matrices
    got = E.heads_from_adjacency(adj, 6)
    assert (got == -1).sum() == 3
    assert np.array_equal(O.dense_adjacency_from_heads(got, 6), adj[:6, :6])
    assert E.heads_from_adjacency(np.eye(4, dtype=np.int64), 1).tolist() == [-1]
    items = [{"dependency_graph": adj.tolist(), "anchor_index": 4, "sentence_length": 6},
             {"dependency_graph": np.eye(9, dtype=np.int64).tolist(), "anchor_index": 0, "sentence_length": 1}]
    pb = E.collate_packed(items)
    assert pb.dist is None and pb.seg_start is None and pb.polarity is None
    assert pb.sent_ptr.tolist() == [0, 6, 7] and pb.max_len == 6 and pb.n_rows == 7
    with pytest.raises(ValueError):
        asym = adj.copy(); asym[0, 5] = 1
        E.heads_from_adjacency(asym, 6)


def test_built_library_contains_tcgen05_and_tma_instructions():
    """No GPU needed: the SASS of the in-tree library must hold what the design claims -- tcgen05.mma (UTCHMMA),
    tcgen05.ld (LDTM), TMA tensor loads (UTMALDG) and bulk copies (UBLKCP) -- per kernel family."""
    import shutil
    from ed_gated_gcn_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    per_fn = {}
    cur = None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            per_fn[cur] = set()
        elif cur:
            for op in ("UTCHMMA", "LDTM", "UTMALDG", "UBLKCP"):
                if op in line:
                    per_fn[cur].add(op)
    def ops_of(substr):
        out = set()
        for fn, ops in per_fn.items():
            if substr in fn:
                out |= ops
        return out
    for kern in ("linear_ws_kernel", "linear_tc_kernel", "wgrad_tc_kernel", "wgrad_tall_kernel", "wgrad_tc_batch_kernel",
                 "mlp_chain_kernel"):
        assert {"UTCHMMA", "UTMALDG"} <= ops_of(kern), kern          # tensor cores fed by TMA
    for kern in ("linear_ws_kernel", "mlp_chain_kernel", "wgrad_tall_kernel"):
        assert "LDTM" in ops_of(kern), kern                          # accumulators read back from TMEM
    for kern in ("aggregate_staged_kernel", "pool_staged_kernel", "scores_staged_kernel", "head_bwd_staged_kernel"):
        assert "UBLKCP" in ops_of(kern), kern                        # windows staged by bulk async copies


def test_head_and_loss_modules_keep_the_reference_parameter_layout_and_refuse_cpu_tensors():
    """E.DenseHead is an nn.Linear(2*hidden, polarities) (bert_amir5.py:573): same state-dict keys and shapes, so a
    reference checkpoint loads; called with ONE argument it is a plain Linear (works on CPU); the two-argument form and the
    loss are CUDA kernels only and say so."""
    import torch
    import ed_gated_gcn_b200 as E
    head = E.DenseHead(600, 34)
    ref = torch.nn.Linear(600, 34)
    assert {k: tuple(v.shape) for k, v in head.state_dict().items()} == {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    head.load_state_dict(ref.state_dict())
    x = torch.randn(3, 600)
    assert torch.equal(head(x), ref(x))
    assert not head.fusable(300)                     # CPU parameters: the block would keep the torch path
    with pytest.raises(E.EdgError):
        head(torch.randn(3, 300), torch.randn(3, 300))
    with pytest.raises(E.EdgError):
        E.cross_entropy(torch.randn(3, 34), torch.zeros(3, dtype=torch.long))


def test_host_side_planning_entry_points_of_the_round_2_additions():
    """No GPU needed: pitches, shape coverage, workspace sizes and the SM budget are host arithmetic."""
    from ed_gated_gcn_b200 import _lib
    lib = _lib.load()
    assert lib.edg_split_pitch(300) == 640 and lib.edg_split_pitch(64) == 128 and lib.edg_split_pitch(65) == 256
    assert lib.edg_split_pitch(0) == 0
    # the hi+lo weight slice of the fp32-parity projection has to fit next to two activation stages
    assert lib.edg_linear_split_ok(300, 300) == 1 and lib.edg_linear_split_ok(768, 768) == 1
    assert lib.edg_linear_split_ok(300, 2000) == 0          # bias table (kMaxBias) exceeded
    assert lib.edg_linear_split_ok(8192, 300) == 0          # no N tile of 16 columns fits any more
    # three products: the hi x hi launch in short chains (more slabs) + two cross-term launches
    assert lib.edg_wgrad_split_workspace(204800, 300, 300) > 3 * 301 * 300 * 4
    assert lib.edg_wgrad_split_workspace(0, 300, 300) == 16
    assert lib.edg_dense_head_bwd_workspace(4096, 300, 34) == 128 * 34 * 601 * 4
    assert lib.edg_cross_entropy_workspace(4096) == (2 * 512 + 1) * 4
    prev = lib.edg_set_sm_budget(116)
    assert prev == 148 and lib.edg_set_sm_budget(1000) == 116 and lib.edg_set_sm_budget(148) == 148
