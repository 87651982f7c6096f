#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/*.npz by executing the REAL
reference modules from /root/reference (read-only) in THIS container.

DGL is absent here, so `dgl_stub.py` supplies the few DGL objects the hot path
touches (documented [M] semantics); every other line that runs is the
reference's own: gcc.contrastive.{memory_moco,criterions}, gcc.utils.misc,
gcc.models.{graph_encoder,gin}, gcc.datasets.{graph_dataset,data_util} and
train.py's train_moco / moment_update / clip_grad_norm / train_finetune / test_finetune.

Run:  python tests/golden/make_golden.py          (needs /root/reference)
The fixtures are committed; the GPU box never needs /root/reference.
"""
import argparse
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
REF = os.environ.get("GCC_REFERENCE", "/root/reference")

import dgl_stub  # noqa: E402

dgl_stub.install()
sys.path.insert(0, REF)

from oracle import rwr as orwr  # noqa: E402
from gcc_b200.datasets import synthetic  # noqa: E402

import gcc.contrastive.criterions as ref_crit  # noqa: E402
import gcc.contrastive.memory_moco as ref_moco  # noqa: E402
import gcc.datasets.data_util as ref_du  # noqa: E402
import gcc.datasets.graph_dataset as ref_gd  # noqa: E402
import gcc.models.graph_encoder as ref_ge  # noqa: E402
import gcc.utils.misc as ref_misc  # noqa: E402

KEY = 0x5EED5EED
PART_BYTES = 900_000        # no fixture file may exceed 1 MB


def save(name, **arrays):
    """tests/golden/<name>.npz; a fixture holding more than PART_BYTES of arrays is written as parts
    <name>.0.npz, <name>.1.npz, ... in key order (the `golden` fixture of tests/conftest.py merges them)."""
    parts, size = [{}], 0
    for k, v in arrays.items():
        if parts[-1] and size + v.nbytes > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = v
        size += v.nbytes
    stem = os.path.join(HERE, name[:-len(".npz")])
    paths = [stem + ".npz"] if len(parts) == 1 else ["%s.%d.npz" % (stem, i) for i in range(len(parts))]
    for path, part in zip(paths, parts):
        np.savez_compressed(path, **part)
        print("wrote", path, "(%d arrays)" % len(part))


# ----------------------------------------------------------------------------- #
def golden_moco():
    """MemoryMoCo.forward + NCE losses, incl. wrap-around enqueue."""
    torch.manual_seed(1)
    d, K, B, T = 8, 20, 6, 0.07
    m = ref_moco.MemoryMoCo(d, None, K, T, use_softmax=True)
    mem0 = m.memory.clone().numpy()
    out = {}
    out["memory0"] = mem0
    idx = [m.index]
    for step in range(5):                       # 5 * 6 = 30 > K = 20 -> wraps
        q = torch.nn.functional.normalize(torch.randn(B, d), dim=1).requires_grad_(True)
        k = torch.nn.functional.normalize(torch.randn(B, d), dim=1)
        o = m(q, k)
        loss = ref_crit.NCESoftmaxLoss()(o)
        loss_ns = ref_crit.NCESoftmaxLossNS()(o[:, :B])
        (dq,) = torch.autograd.grad(loss, q, retain_graph=True)
        out["q%d" % step] = q.detach().numpy()
        out["k%d" % step] = k.numpy()
        out["out%d" % step] = o.detach().numpy()
        out["loss%d" % step] = loss.detach().numpy()
        out["loss_ns%d" % step] = loss_ns.detach().numpy()
        out["dq%d" % step] = dq.numpy()
        out["memory%d" % (step + 1)] = m.memory.clone().numpy()
        idx.append(m.index)
    out["index"] = np.array(idx)
    out["T"] = np.array(T)
    out["state_keys"] = np.array(sorted(m.state_dict().keys()))
    save("moco_golden.npz", **out)


def golden_misc():
    xs = np.linspace(0, 1.2, 25)
    save("misc_golden.npz", x=xs,
         warm01=np.array([ref_misc.warmup_linear(float(x), 0.1) for x in xs]),
         warm_default=np.array([ref_misc.warmup_linear(float(x)) for x in xs]))


# ----------------------------------------------------------------------------- #
def _simple_spectrum(lap, k, gap=1e-3):
    w = np.linalg.eigvalsh(lap)
    top = w[-(k + 1):] if len(w) > k else w
    return np.min(np.diff(top)) > gap if len(top) > 1 else True


def golden_posenc():
    """_add_undirected_graph_positional_embedding on graphs whose wanted
    spectrum is simple, so the reference's answer is unique up to column sign."""
    from oracle import posenc as opos
    cases, out = [], {}
    graphs = [synthetic.path_graph(2), synthetic.path_graph(3), synthetic.path_graph(5),
              synthetic.path_graph(12), synthetic.path_graph(40),
              synthetic.triangle_tail(3), synthetic.triangle_tail(7)]
    rng = np.random.default_rng(3)
    tries = 0
    while len(graphs) < 13 and tries < 400:    # random connected graphs, simple spectrum
        tries += 1
        n = int(rng.integers(6, 30))
        g = synthetic.from_pairs(rng.integers(0, n, 3 * n), rng.integers(0, n, 3 * n), n, "rnd")
        if g.num_nodes < 5:
            continue
        lap = opos.normalized_adjacency(g.indptr, g.indices, g.num_nodes).toarray()
        k = min(g.num_nodes - 2, 32)
        if _simple_spectrum(lap, k):
            graphs.append(g)
    for ci, g in enumerate(graphs):
        sg = dgl_stub.StubGraph.from_csr(g.indptr, g.indices)
        np.random.seed(100 + ci)               # the reference draws v0 from np.random
        sg = ref_du._add_undirected_graph_positional_embedding(sg, 32)
        out["indptr%d" % ci] = g.indptr
        out["indices%d" % ci] = g.indices
        out["pos%d" % ci] = sg.ndata["pos_undirected"].numpy()
        lap = opos.normalized_adjacency(g.indptr, g.indices, g.num_nodes).toarray()
        k = min(g.num_nodes - 2, 32)
        out["simple%d" % ci] = np.array(bool(k <= 0 or _simple_spectrum(lap, k)))
        cases.append(g.name)
    out["num_cases"] = np.array(len(graphs))
    save("posenc_golden.npz", **out)


# ----------------------------------------------------------------------------- #
class _Ctx:
    sample = 0


def _bind_rwr(graph_csr, rw_key):
    """dgl.contrib.sampling.random_walk_with_restart -> oracle pure-Python walk.
    seeds=[s, s]: position in the seeds list is the view index."""
    indptr, indices = graph_csr

    def impl(g, seeds, restart_prob, max_nodes_per_seed):
        rt = orwr.restart_threshold(restart_prob)
        res = []
        for view, s in enumerate(seeds):
            traces = orwr.rwr_traces_py(indptr, indices, rw_key, _Ctx.sample, view, int(s),
                                        int(max_nodes_per_seed), rt)
            res.append([torch.tensor(t, dtype=torch.long) for t in traces])
        return res

    dgl_stub._rwr_impl = impl
    ref_gd.dgl.contrib.sampling.random_walk_with_restart = dgl_stub.random_walk_with_restart


def golden_dataset():
    """LoadBalanceGraphDataset.__getitem__ (budget, RWR call, node order,
    induction, seed one-hot) and batcher(), reference code, stub graph."""
    g = synthetic.erdos_renyi(300, 1200, seed=5)
    _bind_rwr((g.indptr, g.indices), KEY)
    ds = object.__new__(ref_gd.LoadBalanceGraphDataset)   # skip file loading in __init__
    ds.rw_hops, ds.restart_prob, ds.positional_embedding_size = 64, 0.8, 32
    ds.step_dist, ds.aug, ds.graph_transform, ds.num_neighbors = [1.0, 0.0, 0.0], "rwr", None, 5
    ds.graphs = [dgl_stub.StubGraph.from_csr(g.indptr, g.indices)]
    ds.length = g.num_nodes
    seeds = [0, 7, 150, 298, 42, 42]
    out = dict(indptr=g.indptr, indices=g.indices, seeds=np.array(seeds),
               key=np.array(KEY, dtype=np.uint64), rw_hops=np.array(64),
               restart_prob=np.array(0.8))
    pairs = []
    for i, s in enumerate(seeds):
        _Ctx.sample = i
        np.random.seed(7 + i)
        gq, gk = ds.__getitem__(s)
        pairs.append((gq, gk))
        for view, sg in enumerate((gq, gk)):
            sp, si = sg.batched_csr()
            out["subv_%d_%d" % (i, view)] = sg.parent_nid
            out["indptr_%d_%d" % (i, view)] = sp
            out["indices_%d_%d" % (i, view)] = si
            out["seedflag_%d_%d" % (i, view)] = sg.ndata["seed"].numpy()
            out["pos_%d_%d" % (i, view)] = sg.ndata["pos_undirected"].numpy()
    bq, bk = ref_du.batcher()(pairs)
    for name, bg in (("q", bq), ("k", bk)):
        sp, si = bg.batched_csr()
        out["batch_%s_indptr" % name] = sp
        out["batch_%s_indices" % name] = si
        out["batch_%s_num_nodes" % name] = np.array(bg.batch_num_nodes)
        out["batch_%s_seed" % name] = bg.ndata["seed"].numpy()
    # budgets for a degree sweep, straight from the reference formula inside
    # __getitem__ (graph_dataset.py:113-124): observed through max_nodes_per_seed
    budgets = []

    def spy(gg, seeds, restart_prob, max_nodes_per_seed):
        budgets.append(int(max_nodes_per_seed))
        raise StopIteration

    ref_gd.dgl.contrib.sampling.random_walk_with_restart = spy
    degs = [1, 2, 5, 17, 100, 400, 1000, 4296, 20000]
    for d in degs:
        star = synthetic.star_graph(d)
        ds.graphs = [dgl_stub.StubGraph.from_csr(star.indptr, star.indices)]
        for rw_hops, rp in ((256, 0.8), (64, 0.5)):
            ds.rw_hops, ds.restart_prob = rw_hops, rp
            try:
                ds.__getitem__(0)
            except StopIteration:
                pass
    out["budget_degs"] = np.array(degs)
    out["budgets"] = np.array(budgets).reshape(len(degs), 2)
    save("dataset_golden.npz", **out)


# ----------------------------------------------------------------------------- #
class _MaskDrop(torch.nn.Module):
    """Replaces nn.Dropout(0.5) inside the reference model so the q-branch mask
    is the repo's Philox mask spec instead of torch's RNG (not reproducible)."""

    def __init__(self, key, hidden):
        super().__init__()
        self.key, self.hidden, self.step, self.layer = key, hidden, 0, 0
        self.enabled = True

    def forward(self, x):
        if not (self.training and self.enabled):
            return x
        keep = orwr.dropout_mask(self.key, self.step, self.layer, x.numel(), 0.5)
        self.layer += 1
        return x * torch.from_numpy(keep.reshape(x.shape)).to(x.dtype) * 2.0


def _make_batches(num_steps, B, rw_hops, g, cdf, bt, rt):
    from oracle import posenc as opos
    steps = []
    for st in range(num_steps):
        views = [[], []]
        for i in range(B):
            sid = st * B + i
            seed = int(orwr.draw_seeds(cdf, KEY, [sid])[0])
            deg = int(g.indptr[seed + 1] - g.indptr[seed])
            for view in (0, 1):
                r = orwr.rwr_subgraph(g.indptr, g.indices, KEY, sid, view, seed, int(bt[deg]), rt)
                sg = dgl_stub.StubGraph.from_csr(r["indptr"], r["indices"])
                sg.ndata["pos_undirected"] = torch.from_numpy(
                    opos.posenc_exact(r["indptr"], r["indices"], r["n"], 32))
                sd = torch.zeros(r["n"], dtype=torch.long)
                sd[0] = 1
                sg.ndata["seed"] = sd
                views[view].append(sg)
        steps.append((dgl_stub.batch(views[0]), dgl_stub.batch(views[1])))
    return steps


def golden_train(tag, num_layer, hidden, B, K, moco, num_steps=3):
    """train.py:train_moco (reference code) for a few steps on fixed batches."""
    import train as ref_train
    torch.manual_seed(11)
    g = synthetic.erdos_renyi(400, 1600, seed=9)
    cdf = orwr.seed_cdf(g.indptr)
    bt = orwr.budget_table(int(np.diff(g.indptr).max()), 48, 0.8)
    rt = orwr.restart_threshold(0.8)
    batches = _make_batches(num_steps, B, 48, g, cdf, bt, rt)

    def mk():
        return ref_ge.GraphEncoder(positional_embedding_size=32, max_node_freq=16,
                                   max_edge_freq=16, max_degree=512, freq_embedding_size=16,
                                   degree_embedding_size=16, output_dim=hidden,
                                   node_hidden_dim=hidden, edge_hidden_dim=hidden,
                                   num_layers=num_layer, num_step_set2set=6,
                                   num_layer_set2set=3, norm=True, gnn_model="gin",
                                   degree_input=True)

    model, model_ema = mk(), mk()
    drop = _MaskDrop(KEY, hidden)
    model.gnn.drop = drop
    ref_train.moment_update(model, model_ema, 0)
    contrast = ref_moco.MemoryMoCo(hidden, None, K, 0.07, use_softmax=True)
    criterion = ref_crit.NCESoftmaxLoss() if moco else ref_crit.NCESoftmaxLossNS()
    optimizer = torch.optim.Adam(model.parameters(), lr=0.005, betas=(0.9, 0.999),
                                 weight_decay=1e-5)
    opt = types.SimpleNamespace(batch_size=B, gpu="cpu", moco=moco, clip_norm=1.0,
                                learning_rate=0.005, epochs=2, alpha=0.999, print_freq=1000,
                                tb_freq=1000, nce_t=0.07, hidden_size=hidden)
    out = {"num_steps": np.array(num_steps), "B": np.array(B), "K": np.array(K),
           "hidden": np.array(hidden), "num_layer": np.array(num_layer),
           "moco": np.array(moco), "key": np.array(KEY, dtype=np.uint64)}
    for k_, v in model.state_dict().items():
        out["init/" + k_] = v.numpy().copy()
    out["init_memory"] = contrast.memory.numpy().copy()
    out["param_order"] = np.array([n for n, _ in model.named_parameters()])
    losses, gnorms = [], []
    for st, (bq, bk) in enumerate(batches):
        for name, bg in (("q", bq), ("k", bk)):
            sp, si = bg.batched_csr()
            out["s%d_%s_indptr" % (st, name)] = sp
            out["s%d_%s_indices" % (st, name)] = si
            out["s%d_%s_num_nodes" % (st, name)] = np.array(bg.batch_num_nodes)
            out["s%d_%s_pos" % (st, name)] = bg.ndata["pos_undirected"].numpy()
            out["s%d_%s_seed" % (st, name)] = bg.ndata["seed"].numpy()

        drop.step, drop.layer = st, 0   # q view uses mask layers 0..L-1, (E2E) k view L..2L-1
        sw = types.SimpleNamespace(add_scalar=lambda *a, **k: None)

        class _OneStep:
            dataset = types.SimpleNamespace(total=num_steps * B)

            def __iter__(self_inner):
                return iter([(bq, bk)])

        # the reference computes global_step = epoch * n_batch + idx (train.py:411) with
        # n_batch = total // batch_size = num_steps and idx = 0 for a 1-item loader, so
        # epoch = st / num_steps makes global_step == st.
        loss = ref_train.train_moco(st / float(num_steps), _OneStep(), model, model_ema,
                                    contrast, criterion, optimizer, sw, opt)
        losses.append(loss)
        gn = torch.sqrt(sum((p.grad.detach() ** 2).sum() for p in model.parameters()
                            if p.grad is not None))
        gnorms.append(float(gn))
        for k_, v in model.state_dict().items():
            out["s%d_model/%s" % (st, k_)] = v.numpy().copy()
        if st == num_steps - 1:
            for k_, v in model_ema.state_dict().items():
                out["s%d_ema/%s" % (st, k_)] = v.numpy().copy()
        out["s%d_memory" % st] = contrast.memory.numpy().copy()
        for n_, p in model.named_parameters():
            if p.grad is not None:
                out["s%d_grad/%s" % (st, n_)] = p.grad.numpy().copy()
    out["losses"] = np.array(losses)
    out["post_clip_gnorms"] = np.array(gnorms)
    out["final_index"] = np.array(contrast.index)
    save("train_%s_golden.npz" % tag, **out)


def golden_finetune(num_layer=3, hidden=32, B=8, num_classes=3):
    """train.py:train_finetune / test_finetune (reference code) on fixed labeled batches: two ego-net batches
    (NodeClassificationDatasetLabeled items: seed = row 0), one whole-graph batch built by the reference's
    _rwr_trace_to_dgl_graph(entire_graph=True) (GraphClassificationDatasetLabeled items: the seed flag sits on
    the max-degree node, positional features from the reference's own eigsh call), then one validation batch."""
    import train as ref_train
    from oracle import posenc as opos
    torch.manual_seed(23)
    np.random.seed(23)
    g = synthetic.erdos_renyi(300, 1200, seed=4)
    rt = orwr.restart_threshold(0.8)

    def ego_batch(first_sid, budget=24):
        graphs = []
        for i in range(B):
            sid = first_sid + i
            seed = (sid * 37 + 11) % g.num_nodes
            r = orwr.rwr_subgraph(g.indptr, g.indices, KEY, sid, 0, seed, budget, rt)
            sg = dgl_stub.StubGraph.from_csr(r["indptr"], r["indices"])
            sg.ndata["pos_undirected"] = torch.from_numpy(opos.posenc_exact(r["indptr"], r["indices"], r["n"], 32))
            sd = torch.zeros(r["n"], dtype=torch.long)
            sd[0] = 1
            sg.ndata["seed"] = sd
            graphs.append(sg)
        return dgl_stub.batch(graphs)

    def whole_batch(seed0):
        graphs = []
        for i in range(B):
            wg = synthetic.erdos_renyi(12 + 3 * i, 30 + 9 * i, seed=seed0 + i)
            parent = dgl_stub.StubGraph.from_csr(wg.indptr, wg.indices)
            node_idx = int(parent.in_degrees().argmax())             # graph_dataset.py:361 (out == in: symmetric)
            trace = [torch.tensor([node_idx])]
            sg = ref_du._rwr_trace_to_dgl_graph(g=parent, seed=node_idx, trace=trace,
                                                positional_embedding_size=32, entire_graph=True)
            graphs.append(sg)
        return dgl_stub.batch(graphs)

    batches = [ego_batch(0), ego_batch(100), whole_batch(50)]
    valid = ego_batch(200)
    ys = [torch.from_numpy(np.random.randint(0, num_classes, size=B)).long() for _ in range(4)]

    model = ref_ge.GraphEncoder(positional_embedding_size=32, max_node_freq=16, max_edge_freq=16, max_degree=512,
                                freq_embedding_size=16, degree_embedding_size=16, output_dim=hidden,
                                node_hidden_dim=hidden, edge_hidden_dim=hidden, num_layers=num_layer,
                                num_step_set2set=6, num_layer_set2set=3, norm=True, gnn_model="gin",
                                degree_input=True)
    drop = _MaskDrop(KEY, hidden)
    model.gnn.drop = drop
    output_layer = torch.nn.Linear(hidden, num_classes)
    criterion = torch.nn.CrossEntropyLoss()
    optimizer = torch.optim.Adam(model.parameters(), lr=0.005, betas=(0.9, 0.999), weight_decay=1e-5)
    out_opt = torch.optim.Adam(output_layer.parameters(), lr=0.005, betas=(0.9, 0.999), weight_decay=1e-5)
    opt = types.SimpleNamespace(gpu="cpu", hidden_size=hidden, learning_rate=0.005, epochs=6, print_freq=1000,
                                tb_freq=1000)
    sw = types.SimpleNamespace(add_scalar=lambda *a, **k: None)
    out = {"num_steps": np.array(len(batches)), "B": np.array(B), "hidden": np.array(hidden),
           "num_layer": np.array(num_layer), "num_classes": np.array(num_classes),
           "key": np.array(KEY, dtype=np.uint64), "epochs": np.array(opt.epochs)}
    for k_, v in model.state_dict().items():
        out["init/" + k_] = v.numpy().copy()
    out["init_out/weight"] = output_layer.weight.detach().numpy().copy()
    out["init_out/bias"] = output_layer.bias.detach().numpy().copy()

    def dump(prefix, bg, y):
        sp, si = bg.batched_csr()
        out[prefix + "_indptr"], out[prefix + "_indices"] = sp, si
        out[prefix + "_num_nodes"] = np.array(bg.batch_num_nodes)
        out[prefix + "_pos"] = bg.ndata["pos_undirected"].numpy()
        out[prefix + "_seed"] = bg.ndata["seed"].numpy()
        out[prefix + "_y"] = y.numpy()

    losses, f1s = [], []
    for st, (bg, y) in enumerate(zip(batches, ys)):
        dump("s%d" % st, bg, y)
        drop.step, drop.layer = st, 0
        # n_batch = len(loader) = 1, idx = 0: global_step = epoch * n_batch + idx = st  (train.py:231)
        loss, f1 = ref_train.train_finetune(st, [(bg, y)], model, output_layer, criterion, optimizer, out_opt, sw, opt)
        losses.append(loss)
        f1s.append(f1)
        for k_, v in model.state_dict().items():
            out["s%d_model/%s" % (st, k_)] = v.numpy().copy()
        out["s%d_out/weight" % st] = output_layer.weight.detach().numpy().copy()
        out["s%d_out/bias" % st] = output_layer.bias.detach().numpy().copy()
        for n_, p in model.named_parameters():
            if p.grad is not None:
                out["s%d_grad/%s" % (st, n_)] = p.grad.numpy().copy()
    dump("valid", valid, ys[3])
    vloss, vf1 = ref_train.test_finetune(len(batches), [(valid, ys[3])], model, output_layer, criterion, sw, opt)
    with torch.no_grad():
        out["valid_logits"] = output_layer(model(valid)).numpy().copy()
    out["losses"], out["f1"] = np.array(losses), np.array(f1s)
    out["valid_loss"], out["valid_f1"] = np.array(vloss), np.array(vf1)
    save("train_finetune_golden.npz", **out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    todo = a.only.split(",") if a.only else ["moco", "misc", "posenc", "dataset", "train", "finetune"]
    if "moco" in todo:
        golden_moco()
    if "misc" in todo:
        golden_misc()
    if "posenc" in todo:
        golden_posenc()
    if "dataset" in todo:
        golden_dataset()
    if "train" in todo:
        golden_train("moco", num_layer=5, hidden=64, B=8, K=32, moco=True)
        golden_train("e2e", num_layer=2, hidden=32, B=8, K=32, moco=False)
    if "finetune" in todo:
        golden_finetune()


if __name__ == "__main__":
    main()
