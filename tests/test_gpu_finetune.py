"""GPU: the finetune path (SURVEY.md section 8 row N4) -- train.py:train_finetune / test_finetune through the
device kernels against tests/golden/train_finetune_golden.*.npz (produced by the REAL reference train_finetune),
and the labeled datasets (ego-net and whole-graph batches) against the CPU oracle."""
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _encoder(H, L):
    from gcc_b200.models import GraphEncoder
    return GraphEncoder(positional_embedding_size=32, max_node_freq=16, max_edge_freq=16, max_degree=512,
                        freq_embedding_size=16, degree_embedding_size=16, output_dim=H, node_hidden_dim=H,
                        edge_hidden_dim=H, num_layers=L, num_step_set2set=6, num_layer_set2set=3, norm=True,
                        gnn_model="gin", degree_input=True)


def _fixture_batch(z, prefix):
    """Fixture batch -> BatchBuffers (view 0).  A graph whose seed flag is not on row 0 (the reference's
    entire_graph items) is relabelled by the PRODUCT's seed_first, the fixture's positional rows follow."""
    from gcc_b200.datasets.graph_dataset import BatchBuffers
    from gcc_b200.datasets.labeled import fill_whole_graphs, seed_first
    indptr, indices, nn = z[prefix + "_indptr"], z[prefix + "_indices"], z[prefix + "_num_nodes"]
    seed, pos = z[prefix + "_seed"], z[prefix + "_pos"]
    graphs, rows, a = [], [], 0
    for n in nn:
        ip = indptr[a:a + n + 1]
        loc_ip, loc_ix = (ip - ip[0]).astype(np.int64), (indices[ip[0]:ip[-1]] - a).astype(np.int32)
        s = int(np.flatnonzero(seed[a:a + n])[0])
        assert seed[a:a + n].sum() == 1
        new_ip, new_ix, perm = seed_first(loc_ip, loc_ix, s)
        graphs.append((new_ip, new_ix))
        rows.append(a + perm)
        a += n
    buf = BatchBuffers(len(nn), int(a) + 8, len(indices) + 8, 32, 64, "cuda")
    fill_whole_graphs(buf, graphs, view=0)
    buf.pos[0, :a] = torch.from_numpy(pos[np.concatenate(rows)])
    return buf


def test_finetune_vs_reference_golden(golden):
    import train
    from gcc_b200.datasets.data_util import BatchedSubgraphs
    z = golden("train_finetune_golden")
    L, H, S, C = int(z["num_layer"]), int(z["hidden"]), int(z["num_steps"]), int(z["num_classes"])
    model = _encoder(H, L)
    model.load_state_dict({k[5:]: torch.from_numpy(z[k]) for k in z if k.startswith("init/")})
    model = model.cuda()
    model.dropout_key = int(z["key"])
    out_layer = torch.nn.Linear(H, C)
    with torch.no_grad():
        out_layer.weight.copy_(torch.from_numpy(z["init_out/weight"]))
        out_layer.bias.copy_(torch.from_numpy(z["init_out/bias"]))
    out_layer = out_layer.cuda()
    criterion = torch.nn.CrossEntropyLoss()
    opt_m = torch.optim.Adam(model.parameters(), lr=0.005, betas=(0.9, 0.999), weight_decay=1e-5)
    opt_o = torch.optim.Adam(out_layer.parameters(), lr=0.005, betas=(0.9, 0.999), weight_decay=1e-5)
    opt = types.SimpleNamespace(hidden_size=H, learning_rate=0.005, epochs=int(z["epochs"]), print_freq=1000,
                                tb_freq=1000)
    for st in range(S):
        buf = _fixture_batch(z, "s%d" % st)
        y = torch.from_numpy(z["s%d_y" % st]).cuda()
        loss, f1 = train.train_finetune(st, [(BatchedSubgraphs(buf, 0), y)], model, out_layer, criterion, opt_m,
                                        opt_o, None, opt)
        assert np.isclose(loss, z["losses"][st], rtol=1e-3), (st, loss, z["losses"][st])
        assert np.isclose(f1, z["f1"][st]), (st, f1, z["f1"][st])
        sd = {k: v.cpu().numpy() for k, v in model.state_dict().items()}
        for k in z:
            if k.startswith("s%d_model/" % st):
                name = k.split("/", 1)[1]
                if ("mlp.linears" in name and name.endswith("bias")) or \
                        (name.endswith("running_mean") and "apply_func" in name):
                    continue            # zero-gradient biases under BatchNorm: chaotic in the reference too
                assert np.allclose(sd[name], z[k], rtol=2e-3, atol=5e-5), (st, name, np.abs(sd[name] - z[k]).max())
        assert np.allclose(out_layer.weight.detach().cpu().numpy(), z["s%d_out/weight" % st], rtol=2e-3, atol=5e-5)
        assert np.allclose(out_layer.bias.detach().cpu().numpy(), z["s%d_out/bias" % st], rtol=2e-3, atol=5e-5)
    buf = _fixture_batch(z, "valid")
    y = torch.from_numpy(z["valid_y"]).cuda()
    vloss, vf1 = train.test_finetune(S, [(BatchedSubgraphs(buf, 0), y)], model, out_layer, criterion, None, opt)
    assert np.isclose(vloss, float(z["valid_loss"]), rtol=2e-3), (vloss, float(z["valid_loss"]))
    assert np.isclose(vf1, float(z["valid_f1"]))
    with torch.no_grad():
        logits = out_layer(model(BatchedSubgraphs(buf, 0))).cpu().numpy()
    assert np.allclose(logits, z["valid_logits"], rtol=2e-3, atol=2e-4)


def _two_class_graphs(n_graphs, seed=0):
    """Class 0: sparse random graphs; class 1: the same plus a hub joined to every node."""
    from gcc_b200.datasets import synthetic
    from gcc_b200.datasets.labeled import _simple_csr
    rng = np.random.RandomState(seed)
    graphs, labels = [], []
    for i in range(n_graphs):
        n = int(rng.randint(14, 40))
        m = 2 * n
        src, dst = rng.randint(0, n, m), rng.randint(0, n, m)
        lab = i % 2
        if lab:
            hub = int(rng.randint(0, n))
            src = np.concatenate([src, np.full(n, hub)])
            dst = np.concatenate([dst, np.arange(n)])
        graphs.append(_simple_csr(src, dst, n, "g%d" % i))
        labels.append(lab)
    assert isinstance(graphs[0], synthetic.CSRGraph)
    return graphs, np.array(labels)


def test_whole_graph_batches_match_oracle():
    """GraphClassificationDatasetLabeled: relabelled whole graphs (isolated vertices included), device
    eigensolver features, encoder forward -- against the oracle on the SAME features with the seed flag on the
    max-degree node of the ORIGINAL numbering (the reference's entire_graph layout)."""
    from gcc_b200.datasets.labeled import GraphClassificationDatasetLabeled
    from oracle import model as om
    from oracle import posenc as opos
    graphs, labels = _two_class_graphs(12, seed=3)
    ds = GraphClassificationDatasetLabeled((graphs, labels), batch_size=6)
    assert ds.num_classes == 2 and len(ds) == 12
    torch.manual_seed(5)
    model = _encoder(32, 3).cuda().eval()
    params = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    seen = 0
    for gq, y in ds.batches(batch_size=6):
        idx = np.arange(seen, seen + 6)
        seen += 6
        assert y.cpu().tolist() == labels[idx].tolist()
        with torch.no_grad():
            feat = model(gq).cpu().numpy()
        n_tot = gq.number_of_nodes()
        pos_dev = gq.buffers.pos[0, :n_tot].cpu().numpy()
        eig_dev = gq.buffers.eigvals[:6].cpu().numpy()
        # oracle input in the ORIGINAL numbering: undo the relabelling graph by graph
        ip_all, ix_all, pos_all, seed_all, noff = [0], [], [], [], [0]
        a = e_off = 0
        for i in idx:
            g = graphs[i]
            n = g.num_nodes
            s = int(ds.seeds[i])
            assert s == int(np.argmax(np.diff(g.indptr)))
            perm = np.concatenate([[s], np.arange(s), np.arange(s + 1, n)])     # perm[new] = old
            p = np.empty((n, 32), np.float32)
            p[perm] = pos_dev[a:a + n]
            lap = opos.normalized_adjacency(g.indptr, g.indices, n).toarray()
            k = min(n - 2, 32)
            w_exact, _ = opos.eig_topk_exact(lap, k)
            lam = eig_dev[i - idx[0], :k]
            assert np.allclose(lam, w_exact, atol=2e-5), (i, np.abs(lam - w_exact).max())
            rn = np.linalg.norm(p[:, :k], axis=1)
            assert np.allclose(rn[rn > 0], 1.0, atol=1e-4)                    # rows are L2-normalised (data_util.py:258)
            pos_all.append(p)
            sd = np.zeros(n, np.int64)
            sd[s] = 1
            seed_all.append(sd)
            ix_all.append(g.indices.astype(np.int64) + noff[-1])
            ip_all.extend((g.indptr[1:] + e_off).tolist())
            e_off += len(g.indices)
            noff.append(noff[-1] + n)
            a += n
        indptr = np.array(ip_all, dtype=np.int64)
        feat_o, _, _ = om.gin_encoder_forward(params, indptr, np.concatenate(ix_all), torch.from_numpy(np.concatenate(pos_all)),
                                              np.concatenate(seed_all), np.diff(indptr), np.array(noff), num_layers=3,
                                              max_degree=512, norm=True, bn_train=False, dropout_keep=None)
        assert np.allclose(feat, feat_o.numpy(), rtol=1e-3, atol=1e-4), np.abs(feat - feat_o.numpy()).max()
    assert seen == 12


def test_finetune_learns_graph_and_node_classification(tmp_path):
    """End to end through train.py's main_finetune on labeled synthetic data: the whole-graph task (hub vs no
    hub) and a node task (label = degree bucket) both beat chance clearly after a few epochs."""
    import train
    from gcc_b200.datasets import synthetic
    from gcc_b200.datasets.labeled import GraphClassificationDatasetLabeled, NodeClassificationDatasetLabeled
    graphs, labels = _two_class_graphs(120, seed=1)
    args = train.parse_option(["--finetune", "--epochs", "6", "--batch-size", "16", "--hidden-size", "32",
                               "--num-layer", "3", "--rw-hops", "32", "--model-path", str(tmp_path / "m"),
                               "--tb-path", str(tmp_path / "tb"), "--dataset", "synthetic-graphs", "--gpu", "0",
                               "--print-freq", "1000", "--learning_rate", "0.01"])
    f1 = train.main_finetune(args, dataset=GraphClassificationDatasetLabeled((graphs, labels), batch_size=16))
    assert f1 >= 0.8, f1
    g = synthetic.chung_lu(3000, 12000, 0.5, seed=2)
    deg = np.diff(g.indptr)
    y = (deg > np.median(deg)).astype(np.int64)
    args.dataset, args.epochs = "synthetic-nodes", 3
    ds = NodeClassificationDatasetLabeled((g, y), rw_hops=32, batch_size=64)
    assert ds.num_classes == 2
    args.batch_size = 64
    f1 = train.main_finetune(args, dataset=ds)
    assert f1 >= 0.75, f1
