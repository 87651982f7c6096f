"""CPU: host-side logic and the C-ABI surface (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


def test_library_builds_loads_and_exports_every_declared_symbol():
    import __graft_entry__ as ge
    from gcc_b200 import _capi
    lib_path = ge.build()
    lib = _capi.bind(ctypes.CDLL(lib_path))                 # raises if a prototype is missing
    hdr = open(os.path.join(ROOT, "include", "gccb200.h")).read()
    declared = set(re.findall(r"\b(gccb_[a-z0-9_]+)\s*\(", hdr))
    assert declared and declared == set(_capi.SYMBOLS), declared ^ set(_capi.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.gccb_version() == 200
    if not torch.cuda.is_available():
        assert lib.gccb_arch() < 0                          # no device: loud negative status, no fallback
        assert b"CUDA" in lib.gccb_last_error()


def test_no_cpu_fallback_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from gcc_b200 import _lib
    from gcc_b200.datasets import synthetic
    from gcc_b200.datasets.graph_dataset import LoadBalanceGraphDataset
    with pytest.raises(_lib.GccbError):
        LoadBalanceGraphDataset(dgl_graphs_file=synthetic.erdos_renyi(100, 300), batch_size=4)
    from gcc_b200.contrastive.criterions import NCESoftmaxLoss
    with pytest.raises(_lib.GccbError):
        NCESoftmaxLoss()(torch.zeros(2, 3))


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "gcc_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "cuda_emu.h" not in src or f == "common.cuh"      # emu include is #ifdef-guarded
    for f in ("train.py", "generate.py"):                                # the CLIs are product code too
        src = open(os.path.join(ROOT, f)).read()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f


def test_generation_budget_uses_the_plain_degree():
    """GraphDataset.__getitem__ (graph_dataset.py:243-254): max(rw_hops, int(deg*e/(e-1)/restart + 0.5)),
    no deg^0.75 -- unlike the pretraining loader (:113-124)."""
    import math
    from gcc_b200.datasets.graph_dataset import budget_for_degree
    for deg in (1, 3, 17, 64, 500, 4096):
        for hops, rp in ((64, 0.8), (256, 0.8), (16, 0.5)):
            want = max(hops, int((deg * math.e / (math.e - 1) / rp) + 0.5))
            assert budget_for_degree(deg, hops, rp, exponent=1.0) == want
            assert budget_for_degree(deg, hops, rp) == max(hops, int(((deg ** 0.75) * math.e / (math.e - 1) / rp) + 0.5))


def test_param_layout_matches_c_layout_and_reference_state_dict(golden):
    from gcc_b200 import _capi
    from gcc_b200.models import GraphEncoder
    from gcc_b200.models import layout as glayout
    import __graft_entry__ as ge
    lib = _capi.bind(ctypes.CDLL(ge.build()))
    for L, H in ((5, 64), (2, 32), (5, 256)):
        cfg = glayout.make_cfg(num_layers=L, hidden=H)
        lay = glayout.c_layout(lib, cfg)
        sl, total = glayout.param_slices(cfg)
        assert lay.total == total
        for l in range(L - 1):
            p = "gnn.ginlayers.%d.apply_func." % l
            assert lay.w1[l] == sl[p + "mlp.linears.0.weight"][0] and lay.b2[l] == sl[p + "mlp.linears.1.bias"][0]
            assert lay.bnb_w[l] == sl["gnn.batch_norms.%d.weight" % l][0]
        assert lay.wp[L - 1] == sl["gnn.linears_prediction.%d.weight" % (L - 1)][0]
        assert lay.emb == sl["degree_embedding.weight"][0]
    # same torch seed as the golden run -> identical initial weights, identical state_dict keys/order
    z = golden("train_moco_golden")
    torch.manual_seed(11)
    m = GraphEncoder(positional_embedding_size=32, max_node_freq=16, max_edge_freq=16, max_degree=512,
                     freq_embedding_size=16, degree_embedding_size=16, output_dim=64, node_hidden_dim=64,
                     edge_hidden_dim=64, num_layers=5, num_step_set2set=6, num_layer_set2set=3, norm=True,
                     gnn_model="gin", degree_input=True)
    ref_keys = [k[5:] for k in z if k.startswith("init/")]
    sd = m.state_dict()
    assert list(sd.keys()) == ref_keys
    for k in ref_keys:
        assert np.array_equal(sd[k].numpy(), z["init/" + k]), k
    assert sum(p.numel() for p in m.parameters()) == 190544 and m.n_live == 61904      # SURVEY 8b
    # load_state_dict writes through to the flat buffer; named params alias it
    sd2 = {k: torch.full_like(v, 0.5) if v.dtype.is_floating_point else v for k, v in sd.items()}
    m.load_state_dict(sd2)
    assert float(m.flat_params.min()) == 0.5 == float(m.flat_params.max())
    list(m.parameters())[0].data.fill_(2.0)
    assert float(m.flat_params.max()) == 2.0
    names = [n for n, _ in m.named_parameters()]
    assert names == [str(x) for x in z["param_order"]]


def test_set_bn_train_trick_and_misc():
    """train.py:360-365 switches BatchNorm modules to train mode by class name."""
    from gcc_b200.models import GraphEncoder
    from gcc_b200.utils.misc import AverageMeter, warmup_linear
    m = GraphEncoder(positional_embedding_size=32, max_degree=512, degree_embedding_size=16, output_dim=32,
                     node_hidden_dim=32, num_layers=2, norm=True, gnn_model="gin", degree_input=True)
    m.eval()
    assert not m.bn_train and not m.gnn.drop.training

    def set_bn_train(mod):
        if mod.__class__.__name__.find("BatchNorm") != -1:
            mod.train()
    m.apply(set_bn_train)
    assert m.bn_train and not m.gnn.drop.training
    z = np.load(os.path.join(G, "misc_golden.npz"))
    for x, a, b in zip(z["x"], z["warm01"], z["warm_default"]):
        assert warmup_linear(float(x), 0.1) == a and warmup_linear(float(x)) == b
    am = AverageMeter()
    am.update(2.0, 2)
    am.update(4.0, 2)
    assert am.avg == 3.0 and am.val == 4.0
    with pytest.raises(NotImplementedError):
        GraphEncoder(gnn_model="mpnn")


def test_budget_formula_and_graph_invariants():
    from gcc_b200.datasets import synthetic
    from gcc_b200.datasets.graph_dataset import budget_for_degree
    z = np.load(os.path.join(G, "dataset_golden.npz"))
    for d, (b256, b64) in zip(z["budget_degs"], z["budgets"]):      # values observed inside the reference
        assert budget_for_degree(int(d), 256, 0.8) == b256 and budget_for_degree(int(d), 64, 0.5) == b64
    for g in (synthetic.erdos_renyi(500, 2000, 1), synthetic.chung_lu(3000, 20000, seed=2), synthetic.rmat(10, 5000)):
        deg = np.diff(g.indptr)
        assert deg.min() >= 1 and g.indptr[-1] == len(g.indices)
        rows = np.repeat(np.arange(g.num_nodes), deg)
        assert not np.any(rows == g.indices)                          # no self loops
        fwd = set(zip(rows.tolist(), g.indices.tolist()))
        assert all((b, a) in fwd for a, b in list(fwd)[:2000])        # symmetric
        assert len(fwd) == len(g.indices)                             # de-duplicated
