"""GPU parity tests (B200): every kernel family of libgccb200, driven through the product's
Python API (which calls the C ABI), against the CPU oracle and the golden fixtures produced by
the real reference modules.  Integer outputs must be bit-exact; floating point within the
stated tolerances (north_star: 1e-3 relative for embeddings and loss)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _dataset(graph, B, rw_hops, seed=7, **kw):
    from gcc_b200.datasets.graph_dataset import LoadBalanceGraphDataset
    return LoadBalanceGraphDataset(rw_hops=rw_hops, restart_prob=0.8, positional_embedding_size=32,
                                   dgl_graphs_file=graph, num_samples=B * 4, batch_size=B, seed=seed, **kw)


def _split(buf, v):
    B = buf.B
    noff = buf.node_off[v].cpu().numpy()
    indptr = buf.indptr[v].cpu().numpy()
    indices = buf.indices[v].cpu().numpy()
    orig = buf.orig_id[v].cpu().numpy()
    out = []
    for g in range(B):
        a, z = noff[g], noff[g + 1]
        ip = indptr[a:z + 1]
        out.append(dict(subv=orig[a:z], indptr=ip - ip[0], indices=indices[ip[0]:ip[-1]] - a, n=z - a))
    return out


@pytest.mark.parametrize("name,B,hops", [("er", 32, 32), ("cl", 64, 64), ("cl_big", 48, 256), ("star", 8, 16)])
def test_sampler_bit_exact(name, B, hops):
    from gcc_b200.datasets import synthetic
    from oracle import rwr as orwr
    g = {"er": lambda: synthetic.erdos_renyi(1000, 5000, seed=0),
         "cl": lambda: synthetic.chung_lu(20000, 200000, seed=1),
         "cl_big": lambda: synthetic.chung_lu(50000, 1000000, seed=2),
         "star": lambda: synthetic.star_graph(300)}[name]()
    ds = _dataset(g, B, hops, seed=1234)
    buf = ds.sample_batch(first_sample=100, posenc=False)
    torch.cuda.synchronize()
    buf.check_flags()
    cdf = orwr.seed_cdf(g.indptr)
    want_seeds = orwr.draw_seeds(cdf, 1234, range(100, 100 + B))
    assert np.array_equal(buf.seeds.cpu().numpy(), want_seeds)
    bt = orwr.budget_table(int(np.diff(g.indptr).max()), hops, 0.8)
    assert np.array_equal(ds.graph.budget_table.cpu().numpy()[np.unique(np.diff(g.indptr))],
                          bt[np.unique(np.diff(g.indptr))])
    want = orwr.rwr_batch(g.indptr, g.indices, 1234, np.arange(100, 100 + B), want_seeds, bt,
                          orwr.restart_threshold(0.8), int(bt.max()) + 65, 1 << 18)
    cnt = buf.counters.cpu().numpy()
    for v in (0, 1):
        got = _split(buf, v)
        for gi in range(B):
            w = want[2 * gi + v]
            assert np.array_equal(got[gi]["subv"], w["subv"]), (v, gi)
            assert np.array_equal(got[gi]["indptr"], w["indptr"]), (v, gi)
            assert np.array_equal(got[gi]["indices"], w["indices"]), (v, gi)
            assert tuple(cnt[v * B + gi]) == (w["n"], w["m"], w["steps"], w["sumdeg"])
    # idempotence: the batch is a pure function of (seed, sample ids)
    first = [t.clone() for t in (buf.orig_id, buf.indptr, buf.indices)]
    ds.sample_batch(first_sample=100, posenc=False)
    torch.cuda.synchronize()
    for a, b in zip(first, (buf.orig_id, buf.indptr, buf.indices)):
        n = int(buf.node_off[0, B])
        assert torch.equal(a[0, :n], b[0, :n])


def test_sampler_capacity_overflow_flag():
    from gcc_b200 import _lib
    from gcc_b200.datasets import synthetic
    ds = _dataset(synthetic.erdos_renyi(1000, 5000, seed=0), 16, 64, node_cap=100, edge_cap=100000)
    buf = ds.sample_batch(posenc=True)
    torch.cuda.synchronize()
    with pytest.raises(_lib.GccbError):
        buf.check_flags()


def _spectral_check(sub, u, lam, tol_l=2e-5):
    from oracle import posenc as opos
    n = sub["n"]
    k = min(n - 2, 32)
    if k <= 0:
        assert np.all(u == 0)
        return
    lap = opos.normalized_adjacency(sub["indptr"], sub["indices"], n).toarray()
    w, _ = opos.eig_topk_exact(lap, k)
    assert np.allclose(lam[:k], w, atol=tol_l), np.abs(lam[:k] - w).max()
    theta, resid, ortho = opos.spectral_report(lap, u[:, :k].astype(np.float64))
    assert resid.max() < 3e-4 and ortho < 1e-4, (resid.max(), ortho)   # fp32 Rayleigh-Ritz floor
    assert np.all(u[:, k:] == 0)


def test_posenc_spectral_parity_on_sampled_egonets():
    import ctypes as C
    from gcc_b200 import _lib
    from gcc_b200.datasets import synthetic
    g = synthetic.chung_lu(20000, 200000, seed=1)
    B = 48
    ds = _dataset(g, B, 96, seed=5)
    buf = ds.sample_batch(posenc=False)
    lib = _lib.get()
    _lib.check(lib.gccb_posenc(C.byref(buf.c), 32, 0, _lib.dptr(buf.pos), _lib.dptr(buf.eigvals),
                               _lib.dptr(buf.ws_posenc), buf.ws_posenc.numel(), _lib.stream_ptr()))
    torch.cuda.synchronize()
    buf.check_flags()
    raw = buf.pos.cpu().numpy().copy()
    eig = buf.eigvals.cpu().numpy().copy()
    sizes = set()
    for v in (0, 1):
        subs = _split(buf, v)
        noff = buf.node_off[v].cpu().numpy()
        for gi, s in enumerate(subs):
            _spectral_check(s, raw[v, noff[gi]:noff[gi + 1]], eig[v * B + gi])
            sizes.add(0 if s["n"] <= 64 else 1 if s["n"] <= 128 else 2)
    assert len(sizes) >= 2                                  # more than one size class exercised
    # normalised output: rows unit-norm, equals the row-normalised raw vectors
    ds.sample_batch(first_sample=0, posenc=True)
    torch.cuda.synchronize()
    pos = buf.pos.cpu().numpy()
    for v in (0, 1):
        n = int(buf.node_off[v, B])
        nrm = np.linalg.norm(pos[v, :n], axis=1)
        assert np.allclose(nrm, 1.0, atol=1e-5)


def test_posenc_matches_reference_golden():
    """tests/golden/posenc_golden.npz = outputs of the reference's own
    _add_undirected_graph_positional_embedding (simple spectra: unique up to column sign)."""
    import ctypes as C
    from gcc_b200 import _lib
    from gcc_b200.datasets.graph_dataset import BatchBuffers
    z = np.load(os.path.join(G, "posenc_golden.npz"))
    nc = int(z["num_cases"])
    subs = [dict(indptr=z["indptr%d" % i].astype(np.int32), indices=z["indices%d" % i].astype(np.int32))
            for i in range(nc)]
    if nc % 2:
        subs.append(subs[0])
    B = len(subs) // 2
    N = sum(len(s["indptr"]) - 1 for s in subs)
    E = sum(len(s["indices"]) for s in subs)
    buf = BatchBuffers(B, N + 8, E + 8, 32, 64, "cuda")
    _fill_batch(buf, [subs[:B], subs[B:]])
    lib = _lib.get()
    _lib.check(lib.gccb_posenc(C.byref(buf.c), 32, 1, _lib.dptr(buf.pos), _lib.dptr(buf.eigvals),
                               _lib.dptr(buf.ws_posenc), buf.ws_posenc.numel(), _lib.stream_ptr()))
    torch.cuda.synchronize()
    pos = buf.pos.cpu().numpy()
    noff = buf.node_off.cpu().numpy()
    checked = 0
    for ci in range(nc):
        v, gi = (0, ci) if ci < B else (1, ci - B)
        got, want = pos[v, noff[v, gi]:noff[v, gi + 1]], z["pos%d" % ci]
        k = min(len(want) - 2, 32)
        if k <= 0:
            assert np.all(got == 0) and np.all(want == 0)
        elif bool(z["simple%d" % ci]):
            s = np.sign((got[:, :k] * want[:, :k]).sum(axis=0))
            assert np.allclose(got[:, :k] * s, want[:, :k], atol=5e-5)
            checked += 1
    assert checked >= 8


def _fill_batch(buf, views):
    """Write explicit ego-nets (local-id CSR) into a BatchBuffers (test helper)."""
    B = buf.B
    for v, subs in enumerate(views):
        noff = eoff = 0
        node_off, edge_off = [], []
        ip_all, ix_all, deg_all, gid_all = [], [], [], []
        for g, s in enumerate(subs):
            n, m = len(s["indptr"]) - 1, len(s["indices"])
            node_off.append(noff)
            edge_off.append(eoff)
            ip_all.append(eoff + np.asarray(s["indptr"][:n], dtype=np.int32))
            ix_all.append(noff + np.asarray(s["indices"], dtype=np.int32))
            deg_all.append(np.diff(s["indptr"]).astype(np.int32))
            gid_all.append(np.full(n, g, np.int32))
            noff += n
            eoff += m
        node_off.append(noff)
        edge_off.append(eoff)
        ip_all.append(np.array([eoff], np.int32))
        buf.node_off[v] = torch.tensor(node_off, dtype=torch.int32)
        buf.edge_off[v] = torch.tensor(edge_off, dtype=torch.int32)
        buf.indptr[v, :noff + 1] = torch.from_numpy(np.concatenate(ip_all))
        buf.indices[v, :eoff] = torch.from_numpy(np.concatenate(ix_all))
        buf.sub_deg[v, :noff] = torch.from_numpy(np.concatenate(deg_all))
        buf.graph_id[v, :noff] = torch.from_numpy(np.concatenate(gid_all))
        cnt = torch.tensor([[len(s["indptr"]) - 1, len(s["indices"]), 0, 0] for s in subs], dtype=torch.int64)
        buf.counters[v * B:(v + 1) * B] = cnt
    return buf


def _golden_batch(z, st):
    from gcc_b200.datasets.graph_dataset import BatchBuffers
    views = []
    for name in ("q", "k"):
        indptr, nn = z["s%d_%s_indptr" % (st, name)], z["s%d_%s_num_nodes" % (st, name)]
        indices = z["s%d_%s_indices" % (st, name)]
        subs, a = [], 0
        for n in nn:
            ip = indptr[a:a + n + 1]
            subs.append(dict(indptr=(ip - ip[0]).astype(np.int32), indices=(indices[ip[0]:ip[-1]] - a).astype(np.int32)))
            a += n
        views.append(subs)
    B = len(views[0])
    N = max(len(z["s%d_%s_seed" % (st, nm)]) for nm in ("q", "k"))
    E = max(len(z["s%d_%s_indices" % (st, nm)]) for nm in ("q", "k"))
    buf = BatchBuffers(B, N + 8, E + 8, 32, 64, "cuda")
    _fill_batch(buf, views)
    for v, nm in enumerate(("q", "k")):
        p = z["s%d_%s_pos" % (st, nm)]
        buf.pos[v, :len(p)] = torch.from_numpy(p)
    return buf


@pytest.mark.parametrize("tag", ["moco", "e2e"])
def test_train_step_vs_reference_golden(tag, golden):
    """The module-level API (GraphEncoder + MemoryMoCo + NCESoftmaxLoss + torch Adam, wired exactly
    like the reference's train_moco) reproduces tests/golden/train_*_golden.*.npz, which was produced
    by the REAL reference train_moco: losses, weights after Adam, EMA weights, queue."""
    from gcc_b200.contrastive.criterions import NCESoftmaxLoss, NCESoftmaxLossNS
    from gcc_b200.contrastive.memory_moco import MemoryMoCo
    from gcc_b200.datasets.data_util import BatchedSubgraphs
    from gcc_b200.models import GraphEncoder
    from gcc_b200.utils.misc import warmup_linear
    z = golden("train_%s_golden" % tag)
    L, H, S, K, moco = int(z["num_layer"]), int(z["hidden"]), int(z["num_steps"]), int(z["K"]), bool(z["moco"])

    def mk():
        return GraphEncoder(positional_embedding_size=32, max_node_freq=16, max_edge_freq=16, max_degree=512,
                            freq_embedding_size=16, degree_embedding_size=16, output_dim=H, node_hidden_dim=H,
                            edge_hidden_dim=H, num_layers=L, num_step_set2set=6, num_layer_set2set=3,
                            norm=True, gnn_model="gin", degree_input=True)

    model, model_ema = mk(), mk()
    init = {k[5:]: torch.from_numpy(z[k]) for k in z if k.startswith("init/")}
    model.load_state_dict(init)
    model_ema.load_state_dict(init)
    model, model_ema = model.cuda(), model_ema.cuda()
    model.dropout_key = int(z["key"])
    contrast = MemoryMoCo(H, None, K, 0.07, use_softmax=True).cuda()
    contrast.memory.copy_(torch.from_numpy(z["init_memory"]))
    criterion = NCESoftmaxLoss() if moco else NCESoftmaxLossNS()
    opt = torch.optim.Adam(model.parameters(), lr=0.005, betas=(0.9, 0.999), weight_decay=1e-5)
    model.train()
    model_ema.eval()
    for m in model_ema.modules():                          # train.py:360-365
        if m.__class__.__name__.find("BatchNorm") != -1:
            m.train()
    for st in range(S):
        buf = _golden_batch(z, st)
        gq, gk = BatchedSubgraphs(buf, 0), BatchedSubgraphs(buf, 1)
        if moco:
            feat_q = model(gq)
            with torch.no_grad():
                feat_k = model_ema(gk)
            out = contrast(feat_q, feat_k)
        else:
            feat_q = model(gq)
            feat_k = model(gk)
            out = torch.matmul(feat_k, feat_q.t()) / 0.07
        opt.zero_grad()
        loss = criterion(out)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        for pg in opt.param_groups:
            pg["lr"] = 0.005 * warmup_linear(st / (2.0 * S), 0.1)
        opt.step()
        if moco:
            for p1, p2 in zip(model.parameters(), model_ema.parameters()):
                p2.data.mul_(0.999).add_(p1.detach().data, alpha=1 - 0.999)
        assert np.isclose(loss.item(), z["losses"][st], rtol=1e-3), (st, loss.item(), z["losses"][st])
        sd = {k: v.cpu().numpy() for k, v in model.state_dict().items()}
        for k in z:
            if k.startswith("s%d_model/" % st):
                name = k.split("/", 1)[1]
                if ("mlp.linears" in name and name.endswith("bias")) or \
                        (name.endswith("running_mean") and "apply_func" in name):
                    continue            # zero-gradient biases under BatchNorm: chaotic in the reference too
                assert np.allclose(sd[name], z[k], rtol=2e-3, atol=5e-5), (st, name, np.abs(sd[name] - z[k]).max())
        if moco:
            assert np.allclose(contrast.memory.cpu().numpy(), z["s%d_memory" % st], atol=5e-5)
    if moco:
        assert contrast.index == int(z["final_index"])
        sde = {k: v.cpu().numpy() for k, v in model_ema.state_dict().items()}
        for k in z:
            if k.startswith("s%d_ema/" % (S - 1)):
                name = k.split("/", 1)[1]
                if name.endswith("running_mean") and "apply_func" in name:
                    continue
                assert np.allclose(sde[name], z[k], rtol=2e-3, atol=5e-5), name


def test_moco_modules_vs_reference_golden():
    from gcc_b200.contrastive.criterions import NCESoftmaxLoss, NCESoftmaxLossNS
    from gcc_b200.contrastive.memory_moco import MemoryMoCo
    z = np.load(os.path.join(G, "moco_golden.npz"))
    T = float(z["T"])
    K, d = z["memory0"].shape
    m = MemoryMoCo(d, None, K, T, use_softmax=True).cuda()
    assert sorted(m.state_dict().keys()) == list(z["state_keys"])
    m.memory.copy_(torch.from_numpy(z["memory0"]))
    for s in range(5):
        q = torch.from_numpy(z["q%d" % s]).cuda().requires_grad_(True)
        k = torch.from_numpy(z["k%d" % s]).cuda()
        out = m(q, k)
        assert np.allclose(out.detach().cpu().numpy(), z["out%d" % s], rtol=1e-5, atol=1e-5)
        loss = NCESoftmaxLoss()(out)
        assert np.isclose(loss.item(), float(z["loss%d" % s]), rtol=1e-5)
        B = q.shape[0]
        assert np.isclose(NCESoftmaxLossNS()(out[:, :B].contiguous()).item(), float(z["loss_ns%d" % s]), rtol=1e-5)
        loss.backward()
        assert np.allclose(q.grad.cpu().numpy(), z["dq%d" % s], rtol=1e-4, atol=1e-7)
        assert m.index == int(z["index"][s + 1])
        assert np.array_equal(m.memory.cpu().numpy(), z["memory%d" % (s + 1)])      # incl. wrap-around


def test_engine_step_matches_oracle_and_learns():
    """The fused engine (flat Adam, fused InfoNCE, device sampler) against the CPU oracle step on
    the same sampled batch, then a few steps of training: loss finite and decreasing on average."""
    from gcc_b200.contrastive.memory_moco import MemoryMoCo
    from gcc_b200.datasets import synthetic
    from gcc_b200.engine import PretrainEngine
    from gcc_b200.models import GraphEncoder
    from oracle import step as ostep
    torch.manual_seed(3)
    g = synthetic.chung_lu(5000, 40000, seed=4)
    B, H, L, K = 16, 64, 5, 64
    ds = _dataset(g, B, 48, seed=9)

    def mk():
        return GraphEncoder(positional_embedding_size=32, max_degree=512, degree_embedding_size=16, output_dim=H,
                            node_hidden_dim=H, num_layers=L, norm=True, gnn_model="gin", degree_input=True)

    model, ema = mk(), mk()
    ema.load_state_dict(model.state_dict())
    model, ema = model.cuda(), ema.cuda()
    contrast = MemoryMoCo(H, None, K, 0.07, use_softmax=True).cuda()
    eng = PretrainEngine(ds, model, ema, contrast, moco=True)
    # oracle state from the same initial weights
    sd0 = {k: v.detach().cpu().double().clone() for k, v in model.state_dict().items()}
    state = dict(params={k: v.clone() for k, v in sd0.items()}, ema={k: v.clone() for k, v in sd0.items()},
                 memory=contrast.memory.detach().cpu().double().clone(), index=0, adam_m={}, adam_v={}, adam_t=0)
    eng.step(lr=0.005)
    torch.cuda.synchronize()
    s = eng.read_stats()
    buf = eng.cur_buf

    def view(v):
        n, m = int(buf.node_off[v, B]), int(buf.edge_off[v, B])
        noff = buf.node_off[v].cpu().numpy().astype(np.int64)
        seed = np.zeros(n, np.int64)
        seed[noff[:B]] = 1
        return dict(indptr=buf.indptr[v, :n + 1].cpu().numpy().astype(np.int64),
                    indices=buf.indices[v, :m].cpu().numpy().astype(np.int64),
                    pos=buf.pos[v, :n].cpu().double().numpy(), seed=seed,
                    sub_deg=buf.sub_deg[v, :n].cpu().numpy(), node_off=noff)

    r = ostep.train_step(state, view(0), view(1), num_layers=L, moco=True, T=0.07, lr=0.005,
                         dropout_key=model.dropout_key, step_index=0)
    assert np.isclose(s["loss"], r["loss"], rtol=1e-3), (s["loss"], r["loss"])
    assert np.isclose(s["grad_norm"], r["grad_norm"], rtol=2e-3)
    fq = eng.feat_q.cpu().numpy()
    assert np.allclose(fq, r["feat_q"].numpy(), rtol=1e-3, atol=1e-4)
    # raw (pre-clip) gradients of the flat buffer against autograd's
    gflat = eng.grads.cpu().numpy()
    for k, (off, shape) in model._slices.items():
        if "mlp.linears" in k and k.endswith("bias"):
            continue                                    # exactly-zero true gradient (feeds a BatchNorm)
        got = gflat[off:off + int(np.prod(shape))].reshape(shape)
        want = r["grads"][k].numpy() if k in r["grads"] else np.zeros(shape)
        # (floor: apply_func.bn.weight has a true gradient of ~1e-6 at initialisation -- fp32 summation noise)
        scale = max(np.abs(want).max(), 1e-4)
        assert np.allclose(got, want, rtol=5e-3, atol=2e-3 * scale), (k, np.abs(got - want).max(), scale)
    # weights after the first Adam step: update = lr * g/(|g|+eps) is sign-like, so entries whose
    # gradient is ~eps-sized are ill-conditioned in the reference too; require agreement elsewhere
    sd1 = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    for k, v in state["params"].items():
        if ("mlp.linears" in k and k.endswith("bias")) or (k.endswith("running_mean") and "apply_func" in k) \
                or k.endswith("num_batches_tracked") or k.endswith(".eps"):
            continue
        diff = np.abs(sd1[k] - v.numpy())
        assert diff.max() <= 2 * 0.005 + 1e-6, (k, diff.max())
        assert (diff > 5e-5).mean() < 0.02, (k, (diff > 5e-5).mean())
    assert np.allclose(contrast.memory.cpu().numpy(), state["memory"].numpy(), atol=1e-4)
    losses = [s["loss"]]
    for i in range(30):
        eng.step(lr=0.005)
        if i % 10 == 9:
            losses.append(eng.read_stats()["loss"])
    assert all(np.isfinite(losses))


def test_e2e_engine_runs_config1():
    """BASELINE config 1 shape: E2E, B=32, 2-layer GIN hid=32 on ER(1000, 5000)."""
    from gcc_b200.contrastive.memory_moco import MemoryMoCo
    from gcc_b200.datasets import synthetic
    from gcc_b200.engine import PretrainEngine
    from gcc_b200.models import GraphEncoder
    torch.manual_seed(0)
    ds = _dataset(synthetic.erdos_renyi(1000, 5000, seed=0), 32, 256, seed=0)

    def mk():
        return GraphEncoder(positional_embedding_size=32, max_degree=512, degree_embedding_size=16, output_dim=32,
                            node_hidden_dim=32, num_layers=2, norm=True, gnn_model="gin", degree_input=True)

    model, ema = mk().cuda(), mk().cuda()
    contrast = MemoryMoCo(32, None, 32, 0.07, use_softmax=True).cuda()
    eng = PretrainEngine(ds, model, ema, contrast, moco=False)
    for _ in range(5):
        eng.step(lr=0.005)
    s = eng.read_stats()
    assert np.isfinite(s["loss"]) and 0 < s["loss"] < 10 and s["nodes_q"] > 32


def test_engine_prefetch_matches_serial():
    """The loader run-ahead (sampler + eigensolver of batch t+1 on a second stream) must not change
    results: same batches, same order, same weights as the serial engine."""
    from gcc_b200.contrastive.memory_moco import MemoryMoCo
    from gcc_b200.datasets import synthetic
    from gcc_b200.engine import PretrainEngine
    from gcc_b200.models import GraphEncoder
    g = synthetic.chung_lu(3000, 20000, seed=1)
    out = []
    for prefetch in (0, 1, 6, 2):
        torch.manual_seed(0)
        ds = _dataset(g, 16, 48, seed=5)

        def mk():
            return GraphEncoder(positional_embedding_size=32, max_degree=512, degree_embedding_size=16,
                                output_dim=64, node_hidden_dim=64, num_layers=3, norm=True, gnn_model="gin",
                                degree_input=True)

        model, ema = mk(), mk()
        ema.load_state_dict(model.state_dict())
        model, ema = model.cuda(), ema.cuda()
        contrast = MemoryMoCo(64, None, 64, 0.07, use_softmax=True).cuda()
        eng = PretrainEngine(ds, model, ema, contrast, moco=True, prefetch=prefetch)
        losses = []
        for i in range(6):
            eng.step(lr=0.005)
            losses.append(eng.read_stats()["loss"])
        buf = eng.cur_buf
        out.append((losses, buf.orig_id.cpu().numpy().copy(), buf.node_off.cpu().numpy().copy(),
                    model.flat_params.detach().cpu().numpy().copy()))
    l0, o0, n0, p0 = out[0]
    for l1, o1, n1, p1 in out[1:]:
        assert np.array_equal(n0, n1)                                  # same ego-nets in the 6th batch
        for v in (0, 1):
            assert np.array_equal(o0[v, :n0[v, -1]], o1[v, :n1[v, -1]])
        assert np.allclose(l0, l1, rtol=1e-4), (l0, l1)
        assert np.allclose(p0, p1, atol=2e-3), np.abs(p0 - p1).max()


def test_generate_eval_mode_embeddings_match_oracle():
    """generate.py:33-53 -- (f(q) + f(k)) / 2 with eval-mode BatchNorm, seeds = every node in order,
    budget from the plain degree (graph_dataset.py:243-254): walks bit-exact, embeddings <= 1e-3."""
    from gcc_b200.datasets import synthetic
    from gcc_b200.datasets.graph_dataset import NodeClassificationDataset, budget_for_degree
    from gcc_b200.models import GraphEncoder
    from oracle import model as om
    from oracle import rwr as orwr
    torch.manual_seed(3)
    g = synthetic.erdos_renyi(150, 600, seed=4)
    ds = NodeClassificationDataset(g, rw_hops=24, restart_prob=0.8, batch_size=64, seed=11)
    model = GraphEncoder(positional_embedding_size=32, max_degree=512, degree_embedding_size=16, output_dim=64,
                         node_hidden_dim=64, num_layers=3, norm=True, gnn_model="gin", degree_input=True)
    sd = model.state_dict()
    for k_, v in sd.items():                               # non-trivial running statistics
        if k_.endswith("running_mean"):
            v.copy_(torch.randn_like(v) * 0.1)
        elif k_.endswith("running_var"):
            v.copy_(torch.rand_like(v) + 0.5)
    model.load_state_dict(sd)
    model = model.cuda().eval()
    P = {k_: v.detach().cpu().double() for k_, v in model.state_dict().items()}
    deg = np.diff(g.indptr)
    bt = np.array([budget_for_degree(d, 24, 0.8, exponent=1.0) for d in range(int(deg.max()) + 1)], np.int32)
    got, want = [], []
    for gq, gk, count in ds:
        B = gq.batch_size
        with torch.no_grad():
            got.append(((model(gq) + model(gk)) / 2)[:count].cpu().numpy())
        buf = ds.buffers
        seeds = buf.seeds.cpu().numpy()
        sids = buf.sample_ids.cpu().numpy()
        ref = orwr.rwr_batch(g.indptr, g.indices, 11, sids, seeds, bt, orwr.restart_threshold(0.8),
                             int(bt.max()) + 65, 1 << 16)
        feats = []
        for v in (0, 1):
            noff = buf.node_off[v].cpu().numpy().astype(np.int64)
            n = int(noff[B])
            orig = buf.orig_id[v].cpu().numpy()
            for gi in range(B):
                assert np.array_equal(orig[noff[gi]:noff[gi + 1]], ref[2 * gi + v]["subv"])
            seed_flag = np.zeros(n, np.int64)
            seed_flag[noff[:B]] = 1
            f, _, _ = om.gin_encoder_forward(
                P, buf.indptr[v, :n + 1].cpu().numpy().astype(np.int64),
                buf.indices[v, :int(buf.edge_off[v, B])].cpu().numpy().astype(np.int64),
                buf.pos[v, :n].cpu().double(), seed_flag, buf.sub_deg[v, :n].cpu().numpy(), noff,
                num_layers=3, bn_train=False)
            feats.append(f.detach().numpy())
        want.append(((feats[0] + feats[1]) / 2)[:count])
    got, want = np.concatenate(got), np.concatenate(want)
    assert got.shape == (150, 64)
    assert np.allclose(got, want, rtol=1e-3, atol=1e-4), np.abs(got - want).max()
