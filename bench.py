#!/usr/bin/env python
"""bench.py -- subgraphs/sec of the MoCo pretraining step (BASELINE.json metric) on N x B200.

  python bench.py --gpus 1 --steps 50 --warmup 5                  (N>1: launched by torchrun)
  python bench.py --impl reference ...                            (CPU oracle arm, host cores)

Workload (config.workload): BASELINE.json configs[1] = "C2": MoCo K=16384 m=0.999, 5-layer GIN
hid=64, rw_hops=256 restart=0.8, batch 256 (per GPU: weak scaling, configs[2] at N>1), synthetic
power-law Chung-Lu graph 1M nodes / 20M edges (CSR ~168 MB > the 126 MB L2, sampled at random).
One step = sample -> induce -> positional features -> GIN q/k -> InfoNCE -> backward -> clip/Adam
-> EMA -> enqueue = 2*B ego-subgraphs.  `value` has inputs resident in HBM; `e2e` drives the same
step with host-side seeds (pinned -> H2D) and a loss read-back (D2H) inside the timed region.
"""
import argparse
import contextlib
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "subgraphs/sec (MoCo pretrain step)"
CONFIGS = {
    # name: nodes, pairs, batch, K, layers, hidden, rw_hops
    "c2": dict(nodes=1_000_000, pairs=20_000_000, batch=256, K=16384, layers=5, hidden=64, rw_hops=256),
    "small": dict(nodes=50_000, pairs=500_000, batch=64, K=1024, layers=5, hidden=64, rw_hops=64),
    # BASELINE config 4 shapes (K=65536, hid=256, batch 1024) in fp32: the kernels are SIMT fp32 in round 1,
    # the bf16 tensor-core variant is future work -- a capability / stress run, not the headline line
    "c4": dict(nodes=1_000_000, pairs=20_000_000, batch=1024, K=65536, layers=5, hidden=256, rw_hops=256),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps (each of the two timed windows)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--mode", default="moco", choices=["moco", "e2e"],
                    help="moco: the headline MoCo step; e2e: the reference's E2E recipe (train.py without --moco: both "
                         "views through the query encoder, in-batch negatives, no queue / momentum encoder)")
    ap.add_argument("--prefetch", type=int, default=4, choices=[1, 2, 3, 4, 5, 6, 8],
                    help="batches the sampler/eigensolver streams run ahead of the training stream")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (loss, embeddings, weights, queue, "
                         "its batch) to DIR/<name>.npy, under 64 MB in all; same arguments, same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload_name(cfg, n_gpus):
    return ("MoCo K=%d m=0.999 T=0.07, %d-layer GIN hid=%d, rw_hops=%d restart=0.8, batch %d%s, "
            "Chung-Lu power-law %d nodes / %d edges" % (
                cfg["K"], cfg["layers"], cfg["hidden"], cfg["rw_hops"], cfg["batch"],
                " per GPU" if n_gpus > 1 else "", cfg["nodes"], cfg["pairs"]))


# ------------------------------------------------------------------------------------------------
# clocks sampling (pynvml in a thread) -- the recipe's clocks line
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}

    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag, self.max_mhz = [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop_flag and self.nv is not None:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.1)

    def start(self):
        self.t.start()

    def stop(self):
        self.stop_flag = True
        self.t.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (C walk/induce, the reference's own scipy eigsh call, torch-CPU model)
def _cpu_worker(args):
    """One DataLoader-worker-like task: sample + induce + positional features for a slice of the
    batch (OMP/MKL threads = 1, like the reference's workers)."""
    (indptr, indices, key, sample_ids, seeds, btable, rt, cap_n, cap_m, rng_seed) = args
    import numpy as np
    from oracle import posenc as opos
    from oracle import rwr as orwr
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    t0 = time.perf_counter()
    subs = orwr.rwr_batch(indptr, indices, key, sample_ids, seeds, btable, rt, cap_n, cap_m)
    t1 = time.perf_counter()
    rng = np.random.RandomState(rng_seed)
    pos = [opos.posenc_reference_call(s["indptr"], s["indices"], s["n"], 32, rng=rng) for s in subs]
    t2 = time.perf_counter()
    return subs, pos, t1 - t0, t2 - t1


_G = {}


def _cpu_make_batch(st):
    """One DataLoader-worker task = ONE whole batch (the reference's workers each assemble full
    batches, graph_dataset.py:85-92 + data_util.py:26-32): seeds, walks, induction, eigsh, collate."""
    import numpy as np
    from oracle import rwr as orwr
    indptr, indices, cdf, btable, rt, cap_n, B = _G["args"]
    sids = np.arange(st * B, (st + 1) * B, dtype=np.int64)
    seeds = orwr.draw_seeds(cdf, 0, sids)
    subs, pos, t_walk, t_eig = _cpu_worker((indptr, indices, 0, sids, seeds, btable, rt, cap_n, 1 << 16, 1000 + st))
    t0 = time.perf_counter()
    views, posv = [[], []], [[], []]
    for j, (s_, p_) in enumerate(zip(subs, pos)):
        views[j & 1].append(s_)
        posv[j & 1].append(p_)
    batches = []
    for v in (0, 1):
        noff = np.concatenate([[0], np.cumsum([s_["n"] for s_ in views[v]])])
        eoff = np.concatenate([[0], np.cumsum([s_["m"] for s_ in views[v]])])
        ip = np.concatenate([eoff[i] + s_["indptr"][:-1] for i, s_ in enumerate(views[v])] + [[eoff[-1]]])
        ix = np.concatenate([noff[i] + s_["indices"] for i, s_ in enumerate(views[v])])
        seed = np.zeros(noff[-1], np.int64)
        seed[noff[:-1]] = 1
        batches.append(dict(indptr=ip, indices=ix, pos=np.concatenate(posv[v]), seed=seed,
                            sub_deg=np.concatenate([np.diff(s_["indptr"]) for s_ in views[v]]), node_off=noff))
    return st, batches, t_walk, t_eig, time.perf_counter() - t0


def cpu_arm(cfg, graph_np, steps, seconds_budget, cores=None):
    """The CPU pipeline the reference runs, restated with the oracle: `workers` loader processes
    (1 BLAS thread each, like DataLoader workers) produce whole batches; the main process consumes
    them with the torch-CPU encoder / MoCo head / Adam.  Steady-state throughput: the clock starts
    when the first batch is consumed.  Returns dict."""
    import multiprocessing as mp
    import numpy as np
    import torch
    from oracle import rwr as orwr
    from oracle import step as ostep
    from oracle import model as om
    cores = cores or os.cpu_count() or 1
    model_threads = max(1, min(16, cores // 4))
    workers = max(1, cores - model_threads)
    indptr, indices = graph_np
    B, L, H, K = cfg["batch"], cfg["layers"], cfg["hidden"], cfg["K"]
    cdf = orwr.seed_cdf(indptr)
    btable = orwr.budget_table(int(np.diff(indptr).max()), cfg["rw_hops"], 0.8)
    _G["args"] = (indptr, indices, cdf, btable, orwr.restart_threshold(0.8), int(btable.max()) + 65, B)
    torch.manual_seed(0)
    torch.set_num_threads(model_threads)
    shapes = om.param_shapes(num_layers=L, hidden=H)
    params = {}
    for k, shp in shapes.items():
        if k.endswith("running_var") or (k.endswith("weight") and len(shp) == 1):
            params[k] = torch.ones(shp)
        elif k.endswith("num_batches_tracked"):
            params[k] = torch.zeros(shp, dtype=torch.long)
        elif len(shp) == 2:
            params[k] = torch.randn(shp) / math.sqrt(shp[1])
        else:
            params[k] = torch.zeros(shp)
    state = dict(params=params, ema={k: v.clone() for k, v in params.items()},
                 memory=torch.rand(K, H) * 0.4 - 0.2, index=0, adam_m={}, adam_v={}, adam_t=0)
    ctx = mp.get_context("fork")
    # Phase 1 -- loader rate: every loader process assembles ONE whole batch, all in parallel
    # (steady-state DataLoader behaviour); rate = workers * 2B / wall time.
    n_load = workers                                           # one whole batch per loader process
    with ctx.Pool(workers) as pool:
        pool.map(abs, range(workers))                          # processes are up before the clock starts
        t0 = time.perf_counter()
        produced = pool.map(_cpu_make_batch, range(n_load), chunksize=1)
        t_load = time.perf_counter() - t0
    loader_rate = 2 * B * n_load / t_load * (workers / float(min(workers, n_load)))
    split = {"walk_induce": sum(p[2] for p in produced), "eigsh": sum(p[3] for p in produced),
             "collate": sum(p[4] for p in produced), "model": 0.0}
    # Phase 2 -- model rate: the main process consumes produced batches (torch-CPU encoder/head/Adam)
    n_model = min(len(produced), 8) if seconds_budget else min(len(produced), max(steps, 1))
    ostep.train_step(state, produced[0][1][0], produced[0][1][1], num_layers=L, moco=True, T=0.07, lr=0.005,
                     dropout_key=1, step_index=0)            # warm-up
    t0 = time.perf_counter()
    for i in range(n_model):
        b_ = produced[i % len(produced)][1]
        ostep.train_step(state, b_[0], b_[1], num_layers=L, moco=True, T=0.07, lr=0.005, dropout_key=1,
                         step_index=1 + i)
    split["model"] = time.perf_counter() - t0
    model_rate = 2 * B * n_model / split["model"]
    value = min(loader_rate, model_rate)                      # pipeline: the slower stage sets the pace
    return dict(value=value, unit="subgraphs/sec", cores=cores, workers=workers,
                model_threads=model_threads, kind="port",
                sample="loader: %d whole batches of %d pairs on %d processes in parallel (C oracle walk+induce + the "
                       "reference's scipy eigsh call, 1 BLAS thread each) = %.0f subgraphs/s; model: %d steps of the "
                       "torch-CPU encoder/loss/Adam on %d threads = %.0f subgraphs/s; pipeline = min of the two; DGL "
                       "itself is absent" % (n_load, B, workers, loader_rate, n_model, model_threads, model_rate),
                steps=n_model, seconds=t_load + split["model"], ms_per_step=1e3 * 2 * B / value,
                loader_rate=loader_rate, model_rate=model_rate,
                split_seconds={k: round(v, 3) for k, v in split.items()},
                split_note="walk/eigsh/collate are CPU-seconds summed over loader processes; model is wall time")


# ------------------------------------------------------------------------------------------------
def make_graph_device(cfg, device):
    from gcc_b200.datasets import synthetic
    return synthetic.chung_lu_device(cfg["nodes"], cfg["pairs"], 0.5, seed=0, device=device)


def run_reference(args, cfg):
    """--impl reference: the CPU path (oracle port; the reference's DGL path cannot run, DGL is
    absent) on the host cores, same workload / metric.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    import torch
    from gcc_b200.datasets import synthetic
    if torch.cuda.is_available():
        g = make_graph_device(cfg, "cuda")
        graph_np = (g.indptr.cpu().numpy(), g.indices.cpu().numpy())
    else:
        g = synthetic.chung_lu(cfg["nodes"], cfg["pairs"], 0.5, seed=0)
        graph_np = (g.indptr, g.indices)
    cpu_arm(cfg, graph_np, max(args.warmup, 1), 0)                      # warm-up steps
    r = cpu_arm(cfg, graph_np, args.steps, 240.0)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "subgraphs/sec",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "model_steps_timed": r["steps"],
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(cfg, 1), "config": args.config},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "workers", "model_threads", "kind",
                                               "sample", "split_seconds", "split_note")},
            "e2e": {"value": r["value"], "unit": "subgraphs/sec", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}
    emit(line)


def run_ours(args, cfg):
    import numpy as np
    import torch
    import torch.distributed as dist
    from gcc_b200 import _lib
    from gcc_b200.contrastive.memory_moco import MemoryMoCo
    from gcc_b200.datasets.graph_dataset import LoadBalanceGraphDataset
    from gcc_b200.engine import PretrainEngine
    from gcc_b200.models import GraphEncoder

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, L, H, K = cfg["batch"], cfg["layers"], cfg["hidden"], cfg["K"]
    torch.manual_seed(0)
    g = make_graph_device(cfg, dev)
    ds = LoadBalanceGraphDataset(rw_hops=cfg["rw_hops"], restart_prob=0.8, positional_embedding_size=32,
                                 dgl_graphs_file=g, num_samples=2000, num_workers=12, num_copies=6,
                                 batch_size=B, seed=0, device=dev)

    def mk():
        return GraphEncoder(positional_embedding_size=32, max_node_freq=16, max_edge_freq=16, max_degree=512,
                            freq_embedding_size=16, degree_embedding_size=16, output_dim=H, node_hidden_dim=H,
                            edge_hidden_dim=H, num_layers=L, num_step_set2set=6, num_layer_set2set=3,
                            norm=True, gnn_model="gin", degree_input=True)

    model, ema = mk(), mk()
    ema.load_state_dict(model.state_dict())                 # moment_update(model, model_ema, 0), train.py:623-624
    model, ema = model.to(dev), ema.to(dev)
    with contextlib.redirect_stdout(sys.stderr):           # the reference prints the queue shape; keep stdout = one JSON line
        contrast = MemoryMoCo(H, None, K, 0.07, use_softmax=True).to(dev)
    eng = PretrainEngine(ds, model, ema, contrast, moco=args.mode == "moco", rank=rank, world_size=world,
                         prefetch=args.prefetch)
    lib = _lib.get()
    total_steps = 75000                                     # train.py defaults: 100 epochs x 750

    def lr_at(step):
        from gcc_b200.utils.misc import warmup_linear
        return 0.005 * warmup_linear(step / total_steps, 0.1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        eng.step(lr=lr_at(eng.global_step))
    barrier()
    for b_ in eng.bufs:
        b_.check_flags()
    # ---- timed region: K steps, inputs resident in HBM, no host sync inside -------------------
    # eng.step() trains on batch t (main stream) while sampler + eigensolver of batch t+1 run on
    # the engine's data stream (loader run-ahead, as the reference's DataLoader workers do).
    clocks = ClockSampler(local)
    clocks.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    eng.count_acc = torch.zeros(4, dtype=torch.float64, device=dev)   # algorithmic-byte counters (device side)
    eng.timing = []
    for i in range(2):              # the diagnostics above use torch kernels / timed events the warm-up never
        eng.step(lr=lr_at(eng.global_step))   # launched: CUDA loads them lazily (tens of ms) -- not inside the window
    eng.count_acc.zero_()
    eng.timing = []
    launches0 = lib.gccb_launch_count()
    step_ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    barrier()
    ev[0].record()
    for i in range(args.steps):
        eng.step(lr=lr_at(eng.global_step))
        step_ev[i].record()
    # the window closes when the data path has caught up too: every step() issued one prepare (sampler +
    # eigensolver of a later batch) on a data stream; without this wait the window would hold K training
    # parts but only K - prefetch data parts (the pipeline was full when the clock started)
    eng.wait_data_streams()
    ev[1].record()
    barrier()
    ms = ev[0].elapsed_time(ev[1])
    per_step = [ev[0].elapsed_time(step_ev[0])] + [step_ev[i - 1].elapsed_time(step_ev[i]) for i in range(1, args.steps)]
    ps = sorted(per_step)
    med = ps[len(ps) // 2]
    step_dist = {"p50_ms": med, "p95_ms": ps[min(len(ps) - 1, int(0.95 * len(ps)))], "max_ms": ps[-1], "min_ms": ps[0],
                 "steps_over_2x_median": int(sum(1 for x in per_step if x > 2 * med)),
                 "slowest_steps": sorted(range(len(per_step)), key=lambda i: -per_step[i])[:3],
                 "drain_ms": ms - sum(per_step),
                 "note": "CUDA-event time between consecutive steps on the training stream; drain_ms = the trailing "
                         "data-path work included in the window after the last training step"}
    launches = lib.gccb_launch_count() - launches0
    clk = clocks.stop()
    samp_ev, eng.timing = eng.timing, None
    cnt_acc, eng.count_acc = eng.count_acc, None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    rank_skew = None
    if world > 1:
        # per-rank window and step-time percentiles: the collective makes every step cost the slowest rank's time
        mine = torch.tensor([ms, med, ps[min(len(ps) - 1, int(0.95 * len(ps)))]], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        rank_skew = {"window_ms": [round(float(x[0]), 3) for x in allr], "p50_ms": [round(float(x[1]), 3) for x in allr],
                     "p95_ms": [round(float(x[2]), 3) for x in allr]}
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = 2.0 * B * world * args.steps / (ms_max / 1e3)
    for b_ in eng.bufs:
        b_.check_flags()
    stats = eng.read_stats()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng)                  # before the e2e steps below change the state
    samp_ms = sum(a.elapsed_time(b) for a, b, _ in samp_ev) / len(samp_ev)
    eig_ms = sum(b.elapsed_time(c) for _, b, c in samp_ev) / len(samp_ev)
    n_sum, m_sum, t_sum, deg_sum = [float(x) / args.steps for x in cnt_acc.tolist()]
    # SURVEY 8(d): per view bytes = T*(8+4) + sum_{v in subv}(8 + 4 deg v) + 4*(2n + 1 + m)
    alg_bytes = t_sum * 12 + (8 * n_sum + 4 * deg_sum) + 4 * (2 * n_sum + 2 * B + m_sum)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (samp_ms / 1e3) / 1e9
    roofline = {"kernel": "sampler: rwr_walk_unique + batch_offsets + induce_fill (per step, 3 launches)",
                "bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                "frac": achieved / peak_gbs, "traffic": None,
                "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6650 GB/s",
                "algorithmic_bytes_per_step": alg_bytes, "ms_per_launch_group": samp_ms,
                "note": "latency-bound at %d ego-nets/step (tens of MB per launch group); see DESIGN.md" % (2 * B)}
    try:
        if args.config != "c2":
            raise KeyError("the ncu capture is of the C2 workload")
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        roofline["traffic"] = tr["sampler_group_dram_bytes_per_step"]
        roofline["traffic_source"] = tr.get("source", "profiles/traffic.json")
    except Exception:
        pass
    eig = eigensolver_report(eng.cur_buf, eig_ms)
    phases = {"sampler_ms": samp_ms, "eigensolver_ms": eig_ms, "step_ms": ms / args.steps,
              "note": "sampler + eigensolver of batch t+1 run on the data stream concurrently with the "
                      "encoder/head/optimizer of batch t on the main stream; step_ms is the pipeline period"}

    # ---- e2e: host seeds (pinned) -> H2D each step, loss D2H each step ---------------------------
    cdf_host = ds.graph.cdf.cpu().numpy()
    rs = np.random.RandomState(1 + rank)
    n_e2e = args.steps
    host_seeds = torch.from_numpy(np.searchsorted(cdf_host, rs.random_sample((n_e2e + 2, B)), side="right")
                                  .clip(max=len(cdf_host) - 1).astype(np.int64)).pin_memory()
    loss_ring = torch.zeros(4, 4, dtype=torch.float32).pin_memory()
    done = [torch.cuda.Event() for _ in range(4)]
    NSEED = 2 * (args.prefetch + 2)             # a slot is rewritten long after the sampler that reads it has run
    seeds_ring = [torch.zeros(B, dtype=torch.int64, device=dev) for _ in range(NSEED)]
    # untimed e2e steps: every data stream (one per batch in flight) must have run the host-seed variant of the
    # data path once -- its first use allocates from that stream's pool of the caching allocator (a cudaMalloc)
    E2E_WARM = args.prefetch + 2
    for i in range(E2E_WARM):
        seeds_ring[i % NSEED].copy_(host_seeds[i % 2], non_blocking=True)
        eng.step(lr=lr_at(eng.global_step), seeds=seeds_ring[i % NSEED])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_losses = []
    LAG = 2                                    # < ring depth 4
    host_t = np.zeros((n_e2e, 3))
    for i in range(n_e2e):
        host_t[i, 0] = time.perf_counter()
        slot = (i + E2E_WARM) % NSEED
        seeds_ring[slot].copy_(host_seeds[2 + i], non_blocking=True)     # seeds of the batch prepared this step
        eng.step(lr=lr_at(eng.global_step), seeds=seeds_ring[slot])
        loss_ring[i & 3].copy_(eng.stats, non_blocking=True)            # D2H of this step's loss / prob / grad norm
        done[i & 3].record()
        host_t[i, 1] = time.perf_counter()
        if i >= LAG:        # the reference's .item() per step (train.py:420-422), read LAG steps late so that the
            done[(i - LAG) & 3].synchronize()                           # host enqueues ahead while those steps run
            e2e_losses.append(float(loss_ring[(i - LAG) & 3][0]))
        host_t[i, 2] = time.perf_counter()
    for i in range(max(n_e2e - LAG, 0), n_e2e):
        done[i & 3].synchronize()
        e2e_losses.append(float(loss_ring[i & 3][0]))
    eng.wait_data_streams()
    e1.record()
    barrier()
    t2 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = 2.0 * B * world * n_e2e / (float(t2.item()) / 1e3)
    enq, wait = (host_t[:, 1] - host_t[:, 0]) * 1e3, (host_t[:, 2] - host_t[:, 1]) * 1e3
    worst = int(np.argmax(enq + wait))
    e2e_host = {"enqueue_p50": float(np.median(enq)), "enqueue_max": float(enq.max()), "wait_p50": float(np.median(wait)),
                "wait_max": float(wait.max()), "slowest_step": worst, "slowest_enqueue": float(enq[worst]),
                "slowest_wait": float(wait[worst]),
                "note": "host wall time per e2e step: enqueue = seed copy + PretrainEngine.step + stats copy; wait = "
                        "blocking read of the result two steps back"}

    line = {"metric": METRIC, "value": value, "unit": "subgraphs/sec", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_name(cfg, world) + ("" if args.mode == "moco" else " [E2E head: no queue]"),
                       "config": args.config,
                       "global_batch_pairs": B * world, "subgraphs_per_step": 2 * B * world,
                       "parallelism": "dp%d (CSR replicated, seeds sharded, one all-gather/step)" % world,
                       "l2": "inputs larger than L2: %.0f MB CSR sampled at random; no explicit flush" % (
                           ds.graph.nbytes / 1e6),
                       "graph_nodes": ds.graph.num_nodes, "graph_nnz": int(ds.graph.indices.numel()),
                       "max_degree": ds.graph.max_degree, "max_walk_budget": ds.graph.max_budget,
                       "avg_nodes_per_egonet": n_sum / (2 * B), "avg_edges_per_egonet": m_sum / (2 * B)},
            "pairs_per_sec": value / 2.0,
            "e2e": {"value": e2e_value, "unit": "subgraphs/sec", "h2d_bytes_per_step": B * 8,
                    "d2h_bytes_per_step": 16, "steps": n_e2e, "host_step_ms": e2e_host,
                    "path": "host np seed draw -> pinned -> H2D -> PretrainEngine.step (trains batch t, prepares a later batch from these seeds) -> stats D2H every step, the host reads each step's copy two steps later"},
            "gpu_launches": int(launches), "gpu_launches_per_step": launches / args.steps,
            "step_time": step_dist, "mode": args.mode, "rank_skew": rank_skew,
            "clocks": clk, "roofline": roofline, "eigensolver": eig, "phases_ms": phases,
            "loss": stats["loss"], "grad_norm": stats["grad_norm"]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        graph_np = (g.indptr.cpu().numpy(), g.indices.cpu().numpy())
        cb = cpu_arm(cfg, graph_np, 10000, args.cpu_seconds)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "workers", "model_threads", "kind",
                                                   "sample", "split_seconds", "split_note")}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_ARRAY_BYTES = 4 << 20          # per array: 14 arrays at most, so a dump stays under 64 MB


def dump_outputs(out_dir, eng):
    """Write what the engine's last step computed as out_dir/<name>.npy, so that two builds can be compared
    output for output (the inputs depend only on the command line): `loss`, `prob`, `grad_norm`; the query
    and key embeddings `feat_q`, `feat_k`; the float entries of the encoder's state_dict after the update,
    flattened in state_dict order (`model_state`; MoCo: also `ema_state` and the queue `memory`); the batch
    the step trained on, per view v in q, k: `node_off_v` (ego-net offsets), `nodes_v` (parent-graph id of
    every ego-net node) and `pos_v` (positional features).  Integer outputs are stored as float64, the rest
    as float32.  An array larger than DUMP_ARRAY_BYTES keeps every s-th row, s the smallest stride that fits.
    Two runs of one build give the same batch bit for bit, but the floats differ where kernels sum in a varying
    order, so compare them with a tolerance: between two c2 runs on a B200 (1000 W) the largest difference was
    1.7e-3, in a BatchNorm running variance; 4e-5 in the embeddings."""
    import numpy as np
    import torch

    def flat_state(model):
        return torch.cat([v.reshape(-1).float() for v in model.state_dict().values() if v.is_floating_point()])

    buf, B = eng.cur_buf, eng.B
    loss, prob, grad_norm = eng.stats[:3].tolist()
    out = {"loss": np.float32(loss), "prob": np.float32(prob), "grad_norm": np.float32(grad_norm),
           "feat_q": eng.feat_q, "feat_k": eng.feat_k, "model_state": flat_state(eng.model)}
    if eng.moco:
        out["ema_state"] = flat_state(eng.model_ema)
        out["memory"] = eng.contrast.memory
    for v, name in enumerate(("q", "k")):
        n = int(buf.node_off[v, B])
        out["node_off_" + name] = buf.node_off[v].double()
        out["nodes_" + name] = buf.orig_id[v, :n].double()
        out["pos_" + name] = buf.pos[v, :n]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        a = a.detach().cpu().numpy() if torch.is_tensor(a) else a
        if a.nbytes > DUMP_ARRAY_BYTES:
            a = a[::-(-a.nbytes // DUMP_ARRAY_BYTES)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def eigensolver_report(buf, eig_ms):
    """SURVEY 8(d): the eigensolver has no closed-form byte count -- report n, k, iterations and
    an fp32 FLOP estimate against the CUDA-core peak.  Per ChFSI iteration on an n-node, m-edge
    ego-net with a 48-column block: filter deg*(2(m+n)+3n)*48, Gram-Schmidt 2n*48^2 (one pass),
    H = Q^T L Q 2(m+n)*48 + 2n*48^2, 48x48 Jacobi ~6 sweeps * 47 rounds * 14e3, X = QW 2n*48^2,
    residual 2(m+n)*48 + 6n*48; direct Jacobi (n <= 64): sweeps * 4 n^3; dense tridiagonal solver (n <= 228,
    reported with 0 iterations): 4/3 n^3 (Householder) + 4*32 n^2 (back-transformation) + 2*2*32^2 n (two
    Gram-Schmidt passes) + 3*32*8n (inverse iterations) + 7*NT*5n (Sturm counts)."""
    import numpy as np
    it, res = buf.eig_debug()
    it, res = it.cpu().numpy().astype(np.int64), res.cpu().numpy()
    cnt = buf.counters.cpu().numpy().astype(np.float64)
    n, m = cnt[:, 0], cnt[:, 1]
    ch = it > 0
    deg_sum = np.where(it >= 1, 4, 0) + 8 * np.maximum(it - 1, 0)
    per_iter = 2 * n * 48 ** 2 * 3 + (2 * (m + n) * 48) * 2 + 6 * n * 48 + 6 * 47 * 14e3
    dense = 4.0 / 3.0 * n ** 3 + 128.0 * n ** 2 + 4096.0 * n + 768.0 * n + 7 * 256 * 5.0 * n
    flops = np.where(ch, deg_sum * (2 * (m + n) + 3 * n) * 48 + it * per_iter, np.where(it < 0, -it * 4.0 * n ** 3, dense))
    total = float(flops.sum())
    peak = 148 * 128 * 2 * 1.965e9 / 1e12                   # fp32 FMA on the CUDA cores at 1965 MHz
    ach = total / (eig_ms / 1e3) / 1e12
    return {"bound": "fp32 CUDA-core FMA + shared-memory/barrier latency (neither HBM nor tensor; SURVEY 8d)",
            "k": 32, "block": 48, "egonets": int(len(n)), "mean_n": float(n.mean()), "max_n": int(n.max()),
            "mean_iterations_chfsi": float(it[ch].mean()) if ch.any() else 0.0,
            "egonets_dense_solver": int((it == 0).sum()), "egonets_chfsi": int(ch.sum()),
            "max_iterations": int(it.max()), "max_residual": float(res.max()),
            "est_flop_per_batch": total, "achieved": ach, "peak": peak, "unit": "TFLOP/s",
            "frac": ach / peak, "ms_per_batch": eig_ms, "egonets_per_sec": len(n) / (eig_ms / 1e3)}


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else any library prints (NCCL's
    version banner, the reference-style queue-shape print) was diverted to stderr in main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # see gcc_b200/__init__.py (before CUDA starts)
    args = parse()
    cfg = CONFIGS[args.config]
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                                          # fd-level: also catches C libraries
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
