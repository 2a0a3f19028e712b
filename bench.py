#!/usr/bin/env python
"""bench.py — enclosing-subgraphs/sec of the IGMC train step (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (1 process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port)

A *step* is one pass of the hot path over one batch of 50 (user,item) pairs per GPU of the synthetic
ml_1m-shaped matrix (max-nodes-per-hop 100): H2D(indices) -> extract -> adjacency -> fused RGCN
forward+loss -> backward -> gradient assembly(+ARR) -> [NCCL all-reduce] -> Adam.
  value : device-timed throughput, step inputs already resident in HBM, L2 flushed between steps
  e2e   : through the public TrainEngine.step() API with pinned-host indices in, loss read back, per step
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the single JSON line

WORKLOADS = {
    # name: (preset, batch per GPU, description)
    "ml_1m": ("ml_1m", 50, "ml_1m* synthetic 6040x3706 nnz 900188, mnph=100, batch=50/GPU, hop=1, R=5, 4xRGCN(32), "
                           "adj_dropout=0, ARR=0.001, Adam lr 1e-3"),
    "ml_100k": ("ml_100k", 50, "ml_100k* synthetic 943x1682 nnz 80000, mnph=200, batch=50/GPU, adj_dropout=0.2"),
    "ml_1m_r02": ("ml_1m_r02", 256, "ml_1m* ratio 0.2 synthetic nnz 216045, mnph=100, batch=256/GPU"),
    "flixster": ("flixster", 50, "flixster (REAL Monti split, 3000x3000, 23556 train ratings, R=10), no node cap, STATIC "
                                 "pre-extracted subgraphs (device-resident store + batch-assembly kernel), "
                                 "batch=50/GPU, adj_dropout=0.2"),
}
ARR = 0.001
LR = 1e-3
SAMPLE_SEED = 0x51ED270B7F4A7C15   # sampling stream of the timed `value` steps


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port of the reference's extraction + restated PyG-1.4.2 model)
# ------------------------------------------------------------------------------------------------
_G = {}


def _pool_init(adj_blob, cv, mnph, use_ref):
    import scipy.sparse as ssp
    data, indices, indptr, shape = adj_blob
    A = ssp.csr_matrix((data, indices, indptr), shape=shape)
    _G["cv"], _G["mnph"], _G["ref"] = cv, mnph, None
    if use_ref:
        from oracle import ref_shim
        m = ref_shim.load()                      # the reference's own util_functions.py (oracle/_ref)
        _G["ref"] = m
        _G["idx"] = (m.SparseRowIndexer(A), m.SparseColIndexer(A.tocsc()))
    else:
        from oracle import extract_np
        _G["g"] = extract_np.RatingCSR(A)


def _pool_extract(args):
    u, v, lab, pid = args
    m = _G["ref"]
    if m is not None:   # reference code path: subgraph_extraction_labeling + construct_pyg_graph (util_functions.py:208-297)
        import random
        random.seed(pid)
        out = m.subgraph_extraction_labeling((u, v), _G["idx"][0], _G["idx"][1], 1, 1.0, _G["mnph"], None, None,
                                             _G["cv"], lab)
        d = m.construct_pyg_graph(*out)
        return dict(x=d.x.numpy(), edge_index=d.edge_index.numpy(), edge_type=d.edge_type.numpy(),
                    y=d.y.numpy().reshape(-1))
    from oracle import extract_np
    sub = extract_np.extract_subgraph(_G["g"], u, v, 1, 1.0, _G["mnph"], seed=0, pair_id=pid)
    return extract_np.construct_graph(sub, _G["cv"][lab], 1)


def _collate(graphs):
    """PyG Batch.from_data_list (SURVEY A.3) of per-graph dicts."""
    off, xs, eis, ets, ys, bs = 0, [], [], [], [], []
    for gi, g in enumerate(graphs):
        n = g["x"].shape[0]
        xs.append(g["x"]); eis.append(g["edge_index"] + off); ets.append(g["edge_type"]); ys.append(g["y"])
        bs.append(np.full(n, gi, np.int64))
        off += n
    return dict(x=np.concatenate(xs).astype(np.float32), edge_index=np.concatenate(eis, 1).astype(np.int64),
                edge_type=np.concatenate(ets).astype(np.int64), y=np.concatenate(ys).astype(np.float32),
                batch=np.concatenate(bs), num_graphs=len(graphs))


class CpuReference(object):
    """The reference's CPU train path: per-pair extraction in a persistent process pool (its DataLoader workers,
    train_eval.py:40-45) running the reference's OWN extraction code when it is present (oracle/_ref, built by
    oracle/make_ref.py; else the numpy port), + the PyG-1.4.2-formulation model step on the host threads."""

    def __init__(self, ds, batch, cores=None, model_kind="igmc", k=30):
        import multiprocessing as mp
        import torch
        from oracle import pyg_restated, ref_shim
        self.ds, self.B = ds, batch
        self.cores = cores or os.cpu_count()
        self.use_ref = ref_shim.available()
        A = ds["adj_train"]
        self.pool = mp.get_context("fork").Pool(self.cores, _pool_init,
                                                ((A.data, A.indices, A.indptr, A.shape), ds["class_values"],
                                                 ds["max_nodes_per_hop"], self.use_ref))
        self.threads = min(self.cores, 16)
        torch.set_num_threads(self.threads)
        self.pyg = pyg_restated
        self.build_model(model_kind, k)

    def build_model(self, model_kind, k):
        import torch
        from oracle import pyg_restated
        ds = self.ds
        torch.manual_seed(1)
        if model_kind == "dgcnn_rs":
            self.model = pyg_restated.DGCNN_RSRef(4, (32, 32, 32, 1), k, ds["num_relations"], 4,
                                                  ds["adj_dropout"]).train()
        else:
            self.model = pyg_restated.IGMCRef(4, (32, 32, 32, 32), ds["num_relations"], 4, ds["adj_dropout"]).train()
        self.model_kind = model_kind
        self.opt = torch.optim.Adam(self.model.parameters(), lr=LR)

    def extract_graphs(self, idx):
        tu, tv, tl = self.ds["train"]
        return self.pool.map(_pool_extract, [(int(tu[i]), int(tv[i]), int(tl[i]), int(i)) for i in idx],
                             chunksize=max(1, len(idx) // (8 * self.cores)))

    def extract(self, idx):
        return _collate(self.extract_graphs(idx))

    def model_step(self, nb):
        tb = self.pyg.to_torch_batch(nb)
        self.opt.zero_grad()
        if self.model_kind == "dgcnn_rs":
            import torch.nn.functional as F
            out = self.model(tb["x"], tb["edge_index"], tb["edge_type"], tb["batch"], num_graphs=tb["num_graphs"])
            loss = F.mse_loss(out, tb["y"].view(-1)) + ARR * self.pyg.arr_regulariser(self.model)
        else:
            loss, _ = self.pyg.train_loss(self.model, tb, ARR)
        loss.backward()
        self.opt.step()
        return float(loss.detach())

    def close(self):
        self.pool.terminate()


def run_reference(args, ds, B, rank):
    """--impl reference / cpu_baseline: the two halves of the reference's CPU step are timed separately - extraction
    as ONE pool.map over a large set of pairs (>= 1000: steady state of the worker pool, not per-batch fork/IPC jitter)
    and the model step on pre-extracted batches - and combined as the reference overlaps them (DataLoader workers):
    value = min(extraction rate, model rate); the serial figure is listed too."""
    import torch
    ref = CpuReference(ds, B, model_kind=getattr(args, "model", "igmc"), k=getattr(args, "k", None) or 30)
    rng = np.random.default_rng(123)
    n = len(ds["train"][0])
    static = ds["name"] == "flixster"   # the reference pre-extracts this dataset once (MyDataset): model-bound steps
    steps = max(1, int(args.steps))
    ref.extract_graphs(rng.choice(n, min(n, 4 * ref.cores), replace=False))          # warm the workers
    n_pairs = min(n, max(1000, 4 * B))
    idx_all = rng.choice(n, n_pairs, replace=False)
    t = time.perf_counter()
    graphs = ref.extract_graphs(idx_all)
    t_ext = time.perf_counter() - t
    ext_rate = n_pairs / t_ext
    batches = [_collate(graphs[s * B:(s + 1) * B]) for s in range(min(steps + 1, n_pairs // B))]
    nb0 = batches[0]
    if getattr(args, "model", "igmc") == "dgcnn_rs" and not getattr(args, "k", None):
        nn_ = np.sort(np.bincount(nb0["batch"], minlength=B))   # percentile rule of models.py:69-73 on one batch
        ref.build_model("dgcnn_rs", max(10, int(nn_[int(np.ceil(0.6 * len(nn_))) - 1])))
    # the reference's best thread count for the small per-edge bmm ops (oversubscription hurts it)
    best = (1e30, ref.threads)
    for th in sorted({8, 16, 32, 64, ref.cores} & set(range(1, ref.cores + 1))):
        torch.set_num_threads(th)
        ref.model_step(nb0)
        t = time.perf_counter()
        ref.model_step(nb0)
        best = min(best, (time.perf_counter() - t, th))
    ref.threads = best[1]
    torch.set_num_threads(ref.threads)
    budget, t_mod, done = 150.0, 0.0, 0
    t0 = time.perf_counter()
    while done < steps and (time.perf_counter() - t0) < budget:
        a = time.perf_counter()
        ref.model_step(batches[1 + done % (len(batches) - 1)] if len(batches) > 1 else nb0)
        t_mod += time.perf_counter() - a
        done += 1
    ref.close()
    mod_rate = B * done / t_mod
    value = mod_rate if static else min(ext_rate, mod_rate)
    ext_kind = "reference" if ref.use_ref else "port"
    return dict(value=value, steps=done, ms_per_step=1000.0 * B / value, cores=ref.cores,
                extraction_subgraphs_per_s=ext_rate, model_subgraphs_per_s=mod_rate, extraction_kind=ext_kind,
                serial_subgraphs_per_s=1.0 / (1.0 / ext_rate + 1.0 / mod_rate),
                sample="extraction: %d pairs in one map over a %d-process pool (%s); model: %d steps of %d subgraphs, "
                       "PyG-1.4.2-formulation fwd/bwd/Adam on %d torch threads (best of {8,16,32,64,all}); %s"
                       % (n_pairs, ref.cores,
                          "the reference's own subgraph_extraction_labeling + construct_pyg_graph" if ref.use_ref
                          else "numpy port of the reference's extraction", done, B, ref.threads,
                          "value=model rate: the static dataset is pre-extracted once" if static else
                          "value=min(extraction, model) as the reference overlaps them"))


def cpu_baseline_dict(r):
    # kind: the model half is a restatement (PyG 1.4.2 is not installable here), so the arm as a whole is a port;
    # the extraction half runs the reference's own code whenever oracle/_ref is present
    return {"value": r["value"], "unit": "subgraphs/s", "cores": r["cores"], "kind": "port",
            "extraction_kind": r["extraction_kind"], "model_kind": "port (PyG 1.4.2 RGCNConv restated)",
            "sample": r["sample"], "extraction_subgraphs_per_s": r["extraction_subgraphs_per_s"],
            "model_subgraphs_per_s": r["model_subgraphs_per_s"],
            "serial_subgraphs_per_s": r["serial_subgraphs_per_s"]}


def make_config(desc, G, world, no_graph=False):
    """identical keys on both arms (the driver compares the dicts); the l2 / graph / pipeline entries describe how
    OUR arm is timed, the reference arm times whole CPU steps on the same workload"""
    return {"workload": desc, "global_batch": G, "parallelism": "dp%d" % world,
            "l2": "flushed between timed steps (256 MiB fill), per-step CUDA events summed",
            "cuda_graph": not no_graph,
            "pipeline": "extraction of batch k+1 overlaps the model step of batch k (two graph branches)"}


def gpu_baseline(ds, train, steps_idx, B, model_kind="igmc", steps=12):
    """BASELINE config 2 / SURVEY 8(d): "vs PyG on the same B200".  PyG is not installable, so this is the restated
    PyG-1.4.2 formulation (index_select of per-edge weights + bmm + scatter-mean, autograd, torch.optim.Adam) run with
    torch CUDA ops on the same batches - what the reference does when a GPU is present (train_eval.py:20,159-177).
    The batches come from OUR extractor (collated on the device), so only the model half is the baseline's."""
    import torch
    from oracle import pyg_restated
    dev = torch.device("cuda")
    torch.manual_seed(1)
    if model_kind != "igmc":
        return None
    ref = pyg_restated.IGMCRef(4, (32, 32, 32, 32), ds["num_relations"], 4, ds["adj_dropout"]).to(dev).train()
    opt = torch.optim.Adam(ref.parameters(), lr=LR)
    ex = train.extractor
    tbs = []
    for k in range(min(4, len(steps_idx))):
        b = ex.extract(idx=steps_idx[k])
        tbs.append(dict(x=b.x.clone(), edge_index=b.edge_index.clone(), edge_type=b.edge_type.clone(), y=b.y.clone()))

    def one(tb):
        opt.zero_grad()
        loss, _ = pyg_restated.train_loss(ref, tb, ARR)
        loss.backward()
        opt.step()
        return loss

    for k in range(3):
        one(tbs[k % len(tbs)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        one(tbs[k % len(tbs)])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    peak = torch.cuda.max_memory_allocated() / 2 ** 30
    del ref, opt, tbs
    torch.cuda.empty_cache()
    return {"value": B / (ms / 1000.0), "unit": "subgraphs/s", "ms_per_step": ms, "steps": steps,
            "kind": "port (PyG-1.4.2 formulation: index_select + bmm + scatter-mean, autograd, torch.optim.Adam; "
                    "torch CUDA ops on the same B200, model half only - batches pre-extracted on the device)",
            "peak_mem_gib": round(peak, 2)}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def algorithmic_bytes(stats, in_dims=(4, 32, 32, 32), static=False, keep=1.0):
    """SURVEY.md §8(d) compulsory HBM bytes for a batch with the measured totals in `stats`
    (`keep` = 1 - adj_dropout scales the per-edge terms of the model passes; static: 24 E + 24 n slice read)."""
    n, E, d0, Du, B = stats["n"], stats["E"], stats["d0"], stats["Du"], stats["B"]
    b_ext = (24 * E + 24 * n) if static else (4 * d0 + 5 * Du + 24 * E + 16 * n + 8 * n + 4 * B)
    b_fwd = sum(9 * keep * E + 4 * n * (i + 32) for i in in_dims) + (4 * 2 * 128 + 4) * B
    return dict(extract=b_ext, forward=b_fwd, backward=2 * b_fwd, step=b_ext + 3 * b_fwd)


def batch_stats(ds, engine, idx_list):
    """measured sum n, sum E, sum d0, sum D_u over the timed batches (host side, outside timing)."""
    A = ds["adj_train"]
    rowdeg = np.diff(A.indptr)
    coldeg = np.diff(A.tocsc().indptr)
    tu, tv, _ = ds["train"]
    tot = dict(n=0, E=0, d0=0, Du=0, B=0)
    ex = engine.dataset.extractor
    for idx in idx_list:
        b = ex.extract(idx=idx, seed=SAMPLE_SEED)
        cnt = b._priv["counts"].cpu().numpy()
        tot["n"] += int(cnt[0]); tot["E"] += int(cnt[1]); tot["B"] += len(idx)
        if not hasattr(ex, "node_lists"):   # static store: the batch is a slice read, no CSR scan
            continue
        nu, nv, cu, cv = ex.node_lists(len(idx))
        tot["d0"] += int(rowdeg[tu[idx]].sum() + coldeg[tv[idx]].sum())
        for k in range(len(idx)):
            tot["Du"] += int(rowdeg[nu[k, :cu[k]]].sum())
    return tot


def step_outputs(eng, model, opt):
    """Host copies of what a caller of the timed train step receives after its last step: the step's loss, the
    updated parameters and the Adam moments, named by the model's state_dict keys."""
    # last_loss is the tensor the step graphs were captured with; replays of either pipeline slot write into it because
    # the model's workspace (and its loss) is keyed by batch shape, not by slot
    out = {"loss": eng.last_loss.detach().float().cpu().numpy().reshape(-1)}
    for name, p in model.named_parameters():
        out["param." + name] = p.detach().float().cpu().numpy()
        out["adam_exp_avg." + name] = opt.state[p]["exp_avg"].float().cpu().numpy()
        out["adam_exp_avg_sq." + name] = opt.state[p]["exp_avg_sq"].float().cpu().numpy()
    return out


def write_outputs(path, outputs):
    """``path``/<name>.npy per array (float32, a few hundred KB in all)."""
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from igmc_b200.data import make_synthetic_dataset
    from igmc_b200.models import DGCNN_RS, IGMC, FusedAdam
    from igmc_b200.train_eval import TrainEngine
    from igmc_b200.util_functions import MyDataset, MyDynamicDataset

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    preset, B, desc = WORKLOADS[args.workload]
    ds = make_synthetic_dataset(preset, seed=0)
    tu, tv, tl = ds["train"]
    static = preset == "flixster"
    train = (MyDataset if static else MyDynamicDataset)(None, ds["adj_train"], (tu, tv), tl, 1, 1.0,
                                                        ds["max_nodes_per_hop"], None, None, ds["class_values"],
                                                        seed=0)
    torch.manual_seed(1)
    if args.model == "dgcnn_rs":
        model = DGCNN_RS(train, latent_dim=[32, 32, 32, 1], k=0.6, num_relations=ds["num_relations"], num_bases=4,
                         regression=True, adj_dropout=ds["adj_dropout"]).cuda()
        args.k = model.k
        desc = desc.replace("4xRGCN(32)", "DGCNN_RS 4xRGCN(32,32,32,1)") + ", model DGCNN_RS k=%d" % model.k
    else:
        model = IGMC(train, latent_dim=[32, 32, 32, 32], num_relations=ds["num_relations"], num_bases=4,
                     regression=True, adj_dropout=ds["adj_dropout"]).cuda()
    if world > 1:
        dist.broadcast(model.flat_params, 0)
    opt = FusedAdam(model, lr=LR)
    eng = TrainEngine(train, model, opt, B, ARR=ARR, use_graph=not args.no_graph)
    K, W = args.steps, max(args.warmup, 3)
    G = B * world
    rng = np.random.default_rng(1000)
    perm = rng.permutation(len(tu))
    # every step: one global batch of G pairs of the permutation, dealt to the ranks balanced by the pairs' degree
    # estimate (train_eval.deal_balanced, what `train()` does under data parallelism); wraps on small sets
    from igmc_b200.train_eval import deal_balanced
    cost = train.pair_cost()
    steps_idx = []
    for s in range(W + 4 * K + 32):
        chunk = perm[(s * G + np.arange(G)) % len(perm)]
        steps_idx.append(deal_balanced(chunk, cost[chunk], world)[rank] if world > 1 else chunk)
    cursor = [0]

    def next_idx():
        cursor[0] += 1
        return steps_idx[cursor[0]]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (first steps eager, then the graphs of both buffer slots are captured) ----
    # pipelined engine: every step trains on the batch extracted during the previous step and extracts the next
    eng.prime(steps_idx[0], epoch=1, G=G)
    for s in range(W + 4):
        eng.step_pipe(next_idx(), epoch=1, next_G=G)
    eng.check()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    # ---- (1) value: inputs resident in HBM, per-step CUDA events, L2 flushed between steps ----
    staged = torch.zeros(K, B + 4, dtype=torch.int64)
    from igmc_b200.train_eval import _u64_as_i64
    from igmc_b200.models import splitmix64
    value_first = cursor[0] + 1
    for k in range(K):
        staged[k, :B] = torch.as_tensor(steps_idx[value_first + k])   # indices of the batch extracted in step k
        staged[k, B] = _u64_as_i64(SAMPLE_SEED)
        staged[k, B + 1] = _u64_as_i64(eng.drop_seed(100000 + k))
        staged[k, B + 2] = G
        staged[k, B + 3] = _u64_as_i64(eng.drop_seed(100000 + k + 1))   # the next step's draws (list images)
    staged = staged.cuda()
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    # the graphs of the device-resident-input variant are captured here, not inside the timed region (4 untimed steps:
    # per buffer slot one eager launch and one capture), and the clock sampler's process start-up (~90 ms) happens
    # before the barrier so that no rank enters the timed loop late
    for k in range(4):
        eng.stepbuf_dev.copy_(staged[k % K])
        eng.step_pipe(next_idx(), epoch=1, next_G=G, staged=True)
    clocks = ClockSampler(local)
    clocks.start()
    barrier()
    t_wall0 = time.perf_counter()
    if world > 1:
        # the ranks leave the host barrier up to ~1 ms apart; a tiny all-reduce on the device stream lines the GPUs up
        # before the first timed step, which would otherwise absorb that skew as waiting time inside its exchange
        dist.all_reduce(torch.zeros(1, device="cuda"))
    for k in range(K):
        flush.fill_(k & 0xff)
        ev0[k].record()
        eng.stepbuf_dev.copy_(staged[k])
        eng.step_pipe(next_idx(), epoch=1, next_G=G, staged=True)
        ev1[k].record()
    barrier()
    wall = time.perf_counter() - t_wall0
    clk = clocks.stop()
    per_step = np.array([a.elapsed_time(b) for a, b in zip(ev0, ev1)])
    dev_ms = float(per_step.sum())
    outputs = step_outputs(eng, model, opt) if args.dump_outputs and rank == 0 else None
    if os.environ.get("IGMC_BENCH_DEBUG"):
        span = ev0[0].elapsed_time(ev1[-1])
        gaps = np.array([ev1[k].elapsed_time(ev0[k + 1]) for k in range(K - 1)])
        top = np.argsort(-per_step)[:6]
        sys.stderr.write("[rank %d] value loop: sum of steps %.2f ms, first-to-last span %.2f ms, wall %.2f ms; step us "
                         "min/med/max %.0f/%.0f/%.0f; flush gap us med/max %.0f/%.0f; longest steps %s\n" % (
                             rank, dev_ms, span, 1000 * wall, 1000 * per_step.min(), 1000 * np.median(per_step),
                             1000 * per_step.max(), 1000 * np.median(gaps), 1000 * gaps.max(),
                             [(int(i), round(1000 * per_step[i])) for i in top]))
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    value = G * K / (dev_ms / 1000.0)

    # ---- (1b) informative: back-to-back steps, warm L2 (what a real epoch looks like) ----
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        eng.stepbuf_dev.copy_(staged[k])
        eng.step_pipe(next_idx(), epoch=1, next_G=G, staged=True)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    warm_ms = float(t.item())

    # ---- (2) e2e: public API, pinned host indices -> H2D every step, loss D2H every step ----
    # two repetitions, both reported (`e2e.runs_ms_per_step`), the faster one is the value: the region is host-paced
    # wall clock and an occasional multi-millisecond stall of the host process was observed on the short-step workloads
    # every step: (B+4) int64 of inputs travel host -> device (the kernels read them out of pinned host memory) and the
    # step's loss travels device -> host (the update kernel stores it into a pinned ring); without the zero-copy path
    # (IGMC_ZERO_COPY=0 or a non-fused plan) the same bytes move by one H2D and one D2H memcpy per step
    loss_host = torch.zeros(K, dtype=torch.float32).pin_memory()
    zc = eng.zero_copy and eng.exchange is not None
    e2e_runs = []
    for rep in range(2):
        barrier()
        u0 = eng._updates
        t0 = time.perf_counter()
        for k in range(K):
            eng.step_pipe(next_idx(), epoch=2, next_G=G)
            if not zc:
                loss_host[k:k + 1].copy_(eng.last_loss, non_blocking=True)
        barrier()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_runs.append(float(t.item()))
        if zc:   # the ring keeps the losses of the last LOSS_RING updates
            for k in range(max(0, K - eng.LOSS_RING), K):
                loss_host[k] = eng.loss_of_update(u0 + k)
    e2e_s = min(e2e_runs)
    eng.check()
    assert bool(torch.isfinite(loss_host).all()) and float(loss_host.abs().sum()) > 0, "bad training loss read-back"

    out = None
    if rank == 0:
        # ---- per-kernel times (eager launches, CUDA events on the launching stream) + roofline ----
        stats = batch_stats(ds, eng, [steps_idx[value_first + k] for k in range(min(K, 20))])
        ab = algorithmic_bytes(stats, static=static, keep=1.0 - ds["adj_dropout"])
        nb_batches = min(K, 20)
        names = ("extract", "forward", "backward", "grad_reduce", "adam")
        # the engine's step runs forward + loss + backward as ONE launch (igmc_forward_backward) when the model allows
        one_launch = args.model != "dgcnn_rs" and os.environ.get("IGMC_FUSED_FB", "1") != "0"
        acc = {n: 0.0 for n in names + ("forward_backward",)}
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 3)]
        ex = train.extractor
        reps = min(K, 50)
        for k in range(reps):
            idx = torch.as_tensor(steps_idx[value_first + k]).cuda()
            flush.fill_(1)
            evs[0].record()
            b = ex.extract(idx=idx, reuse=True)
            model._step += 1
            drop = model.make_dropout(True)
            model.stage_batch(b, True, drop)   # list images: part of the extraction branch of the step graph
            evs[1].record()
            _, saved = model._launch_forward(b, True, drop, y=b.y, loss_scale=1.0 / G)
            evs[2].record()
            model._launch_backward(b, drop, saved, saved["ws"]["dpred"])
            evs[3].record()
            model._launch_grad_reduce(b, saved, 1.0 / G, ARR, True)
            evs[4].record()
            opt.step(lr_dev=eng.lr_dev)
            evs[5].record()
            if one_launch and model.fused_update_ok(b):
                model.prep_weights(mark=True)      # (its own launch in this eager sequence; the step's update kernel
                flush.fill_(1)                     #  rebuilds the prepared weights itself)
                evs[6].record()
                model._launch_train(b, drop, b.y, 1.0 / G)
                evs[7].record()
            else:
                one_launch = False
            torch.cuda.synchronize()
            for i, n in enumerate(names):
                acc[n] += evs[i].elapsed_time(evs[i + 1])
            if one_launch:
                acc["forward_backward"] += evs[6].elapsed_time(evs[7])
        kern_ms = {n: acc[n] / reps for n in names}
        if one_launch:
            kern_ms["forward_backward"] = acc["forward_backward"] / reps
        ab["forward_backward"] = ab["forward"] + ab["backward"]
        # dominant kernel of the step's critical path; the extraction kernels run under it on the second
        # branch of the step graph and get their own line (`roofline.extract`)
        dom = "forward_backward" if one_launch else max(("forward", "backward"), key=lambda n: kern_ms[n])
        peak, peak_src = peaks()
        traffic = None     # DRAM bytes per launch from an `ncu --set full` capture OF THIS workload + model, else null
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f).get("%s/%s" % (args.workload, args.model), {}).get(dom)
        per_launch_bytes = ab[dom] / nb_batches
        achieved = per_launch_bytes / (kern_ms[dom] * 1e-3) / 1e9
        step_bytes = ab["step"] / nb_batches
        cpu, gpub = None, None
        if not args.skip_cpu_baseline:
            if world == 1 and not static:
                gpub = gpu_baseline(ds, train, [steps_idx[value_first + k] for k in range(4)], B, args.model)
            ns = argparse.Namespace(steps=args.cpu_steps, warmup=1, model=args.model, k=getattr(args, "k", 30))
            cpu = cpu_baseline_dict(run_reference(ns, ds, B, 0))
        out = {
            "metric": "enclosing-subgraphs/sec (train step)", "value": value, "unit": "subgraphs/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "real (tests/golden/flixster_ratings.npz)" if ds.get("real") else "synthetic",
            "config": make_config(desc, G, world, args.no_graph),
            "clocks": clk,
            "e2e": {"value": G * K / e2e_s, "unit": "subgraphs/s", "h2d_bytes_per_step": (B + 4) * 8,
                    "d2h_bytes_per_step": 4, "ms_per_step": 1000.0 * e2e_s / K,
                    "transport": "zero-copy (kernels read the pinned host inputs; loss stored into a pinned host ring)"
                                 if zc else "cudaMemcpyAsync H2D + D2H per step",
                    "runs_ms_per_step": [1000.0 * x / K for x in e2e_runs]},
            # our kernels per pipelined step.  IGMC: gate + extraction (one launch; static store: assembly) + list
            # images + forward/loss/backward (one launch; two with IGMC_FUSED_FB=0) + fused
            # reduce/exchange/Adam/weight-prep = 5 (6).  DGCNN_RS (external readout, no
            # fused update): + weight prep + 3 SortPooling launches + gradient assembly + Adam = 11
            "gpu_launches": (11 if args.model == "dgcnn_rs" else 5 if one_launch else 6) * K,
            "warm_l2": {"value": G * K / (warm_ms / 1000.0), "ms_per_step": warm_ms / K,
                        "note": "same steps back to back without the L2 flush (informative)"},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": per_launch_bytes,
                         "kernel_ms": kern_ms, "step_algorithmic_bytes": step_bytes,
                         "extract": {"achieved": ab["extract"] / nb_batches / (kern_ms["extract"] * 1e-3) / 1e9,
                                     "unit": "GB/s", "algorithmic_bytes_per_launch_pair": ab["extract"] / nb_batches,
                                     "note": "k_extract_fast + k_stage_lists (static store: k_assemble), on the second "
                                             "graph branch under the model kernels"},
                         "step_frac": (step_bytes / (dev_ms / K * 1e-3) / 1e9) / peak},
            "cpu_baseline": cpu,
            "gpu_baseline": gpub,
            "batch_stats": {k: v / stats["B"] for k, v in stats.items() if k != "B"},
            "wall_s_timed_region": wall,
        }
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
    if world > 1:
        # NCCL communicators that were captured into CUDA graphs do not tear down reliably
        # (destroy_process_group was observed to hang): drop the graphs, align the ranks, and let main() leave
        # through os._exit after the JSON line is flushed.
        torch.cuda.synchronize()
        dist.barrier()
        eng.graphs.clear()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ml_1m", choices=sorted(WORKLOADS))
    ap.add_argument("--model", default="igmc", choices=["igmc", "dgcnn_rs"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=12)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss, parameters and Adam moments of the last timed step "
                         "as DIR/<name>.npy (float32); the inputs are seeded, so runs with the same arguments compare "
                         "output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    # stdout carries exactly ONE line (the JSON): anything a library prints to fd 1 during the run (NCCL's version
    # banner, for one) is sent to stderr, and the result is written to the saved descriptor at the end
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.write(result_fd, (json.dumps(obj) + "\n").encode())

    if args.impl == "reference":
        if rank != 0:
            return
        from igmc_b200.data import make_synthetic_dataset
        preset, B, desc = WORKLOADS[args.workload]
        ds = make_synthetic_dataset(preset, seed=0)
        r = run_reference(args, ds, B, rank)
        world = max(1, int(args.gpus))
        line = {"impl": "reference", "metric": "enclosing-subgraphs/sec (train step)", "value": r["value"],
                "unit": "subgraphs/s", "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "real (tests/golden/flixster_ratings.npz)" if ds.get("real") else "synthetic",
                "config": make_config(desc, B * world, world),
                "reference_note": "one CPU process on the host cores (the reference has no data parallelism, "
                                  "train_eval.py:20); `config` is our arm's so that both lines name the same workload",
                "cpu_baseline": cpu_baseline_dict(r),
                "e2e": {"value": r["value"], "unit": "subgraphs/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}}
        emit(line)
        return
    out = run_ours(args)
    if out is not None:
        emit(out)
    sys.stdout.flush()
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        os._exit(0)


if __name__ == "__main__":
    main()
