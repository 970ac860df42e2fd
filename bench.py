#!/usr/bin/env python
"""bench.py — DeepFM train samples/s on Criteo-shaped synthetic data (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU PyTorch path (baseline/_ref)

A "step" is one full training iteration of the reference's trainer loop
(src/trainer/deepfm.py:44-62): forward -> BCEWithLogits -> zero_grad -> backward ->
optimizer.step, on one batch of synthetic Criteo-shaped ids (65 536 per GPU).

Default workload = BASELINE.json configs[4] / north_star: DeepFM with the FULL Criteo-shaped table
(configs/deepfm/base_config.yaml: D = 16, MLP 400x3 + BatchNorm, dropout 0.5, Adam lr 1e-3 wd 1e-6) row-sharded
over the N GPUs of the box - at N = 1 the same model with one shard, so the 1/2/4/8-GPU lines are the same
experiment.  At N = 1 the line also carries `other_configs`: configs[1] (QR-hashing, qr_80.yaml), configs[0]'s
shape on one GPU with the fused sparse row update, configs[2] (DCN-Mix, Avazu shape), configs[3] (PEP and OptEmbed,
KDD shape) and the SURVEY 8(d) roofline shape (17 M rows: a table far larger than L2), each with its own rooflines.

Prints ONE JSON line (rank 0).  `value` = device-resident inputs; `e2e` = the reference trainer's loop verbatim fed
from pinned host memory with loss.item() every step; `roofline` = the kernel with the largest share of the step
(`roofline_top3`, `roofline_hot_path` list more), measured with CUDA events in a separate pass; `parity_check` = the
in-run check of the sharded path against the single-GPU model; `cpu_baseline` = the unmodified reference classes
timed on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CRITEO_DIMS = [49, 101, 126, 45, 223, 118, 84, 76, 95, 9, 30, 40, 75, 1458, 555, 193949, 138801, 306, 19, 11970, 634,
               4, 42646, 5178, 192773, 3175, 27, 11422, 181075, 11, 4654, 2032, 5, 189657, 18, 16, 59697, 86, 45571]
AVAZU_DIMS = [100000] * 10 + [1000] * 12
KDD_DIMS = [600000] * 8 + [400000] * 3
# SURVEY 8(d) "roofline shape": Criteo field structure with every field > 10k ids scaled x16 -> 17.1 M rows,
# a 1.1 GB fp32 table (>> 126 MB L2), so the gather really runs out of HBM
ROOFLINE_DIMS = [d * 16 if d > 10000 else d for d in CRITEO_DIMS]

METRIC = "DeepFM train samples/s (Criteo shape)"

WORKLOADS = {
    # BASELINE.json configs[1] (default)
    "deepfm_qr_criteo": dict(model="deepfm", dims=CRITEO_DIMS, emb={"name": "qr", "divider": 5}, use_bn=False,
                             p_dropout=0.5, opt=dict(learning_rate=1e-3, weight_decay=1e-6, fused_adam="rsb")),
    # configs[0] shape on the GPU, sparse=True variant (configs/deepfm/base_config_sparse.yaml) with the fused row update
    "deepfm_full_criteo": dict(model="deepfm", dims=CRITEO_DIMS, emb={"name": "vanilla", "sparse": True}, use_bn=True,
                               p_dropout=0.5,
                               opt=dict(learning_rate=1e-3, weight_decay=1e-6, sparse=True, fused_sparse=True, fused_adam="rsb")),
    "deepfm_full_criteo_dense_adam": dict(model="deepfm", dims=CRITEO_DIMS, emb={"name": "vanilla"}, use_bn=True,
                                          p_dropout=0.5, opt=dict(learning_rate=1e-3, weight_decay=1e-6, fused_adam="rsb")),
    "deepfm_full_roofline": dict(model="deepfm", dims=ROOFLINE_DIMS, emb={"name": "vanilla", "sparse": True}, use_bn=True,
                                 p_dropout=0.5,
                                 opt=dict(learning_rate=1e-3, weight_decay=1e-6, sparse=True, fused_sparse=True, fused_adam="rsb")),
    # BASELINE.json configs[4]: full table row-sharded over the GPUs (NVLink peer gathers + shard atomics),
    # dense Adam on each shard (= configs/deepfm/base_config.yaml semantics), dense MLP grads allreduced
    "deepfm_full_criteo_sharded": dict(model="deepfm", dims=CRITEO_DIMS, emb={"name": "vanilla"}, use_bn=True,
                                       p_dropout=0.5, opt=dict(learning_rate=1e-3, weight_decay=1e-6, fused_adam="rsb"), sharded=True),
    # BASELINE.json configs[3]: pruned-mask embeddings on KDD-shaped data (11 fields, 6 M ids, configs/kdd/deepfm)
    "deepfm_pep_kdd": dict(model="deepfm", dims=KDD_DIMS, emb={"name": "pep", "threshold_type": "feature_dim",
                                                                 "init_threshold": -150,
                                                                 "checkpoint_weight_dir": "/tmp/rsb_pep_ckpt"},
                           use_bn=True, p_dropout=0.2, opt=dict(learning_rate=1e-3, weight_decay=1e-5, fused_adam="rsb")),
    "deepfm_optembed_kdd": dict(model="deepfm", dims=KDD_DIMS, emb={"name": "deepfm_optembed"}, use_bn=True,
                                p_dropout=0.2, opt=dict(learning_rate=3e-5, weight_decay=1e-3, fused_adam="rsb")),
    # SURVEY 8 f-3: deep hash embedding, configs/deepfm/dhe_config-50.yaml (k = 1024 codes generated in-kernel,
    # 4 x 1536 Mish/BatchNorm encoder, reference batch 2048: 79 872 encoder rows per step, ~4 TFLOP per step)
    "deepfm_dhe_criteo": dict(model="deepfm", dims=CRITEO_DIMS, batch=2048,
                              emb={"name": "dhe", "hidden_sizes": [1536, 1536, 1536, 1536], "compute_v2": False},
                              use_bn=True, p_dropout=0.5, opt=dict(learning_rate=1e-3, weight_decay=1e-6, fused_adam="rsb")),
    # SURVEY 8(e) widened: the lightweight variants row-sharded too (PEP weight + per-row thresholds on the KDD shape,
    # QR emb2 on the Criteo shape, DCN-Mix over a sharded Avazu-shaped table); --workload ... under torchrun
    "deepfm_pep_kdd_sharded": dict(model="deepfm", dims=KDD_DIMS, emb={"name": "pep", "threshold_type": "feature_dim",
                                                                         "init_threshold": -150,
                                                                         "checkpoint_weight_dir": "/tmp/rsb_pep_ckpt"},
                                   use_bn=True, p_dropout=0.2, opt=dict(learning_rate=1e-3, weight_decay=1e-5, fused_adam="rsb"),
                                   sharded=True),
    "deepfm_qr_criteo_sharded": dict(model="deepfm", dims=CRITEO_DIMS, emb={"name": "qr", "divider": 5}, use_bn=True,
                                     p_dropout=0.5, opt=dict(learning_rate=1e-3, weight_decay=1e-6, fused_adam="rsb"),
                                     sharded=True),
    "dcnmix_full_avazu_sharded": dict(model="dcn_mix", dims=AVAZU_DIMS, emb={"name": "vanilla"}, use_bn=True, p_dropout=0.5,
                                      opt=dict(learning_rate=1e-3, weight_decay=1e-6, fused_adam="rsb"), sharded=True),
    "dcnmix_full_avazu": dict(model="dcn_mix", dims=AVAZU_DIMS, emb={"name": "vanilla"}, use_bn=True, p_dropout=0.5,
                              opt=dict(learning_rate=1e-3, weight_decay=1e-6, fused_adam="rsb")),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            v = json.load(fh).get("hbm_gbs")
        if v:
            return float(v), "measured (MEASURED_PEAKS.json)"
    except (OSError, ValueError):
        pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _zipf_ids(d, batch, g, alpha=1.05):
    """Zipf(alpha) over the ids of one field, clipped to the field size (SURVEY 8(d)): id k has weight
    (k+1)^-alpha, drawn by inverting the CDF with seeded uniforms."""
    import torch

    w = torch.arange(1, d + 1, dtype=torch.float64).pow_(-alpha)
    cdf = torch.cumsum(w, 0)
    u = torch.rand(batch, generator=g, dtype=torch.float64) * cdf[-1]
    return torch.searchsorted(cdf, u).clamp_(max=d - 1)


def make_batches(dims, batch, n, seed, dtype, dist_name="uniform"):
    import torch

    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        if dist_name == "zipf":
            x = torch.stack([_zipf_ids(d, batch, g) for d in dims], 1).to(dtype)
        else:
            x = torch.stack([torch.randint(0, d, (batch,), generator=g) for d in dims], 1).to(dtype)
        y = torch.randint(0, 2, (batch,), generator=g).float()
        out.append((x, y))
    return out


# ------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ------------------------------------------------------------------------------------
# `--impl reference` and the `cpu_baseline` leg time the reference's CPU PyTorch path on this box's host cores:
#   kind "reference": the UNMODIFIED reference classes (src.models.get_ctr_model + src.models.deepfm.get_optimizers,
#                     the loop of src/trainer/deepfm.py:44-62) imported from baseline/_ref, where
#                     __graft_entry__.build() stages the pure-Python reference (it travels to the GPU box with the
#                     snapshot like librsb.so); /root/reference itself is never read here;
#   kind "port":      oracle/torch_port.py (the functional restatement, pinned against the golden vectors) when
#                     baseline/_ref is absent.
PORT_EMBEDDINGS = ("vanilla", "qr", "pep")
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def _reference_available():
    return os.path.isdir(os.path.join(REF_DIR, "src", "models"))


def _port_model(TP, wl, device):
    """Parameters, optimizers and forward function of oracle/torch_port.py for a workload, on `device`."""
    dims = wl["dims"]
    emb = {k: v for k, v in wl["emb"].items() if k != "checkpoint_weight_dir"}
    if emb.get("name", "vanilla") not in PORT_EMBEDDINGS:
        raise NotImplementedError(f"torch port: embedding {emb.get('name')}")
    if wl["model"] == "deepfm":
        p = TP.make_deepfm_params(dims, 16, [400, 400, 400], emb, wl["use_bn"], seed=0)
        fwd = TP.deepfm_forward
    else:
        p = TP.make_dcn_params(dims, 16, [400, 400, 400], emb, seed=0)
        fwd = TP.dcn_mix_forward
    if device.type != "cpu":
        p = {k: v.detach().to(device).requires_grad_(True) for k, v in p.items()}
    opts = TP.make_optimizers(p, {k: v for k, v in wl["opt"].items() if k not in ("fused_sparse", "fused_adam")})
    return p, opts, emb, fwd


def model_config(wl):
    if wl["model"] == "deepfm":
        return dict(num_factor=16, hidden_sizes=[400, 400, 400], p_dropout=wl["p_dropout"], use_batchnorm=wl["use_bn"],
                    embedding_config=dict(wl["emb"]))
    return dict(name="dcn_mix", num_factor=16, hidden_sizes=[400, 400, 400], p_dropout=wl["p_dropout"],
                compile_model=False, embedding_config=dict(wl["emb"]))


def run_cpu_reference(wl, sample_batch, steps, warmup, budget_s=25.0, ids="uniform"):
    """The unmodified reference on the CPU: its own model classes, its own get_optimizers, its trainer's step."""
    import types

    import torch

    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    sys.modules.setdefault("lmdb", types.ModuleType("lmdb"))
    sys.modules.setdefault("optuna", types.ModuleType("optuna"))
    from loguru import logger

    logger.remove()
    import src.models as ref_models
    import src.models.deepfm as ref_deepfm

    if not type(ref_models.DeepFM).__module__ or not ref_models.DeepFM.__module__.startswith("src."):
        raise RuntimeError("the reference registry is rebound to the B200 classes in this process")
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    torch.manual_seed(2023)
    cfg = model_config(wl)
    model = ref_models.get_ctr_model(wl["dims"], cfg)
    opt_cfg = {k: v for k, v in wl["opt"].items() if k not in ("fused_sparse", "fused_adam")}
    opts = ref_deepfm.get_optimizers(model, opt_cfg)
    crit = torch.nn.BCEWithLogitsLoss()
    model.train()
    batches = make_batches(wl["dims"], sample_batch, 2, 2023, torch.int32, ids)

    def step(x, y):                       # src/trainer/deepfm.py:44-62
        out = model(x)
        loss = crit(out, y.float())
        for o in opts:
            o.zero_grad()
        loss.backward()
        for o in opts:
            o.step()
        return loss.item()

    for i in range(warmup):
        step(*batches[i % 2])
    times = []
    t_all = time.perf_counter()
    for i in range(steps):
        t0 = time.perf_counter()
        step(*batches[i % 2])
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s and len(times) >= 3:
            break
    med = statistics.median(times)
    return dict(value=sample_batch / med, ms_per_step=med * 1e3, steps=len(times), cores=cores, kind="reference",
                sample=f"{len(times)} steps of {sample_batch} samples (median step) of the unmodified reference classes "
                       f"(baseline/_ref), torch {torch.__version__} CPU, {cores} threads")


def run_cpu_port(wl, sample_batch, steps, warmup, budget_s=25.0, ids="uniform"):
    import torch

    from oracle import torch_port as TP

    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    dims = wl["dims"]
    p, opts, emb, fwd = _port_model(TP, wl, torch.device("cpu"))
    offsets = torch.tensor([0] + dims[:-1]).cumsum(0)[None, :]
    batches = make_batches(dims, sample_batch, 2, 2023, torch.int64, ids)
    for i in range(warmup):
        TP.train_step(p, opts, *batches[i % 2], offsets, emb, wl["p_dropout"], forward=fwd)
    times = []
    t_all = time.perf_counter()
    for i in range(steps):
        t0 = time.perf_counter()
        TP.train_step(p, opts, *batches[i % 2], offsets, emb, wl["p_dropout"], forward=fwd)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s and len(times) >= 3:
            break
    med = statistics.median(times)
    return dict(value=sample_batch / med, ms_per_step=med * 1e3, steps=len(times), cores=cores, kind="port",
                sample=f"{len(times)} steps of {sample_batch} samples (median step), oracle/torch_port.py, "
                       f"torch {torch.__version__} CPU, {cores} threads")


def run_cpu_arm(wl, sample_batch, steps, warmup, budget_s, ids):
    if _reference_available():
        try:
            return run_cpu_reference(wl, sample_batch, steps, warmup, budget_s, ids)
        except Exception as exc:  # noqa: BLE001 - fall back to the port, say why
            r = run_cpu_port(wl, sample_batch, steps, warmup, budget_s, ids)
            r["sample"] += f" (reference classes failed: {type(exc).__name__}: {exc})"[:200]
            return r
    return run_cpu_port(wl, sample_batch, steps, warmup, budget_s, ids)


def torch_eager_gpu_leg(wl, dims, b, dev, dev_pool, steps):
    """The reference's own operators (the oracle's functional port of its PyTorch path: F.embedding,
    embedding_bag, element-wise FM, cuBLAS fp32 Linear, torch Adam) run eagerly on the SAME GPU and the same
    batches: the 'library kernels to beat' of SURVEY 8(d).  A comparison only - never on the product path."""
    import torch

    from oracle import torch_port as TP

    p, opts, emb, fwd = _port_model(TP, wl, dev)
    offsets = torch.tensor([0] + dims[:-1]).cumsum(0)[None, :].to(dev)
    pool = [(x.long(), y) for x, y in dev_pool[:4]]
    for i in range(3):
        TP.train_step(p, opts, *pool[i % len(pool)], offsets, emb, wl["p_dropout"], sync=False, forward=fwd)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(steps):
        TP.train_step(p, opts, *pool[i % len(pool)], offsets, emb, wl["p_dropout"], sync=False, forward=fwd)
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / steps
    return {"ms_per_step": round(ms, 4), "samples_per_s": round(b / ms * 1e3, 1), "batch": b,
            "note": "oracle/torch_port.py (the reference's torch operators, fp32, TF32 off) eager on this GPU, "
                    "inputs resident, no loss read-back"}


def main_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the same workload and the same per-step batch as our arm's per-GPU batch, on this box's host cores
    sample = args.batch
    r = run_cpu_arm(wl, sample, max(args.steps, 3), max(args.warmup, 1), budget_s=150.0, ids=args.ids)
    line = {
        "impl": "reference",
        "metric": METRIC if wl["model"] == "deepfm" else "DCN-Mix train samples/s",
        "value": r["value"],
        "unit": "samples/s", "n_gpus": args.gpus, "steps": r["steps"], "warmup": max(args.warmup, 1),
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "batch_per_step": sample, "fields": len(wl["dims"]),
                   "rows": sum(wl["dims"]), "embedding": wl["emb"], "device": "cpu",
                   "note": "single process on the host cores (the reference has no multi-GPU path); same model, "
                           "optimizer recipe and batch as one GPU of our arm"},
        "cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": r["kind"],
                         "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [s.strip() for s in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                   "samples": len(sm)}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


def small_batch_leg(args, wl, dims, cfg, dev, R, crit, batch=None):
    """The reference yaml batch (configs/deepfm/*.yaml: 2048) is launch-latency-bound on a B200
    (~70 launches of a few microseconds each), so the same training step is also measured captured in
    ONE CUDA graph (static input buffers, capturable Adam, dropout stream position in device memory)."""
    import torch

    b = batch or args.small_batch
    torch.manual_seed(2023)
    cfg = {k: (dict(v) if isinstance(v, dict) else v) for k, v in cfg.items()}
    cfg["embedding_config"].pop("sparse", None)   # dense gradients: the sparse optimizers are not capturable
    model = R.get_ctr_model(dims, cfg).to(dev)
    model.train()
    opt_cfg = dict(wl["opt"])
    opt_cfg.update(capturable=True, fused_adam="rsb")
    opt_cfg.pop("fused_sparse", None)
    if opt_cfg.get("sparse"):
        opt_cfg.pop("sparse")          # the sparse optimizers are not capturable: dense Adam for this leg
    opts = R.get_optimizers(model, opt_cfg)
    pool = make_batches(dims, b, 8, 77, torch.int32)
    dev_pool = [(x.to(dev), y.to(dev)) for x, y in pool]
    sx, sy = dev_pool[0][0].clone(), dev_pool[0][1].clone()

    def step(x, y):
        logits = model(x)
        loss = crit(logits, y)
        for o in opts:
            o.zero_grad(set_to_none=True)
        loss.backward()
        for o in opts:
            o.step()
        return loss

    def run(fn, steps):
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            fn(i)
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / steps

    steps = max(args.steps, 20)
    for i in range(5):
        step(*dev_pool[i % 8])
    eager_ms = run(lambda i: step(*dev_pool[i % 8]), steps)

    from recsys_benchmark_b200.graphed import GraphedTrainStep

    gstep = GraphedTrainStep(model, opts, crit, sx, sy)
    static_loss = gstep.loss

    def replay(i):
        gstep(*dev_pool[i % 8])

    for i in range(5):
        replay(i)
    graph_ms = run(replay, steps)
    l1 = float(static_loss.item())
    replay(1)
    l2 = float(static_loss.item())
    # end to end through the graph: pinned host ids -> static device buffers -> one graph launch -> loss.item()
    host_pool = [(x.pin_memory(), y.pin_memory()) for x, y in pool]
    for i in range(3):
        gstep(*host_pool[i % 8]).item()
    e2e_ms = run(lambda i: gstep(*host_pool[i % 8]).item(), steps)
    return {"batch": b, "cuda_graph_e2e_ms_per_step": round(e2e_ms, 4),
            "cuda_graph_e2e_samples_per_s": round(b / e2e_ms * 1e3, 1), "eager_ms_per_step": round(eager_ms, 4), "eager_samples_per_s": round(b / eager_ms * 1e3, 1),
            "cuda_graph_ms_per_step": round(graph_ms, 4), "cuda_graph_samples_per_s": round(b / graph_ms * 1e3, 1),
            "loss_changes_between_replays": l1 != l2,
            "note": "whole step (fwd, BCE, bwd, Adam) captured in one CUDA graph; inputs copied into static buffers"}


def _peaks_all():
    out = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            d = json.load(fh)
        for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained"):
            if d.get(k):
                out[k] = float(d[k])
        out["source"] = "measured (MEASURED_PEAKS.json)"
    except (OSError, ValueError):
        pass
    return out


NVLINK_GBS = 770.0     # measured peer-copy bandwidth per direction per GPU on this pool (B200_PROFILING.md); nominal 900


def _hot_rows():
    from recsys_benchmark_b200.sharded import HOT_FIELD_ROWS
    return HOT_FIELD_ROWS


def kernel_rooflines(kern, ksteps, ms_kpass, world, b, n_fields, traffic_for, n_sharded_fields=None):
    """One roofline entry per timed C-ABI call name.  HBM-bound kernels: algorithmic bytes (SURVEY 8d) / CUDA-event
    time vs the measured copy bandwidth.  The GEMM: real bf16 MMA FLOPs (6 plane products per fp32 product, stated
    separately) vs the measured cuBLAS bf16 throughput sustained inside a long step."""
    pk = _peaks_all()
    out = {}
    for name, r in kern.items():
        if r["ms_avg"] <= 0:
            continue
        share = r["ms_total"] / ms_kpass
        base = {"calls_per_step": r["calls"] / ksteps, "ms_per_launch": round(r["ms_avg"], 4),
                "share_of_step": round(share, 4)}
        if name.startswith("gemm_planes"):
            flops = r["bytes_avg"]                       # planes.gemm stores 2*M*N*K*batch in the timer's slot
            tf = flops / (r["ms_avg"] * 1e-3) / 1e12
            mma = 3 if name.endswith("_h") else 6        # FP16X2 operands: 3 plane products; BF16X3: 6
            base.update(bound="tensor", achieved=round(mma * tf, 1), peak=pk["bf16_tflops_sustained"], unit="TFLOP/s",
                        frac=round(mma * tf / pk["bf16_tflops_sustained"], 4), fp32_equivalent_tflops=round(tf, 1),
                        mma_per_fp32_product=mma, traffic=None,
                        note=f"achieved = 16-bit tensor-core FLOPs actually issued ({mma} plane products per fp32 "
                             "product); peak = cuBLAS bf16 sustained (fp16 runs at the same rate)")
        elif r["bytes_avg"] > 0:
            gbs = r["bytes_avg"] / (r["ms_avg"] * 1e-3) / 1e9
            base.update(bound="hbm", achieved=round(gbs, 1), peak=pk["hbm_gbs"], unit="GB/s",
                        frac=round(gbs / pk["hbm_gbs"], 4), alg_bytes_per_launch=int(r["bytes_avg"]),
                        traffic=traffic_for(name))
            if name == "lookup_fwd_sharded" and world > 1:
                # rows fetched from peer shards: only the SHARDED fields' lookups leave the GPU (small fields are
                # replicated, sharded.HOT_FIELD_ROWS)
                nsf = n_fields if n_sharded_fields is None else n_sharded_fields
                remote = b * nsf * 64 * (world - 1) / world
                base["nvlink"] = {"remote_bytes_per_launch": int(remote), "achieved": round(remote / (r["ms_avg"] * 1e-3) / 1e9, 1),
                                  "peak": NVLINK_GBS, "unit": "GB/s",
                                  "frac": round(remote / (r["ms_avg"] * 1e-3) / 1e9 / NVLINK_GBS, 4),
                                  "note": "64-byte rows read from the peers' shards inside the gather kernel"}
        else:
            continue
        base["peak_source"] = pk["source"]
        out[name] = base
    return out


def run_workload(args, name, wl, dev, rank, world, R, primary):
    """Build the workload's model and measure it.  primary: every leg; otherwise value + kernel pass + the reference
    trainer loop only (the extra BASELINE configs reported beside the headline at N = 1)."""
    import torch
    import torch.distributed as dist

    import recsys_benchmark_b200.functional as RF
    from recsys_benchmark_b200 import _lib

    torch.manual_seed(2023)
    dims = wl["dims"]
    b = int(wl.get("batch", args.batch)) if not primary else args.batch
    cfg = model_config(wl)
    sharded = bool(wl.get("sharded", False))
    if sharded:
        from recsys_benchmark_b200.sharded import ShardedDCNMix, ShardedDeepFM

        if wl["model"] == "dcn_mix":
            model = ShardedDCNMix(dims, 16, [400, 400, 400], p_dropout=wl["p_dropout"],
                                  embedding_config=dict(wl["emb"])).to(dev)
        else:
            model = ShardedDeepFM(dims, 16, [400, 400, 400], p_dropout=wl["p_dropout"], use_batchnorm=wl["use_bn"],
                                  embedding_config=dict(wl["emb"])).to(dev)
    else:
        model = R.get_ctr_model(dims, dict(cfg)).to(dev)     # a copy: get_ctr_model pops "name" like the reference
    model.train()
    opts = R.get_optimizers(model, dict(wl["opt"]))
    crit = torch.nn.BCEWithLogitsLoss()
    params = [p for p in model.parameters() if p.requires_grad]

    def allreduce_grads():
        grads = [p.grad for p in params if p.grad is not None]
        flat = torch.cat([g.reshape(-1) for g in grads])
        dist.all_reduce(flat)
        flat.div_(world)
        off = 0
        views = []
        for g in grads:
            views.append(flat[off:off + g.numel()].view_as(g))
            off += g.numel()
        torch._foreach_copy_(grads, views)

    dump = primary and args.dump_outputs is not None
    last = {}

    def step(x, y):
        logits = model(x)
        loss = crit(logits, y)
        for o in opts:
            o.zero_grad()
        loss.backward()
        if sharded:
            model.sync_gradients()
        elif world > 1:
            allreduce_grads()
        for o in opts:
            o.step()
        if sharded:
            model.finish_step()
        if dump:
            last["logits"], last["loss"] = logits.detach(), loss.detach()
        return loss

    pool = make_batches(dims, b, args.pool, 2023 + rank, torch.int32, args.ids)
    dev_pool = [(x.to(dev), y.to(dev)) for x, y in pool]
    host_pool = [(x.pin_memory(), y.pin_memory()) for x, y in pool]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        sync_all()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            fn(i)
        e.record()
        sync_all()
        ms = s.elapsed_time(e)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    steps = args.steps if primary else max(5, min(args.steps, 10))
    # ---- value: inputs resident in HBM -------------------------------------------------
    for i in range(args.warmup):
        step(*dev_pool[i % len(dev_pool)])
    sampler = ClockSampler(dev.index) if (rank == 0 and primary) else None
    l0 = _lib.load().rsb_launch_count()
    ms_total = timed(lambda i: step(*dev_pool[i % len(dev_pool)]), steps)
    launches = _lib.load().rsb_launch_count() - l0
    outputs = snapshot_outputs(model, last) if dump else None
    # per-kernel CUDA-event timing in a SEPARATE pass of the same steps (an event pair around every C call keeps
    # consecutive kernels from overlapping their launch latency, so it must not sit inside the `value` region)
    timer = RF.KernelTimer()
    RF.set_timer(timer)
    ksteps = max(3, min(steps, 10))
    ms_kpass = timed(lambda i: step(*dev_pool[i % len(dev_pool)]), ksteps)
    RF.set_timer(None)
    kern = timer.summary()
    ms_step = ms_total / steps
    value = world * b / (ms_step * 1e-3)

    # ---- e2e: host buffers, H2D inside the timed region, loss read back every step ----------
    # (1) the reference trainer's loop verbatim (src/trainer/deepfm.py:44-62)
    def e2e_step(i):
        xh, yh = host_pool[i % len(host_pool)]
        loss = step(xh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True))
        return loss.item()

    for i in range(min(args.warmup, 3)):
        e2e_step(i)
    ms_e2e = timed(e2e_step, steps) / steps
    res = {"workload": name, "value": round(value, 1), "ms_per_step": round(ms_step, 4), "batch_per_gpu": b,
           "gpu_launches": int(launches), "steps": steps,
           "reference_trainer_loop": {"value": round(world * b / (ms_e2e * 1e-3), 1), "ms_per_step": round(ms_e2e, 4),
                                      "note": "src/trainer/deepfm.py:44-62 verbatim: blocking inputs.to(device) on the "
                                              "compute stream, loss.item() right after optimizer.step()"}}
    h2d = pool[0][0].numel() * pool[0][0].element_size() + pool[0][1].numel() * 4
    res["h2d_bytes_per_step"] = int(h2d)

    if primary:
        # (2) the library's own loop: DevicePrefetcher (H2D of step i+1 on a side stream under step i) and the loss
        #     copied D2H every step through DeferredScalar, consumed one step late
        from recsys_benchmark_b200.data import DeferredScalar, DevicePrefetcher

        class HostCycle:          # a re-iterable "loader" over the pinned host batches
            n = 0

            def __iter__(self):
                return (host_pool[i % len(host_pool)] for i in range(self.n))

        loader = HostCycle()
        prefetcher = DevicePrefetcher(loader, dev)

        def deferred_run(n):
            loader.n = n
            reader = DeferredScalar(dev)
            for xd, yd in prefetcher:
                reader.push(step(xd, yd))
            return reader.flush()

        deferred_run(3)
        sync_all()
        s_ev, e_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s_ev.record()
        deferred_run(steps)
        e_ev.record()
        sync_all()
        ms_df = s_ev.elapsed_time(e_ev) / steps
        if world > 1:
            t = torch.tensor([ms_df], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_df = float(t.item())
        res["pipelined_loop"] = {"value": round(world * b / (ms_df * 1e-3), 1), "ms_per_step": round(ms_df, 4),
                                 "note": "data.DevicePrefetcher + data.DeferredScalar (loss read one step late)"}
        # (3) the caches' record format end to end (SURVEY 8 f-2): [B, F+1] int32 blocks (label in column 0) staged by
        #     data.RecordStager - one H2D copy + the unpack kernel on a side stream - loss through DeferredScalar
        from recsys_benchmark_b200.data import RecordStager

        rec_pool = [torch.cat([y.to(torch.int32).unsqueeze(1), x], 1).contiguous().pin_memory() for x, y in pool]

        class RecCycle:
            n = 0

            def __iter__(self):
                return (rec_pool[i % len(rec_pool)] for i in range(self.n))

        rloader = RecCycle()
        stager = RecordStager(rloader, dev)

        def record_run(n):
            rloader.n = n
            reader = DeferredScalar(dev)
            for xd, yd in stager:
                reader.push(step(xd, yd))
            return reader.flush()

        record_run(3)
        sync_all()
        s_ev, e_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s_ev.record()
        record_run(steps)
        e_ev.record()
        sync_all()
        ms_rs = s_ev.elapsed_time(e_ev) / steps
        if world > 1:
            t = torch.tensor([ms_rs], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_rs = float(t.item())
        res["record_staged_loop"] = {"value": round(world * b / (ms_rs * 1e-3), 1), "ms_per_step": round(ms_rs, 4),
                                     "h2d_bytes_per_step": int(rec_pool[0].numel() * 4),
                                     "note": "lmdb record blocks [B, F+1] int32 -> data.RecordStager (pinned copy, one H2D, "
                                             "rsb_records_unpack) + data.DeferredScalar"}
        res["clocks"] = sampler.stop() if sampler else None

    # ---- rooflines -----------------------------------------------------------------------------
    unique_rows = None
    if wl["opt"].get("fused_sparse") and "segment_reduce_apply" in kern and not sharded:
        # fused SparseAdam: + read/write of w, m, v per UNIQUE row (SURVEY 8d: 6*D*4 B); U is counted here, on batch 0,
        # outside the timed region (the product path never synchronises to learn it)
        offs = torch.tensor([0] + dims[:-1]).cumsum(0)
        unique_rows = int(torch.unique(pool[0][0].long() + offs).numel())
        kern["segment_reduce_apply"]["bytes_avg"] += 6 * 16 * 4 * unique_rows
    res["unique_rows_per_step"] = unique_rows
    traffic_tab = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as fh:
            traffic_tab = json.load(fh).get(name, {})
    n_sharded_fields = None
    if sharded:
        from recsys_benchmark_b200.sharded import HOT_FIELD_ROWS
        # small fields are replicated for the vanilla table only; the variants shard every field
        n_sharded_fields = (sum(1 for d in dims if d > HOT_FIELD_ROWS)
                            if (world > 1 and wl["emb"]["name"] == "vanilla") else len(dims))
    roofs = kernel_rooflines(kern, ksteps, ms_kpass, world, b, len(dims), lambda k: traffic_tab.get(k),
                             n_sharded_fields)
    top = sorted(roofs, key=lambda k: -roofs[k]["share_of_step"])
    res["roofline_top3"] = [dict(kernel=k, **roofs[k]) for k in top[:3]]
    res["roofline"] = dict(kernel=top[0], **roofs[top[0]]) if top else None
    hot = [k for k in top if k.startswith(("lookup_", "segment_", "sort_rows", "small_table", "csr_lookup", "dhe_"))]
    res["roofline_hot_path"] = [dict(kernel=k, **roofs[k]) for k in hot[:4]]
    res["kernels"] = {k: {"calls_per_step": r["calls"] / ksteps, "ms_avg": round(r["ms_avg"], 4),
                          "share_of_step": round(r["ms_total"] / ms_kpass, 4)} for k, r in kern.items()}
    res["_objects"] = (model, opts, crit, cfg, dev_pool, pool)
    res["_outputs"] = outputs
    return res


DUMP_MAX_ELEMENTS = 1 << 20      # per array: at most 4 MB of float32


def snapshot_outputs(model, last):
    """What the last timed step handed back: its loss and logits, and the model's parameters and floating-point
    buffers as the optimizer step left them.  An array of more than DUMP_MAX_ELEMENTS keeps a fixed, seeded
    sample of its rows (sorted row ids, the same for every run of the same shape)."""
    import torch

    out = {"loss": last["loss"].float().reshape(1), "logits": last["logits"].float()}
    tensors = list(model.named_parameters()) + [(n, b) for n, b in model.named_buffers() if b.is_floating_point()]
    for name, t in tensors:
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMENTS:
            keep = max(1, DUMP_MAX_ELEMENTS // max(1, t[0].numel()))
            g = torch.Generator().manual_seed(0)
            rows = torch.randperm(t.shape[0], generator=g)[:keep].sort().values
            t = t[rows.to(t.device)]
        out[name] = t.float()
    return {k: v.cpu().numpy() for k, v in out.items()}


def write_outputs(outputs, out_dir, max_bytes=64 << 20):
    import numpy as np

    total = sum(a.nbytes for a in outputs.values())
    if total > max_bytes:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {max_bytes}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def sharded_parity_check(dims, dev, rank, world, R):
    """In-run parity of the row-sharded path (SURVEY 8e "Parity"): (1) the sharded forward over local + peer shards
    gives the SAME logits, bit for bit, as the single-GPU gather on this rank's batch; (2) after two data-parallel
    training steps the gathered table equals the single-GPU model trained on the global batch within 1e-4.
    Dropout and BatchNorm are off here (dropout draws per-rank masks; BatchNorm statistics are per-rank by design)."""
    import torch
    import torch.distributed as dist

    from recsys_benchmark_b200.sharded import ShardedDeepFM

    torch.manual_seed(77)
    bl = 4096
    sh = ShardedDeepFM(dims, 16, [400, 400, 400], p_dropout=0.0, use_batchnorm=False).to(dev)
    full = R.get_ctr_model(dims, dict(num_factor=16, hidden_sizes=[400, 400, 400], p_dropout=0.0, use_batchnorm=False,
                                      embedding_config={"name": "vanilla"})).to(dev)
    st = {k: v for k, v in sh.state_dict().items() if not k.startswith("embedding.")}
    full.load_state_dict(st, strict=False)
    with torch.no_grad():
        full.embedding.get_weight().copy_(sh.embedding.gather_full_weight())
    g = torch.Generator().manual_seed(5)
    xg = torch.stack([torch.randint(0, d, (bl * world,), generator=g) for d in dims], 1).int()
    yg = torch.randint(0, 2, (bl * world,), generator=g).float()
    xl, yl = xg[rank::world].to(dev), yg[rank::world].to(dev)
    xg, yg = xg.to(dev), yg.to(dev)
    crit = torch.nn.BCEWithLogitsLoss()
    o_sh = torch.optim.Adam(sh.parameters(), lr=1e-3)
    o_full = torch.optim.Adam(full.parameters(), lr=1e-3)
    out = {"world": world, "local_batch": bl}
    with torch.no_grad():
        # the sharded gather (local + peer shards over NVLink) against the single-GPU gather: bit for bit
        e_sh, y_sh = sh.embedding.lookup(xl, sh.offsets, sh.fc.weight, sh._bias)
        e_full, y_full = full.embedding.lookup(xg, full.offsets, full.fc.weight, full._bias)
        out["gather_fm_bit_identical"] = bool(torch.equal(e_sh, e_full[rank::world]) and torch.equal(y_sh, y_full[rank::world]))
    for s in range(2):
        lg_sh = sh(xl)
        lg_full = full(xg)
        if s == 0:
            # (the MLP's one-output Linear is a library GEMV whose kernel choice depends on the batch size: the logits
            #  of a 4096-row and an 8192-row call agree to fp32 rounding, not necessarily bit for bit)
            ref = lg_full[rank::world]
            out["logits_max_rel_err"] = float((lg_sh - ref).abs().max() / ref.abs().max())
            out["logits_bit_identical"] = bool(torch.equal(lg_sh, ref))
        o_sh.zero_grad()
        crit(lg_sh, yl).backward()
        sh.sync_gradients()
        o_sh.step()
        sh.finish_step()
        o_full.zero_grad()
        crit(lg_full, yg).backward()
        o_full.step()
    w_sh, w_full = sh.embedding.gather_full_weight(), full.embedding.get_weight().detach()
    err = float((w_sh - w_full).abs().max() / w_full.abs().max())
    flags = torch.tensor([float(out["gather_fm_bit_identical"]), float(out["logits_bit_identical"]),
                          -out["logits_max_rel_err"], -err], device=dev)
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)          # worst rank
    out["gather_fm_bit_identical"] = bool(flags[0].item() == 1.0)
    out["logits_bit_identical"] = bool(flags[1].item() == 1.0)
    out["logits_max_rel_err"] = float(-flags[2].item())
    err = float(-flags[3].item())
    out["table_rel_err_after_2_steps"] = err
    out["ok"] = bool(out["gather_fm_bit_identical"] and out["logits_max_rel_err"] < 1e-5 and err < 1e-4)
    del sh, full
    torch.cuda.empty_cache()
    return out


def main_ours(args, wl):
    import torch
    import torch.distributed as dist

    import __graft_entry__ as G

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (our arm) needs a CUDA device: there is no CPU fallback for the hot path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL_DEBUG=VERSION makes NCCL printf() its version banner to stdout: keep stdout to the ONE JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        G.build()
    if world > 1:
        dist.barrier()
    import recsys_benchmark_b200 as R

    sharded = bool(wl.get("sharded", False))
    parity = None
    if sharded and not args.no_parity_check and wl["model"] == "deepfm" and wl["emb"]["name"] == "vanilla":
        # (the sharded variants are held to the single-device model by tests/test_gpu_sharded_kinds.py)
        try:
            parity = sharded_parity_check(wl["dims"], dev, rank, world, R)
        except Exception as exc:  # noqa: BLE001 - reported, never hidden
            parity = {"ok": False, "error": f"{type(exc).__name__}: {exc}"[:300]}
    res = run_workload(args, args.workload, wl, dev, rank, world, R, primary=True)
    model, opts, crit, cfg, dev_pool, pool = res.pop("_objects")
    outputs = res.pop("_outputs")
    if outputs is not None and rank == 0:
        write_outputs(outputs, args.dump_outputs)
    dims, b = wl["dims"], args.batch

    # ---- reference-yaml batch (2048): launch-bound -> whole step captured in a CUDA graph -------------
    small = None
    if world == 1 and args.small_batch > 0 and not sharded:
        try:
            small = small_batch_leg(args, wl, dims, cfg, dev, R, crit)
        except Exception as exc:  # noqa: BLE001 - a secondary number must never break the main line
            small = {"batch": args.small_batch, "error": f"{type(exc).__name__}: {exc}"[:300]}
    # ---- the reference's torch operators, eager, on this GPU (comparison only) ----------------------
    eager = None
    if world == 1 and not args.no_torch_eager and wl["emb"].get("name", "vanilla") in PORT_EMBEDDINGS:
        try:
            eager = torch_eager_gpu_leg(wl, dims, b, dev, dev_pool, max(3, min(args.steps, 10)))
        except Exception as exc:  # noqa: BLE001
            eager = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    del model, opts, dev_pool
    torch.cuda.empty_cache()

    # ---- the other BASELINE.json configs, beside the headline (N = 1 only) -----------------------------
    others = {}
    if world == 1 and not args.no_other_configs:
        for other in OTHER_CONFIGS:
            if other == args.workload:
                continue
            try:
                r = run_workload(args, other, WORKLOADS[other], dev, rank, world, R, primary=False)
                r.pop("_objects")
                r.pop("_outputs")
                r.pop("kernels", None)
                if other == "deepfm_qr_criteo" and args.small_batch > 0:
                    try:
                        r["small_batch"] = small_batch_leg(args, WORKLOADS[other], WORKLOADS[other]["dims"],
                                                           model_config(WORKLOADS[other]), dev, R, crit)
                    except Exception as exc:  # noqa: BLE001
                        r["small_batch"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
                others[other] = r
            except Exception as exc:  # noqa: BLE001
                others[other] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- cpu baseline (the reference's CPU path), rank 0, N=1 only ----------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = run_cpu_arm(wl, min(args.cpu_batch, b), 6, 1, budget_s=20.0, ids=args.ids)
        cpu = {"value": round(r["value"], 1), "unit": "samples/s", "cores": r["cores"], "kind": r["kind"],
               "sample": r["sample"]}

    e2e_ref = res["reference_trainer_loop"]
    line = {
        "metric": METRIC if wl["model"] == "deepfm" else "DCN-Mix train samples/s",
        "value": res["value"], "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "global_batch": world * b, "batch_per_gpu": b, "fields": len(dims),
                   "rows": sum(dims), "embedding": wl["emb"], "num_factor": 16, "mlp": [400, 400, 400],
                   "use_batchnorm": wl["use_bn"], "optimizer": wl["opt"],
                   "ids": f"int32, {'Zipf(1.05) clipped' if args.ids == 'zipf' else 'uniform'} per field, seed 2023",
                   "parallelism": (f"row-sharded table x{world} (rows r % {world} on rank r, forward gather over NVLink "
                                   f"peer memory, gradients pushed to the owner shard"
                                   + (f"; the {sum(1 for d in dims if d <= _hot_rows())} fields of <= {_hot_rows()} ids "
                                      f"replicated" if world > 1 else "")
                                   + f") + dp{world} dense allreduce"
                                   if sharded else (f"dp{world} (replicated tables, flat grad allreduce)"
                                                    if world > 1 else "single")),
                   "l2": f"{args.pool} distinct batches cycled; per-step traffic "
                         f"{round(b * 13.4e3 / 1e6)} MB vs 126 MB L2 (no flush)"},
        "clocks": res.get("clocks"),
        # the headline end-to-end number is the reference trainer's own loop (blocking H2D, loss.item() every step);
        # the library's pipelined loop is reported beside it
        "e2e": {"value": e2e_ref["value"], "unit": "samples/s", "ms_per_step": e2e_ref["ms_per_step"],
                "h2d_bytes_per_step": res["h2d_bytes_per_step"], "d2h_bytes_per_step": 4,
                "loop": e2e_ref["note"], "pipelined_loop": res.get("pipelined_loop"),
                "record_staged_loop": res.get("record_staged_loop")},
        "reference_trainer_loop": e2e_ref,
        "gpu_launches": res["gpu_launches"],
        "roofline": res["roofline"],
        "roofline_top3": res["roofline_top3"],
        "roofline_hot_path": res["roofline_hot_path"],
        "parity_check": parity,
        "kernels": res["kernels"],
        "cpu_baseline": cpu,
        "small_batch": small if small is not None else others.get("deepfm_qr_criteo", {}).get("small_batch"),
        "torch_eager_gpu": eager,
        "unique_rows_per_step": res["unique_rows_per_step"],
        "other_configs": others,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# BASELINE.json configs reported beside the headline at N = 1: [1] QR, [0] full table on one GPU (fused SparseAdam),
# [2] DCN-Mix Avazu, [3] PEP / OptEmbed KDD, and the SURVEY 8(d) roofline shape (17 M rows, table >> L2)
OTHER_CONFIGS = ["deepfm_qr_criteo", "deepfm_full_criteo", "dcnmix_full_avazu", "deepfm_pep_kdd", "deepfm_optembed_kdd",
                 "deepfm_full_roofline"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="deepfm_full_criteo_sharded", choices=sorted(WORKLOADS),
                    help="default: BASELINE.json configs[4], the full Criteo-shaped table row-sharded over the N GPUs "
                         "(N = 1: one shard), so that the 1/2/4/8-GPU lines measure the same model")
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU per step (default: 65536, or the "
                                                            "workload's own batch)")
    ap.add_argument("--pool", type=int, default=8, help="distinct synthetic batches cycled through")
    ap.add_argument("--cpu-batch", type=int, default=65536, help="samples per CPU step of the cpu_baseline leg "
                                                                 "(default: the GPU arm's own batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true", help="skip the in-run sharded parity check")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="N = 1: do not also measure the other BASELINE configs (QR, DCN-Mix, PEP, OptEmbed, roofline shape)")
    ap.add_argument("--ids", default="uniform", choices=["uniform", "zipf"],
                    help="per-field id distribution: uniform, or Zipf(1.05) clipped to the field size")
    ap.add_argument("--no-torch-eager", action="store_true", help="skip the torch-eager-on-GPU comparison leg")
    ap.add_argument("--small-batch", type=int, default=2048,
                    help="also time this (reference yaml) batch eagerly and as one CUDA graph; 0 = skip")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, logits and model state after the last timed step as DIR/<name>.npy "
                         "(float32; arrays over 2^20 elements as a seeded row sample), so that two builds can be "
                         "compared output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = WORKLOADS[args.workload]
    if args.batch is None:
        args.batch = int(wl.get("batch", 65536))
    if args.impl == "reference":
        main_reference(args, wl)
    else:
        main_ours(args, wl)


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the tree bench.py runs from may be read-only: no __pycache__ written into it
    main()
