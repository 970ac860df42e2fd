"""bench.py contract checks that need no GPU: the reference arm's JSON line, the synthetic id generators and
the workload table (SURVEY.md section 8d)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--batch", "256"], capture_output=True, text=True, timeout=600,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["value"] > 0 and d["gpu_launches"] == 0
    # the unmodified reference classes when baseline/_ref is staged (build container and GPU box), else the oracle port
    assert d["cpu_baseline"]["kind"] == ("reference" if bench._reference_available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["config"]["batch_per_step"] == 256
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "deepfm_full_criteo_sharded" and d["vs_baseline"] is None


def test_reference_arm_is_silent_on_non_zero_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_synthetic_id_generators():
    dims = [4, 1000, 200000]
    (x, y), = bench.make_batches(dims, 8192, 1, 2023, torch.int32)
    assert x.dtype == torch.int32 and tuple(x.shape) == (8192, 3) and set(y.unique().tolist()) <= {0.0, 1.0}
    assert all(int(x[:, i].max()) < d and int(x[:, i].min()) >= 0 for i, d in enumerate(dims))
    (z, _), = bench.make_batches(dims, 8192, 1, 2023, torch.int64, "zipf")
    assert all(int(z[:, i].max()) < d and int(z[:, i].min()) >= 0 for i, d in enumerate(dims))
    counts = np.bincount(z[:, 2].numpy(), minlength=16)[:16]
    assert counts[0] > counts[1] > counts[3] > counts[15] > 0          # heavy head, Zipf(1.05)
    assert z[:, 2].unique().numel() < x[:, 2].unique().numel()          # far more duplicates than uniform ids
    again = bench.make_batches(dims, 8192, 1, 2023, torch.int64, "zipf")[0][0]
    assert torch.equal(z, again)                                        # seeded


def test_dump_outputs_snapshot_is_seeded_float_and_bounded(tmp_path):
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Embedding(bench.DUMP_MAX_ELEMENTS // 4 + 3, 8), torch.nn.BatchNorm1d(8))
    last = {"logits": torch.randn(64), "loss": torch.tensor(0.5)}
    a = bench.snapshot_outputs(model, last)
    b = bench.snapshot_outputs(model, last)
    assert set(a) == {"loss", "logits", "0.weight", "1.weight", "1.bias", "1.running_mean", "1.running_var"}
    assert all(v.dtype == np.float32 for v in a.values())
    assert a["loss"].shape == (1,) and a["logits"].shape == (64,)
    table = model[0].weight.detach().numpy()
    assert a["0.weight"].shape == (bench.DUMP_MAX_ELEMENTS // 8, 8)
    assert np.array_equal(a["0.weight"], b["0.weight"])                   # the same rows every time
    rows = [int(np.flatnonzero((table == r).all(1))[0]) for r in a["0.weight"][:5]]
    assert rows == sorted(rows)
    bench.write_outputs(a, str(tmp_path / "out"))
    assert np.array_equal(np.load(tmp_path / "out" / "0.weight.npy"), a["0.weight"])
    with pytest.raises(RuntimeError):
        bench.write_outputs(a, str(tmp_path / "small"), max_bytes=1024)


def test_workload_table_matches_the_survey_shapes():
    assert sum(bench.CRITEO_DIMS) == 1086810 and len(bench.CRITEO_DIMS) == 39
    assert len(bench.AVAZU_DIMS) == 22 and len(bench.KDD_DIMS) == 11 and sum(bench.KDD_DIMS) == 6_000_000
    assert sum(bench.ROOFLINE_DIMS) >= 16_000_000 and len(bench.ROOFLINE_DIMS) == 39
    wl = bench.WORKLOADS
    assert wl["deepfm_qr_criteo"]["emb"] == {"name": "qr", "divider": 5} and not wl["deepfm_qr_criteo"]["use_bn"]
    assert wl["dcnmix_full_avazu"]["model"] == "dcn_mix" and wl["deepfm_full_criteo_sharded"]["sharded"]
    for name, w in wl.items():
        assert w["model"] in ("deepfm", "dcn_mix") and "opt" in w and "dims" in w, name
    # the sharded variants of SURVEY 8e keep their unsharded twins' shapes and optimizer recipes
    for sh, base in (("deepfm_pep_kdd_sharded", "deepfm_pep_kdd"), ("dcnmix_full_avazu_sharded", "dcnmix_full_avazu")):
        assert wl[sh]["sharded"] and wl[sh]["dims"] == wl[base]["dims"] and wl[sh]["emb"] == wl[base]["emb"]
        assert wl[sh]["opt"] == wl[base]["opt"]
    assert wl["deepfm_qr_criteo_sharded"]["emb"] == wl["deepfm_qr_criteo"]["emb"]
    # every dense optimizer recipe asks for the library's one-launch Adam
    assert all(w["opt"].get("fused_adam") == "rsb" for w in wl.values())
