"""The reference arm of bench.py (`--impl reference`) runs on host cores only, so its JSON contract can be checked without a GPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "points/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["metric"] == "CRFConv fwd+bwd points/s (N=40960,k=16)" and d["value"] > 0 and d["n_gpus"] == 1
    assert "workload" in d["config"] and "model" not in d["config"]
    cb, e2e = d["cpu_baseline"], d["e2e"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_product_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: without CUDA the product arm must fail loudly instead of measuring something else."""
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode != 0
    assert not [l for l in r.stdout.strip().splitlines() if l.startswith("{") and '"value"' in l]


def test_dump_outputs_writes_float32_on_fixed_rows(tmp_path):
    """--dump-outputs: the same sampled rows in every run, every array written as float32; --steps 0 is refused."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    rows = bench.sample_rows(torch, 6 * 40960, 32768, "cpu")
    assert torch.equal(rows, bench.sample_rows(torch, 6 * 40960, 32768, "cpu")) and bool((rows[1:] > rows[:-1]).all())
    bench.dump_outputs(str(tmp_path), {"loss": torch.tensor([2.5], dtype=torch.float64), "out_rows": rows})
    assert np.load(tmp_path / "loss.npy").dtype == np.float32 and np.array_equal(np.load(tmp_path / "out_rows.npy"), rows.numpy())
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_algorithmic_bytes_match_the_survey():
    """SURVEY.md §8(d): 79,298,560 algorithmic bytes per 40,960-point cloud for one CRF layer fwd+bwd at S1 — the roofline numerator."""
    sys.path.insert(0, ROOT)
    import bench
    assert bench.ALGO_BYTES_PER_CLOUD == 79_298_560
    assert bench.crf_layer_algo_bytes(40960, 10240, 128, 64, 64, 16) == bench.ALGO_BYTES_PER_CLOUD
    a3 = bench.network_algo_bytes(40960, 13)
    assert 230e6 < a3 < 240e6                                  # DESIGN.md §6: 236 MB per cloud for the whole network at C3
    assert bench.network_algo_bytes(45056, 19) > a3 and bench.network_algo_bytes(65536, 8) > a3
