"""bench.py's reference arm runs on host cores only (it is the one bench leg a CPU box can execute): check that it follows the
JSON-line contract of the driver -- one line, the BASELINE.json metric, the keys and types the base contract names."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert j["impl"] == "reference" and j["unit"] == "pairs/s" and j["higher_is_better"] is True and j["scaling"] == "weak"
    assert "pairs/sec" in j["metric"] and "36 regions" in j["metric"]
    assert str(base.get("metric", "")).split()[0].lower() in j["metric"].lower() or "pairs" in j["metric"]
    assert j["n_gpus"] == 1 and j["steps"] == 1 and j["value"] > 0 and j["ms_per_step"] > 0
    assert j["data"] == "synthetic" and j["dtype"] == "f32" and j["vs_baseline"] is None
    assert "workload" in j["config"] and "model" not in j["config"]
    cb = j["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == j["value"] and cb["sample"]
    e2e = j["e2e"]
    assert e2e["value"] == j["value"] and e2e["unit"] == j["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_gpu_arm_fails_loudly_without_a_gpu():
    """No CUDA device: the product arm must refuse (non-zero exit, no JSON line) instead of falling back to anything."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--no-cpu-baseline"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_keeps_a_fixed_row_sample_within_the_budget(tmp_path, monkeypatch):
    """Under the budget every output is written whole, as float32; over it every output keeps the same share of its rows, and
    the same rows on every call, so dumps of two runs stay comparable."""
    import numpy as np
    import torch
    import bench
    a, b = torch.randn(100, 30, dtype=torch.float64), torch.randn(50, 4, 2)
    bench.dump_outputs(str(tmp_path / "all"), {"a": a, "b": b})
    whole = np.load(tmp_path / "all" / "a.npy")
    assert whole.dtype == np.float32 and np.array_equal(whole, a.float().numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", (a.numel() + b.numel()) * 4 // 4)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), {"a": a, "b": b})
    sa, sb = np.load(tmp_path / "s1" / "a.npy"), np.load(tmp_path / "s1" / "b.npy")
    assert sa.shape == (25, 30) and sb.shape == (12, 4, 2)
    assert sa.nbytes + sb.nbytes <= bench.DUMP_BYTES
    assert np.array_equal(sa, np.load(tmp_path / "s2" / "a.npy")) and np.array_equal(sb, np.load(tmp_path / "s2" / "b.npy"))
    rows = {tuple(r) for r in a.float().numpy()}
    assert all(tuple(r) in rows for r in sa)


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs writes what the last of the --steps timed steps returned: 5 steps over 3 rotating input batches end on
    batch (5 - 1) % 3 = 1, and a fresh engine given that batch returns the same bits."""
    import numpy as np
    import vilbert_b200 as vb
    from vilbert_b200 import synthetic as S
    out_dir = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "5", "--warmup", "1", "--rotate", "3", "--batch", "8",
                        "--dtype", "bf16", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 5
    assert sorted(os.listdir(out_dir)) == ["vil_prediction.npy"]
    got = np.load(out_dir / "vil_prediction.npy")
    assert got.dtype == np.float32 and got.shape == (8, 3129)
    cfg = vb.BertConfig(task_specific_tokens=True, visualization=True)
    model = vb.VILBertForVLTasks.from_pretrained(S.synthetic_state_dict(cfg, seed=42), config=cfg, num_labels=3129,
                                                 compute_dtype="bf16").eval().cuda(0)
    req = S.synthetic_request(8, 30, 36, seed=1234 + 1)
    want = model(*[t.cuda() for t in req], select=vb.OUT_VIL_PREDICTION)[0].cpu().numpy()
    model.close()
    assert np.array_equal(got, want)
