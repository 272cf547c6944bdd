"""bench.py contract (driver-facing): the reference arm runs on the host CPU and prints ONE json line with the agreed keys."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, GIMMVFI_CPU_THREADS="8", GIMMVFI_CPU_SAMPLE="128x160")   # small sample: this test checks the contract, not the number
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("interpolated frames/sec") and d["unit"] == "frames/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_of_the_f_configs_says_unavailable():
    """--config f2k / f4k (GIMM-VFI-F): the reference arm cannot run offline (timm + pretrained FlowFormer) - one json line, exit 0."""
    for cfg in ("f2k", "f4k"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", cfg, "--impl", "reference"],
                           capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
        assert len(lines) == 1
        d = json.loads(lines[0])
        assert d["impl"] == "reference" and isinstance(d.get("unavailable"), str) and d["unavailable"]


def test_reference_arm_times_steps_and_dumps_outputs(tmp_path):
    """--steps sets the number of timed forwards; --dump-outputs writes the last one's outputs, which are those of the seeded input."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gimmvfi_r_oracle as O
    from gimmvfi_b200.synth import synth_batch
    from gimmvfi_b200.weights import random_state_dict

    env = dict(os.environ, GIMMVFI_CPU_THREADS="8", GIMMVFI_CPU_SAMPLE="128x160")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "0",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == d["steps_timed"] == 3
    with torch.no_grad():
        ref = O.gimmvfi_r_forward(random_state_dict(0), synth_batch(1, 128, 160, seed=100), [(O.sample_coord_input(1, (128, 160), [0.5]), None)],
                                  [0.5 * torch.ones(1)])
    for name, t in bench.flatten_outputs(ref).items():
        a = np.load(tmp_path / (name + ".npy"))
        assert a.dtype == np.float32 and a.shape == tuple(t.shape) and np.isfinite(a).all(), name
    # this process may run on more CPU threads than the bench's 8, which reorders sums that RAFT's 20 iterations amplify in the flows;
    # the frame stays within the parity tolerance
    assert np.abs(np.load(tmp_path / "imgt_pred_0.npy") - ref["imgt_pred"][0].numpy()).max() <= 1e-3


def test_dump_outputs_samples_large_outputs_within_the_budget(tmp_path):
    g = torch.Generator().manual_seed(0)
    out = {"imgt_pred": [torch.rand(1, 3, 1088, 1920, generator=g) for _ in range(7)], "raft_flow": torch.rand(1, 2, 2, 136, 240, generator=g),
           "nflow": torch.rand(4, dtype=torch.float64, generator=g)}
    bench.dump_outputs(str(tmp_path / "a"), out)
    bench.dump_outputs(str(tmp_path / "b"), out)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["imgt_pred_%d.npy" % i for i in range(7)] + ["nflow.npy", "raft_flow.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 << 20
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    assert np.array_equal(np.load(tmp_path / "a" / "raft_flow.npy"), out["raft_flow"].numpy())
    nflow = np.load(tmp_path / "a" / "nflow.npy")
    assert nflow.dtype == np.float64 and np.array_equal(nflow, out["nflow"].numpy())
    s = np.load(tmp_path / "a" / "imgt_pred_3.npy")
    assert s.dtype == np.float32 and s.ndim == 1 and 0 < s.size < out["imgt_pred"][3].numel()
    idx = np.sort(np.random.default_rng(0).choice(out["imgt_pred"][3].numel(), s.size, replace=False))
    assert np.array_equal(s, out["imgt_pred"][3].numpy().reshape(-1)[idx])
