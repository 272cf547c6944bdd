"""Parity AT THE BENCHMARKED CONFIGURATIONS (VERDICT r01 item 1): the CUDA path through the drop-in GIMMVFI_R against
fixtures produced by the UNMODIFIED reference on CPU at those sizes (oracle/make_golden_big.py, stride-8 sub-sampled):

  big_r_1088x1920_t0.5       BASELINE config 2 — the exact pair bench.py times (synth seed 100)
  big_r_736x1280_t0.5        BASELINE config 5 — one 1280x720 pair padded to 736x1280
  big_r_ds0.5_1088x2048_T7   the reference's 2K video setting: ds_factor 0.5, N = 8 -> 7 timesteps (README.md:87-96)
  big_r_demo_736x864_t0.5    the reference's own demo frames (demo/input_frames), replicate-padded by InputPadder(.., 32)

Contract (BASELINE.json north_star): max |d imgt_pred| <= 1e-3 in the DEFAULT precision mode, every pixel of the sub-sampled
grid; additionally the PSNR-equivalent (RMSE) and the flow fields' percentiles are bounded as in test_forward_gpu.py."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gimmvfi_r_oracle as O
from conftest import GOLDEN_DIR
from gimmvfi_b200 import GIMMVFI_R
from gimmvfi_b200.synth import synth_batch

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL_IMG = 1e-3

with open(os.path.join(GOLDEN_DIR, "manifest_big.json")) as _f:
    MANIFEST = json.load(_f)


@pytest.fixture(scope="module")
def model(weights0):
    m = GIMMVFI_R(seed=0).to(DEV).eval()
    m.load_state_dict(weights0, strict=True)
    if os.environ.get("GIMMVFI_TEST_MODE"):   # builder experiments only (e.g. validating a candidate default); the driver runs the shipped default
        m.tensor_cores = int(os.environ["GIMMVFI_TEST_MODE"])
    return m   # default precision mode (model.tensor_cores as shipped)


def case_input(meta, g):
    if meta["input_seed"] is None:   # demo frames travel inside the fixture (uint8 RGB): video_Nx.py:46-50,151-156
        x = torch.from_numpy(g["frames_u8"].copy()).permute(0, 3, 1, 2).float() / 255.0
        ht, wd = x.shape[-2:]
        ph, pw = (((ht // 32) + 1) * 32 - ht) % 32, (((wd // 32) + 1) * 32 - wd) % 32
        x = F.pad(x, [pw // 2, pw - pw // 2, ph // 2, ph - ph // 2], mode="replicate")
        return torch.stack([x[0], x[1]], 1).unsqueeze(0).contiguous()
    return synth_batch(1, meta["H"], meta["W"], seed=meta["input_seed"])


def stats(a, b):
    d = (a.double() - b.double()).abs().flatten()
    return d.max().item(), torch.quantile(d[:: max(1, d.numel() // 2_000_000)], 0.9999).item(), d.pow(2).mean().sqrt().item()


@pytest.mark.parametrize("name", sorted(MANIFEST))
def test_benchmarked_config_matches_reference(name, model):
    meta = MANIFEST[name]
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    s = int(g["stride"])
    H, W, ts, ds = meta["H"], meta["W"], meta["timesteps"], meta["ds_factor"]
    xs = case_input(meta, g)
    assert tuple(xs.shape) == (1, 3, 2, H, W)
    ratio = 1.0 if ds is None else ds
    coord = [(model.sample_coord_input(1, (H, W), [t], device=DEV, upsample_ratio=ratio), None) for t in ts]
    tt = [t * torch.ones(1, device=DEV) for t in ts]
    out = model(xs.to(DEV), coord, t=tt, ds_factor=ds)
    torch.cuda.synchronize()
    checks = []
    for i in range(len(ts)):
        img = out["imgt_pred"][i]
        assert tuple(img.shape) == (1, 3, H, W) and torch.isfinite(img).all()
        mx, p9999, rmse = stats(img[..., ::s, ::s].cpu(), torch.from_numpy(g["imgt_pred_%d" % i]))
        checks += [("imgt_pred[%d] max" % i, mx, TOL_IMG), ("imgt_pred[%d] rmse" % i, rmse, 2e-4)]
        mean_d = abs(img.double().sum().item() - float(g["imgt_pred_sum_%d" % i])) / img.numel()
        checks.append(("imgt_pred[%d] |mean diff|" % i, mean_d, 1e-4))
        ft = out["flowt"][i]
        ft = ft if ft.dim() == 4 else ft[None]
        _, fp, frm = stats(ft[..., ::s, ::s].cpu(), torch.from_numpy(g["flowt_%d" % i]))
        checks += [("flowt[%d] p99.99" % i, fp, 1e-1), ("flowt[%d] rmse" % i, frm, 2e-2)]
    rmx = stats(out["raft_flow"][..., ::s, ::s].cpu(), torch.from_numpy(g["raft_flow"]))[0]
    checks.append(("raft_flow max (|flow| up to %.1f px)" % float(g["raft_flow_absmax"]), rmx, 1e-2))
    report = "; ".join("%s %.3e (<= %.1e)%s" % (n, v, lim, "" if v <= lim else " FAIL") for n, v, lim in checks)
    print(name, "mode", model.tensor_cores, report)
    assert all(v <= lim for _, v, lim in checks), report


def test_bench_dump_outputs_hold_the_timed_forward(tmp_path, weights0):
    """bench.py --dump-outputs on the GPU path: the files hold the last timed forward's outputs on the seeded input (synth seed 100,
    weights seed 0) - imgt_pred within the parity tolerance of the CPU oracle on the same input."""
    H, W = 128, 160
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--height", str(H), "--width", str(W), "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--no-torch-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2 and d["config"]["height"] == H and d["config"]["width"] == W
    names = sorted(p.name for p in tmp_path.iterdir())
    assert {"imgt_pred_0.npy", "flowt_0.npy", "raft_flow.npy", "nflow.npy"} <= set(names), names
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    assert all(np.load(tmp_path / n).dtype == np.float32 for n in names)
    with torch.no_grad():
        ref = O.gimmvfi_r_forward(weights0, synth_batch(1, H, W, seed=100), [(O.sample_coord_input(1, (H, W), [0.5]), None)], [0.5 * torch.ones(1)])
    img = np.load(tmp_path / "imgt_pred_0.npy")
    assert img.shape == (1, 3, H, W)
    err = np.abs(img - ref["imgt_pred"][0].numpy()).max()
    print("bench dump: imgt_pred max|d| vs oracle = %.3e" % err)
    assert err <= TOL_IMG, err
