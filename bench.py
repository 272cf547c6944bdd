#!/usr/bin/env python
"""bench.py — interpolated frames/s of the GIMM-VFI-R per-pair path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" = one GIMMVFI_R.forward over one batch of synthetic frame pairs.  Workload at
every N: BASELINE.json configs[1] — one 1920x1080 pair per GPU (caller-padded to
1088x1920), t=0.5, GIMM-VFI-R, random-init weights (no checkpoints offline), all
reference outputs produced.  N>1: one process per GPU (torchrun), pairs sharded with no
data-path collective, ONE all-gather of the output frames per step (weak scaling).

Prints one JSON line (rank 0).  `value` = device-timed frames/s with inputs resident in
HBM; `e2e` = the same through the public API with pinned-host inputs, H2D + D2H inside the
timed region; `roofline` = the dominant kernel timed live with CUDA events on the
launching stream; `cpu_baseline` = the CPU oracle port on the box's host cores (bounded
sample).  `--impl reference` times that CPU path only (the reference is Python/PyTorch:
its own path on host cores is the oracle port, bit-identical to it here).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "interpolated frames/sec @1080p t=0.5"
UNIT = "frames/s"
H_PAD, W_PAD = 1088, 1920          # InputPadder(1080x1920, 32)  src/utils/utils.py:156-185
SAMPLE_H, SAMPLE_W = 256, 448      # bounded CPU sample (BASELINE config 1 size)
if os.environ.get("GIMMVFI_CPU_SAMPLE"):   # tests shrink the sample (e.g. "128x160"); the scaling to 1080p is by pixel count either way
    SAMPLE_H, SAMPLE_W = (int(v) for v in os.environ["GIMMVFI_CPU_SAMPLE"].lower().split("x"))


def flops_per_frame(P, T=1, P_full=None):
    """SURVEY.md §8(d): algorithmic FLOPs (2*MAC, conv+matmul) of GIMM-VFI-R for one pair."""
    P_full = P if P_full is None else P_full
    return 4.981e6 * P + 0.375 * float(P) ** 2 + T * (13.770e6 * P + 0.0212e6 * P_full)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]), which="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, which="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = max((float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(self.rows)}


DUMP_BUDGET = 60 << 20   # bytes of array data --dump-outputs writes at most (the .npy headers stay well inside 64 MB)


def flatten_outputs(out, prefix=""):
    """{name: tensor} of a forward's output dict; list entries append their index (imgt_pred_0, flowt0_pred_0_1, ...)"""
    if torch.is_tensor(out):
        return {prefix: out}
    items = {}
    for k, v in (out.items() if isinstance(out, dict) else enumerate(out)):
        items.update(flatten_outputs(v, "%s_%s" % (prefix, k) if prefix else str(k)))
    return items


def dump_outputs(path, out):
    """Writes every array of `out` as <path>/<name>.npy in float32 (float64 stays float64).  If they exceed DUMP_BUDGET together,
    each array larger than an equal share of it is replaced by a 1-D sample of that many elements: flat indices drawn without
    replacement by numpy.random.default_rng(0), in increasing order, so runs of two builds write the same elements."""
    arrays = flatten_outputs(out)
    os.makedirs(path, exist_ok=True)
    total = sum(t.numel() * (8 if t.dtype == torch.float64 else 4) for t in arrays.values())
    share = DUMP_BUDGET // len(arrays)
    for name, t in arrays.items():
        a = t.detach().to("cpu", torch.float64 if t.dtype == torch.float64 else torch.float32).numpy()
        cap = share // a.itemsize
        if total > DUMP_BUDGET and a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def cpu_threads():
    """Threads for the CPU arm: all host cores up to GIMMVFI_CPU_THREADS (default 64: the builder's 1080p run, 104.5 s per frame,
    used 64 of the GPU box's 128 cores; the reference's small RAFT convolutions oversubscribe oneDNN beyond that)."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get("GIMMVFI_CPU_THREADS", "64"))))


def workload_config(H, W, T, B=1, precision=None, world=1):
    """`config` of the JSON line — IDENTICAL in both arms (the driver compares them: same workload, same metric)."""
    frame = "1920x1080 pair per GPU (padded %dx%d)" % (H, W) if (H, W) == (H_PAD, W_PAD) else "%dx%d pair per GPU (--height/--width)" % (H, W)
    return {"workload": "%d x %s, %s, GIMM-VFI-R (RAFT 20 iters), random-init weights, all reference outputs produced"
                        % (B, frame, "t=0.5, T=1" if T == 1 else "T=%d frames per pair at t=i/%d" % (T, T + 1)),
            "height": H, "width": W, "timesteps": T, "pairs_per_step_per_gpu": B}


def cpu_reference_fps(steps, warmup, H=H_PAD, W=W_PAD, T=1):
    """The reference's own PyTorch path (fp32, torch.no_grad) on the host cores via the oracle port (bit-identical to the unmodified
    reference in the build container at every fixture size incl. 736x1280: tests/golden/manifest*.json).  One step = one full
    forward of ONE HxW pair — the same workload the GPU arm times, no extrapolation."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gimmvfi_r_oracle as O
    from gimmvfi_b200.synth import synth_batch
    from gimmvfi_b200.weights import random_state_dict

    torch.set_num_threads(cpu_threads())
    sd = random_state_dict(0)
    xs = synth_batch(1, H, W, seed=100)
    tvals = [0.5] if T == 1 else [i / (T + 1) for i in range(1, T + 1)]
    coord = [(O.sample_coord_input(1, (H, W), [tv]), None) for tv in tvals]
    t = [tv * torch.ones(1) for tv in tvals]
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            out = O.gimmvfi_r_forward(sd, xs, coord, t)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    sec = sum(times) / len(times)
    return dict(sec_per_step=sec, fps=T / sec, cores=torch.get_num_threads(), times=times, out=out)


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation of the SAME config (one 1088x1920 pair per step).  A forward takes
    ~100 s on the box's host cores, so the warm-up is bounded (at most GIMMVFI_REF_MAX_WARMUP forwards, default 1); --steps
    forwards are timed.  `steps`/`warmup` echo the request, `steps_timed`/`warmup_run` say what ran."""
    if rank != 0:
        return
    H, W = args.height, args.width
    scaled = None
    if os.environ.get("GIMMVFI_CPU_SAMPLE"):   # contract tests only: a small frame instead of the workload (NOT the same config; flagged)
        H, W = (int(v) for v in os.environ["GIMMVFI_CPU_SAMPLE"].lower().split("x"))
        scaled = (H * W) / float(args.height * args.width)
    T = max(1, args.timesteps)
    timed = args.steps
    warm = min(max(0, args.warmup), int(os.environ.get("GIMMVFI_REF_MAX_WARMUP", "1")))
    r = cpu_reference_fps(timed, warm, H, W, T)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["out"])
    fps = r["fps"] * (scaled if scaled else 1.0)
    sample = ("oracle port (== reference PyTorch fp32 path, bit-identical to it on the golden fixtures) on the full %dx%d pair, "
              "%d warm-up + %d timed forwards (~100 s each)" % (H, W, warm, timed))
    if scaled:
        sample = "TEST SAMPLE %dx%d pixel-scaled to %dx%d — not the benchmark config" % (H, W, args.height, args.width)
    cfg = workload_config(args.height, args.width, T)
    if scaled:
        cfg["timed_sample"] = "%dx%d" % (H, W)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "steps_timed": timed, "warmup_run": warm, "ms_per_step": 1000.0 * r["sec_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def gpu_torch_baseline(H, W, T, dev, steps=3, warmup=1):
    """The 'stock PyTorch on the same B200' bar of SURVEY 2a / 8(d): the oracle port (== the reference's own torch ops: cuDNN / cuBLAS
    convolutions, grid_sample, index_add_ splat) in fp32 with TF32 disabled, eager, same input, CUDA-event timed.  Test
    infrastructure used as a measured baseline only; nothing of it is on the product path."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gimmvfi_r_oracle as O
    from gimmvfi_b200.synth import synth_batch
    from gimmvfi_b200.weights import random_state_dict

    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    try:
        sd = {k: v.to(dev) for k, v in random_state_dict(0).items()}
        xs = synth_batch(1, H, W, seed=100).to(dev)
        tvals = [0.5] if T == 1 else [i / (T + 1) for i in range(1, T + 1)]
        ms = []
        with torch.no_grad(), torch.device(dev):   # the oracle's factory calls (linspace / arange / zeros) follow the default device
            coord = [(O.sample_coord_input(1, (H, W), [tv]), None) for tv in tvals]
            t = [tv * torch.ones(1) for tv in tvals]
            out = None
            for i in range(warmup + steps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = O.gimmvfi_r_forward(sd, xs, coord, t)
                e1.record()
                torch.cuda.synchronize(dev)
                if i >= warmup:
                    ms.append(e0.elapsed_time(e1))
        peak = torch.cuda.max_memory_allocated(dev)
        img = out["imgt_pred"][0]
        del out
        torch.cuda.empty_cache()
        m = sum(ms) / len(ms)
        return {"value": T / (m * 1e-3), "unit": UNIT, "ms_per_step": m, "steps": steps, "warmup": warmup, "peak_mem_gb": peak / 2 ** 30,
                "what": "oracle port == the reference's own torch ops (cuDNN/cuBLAS eager, fp32, allow_tf32=False, cudnn.benchmark=True, "
                        "splat via index_add_) on the same B200 and the same 1x%dx%d input; CUDA-event timed" % (H, W)}, img
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark = old


def load_ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant layer shape of each kernel, written by
    scripts/summarize_ncu.py from the committed `ncu --set full` captures (profiles/ncu_traffic.json); absent -> traffic null."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return {}
    with open(p) as f:
        return json.load(f)


PRECISIONS = {"fp32": 0, "tf32": 1, "3xtf32": 2, "mixed3": 3, "mixed": 4}
PRECISION_NOTES = {
    "fp32": "fp32 CUDA cores everywhere",
    "tf32": "RAFT fp32 (CUDA cores); post-RAFT convs TF32 tcgen05, fp32 accumulate",
    "3xtf32": "RAFT + its correlation volume: tcgen05 3xF16 (fp16 hi/lo operand split, fp32 register-promoted accumulation: fp32-class); post-RAFT convs: "
              "tcgen05 TF32, fp32 accumulate; HypoNet fused, fp32-class",
    "mixed3": "as 3xtf32 + the final decoder's 256-channel residual trunk stored in fp16 on tcgen05 kind::f16; fp32 accumulate everywhere",
    "mixed": "RAFT + its correlation volume: tcgen05 3xF16 (fp16 hi/lo operand split, fp32 register-promoted accumulation: fp32-class); HypoNet fused, "
             "fp32-class; post-RAFT convs: tcgen05 TF32 or, where the activations are stored in fp16 (final-decoder trunk, the 32/64-channel "
             "full-resolution chains, init-decoder trunk, decoder concat), kind::f16; fp32 accumulate everywhere.  Parity at this exact workload: "
             "tests/test_bench_parity_gpu.py::big_r_1088x1920_t0.5 (reference-generated fixture, max|d imgt_pred| <= 1e-3)",
}
DTYPES = {"fp32": "f32", "tf32": "tf32", "3xtf32": "tf32", "mixed3": "tf32+f16 operands, f32 accumulate", "mixed": "tf32+f16 operands, f32 accumulate"}
NOTES = {"conv2d_tc_f16": "tcgen05 kind::f16 implicit GEMM on fp16-stored activations (TMA halo tiles, TMEM fp32 accumulators)",
         "conv2d_tc_tf32": "tcgen05 kind::tf32 implicit GEMM (TMA halo tiles, TMEM accumulators); the TF32 tensor peak is half the bf16 peak used as denominator (ceiling 0.5)",
         "conv2d_tc_3xtf32": "tcgen05 3xTF32 (3 MMAs per K step + register-promoted accumulation): 'achieved' counts ALGORITHMIC flops, the tensor pipe "
                             "executes 3x that at the TF32 rate (= bf16 peak / 2), so the ceiling of this ratio is 1/6",
         "conv2d_tc_3xf16": "tcgen05 3-term fp16 hi/lo split (3 kind::f16 MMAs per K step + register-promoted accumulation): 'achieved' counts ALGORITHMIC "
                            "flops, the tensor pipe executes 3x that at the f16 rate, so the ceiling of this ratio is 1/3",
         "conv2d_simt_n64": "fp32 CUDA-core implicit GEMM measured against the tensor-pipe peak (the layer class is tensor-bound, SURVEY 8(d))"}
CEILING = {"conv2d_tc_tf32": 0.5, "conv2d_tc_3xtf32": 1.0 / 6.0, "conv2d_tc_3xf16": 1.0 / 3.0, "conv2d_tc_f16": 1.0}


def build_roofline(prof, raw_prof, peaks):
    """The dominant kernel of the profiled step: algorithmic work / CUDA-event time of its launches."""
    total_ms = sum(v["ms"] for v in prof.values()) or 1.0
    dname, d = max(prof.items(), key=lambda kv: kv[1]["ms"])
    traffic = load_ncu_traffic()
    if dname.startswith(("conv2d", "corr_gemm", "hyponet")):
        ach = d["work"] / (d["ms"] * 1e-3) / 1e12
        tr = traffic.get(dname, {})
        roof = {"bound": "tensor", "kernel": dname, "achieved": ach, "peak": peaks["tf_sust"], "unit": "TFLOP/s", "frac": ach / peaks["tf_sust"],
                "traffic": tr.get("bytes"), "traffic_detail": tr or None,
                "peak_source": "%s bf16 sustained (MEASURED_PEAKS.json)" % peaks["which"], "format_ceiling_frac": CEILING.get(dname),
                "launches": d["launches"], "avg_launch_ms": d["ms"] / d["launches"], "share_of_step": d["ms"] / total_ms, "note": NOTES.get(dname, "")}
        top = max(((k, v) for k, v in raw_prof.items() if k.startswith(("conv2d", "corr_gemm", "hyponet"))), key=lambda kv: kv[1]["ms"])
        roof["top_layer"] = {"name": top[0], "ms_total": top[1]["ms"], "launches": top[1]["launches"],
                             "tflops": top[1]["work"] / (top[1]["ms"] * 1e-3) / 1e12, "frac_of_peak": top[1]["work"] / (top[1]["ms"] * 1e-3) / 1e12 / peaks["tf_sust"]}
    else:   # pointwise / gather kernels report `work` in fp32 elements touched
        ach = 4.0 * d["work"] / (d["ms"] * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": dname, "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach / peaks["hbm"],
                "traffic": traffic.get(dname, {}).get("bytes"), "launches": d["launches"], "share_of_step": d["ms"] / total_ms}
    return roof, total_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="pair1080", choices=["pair1080", "batch720", "f2k", "f4k"],
                    help="pair1080 (default, BASELINE configs[1], the headline metric): one 1920x1080 pair per GPU per step, weak scaling.  "
                         "batch720 (BASELINE configs[4]): 256 1280x720 pairs (padded 736x1280) sharded across the ranks, a step = the whole "
                         "batch in micro-batches of --micro-batch pairs per forward, ONE all-gather of the output frames, strong scaling.  "
                         "f2k / f4k (BASELINE configs[2] / [3]): GIMM-VFI-F (native FlowFormer estimator) on one 2K pair at ds_factor 0.5 / one 4K "
                         "pair at ds_factor 0.25 per GPU, N = 8 -> 7 interpolated frames per pair")
    ap.add_argument("--pairs", type=int, default=256)
    ap.add_argument("--micro-batch", type=int, default=8)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-baseline", action="store_true")
    ap.add_argument("--precision", default="mixed", choices=list(PRECISIONS))
    ap.add_argument("--profile-json", default="", help="write the per-kernel CUDA-event breakdown here")
    ap.add_argument("--timesteps", type=int, default=1,
                    help="T interpolated frames per pair at t = i/(T+1): 1 = the headline metric (t=0.5); 7 = the reference's N=8 video setting")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32; at most 64 MB in all, larger "
                         "outputs as a fixed seeded sample of their elements) - the inputs are seeded, so runs of two builds compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    batch_mode = args.config == "batch720"
    f_mode = args.config in ("f2k", "f4k")
    ds = None
    if f_mode:   # src/video_Nx.py: 2K -> ds 0.5, 4K -> ds 0.25 (README of the reference), InputPadder(32): 2048x1080 -> 1088x2048, 4096x2160 -> 2176x4096
        ds = 0.5 if args.config == "f2k" else 0.25
        if not args.height:
            args.height, args.width = (1088, 2048) if args.config == "f2k" else (2176, 4096)
        if args.timesteps == 1:
            args.timesteps = 7
        args.no_cpu_baseline = args.no_torch_baseline = True   # (the CPU / stock-PyTorch legs are GIMM-VFI-R's; FlowFormer on host cores takes minutes per pair)
        if args.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                print(json.dumps({"impl": "reference", "unavailable": "GIMM-VFI-F's reference needs timm 0.4.12 + pretrained FlowFormer weights (absent offline); "
                                  "its CPU path at this size runs for minutes per pair - the timed reference arm is the GIMM-VFI-R headline config"}))
            return
    fkw = {"ds_factor": ds} if f_mode else {}
    ckw = {"upsample_ratio": ds} if f_mode else {}
    if not args.height:
        args.height, args.width = (736, 1280) if batch_mode else (H_PAD, W_PAD)
    args.warmup = max(args.warmup, 3 if not batch_mode else 1) if args.impl == "ours" else args.warmup

    from gimmvfi_b200.parallel import init_from_env, shard_range

    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")))
        return

    import torch.distributed as dist

    rank, local, world = init_from_env("nccl")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    from gimmvfi_b200 import GIMMVFI_R
    from gimmvfi_b200.synth import synth_batch

    H, W, T = args.height, args.width, max(1, args.timesteps)
    tvals = [0.5] if T == 1 else [i / (T + 1) for i in range(1, T + 1)]
    if f_mode:
        from gimmvfi_b200 import GIMMVFI_F
        from gimmvfi_b200.weights import random_state_dict_f

        model = GIMMVFI_F(seed=0).to(dev).eval()
        model.load_state_dict(random_state_dict_f(0), strict=True)
    else:
        model = GIMMVFI_R(seed=0).to(dev).eval()
    model.tensor_cores = PRECISIONS[args.precision]
    if batch_mode:
        mine = shard_range(args.pairs, rank, world)
        MB = max(1, args.micro_batch)
        nmb = (len(mine) + MB - 1) // MB
        B = MB
        distinct = synth_batch(min(4, MB), H, W, seed=100 + 7 * rank)              # a few distinct pairs, tiled to the micro-batch
        xs_host = distinct.repeat((MB + distinct.shape[0] - 1) // distinct.shape[0], 1, 1, 1, 1)[:MB].contiguous().pin_memory()
        per_rank_max = len(shard_range(args.pairs, 0, world))
    else:
        B, nmb, MB = 1, 1, 1
        xs_host = synth_batch(1, H, W, seed=100 + rank).pin_memory()
    xs = xs_host.to(dev, non_blocking=True)
    coord = [(model.sample_coord_input(B, (H, W), [tv], device=dev, **ckw), None) for tv in tvals]
    tt = [tv * torch.ones(B, device=dev) for tv in tvals]
    frames_per_step_rank = (len(mine) if batch_mode else B) * T
    if batch_mode:
        outbuf = torch.empty(per_rank_max * T, 3, H, W, device=dev)
        gathered = torch.empty(world * per_rank_max * T, 3, H, W, device=dev) if world > 1 else None
    else:
        outbuf = None
        gathered = torch.empty(world * B * T, 3, H, W, device=dev) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def frames_of(out, b):
        return (torch.stack(out["imgt_pred"], 1).reshape(-1, 3, H, W) if T > 1 else out["imgt_pred"][0])[: b * T]

    def step(x=None):
        """one step on device-resident inputs: pair1080 = one forward; batch720 = this rank's shard in micro-batches + ONE all-gather.
        Returns what the caller receives: the forward's output dict, or this rank's frames (batch720)."""
        if not batch_mode:
            out = model(xs if x is None else x, coord, t=tt, **fkw)
            img = frames_of(out, B)
            if world > 1:
                dist.all_gather_into_tensor(gathered, img.contiguous())   # the single output collective
            return out
        done = 0
        for m in range(nmb):
            b = min(MB, len(mine) - done)
            outbuf[done * T:(done + b) * T].copy_(frames_of(model(xs, coord, t=tt), b))   # (a ragged last micro-batch computes MB pairs, keeps b)
            done += b
        if world > 1:
            dist.all_gather_into_tensor(gathered, outbuf)
        return {"imgt_pred": outbuf}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    aux = model.aux_outputs
    if batch_mode:
        model.aux_outputs = False   # config 5 collects frames only (SURVEY 8(e)); pair1080 produces every reference output
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    # ---- device-timed steps (CUDA events on the launching stream; L2 flushed between steps)
    evs = []
    barrier()
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        last = None   # a step's outputs are released before the next step starts
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = step()
        e1.record()
        evs.append((e0, e1))
    barrier()
    wall = time.perf_counter() - wall0
    if args.dump_outputs and rank == 0:   # written after the measurements below
        dumped = {k: v.cpu() for k, v in flatten_outputs(last).items()}
    del last
    ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps
    launches = model.engine.last_launches * nmb
    # ---- end-to-end through the public API: pinned host input -> H2D -> forward -> D2H of the frames, every forward.
    # The loop is what a video / batch caller runs (src/video_Nx.py:134-216 walks consecutive pairs): the copies of forward i+1 / i-1
    # travel on a second stream while forward i computes; nothing is reused across forwards and the whole region (all copies
    # included) is timed by the wall clock between two full synchronisations.
    out_host = [torch.empty(B * T, 3, H, W).pin_memory() for _ in range(2)]
    x_dev = [torch.empty_like(xs) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)
    ev_in = [torch.cuda.Event() for _ in range(2)]     # H2D of the buffer landed
    ev_free = [torch.cuda.Event() for _ in range(2)]   # forward that read the buffer finished
    ev_out = [torch.cuda.Event() for _ in range(2)]    # D2H of the result buffer finished
    keep = [None, None]
    n_fwd = args.steps * nmb

    def h2d(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[i % 2])
            x_dev[i % 2].copy_(xs_host, non_blocking=True)
            ev_in[i % 2].record(copy_stream)

    def e2e_loop(n):
        """n pipelined forwards; returns wall seconds between two full synchronisations"""
        barrier()
        for e in ev_free + ev_out:
            e.record(main_stream)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        h2d(0)
        for i in range(n):
            main_stream.wait_event(ev_in[i % 2])
            if i + 1 < n:
                h2d(i + 1)
            c = [(model.sample_coord_input(B, (H, W), [tv], device=dev, **ckw), None) for tv in tvals]
            o = model(x_dev[i % 2], c, t=[tv * torch.ones(B, device=dev) for tv in tvals], **fkw)
            img = frames_of(o, B)
            if world > 1 and not batch_mode:
                dist.all_gather_into_tensor(gathered, img.contiguous())
            ev_free[i % 2].record(main_stream)
            keep[i % 2] = img
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_free[i % 2])
                copy_stream.wait_event(ev_out[i % 2])
                img.record_stream(copy_stream)
                out_host[i % 2].copy_(img, non_blocking=True)
                ev_out[i % 2].record(copy_stream)
            if batch_mode and world > 1 and (i + 1) % nmb == 0:
                dist.all_gather_into_tensor(gathered, outbuf)
        torch.cuda.synchronize(dev)
        return time.perf_counter() - t0

    # untimed warm-up of the copy stream / pinned buffers / pipelined path: as many forwards as the timed loop, so that the caching allocator has
    # already grown to the loop's steady state (outputs handed to the copy stream are freed late; a first-time cudaMalloc in the timed loop
    # synchronises the device - seen as +8 ms per step in 2 of 5 otherwise identical runs)
    e2e_loop(max(2 * nmb, n_fwd) if not batch_mode else nmb)
    e2e_ms = 1000.0 * e2e_loop(n_fwd) / args.steps
    barrier()
    clocks = sampler.stop() if sampler else None
    # ---- per-kernel breakdown (CUDA events around every launch of one extra forward)
    model.engine.set_profile(True)
    model(xs, coord, t=tt, **fkw)
    prof = model.engine.profile()
    model.engine.set_profile(False)
    model.aux_outputs = aux
    # max over ranks
    if world > 1:
        tm = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ms, e2e_ms = tm.tolist()
    if rank == 0:
        peaks = load_peaks()
        raw_prof = prof
        agg = {}
        for k, v in prof.items():   # labels carry the layer shape; aggregate per kernel for the headline
            a = agg.setdefault(k.split(" ")[0], {"ms": 0.0, "work": 0.0, "launches": 0})
            a["ms"] += v["ms"]; a["work"] += v["work"]; a["launches"] += v["launches"]
        prof = agg
        roof, total_ms = build_roofline(prof, raw_prof, peaks)
        conv_ms = sum(v["ms"] for k, v in prof.items() if k.startswith("conv2d"))
        conv_fl = sum(v["work"] for k, v in prof.items() if k.startswith("conv2d"))
        if args.profile_json:
            with open(args.profile_json, "w") as f:
                json.dump({"per_kernel": prof, "per_layer": raw_prof, "sum_ms": total_ms, "step_ms": ms}, f, indent=1)
        total_frames = (args.pairs if batch_mode else world * B) * T
        fl = flops_per_frame(H * W, T)
        n_pairs_total = args.pairs if batch_mode else world * B
        cfg = workload_config(H, W, T, B)
        if f_mode:
            cfg["workload"] = ("%d x %s pair per GPU (padded %dx%d), ds_factor %s, T=%d frames per pair at t=i/%d, GIMM-VFI-F (native FlowFormer estimator, 32 "
                               "decoder iterations, both directions), seeded random weights, all reference outputs produced"
                               % (B, "2K (2048x1080)" if args.config == "f2k" else "4K (4096x2160)", H, W, ds, T, T + 1))
            cfg["ds_factor"] = ds
        if batch_mode:
            cfg["workload"] = ("%d x 1280x720 pairs (padded %dx%d), t=0.5, GIMM-VFI-R (RAFT 20 iters), random-init weights, sharded over %d GPU(s), "
                               "micro-batch %d pairs per forward, frames only" % (args.pairs, H, W, world, MB))
            cfg["pairs"] = args.pairs
            cfg["micro_batch"] = MB
        if f_mode:
            fl = None
        cfg.update({"precision": PRECISION_NOTES[args.precision] if not f_mode else
                    "FlowFormer estimator (Twins-SVT x2, cost-perceiver memory encoder, GMA decoder) and HypoNet: tcgen05 3xF16 (fp32-class) convolutions / GEMMs, fp32 "
                    "CUDA-core attention, softmax and LayerNorm; synthesis half as GIMM-VFI-R's default mode.  Parity: tests/test_f_gpu.py (reference-generated "
                    "ff_* fixtures: flows <= 2e-3 px, max|d imgt_pred| <= 1e-3)",
                    "parallelism": ("pairs sharded rank::world, ONE all-gather of the output frames per step" if world > 1 else "single GPU"),
                    "l2": "256 MiB L2 flush between timed steps; per-step working set ~30 GB >> L2",
                    "algorithmic_tflop_per_frame": fl / T / 1e12 if fl else None,
                    "achieved_tflops_end_to_end": n_pairs_total * fl / (ms * 1e-3) / 1e12 if fl else None})
        line = {
            "metric": (METRIC if not batch_mode else "interpolated frames/sec, batch of 256 1280x720 pairs, t=0.5") if not f_mode else
                      "interpolated frames/sec, %s pair DS_SCALE=%s, N=8 timesteps, GIMM-VFI-F" % ("2K" if args.config == "f2k" else "4K", ds),
            "value": total_frames / (ms * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if batch_mode else "weak", "vs_baseline": None, "dtype": DTYPES[args.precision], "data": "synthetic",
            "config": cfg,
            "e2e": {"value": total_frames / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": xs_host.numel() * 4 * nmb,
                    "d2h_bytes_per_step": out_host[0].numel() * 4 * nmb,
                    "how": "K-step loop, wall clock between full syncs; per-forward H2D/D2H on a copy stream overlapped with the previous/next forward"},
            "gpu_launches": int(launches) * args.steps,
            "launches_per_step": int(launches),
            "roofline": roof,
            "kernel_shares": {k: round(v["ms"] / total_ms, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])[:8]},
            "conv_tflops": conv_fl / (conv_ms * 1e-3) / 1e12 if conv_ms else None,
            "clocks": clocks,
            "wall_s_timed_region": wall,
        }
        if world == 1 and not args.no_torch_baseline and not batch_mode:
            try:
                del flush
                torch.cuda.empty_cache()
                tb, ref_img = gpu_torch_baseline(H, W, T, dev)
                mine_img = frames_of(model(xs, coord, t=tt), B)[:1]
                tb["max_abs_diff_imgt_pred_vs_this_arm"] = (ref_img - mine_img).abs().max().item()
                tb["speedup_of_this_arm"] = line["value"] / tb["value"]
                line["gpu_torch_baseline"] = tb
            except Exception as ex:  # noqa: BLE001
                line["gpu_torch_baseline"] = {"value": None, "error": repr(ex)[:300]}
        if world == 1 and not args.no_cpu_baseline and not batch_mode:
            # bounded sample (~10-30 s of CPU work): ONE 256x448 pair per step (BASELINE config 1 size), frames/s EXTRAPOLATED to the
            # workload by the pixel ratio — the same-config CPU measurement is the `--impl reference` arm (~100 s per forward)
            try:
                env = dict(os.environ, GIMMVFI_CPU_SAMPLE="%dx%d" % (SAMPLE_H, SAMPLE_W), GIMMVFI_CPU_THREADS=os.environ.get("GIMMVFI_CPU_THREADS", "32"))
                o = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                                   capture_output=True, text=True, timeout=240, env=env).stdout.strip().splitlines()
                cb = json.loads([l for l in o if l.startswith("{")][-1])["cpu_baseline"]
                cb["sample"] = ("EXTRAPOLATED: oracle port (== reference PyTorch fp32 path) on one %dx%d pair, 1 warm-up + 2 timed, frames/s scaled by the "
                                "pixel ratio to %dx%d (the all-pairs correlation grows faster, so this flatters the CPU; the measured same-config "
                                "figure is the --impl reference arm)" % (SAMPLE_H, SAMPLE_W, H, W))
                line["cpu_baseline"] = cb
            except Exception as ex:  # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": cpu_threads(), "kind": "port", "sample": "CPU arm did not finish within 240 s: %r" % (ex,)}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
