"""bench.py - FullSubNet inference throughput on B200 (BASELINE.json metric: frames/s and x real-time,
16 kHz, n_fft=512, hop=256) for the workload `configs[1]`: batch = 256 x 4 s synthetic clips per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--precision auto|fp32|f16x3_tc|f16_tc] [--no-extras]
                  [--dump-outputs DIR]
  python bench.py --impl reference      # the CPU arm (oracle port of the reference path, all host threads)

One "step" = one pass of the hot path (stft -> model -> decompress/mask -> istft) over one batch.
--dump-outputs DIR writes what the last of the K timed steps returned as DIR/<name>.npy (float32); the inputs and weights
are fixed by their seeds, so two builds run with the same arguments can be compared output for output.
`value` is measured with the inputs resident in HBM; `e2e` goes through the public API with pinned HOST
buffers, the H2D copy of the waveforms and the D2H copy of the result inside the timed region.
Multi-GPU: one process per GPU (torchrun), clips sharded over ranks, no data-path collective (weak
scaling: every rank enhances its own B clips); time = max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR, N_FFT, HOP, WIN = 16000, 512, 256, 512
CLIP_SECONDS = 4
FLOP_PER_FRAME_STEP_SB = 257 * 3_638_784  # SURVEY 8d: sub-band stack, per clip per LSTM step
FLOP_PER_FRAME_STEP_ALL = 942_774_784
DUMP_BYTES = 63 * 10**6  # array bytes --dump-outputs writes at most: under 64 MB in all with the .npy headers


def dump_outputs(out_dir: str, arrays: dict, rank: int = 0, world: int = 1) -> None:
    """Writes each tensor of ``arrays`` as out_dir/<name>.npy in float32 (<name>_rank<r>.npy with several ranks).  Where
    they exceed this rank's share of DUMP_BYTES, every array keeps the same fixed, seeded sample of its leading (clip)
    dimension, in order, so that repeated runs write the same sample."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total, budget = sum(a.nbytes for a in arrays.values()), DUMP_BYTES // world
    for name, a in arrays.items():
        if total > budget and a.ndim:
            keep = a.shape[0] * budget // total
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}_rank{rank}.npy" if world > 1 else f"{name}.npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


_CPU_THREADS = None
_CPU_SWEEP = {}


def _cpu_model():
    from oracle import fullsubnet_oracle as O
    from oracle import libcall_port as P
    return P.LibcallModel(O.make_state_dict(seed=0))


def pick_cpu_threads() -> int:
    """Thread count of the CPU arm.  The per-step LSTM matmuls are small, so more threads are not always faster;
    every candidate count enhances one warm-up clip and then three full 4 s clips (>= 1 s of work each) and the count
    with the best MEDIAN clip time is kept - long enough that the choice does not flap between runs."""
    global _CPU_THREADS
    if _CPU_THREADS is None:
        from oracle import fullsubnet_oracle as O
        from oracle import libcall_port as P
        cores = os.cpu_count() or 1
        model = _cpu_model()
        y = O.make_noisy(1, SR * CLIP_SECONDS, seed=0)
        best = (1e30, 1)
        for n in sorted({c for c in (8, 16, 32, 64) if c <= cores} | {min(cores, 8)}):
            torch.set_num_threads(n)
            P.enhance(y, model)
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                P.enhance(y, model)
                ts.append(time.perf_counter() - t0)
            med = sorted(ts)[1]
            _CPU_SWEEP[n] = round((1 + (SR * CLIP_SECONDS) // HOP) / med, 1)
            best = min(best, (med, n))
            if med > 20:
                break
        _CPU_THREADS = best[1]
    return _CPU_THREADS


def cpu_oracle_time(n_clips: int, threads: int):
    """Times the CPU arm: Inferencer.full_band_crm_mask restated with the reference's own PyTorch library calls
    (oracle/libcall_port.py: torch.stft / nn.LSTM / F.unfold / torch.istft, bit-identical to the reference's output
    on the goldens), B=1 loop - the reference's only inference batch."""
    from oracle import fullsubnet_oracle as O
    from oracle import libcall_port as P
    torch.set_num_threads(threads)
    model = _cpu_model()
    y = O.make_noisy(n_clips, SR * CLIP_SECONDS, seed=0)
    t0 = time.perf_counter()
    P.enhance(y, model)
    dt = time.perf_counter() - t0
    frames = n_clips * (1 + (SR * CLIP_SECONDS) // HOP)
    return frames / dt, dt


CPU_KIND_NOTE = ("port = the reference path written with the reference's own torch library calls (torch.stft, nn.LSTM, "
                 "F.unfold, torch.istft), output bit-identical to the unmodified reference on tests/golden; the reference "
                 "is pure Python without setup.py and with uninstalled deps, so it cannot be installed or travel")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = pick_cpu_threads()
    n_clips = 4
    vals = []
    for _ in range(1 if args.warmup > 0 else 0):
        cpu_oracle_time(1, cores)
    t_all = time.perf_counter()
    for _ in range(args.steps):
        v, _ = cpu_oracle_time(n_clips, cores)
        vals.append(v)
    dt = time.perf_counter() - t_all
    v = sorted(vals)[len(vals) // 2]
    T = 1 + (SR * CLIP_SECONDS) // HOP
    line = {
        "impl": "reference", "metric": "frames_per_sec", "value": v, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "rtf_x": v / (SR / HOP),
        "config": {"workload": "fullsubnet inference, 4 s 16 kHz synthetic clips, n_fft=512 hop=256 N=15, 2xLSTM-512 fb + "
                               "2xLSTM-384 sb (CPU: B=1 loop over 4 clips per step; per-frame throughput is batch-"
                               "independent on this arm, the GPU arm runs 256 clips per step)",
                   "clip_seconds": CLIP_SECONDS, "frames_per_clip": T, "clips_per_step": n_clips},
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{n_clips} x 4 s clips per step, B=1 loop, torch CPU fp32 library calls, {cores} "
                                   f"threads (best median of a sweep {_CPU_SWEEP} frames/s; host has "
                                   f"{os.cpu_count()} logical cores)",
                         "note": CPU_KIND_NOTE},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256, help="clips per GPU (configs[1]: 256)")
    ap.add_argument("--precision", default="auto")
    ap.add_argument("--model", default="fullsubnet", choices=["fullsubnet", "fast_fullsubnet", "improved_fullsubnet", "fullsubnet_train"],
                    help="fullsubnet = BASELINE configs[1] (the headline); fast_fullsubnet = configs[3] (use --batch 512); "
                         "improved_fullsubnet = configs[4] (48 kHz, n_fft 1024, use --batch 128; --variant k48_960 = the "
                         "reference's own 48 kHz example, k16 = the class defaults); "
                         "fullsubnet_train = configs[2], the training step (bench_train.py)")
    ap.add_argument("--variant", default="k48", choices=["k48", "k48_960", "k16"], help="improved_fullsubnet constructor args")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `precisions`, `latency_b1` and `train_dp` objects")
    ap.add_argument("--no-train", action="store_true", help="skip the `train_dp` object")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy "
                                                          "(float32; above 64 MB, a fixed, seeded sample of the clips)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA implementation (--impl b200)")
    if args.model == "fullsubnet_train":
        import bench_train
        return bench_train.main(args)
    if args.impl == "reference":
        return run_reference(args)

    import ctypes as C
    from fullsubnet_b200 import _lib
    from fullsubnet_b200.fullsubnet.model import Model
    from fullsubnet_b200.inferencer import Inferencer
    from oracle import fullsubnet_oracle as O  # weights / inputs generator only (+ cpu_baseline leg)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist_mod.init_process_group("nccl", device_id=dev)
        dist = dist_mod

    lib = _lib.load()
    B, L = args.batch, SR * CLIP_SECONDS
    T = 1 + L // HOP
    imp_args = None
    frame_rate = SR / HOP  # frames per second of real time (x RT = frames/s / frame_rate)
    if args.model == "improved_fullsubnet":
        from fullsubnet_b200.improved_fullsubnet.model import Model as ImpModel
        from oracle import improved_fullsubnet_oracle as IO
        imp_args = {"k48": IO.ARGS_48K_1024, "k48_960": IO.ARGS_48K_960, "k16": IO.DEFAULT_IMPROVED_ARGS}[args.variant]
        sr = 16000 if args.variant == "k16" else 48000
        L = sr * 2  # BASELINE configs[4]: 2 s clips
        T = 1 + L // imp_args["hop_length"]
        frame_rate = sr / imp_args["hop_length"]
        model = ImpModel(**imp_args)
        model.load_state_dict(IO.make_improved_state_dict(seed=5, args=imp_args), strict=True)
        if args.precision != "auto":
            model.precision = args.precision
        model = model.to(dev).eval()
        precision = model._resolve_precision()
    elif args.model == "fast_fullsubnet":
        from fullsubnet_b200.fast_fullsubnet.model import Model as FastModel
        from oracle import fast_fullsubnet_oracle as FO
        model = FastModel(**FO.DEFAULT_FAST_ARGS, **({"precision": args.precision} if "precision" in
                                                     FastModel.__init__.__code__.co_varnames else {}))
        model.load_state_dict(FO.make_fast_state_dict(seed=0), strict=True)
        model = model.to(dev).eval()
        precision = getattr(model, "_resolve_precision", lambda: "fp32")()
    else:
        model = Model(**O.DEFAULT_MODEL_ARGS, precision=args.precision)
        model.load_state_dict(O.make_state_dict(seed=0), strict=True)
        model = model.to(dev).eval()
        precision = model._resolve_precision()
    inf = Inferencer(model=model, device=dev) if imp_args is None else None
    host_in = O.make_noisy(B, L, seed=rank).pin_memory()  # every rank enhances its own clips
    host_out = torch.empty(B, L, dtype=torch.float32).pin_memory()
    x_dev = host_in.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, prof=False):
        for _ in range(warmup):
            fn()
        barrier()
        lib.fsn_set_profiling(1 if prof else 0)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stage = [0.0] * 4
        ev0.record()
        for _ in range(steps):
            flush.zero_()  # L2 flush between timed iterations (inside the region, ~0.1 ms)
            fn()
            if prof:
                torch.cuda.synchronize()
                for s in range(4):
                    stage[s] += max(0.0, lib.fsn_last_stage_ms(s))
        ev1.record()
        barrier()
        lib.fsn_set_profiling(0)
        ms = ev0.elapsed_time(ev1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, [s / steps for s in stage]

    last = {}  # output of the latest step_resident(): --dump-outputs writes the one of the last timed step

    def step_resident():
        if args.model == "fullsubnet":
            last["enhanced"] = model.enhance(x_dev, N_FFT, HOP, WIN)
        elif args.model == "improved_fullsubnet":
            with torch.no_grad():
                last["enhanced"] = model(x_dev)  # wav -> wav (improved_fullsubnet/model.py:541-591)
        else:
            last["enhanced"] = inf.enhance_batch(x_dev)

    def step_e2e():
        if args.model == "improved_fullsubnet":
            with torch.no_grad():
                out = model(host_in.to(dev, non_blocking=True))
        else:
            out = inf.enhance_batch(host_in)  # H2D inside
        host_out.copy_(out.reshape(B, L), non_blocking=True)  # D2H inside
        torch.cuda.current_stream().synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    ms_step, _ = timed(step_resident, args.steps, args.warmup)
    clocks = sampler.stop()
    launches = int(lib.fsn_last_launch_count())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, rank, world)
    # second pass with stage events on (separate from the headline timing)
    _, stage_ms = timed(step_resident, max(2, min(args.steps, 3)), 1, prof=True)
    ms_e2e, _ = timed(step_e2e, args.steps, 1)

    frames = B * T * world
    value = frames / (ms_step * 1e-3)
    e2e_value = frames / (ms_e2e * 1e-3)
    peaks, peak_kind = load_peaks()
    peak_tf = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    sb_flops = B * (T + 2) * FLOP_PER_FRAME_STEP_SB
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    tj = json.load(open(tpath)) if os.path.exists(tpath) else {}

    def sb_roofline(prec, sb_ms):
        """Tensor roofline of the sub-band stack: ALGORITHMIC FLOPs (SURVEY 8d; one product per MAC, whatever the
        number of MMA passes the precision needs) over the CUDA-event time of the stage."""
        achieved = sb_flops / (sb_ms * 1e-3) / 1e12 if sb_ms > 0 else None
        passes = {"f16x3_tc": 3, "f16_tc": 1}.get(prec)
        key = {"f16x3_tc": "sb_lstm_tc2_kernel<x3>", "f16_tc": "sb_lstm_tc2_kernel"}.get(prec)
        if prec == "f16_tc" and os.environ.get("FSN_TC_PAIR", "1") == "0":
            key = "sb_lstm_tc_kernel"
        r = {"kernel": f"sub-band LSTM stack ({prec})", "bound": "tensor" if passes else "fma", "achieved": achieved,
             "peak": peak_tf, "unit": "TFLOP/s", "frac": (achieved / peak_tf) if achieved else None,
             "traffic": tj.get(key, {}).get("dram_bytes_per_launch") if (key and B == 256) else None,
             "peak_source": f"{peak_kind} bf16_tflops_sustained (fp16 and bf16 share the dense tensor rate)",
             "flops_per_launch": sb_flops, "ms_per_launch": sb_ms}
        if passes:
            r["mma_passes"] = passes
            r["executed_frac"] = (passes * achieved / peak_tf) if achieved else None
        return r

    line = {
        "metric": "frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None,
        "dtype": {"f16_tc": "f16xf32acc", "f16x3_tc": "f16x3(hi+lo split, fp32-class)xf32acc"}.get(precision, "f32"),
        "data": "synthetic", "rtf_x": value / frame_rate,
        "config": {"workload": (f"fullsubnet inference, batch={B} x 4 s 16 kHz synthetic clips per GPU, "
                                "n_fft=512 hop=256 N=15, 2xLSTM-512 fb + 2xLSTM-384 sb (BASELINE configs[1])"
                                if args.model == "fullsubnet" else
                                (f"improved_fullsubnet inference ({args.variant}: n_fft={imp_args['n_fft']} "
                                 f"hop={imp_args['hop_length']}), batch={B} x 2 s synthetic clips per GPU (BASELINE configs[4])"
                                 if imp_args is not None else
                                 f"fast_fullsubnet inference, batch={B} x 4 s 16 kHz synthetic clips per GPU "
                                 "(BASELINE configs[3])")),
                   "clips_per_gpu": B, "frames_per_clip": T, "precision": precision,
                   "precision_note": "headline = the fastest arithmetic that meets BOTH parity gates (cRM 1e-3 rel, "
                                     "waveform 1e-4 abs) on BOTH weight sets W-a and W-b (tests/test_gpu_parity.py); "
                                     "single-pass f16_tc and fp32 are under `precisions`",
                   "l2": "256 MiB flush write between timed iterations", "parallelism": f"clips sharded x{world}"},
        "e2e": {"value": e2e_value, "unit": "frames/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": B * L * 4, "d2h_bytes_per_step": B * L * 4, "rtf_x": e2e_value / frame_rate},
        "gpu_launches": launches,
        "clocks": clocks,
        "stage_ms": {"stft": stage_ms[0], "fullband": stage_ms[1], "subband": stage_ms[2], "mask_istft": stage_ms[3]},
        "roofline": sb_roofline(precision, stage_ms[2]),
    }

    extras = args.model == "fullsubnet" and not args.no_extras
    if extras and args.precision == "auto":
        # the other arithmetic modes on the same workload (fewer iterations; same timing rules)
        line["precisions"] = {}
        for p in ("f16_tc", "fp32"):
            model.precision = p
            ms_p, _ = timed(step_resident, 2, 1)
            _, st_p = timed(step_resident, 2, 0, prof=True)
            line["precisions"][p] = {"ms_per_step": ms_p, "value": frames / (ms_p * 1e-3), "unit": "frames/s",
                                     "rtf_x": frames / (ms_p * 1e-3) / (SR / HOP),
                                     "stage_ms": {"fullband": st_p[1], "subband": st_p[2]},
                                     "roofline": sb_roofline(p, st_p[2]),
                                     "parity": {"f16_tc": "cRM gate on W-a and W-b, waveform gate on W-a only",
                                                "fp32": "both gates, both weight sets"}[p]}
        model.precision = args.precision
    if extras:
        # regime (ii) of SURVEY 8d: ONE 4 s clip (BASELINE configs[0] shape) - latency, not throughput
        x1 = x_dev[:1].contiguous()
        lat = {}
        for p in ([args.precision] if args.precision != "auto" else ["auto", "f16_tc", "fp32"]):
            model.precision = p
            for _ in range(3):
                model.enhance(x1, N_FFT, HOP, WIN)
            torch.cuda.synchronize()
            ts = []
            lib.fsn_set_profiling(1)
            st = [0.0] * 4
            for _ in range(10):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                model.enhance(x1, N_FFT, HOP, WIN)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
                for k in range(4):
                    st[k] += max(0.0, lib.fsn_last_stage_ms(k)) / 10
            lib.fsn_set_profiling(0)
            ms1 = sorted(ts)[len(ts) // 2]
            fb_bytes = 15.21e6  # SURVEY 8d: fp32 weights of the full-band stack one LSTM step touches
            lat[model._resolve_precision()] = {
                "ms_per_clip": ms1, "rtf_x": CLIP_SECONDS * 1e3 / ms1, "frames_per_sec": T / (ms1 * 1e-3),
                "stage_ms": {"stft": st[0], "fullband": st[1], "subband": st[2], "mask_istft": st[3]},
                "fullband_us_per_lstm_step": 1e3 * st[1] / (T + 2),
                "fullband_weight_stream": {
                    "bytes_per_step": fb_bytes, "achieved_gbs": fb_bytes / (1e-3 * st[1] / (T + 2)) / 1e9,
                    "hbm_peak_gbs": peaks.get("hbm_gbs"),
                    "frac_of_hbm_peak": fb_bytes / (1e-3 * st[1] / (T + 2)) / 1e9 / peaks.get("hbm_gbs", 6582.5),
                    "note": "the persistent kernel keeps the weights in shared memory for all 253 steps (HBM is read "
                            "once, 15.2 MB per launch); the figure is the SMEM-resident weight bytes one step consumes "
                            "over the step time, i.e. what an HBM-streaming GEMV would have to sustain to keep up; "
                            "the step is bound by the grid barrier + the h exchange through L2"}}
        model.precision = args.precision
        line["latency_b1"] = {"workload": "1 x 4 s clip (BASELINE configs[0] shape), inputs resident, median of 10",
                              "by_precision": lat}

    if rank == 0 and not args.no_cpu_baseline and world == 1:
        cores = pick_cpu_threads()
        v, dt = cpu_oracle_time(4, cores)
        line["cpu_baseline"] = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                                "sample": f"4 x 4 s clips, B=1 loop, torch CPU fp32 library calls "
                                          f"(oracle/libcall_port.py), {cores} threads (best median of a sweep "
                                          f"{_CPU_SWEEP} frames/s; host has {os.cpu_count()} logical cores), {dt:.1f} s",
                                "note": CPU_KIND_NOTE}
    if extras and not args.no_train:
        # BASELINE configs[2]: the training step with its gradient all-reduce - the one collective on the path
        del x_dev, flush
        torch.cuda.empty_cache()
        import bench_train
        targs = argparse.Namespace(**vars(args))
        targs.batch, targs.steps, targs.warmup, targs.dump_outputs = 64, max(2, min(args.steps, 5)), 3, None
        tl = bench_train.measure(targs, dist, dev, rank, world, local, cpu_leg=False)
        line["train_dp"] = {k: tl[k] for k in ("value", "unit", "ms_per_step", "n_gpus", "dtype", "gpu_launches")}
        line["train_dp"].update({"workload": tl["config"]["workload"], "parallelism": tl["config"]["parallelism"],
                                 "allreduce": tl.get("allreduce"), "e2e": tl["e2e"], "roofline": tl["roofline"]})
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
