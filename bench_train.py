"""bench_train.py - FullSubNet TRAINING step on B200 (BASELINE configs[2]: batch = 64 x 3 s clips per GPU, cIRM MSE
loss, data-parallel with one gradient all-reduce).  Same JSON contract as bench.py (which dispatches here for
``--model fullsubnet_train``).

One "step" = fullsubnet/trainer.py:41-71: STFT of noisy + clean -> cIRM target (+ drop_band) -> Model.forward ->
MSE -> backward (BPTT) -> [all-reduce of the flat gradient buffer] -> clip_grad_norm_(10) -> Adam.  `value` has
the waveforms resident in HBM; `e2e` feeds pinned HOST waveforms (H2D inside) and reads the loss back (D2H inside).
Weak scaling: every rank trains on its own 64 clips, like the reference's per-rank batch_size (train.py:38-43).
"""
from __future__ import annotations

import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR, N_FFT, HOP, WIN = 16000, 512, 256, 512
CLIP_SECONDS = 3
FLOP_FWD_PER_FRAME_STEP = 7_607_296 + 128 * 3_638_784  # SURVEY 8d cfg3: full band + 128 kept sub-band units


def cpu_train_time(n_clips: int, threads: int):
    from oracle import fullsubnet_oracle as O
    from oracle import train_oracle as TO
    torch.set_num_threads(threads)
    sd = O.make_state_dict(seed=0)
    L = SR * CLIP_SECONDS
    noisy, clean = O.make_noisy(n_clips, L, seed=0), 0.5 * O.make_noisy(n_clips, L, seed=100)
    t0 = time.perf_counter()
    TO.train_step(noisy, clean, sd)
    dt = time.perf_counter() - t0
    return n_clips * (1 + L // HOP) / dt, dt


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from bench import pick_cpu_threads
    cores = pick_cpu_threads()
    n_clips = 3
    vals = []
    t_all = time.perf_counter()
    for _ in range(args.steps):
        vals.append(cpu_train_time(n_clips, cores)[0])
    dt = time.perf_counter() - t_all
    v = sorted(vals)[len(vals) // 2]
    print(json.dumps({
        "impl": "reference", "metric": "frames_per_sec", "value": v, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "fullsubnet training step, 3 s 16 kHz clips, cIRM MSE (CPU: 3 clips per step)"},
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{n_clips} x 3 s clips per step, oracle port of trainer.py:41-68 (torch CPU "
                                   f"autograd, fp32), {cores} threads"},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def main(args):
    if args.impl == "reference":
        return run_reference(args)
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
    line = measure(args, dist, dev, rank, world, local, cpu_leg=not args.no_cpu_baseline)
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def measure(args, dist, dev, rank, world, local, cpu_leg=True):
    """One measurement of the training step on an initialised process group (``dist`` = torch.distributed or None);
    returns the JSON line as a dict.  bench.py embeds it as `train_dp` next to the inference numbers."""
    from bench import ClockSampler, dump_outputs, load_peaks, pick_cpu_threads
    from fullsubnet_b200 import _lib
    from fullsubnet_b200.fullsubnet.model import Model
    from fullsubnet_b200.loss import mse_loss
    from fullsubnet_b200.optim import FusedClipAdam
    from fullsubnet_b200.trainer import Trainer
    from oracle import fullsubnet_oracle as O  # weights / inputs generator only (+ cpu_baseline leg)

    lib = _lib.load()
    B = args.batch if args.batch != 256 else 64  # bench.py's default batch belongs to the inference config
    L = SR * CLIP_SECONDS
    T = 1 + L // HOP
    margs = dict(O.DEFAULT_MODEL_ARGS, weight_init=False)
    model = Model(**margs)
    model.load_state_dict(O.make_state_dict(seed=0), strict=True)  # identical replicas on every rank
    model = model.to(dev).train()
    cfg = {"meta": {"use_amp": False, "save_dir": "/tmp/fsn_bench", "experiment_name": "bench"},
           "acoustics": {"n_fft": N_FFT, "hop_length": HOP, "win_length": WIN},
           "trainer": {"train": {"epochs": 1, "save_checkpoint_interval": 1, "clip_grad_norm_value": 10}}}
    trainer = Trainer(dist, local, cfg, False, False, model, mse_loss(), FusedClipAdam(model.parameters(), lr=1e-3),
                      None, None)
    host_noisy = O.make_noisy(B, L, seed=rank).pin_memory()
    host_clean = (0.5 * O.make_noisy(B, L, seed=100 + rank)).pin_memory()
    dev_noisy, dev_clean = host_noisy.to(dev), host_clean.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    host_loss = torch.empty((), dtype=torch.float32).pin_memory()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            flush.zero_()
            fn()
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    last = {}

    def step_resident():
        last["loss"] = trainer.train_step(dev_noisy, dev_clean)

    def step_e2e():
        loss = trainer.train_step(host_noisy, host_clean)  # H2D of both waveforms inside
        host_loss.copy_(loss, non_blocking=True)  # the reference's loss.item() (trainer.py:71)
        torch.cuda.current_stream().synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    ms_step = timed(step_resident, args.steps, args.warmup)
    clocks = sampler.stop()
    if args.dump_outputs:  # the loss of the last timed step and the parameters its Adam update left
        dump_outputs(args.dump_outputs, dict(last, **{"param." + k: p for k, p in model.named_parameters()}), rank, world)
    n0 = lib.fsn_total_launch_count()
    step_resident()
    torch.cuda.synchronize()
    launches = int(lib.fsn_total_launch_count() - n0)
    ms_e2e = timed(step_e2e, args.steps, 1)
    allreduce = None
    if dist is not None:  # the collective alone: K all-reduces of the flat gradient buffer, device-timed, max over ranks
        flat = model.flat_grad()
        for _ in range(3):
            dist.all_reduce(flat)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(20):
            dist.all_reduce(flat)
        ev1.record()
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1) / 20], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ar_ms = float(t.item())
        nbytes = flat.numel() * 4
        allreduce = {"ms": ar_ms, "bytes": nbytes, "ranks": world, "backend": "nccl",
                     "busbw_gbs": 2 * (world - 1) / world * nbytes / (ar_ms * 1e-3) / 1e9,
                     "share_of_step": ar_ms / ms_step}

    frames = B * T * world
    value, e2e_value = frames / (ms_step * 1e-3), frames / (ms_e2e * 1e-3)
    peaks, peak_kind = load_peaks()
    flops = 3.0 * B * (T + 2) * FLOP_FWD_PER_FRAME_STEP  # forward + 2x for backward (dX and dW)
    achieved = flops / (ms_step * 1e-3) / 1e12
    peak_tf = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    precision = model._resolve_train_precision()
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if precision == "tf32_tc" and os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("tgemm_tma_kernel", {}).get("dram_bytes_per_launch")
    line = {
        "metric": "frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "tf32+f16 operands, f32 accumulate/state" if precision == "tf32_tc" else "f32", "data": "synthetic",
        "rtf_x": value / (SR / HOP),
        "config": {"workload": f"fullsubnet training step, batch={B} x 3 s 16 kHz synthetic clips per GPU, cIRM MSE "
                               "loss, drop_band G=2, clip 10 + Adam 1e-3 (BASELINE configs[2])",
                   "clips_per_gpu": B, "frames_per_clip": T, "precision": precision,
                   "l2": "256 MiB flush write between timed iterations",
                   "parallelism": f"dp{world}: one all-reduce of the 22.55 MB flat gradient buffer per step"},
        "e2e": {"value": e2e_value, "unit": "frames/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": 2 * B * L * 4,
                "d2h_bytes_per_step": 4},
        "gpu_launches": launches, "clocks": clocks,
        "roofline": {"kernel": "whole training step; tcgen05 kernels: lstm_fwd_step_kernel (fused recurrent GEMM + cell, "
                               "kind::f16 / tf32) and tgemm_tma_kernel (kind::tf32: BPTT and weight-gradient GEMMs), "
                               "together about 60 % of the step (profiles/r02h_train_step_launches_summary.txt)"
                               if precision == "tf32_tc" else "whole training step (fp32 FMA GEMMs)",
                     "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": achieved / peak_tf, "traffic": traffic,
                     "peak_source": f"{peak_kind} bf16_tflops_sustained (the dense tf32 rate is half of it)",
                     "flops_per_launch": flops, "ms_per_launch": ms_step,
                     "note": "achieved = algorithmic FLOPs of the whole step (3 x forward) / step time; traffic = DRAM "
                             "bytes of one BPTT-step GEMM launch (profiles/traffic.json)"},
    }
    line["allreduce"] = allreduce
    if rank == 0 and cpu_leg and world == 1:
        cores = pick_cpu_threads()
        v, dt = cpu_train_time(3, cores)
        line["cpu_baseline"] = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                                "sample": f"one step on 3 x 3 s clips, oracle port of trainer.py:41-68 (torch CPU "
                                          f"autograd fp32), {cores} threads, {dt:.1f} s"}
    del trainer, model, dev_noisy, dev_clean, flush
    torch.cuda.empty_cache()
    return line


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss and parameters after the last timed step")
    main(ap.parse_args())
