#!/usr/bin/env python
"""bench.py -- clips/sec for 30 s audio -> beats (final0-shaped checkpoint) on N B200 GPUs.

    python bench.py --gpus 1 --steps K --warmup W            # our CUDA path, BASELINE config 2 (default)
    python bench.py --impl reference --gpus 1 --steps K ...  # the UNMODIFIED reference (baseline/_ref) on host cores
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --config 3|4|5 ...                       # the other BASELINE configs (files / --dbn / ragged)
    python bench.py --dump-outputs DIR ...                   # also write the last timed step's outputs as DIR/*.npy

One "step" = one pass of the hot path over one batch of `--batch` synthetic 30 s clips per GPU (BASELINE config 2:
Audio2Frames final0, batch 64; the minimal peak picker is included so that the step is audio -> beats).  Prints ONE
JSON line (rank 0).

value    : device-resident throughput (audio already in HBM; CUDA events; max over ranks); no per-kernel events.
e2e      : the reference-signature call -- Audio2Beats.batch(list of float64 numpy arrays as load_audio returns
           them) -- for steps*batch clips: threaded mono-mix/cast into pinned memory, H2D copy, all kernels, D2H of
           the timestamp arrays, every step, staging of step i+1 overlapping the kernels of step i.
roofline : the dominant kernel (time-direction flash attention, tcgen05) -- algorithmic FLOPs / CUDA-event time,
           measured live in a second timed pass with one event per launch (bt_profile_*).
parity   : the GPU results of the timed path checked against the CPU run of the cpu_baseline leg on the same clips.
cpu_baseline: the unmodified reference (kind "reference") -- or the oracle port when baseline/_ref is absent --
           timed on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

# stdout carries exactly ONE line, the JSON result: everything else that writes to file descriptor 1 -- Python
# prints, the NCCL version banner (printed from C at NCCL_DEBUG >= VERSION), library chatter -- goes to stderr.
_REAL_STDOUT = os.dup(1)
sys.stdout.flush()
os.dup2(2, 1)


def emit(line: dict) -> None:
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

from beat_this_b200.synthetic import cache_dir

SR = 22050
METRIC = "clips/sec (30 s audio->beats, final0)"
CACHE = cache_dir()
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": float(max(power)), "samples": len(sm)}


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def synth_clips(n_clips: int, seconds: float, seed0: int):
    """n distinct seeded clips, float64 mono in [-1, 1] -- what the reference's load_audio hands to Audio2Beats."""
    from beat_this_b200 import synthetic

    return [synthetic.synth_clip(seed0 + i, seconds) for i in range(n_clips)]


# ================================================================================== reference arm
def import_reference():
    """(beat_this.inference module of the UNMODIFIED reference, kind).  baseline/_ref = `pip install --no-deps
    --target baseline/_ref /root/reference`; the two third-party packages it imports that are not installable
    offline (rotary_embedding_torch, soxr) come from oracle/shims.  None when baseline/_ref is absent."""
    if not os.path.isdir(os.path.join(REF_DIR, "beat_this")):
        return None
    for p in (os.path.join(ROOT, "oracle", "shims"), REF_DIR):
        if p not in sys.path:
            sys.path.insert(0, p)
    try:
        import beat_this.inference as ref_inf

        if not os.path.abspath(ref_inf.__file__).startswith(os.path.abspath(REF_DIR)):
            return None
        return ref_inf
    except Exception as e:  # pragma: no cover
        print(f"reference import failed: {e}", file=sys.stderr)
        return None


class CpuArm:
    """The reference's CPU path: Audio2Beats(ckpt, "cpu", float16=False)(signal, sr) per clip, chunk by chunk, as
    it really runs (inference.py:215) -- through baseline/_ref when present, else the oracle port."""

    def __init__(self, seconds: float):
        from beat_this_b200 import synthetic

        self.ckpt = synthetic.write_checkpoint(os.path.join(CACHE, "final0_s0.ckpt"), "final0", 0)
        self.ref = import_reference()
        if self.ref is not None:
            self.kind = "reference"
            self.a2b = self.ref.Audio2Beats(self.ckpt, "cpu", False, False)
            self.what = "UNMODIFIED reference beat_this.inference.Audio2Beats (baseline/_ref, fp32, torch CPU)"
        else:
            from oracle import beat_this_oracle as O

            self.kind = "port"
            self.O = O
            self.sd = O.strip_prefix(torch.load(self.ckpt, weights_only=True)["state_dict"])
            self.what = "oracle port of the reference forward (oracle/beat_this_oracle.py, fp32, torch CPU)"
        self.seconds = seconds
        self.threads = self.calibrate()

    def run(self, x, want_logits=False):
        if self.kind == "reference":
            with torch.inference_mode():
                beat, down = self.ref.Audio2Frames.__call__(self.a2b, x, SR)
                bt, dt = self.a2b.frames2beats(beat, down)
        else:
            beat, down = self.O.spect2frames(self.sd, self.O.signal2spect(x, SR))
            bt, dt = self.O.postp_minimal(beat, down)
        return (bt, dt, beat.numpy(), down.numpy()) if want_logits else (bt, dt)

    def calibrate(self) -> int:
        """torch CPU ops get slower with more threads than the box can feed (128 logical CPUs: 10x slower than 16):
        time the REAL workload (one 30 s clip = two 1500-frame chunks) at a few thread counts, best of 2, keep the
        fastest.  The choice is printed and reported."""
        from beat_this_b200 import synthetic

        n = host_cores()
        # more than ~32 threads only slows torch's CPU kernels down on these shapes (measured on the 128-CPU bench
        # box: 64 threads 1.6-1.9 s per clip, 128 threads 22 s, 16 threads 0.33-0.47 s), so the sweep stops at 32
        cands = sorted({c for c in (min(n, 32), 24, 16, 12, 8) if 1 <= c <= n}, reverse=True)
        x = synthetic.synth_clip(999, self.seconds)
        best, best_t, table = cands[-1], float("inf"), {}
        for c in cands:
            torch.set_num_threads(c)
            self.run(x)
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                self.run(x)
                ts.append(time.perf_counter() - t0)
            table[c] = sorted(ts)[1]  # median of 3
            if table[c] < best_t:
                best, best_t = c, table[c]
        torch.set_num_threads(best)
        print("cpu arm thread calibration (s per clip): " + ", ".join(f"{c}: {t:.2f}" for c, t in table.items()) + f" -> {best}", file=sys.stderr)
        self.table = table
        return best


def run_reference(args, rank, world):
    if rank != 0:
        return
    arm = CpuArm(args.seconds)
    n = args.ref_clips_per_step
    clips = synth_clips(n, args.seconds, 1000)
    for _ in range(max(1, min(args.warmup, 2))):
        arm.run(clips[0])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for c in clips:
            arm.run(c)
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    sample = (f"{n} clip(s) of {args.seconds:g} s per step x {args.steps} steps, {arm.what}, {arm.threads} threads "
              f"(calibrated on a full clip; {host_cores()} usable CPUs)")
    emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "clips/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"Audio2Beats final0-shaped synthetic checkpoint, {args.seconds:g} s clips @22.05 kHz mono, minimal peak picking",
                   "batch_per_gpu": n, "bounded_sample": sample, "device": "host CPU (no GPU work)"},
        "cpu_baseline": {"value": value, "unit": "clips/s", "cores": arm.threads, "kind": arm.kind, "sample": sample},
        "e2e": {"value": value, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ================================================================================== parity helpers
def peak_mismatch_report(ref_logits, our_logits, ref_times, our_times, err):
    """Frames whose peak decision differs between two logit curves, and whether the reference's decision margin at
    that frame (distance to the `> 0` threshold / to the competing maximum in the +-3 window, postprocessor.py:95-99)
    is within 2*err -- i.e. the flip is explained by the measured logit error, not by a bug."""
    def peaks(x):
        T = len(x)
        pad = np.full(T + 6, -np.inf, dtype=np.float64)
        pad[3:T + 3] = x
        win = np.stack([pad[k:k + T] for k in range(7)])
        mx = win.max(0)
        others = np.delete(win, 3, axis=0).max(0)
        return (x == mx) & (x > 0), others

    pr, others = peaks(ref_logits.astype(np.float64))
    po, _ = peaks(our_logits.astype(np.float64))
    diff = np.flatnonzero(pr != po)
    unexplained = 0
    for t in diff:
        x = float(ref_logits[t])
        margin = min(x, x - others[t]) if pr[t] else max(-x, others[t] - x)
        if abs(margin) > 2 * err + 1e-6:
            unexplained += 1
    same = len(ref_times) == len(our_times) and np.array_equal(np.asarray(ref_times), np.asarray(our_times))
    return {"frames_differing": int(len(diff)), "unexplained": int(unexplained), "times_identical": bool(same)}


def cpu_baseline_and_parity(args, gpu_run, budget_s: float = 25.0):
    """Time the CPU arm on a bounded sample of the bench workload and check the GPU path against it on those clips."""
    arm = CpuArm(args.seconds)
    clips = synth_clips(min(8, args.batch), args.seconds, 2000)  # the first clips of the rank-0 bench batch
    arm.run(clips[0])
    cpu, t0 = [], time.perf_counter()
    for c in clips:
        cpu.append(arm.run(c, want_logits=True))
        if time.perf_counter() - t0 > budget_s:
            break
    el = time.perf_counter() - t0
    n = len(cpu)
    base = {"value": n / el, "unit": "clips/s", "cores": arm.threads, "kind": arm.kind,
            "sample": f"{n} x {args.seconds:g} s clip(s), {arm.what}, {arm.threads} threads (calibrated on a full clip), {el:.1f} s"}
    frames, beats = gpu_run(clips[:n])
    par = {"clips": n, "max_abs_logit_err": 0.0, "beats_ref": 0, "clips_with_identical_timestamps": 0,
           "peak_frames_differing": 0, "unexplained_by_margin": 0}
    for (bt, dt, rb, rd), (b, d), (gbt, gdt) in zip(cpu, frames, beats):
        b, d = b.cpu().numpy(), d.cpu().numpy()
        err = float(max(np.abs(b - rb).max(), np.abs(d - rd).max()))
        par["max_abs_logit_err"] = max(par["max_abs_logit_err"], err)
        rep_b = peak_mismatch_report(rb, b, bt, gbt, err)
        rep_d = peak_mismatch_report(rd, d, dt, gdt, err)
        par["beats_ref"] += len(bt)
        par["clips_with_identical_timestamps"] += int(rep_b["times_identical"] and rep_d["times_identical"])
        par["peak_frames_differing"] += rep_b["frames_differing"] + rep_d["frames_differing"]
        par["unexplained_by_margin"] += rep_b["unexplained"] + rep_d["unexplained"]
    par["against"] = f"{arm.kind} CPU run of the same clips (fp32)"
    return base, par


def gpu_reference_arm(args, dev, n_clips=8):
    """The unmodified reference on the SAME GPU (eager PyTorch, float16=True autocast): the 'existing Blackwell path'."""
    ref = import_reference()
    if ref is None:
        return None
    from beat_this_b200 import synthetic

    try:
        ckpt = synthetic.write_checkpoint(os.path.join(CACHE, "final0_s0.ckpt"), "final0", 0)
        a2b = ref.Audio2Beats(ckpt, str(dev), True, False)
        clips = synth_clips(n_clips, args.seconds, 2000)
        a2b(clips[0], SR)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for c in clips:
            a2b(c, SR)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        return {"value": n_clips / dt, "unit": "clips/s", "what": "UNMODIFIED reference Audio2Beats(device=cuda, float16=True), eager PyTorch, one clip per call",
                "clips": n_clips}
    except Exception as e:
        return {"unavailable": f"{type(e).__name__}: {e}"[:200]}


# ================================================================================== our arm
def make_model(args, dev, rank):
    from beat_this_b200 import synthetic
    from beat_this_b200.distributed import load_model_distributed

    ckpt = synthetic.write_checkpoint(os.path.join(CACHE, "final0_s0.ckpt"), "final0", 0) if rank == 0 else None
    return load_model_distributed(ckpt, dev, float16=not args.float32, wave_chunks=args.wave)


def reduce_max(world, dev, *vals):
    import torch.distributed as dist

    if world == 1:
        return vals
    t = torch.tensor(vals, dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return tuple(float(v) for v in t)


def reduce_sum(world, dev, v):
    import torch.distributed as dist

    if world == 1:
        return v
    t = torch.tensor([v], dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return int(t[0])


DUMP_LIMIT_BYTES = 63 << 20  # array data; with the .npy headers the files stay below 64 MB


def dump_outputs(out_dir: str, beat: torch.Tensor, down: torch.Tensor, times: list) -> None:
    """Write what one step of the timed path returned, so that two builds can be compared output for output:
    beat_logits / downbeat_logits (float32, [clips, frames]; every clip of the batch has the same length),
    beat_times / downbeat_times (float64, all clips concatenated) with beat_counts / downbeat_counts per clip, and
    clip_index, the clips of the batch they belong to.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of
    clips is written."""
    n = len(times)
    beat = beat.view(n, -1).cpu().numpy()
    down = down.view(n, -1).cpu().numpy()
    size = np.asarray([beat.shape[1] * 8 + (len(b) + len(d) + 3) * 8 for b, d in times])
    keep = np.arange(n)
    if size.sum() > DUMP_LIMIT_BYTES:
        order = np.random.default_rng(0).permutation(n)
        keep = np.sort(order[np.cumsum(size[order]) <= DUMP_LIMIT_BYTES])
    out = {
        "beat_logits": beat[keep],
        "downbeat_logits": down[keep],
        "beat_times": np.concatenate([times[i][0] for i in keep]).astype(np.float64),
        "downbeat_times": np.concatenate([times[i][1] for i in keep]).astype(np.float64),
        "beat_counts": np.asarray([len(times[i][0]) for i in keep], dtype=np.float64),
        "downbeat_counts": np.asarray([len(times[i][1]) for i in keep], dtype=np.float64),
        "clip_index": keep.astype(np.float64),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), arr)
    print(f"outputs of the last timed step ({len(keep)} of {n} clips) written to {out_dir}", file=sys.stderr)


def run_ours(args, rank, world, local):
    import torch.distributed as dist

    from beat_this_b200.inference import Audio2Beats, Audio2Frames

    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    half = not args.float32
    a2b = Audio2Beats.from_model(make_model(args, dev, rank))
    eng = a2b.model.engine
    act = eng.act_dtype

    clips = synth_clips(args.batch, args.seconds, 2000 + 100 * rank)  # float64, as load_audio returns them
    so = [0]
    for c in clips:
        so.append(so[-1] + len(c))
    host = torch.empty(so[-1], dtype=torch.float32, pin_memory=True)
    a2b.pipeline.stage_signals(clips, host)
    audio_dev = host.to(dev)
    fo = eng.frame_offsets(so)
    n_chunks = sum(int(eng.lib.bt_plan_chunks(fo[i + 1] - fo[i], None, None, 0)) for i in range(len(clips)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step_device():
        beat, down, f = eng.audio2frames_cat(audio_dev, so)
        return beat, down, eng.peakpick_cat(beat, down, f)

    def timed_device_steps():
        """(elapsed ms, what the last step returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            out = step_device()
        e1.record()
        barrier()
        return e0.elapsed_time(e1), out

    # ---- device-resident timing (no per-kernel events) ----------------------------------------------------
    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = eng.launches
    ms, last_step = timed_device_steps()
    launches = eng.launches - l0
    clocks = sampler.stop()
    # ---- second timed pass with one CUDA event per launch: per-kernel times for the roofline ---------------
    eng.profile_reset()
    eng.profile_enable(True)
    ms_prof, _ = timed_device_steps()
    eng.profile_enable(False)
    prof = eng.profile_results()
    # ---- end to end through the reference-signature API ---------------------------------------------------
    many = [clips[i % len(clips)] for i in range(args.batch * args.steps)]
    a2b.batch(clips, SR)  # warm-up: pinned ring, streams
    a2b.batch(clips + clips, SR)
    pipe = a2b.pipeline
    barrier()
    h0, d0 = pipe.h2d_bytes, pipe.d2h_bytes
    t0 = time.perf_counter()
    res = a2b.batch(many, SR)
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    h2d, d2h = (pipe.h2d_bytes - h0) // args.steps, (pipe.d2h_bytes - d0) // args.steps
    assert len(res) == len(many) and all(r is not None for r in res)
    # one synchronous call per step (no overlap across calls), for transparency
    t0 = time.perf_counter()
    for _ in range(min(args.steps, 5)):
        a2b.batch(clips, SR)
    sync_s = (time.perf_counter() - t0) / min(args.steps, 5)

    ms, ms_prof, e2e_ms, sync_ms = reduce_max(world, dev, ms, ms_prof, e2e_s * 1000.0, sync_s * 1000.0)
    launches = reduce_sum(world, dev, launches)
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last_step)
    peaks, peak_src = load_peaks()
    total_clips = args.batch * world
    value = total_clips * args.steps / (ms / 1000.0)
    e2e_value = total_clips * args.steps / (e2e_ms / 1000.0)
    # roofline of the dominant kernel: time-direction attention (frontend + main layers).
    # algorithmic FLOPs = 4 * L^2 * d per (sequence, head) (QK^T and PV, 2 flops per MAC), L = chunk length
    D = eng.hparams.get("transformer_dim", 512)
    headseqs_per_chunk = 3 * 32 + eng.hparams.get("n_layers", 6) * (D // 32)
    Lc = 1500 if args.seconds >= 29.76 else fo[1] + 12
    attn_flops = 4.0 * Lc * Lc * 32 * headseqs_per_chunk * n_chunks * args.steps
    key = "attn_time_tc" if half else "attn_time_simt"
    a_ms, a_n = prof.get(key, (0.0, 0))
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "attn_traffic.json")
    if half and os.path.exists(tpath) and args.batch == 64 and args.seconds == 30.0:
        with open(tpath) as f:
            tj = json.load(f)
        traffic, traffic_src = tj.get("dram_bytes_per_launch_mean"), tj.get("source")
    roof = {"bound": "tensor", "kernel": key, "achieved": (attn_flops / (a_ms / 1000.0) / 1e12) if a_ms > 0 else None,
            "peak": peak_tf, "peak_source": f"{peak_src} bf16_tflops_sustained (fp16 and bf16 tcgen05 run at the same rate; kernel timed inside a long step)",
            "unit": "TFLOP/s", "traffic": traffic, "traffic_source": traffic_src, "launches": a_n, "avg_launch_ms": (a_ms / a_n) if a_n else None,
            "algorithmic_flops_per_launch": attn_flops / a_n if a_n else None,
            "timed_in": f"second timed pass of {args.steps} steps with one CUDA event per launch ({ms_prof / args.steps:.2f} ms/step vs {ms / args.steps:.2f} without)"}
    roof["frac"] = (roof["achieved"] / peak_tf) if roof["achieved"] else None
    tot_ms = sum(v[0] for v in prof.values()) or 1.0
    shares = {k: {"ms_per_step": round(v[0] / args.steps, 3), "launches_per_step": v[1] // max(1, args.steps), "share": round(v[0] / tot_ms, 4)}
              for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    line = {
        "metric": METRIC, "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": act, "data": "synthetic",
        "config": {"workload": f"Audio2Beats final0-shaped synthetic checkpoint (seeded random weights), batch {args.batch} x {args.seconds:g} s clips "
                               f"@22.05 kHz mono per GPU ({n_chunks} chunks of {Lc} frames, {args.batch} distinct clips), log-mel + BeatThis forward + minimal peak picking",
                   "batch_per_gpu": args.batch, "global_batch": total_clips, "parallelism": f"dp{world} (clips sharded, weights broadcast once over NCCL)",
                   "wave_chunks": args.wave, "l2_policy": f"inputs larger than L2: {so[-1] * 4 / 1e6:.0f} MB audio per step per GPU; activations stream through HBM",
                   "operands": f"{act} tcgen05 operands, fp32 accumulate, fp32 residual stream" if half else "fp32 CUDA cores"},
        "roofline": roof, "kernel_time_shares": shares,
        "e2e": {"value": e2e_value, "unit": "clips/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_ms / args.steps,
                "api": f"beat_this_b200.inference.Audio2Beats.batch(list of {args.batch * args.steps} float64 numpy signals, sr=22050) -> list of (beats, downbeats); "
                       "internally groups of 64 clips: threaded mono-mix + fp32 cast into a pinned ring, H2D, kernels, D2H, staging of group g+1 overlapping the kernels of group g",
                "one_call_per_step": {"value": total_clips / (sync_ms / 1000.0), "ms_per_step": sync_ms,
                                      "api": f"Audio2Beats.batch(list of {args.batch} signals), one synchronous call per step (nothing overlaps across calls)"},
                "host_threads": pipe.host_threads},
        "gpu_launches": int(launches), "clocks": clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        def gpu_run(cs):
            return Audio2Frames.batch(a2b, cs, SR), a2b.batch(cs, SR)

        line["cpu_baseline"], line["parity"] = cpu_baseline_and_parity(args, gpu_run)
        if not args.no_gpu_reference:
            line["reference_on_this_gpu"] = gpu_reference_arm(args, dev)
    emit(line)


# ================================================================================== other BASELINE configs
def run_config(args, rank, world, local):
    """--config 3: File2Beats over int16 WAV files; 4: Audio2Beats --dbn; 5: ragged 5-300 s Audio2Frames.  Clips are
    sharded over the ranks (3, 4: round robin; 5: by chunk count), no collective on the path; time = max over ranks."""
    import torch.distributed as dist

    from beat_this_b200 import synthetic
    from beat_this_b200.distributed import shard_by_cost
    from beat_this_b200.inference import Audio2Beats, Audio2Frames, File2Beats

    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    model = make_model(args, dev, rank)
    eng = model.engine
    cfg = args.config
    extra = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    if cfg == 3:
        from scipy.io import wavfile

        n_total, n_distinct = args.clips or 10000, 256
        wdir = os.path.join(CACHE, "wavs30")
        os.makedirs(wdir, exist_ok=True)
        for i in range(rank, n_distinct, world):  # every rank writes its share of the distinct files (untimed)
            p = os.path.join(wdir, f"clip{i:03d}.wav")
            if not os.path.exists(p):
                x = synthetic.synth_clip(5000 + i, args.seconds)
                wavfile.write(p + ".tmp.wav", SR, np.clip(np.round(x * 32767.0), -32768, 32767).astype(np.int16))
                os.replace(p + ".tmp.wav", p)
        barrier()
        mine = [os.path.join(wdir, f"clip{(i % n_distinct):03d}.wav") for i in range(rank, n_total, world)]
        runner = File2Beats.from_model(model)
        runner.batch(mine[:128])  # warm-up
        barrier()
        t0 = time.perf_counter()
        res = runner.batch(mine)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        n_mine, units = len(mine), n_total
        workload = (f"File2Beats.batch over {n_total} int16 mono WAV files of {args.seconds:g} s ({n_distinct} distinct seeded files on local disk, cycled; "
                    f"page cache warm), sharded i % {world}: native threaded WAV decode -> pinned ring -> device -> timestamps")
    elif cfg == 4:
        n_total = args.clips or 1000
        base = synth_clips(64, args.seconds, 7000 + 100 * rank)
        mine_idx = list(range(rank, n_total, world))
        mine = [base[i % 64] for i in mine_idx]
        runner = Audio2Beats.from_model(model, dbn=True)
        runner.batch(mine[:128], SR)
        barrier()
        t0 = time.perf_counter()
        res = runner.batch(mine, SR)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        n_mine, units = len(mine), n_total
        impl = type(runner.frames2beats.dbn).__name__
        workload = (f"Audio2Beats(dbn=True).batch over {n_total} clips of {args.seconds:g} s (64 distinct), device frames + host DBN ({impl}; "
                    "madmom itself is not installable offline), DBN of group g overlapping the kernels of group g+1")
    else:
        n_total = args.clips or 512
        rng = np.random.default_rng(7)
        secs = rng.uniform(5.0, 300.0, n_total)
        frames = [1 + int(s * SR) // 441 for s in secs]
        costs = [int(eng.lib.bt_plan_chunks(f, None, None, 0)) for f in frames]
        shards = shard_by_cost(costs, world)
        mine_idx = shards[rank]
        mine = []
        for i in mine_idx:  # cheap seeded audio: noise + a click track (kernels are data independent)
            n = int(secs[i] * SR)
            g = np.random.default_rng(9000 + i)
            x = (0.05 * g.standard_normal(n)).astype(np.float32)
            x[:: int(SR * 60.0 / g.uniform(60, 180))] += 0.8
            mine.append(x)
        runner = Audio2Frames.from_model(model)
        runner.batch(mine[: max(4, len(mine) // 2)], SR)  # warm-up: pinned staging ring (3 slots), plans of common lengths
        barrier()
        t0 = time.perf_counter()
        res = runner.batch(mine, SR)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        n_mine, units = len(mine), n_total
        my_chunks = sum(costs[i] for i in mine_idx)
        short = sum(1 for i in mine_idx if frames[i] <= 1488)
        if world > 1:
            t = torch.tensor([my_chunks, short, int(dt * 1e6)], dtype=torch.int64, device=dev)
            allv = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allv, t)
            per = [[int(v) for v in a] for a in allv]
        else:
            per = [[my_chunks, short, int(dt * 1e6)]]
        ch = [p[0] for p in per]
        extra = {"chunks_per_rank": ch, "short_chunks_per_rank": [p[1] for p in per], "seconds_per_rank": [p[2] / 1e6 for p in per],
                 "chunk_imbalance_max_over_mean": max(ch) / (sum(ch) / len(ch)), "total_chunks": sum(ch),
                 "equivalent_30s_clips_per_s": None}
        workload = (f"Audio2Frames.batch over {n_total} clips of 5-300 s (rng(7).uniform), sharded by chunk count (greedy longest first); "
                    "full 1500-frame chunks batch into waves of <=128, every short clip (<29.76 s) is a wave of its own length")
    assert len(res) == n_mine and all(r is not None for r in res)
    st = runner.pipeline.stats
    extra["host_pipeline_rank0"] = {k: (round(v, 4) if isinstance(v, float) else v) for k, v in st.items()}
    extra["host_pipeline_rank0"]["host_threads"] = runner.pipeline.host_threads
    extra["host_pipeline_rank0"]["note"] = "seconds on the calling thread since the runner was created (warm-up included)"
    (dt_max,) = reduce_max(world, dev, dt)
    if rank != 0:
        return
    value = units / dt_max
    if cfg == 5:
        extra["equivalent_30s_clips_per_s"] = extra["total_chunks"] / 2.0 / dt_max
    emit({"metric": {3: "clips/sec (30 s WAV file -> beats, final0)", 4: "clips/sec (30 s audio -> beats with --dbn, final0)",
                     5: "clips/sec (5-300 s audio -> frames, final0)"}[cfg],
          "value": value, "unit": "clips/s", "n_gpus": world, "steps": 1, "warmup": 1, "ms_per_step": dt_max * 1000.0,
          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": eng.act_dtype, "data": "synthetic",
          "config": {"workload": workload, "baseline_config": cfg, "clips": units, "parallelism": f"dp{world}"},
          "e2e": {"value": value, "unit": "clips/s", "api": type(runner).__name__ + ".batch", "note": "host buffers / files in, host results out: the timed call is end to end"},
          "gpu_launches": int(reduce_sum(1, dev, eng.launches)), **extra})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json config (2 = the headline bench line)")
    ap.add_argument("--clips", type=int, default=0, help="configs 3/4/5: total clips over all ranks (default 10000 / 1000 / 512)")
    ap.add_argument("--batch", type=int, default=64, help="clips per GPU per step")
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--wave", type=int, default=128, help="chunks per wave (one wave = one launch of every kernel)")
    ap.add_argument("--float32", action="store_true", help="fp32 CUDA-core path instead of the 16-bit tcgen05 path")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--ref-clips-per-step", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", help="config 2: write the logits and beat / downbeat times of the "
                    "last timed step (rank 0) as .npy files to DIR")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "ours" or args.config != 2):
        ap.error("--dump-outputs writes the outputs of the config 2 timed path (--impl ours)")
    from beat_this_b200.distributed import init_from_env

    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        run_reference(args, rank, int(os.environ.get("WORLD_SIZE", "1")))
        return
    rank, world, local = init_from_env("nccl")
    try:
        if args.config == 2:
            run_ours(args, rank, world, local)
        else:
            run_config(args, rank, world, local)
    finally:
        import torch.distributed as dist

        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
