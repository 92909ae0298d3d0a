#!/usr/bin/env python
"""Benchmark of the FLowHigh `generate` hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): midpoint ODE (2 NFE), batch of 64 x 10 s clips, 12 kHz -> 48 kHz,
basic_cfm, transformer 2L x 16H x 64, BigVGAN 48 kHz / 256-band (ASSUMED vocoder config, SURVEY A.6),
random-init weights, synthetic speech-like audio, 16-bit tensor-core path (fp16 operands by default,
--precision bf16 selects bfloat16: same MMA rate and bytes).  One "step" = one pass of the
whole path (resample -> log-mel -> CFM -> vocoder -> post-processing) over one batch per GPU.

  value : 48 kHz audio-seconds produced per wall second, whole job, inputs resident in HBM
  e2e   : same through the public API (FlowHighSR.generate_batch) from pinned host buffers, H2D and
          D2H copies inside the timed region
  roofline : the dominant kernel (tcgen05 implicit-GEMM conv), algorithmic FLOPs / CUDA-event time
  cpu_baseline : the oracle port of the reference (fp32 PyTorch-CPU restatement) on a bounded sample

N > 1: launched by torchrun, one rank per GPU, each rank runs its own batch (weak scaling, clips are
independent: no data-path collective); time = max over ranks.

--dump-outputs DIR: after the timed steps, rank 0 writes the waveforms its last timed step returned as
DIR/audio.npy (float32).  Inputs, noise and weights come from fixed seeds, so two builds run with the same
arguments can be compared output for output; an output above DUMP_BYTES is cut to a fixed seeded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "48kHz audio-sec/sec (whole job)"
UNIT = "audio-s/s"
CLIP_SECONDS = 10.0
SR_IN = 12000
BATCH = 64
STEPS_ODE = 1  # time_step = 1, midpoint -> 2 NFE
DUMP_BYTES = 48 << 20  # --dump-outputs: bound on what one run writes (batch64 at B = 64: 26 of the 64 clips)


def config_dict(n_gpus, batch):
    return {
        "workload": f"configs[1]: {batch} x 10 s clips/GPU, 12 kHz -> 48 kHz, basic_cfm, midpoint (2 NFE), "
                    "transformer 2Lx16Hx64, BigVGAN 48k/256-band (assumed cfg: rates 5,4,3,2,2,2, C0 1536, "
                    "AMPBlock1 k 3/7/11 d 1/3/5, snakebeta), random-init weights",
        "clips_per_gpu": batch, "clip_seconds": CLIP_SECONDS, "sr_in": SR_IN, "sr_out": 48000, "nfe": 2,
        "parallelism": f"clips sharded over {n_gpus} GPU(s), no data-path collective",
        "l2_policy": "per-step working set (>= 40 GB of activations) far exceeds the 126 MB L2; no flush needed",
    }


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d["bf16_tflops_sustained"], "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw,power.limit")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower() == "active" for r in self.rows)]
        def col(i):
            out = []
            for r in self.rows:
                try:
                    out.append(float(r[i]))
                except (IndexError, ValueError):
                    pass
            return out
        pw, pl = col(6), col(7)
        # the step is energy-bound at the board power cap (DESIGN.md section 4): the draw belongs next to the clock
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "sm_mhz_min": min(sm) if sm else None, "sm_mhz_peak": max(sm) if sm else None,
                "reasons": reasons, "samples": len(sm), "power_w": statistics.median(pw) if pw else None,
                "power_limit_w": max(pl) if pl else None}


def dump_outputs(path, name, out):
    """Writes `out` as <path>/<name>.npy in float32.  Above DUMP_BYTES, whole rows (clips) drawn with a fixed seed
    are kept, in ascending order; a single row longer than that is cut to fixed seeded sample positions instead."""
    import torch
    a = out.detach().float()
    if a.numel() * 4 > DUMP_BYTES:
        rng = np.random.default_rng(0)
        row = a[0].numel() * 4
        if a.shape[0] > 1 and row <= DUMP_BYTES:
            idx = np.sort(rng.choice(a.shape[0], DUMP_BYTES // row, replace=False))
        else:
            a = a.flatten()
            idx = np.sort(rng.choice(a.numel(), DUMP_BYTES // 4, replace=False))
        a = a[torch.from_numpy(idx).to(a.device)]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, name + ".npy"), a.cpu().numpy())


# ------------------------------------------------------------------------------------------- CPU arm
def cpu_weights():
    from flowhigh_b200.config import BackboneConfig, VocoderConfig
    from flowhigh_b200.weights import random_state_dict
    vcfg = VocoderConfig.assumed_48k()
    return vcfg, random_state_dict(BackboneConfig(), vcfg, seed=0, vocoder_gain=0.7)


class CpuReference:
    """The reference's CPU implementation of the path, one clip per step (its generate() is batch-1).
    kind "reference": the UNMODIFIED reference package (baseline/_ref, or /root/reference in the build container),
    imported through oracle/ref_harness.py (stubs for the four packages missing offline, `.cuda()` neutralised --
    the caller hides the GPU); kind "port": the oracle restatement, only when no reference tree is present."""

    def __init__(self):
        import torch
        from oracle import ref_harness
        self.vcfg, self.sd = cpu_weights()
        self.kind = "reference" if ref_harness.available() and not torch.cuda.is_available() else "port"
        if self.kind == "reference":
            self.model = ref_harness.build_reference_model(self.sd, self.vcfg, cfm_method="basic_cfm",
                                                           ode_method="midpoint", sigma=0.0)
        else:
            from oracle import pipeline
            self.model = pipeline.OracleFlowHigh(self.sd, self.vcfg, cfm_method="basic_cfm", ode_method="midpoint")

    def step(self, sample_seconds, seed):
        import torch
        from flowhigh_b200.synth import synth_speech
        wav = synth_speech(int(sample_seconds * SR_IN), SR_IN, seed)
        t0 = time.perf_counter()
        if self.kind == "reference":
            with torch.no_grad():
                out = self.model.generate(wav, SR_IN, 48000, timestep=STEPS_ODE)
        else:
            N = int(sample_seconds * 48000) // 480
            eps = torch.from_numpy(np.random.default_rng(seed).standard_normal((1, N, 256)).astype(np.float32))
            out = self.model.generate(wav, SR_IN, eps, timestep=STEPS_ODE)
        dt = time.perf_counter() - t0
        assert out.shape[-1] == int(sample_seconds * 48000) and bool(torch.isfinite(out).all())
        return dt


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation on the box's host cores, all threads, one 10 s clip of
    the configs[1] workload per step (BASELINE.md section 3).  The run is bounded to a few minutes: when K + W steps of
    the measured step time would not fit, fewer steps are executed and the line says so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["CUDA_VISIBLE_DEVICES"] = ""  # the reference hard-codes .cuda() (SURVEY F7): this arm is its CPU path
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = CpuReference()
    sample = float(args.ref_clip_seconds)
    budget = float(args.ref_budget_seconds)
    t_first = ref.step(sample, 0)  # warm-up 1 (also sizes the run)
    n_warm = 1
    steps = args.steps
    if t_first * (args.steps + args.warmup) > budget:
        steps = max(3, min(args.steps, int(budget / t_first) - 1))
    else:
        for i in range(1, args.warmup):
            ref.step(sample, i)
            n_warm += 1
    t = [ref.step(sample, 100 + i) for i in range(steps)]
    total = sum(t)
    value = sample * steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": n_warm, "requested": {"steps": args.steps, "warmup": args.warmup},
        "ms_per_step": 1000 * total / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args.gpus, BATCH),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": ref.kind,
                         "sample": f"1 clip x {sample:g} s per step ({'unmodified reference package, generate()' if ref.kind == 'reference' else 'oracle port'}; "
                                   f"the reference generate() is batch-1), median step {1000 * statistics.median(t):.0f} ms"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(clip_seconds=10.0, steps=2, timeout=600):
    """cpu_baseline leg of the GPU arm: the reference arm in a child process with the GPU hidden (the reference would
    otherwise run on CUDA), bounded to ~10-30 s of CPU work."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", "1",
           "--ref-clip-seconds", str(clip_seconds), "--ref-budget-seconds", "60"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return {"error": (r.stderr or r.stdout)[-300:]}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


# ------------------------------------------------------------------------------------------- sharded workloads
def run_sharded_workload(args, model, eng, dev, world, rank, local):
    """BASELINE configs[2] (`mixed512`) and configs[3] (`longform`): ONE job partitioned over the ranks (strong scaling),
    through the public API from host buffers, the output gather (one ncclAllGather) and the D2H read inside the timed
    region; time = max over ranks.  `value` = audio-seconds of the whole job per wall second."""
    import torch
    import torch.distributed as dist
    from flowhigh_b200.synth import synth_speech

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    W = max(args.warmup, 3)
    if args.workload == "mixed512":
        rates = [8000, 12000, 16000, 24000]
        base = {sr: [synth_speech(int(CLIP_SECONDS * sr), sr, seed=sr + i) for i in range(4)] for sr in rates}
        srs = [rates[i % 4] for i in range(args.clips)]
        audios = [base[srs[i]][(i // 4) % 4] for i in range(args.clips)]
        N = int(CLIP_SECONDS * 48000) // 480
        gen = torch.Generator(dev).manual_seed(99)
        eps_all = torch.randn((args.clips, N, 256), device=dev, generator=gen)  # same on every rank
        eps = [eps_all[i] for i in range(args.clips)]
        out_host = torch.empty((args.clips, int(CLIP_SECONDS * 48000)), dtype=torch.float32).pin_memory() if rank == 0 else None
        audio_s = args.clips * CLIP_SECONDS

        def step():
            out = model.generate_sharded(audios, srs, 48000, timestep=STEPS_ODE, eps=eps, gather=True)
            if rank == 0:
                out_host.copy_(out, non_blocking=True)
            torch.cuda.synchronize(dev)
            return out
        h2d = sum(a.size * 4 for a in audios)
        d2h = args.clips * int(CLIP_SECONDS * 48000) * 4
        wl = (f"configs[2]: {args.clips} x 10 s clips, 8/12/16/24 kHz mixed -> 48 kHz, sharded over {world} GPU(s) by assign_clips, "
              "batches of <= 64 per rate group, outputs gathered with one all_gather_into_tensor (NCCL); basic_cfm, midpoint (2 NFE)")
    else:
        sr_in = 16000
        ten = synth_speech(10 * sr_in, sr_in, seed=3)
        reps = int(round(args.minutes * 6))
        clip = np.concatenate([ten * (0.6 + 0.4 * np.cos(0.37 * k)) for k in range(reps)]).astype(np.float32)
        T = clip.shape[0] * 3
        clen, ov = 480000, 24000
        K = -(-(T - clen) // (clen - ov)) + 1
        eps_all = torch.randn((K, clen // 480, 256), device=dev, generator=torch.Generator(dev).manual_seed(7))
        out_host = torch.empty((1, T), dtype=torch.float32).pin_memory() if rank == 0 else None
        audio_s = T / 48000.0

        def step():
            out = model.generate_long(clip, sr_in, 48000, timestep=STEPS_ODE, chunk_seconds=10.0, overlap_seconds=0.5, eps=eps_all)
            if rank == 0:
                out_host.copy_(out, non_blocking=True)
            torch.cuda.synchronize(dev)
            return out
        h2d, d2h = clip.size * 4, T * 4
        wl = (f"configs[3]: one {args.minutes:g}-minute clip 16 kHz -> 48 kHz, {K} overlapped 10 s chunks (0.5 s overlap) in contiguous "
              f"blocks over {world} GPU(s), one all_gather_into_tensor of the chunk waveforms, overlap-add + global post-processing; "
              "basic_cfm, midpoint (2 NFE)")
    for _ in range(W):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ts = []
    for _ in range(args.steps):
        barrier()
        t0 = time.perf_counter()
        out = step()
        barrier()
        ts.append(time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor(ts, device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ts = [float(v) for v in t]
    finite = bool(torch.isfinite(out).all())
    if not finite:
        raise RuntimeError("bench: non-finite output")
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, "audio", out)
    if rank == 0:
        total = sum(ts)
        med = statistics.median(ts)
        line = {"metric": METRIC, "value": audio_s * args.steps / total, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": W, "ms_per_step": 1000 * total / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
                "config": {"workload": wl, "audio_seconds_per_step": audio_s, "sr_out": 48000, "nfe": 2,
                           "parallelism": f"one job partitioned over {world} GPU(s); one NCCL all-gather of the outputs",
                           "l2_policy": "per-step working set far exceeds the 126 MB L2; no flush needed"},
                "e2e": {"value": audio_s * args.steps / total, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(d2h), "note": "the whole timed region IS the end-to-end path (host buffers in, "
                        "gathered result read back on rank 0); max over ranks, wall clock around barriers"},
                "latency_ms": {"p50": 1000 * med, "min": 1000 * min(ts), "max": 1000 * max(ts)},
                "clocks": clocks, "self_check": {"finite": finite, "out_shape": list(out.shape)}}
        print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "fp16x2"],
                    help="16-bit tensor-core operand format (same rate and bytes; fp16 meets the LSD bar, see DESIGN.md)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-clip-seconds", type=float, default=CLIP_SECONDS, help="reference arm: clip length per step")
    ap.add_argument("--ref-budget-seconds", type=float, default=240.0, help="reference arm: bound on the whole run")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-accurate", action="store_true", help="skip the fp16x2 (tolerance-on-every-fixture) leg")
    ap.add_argument("--latency-samples", type=int, default=200)
    ap.add_argument("--breakdown", default=None, help="write the per-kernel CUDA-event breakdown to this JSON file")
    ap.add_argument("--workload", default="batch64", choices=["batch64", "mixed512", "longform"],
                    help="batch64 = BASELINE configs[1] (the metric's configuration, default); mixed512 = configs[2]: 512 x 10 s "
                         "clips, 8/12/16/24 kHz mixed, SHARDED over the ranks (strong scaling, outputs gathered with one "
                         "ncclAllGather); longform = configs[3]: one 10-minute clip, overlapped chunks over the ranks + overlap-add")
    ap.add_argument("--clips", type=int, default=512, help="mixed512: total number of clips")
    ap.add_argument("--minutes", type=float, default=10.0, help="longform: clip length")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/audio.npy (float32, a fixed seeded sample above "
                         f"{DUMP_BYTES >> 20} MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs applies to the GPU implementation")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from flowhigh_b200 import FlowHighSR, VocoderConfig, _lib
    from flowhigh_b200.synth import synth_speech

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL prints its version banner on fd 1 when the communicator is created: keep stdout to the ONE JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    dev = torch.device(f"cuda:{local}")
    W = max(args.warmup, 3)
    B = args.batch

    model = FlowHighSR.from_random(VocoderConfig.assumed_48k(), device=dev, seed=0, precision=args.precision)
    eng = model._engine()
    if args.workload != "batch64":
        run_sharded_workload(args, model, eng, dev, world, rank, local)
        if world > 1:
            dist.destroy_process_group()
        return
    n_in = int(CLIP_SECONDS * SR_IN)
    host = np.stack([synth_speech(n_in, SR_IN, seed=rank * B + i) for i in range(min(B, 8))])
    host = np.concatenate([host] * (-(-B // host.shape[0])))[:B]  # 8 distinct clips tiled (synthesis is slow)
    host_t = torch.from_numpy(np.ascontiguousarray(host)).pin_memory()
    x_dev = host_t.to(dev)
    T = 48000 * int(CLIP_SECONDS)
    N = T // 480
    eps = torch.randn((B, N, 256), device=dev, generator=torch.Generator(dev).manual_seed(1234 + rank))

    def step_resident():
        eng.new_call()
        eng.status_begin()  # overflow / NaN guard of the 16-bit path: reset here, read once after the timed loop
        cond = eng.resample_normalise(x_dev, SR_IN)
        cond_mel = eng.encode(cond)
        mel = eng.sample_mel(cond_mel, eps, steps=STEPS_ODE, ode_method="midpoint", cfm_method="basic_cfm", sigma=0.0)
        wave = eng.vocoder(mel)
        out = eng.postprocess(wave, cond)
        eng.status_end()
        return out

    out_host = torch.empty((B, T), dtype=torch.float32).pin_memory()

    def step_e2e():
        # host clips in, host results out, through the public call: uploads from a page-locked staging buffer, results
        # copied into the caller's page-locked buffer on a side stream (generate_batch docstring)
        model.generate_batch(list(host_t), SR_IN, 48000, timestep=STEPS_ODE, eps=list(eps), pinned=True, out_host=out_host)
        torch.cuda.synchronize(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(W):
        step_resident()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        out = step_resident()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - n0
    clocks = sampler.stop() if rank == 0 else None

    # ---- the timed output is checked, not just produced: finite, guard clean, and clip 0 of the batch against its own
    #      B = 1 run through the public API (different tile shapes, parallel AMP branches, CUDA-graph-free)
    status = eng.status_read()
    finite = bool(torch.isfinite(out).all())
    if not finite or status:
        raise RuntimeError(f"bench: the timed step produced a non-finite output (finite={finite}) or tripped the 16-bit "
                           f"overflow guard (status {status:#x})")
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, "audio", out)
    self_check = None
    if rank == 0:
        model.cuda_graphs = False
        single = model.generate(host[0], SR_IN, 48000, timestep=STEPS_ODE, eps=eps[0:1])[0].double()
        model.cuda_graphs = True
        b0 = out[0].double()
        snr = float(10 * torch.log10((single ** 2).sum() / ((single - b0) ** 2).sum().clamp_min(1e-300)))
        self_check = {"finite": finite, "overflow_status": status, "clip0_snr_vs_b1_generate_db": round(snr, 1),
                      "out_absmax": float(out.abs().max())}
        if snr < 50.0:
            raise RuntimeError(f"bench: clip 0 of the timed batch differs from its own B=1 generate(): SNR {snr:.1f} dB")

    # ---- e2e through the public API with host buffers
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0

    if world > 1:
        t = torch.tensor([ms, e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(t[0]), float(t[1])

    # ---- latency leg (BASELINE metric, second half): p50 of one 10 s clip and of 1 s streaming chunks, B = 1,
    #      through the public generate() call from a host array to a synchronised device result
    latency = None
    if rank == 0 and not args.no_latency:
        def p50_p99(fn, n):
            ts = []
            for _ in range(n):
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize(dev)
                ts.append(1000 * (time.perf_counter() - t0))
            raw = list(ts)
            ts.sort()
            p50 = ts[len(ts) // 2]
            slow = [i for i, v in enumerate(raw) if v > 2 * p50]
            return p50, ts[min(len(ts) - 1, int(0.99 * len(ts)))], {"n": n, "max_ms": ts[-1], "p90_ms": ts[int(0.9 * n)],
                                                                    "samples_over_2x_p50": len(slow), "their_index": slow[:8]}
        NL = args.latency_samples
        clip = host[0]
        for _ in range(5):
            model.generate(clip, SR_IN, 48000, timestep=STEPS_ODE)
        l50, l99, ltail = p50_p99(lambda: model.generate(clip, SR_IN, 48000, timestep=STEPS_ODE), NL)
        # config 5: basic_cfm, euler, time_step 4, 1 s chunks at 16 kHz
        m5 = FlowHighSR.from_random(VocoderConfig.assumed_48k(), device=dev, seed=0, precision=args.precision,
                                    torchdiffeq_ode_method="euler")
        chunk = synth_speech(16000, 16000, seed=7)
        for _ in range(5):
            m5.generate(chunk, 16000, 48000, timestep=4)
        c50, c99, ctail = p50_p99(lambda: m5.generate(chunk, 16000, 48000, timestep=4), NL)
        latency = {"clip_10s_midpoint_p50_ms": l50, "clip_10s_midpoint_p99_ms": l99,
                   "chunk_1s_euler4_p50_ms": c50, "chunk_1s_euler4_p99_ms": c99,
                   "samples": NL, "clip_10s_tail": ltail, "chunk_1s_tail": ctail,
                   "note": "B=1, host numpy in -> device tensor out, stream-synchronised (overflow-guard read included), "
                           "CUDA-graph replay of the whole pipeline"}
        del m5

    # ---- roofline leg: per-kernel CUDA-event timing of one more step (rank 0)
    breakdown = None
    if rank == 0:
        eng.start_profile()
        step_resident()
        breakdown = eng.stop_profile()
    audio_s = B * CLIP_SECONDS * world
    value = audio_s * args.steps / (ms / 1000.0)
    e2e_value = audio_s * e2e_steps / e2e_s

    if rank == 0:
        hbm_peak, tf_peak, peak_src = peaks()
        tc = {k: v for k, v in breakdown.items() if k.startswith("tc_conv")}
        tc_ms = sum(v["ms"] for v in tc.values())
        tc_fl = sum(v["flops"] for v in tc.values())
        tc_n = sum(v["launches"] for v in tc.values())
        tot_ms = sum(v["ms"] for v in breakdown.values())
        achieved = tc_fl / (tc_ms / 1000.0) / 1e12 if tc_ms > 0 else 0.0
        traffic = None  # DRAM bytes per launch from the committed ncu capture of this same workload (B = 64)
        tpath = os.path.join(ROOT, "profiles", "r2_dram_traffic_b64.json")  # the final build's capture (tools/evidence_r2.sh)
        if not os.path.exists(tpath):
            tpath = os.path.join(ROOT, "profiles", "r1_dram_traffic_b64.json")
        if B == BATCH and os.path.exists(tpath):
            tj = json.load(open(tpath))["tc_conv"]
            traffic = (tj["dram_read_bytes"] + tj["dram_write_bytes"]) / tj["launches"]
        tc_by = sum(v["bytes"] for v in tc.values())
        roofline = {"kernel": "tc_conv_kernel<8|12|16> + tc_conv2_kernel (tcgen05 implicit-GEMM conv, all launches of one step)", "bound": "tensor",
                    "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
                    "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram__bytes_read+write, B=64 capture)",
                    "algorithmic_bytes_per_launch": tc_by / max(tc_n, 1),
                    "peak_source": peak_src, "launches_per_step": tc_n,
                    "avg_launch_ms": tc_ms / max(tc_n, 1), "share_of_step": tc_ms / tot_ms if tot_ms else None,
                    "algorithmic_flops_per_step": tc_fl}
        # second roofline: the HBM / FP32-issue-bound anti-aliased snake (all launches of one step)
        sn = breakdown.get("fh_snake_aa_chunked")
        roofline_snake = None
        if sn and sn["ms"] > 0:
            gbs = sn["bytes"] / (sn["ms"] / 1000.0) / 1e9
            straffic = None
            if B == BATCH and os.path.exists(tpath) and "snake" in json.load(open(tpath)):
                tj = json.load(open(tpath))["snake"]
                straffic = (tj["dram_read_bytes"] + tj["dram_write_bytes"]) / tj["launches"]
            roofline_snake = {"kernel": "snake_aa_mma_kernel (fused up2x -> Snake -> down2x, both FIR filters as Toeplitz MMAs)", "bound": "hbm",
                              "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "traffic": straffic,
                              "algorithmic_bytes_per_launch": sn["bytes"] / sn["launches"], "launches_per_step": sn["launches"],
                              "avg_launch_ms": sn["ms"] / sn["launches"], "share_of_step": sn["ms"] / tot_ms if tot_ms else None,
                              "note": "fp32 rows in (fp16 rows behind the first conv of an AMP unit), fp16 rows out; ncu: profiles/r2_ncu_snake.txt"}
        # every other kernel class of the path: HBM roofline from its algorithmic bytes (attention: tensor roofline)
        roofline_stages = {}
        for k, v in breakdown.items():
            if k.startswith("tc_conv") or k == "fh_snake_aa_chunked" or v["ms"] <= 0:
                continue
            if k == "fh_attention_tc" and v["flops"] > 0:
                tf = v["flops"] / (v["ms"] / 1000.0) / 1e12
                roofline_stages[k] = {"bound": "tensor", "achieved": tf, "peak": tf_peak, "unit": "TFLOP/s", "frac": tf / tf_peak,
                                      "ms": v["ms"], "launches": v["launches"],
                                      "note": "attention_tc5_kernel (tcgen05 / TMEM; FH_ATTN_TC5=0: the mma.sync kernel) with the hi/lo operand split (q k^T executed 3 x): algorithmic 4 N^2 Dh per head"}
            elif v["bytes"] > 0:
                gbs = v["bytes"] / (v["ms"] / 1000.0) / 1e9
                roofline_stages[k] = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                                      "ms": v["ms"], "launches": v["launches"]}
        groups = {}
        for k, v in breakdown.items():
            gname = "tc_conv" if k.startswith("tc_conv") else k
            g = groups.setdefault(gname, {"ms": 0.0, "launches": 0})
            g["ms"] += v["ms"]
            g["launches"] += v["launches"]
        if args.breakdown:
            os.makedirs(os.path.dirname(os.path.abspath(args.breakdown)), exist_ok=True)
            json.dump({"per_kernel": breakdown, "groups": groups, "step_ms_profiled": tot_ms}, open(args.breakdown, "w"),
                      indent=1)
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu = cpu_baseline_subprocess()
        # ---- the same step in the mode that meets the LSD <= 0.05 dB bar on EVERY fixture (hi + lo activation operands):
        #      reported beside the headline, never instead of it (tests: test_big_config_16bit_golden)
        accurate = None
        if world == 1 and args.precision == "fp16" and not args.no_accurate and B == BATCH:
            del model, eng, step_resident, step_e2e
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            m2 = FlowHighSR.from_random(VocoderConfig.assumed_48k(), device=dev, seed=0, precision="fp16x2")
            e2 = m2._engine()

            def step_x2():
                e2.new_call()
                e2.status_begin()
                cond = e2.resample_normalise(x_dev, SR_IN)
                mel = e2.sample_mel(e2.encode(cond), eps, steps=STEPS_ODE, ode_method="midpoint", cfm_method="basic_cfm", sigma=0.0)
                o = e2.postprocess(e2.vocoder(mel), cond)
                e2.status_end()
                return o
            for _ in range(3):
                step_x2()
            torch.cuda.synchronize(dev)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(3):
                o2 = step_x2()
            a1.record()
            torch.cuda.synchronize(dev)
            ams = a0.elapsed_time(a1) / 3
            accurate = {"precision": "fp16x2", "ms_per_step": ams, "value": B * CLIP_SECONDS / (ams / 1000.0), "unit": UNIT,
                        "finite": bool(torch.isfinite(o2).all()), "overflow_status": e2.status_read(),
                        "note": "hi + lo fp16 activation operands against duplicated weights (2 x the vocoder MMAs): "
                                "LSD 0.016-0.028 dB on every golden fixture; the default fp16 path meets 0.05 dB on this "
                                "workload's own clip (0.019) and reaches 0.08 dB only on the high-dynamic-range configs[0] clip"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic", "config": config_dict(world, B),
            "per_gpu": value / world, "realtime_factor_per_gpu": value / world,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(host_t.numel() * 4),
                    "d2h_bytes_per_step": int(out_host.numel() * 4), "steps": e2e_steps},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "roofline_snake": roofline_snake,
            "roofline_stages": roofline_stages, "cpu_baseline": cpu,
            "latency": latency, "self_check": self_check, "accurate_mode": accurate,
            "stage_ms": {k: round(v["ms"], 3) for k, v in sorted(groups.items(), key=lambda kv: -kv[1]["ms"])},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
