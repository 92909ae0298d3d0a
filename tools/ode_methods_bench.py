"""Cost of the torchdiffeq ODE methods: `generate_batch` of 8 x 10 s clips (12 -> 48 kHz, fp16, timestep 1) with euler,
midpoint, rk4 and dopri5 at tol 1e-3 and 1e-5, after warm-up.  Prints one JSON line: ms per call (median of --reps),
field evaluations (NFE) per clip, the card's name and power limit.  Fixed-grid groups of <= 8 clips replay a CUDA graph;
dopri5 runs its host-driven loop clip by clip.

    python tools/ode_methods_bench.py [--reps 5] [--out ode_methods.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flowhigh_b200 import FlowHighSR, VocoderConfig  # noqa: E402
from flowhigh_b200.synth import synth_speech  # noqa: E402

CASES = [("euler", None), ("midpoint", None), ("rk4", None), ("dopri5", 1e-3), ("dopri5", 1e-5)]
NFE_FIXED = {"euler": 1, "midpoint": 2, "rk4": 4}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in q.split(",")]
        return name, limit
    except Exception:  # noqa: BLE001
        return torch.cuda.get_device_name(0), None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--clips", type=int, default=8)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    sr = 12000
    clips = [synth_speech(int(args.seconds * sr), sr, seed=i) for i in range(args.clips)]
    n_frames = int(args.seconds * 48000) // 480
    gen = torch.Generator().manual_seed(0)
    eps = [torch.randn((1, n_frames, 256), generator=gen) for _ in clips]
    rows = []
    for method, tol in CASES:
        kw = {} if tol is None else dict(ode_atol=tol, ode_rtol=tol)
        m = FlowHighSR.from_random(VocoderConfig.assumed_48k(), device="cuda:0", seed=0, precision="fp16",
                                   torchdiffeq_ode_method=method, **kw)
        for _ in range(3):  # first sighting, graph capture, replay
            m.generate_batch(clips, sr, eps=eps)
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            m.generate_batch(clips, sr, eps=eps)
            torch.cuda.synchronize()
            ms.append((time.perf_counter() - t0) * 1e3)
        stats = m._engine().ode_stats if method == "dopri5" else None
        nfe = [s["n_f_evals"] for s in stats] if stats else [NFE_FIXED[method]] * len(clips)
        rows.append({"method": method, "tol": tol, "ms_per_call": float(np.median(ms)), "ms_all": [round(x, 2) for x in ms],
                     "nfe_per_clip": nfe, "graphed": len(m._graphs) > 0})
        print(f"{method:9s} tol {tol}: {np.median(ms):9.2f} ms per call, NFE per clip {nfe}", flush=True)
        del m
        torch.cuda.empty_cache()
    name, limit = card()
    res = {"workload": f"generate_batch {args.clips} x {args.seconds:g} s, 12 -> 48 kHz, fp16, timestep 1",
           "card": name, "power_limit": limit, "rows": rows}
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
