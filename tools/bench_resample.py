"""Output-rate conversion on the bench workload (DESIGN.md 3.4): one JSON line.

  resident   the resident-plan step of the bench workload (4096 utterances, ~200 characters, speed 1.0) at 22050,
             16000, 8000 and 48000 Hz, the rates alternated round by round in one process (CUDA events), and the
             resample kernel's own time per step (torch.profiler, CUDA activity)
  e2e        text -> pinned host PCM through ctts_b200_synth_texts at the same rates: seconds, bytes, GB/s

The device name and power limit are read in the same run.  Usage:
  python tools/bench_resample.py [--utts 4096] [--rounds 3] [--steps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

RATES = (22050, 16000, 8000, 48000)


def power_limit_w(index: int) -> float | None:
    try:
        r = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=20)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:
        return None


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import harness as H
    pkg = importlib.import_module("2026-simple-c-tts_b200")
    gpu = importlib.import_module("2026-simple-c-tts_b200.gpu")
    pipe = importlib.import_module("2026-simple-c-tts_b200.pipeline")

    dev = 0
    torch.cuda.set_device(dev)
    db = H.synthetic_db()
    fr = pkg.front.Front(db, H.shipped_config(), H.NORM_CSV)
    prm = fr.params()
    texts = pkg.corpus.batch(args.utts, seed=1234, target_chars=200)
    plan = fr.plan(texts)
    g = gpu.GpuSynth(db, dev)
    stream = torch.cuda.Stream(device=dev)
    g.set_stream(stream.cuda_stream)

    plans, outs = {}, {}
    for hz in RATES:
        g.set_output_rate(hz)
        plans[hz] = g.create_plan(plan, prm)
        outs[hz] = torch.empty(max(plans[hz].out_samples, 8), dtype=torch.int16, device=f"cuda:{dev}")
    native_cnt = None
    counts = {}
    for hz in RATES:
        plans[hz].run(outs[hz].data_ptr())
        counts[hz] = plans[hz].counts().astype(np.int64)
        if hz == 22050:
            native_cnt = counts[hz]
    for hz in RATES:   # the counts follow ceil(n L / M) of the native run
        L, M = {22050: (1, 1), 16000: (320, 441), 8000: (160, 441), 48000: (320, 147)}[hz]
        assert np.array_equal(counts[hz], -(-native_cnt * L // M)), hz

    step_ms = {hz: [] for hz in RATES}
    with torch.cuda.stream(stream):
        for _ in range(args.rounds):
            for hz in RATES:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                plans[hz].run(outs[hz].data_ptr())
                a.record(stream)
                for _ in range(args.steps):
                    plans[hz].run(outs[hz].data_ptr())
                b.record(stream)
                b.synchronize()
                step_ms[hz].append(a.elapsed_time(b) / args.steps)

    # the resample kernel's own time, from the profiler's CUDA activity
    kernel_ms = {}
    from torch.profiler import ProfilerActivity, profile
    for hz in RATES[1:]:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                plans[hz].run(outs[hz].data_ptr())
            torch.cuda.synchronize(dev)
        tot = 0.0
        for e in prof.events():
            if "resample_kernel" in e.name:
                tot += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        kernel_ms[hz] = tot / 1e3 / args.steps

    # text -> host PCM at every rate
    tb = pipe.TextBatch(texts)
    e2e = {}
    for hz in RATES:
        g.set_output_rate(hz)
        cap = pipe.capacity_hint(fr, tb, hz)
        host = torch.empty(cap, dtype=torch.int16, pin_memory=True).numpy()
        pipe.synth_texts(fr, g, tb, host)   # warm-up
        torch.cuda.synchronize(dev)
        t = time.perf_counter()
        for _ in range(args.e2e_steps):
            _, cnt, used, _ = pipe.synth_texts(fr, g, tb, host)
        s = (time.perf_counter() - t) / args.e2e_steps
        assert np.array_equal(cnt.astype(np.int64), counts[hz]), hz
        e2e[hz] = {"ms": round(1e3 * s, 2), "bytes": 2 * used, "GB_per_s": round(2 * used / s / 1e9, 2),
                   "audio_s_per_s": round(float(cnt.sum()) / hz / s, 1)}

    line = {
        "tool": "tools/bench_resample.py",
        "device": torch.cuda.get_device_name(dev),
        "power_limit_w": power_limit_w(dev),
        "utterances": args.utts,
        "workload": "corpus.batch(n, seed=1234, target_chars=200), speed 1.0 (bench.py's default workload)",
        "resident_step_ms": {str(hz): {"median": round(float(np.median(v)), 3), "all": [round(x, 3) for x in v]}
                             for hz, v in step_ms.items()},
        "resample_kernel_ms_per_step": {str(hz): round(v, 3) for hz, v in kernel_ms.items()},
        "output_samples": {str(hz): int(counts[hz].sum()) for hz in RATES},
        "e2e_synth_texts": {str(hz): v for hz, v in e2e.items()},
        "rounds": args.rounds, "steps": args.steps, "e2e_steps": args.e2e_steps,
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    for p in plans.values():
        p.close()
    g.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
