"""Loudness normalization on the bench workload (DESIGN.md 3.6): one JSON line.

  resident   the resident-plan step of the bench workload (4096 utterances, ~200 characters, speed 1.0) at 22050 and
             16000 Hz with the stage off, at -16 LUFS with a -1 dBFS sample-peak ceiling and at -16 LUFS with a
             -1 dBTP true-peak ceiling, the three alternated round by round in one process (CUDA events), medians
  kernels    the loudness kernels' own time per step, from torch.profiler (CUDA activity) in a run of its own
  e2e        text -> pinned host PCM (ctts_b200_synth_texts) and text -> pinned host FLAC (ctts_b200_synth_texts_flac),
             the three settings alternated round by round

The device name and power limit are read in the same run.  Usage:
  python tools/bench_loudness.py [--utts 4096] [--rounds 3] [--steps 5] [--out FILE]
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

RATES = (22050, 16000)
TARGETS = (0.0, -16.0, "tp")   # 0: off; "tp": -16 LUFS with a -1 dBTP true-peak ceiling
LABEL = {0.0: "off", -16.0: "minus16", "tp": "minus16_tp"}
KERNELS = ("ld_chunk_kernel", "ld_scan_kernel", "ld_true_peak_kernel", "ld_gain_kernel", "ld_apply_kernel")


def power_limit_w(index: int) -> float | None:
    try:
        r = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=20)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:
        return None


def _med(v):
    return {"median": round(float(np.median(v)), 3), "all": [round(x, 3) for x in v]}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
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

    def configure(hz, target):
        g.set_output_rate(hz)
        g.set_loudness(-16.0 if target == "tp" else target, -1.0, true_peak=target == "tp")

    plans, outs, launches = {}, {}, {}
    for hz in RATES:
        for t in TARGETS:
            configure(hz, t)
            plans[hz, t] = g.create_plan(plan, prm)
            outs[hz, t] = torch.empty(max(plans[hz, t].out_samples, 8), dtype=torch.int16, device=f"cuda:{dev}")
            launches[hz, t] = plans[hz, t].info().kernel_launches
    gains = {}
    for hz in RATES:
        for t in TARGETS:
            plans[hz, t].run(outs[hz, t].data_ptr())
            plans[hz, t].counts()
        lufs, gain = plans[hz, -16.0].loudness()
        gains[hz] = {"defined": int(np.isfinite(lufs).sum()), "unity": int((gain == 65536).sum()),
                     "lufs_median": round(float(np.median(lufs[np.isfinite(lufs)])), 2)}
        _, gain_tp = plans[hz, "tp"].loudness()
        peak = plans[hz, "tp"].true_peak()
        gains[hz]["true_peak_limited"] = int((gain_tp < gain).sum())
        # the stage-off output of the same batch: the sample peaks
        pk = np.array([np.abs(u.astype(np.int32)).max() if len(u) else 0 for u in plans[hz, 0.0].utterances()], np.float64)
        ok = pk > 0
        gains[hz]["true_peak_over_sample_peak_db_max"] = round(float(np.max(20 * np.log10(peak[ok] / pk[ok]))), 3)

    step_ms = {(hz, t): [] for hz in RATES for t in TARGETS}
    with torch.cuda.stream(stream):
        for _ in range(args.rounds):
            for hz in RATES:
                for t in TARGETS:
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    plans[hz, t].run(outs[hz, t].data_ptr())
                    a.record(stream)
                    for _ in range(args.steps):
                        plans[hz, t].run(outs[hz, t].data_ptr())
                    b.record(stream)
                    b.synchronize()
                    step_ms[hz, t].append(a.elapsed_time(b) / args.steps)

    kernel_ms = {}
    from torch.profiler import ProfilerActivity, profile
    for hz in RATES:
        for t in (-16.0, "tp"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    plans[hz, t].run(outs[hz, t].data_ptr())
                torch.cuda.synchronize(dev)
            tot = {k: 0.0 for k in KERNELS}
            for e in prof.events():
                for k in KERNELS:
                    if k in e.name:
                        tot[k] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            kernel_ms[f"{hz}_{LABEL[t]}"] = {k: round(v / 1e3 / args.steps, 3) for k, v in tot.items()}

    tb = pipe.TextBatch(texts)
    e2e = {}
    for hz in RATES:
        pcm = torch.empty(pipe.capacity_hint(fr, tb, hz), dtype=torch.int16, pin_memory=True).numpy()
        flac = torch.empty(pipe.capacity_hint_flac(fr, tb, hz), dtype=torch.uint8, pin_memory=True).numpy()
        for t in TARGETS:   # warm-up
            configure(hz, t)
            pipe.synth_texts(fr, g, tb, pcm)
            pipe.synth_texts_flac(fr, g, tb, flac)
        res = {(k, t): [] for k in ("pcm", "flac") for t in TARGETS}
        used = {}
        for _ in range(args.rounds):
            for t in TARGETS:
                configure(hz, t)
                torch.cuda.synchronize(dev)
                s = time.perf_counter()
                _, _, used["pcm", t], _ = pipe.synth_texts(fr, g, tb, pcm)
                res["pcm", t].append(1e3 * (time.perf_counter() - s))
                s = time.perf_counter()
                _, _, _, used["flac", t], _ = pipe.synth_texts_flac(fr, g, tb, flac)
                res["flac", t].append(1e3 * (time.perf_counter() - s))
        e2e[hz] = {f"{k}_{LABEL[t]}_ms": _med(v) for (k, t), v in res.items()}
        e2e[hz]["bytes"] = {f"{k}_{LABEL[t]}": int(v) * (2 if k == "pcm" else 1) for (k, t), v in used.items()}

    line = {
        "tool": "tools/bench_loudness.py",
        "device": torch.cuda.get_device_name(dev),
        "power_limit_w": power_limit_w(dev),
        "utterances": args.utts,
        "workload": "corpus.batch(n, seed=1234, target_chars=200), speed 1.0 (bench.py's default workload)",
        "setting_on": {"target_lufs": -16.0, "ceiling_dbfs": -1.0},
        "setting_tp": {"target_lufs": -16.0, "ceiling_dbtp": -1.0},
        "resident_step_ms": {f"{hz}_{LABEL[t]}": _med(v) for (hz, t), v in step_ms.items()},
        "kernel_launches": {f"{hz}_{LABEL[t]}": v for (hz, t), v in launches.items()},
        "loudness_kernels_ms_per_step": kernel_ms,
        "utterances_at_minus16": {str(hz): v for hz, v in gains.items()},
        "e2e": {str(hz): v for hz, v in e2e.items()},
        "rounds": args.rounds, "steps": args.steps,
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
