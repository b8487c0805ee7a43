"""FLAC output on the bench workloads (DESIGN.md 3.5): one JSON line.

  e2e       text -> pinned host PCM (ctts_b200_synth_texts) and text -> pinned host FLAC (ctts_b200_synth_texts_flac),
            alternated round by round in one process, at 22 050 and 16 000 Hz, for the bench workload (4096 sentences
            of ~200 characters, speed 1.0, BASELINE configs[2]) and configs[3] (the same texts at mixed speeds 0.5-2.0):
            seconds, bytes over PCIe, GB/s, the compression ratio
  kernels   each FLAC kernel's time per batch, from torch.profiler with CUDA activity, in a separate run

The device name and power limit are read in the same run.  Usage:
  python tools/bench_flac.py [--utts 4096] [--rounds 3] [--out FILE]
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
KERNELS = ("flac_analyze_kernel", "flac_scan_kernel", "flac_emit_kernel")


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
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    import harness as H
    pkg = importlib.import_module("2026-simple-c-tts_b200")
    gpu = importlib.import_module("2026-simple-c-tts_b200.gpu")
    pipe = importlib.import_module("2026-simple-c-tts_b200.pipeline")

    dev = 0
    torch.cuda.set_device(dev)
    db = H.synthetic_db()
    fr = pkg.front.Front(db, H.shipped_config(), H.NORM_CSV)
    texts = pkg.corpus.batch(args.utts, seed=1234, target_chars=200)
    workloads = {"speed1": pipe.TextBatch(texts), "mixed": pipe.TextBatch(texts, pkg.corpus.mixed_speeds(args.utts, seed=99))}
    g = gpu.GpuSynth(db, dev)

    result = {}
    for hz in RATES:
        g.set_output_rate(hz)
        for wname, tb in workloads.items():
            # warm-up of both paths into pageable buffers of the capacity hints (untouched pages cost nothing); the
            # timed runs go to page-locked buffers of exactly the space they take (the output is deterministic)
            _, _, pneed, _ = pipe.synth_texts(fr, g, tb, np.zeros(pipe.capacity_hint(fr, tb, hz), np.int16))
            _, _, _, fneed, _ = pipe.synth_texts_flac(fr, g, tb, np.zeros(pipe.capacity_hint_flac(fr, tb, hz), np.uint8))
            pcm = torch.empty(pneed, dtype=torch.int16, pin_memory=True).numpy()
            flac = torch.empty(fneed, dtype=torch.uint8, pin_memory=True).numpy()
            pipe.synth_texts(fr, g, tb, pcm)
            pipe.synth_texts_flac(fr, g, tb, flac)
            times = {"pcm": [], "flac": []}
            for _ in range(args.rounds):
                t = time.perf_counter()
                _, pcnt, pused, _ = pipe.synth_texts(fr, g, tb, pcm)
                times["pcm"].append(time.perf_counter() - t)
                t = time.perf_counter()
                _, fbytes, fcnt, fused, _ = pipe.synth_texts_flac(fr, g, tb, flac)
                times["flac"].append(time.perf_counter() - t)
            assert np.array_equal(pcnt, fcnt), (hz, wname)
            pcm_bytes = 2 * int(pcnt.astype(np.int64).sum())
            flac_bytes = int(fbytes.astype(np.int64).sum())
            entry = {"compression_ratio": round(flac_bytes / pcm_bytes, 4), "pcm_sample_bytes": pcm_bytes,
                     "flac_file_bytes": flac_bytes}
            for kind, used in (("pcm", 2 * pused), ("flac", fused)):
                s = float(np.median(times[kind]))
                entry[kind] = {"ms_median": round(1e3 * s, 2), "ms_all": [round(1e3 * x, 2) for x in times[kind]],
                               "bytes_over_pcie": used, "GB_per_s": round(used / s / 1e9, 2)}
            result[f"{wname}_{hz}"] = entry

    # each FLAC kernel's device time per batch, profiler on, in a run of its own
    kernels = {}
    for hz in RATES:
        g.set_output_rate(hz)
        tb = workloads["speed1"]
        flac = np.zeros(pipe.capacity_hint_flac(fr, tb, hz), np.uint8)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            pipe.synth_texts_flac(fr, g, tb, flac)
            torch.cuda.synchronize(dev)
        tot = {k: 0.0 for k in KERNELS + ("pack_scan_kernel", "assemble_kernel")}
        for e in prof.events():
            for k in tot:
                if k in e.name:
                    tot[k] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        kernels[str(hz)] = {k: round(v / 1e3, 3) for k, v in tot.items()}

    line = {
        "tool": "tools/bench_flac.py",
        "device": torch.cuda.get_device_name(dev),
        "power_limit_w": power_limit_w(dev),
        "utterances": args.utts,
        "workloads": {"speed1": "corpus.batch(n, seed=1234, target_chars=200), speed 1.0 (BASELINE configs[2], bench.py's default)",
                      "mixed": "the same texts at corpus.mixed_speeds(n, seed=99), 0.5-2.0 (BASELINE configs[3])"},
        "e2e_text_to_host": result,
        "kernel_ms_per_batch": kernels,
        "rounds": args.rounds,
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    g.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
