"""G.711 output on the bench workload (DESIGN.md 3.7): one JSON line.

  e2e       text -> pinned host PCM (ctts_b200_synth_texts), μ-law and A-law (ctts_b200_synth_texts_g711), alternated
            round by round in one process, at 8 000 and 22 050 Hz, for the bench workload (4096 sentences of ~200
            characters, speed 1.0, BASELINE configs[2]): milliseconds (medians), bytes over PCIe, GB/s
  kernels   g711_pack_kernel against pack_copy_kernel (and the resampler beside them) per batch, from torch.profiler
            with CUDA activity, in a separate run

The device name and power limit are read in the same run.  Usage:
  python tools/bench_g711.py [--utts 4096] [--rounds 3] [--out FILE]
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

RATES = (8000, 22050)
KERNELS = ("g711_pack_kernel", "pack_copy_kernel", "pack_scan_kernel", "resample_kernel", "assemble_kernel")


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
    tb = pipe.TextBatch(pkg.corpus.batch(args.utts, seed=1234, target_chars=200))
    g = gpu.GpuSynth(db, dev)
    laws = {"ulaw": gpu.G711_ULAW, "alaw": gpu.G711_ALAW}

    result = {}
    for hz in RATES:
        g.set_output_rate(hz)
        # warm-up of every path into a pageable buffer of the capacity hint (untouched pages cost nothing); the timed
        # runs go to page-locked buffers of exactly the space they take (the output is deterministic)
        cap = pipe.capacity_hint(fr, tb, hz)
        _, _, pneed, _ = pipe.synth_texts(fr, g, tb, np.zeros(cap, np.int16))
        pcm = torch.empty(pneed, dtype=torch.int16, pin_memory=True).numpy()
        codes = torch.empty(pneed, dtype=torch.uint8, pin_memory=True).numpy()
        for law in laws.values():
            pipe.synth_texts_g711(fr, g, tb, law, np.zeros(cap, np.uint8))
        pipe.synth_texts(fr, g, tb, pcm)
        for law in laws.values():
            pipe.synth_texts_g711(fr, g, tb, law, codes)
        times = {"pcm": [], "ulaw": [], "alaw": []}
        used = {}
        for _ in range(args.rounds):
            t = time.perf_counter()
            _, pcnt, pused, _ = pipe.synth_texts(fr, g, tb, pcm)
            times["pcm"].append(time.perf_counter() - t)
            used["pcm"] = 2 * pused
            for name, law in laws.items():
                t = time.perf_counter()
                _, cnt, gused, _ = pipe.synth_texts_g711(fr, g, tb, law, codes)
                times[name].append(time.perf_counter() - t)
                assert np.array_equal(cnt, pcnt) and gused == pused, (hz, name)
                used[name] = gused
        entry = {"samples": int(pcnt.astype(np.int64).sum())}
        for kind in times:
            s = float(np.median(times[kind]))
            entry[kind] = {"ms_median": round(1e3 * s, 2), "ms_all": [round(1e3 * x, 2) for x in times[kind]],
                           "bytes_over_pcie": used[kind], "GB_per_s": round(used[kind] / s / 1e9, 2)}
        result[str(hz)] = entry

    # device time per batch of the packing kernels (and the resampler), profiler on, in a run of its own
    kernels = {}
    for hz in RATES:
        g.set_output_rate(hz)
        cap = pipe.capacity_hint(fr, tb, hz)
        for kind in ("pcm", "ulaw"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                if kind == "pcm":
                    pipe.synth_texts(fr, g, tb, np.zeros(cap, np.int16))
                else:
                    pipe.synth_texts_g711(fr, g, tb, laws[kind], np.zeros(cap, np.uint8))
                torch.cuda.synchronize(dev)
            tot = {k: 0.0 for k in KERNELS}
            for e in prof.events():
                for k in tot:
                    if k in e.name:
                        tot[k] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            kernels[f"{kind}_{hz}"] = {k: round(v / 1e3, 3) for k, v in tot.items() if v}

    line = {
        "tool": "tools/bench_g711.py",
        "device": torch.cuda.get_device_name(dev),
        "power_limit_w": power_limit_w(dev),
        "utterances": args.utts,
        "workload": "corpus.batch(n, seed=1234, target_chars=200), speed 1.0 (BASELINE configs[2], bench.py's default)",
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
