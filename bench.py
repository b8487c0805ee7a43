#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 CTTS back end (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path
  python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/*.npy

One "step" is one pass of the audio-assembly hot path over one batch of
synthetic utterances (default: BASELINE.json configs[2], 4096 sentences of ~200
characters at speed 1.0 on the seeded synthetic voice).  Prints ONE JSON line.

value      audio-seconds synthesised per second, plan and voice resident in HBM,
           timed with CUDA events on the launching stream, max over ranks.
e2e        TEXT -> host PCM through ctts_b200_synth_texts (libctts_b200.so): the text front end's planner
           threads feeding a device session, host buffers, every copy inside the timed region.  This
           is what the reference arm times (texts as C strings in memory -> PCM in memory), so the two are
           like for like.  e2e.plan_to_pcm is the back end alone (ctts_gpu_synth_batch on a ready plan).
roofline   algorithmic bytes of the assembly kernel / its duration / measured HBM peak.
cpu_baseline  the unmodified reference (oracle/_ref/ctts_ref_bench, N processes) on a
           bounded sample of the same workload, rank 0 only.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SAMPLE_RATE = 22050
METRIC = "audio_seconds_per_second"
UNIT = "audio-s/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--utts", type=int, default=4096, help="utterances per GPU (weak scaling)")
    ap.add_argument("--workload", default="speed1", choices=["speed1", "mixed", "long"],
                    help="speed1 = BASELINE configs[2]; mixed = configs[3] (speeds 0.5-2.0, WSOLA); "
                         "long = configs[4] (paragraphs of ~30 s audio, speed 1.0; use --utts 8192 on 8 GPUs for 65536)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (BASELINE configs[3] sharded over the ranks)")
    ap.add_argument("--strong-utts", type=int, default=4096, help="utterances of the ONE batch the strong-scaling leg shards")
    ap.add_argument("--vocab", type=int, default=0,
                    help="draw the words from a Zipf vocabulary of this many types instead of the round-1 word list "
                         "(sensitivity of the word-region deduplication; the default line reports one such point itself)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload(args, rank: int):
    """Synthetic batch for one rank: texts, speeds."""
    pkg = importlib.import_module("2026-simple-c-tts_b200")
    vocab = pkg.corpus.Vocabulary(args.vocab) if args.vocab else None
    texts = pkg.corpus.batch(args.utts, seed=1234 + 7919 * rank, target_chars=215 if args.workload == "long" else 200, vocab=vocab)
    if args.workload == "mixed":
        speeds = pkg.corpus.mixed_speeds(args.utts, seed=99 + rank)
    else:
        speeds = np.ones(args.utts, dtype=np.float32)
    return texts, speeds


def workload_name(args) -> str:
    if args.vocab:
        return (f"NOT a BASELINE config: {args.utts} sentences (~200 chars) per GPU, words drawn from a Zipf vocabulary of "
                f"{args.vocab} types, workload {args.workload}")
    if args.workload == "mixed":
        return f"BASELINE configs[3]: {args.utts} synthetic sentences (~200 chars) per GPU at mixed speeds 0.5-2.0 (WSOLA)"
    if args.workload == "long":
        return f"BASELINE configs[4]: {args.utts} paragraph-length utterances (~30 s of audio each) per GPU at speed 1.0"
    return f"BASELINE configs[2]: {args.utts} synthetic Portuguese sentences (~200 chars) per GPU at speed 1.0"


def strong_scaling_leg(args, rank, local_rank, world, fr, g, prm, pkg, gpu, sync_all, dist, torch):
    """BASELINE configs[3]: ONE seeded batch at mixed speeds 0.5-2.0, sharded by utterance over the ranks
    (greedy LPT, sharding.py), every rank synthesising its shard, outputs gathered on the host in batch
    order through one shared buffer (hostgather.py).  No data-path collective.  Returns rank 0's report."""
    pipe = importlib.import_module("2026-simple-c-tts_b200.pipeline")
    hg, sh = pkg.hostgather, pkg.sharding
    n = args.strong_utts
    texts = pkg.corpus.batch(n, seed=1234, target_chars=200)          # the same batch on every rank
    speeds = pkg.corpus.mixed_speeds(n, seed=99)
    shards = sh.shard_indices(hg.text_costs(texts, speeds), world)
    mine = shards[rank]
    my_texts = [texts[i] for i in mine]
    my_speeds = speeds[mine]
    dev = f"cuda:{local_rank}"

    # ---- device-timed: the shard as a resident plan (plan and voice in HBM)
    plan = fr.plan(my_texts, my_speeds)
    rp = g.create_plan(plan, prm)
    d_out = torch.empty(max(rp.out_samples, 8), dtype=torch.int16, device=dev)
    for _ in range(max(args.warmup, 3)):
        rp.run(d_out.data_ptr())
    my_counts = rp.counts().astype(np.int64)
    steps = max(3, min(args.steps, 10))
    sync_all()
    stream = torch.cuda.Stream(device=local_rank)   # the context launches on this stream; the events go on it too
    g.set_stream(stream.cuda_stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        e0.record(stream)
        for _ in range(steps):
            rp.run(d_out.data_ptr())
        e1.record(stream)
    sync_all()
    dev_ms = e0.elapsed_time(e1) / steps
    ws = rp.wsola_stats()
    del rp, d_out

    # ---- e2e: texts -> the shared host buffer (text front end + device + copies inside the timed region)
    tb = pipe.TextBatch(my_texts, my_speeds)
    scratch = torch.empty(int(g.layout(plan)[-1]) + 4096, dtype=torch.int16).pin_memory()
    _, _, used, _ = pipe.synth_texts(fr, g, tb, scratch.numpy())       # warm-up; learns the slot space of my shard
    del scratch
    t = torch.tensor([used], dtype=torch.int64, device=dev)
    if world > 1:
        all_used = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(all_used, t)
        all_used = [int(x) for x in all_used]
    else:
        all_used = [int(used)]
    bases = hg.region_bases(all_used)
    name = f"ctts_b200_bench_{os.environ.get('MASTER_PORT', '0')}_{n}"
    if rank == 0:
        shared = hg.SharedBatch(name, n, int(bases[-1]), create=True)
    sync_all()
    if rank != 0:
        shared = hg.SharedBatch(name, n, int(bases[-1]), create=False)
    pinned = shared.pin(bases[rank], bases[rank + 1])
    region = shared.region(bases[rank], bases[rank + 1])
    pipe.synth_texts(fr, g, tb, region)                                # warm-up into the shared buffer (page faults)
    e2e_steps = max(1, min(args.e2e_steps, args.steps))
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        off, cnt, _, tm = pipe.synth_texts(fr, g, tb, region)
        shared.publish(mine, int(bases[rank]), off, cnt)
    torch.cuda.synchronize(local_rank)
    e2e_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
    assert np.array_equal(cnt.astype(np.int64), my_counts)
    red = torch.tensor([dev_ms, e2e_ms, float(my_counts.sum()), float(ws.walked_utterances)], dtype=torch.float64, device=dev)
    per_rank = [red.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, red)
    sync_all()
    report = None
    if rank == 0:
        per = np.array([p.cpu().numpy() for p in per_rank])
        total_audio = float(per[:, 2].sum()) / SAMPLE_RATE
        # the gather: every utterance of the batch is in MY mapping of the shared buffer, in batch order
        assert int(shared.counts.astype(np.int64).sum()) == int(per[:, 2].sum())
        checked = 0
        if world > 1:   # utterances other ranks wrote equal what this rank synthesises for the same text
            probe = [int(shards[r][len(shards[r]) // 2]) for r in range(1, world)][:3]
            pp = fr.plan([texts[i] for i in probe], speeds[probe])
            for k, got in enumerate(g.synth_list(pp, prm)):
                assert np.array_equal(got, shared.utterance(probe[k])), f"gathered utterance {probe[k]} differs"
                checked += 1
        dev_max, e2e_max = float(per[:, 0].max()), float(per[:, 1].max())
        report = {
            "workload": f"BASELINE configs[3]: ONE batch of {n} synthetic sentences (~200 chars) at mixed speeds 0.5-2.0 (WSOLA), "
                        f"sharded by utterance over {world} GPU(s) (greedy LPT on text length / speed), host-side gather into one "
                        "shared buffer in batch order, no data-path collective",
            "scaling": "strong", "n_gpus": world, "audio_seconds": total_audio,
            "value": total_audio / (dev_max / 1e3), "unit": UNIT, "ms_per_step": dev_max,
            "per_rank_device_ms": [float(x) for x in per[:, 0]],
            "e2e": {"value": total_audio / (e2e_max / 1e3), "unit": UNIT, "ms_per_step": e2e_max,
                    "per_rank_ms": [float(x) for x in per[:, 1]],
                    "call": "ctts_b200_synth_texts per rank, device->host copies straight into the shared buffer",
                    "d2h_GBps_all_gpus": 2e-9 * sum(all_used) / (e2e_max / 1e3),
                    "shared_buffer_page_locked": bool(pinned)},
            "gather": {"utterances_in_shared_buffer": int(n), "cross_rank_utterances_checked_bit_exact": checked},
            "chain_walked_utterances": int(per[:, 3].sum()),
            "limiter": "device: per-rank kernel time (assemble + WSOLA verify + overlap-add) scales with the shard; e2e: "
                       "the box's aggregate device->host bandwidth (see d2h_GBps_all_gpus) and, on few host cores per GPU, the planner threads",
        }
    sync_all()
    shared.close(unlink=rank == 0)
    return report


VOICE = "seeded synthetic voice.db (1787 units, 9.2 M samples), shipped config values"


def base_config(args) -> dict:
    """The `config` object: identical in both arms (ours and --impl reference)."""
    return {"workload": workload_name(args), "voice": VOICE,
            "l2": "inputs and outputs of a step (GBs) exceed the 126 MB L2; the 18 MB voice pool is L2-resident by design"}


DUMP_PCM_BYTES = 48 << 20   # float32 PCM that --dump-outputs writes over all ranks; with the counts it stays under 64 MB


def dump_outputs(out_dir: str, rp, counts: np.ndarray, rank: int, world: int) -> None:
    """What the caller of the timed path (ctts_gpu_plan_run) receives from its last step, as .npy files:
      counts.npy          samples of every utterance (float64)
      pcm.npy             the PCM of a seeded sample of whole utterances, concatenated in batch order (float32)
      pcm_utterances.npy  the utterances pcm.npy holds, ascending (float64)
      pcm_strided.npy     every k-th sample of the batch's PCM (all utterances concatenated in batch order) from a
                          seeded start, k as small as the budget allows (float32)
    Each PCM file gets half of the budget.  The whole utterances are a seeded permutation's first ones whose counts
    fit, so two correct builds run with the same arguments dump the same ones, whatever their output layout; with a
    batch that fits, pcm.npy holds every utterance and pcm_strided.npy every sample.  Ranks > 1 add _rank<r> to the
    names."""
    budget = DUMP_PCM_BYTES // world // (2 * 4)                 # float32 samples of each of the two PCM files
    off = rp.out_offsets().astype(np.int64)
    cnt = counts.astype(np.int64)
    order = np.random.default_rng(0).permutation(rp.n_utts)
    pick = np.sort(order[np.cumsum(cnt[order]) <= budget])
    starts = np.concatenate([[0], np.cumsum(cnt)])
    stride = max(1, -(-int(starts[-1]) // budget))
    first = int(np.random.default_rng(1).integers(stride))    # position of the first strided sample in the batch
    picked = set(pick.tolist())
    whole, strided = [np.zeros(0, np.int16)], [np.zeros(0, np.int16)]
    for u in range(rp.n_utts):
        lo = first + max(0, -(-(int(starts[u]) - first) // stride)) * stride - int(starts[u])
        if u not in picked and lo >= cnt[u]:
            continue
        x = rp.read_pcm(int(off[u]), int(cnt[u]))
        if u in picked:
            whole.append(x)
        strided.append(x[lo::stride].copy())                   # not a view: x is freed once used
    sfx = f"_rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"counts{sfx}.npy"), counts.astype(np.float64))
    np.save(os.path.join(out_dir, f"pcm{sfx}.npy"), np.concatenate(whole).astype(np.float32))
    np.save(os.path.join(out_dir, f"pcm_utterances{sfx}.npy"), pick.astype(np.float64))
    np.save(os.path.join(out_dir, f"pcm_strided{sfx}.npy"), np.concatenate(strided).astype(np.float32))


def peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_facts(kernel: str) -> dict:
    """What the committed ncu captures say about one launch of a kernel at full batch size (profiles/traffic.json):
    dram_bytes, issue_active_pct, warp_instructions, ms, share_of_step_pct."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return dict(json.load(f).get(kernel) or {})
    except Exception:
        return {}


class ClockSampler:
    """nvidia-smi sampled every 50 ms in the background; mark() brackets the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.path = tempfile.mktemp(suffix=".csv")
        self.out = open(self.path, "w")
        self.proc = None
        self.lo = self.hi = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=self.out, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def _lines(self) -> int:
        try:
            with open(self.path) as f:
                return sum(1 for _ in f)
        except OSError:
            return 0

    def wait_ready(self, timeout: float = 8.0) -> None:
        t0 = time.time()
        while self.proc is not None and self._lines() < 2 and time.time() - t0 < timeout:
            time.sleep(0.05)

    def mark_begin(self) -> None:
        self.lo = self._lines()

    def mark_end(self) -> None:
        time.sleep(0.06)  # let the sample that covers the end of the region land
        self.hi = self._lines()

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.close()
        rows = []
        with open(self.path) as f:
            for line in f:
                parts = [p.strip() for p in line.split(",")]
                if len(parts) >= 7:
                    rows.append(parts)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        lo = max((self.lo or 0) - 1, 0)
        hi = min(self.hi if self.hi is not None else len(rows), len(rows))
        sel = rows[lo:max(hi, lo + 1)] or rows[-1:]
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for parts in sel:
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(max(smax))
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


def run_reference_cpu(texts, speeds, db_bytes: bytes, n_sample: int, procs: int):
    """Times oracle/_ref/ctts_ref_bench (the unmodified reference, N processes) on texts[:n_sample]."""
    import harness as H
    if not os.path.exists(H.REF_BENCH):
        raise RuntimeError("oracle/_ref/ctts_ref_bench is missing (built from /root/reference by oracle/Makefile)")
    with tempfile.TemporaryDirectory() as d:
        dbp = os.path.join(d, "voice.db")
        with open(dbp, "wb") as f:
            f.write(db_bytes)
        tsv = os.path.join(d, "texts.tsv")
        with open(tsv, "w", encoding="utf-8") as f:
            for t, s in zip(texts[:n_sample], speeds[:n_sample]):
                f.write(f"{float(s):.3f}\t{t}\n")
        r = subprocess.run([H.REF_BENCH, dbp, H.SHIPPED_YAML, H.NORM_CSV, tsv, str(procs)],
                           capture_output=True, text=True, timeout=1800)
        if r.returncode != 0:
            raise RuntimeError(f"ctts_ref_bench failed: {r.stderr[-400:]}")
        res = json.loads(r.stdout.strip().splitlines()[-1])
    return res


def cpu_sample_size(n_utts: int, cores: int, mixed: bool) -> int:
    # ~30 ms/utt/core at speed 1.0, ~0.3 s/utt/core through WSOLA; aim at 10-20 s of wall time
    per_core = 40 if mixed else 400
    return int(max(1, min(n_utts, cores * per_core)))


def main() -> int:
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1

    if args.impl == "reference":
        # the reference's own CPU implementation on the host cores; rank 0 alone runs it
        if rank != 0:
            return 0
        import harness as H
        texts, speeds = workload(args, 0)
        db = H.synthetic_db()
        n_sample = cpu_sample_size(args.utts, cores, args.workload == "mixed")
        for _ in range(max(args.warmup, 0) and 1):
            run_reference_cpu(texts, speeds, db, min(n_sample, cores), cores)
        secs, samples = 0.0, 0
        for _ in range(args.steps):
            r = run_reference_cpu(texts, speeds, db, n_sample, cores)
            secs += r["seconds"]
            samples += r["samples"]
        value = samples / SAMPLE_RATE / secs
        line = {
            "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16/f32",
            "data": "synthetic",
            "config": base_config(args),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
                             "sample": f"first {n_sample} utterances of the workload per step, {cores} processes of the unmodified reference (oracle/_ref/ctts_ref_bench)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the back end has no CPU fallback"}))
        return 1
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import harness as H
    pkg = importlib.import_module("2026-simple-c-tts_b200")
    gpu = importlib.import_module("2026-simple-c-tts_b200.gpu")

    db = H.synthetic_db()
    cfg = H.shipped_config()
    fr = pkg.front.Front(db, cfg, H.NORM_CSV)
    prm = fr.params()
    texts, speeds = workload(args, rank)
    t0 = time.time()
    plan = fr.plan(texts, speeds)
    plan_s = time.time() - t0

    g = gpu.GpuSynth(db, local_rank)
    stream = torch.cuda.Stream(device=local_rank)
    g.set_stream(stream.cuda_stream)
    rp = g.create_plan(plan, prm)
    info = rp.info()
    out_samples = rp.out_samples
    d_out = torch.empty(max(out_samples, 8), dtype=torch.int16, device=f"cuda:{local_rank}")

    def sync_all():
        torch.cuda.synchronize(local_rank)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(local_rank)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    try:
        for _ in range(args.warmup):
            rp.run(d_out.data_ptr())
        sync_all()
        if sampler:
            sampler.wait_ready()
            sampler.mark_begin()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        with torch.cuda.stream(stream):
            evs[0].record(stream)
            for k in range(args.steps):
                rp.run(d_out.data_ptr())
                evs[k + 1].record(stream)
        sync_all()
        if sampler:
            sampler.mark_end()
    finally:   # a failed step must not leave nvidia-smi polling
        clocks = sampler.stop() if sampler else None
    step_ms = [evs[k].elapsed_time(evs[k + 1]) for k in range(args.steps)]
    total_ms = evs[0].elapsed_time(evs[args.steps])
    counts = rp.counts()  # of the last timed step (there may be no warm-up); surfaces device error flags
    audio_s = float(counts.astype(np.int64).sum()) / SAMPLE_RATE
    n_out = int(counts.astype(np.int64).sum())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rp, counts, rank, world)

    # ---- the same resident plan with the word-region deduplication switched off (every region assembled): reported
    #      beside `value` so that the share of the speed-up that comes from repeated words in the batch is visible
    nodedup_ms = level1_ms = None
    zipf = None
    if rank == 0 and info.n_canon_tasks:
        os.environ["CTTS_GPU_REGION_DEDUP"] = "0"       # knobs are read once, by ctts_gpu_init
        g0 = gpu.GpuSynth(db, local_rank)
        os.environ.pop("CTTS_GPU_REGION_DEDUP")
        g0.set_stream(stream.cuda_stream)
        k0 = max(3, min(args.steps, 10))

        def resident_ms(ctx, pl, out=None):
            r = ctx.create_plan(pl, prm)
            if out is None:
                out = torch.empty(max(r.out_samples, 8), dtype=torch.int16, device=f"cuda:{local_rank}")
            for _ in range(3):
                r.run(out.data_ptr())
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                a0.record(stream)
                for _ in range(k0):
                    r.run(out.data_ptr())
                a1.record(stream)
            torch.cuda.synchronize(local_rank)
            c, i = r.counts(), r.info()
            r.close()
            return a0.elapsed_time(a1) / k0, c, i

        nodedup_ms, c0, _ = resident_ms(g0, plan, d_out)
        assert np.array_equal(c0, counts)
        os.environ["CTTS_GPU_REGION_DEDUP"] = "1"       # regions up to their contour only
        g1 = gpu.GpuSynth(db, local_rank)
        os.environ.pop("CTTS_GPU_REGION_DEDUP")
        g1.set_stream(stream.cuda_stream)
        level1_ms, c1, _ = resident_ms(g1, plan, d_out)
        assert np.array_equal(c1, counts)
        g1.close()
        # ---- one more point on the same axis: the same sentence generator over a Zipf vocabulary of 20 000 word types
        #      (rank r has probability ~ 1 / (r + 2.7)): about one token in ten occurs once in the batch
        if args.workload == "speed1" and not args.vocab and args.utts >= 1024:
            zt = pkg.corpus.batch(args.utts, seed=1234, target_chars=200, vocab=pkg.corpus.Vocabulary(20000))
            zplan = fr.plan(zt, np.ones(args.utts, dtype=np.float32))
            z_ms, zc, zi = resident_ms(g, zplan)
            z0_ms, zc0, _ = resident_ms(g0, zplan)
            assert np.array_equal(zc, zc0)
            z_audio = float(zc.astype(np.int64).sum()) / SAMPLE_RATE
            zipf = {"vocabulary": 20000, "utterances": args.utts, "audio_seconds": z_audio,
                    "ms_per_step": z_ms, "value": z_audio / (z_ms / 1e3),
                    "ms_per_step_without": z0_ms, "value_without_region_dedup": z_audio / (z0_ms / 1e3),
                    "region_tasks": int(zi.n_tasks), "canonical_regions": int(zi.n_canon_tasks),
                    "tasks_served_from_them": int(zi.n_dedup_tasks),
                    "share_of_bound_samples": float(zi.dedup_bound_samples) / max(float(zi.bound_samples), 1.0),
                    "whole_task_sources": int(zi.n_source_tasks), "tasks_copied_whole": int(zi.n_reuse_tasks),
                    "share_of_bound_samples_copied_whole": float(zi.reuse_bound_samples) / max(float(zi.bound_samples), 1.0)}
        g0.close()

    # ---- e2e, host buffers, copies inside the timed region: (1) plan -> PCM through the drop-in call
    #      ctts_gpu_synth_batch, (2) TEXT -> PCM through ctts_b200_synth_texts (planner threads + device session)
    e2e = None
    if not args.no_e2e:
        pipe = importlib.import_module("2026-simple-c-tts_b200.pipeline")
        offsets = rp.out_offsets()
        host_out = torch.empty(max(out_samples, 8) + 4096, dtype=torch.int16).pin_memory()
        host_np = host_out.numpy()
        e2e_steps = max(1, min(args.e2e_steps, args.steps))
        g.synth_batch(plan, prm, host_np, offsets)  # warm-up (allocates the lanes' buffers once)
        sync_all()
        te = time.perf_counter()
        for _ in range(e2e_steps):
            _, _, c2 = g.synth_batch(plan, prm, host_np, offsets)
        torch.cuda.synchronize(local_rank)
        plan_s_e2e = (time.perf_counter() - te) / e2e_steps
        g.synth_batch_packed(plan, prm, host_np)
        sync_all()
        te = time.perf_counter()
        for _ in range(e2e_steps):
            g.synth_batch_packed(plan, prm, host_np)
        torch.cuda.synchronize(local_rank)
        plan_packed_s = (time.perf_counter() - te) / e2e_steps
        tb = pipe.TextBatch(texts, speeds)
        pipe.synth_texts(fr, g, tb, host_np)          # warm-up
        sync_all()
        te = time.perf_counter()
        for _ in range(e2e_steps):
            _, c3, used, tm = pipe.synth_texts(fr, g, tb, host_np)
        torch.cuda.synchronize(local_rank)
        e2e_s = (time.perf_counter() - te) / e2e_steps
        assert np.array_equal(c3, c2), "text pipeline and planned batch disagree"
        # the same texts again through a warm plan cache (a server that is asked for the same sentences again)
        cache = pipe.PlanCache(1 << 30)
        pipe.synth_texts(fr, g, tb, host_np, cache=cache)
        sync_all()
        te = time.perf_counter()
        _, c4, _, tmc = pipe.synth_texts(fr, g, tb, host_np, cache=cache)
        torch.cuda.synchronize(local_rank)
        cached_ms = 1e3 * (time.perf_counter() - te)
        cache_stats = cache.stats()
        cache.close()
        assert np.array_equal(c4, c2)
        h2d = int(plan.ops.nbytes + plan.utt_op_begin.nbytes + plan.speed.nbytes)
        d2h = int(used * 2 + 8 * plan.n_utts)
        e2e = {"seconds_per_step": e2e_s, "h2d": h2d, "d2h": d2h, "steps": e2e_steps,
               "audio_s": float(c3.astype(np.int64).sum()) / SAMPLE_RATE, "plan_to_pcm_s": plan_s_e2e,
               "plan_to_pcm_packed_ms": 1e3 * plan_packed_s,
               "cached": {"ms_per_step": cached_ms, "all_planned_ms": 1e3 * tmc.all_plans_s, **cache_stats},
               "timing": {"first_piece_planned_ms": 1e3 * tm.first_plan_s, "all_planned_ms": 1e3 * tm.all_plans_s,
                          "all_submitted_ms": 1e3 * tm.all_submitted_s, "done_ms": 1e3 * tm.done_s,
                          "submitter_waited_for_plans_ms": 1e3 * tm.wait_for_plans_s, "device_pieces": int(tm.pieces)}}

    # ---- reduce over ranks: time = max, work = sum
    t_rank = torch.tensor([total_ms, audio_s, e2e["seconds_per_step"] if e2e else 0.0,
                           e2e["audio_s"] if e2e else 0.0, e2e["plan_to_pcm_s"] if e2e else 0.0],
                          dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        mx = t_rank.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t_rank.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        total_ms_all, audio_all = float(mx[0]), float(sm[1])
        e2e_s_all, e2e_audio_all, e2e_plan_s_all = float(mx[2]), float(sm[3]), float(mx[4])
    else:
        total_ms_all, audio_all = total_ms, audio_s
        e2e_s_all, e2e_audio_all, e2e_plan_s_all = (e2e["seconds_per_step"], e2e["audio_s"], e2e["plan_to_pcm_s"]) if e2e else (0.0, 0.0, 0.0)

    strong = None
    if not args.no_strong and args.workload == "speed1":
        d_out = host_out = host_np = None   # give the memory back before the second workload
        strong = strong_scaling_leg(args, rank, local_rank, world, fr, g, prm, pkg, gpu, sync_all, dist, torch)

    if rank == 0:
        ms_per_step = total_ms_all / args.steps
        value = audio_all / (ms_per_step / 1e3)
        peak, peak_src = peak_hbm()
        # algorithmic bytes of one launch of the assembly kernel (SURVEY.md 8d):
        # 2 B per gathered unit sample + 2 B per output sample + 32 B per plan op
        alg_bytes = 2 * int(info.gather_samples) + 2 * n_out + int(plan.ops.nbytes)
        kern_ms = float(np.mean(step_ms))
        achieved = alg_bytes / (kern_ms / 1e3) / 1e9
        dominant = "assemble_kernel"      # the largest kernel of the step in every workload (mixed: 46 %, see kernels_ncu)
        facts = ncu_facts(dominant)
        traffic = facts.get("dram_bytes")
        step_kernels = ["assemble_kernel"] + (["wsola_verify_kernel", "wsola_ola_kernel"] if args.workload == "mixed" else [])
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int16/f32", "data": "synthetic",
            "config": base_config(args),
            "details": {
                "audio_seconds_per_gpu_step": audio_s, "plan_ops": int(plan.ops.shape[0]),
                "output_GB_per_step": 2 * n_out / 1e9,
                "value_is": "one ctts_gpu_plan_run of a RESIDENT plan (compiled and uploaded once; plan, voice and voice tables in HBM)",
                "voice_tables": "per context, built by device kernels before the first plan runs: normalize_rms of every unit "
                                "(normalized pool, one per target_rms) and estimate_pitch of untouched unit heads per analysis "
                                "length; the e2e warm-up call pays for them, later calls reuse them",
                "front_end_plan_seconds": plan_s,
                "window_samples": int(info.window_samples), "smem_bytes": int(info.smem_bytes),
                "region_tasks": int(info.n_tasks), "region_tasks_in_hbm_window": int(info.n_global_tasks),
                "persistent_ctas": int(info.grid), "ctas_per_sm": int(info.ctas_per_sm),
                "region_dedup": {
                    "what": "equal word regions of the batch are assembled ONCE PER LAUNCH (canonical tasks, inside the timed step) and "
                            "copied by their other occurrences, which run their own contour; tasks that are equal as a whole (same "
                            "region, same contour factors, same pause) are run once and copied; nothing is kept from one step to the "
                            "next; CTTS_GPU_REGION_DEDUP=0 switches it off (value_without_region_dedup), =1 keeps the first level only",
                    "canonical_regions": int(info.n_canon_tasks), "tasks_served_from_them": int(info.n_dedup_tasks),
                    "share_of_bound_samples": float(info.dedup_bound_samples) / max(float(info.bound_samples), 1.0),
                    "whole_task_sources": int(info.n_source_tasks), "tasks_copied_whole": int(info.n_reuse_tasks),
                    "share_of_bound_samples_copied_whole": float(info.reuse_bound_samples) / max(float(info.bound_samples), 1.0),
                    "ms_per_step_regions_only": level1_ms,
                    "ms_per_step_without": nodedup_ms,
                    "value_without_region_dedup": (audio_s / (nodedup_ms / 1e3)) if nodedup_ms else None,
                    "corpus_note": "the benchmark corpus (round-1 generator, SURVEY 8d) draws its sentences from ~190 words plus numbers "
                                   "and abbreviations, so few distinct regions serve most tasks; a batch of all-distinct words costs what "
                                   "value_without_region_dedup says; zipf_vocabulary is the same generator over 20 000 word types",
                    "zipf_vocabulary": zipf},
                "threads_per_cta": int(info.threads),
            },
            "gpu_launches": int(info.kernel_launches) * args.steps,
            "clocks": clocks,
            "roofline": {
                "bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                # the same on DRAM-counter bytes (the pool gather is served by L2, so this is about half of frac)
                "frac_dram": (traffic / (kern_ms / 1e3) / 1e9 / peak) if traffic and args.workload == "speed1" and args.utts == 4096 else None,
                # SURVEY 8(d): the stage is instruction-issue bound, so the issue-slot utilisation is the fraction that
                # says how far the kernel is from ITS ceiling (ncu, committed captures; FP32 pipe utilisation beside it)
                "issue_active_pct": facts.get("issue_active_pct"), "fma_pipe_pct": facts.get("fma_pipe_pct"),
                "ceiling": "at 100 % issue slots the measured instruction count of a 4096-utterance launch (4.69 G warp instructions with "
                           "both levels of the deduplication, 6.67 G with equal regions only, 10.82 G without; what is left is fixed by "
                           "bit-exactness: DESIGN.md 6) takes 4.0 ms = 0.40 of the HBM peak (5.7 ms / 9.3 ms for the other two); the "
                           "north star's 0.60 is 1.6 ms",
                "kernels_ncu": {k: ncu_facts(k) for k in step_kernels},
                "frac_of_nominal_8000_GBs": achieved / 8000.0,   # the north star quotes ~8 TB/s; SURVEY 8d asks for both
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": kern_ms,
                "kernel_ms_min_max": [float(np.min(step_ms)), float(np.max(step_ms))],
                "note": "step = one assemble_kernel launch (+4 small memsets)" if args.workload != "mixed"
                        else "step = assemble + wsola_scan + wsola_verify + wsola_search (exits) + wsola_ola: achieved / frac are for the WHOLE step "
                             "(algorithmic bytes / step time); the stretch kernels are shared-memory / issue bound (kernels_ncu), the HBM "
                             "fraction is reported because the metric demands it",
            },
        }
        if args.workload == "mixed":
            ws = rp.wsola_stats()
            line["details"]["wsola"] = {"frames": int(ws.frames), "tier2_candidates": int(ws.tier2_candidates),
                                       "exact_evaluations": int(ws.exact_evaluations),
                                       "chain_walked_utterances": int(ws.walked_utterances),
                                       "chain_walked_frames": int(ws.walked_frames)}
        if e2e:
            line["e2e"] = {"value": e2e_audio_all / e2e_s_all, "unit": UNIT,
                           "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                           "steps": e2e["steps"], "ms_per_step": 1e3 * e2e_s_all,
                           "call": "ctts_b200_synth_texts: texts (C strings) -> pinned host PCM; planner threads feed a device "
                                   "session piece by piece, like for like with the reference arm (text -> PCM)",
                           "host_threads": cores, "rank0_timing": e2e["timing"],
                           "rank0_warm_plan_cache": e2e["cached"],
                           "d2h_GBps_all_gpus": 1e-9 * world * e2e["d2h"] / e2e_s_all,
                           "plan_to_pcm": {"value": e2e_audio_all / e2e_plan_s_all, "ms_per_step": 1e3 * e2e_plan_s_all,
                                           "call": "ctts_gpu_synth_batch on a ready plan (the back end alone; caller-defined slots, span copies)",
                                           "rank0_packed_ms_per_step": e2e["plan_to_pcm_packed_ms"],
                                           "packed_call": "ctts_gpu_synth_batch_packed (library layout, exact-size copies)"}}
        if strong:
            line["strong"] = strong
        if not args.no_cpu_baseline:
            try:
                n_sample = cpu_sample_size(args.utts, cores, args.workload == "mixed")
                r = run_reference_cpu(texts, speeds, db, n_sample, cores)
                line["cpu_baseline"] = {
                    "value": r["samples"] / SAMPLE_RATE / r["seconds"], "unit": UNIT, "cores": cores,
                    "kind": "reference",
                    "sample": f"first {n_sample} utterances of the same workload, {cores} processes of the unmodified reference (oracle/_ref/ctts_ref_bench), {r['seconds']:.1f} s",
                }
            except Exception as e:  # the GPU number stands on its own
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": cores, "kind": "reference",
                                        "sample": f"failed: {e}"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
