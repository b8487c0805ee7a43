"""bench.py --dump-outputs: the files it writes and that they hold what the timed path computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest


class _Plan:
    """Stand-in for gpu.ResidentPlan: slots of the given bounds, PCM already in them."""

    def __init__(self, bounds, counts, seed=0):
        self.n_utts = len(bounds)
        self.off = np.concatenate([[0], np.cumsum(bounds)]).astype(np.uint64)
        self.buf = np.random.default_rng(seed).integers(-32768, 32768, int(self.off[-1]), dtype=np.int16)
        self.counts = np.asarray(counts, dtype=np.uint32)

    def out_offsets(self):
        return self.off

    def read_pcm(self, first, n):
        return self.buf[first:first + n].copy()


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_outputs_writes_every_utterance_when_it_fits(tmp_path):
    import bench
    rp = _Plan([10, 7, 0, 12], [9, 7, 0, 3])
    bench.dump_outputs(str(tmp_path), rp, rp.counts, 0, 1)
    got = _load(tmp_path)
    assert set(got) == {"counts", "pcm", "pcm_utterances", "pcm_strided"}
    assert got["counts"].dtype == np.float64 and got["pcm"].dtype == got["pcm_strided"].dtype == np.float32
    assert np.array_equal(got["counts"], [9, 7, 0, 3]) and np.array_equal(got["pcm_utterances"], [0, 1, 2, 3])
    want = np.concatenate([rp.buf[0:9], rp.buf[10:17], rp.buf[17:20]]).astype(np.float32)
    assert np.array_equal(got["pcm"], want) and np.array_equal(got["pcm_strided"], want)


def test_dump_outputs_samples_within_the_budget(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_PCM_BYTES", 2 * 4 * 500)    # 500 float32 samples for each of the two PCM files
    bounds = np.random.default_rng(3).integers(50, 200, 40)
    counts = bounds - np.random.default_rng(4).integers(0, 50, 40)
    rp = _Plan(bounds, counts)
    every = np.concatenate([rp.buf[int(rp.off[u]):int(rp.off[u]) + counts[u]] for u in range(40)]).astype(np.float32)
    bench.dump_outputs(str(tmp_path / "a"), rp, rp.counts, 0, 1)
    bench.dump_outputs(str(tmp_path / "b"), rp, rp.counts, 1, 2)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert set(b) == {"counts_rank1", "pcm_rank1", "pcm_utterances_rank1", "pcm_strided_rank1"}
    pick = a["pcm_utterances"].astype(np.int64)
    assert 0 < len(pick) < 40 and np.all(np.diff(pick) > 0) and counts[pick].sum() <= 500
    assert np.array_equal(a["pcm"], np.concatenate([rp.buf[int(rp.off[u]):int(rp.off[u]) + counts[u]] for u in pick]))
    stride = -(-len(every) // 500)
    assert stride > 1 and any(np.array_equal(a["pcm_strided"], every[f::stride]) for f in range(stride))
    # the budget is shared by the ranks
    assert counts[b["pcm_utterances_rank1"].astype(np.int64)].sum() <= 250 and len(b["pcm_strided_rank1"]) <= 250
    # the sample depends on the counts, not on how the output is laid out
    bench.dump_outputs(str(tmp_path / "c"), _Plan(bounds + 64, counts, seed=1), counts.astype(np.uint32), 0, 1)
    assert np.array_equal(_load(tmp_path / "c")["pcm_utterances"], a["pcm_utterances"])


@pytest.mark.gpu
def test_bench_dumps_what_the_timed_steps_computed(H, tmp_path):
    """A small run without warm-up: the dumped PCM is the oracle's, and the same again on a second run."""
    args = [sys.executable, os.path.join(H.ROOT, "bench.py"), "--utts", "6", "--steps", "2", "--warmup", "0",
            "--no-e2e", "--no-strong", "--no-cpu-baseline", "--dump-outputs"]
    lines = []
    for d in ("a", "b"):
        r = subprocess.run(args + [str(tmp_path / d)], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads(r.stdout.strip().splitlines()[-1]))
    assert lines[0]["steps"] == 2 and lines[0]["value"] > 0
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert np.array_equal(a["pcm_utterances"], np.arange(6))
    db = H.synthetic_db()
    fr = H.front.Front(db, H.shipped_config(), H.NORM_CSV)
    texts = H.corpus.batch(6, seed=1234, target_chars=200)
    plan = fr.plan(texts, np.ones(6, dtype=np.float32))
    orc = H.Oracle(db)
    want = [orc.synth(fr.params(), plan.utt_ops(u), 1.0)[0] for u in range(6)]
    assert np.array_equal(a["counts"], [len(w) for w in want])
    want = np.concatenate(want).astype(np.float32)
    assert np.array_equal(a["pcm"], want) and np.array_equal(a["pcm_strided"], want)
