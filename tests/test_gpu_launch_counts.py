"""GPU tests of the launch count a resident plan reports (ctts_gpu_run_info.kernel_launches, DESIGN.md 3.3): the
kernels one ctts_gpu_plan_run enqueues, as torch.profiler (CUDA activity) sees them, are exactly that many.  The plans
take every launch condition of the stage chain: speed 1.0 and mixed speeds, the native rate and 16 kHz, loudness off,
with a sample-peak and with a true-peak ceiling, WSOLA without speculation, and a plan of more than 65 535 stretched
utterances whose grids are split at the grid.y limit.  A plan without tasks is left out on purpose: it counts the
assembly kernel it skips.

Run on a B200 with:  python -m pytest tests/test_gpu_launch_counts.py -m gpu
"""
import collections

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GRID_Y = 65535
PAIRS = [("olá", 1.5), ("bom dia", 0.75), ("casa", 1.25), ("sim", 0.6180339), ("não", 2.0), ("mar azul", 1.2345678),
         ("olá dia", 1.0)]
N_BIG = 80000


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


@pytest.fixture(scope="module")
def batches(H, front_small):
    texts = H.corpus.batch(48, seed=31, target_chars=120)
    return {"speed 1.0": front_small.plan(texts, [1.0] * len(texts)),
            "mixed speeds": front_small.plan(texts, list(H.corpus.mixed_speeds(len(texts), seed=7)))}


def _ctx(gpu, db, hz, loudness):
    g = gpu.GpuSynth(db, 0)
    g.set_output_rate(hz)
    if loudness != "off":
        g.set_loudness(-16.0, -1.0, true_peak=loudness == "true peak")
    return g


def _profiled_kernels(rp):
    """The ctts:: kernels one run() of the plan enqueues, after a run that warms it up: name -> launches."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    rp.run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rp.run()
        torch.cuda.synchronize()
    return collections.Counter(e.name for e in prof.events() if "ctts::" in e.name)


def _check(rp):
    got = _profiled_kernels(rp)
    assert sum(got.values()) == rp.info().kernel_launches, got
    return got


@pytest.mark.parametrize("loudness", ("off", "sample peak", "true peak"))
@pytest.mark.parametrize("hz", (22050, 16000))
@pytest.mark.parametrize("speeds", ("speed 1.0", "mixed speeds"))
def test_launches_equal_the_reported_count(gpu, small_db, front_small, batches, speeds, hz, loudness):
    g = _ctx(gpu, small_db, hz, loudness)
    try:
        rp = g.create_plan(batches[speeds], front_small.params())
        assert (rp.info().n_stretch > 0) == (speeds == "mixed speeds")
        _check(rp)
    finally:
        g.close()


def test_without_wsola_speculation(gpu, small_db, front_small, batches, monkeypatch):
    monkeypatch.setenv("CTTS_GPU_WSOLA_SPECULATE", "0")   # read at init
    g = _ctx(gpu, small_db, 22050, "off")
    try:
        got = _check(g.create_plan(batches["mixed speeds"], front_small.params()))
        assert not any("wsola_verify_kernel" in k for k in got), got
    finally:
        g.close()


def test_grids_split_at_the_grid_y_limit(gpu, small_db, front_small):
    """N_BIG short utterances at 16 kHz with a true-peak ceiling, 6 in 7 stretched: the WSOLA verify, resample, both
    chunk passes, true-peak and apply grids are each launched in two slices."""
    pick = np.arange(N_BIG) % len(PAIRS)
    plan = front_small.plan([PAIRS[k][0] for k in pick], [PAIRS[k][1] for k in pick])
    g = _ctx(gpu, small_db, 16000, "true peak")
    try:
        rp = g.create_plan(plan, front_small.params())
        assert rp.info().n_stretch > GRID_Y
        got = _check(rp)
        per_kernel = {k: sum(v for name, v in got.items() if k in name) for k in
                      ("wsola_verify_kernel", "resample_kernel", "ld_chunk_kernel", "ld_true_peak_kernel", "ld_apply_kernel")}
        assert per_kernel == {"wsola_verify_kernel": 2, "resample_kernel": 2, "ld_chunk_kernel": 4,
                              "ld_true_peak_kernel": 2, "ld_apply_kernel": 2}, got
    finally:
        g.close()
