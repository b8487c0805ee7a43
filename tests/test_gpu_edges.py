"""GPU parity on the constructed voices of edge_voices.py (short units, pitch decisions at their bounds,
WSOLA near fixed points, tiny stretched utterances, amplitude extremes, trim edges): every utterance
bit-exact against the oracle, through a resident plan run twice and through the drop-in call, under the
execution-path knobs that change how joins and regions are assembled.  test_edge_voices.py proves on the
CPU that each family reaches its edge.

Run on a B200 with:  python -m pytest tests/test_gpu_edges.py -m gpu
"""
import numpy as np
import pytest

import edge_voices as E

pytestmark = pytest.mark.gpu

ENVS = {
    "default": {},
    "pitch_slots3": {"CTTS_GPU_PITCH_SLOTS": "3"},    # unit heads estimated in the join, as a pair
    "window2048": {"CTTS_GPU_WINDOW": "2048"},        # HBM-slot regions, joins reaching back across tasks
    "no_dedup": {"CTTS_GPU_REGION_DEDUP": "0"},
}


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


def _assert_same(got, want, what=""):
    assert len(got) == len(want), f"{what}: length {len(got)} != {len(want)}"
    if not np.array_equal(got, want):
        d = np.nonzero(got != want)[0]
        raise AssertionError(f"{what}: {len(d)} of {len(want)} samples differ, first at {d[:5]}, "
                             f"max |d| {np.abs(got.astype(int) - want.astype(int)).max()}")


@pytest.mark.parametrize("env", list(ENVS))
@pytest.mark.parametrize("name", list(E.FAMILIES))
def test_edge_family_bit_exact(gpu, monkeypatch, name, env):
    fam = E.family(name)
    plan, prm, want = fam.plan(), fam.prm(), fam.expected()
    for k, v in ENVS[env].items():
        monkeypatch.setenv(k, v)
    g = gpu.GpuSynth(fam.db, 0)
    try:
        rp = g.create_plan(plan, prm)
        for run in range(2):            # the second run is a new epoch of the plan's region states
            rp.run()
            for u, got in enumerate(rp.utterances()):
                _assert_same(got, want[u], f"{name} {env} resident run {run} utt {u} {fam.texts[u][:30]!r} speed {plan.speed[u]}")
        if name == "wsola":
            st = rp.wsola_stats()
            assert st.tier2_candidates > 0 and st.exact_evaluations > 0, (st.tier2_candidates, st.exact_evaluations)
            assert st.walked_utterances >= 1
        outs = g.synth_list(plan, prm)
        for u in range(plan.n_utts):
            _assert_same(outs[u], want[u], f"{name} {env} pieces utt {u} {fam.texts[u][:30]!r} speed {plan.speed[u]}")
    finally:
        g.close()


def test_wsola_noiseless_patterns_are_walked(gpu):
    """The noiseless near-periodic units alone: a candidate one period away scores 1.0f as well, so the
    speculated chain is wrong somewhere and the chain walk resolves it."""
    fam = E.family("wsola")
    plan = fam.plan()
    pick = [u for u, ws in enumerate(fam.words) if ws[0][0] in fam.info["noiseless"]]
    sub = plan.select(pick)
    want = fam.expected()
    g = gpu.GpuSynth(fam.db, 0)
    try:
        rp = g.create_plan(sub, fam.prm())
        rp.run()
        for k, got in enumerate(rp.utterances()):
            _assert_same(got, want[pick[k]], f"noiseless utt {pick[k]}")
        assert rp.wsola_stats().walked_utterances >= 1
    finally:
        g.close()


XF_SWEEP_MS = {4.49: 198, 4.54: 200, 4.99: 220, 6.31: 278, 9.94: 438, 9.98: 440, 12.5: 550, 12.55: 552}


@pytest.mark.parametrize("ms", list(XF_SWEEP_MS))
def test_crossfade_sweep_on_the_small_voice(H, gpu, small_db, oracle_small, ms):
    """Crossfades whose 2 xf lands at 198 .. 552 samples: the pitch search of ordinary joins runs over a
    truncated lag range and fewer than 220 terms."""
    assert 2 * E.ms_to_samples(ms) == XF_SWEEP_MS[ms]
    cfg = H.shipped_config()
    cfg.crossfade_ms = ms
    cfg.crossfade_vowel_ms = ms
    fr = H.front.Front(small_db, cfg, H.NORM_CSV)
    prm = fr.params()
    texts = H.corpus.batch(40, seed=int(ms * 100), target_chars=70)
    speeds = [1.0] * 32 + [1.5] * 8
    plan = fr.plan(texts, speeds)
    assert any(int(op["b"]) == XF_SWEEP_MS[ms] // 2 for op in plan.ops[plan.ops["kind"] == H.front.OP_UNIT])
    g = gpu.GpuSynth(small_db, 0)
    outs = g.synth_list(plan, prm)
    for u in range(plan.n_utts):
        want, _ = oracle_small.synth(prm, plan.utt_ops(u), float(speeds[u]))
        _assert_same(outs[u], want, f"xf {ms} ms utt {u} speed {speeds[u]}")
