"""Word regions longer than the assembly kernel's shared window in the region deduplication.

Such regions are assembled in place: a canonical one in its region-store slot, an occurrence copies the store straight
into its utterance slot and resumes at its contour there, a whole task that is shared copies what it appended from its
utterance slot into the store, and its copies take it from there.  Every case is bit-exact against the oracle at every
deduplication level, for two runs of a resident plan (a new epoch of the region states) and for the drop-in call.

Run on a B200 with:  python -m pytest tests -m gpu
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


@pytest.fixture(scope="module")
def syn_db(H):
    return H.synthetic_db()


@pytest.fixture(scope="module")
def front_syn(H, syn_db):
    return H.front.Front(syn_db, H.shipped_config(), H.NORM_CSV)


@pytest.fixture(scope="module")
def oracle_syn(H, syn_db):
    return H.Oracle(syn_db)


def _assert_same(got, want, what=""):
    assert len(got) == len(want), f"{what}: length {len(got)} != {len(want)}"
    if not np.array_equal(got, want):
        d = np.nonzero(got != want)[0]
        raise AssertionError(f"{what}: {len(d)} of {len(want)} samples differ, first at {d[:5]}, "
                             f"max |d| {np.abs(got.astype(int) - want.astype(int)).max()}")


def _plan_info(gpu, db, plan, prm, monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    g = gpu.GpuSynth(db, 0)
    rp = g.create_plan(plan, prm)
    info = rp.info()
    rp.close()
    g.close()
    return info


def _check_levels(gpu, db, oracle, prm, plan, monkeypatch, env, what):
    """The plan at deduplication levels 2, 1 and 0 under `env`: resident plan run twice, then the drop-in call.
    Returns the plan info of each level."""
    want = [oracle.synth(prm, plan.utt_ops(u), float(plan.speed[u]))[0] for u in range(plan.n_utts)]
    infos = {}
    for mode in ("2", "1", "0"):
        monkeypatch.setenv("CTTS_GPU_REGION_DEDUP", mode)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        g = gpu.GpuSynth(db, 0)
        rp = g.create_plan(plan, prm)
        infos[mode] = rp.info()
        for _ in range(2):
            rp.run()
        outs = rp.utterances()
        for u in range(plan.n_utts):
            _assert_same(outs[u], want[u], f"{what}, level {mode}, utt {u}")
        rp.close()
        piece_outs = g.synth_list(plan, prm)
        for u in range(plan.n_utts):
            _assert_same(piece_outs[u], want[u], f"{what}, level {mode}, drop-in, utt {u}")
        g.close()
    assert infos["0"].n_canon_tasks == 0 and infos["0"].n_dedup_tasks == 0
    assert infos["1"].n_source_tasks == 0 and infos["1"].n_reuse_tasks == 0
    monkeypatch.delenv("CTTS_GPU_REGION_DEDUP")
    return infos


# the longest word regions of bench.py's batch (hyphenated compounds of long words: about 52 k output samples, 54 k
# bound), spelled-out numbers and long words, at the start of utterances, after a short first word, in the middle
LONG = ["computador-computador", "universidade-escuro", "importante-presidente", "universidade", "computador",
        "importante", "novecentos", "quatrocentos", "seiscentos"]


def _long_word_texts(rng, n):
    texts = []
    for i in range(n):
        words = list(rng.choice(LONG + ["casa", "a", "o", "bom", "dia"], size=int(rng.integers(3, 9))))
        if i % 3 == 0:
            words.insert(0, str(rng.choice(LONG)))              # the first region: the count threshold is not met
        elif i % 3 == 1:
            words.insert(0, "a")                                  # short first word: the threshold may not be met
        texts.append(" ".join(words) + str(rng.choice([".", ",", "!", ""])))
    texts += ["computador-computador computador-computador computador-computador."] * 3     # equal whole tasks
    texts += ["900 e 400 e 600", "900 e 400 e 600", "a 999 e 999"]
    return texts


def test_long_words_repeated(H, gpu, syn_db, front_syn, oracle_syn, monkeypatch):
    """Long words repeated at many positions with the window sized for the batch: the regions longer than it are
    deduplicated (canonical regions assembled in the store, occurrences resumed and whole tasks copied in their
    utterance slots)."""
    rng = np.random.default_rng(31)
    texts = _long_word_texts(rng, 36)
    plan = front_syn.plan(texts, [1.0] * len(texts))
    prm = front_syn.params()
    infos = _check_levels(gpu, syn_db, oracle_syn, prm, plan, monkeypatch, {}, "long words")
    i2 = infos["2"]
    assert i2.n_global_tasks > 20, i2.n_global_tasks
    assert i2.n_canon_tasks >= 5 and i2.n_reuse_tasks >= 3, (i2.n_canon_tasks, i2.n_reuse_tasks)
    # the same plan with every region deduplicated that can be: the longest regions are counted as well
    assert infos["1"].n_dedup_tasks == i2.n_dedup_tasks and infos["1"].n_canon_tasks == i2.n_canon_tasks


def test_small_window_every_region_is_long(H, gpu, small_db, front_small, oracle_small, monkeypatch):
    """A 2 048-sample window: nearly every region is longer than it, so canonical regions, resumes, sources and whole
    copies run in place."""
    words = ["casa", "mundo", "olá", "bom", "dia", "rato", "rua", "importante", "água", "trabalho"]
    rng = np.random.default_rng(5)
    texts = [" ".join(rng.choice(words, size=int(rng.integers(3, 12)))) + str(rng.choice([".", "?", ",", ""])) for _ in range(30)]
    texts += ["bom dia mundo", "bom dia mundo", "olá bom dia mundo", "casa casa casa casa", "casa casa casa casa"]
    speeds = [1.0] * len(texts)
    speeds[4] = 0.7
    plan = front_small.plan(texts, speeds)
    prm = front_small.params()
    infos = _check_levels(gpu, small_db, oracle_small, prm, plan, monkeypatch, {"CTTS_GPU_WINDOW": "2048"}, "window 2048")
    monkeypatch.delenv("CTTS_GPU_WINDOW")
    i2 = infos["2"]
    assert i2.n_global_tasks > i2.n_tasks // 2, (i2.n_global_tasks, i2.n_tasks)
    assert i2.n_canon_tasks >= 5 and i2.n_dedup_tasks > 2 * i2.n_canon_tasks and i2.n_reuse_tasks >= 5, \
        (i2.n_canon_tasks, i2.n_dedup_tasks, i2.n_reuse_tasks)


def test_fade_out_reaching_back_in_place(H, gpu, small_db, oracle_small, monkeypatch):
    """Fade-outs longer than short words (150 ms) with every region longer than the window: a source whose fade-out
    reaches back into the previous word gives up its samples and its copies fall back to the canonical region or
    assemble themselves."""
    for variant in range(2):
        cfg = H.shipped_config()
        cfg.fade_out_ms = 150.0
        if variant == 1:
            cfg.word_pause_ms = 0.0
            cfg.crossfade_ms = 120.0
            cfg.crossfade_vowel_ms = 160.0
        fr = H.front.Front(small_db, cfg, H.NORM_CSV)
        base = ["a e o a e o casa a e o", "o a o a o a mundo o a", "e casa e casa e casa e casa", "a o e bom dia a o e bom dia"]
        texts = base * 3 + ["casa " + base[0], base[1] + " dia"]
        plan = fr.plan(texts, [1.0] * len(texts))
        infos = _check_levels(gpu, small_db, oracle_small, fr.params(), plan, monkeypatch, {"CTTS_GPU_WINDOW": "2048"},
                              f"fade-out variant {variant}")
        monkeypatch.delenv("CTTS_GPU_WINDOW")
        assert infos["2"].n_global_tasks > 0 and infos["2"].n_source_tasks >= 4, (infos["2"].n_global_tasks, infos["2"].n_source_tasks)


def test_regions_just_above_and_below_the_window(H, gpu, small_db, front_small, oracle_small, monkeypatch):
    """The window set 8 samples below and at the largest task bound of a batch of repeated phrases: the longest
    tasks are in place in one case and in the window in the other, with identical deduplication counts."""
    texts = ["casa mundo casa mundo casa.", "bom dia casa mundo casa.", "casa mundo casa mundo casa."] * 3
    plan = front_small.plan(texts, [1.0] * len(texts))
    prm = front_small.params()
    monkeypatch.setenv("CTTS_GPU_REGION_DEDUP", "2")

    def n_global(w):
        return _plan_info(gpu, small_db, plan, prm, monkeypatch, {"CTTS_GPU_WINDOW": str(w)}).n_global_tasks

    lo, hi = 256, 1 << 17           # smallest window (multiple of 8) with no task longer than it: bisection
    assert n_global(hi) == 0
    while hi - lo > 8:
        mid = (lo + hi) // 16 * 8
        if n_global(mid) == 0:
            hi = mid
        else:
            lo = mid
    assert n_global(hi - 8) > 0
    infos = {w: _check_levels(gpu, small_db, oracle_small, prm, plan, monkeypatch, {"CTTS_GPU_WINDOW": str(w)}, f"window {w}")
             for w in (hi - 8, hi)}
    monkeypatch.delenv("CTTS_GPU_WINDOW")
    a, b = infos[hi - 8]["2"], infos[hi]["2"]
    assert a.n_global_tasks > 0 and b.n_global_tasks == 0
    assert a.n_canon_tasks > 0 and a.n_reuse_tasks > 0, (a.n_canon_tasks, a.n_reuse_tasks)
    assert (a.n_canon_tasks, a.n_dedup_tasks, a.n_source_tasks, a.n_reuse_tasks) == \
        (b.n_canon_tasks, b.n_dedup_tasks, b.n_source_tasks, b.n_reuse_tasks)
