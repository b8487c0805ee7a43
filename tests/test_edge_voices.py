"""CPU witnesses of the constructed voices (edge_voices.py): each family really sits on the edge it is
built for, proved from the plans, the voices' units and the oracle's buffers.  The GPU parity of the
same families is in test_gpu_edges.py."""
import ctypes as C

import numpy as np
import pytest

import edge_voices as E

F = E.F


def _unit_ops(fam):
    """Per utterance: list of (unit length, op b, after_boundary, unit name) in op order, words split."""
    plan, lengths = fam.plan(), fam.unit_lengths()
    out = []
    for u in range(plan.n_utts):
        words, cur = [], []
        for op in plan.utt_ops(u):
            if op["kind"] == F.OP_UNIT:
                if op["flags"] & F.UNIT_AFTER_BOUNDARY and cur:
                    words.append(cur)
                    cur = []
                cur.append((int(lengths[op["a"]]), int(op["b"]), bool(op["flags"] & F.UNIT_AFTER_BOUNDARY)))
        if cur:
            words.append(cur)
        out.append(words)
    return out


def _abs16(x):
    x = x.astype(np.int32)
    a = np.where(x > 0, x, -x)
    return np.where(a == 32768, -32768, a)


def _runs(mask):
    """(start, length) of the True runs of a boolean array."""
    d = np.diff(np.concatenate([[0], mask.astype(np.int8), [0]]))
    s, e = np.nonzero(d == 1)[0], np.nonzero(d == -1)[0]
    return list(zip(s.tolist(), (e - s).tolist()))


def test_short_units_reach_every_length_threshold():
    fam = E.family("short_units")
    utts = _unit_ops(fam)
    joins = [(w[i - 1][0], n, b) for ws in utts for w in ws for i, (n, b, _) in enumerate(w) if i > 0]
    used = {n for ws in utts for w in ws for (n, _, _) in w}
    assert set(E.A_LENGTHS) <= used
    for cls, lens in fam.info["xf_lengths"].items():
        xf = E.join_xf(fam.config, cls)
        for n in lens:      # xf - 1, xf, xf + 1, 2 xf - 1, 2 xf + 1, joined with that crossfade
            assert any(m == n and b == xf for _, m, b in joins), (cls, n, xf)
    for n in E.A_LENGTHS:
        assert any(ws[0][0][0] == n for ws in utts), f"{n} never first in an utterance"
        assert any(p < 16 and m == n for p, m, _ in joins), f"{n} never after a short predecessor"
        assert any(p == n and m >= 4000 for p, m, _ in joins), f"{n} never before a long unit"
    # one-letter words, and words made only of short units
    names = {nm for ws in fam.words for w in ws for nm in w if len(w) == 1}
    assert any(len(nm) == 1 for nm in names)
    assert sum(all(n < 600 for n, _, _ in w) and len(w) >= 3 for ws in utts for w in ws) >= 10


def _scored(seg):
    sc = E.pitch_scores(seg)
    return sc, max(sc.values())


def test_pitch_heads_sit_on_the_decision_bounds():
    fam = E.family("pitch")
    pcm = dict(fam.units)
    eps = 1e-4
    thr = {}
    for g, nm, n in fam.info["thr"]:
        seg = E.normalized(pcm[nm])[:n // 2]
        _, mx = _scored(seg)
        assert abs(mx - 0.3) < 5e-5, (nm, mx)
        thr.setdefault(g, []).append(E.oracle_lag(seg))
    assert len(thr) == len(E.B_HEAD_LENGTHS)
    assert all(len(v) == 2 and (v[0] == 0) != (v[1] == 0) for v in thr.values()), thr
    ties = {}
    for g, nm, n in fam.info["tie"]:
        seg = E.normalized(pcm[nm])[:n // 2]
        ties.setdefault(g, []).append((E.oracle_lag(seg), seg))
    for g, ((l1, s1), (l2, s2)) in ties.items():
        assert l1 and l2 and l1 != l2, (g, l1, l2)
        for seg in (s1, s2):
            sc, _ = _scored(seg)
            assert abs(sc[l1] - sc[l2]) < eps, (g, l1, l2, sc[l1] - sc[l2])
    assert {55, 56, 274, 275} <= {l for v in ties.values() for l, _ in v}
    for g, nm, n in fam.info["degenerate"]:
        sc, mx = _scored(E.normalized(pcm[nm])[:n // 2])
        assert sum(v >= mx - eps for v in sc.values()) > 64, nm
    for g, nm, n in fam.info["noise"]:
        seg = E.normalized(pcm[nm])[:n // 2]
        assert E.oracle_lag(seg) == 0 and _scored(seg)[1] < 0.3 - eps
    regs = [n // 2 for k in ("thr", "tie", "degenerate", "noise") for _, _, n in fam.info[k]]
    assert min(regs) < 440 and any(r < 550 for r in regs) and max(regs) >= 550
    # the analysis length at every join is n / 2 of the head: 2 xf and count / 2 are larger
    plan, lengths = fam.plan(), fam.unit_lengths()
    for u in range(plan.n_utts):
        ops = plan.utt_ops(u)
        t, h = ops[ops["kind"] == F.OP_UNIT]
        assert 2 * int(h["b"]) > int(lengths[h["a"]]) // 2 and lengths[t["a"]] >= lengths[h["a"]]


def test_pitch_tails_sit_on_the_threshold_in_the_oracle_buffer():
    fam = E.family("pitch")
    plan, prm, orc = fam.plan(), fam.prm(), fam.oracle()
    index = {nm: k for k, nm in enumerate(fam.texts)}
    got = {}
    for g, nm, hn, reg in fam.info["tails"]:
        ops = plan.utt_ops(index[nm + hn])
        k_head = int(np.nonzero(ops["kind"] == F.OP_UNIT)[0][1])
        _, _, pre = orc.synth(prm, ops[:k_head], 1.0, want_pre=True)     # the buffer the join sees
        seg = pre[-reg:]
        _, mx = _scored(seg)
        assert abs(mx - 0.3) < 5e-5, (nm, mx)
        got.setdefault(g, []).append(E.oracle_lag(seg))
    assert len(got) == 4 and all((v[0] == 0) != (v[1] == 0) for v in got.values()), got


def _walk(orc_lib, pre):
    """The reference's WSOLA chain on a pre-stretch buffer: offsets of frames 1.. and, for each, the best
    1 - rho (float64) among the candidates other than the previous offset."""
    n = len(pre)
    x = pre.astype(np.float64)
    pos_prev, offs, gaps, moved = 0, [0], [], False
    nominal = 128
    while nominal + 512 <= n:
        prev = np.ascontiguousarray(pre[pos_prev:pos_prev + 512])
        off = orc_lib.ctts_oracle_wsola_offset(pre.ctypes.data, n, prev.ctypes.data, nominal)
        t = x[pos_prev + 128:pos_prev + 512]
        h = offs[-1]
        cand = set(range(-128, 129, 4)) | set(range(max(h - 3, -128), min(h + 3, 128) + 1))
        best = np.inf
        tt = t @ t
        for c in cand - {h}:
            p = nominal + c
            if p < 0 or p + 512 > n:
                continue
            w = x[p:p + 384]
            den = np.sqrt((w @ w) * tt)
            if den >= 1.0:
                best = min(best, 1.0 - (w @ t) / den)
        if tt > 0:
            gaps.append(best)
            moved |= off != h
        offs.append(off)
        pos = nominal + off
        pos_prev = min(pos, n - 512)
        nominal += 128
    return gaps, moved


def test_wsola_candidates_sweep_every_tier_band():
    fam = E.family("wsola")
    plan, prm, orc = fam.plan(), fam.prm(), fam.oracle()
    L = E.H.oracle_lib()
    L.ctts_oracle_wsola_offset.restype = C.c_int
    gaps, moved = [], 0
    for u in range(plan.n_utts):
        _, _, pre = orc.synth(prm, plan.utt_ops(u), float(plan.speed[u]), want_pre=True)
        g, m = _walk(L, np.ascontiguousarray(pre))
        gaps += g
        moved += m
    gaps = np.array(gaps)
    bands = [(0.0, 6e-8), (6e-8, 2e-5), (2e-5, 1e-4), (1e-4, 1.25e-3)]
    counts = [int(((gaps >= lo) & (gaps < hi)).sum()) for lo, hi in bands]
    assert all(c >= 20 for c in counts), counts
    assert moved >= 1
    assert {float(np.float32(s)) for s in E.WSOLA_SPEEDS} <= set(plan.speed.tolist())


def test_tiny_stretch_lengths_and_empty_outputs():
    fam = E.family("tiny_stretch")
    plan, prm, orc = fam.plan(), fam.prm(), fam.oracle()
    seen = {}
    empty = 0
    for u in range(plan.n_utts):
        pcm, st = orc.synth(prm, plan.utt_ops(u), float(plan.speed[u]))
        seen.setdefault(float(plan.speed[u]), set()).add(int(st.pre_count))
        empty += len(pcm) == 0
    assert len(seen) == len(E.WSOLA_SPEEDS)
    for sp, pres in seen.items():
        assert set(E.D_LENGTHS) <= pres, (sp, sorted(pres))
    assert empty >= len(E.D_LENGTHS) * len(E.WSOLA_SPEEDS)      # every all-zero utterance, at least


def test_amplitude_extremes_reach_full_scale_and_the_gain_clamps():
    for name in ("amplitude_rms0", "amplitude_rms3000"):
        fam = E.family(name)
        plan, prm, orc = fam.plan(), fam.prm(), fam.oracle()
        lo = hi = 0
        for u in range(plan.n_utts):
            _, _, pre = orc.synth(prm, plan.utt_ops(u), 1.0, want_pre=True)
            lo += int((pre == -32768).sum())
            hi += int((pre == 32767).sum())
        assert lo > 0 and hi > 0, (name, lo, hi)
    fam = E.family("amplitude_rms0")      # (both variants share the units)
    L = E.H.oracle_lib()
    rms = [L.ctts_oracle_rms(np.ascontiguousarray(p).ctypes.data, len(p)) for _, p in fam.units]
    gains = [3000.0 / r for r in rms if r >= 1.0]
    assert any(r < 1.0 for r in rms)
    assert any(np.float32(g) == np.float32(3.0) for g in gains) and any(np.float32(3000.0) / np.float32(r) == np.float32(0.1) for r in rms)
    assert any(g > 3.0 for g in gains) and any(g < 0.1 for g in gains)
    pcm = [p for _, p in fam.units]
    assert any(set(np.unique(p).tolist()) <= {-1, 0, 1} for p in pcm)
    assert any(set(np.unique(p).tolist()) == {-32768, 0} for p in pcm)
    # DC removal saturates (raw units reach it unchanged when target_rms is 0)
    assert any(((p.astype(np.int64) - int(p.astype(np.int64).sum() // len(p))) > 32767).any() for p in pcm if len(p))


def _untrimmed_regions(fam):
    """The first word of every utterance as the trim sees it: the op prefix before its WORD_END."""
    plan, prm, orc = fam.plan(), fam.prm(), fam.oracle()
    out = []
    for u in range(plan.n_utts):
        ops = plan.utt_ops(u)
        k = int(np.nonzero(ops["kind"] == F.OP_WORD_END)[0][0])
        _, _, pre = orc.synth(prm, ops[:k], 1.0, want_pre=True)
        out.append(pre)
    return out


@pytest.mark.parametrize("name", ["trim", "trim_short_runs", "trim_negative"])
def test_trim_runs_at_min_silence_on_every_residue(name):
    fam = E.family(name)
    prm = fam.prm()
    min_sil = int(prm.min_silence_samples)
    assert min_sil == fam.info["min_sil"]
    starts = {min_sil - 1: set(), min_sil: set(), min_sil + 1: set()}
    most, longest, prepass = 0, 0, set()
    for reg in _untrimmed_regions(fam):
        a = _abs16(reg)
        peak = int(a.max())
        limit = int(np.float32(peak) * np.float32(prm.silence_threshold))
        runs = _runs(a <= limit)
        for s, n in runs:
            if n in starts:
                starts[n].add(s % 8)
        cut = sum(n >= min_sil for _, n in runs)
        most = max(most, cut)
        if cut > E.TRIM_MAX_CAND:
            longest = max(longest, len(reg))
        if limit >= 0 and E.trim_prepass_runs(len(reg), min_sil):
            prepass.add(cut)
        if name != "trim_negative":
            assert limit == fam.info["limit"] or len(reg) > 5000      # the words [P_k S]: F_PEAK sets it
        else:
            assert limit < 0 and all((reg[s:s + n] == -32768).all() for s, n in runs)
    assert all(len(v) == 8 for v in starts.values()), starts
    assert most > E.TRIM_MAX_CAND
    if name == "trim_short_runs":
        # regions the candidate pre-pass scans, with a full candidate list and with one run too many
        assert {47, 48, 49, 64} <= prepass, sorted(prepass)
    else:
        assert longest > 200000, longest      # beyond the shared-memory trim mask


@pytest.mark.parametrize("name", E.SIGNAL_FAMILIES)
def test_signal_families_deliver_their_samples(name):
    """The pass-through the loudness and FLAC signal tests rely on: the oracle's native output of every utterance is
    its signal bit for bit, the longest unit (6.3 minutes) included."""
    fam = E.signal_family(name)
    plan, prm, orc = fam.plan(), fam.prm(), fam.oracle()
    sig = fam.info["signals"]
    first = {}
    for u, ws in enumerate(fam.words):
        first.setdefault(ws[0][0], u)
    assert len(first) == len(fam.units)   # utterances of one signal share its unit: one of them stands for all
    for u in first.values():
        got = orc.synth(prm, plan.utt_ops(u), 1.0)[0]
        assert np.array_equal(got, sig[u]), f"{name}: utterance {u} ({len(sig[u])} samples) is not its signal"
