"""Seeded generators of constructed voices that drive the back end's rare decision paths.

The harmonic-pulse voice of voicedb.synth_unit_pcm never reaches them: its units are 2 650-7 708 samples
long, always clearly voiced or unvoiced, never silent for a whole crossfade, never at full scale.  Each
family here builds a small voice.db whose units sit on one kind of edge, the texts that join them, and the
config / assembly-parameter changes it needs:

  A  short units       unit lengths at and around every length threshold of the assembly code
  B  pitch             unit heads and buffer tails whose pitch decision is within eps of a bound
  C  wsola             near-periodic units whose competing WSOLA candidates sweep the tier bands
  D  tiny stretch      pre-stretch lengths around one and two WSOLA frames, and all-zero ones
  E  amplitude         full scale, rms below 1, gain clamps, large DC
  F  trim              silent runs of min_sil - 1 .. min_sil + 1 samples at all 8 grid residues,
                       47 .. 64 cuttable runs in a region (inside and beyond the trim's candidate
                       pre-pass), a negative silence threshold

Every family goes through the front end.  Units are named by syllables (consonant + vowel, or one
vowel), so a word is parsed in exactly one way and the crossfade of a join is set by the class of the
next unit's first letter (the previous unit always ends in a vowel): plosive, fricative, other
consonant or vowel.  The builders check that every planned utterance holds the intended units.

The parity tests (test_gpu_edges.py) compare the CUDA path with the oracle (oracle/ctts_oracle.c).
At these edges the oracle is trusted by its construction: it restates the reference line by line
(same operand types, same order, no FMA), and where the reference tree is present test_oracle.py
compares its stage functions with the reference's.  An edge the reference handles in a way the
oracle does not restate would go unnoticed here.
"""
from __future__ import annotations

import copy
import ctypes as C
from dataclasses import dataclass, field

import numpy as np

import harness as H

F = H.front
SR = 22050

VOWELS = list("aeiou") + list("áéíóúâêôãõ")
CLASS_CONSONANTS = {"plosive": "pbtdgk", "fricative": "fvzjx", "other": "mnlhw"}  # no r, s: rewritten by the rules
WSOLA_SPEEDS = [0.5, 0.75, 1.5, 2.0, 0.6180339, 1.2345678, 1.8765432]


def ms_to_samples(ms: float) -> int:
    """(size_t)(ms * 22050 / 1000.0f) in float arithmetic, as the front end and the reference convert."""
    return int(np.float32(np.float32(ms) * np.float32(SR)) / np.float32(1000.0))


def join_xf(cfg, cls: str) -> int:
    """Crossfade of a join from a unit ending in a vowel into a unit of class `cls` (get_adaptive_crossfade)."""
    base = np.float32(cfg.crossfade_ms)
    ms = {"plosive": base * np.float32(0.2), "fricative": base * np.float32(0.4),
          "vowel": np.float32(cfg.crossfade_vowel_ms),
          "other": base * np.float32(cfg.vowel_to_consonant_factor)}[cls]
    return ms_to_samples(float(ms))


class Names:
    """Unique unit names of a crossfade class, in a fixed order."""

    def __init__(self):
        self._it = {c: iter([k + v for v in VOWELS for k in ks]) for c, ks in CLASS_CONSONANTS.items()}
        self._it["vowel"] = iter(VOWELS)

    def take(self, cls: str) -> str:
        return next(self._it[cls])


@dataclass
class Family:
    name: str
    units: list                    # (text, int16 pcm) for voicedb.build_voice_db
    words: list                    # per utterance: list of words, a word = list of unit names
    speeds: list
    config: object
    params: dict = field(default_factory=dict)   # assembly-parameter overrides (ctts_assembly_params fields)
    info: dict = field(default_factory=dict)     # what the witnesses need to know about the construction
    _cache: dict = field(default_factory=dict, repr=False)

    @property
    def texts(self) -> list:
        return [" ".join("".join(w) for w in ws) for ws in self.words]

    @property
    def db(self) -> bytes:
        if "db" not in self._cache:
            self._cache["db"] = H.voicedb.build_voice_db(self.units)
        return self._cache["db"]

    def front(self):
        if "front" not in self._cache:
            self._cache["front"] = F.Front(self.db, self.config, H.NORM_CSV)
        return self._cache["front"]

    def oracle(self):
        if "oracle" not in self._cache:
            self._cache["oracle"] = H.Oracle(self.db)
        return self._cache["oracle"]

    def prm(self):
        p = copy.copy(self.front().params())
        for k, v in self.params.items():
            setattr(p, k, v)
        return p

    def unit_index(self) -> dict:
        vdb = H.voicedb.parse_voice_db(self.db)
        return {vdb.unit_text(i): i for i in range(vdb.unit_count)}

    def unit_lengths(self) -> np.ndarray:
        return H.voicedb.parse_voice_db(self.db).index["sample_count"].astype(np.int64)

    def plan(self):
        """The batch plan, checked: every utterance holds exactly the intended units, in order."""
        if "plan" not in self._cache:
            plan = self.front().plan(self.texts, self.speeds)
            idx = self.unit_index()
            for u, ws in enumerate(self.words):
                ops = plan.utt_ops(u)
                got = ops["a"][ops["kind"] == F.OP_UNIT].tolist()
                want = [idx[H.voicedb.normalize_text(n)] for w in ws for n in w]
                assert got == want, f"{self.name}: utterance {u} {self.texts[u]!r} planned as other units"
                assert plan.missing[u] == 0
            self._cache["plan"] = plan
        return self._cache["plan"]

    def expected(self):
        """The oracle's PCM of every utterance."""
        if "want" not in self._cache:
            prm, plan, orc = self.prm(), self.plan(), self.oracle()
            self._cache["want"] = [orc.synth(prm, plan.utt_ops(u), float(plan.speed[u]))[0] for u in range(plan.n_utts)]
        return self._cache["want"]


def harmonic(rng, n: int, f0: float | None = None, peak: float | None = None) -> np.ndarray:
    """A voiced unit of exactly n samples: 6 harmonics, a little DC and noise."""
    f0 = rng.uniform(100.0, 180.0) if f0 is None else f0
    peak = rng.uniform(3000.0, 12000.0) if peak is None else peak
    t = np.arange(n) / SR
    x = sum(np.sin(2 * np.pi * h * f0 * t + rng.uniform(0, 6.28)) / h for h in range(1, 7))
    x = peak * x / 2.5 + rng.uniform(-150, 150) + rng.normal(0, 20, n)
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


def periodic(rng, n: int, period: int, amp: float = 9000.0) -> np.ndarray:
    """A seeded random pattern of `period` samples, tiled (float64)."""
    pat = rng.uniform(-amp, amp, period)
    return np.tile(pat, n // period + 1)[:n]


def i16(x) -> np.ndarray:
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


# ---------------------------------------------------------------------------------- oracle helpers

def normalized(x: np.ndarray, target: float = 3000.0) -> np.ndarray:
    """normalize_rms as the oracle computes it (ctts.c:1709)."""
    y = np.ascontiguousarray(x, dtype=np.int16).copy()
    H.oracle_lib().ctts_oracle_normalize_rms(y.ctypes.data, len(y), C.c_float(target))
    return y


def dc_removed(x: np.ndarray) -> np.ndarray:
    y = np.ascontiguousarray(x, dtype=np.int16).copy()
    H.oracle_lib().ctts_oracle_remove_dc(y.ctypes.data, len(y))
    return y


def oracle_lag(s: np.ndarray) -> int:
    """The oracle's estimate_pitch of s as a lag (0 = unvoiced)."""
    s = np.ascontiguousarray(s, dtype=np.int16)
    f = H.oracle_lib().ctts_oracle_estimate_pitch(s.ctypes.data, len(s))
    return int(round(SR / f)) if f > 0 else 0


def pitch_scores(s: np.ndarray) -> dict:
    """estimate_pitch's normalized correlation of every lag, in float64 (ctts.c:1899)."""
    n = len(s)
    hi = min(SR // 80, n // 2)
    ln = min(SR // 100, n - hi)
    x = s.astype(np.float64)
    a = x[:ln]
    e1 = a @ a
    out = {}
    for lag in range(SR // 400, hi + 1):
        b = x[lag:lag + ln]
        den = np.sqrt(e1 * (b @ b))
        out[lag] = (a @ b) / den if den > 0 else 0.0
    return out


def tail_lag_for(p: int) -> int:
    """A lag Q for the other side of a join such that the pitch ratio Q / p falls where the head is
    really resampled (ratio in (1.15, 1.25] or [0.834, 0.85)): the decision changes the PCM."""
    q = int(round(1.2 * p))
    return q if q <= SR // 80 else int(round(0.84 * p))


def bisect(make, decide, lo: float = 0.0, hi: float = 1.0, steps: int = 48):
    """make(w) -> int16 unit; decide(unit) -> answer.  Returns the two units one bisection step apart
    whose answers differ (None if the answers at lo and hi agree)."""
    ulo, uhi = make(lo), make(hi)
    alo, ahi = decide(ulo), decide(uhi)
    if alo == ahi:
        return None
    for _ in range(steps):
        mid = 0.5 * (lo + hi)
        um = make(mid)
        am = decide(um)
        if np.array_equal(um, ulo) or np.array_equal(um, uhi):
            break
        if am == alo:
            lo, ulo = mid, um
        else:
            hi, uhi, ahi = mid, um, am
    return ulo, uhi


# ---------------------------------------------------------------------------------- A: short units

A_LENGTHS = [0, 1, 7, 8, 9, 15, 99, 100, 101, 199, 200, 201, 255, 256, 257,
             439, 440, 441, 495, 496, 497, 549, 550, 551]
XF_CLASSES = ["plosive", "fricative", "other", "vowel"]


def family_short_units(seed: int = 11) -> Family:
    rng = np.random.default_rng(seed)
    cfg = H.shipped_config()
    names = Names()
    units, short = [], []
    for cls in ("plosive", "fricative", "other"):
        for n in A_LENGTHS:
            nm = names.take(cls)
            units.append((nm, harmonic(rng, n)))
            short.append(nm)
    for n in (0, 1, 8, 100, 200, 256, 441, 550):       # vowel names are scarce
        nm = names.take("vowel")
        units.append((nm, harmonic(rng, n)))
        short.append(nm)
    xf_lengths = {}
    for cls in XF_CLASSES:
        xf = join_xf(cfg, cls)
        xf_lengths[cls] = [xf - 1, xf, xf + 1, 2 * xf - 1, 2 * xf + 1]
        for n in xf_lengths[cls]:
            nm = names.take(cls)
            units.append((nm, harmonic(rng, n)))
            short.append(nm)
    longs = []
    for cls in XF_CLASSES:
        nm = names.take(cls)
        units.append((nm, harmonic(rng, int(rng.integers(4000, 6000)))))
        longs.append(nm)
    tiny = [nm for nm, pcm in units if len(pcm) < 16]
    words = []
    for k, u in enumerate(short):
        L = longs[k % 4]
        s = tiny[k % len(tiny)]
        first = [[u], [u, L]][k % 2]        # u is the first unit of the utterance
        ws = [[u] if k % 2 else [u, L], [L, u], [s, u, L], [s, s, u]]
        words.append([first] + [ws[i] for i in rng.permutation(len(ws))])
    for _ in range(24):   # words made only of short units, the first unit of the utterance short too
        words.append([list(rng.choice(short, size=int(rng.integers(1, 6)))) for _ in range(int(rng.integers(1, 4)))])
    speeds = [1.0] * len(words)
    for k in range(0, len(words), 9):
        speeds[k] = 1.3
    return Family("short_units", units, words, speeds, cfg,
                  info={"short": short, "longs": longs, "xf_lengths": xf_lengths})


# ---------------------------------------------------------------------------------- B: pitch decisions

B_HEAD_LENGTHS = [420, 560, 880, 1100, 1500]   # n / 2 < 2 * xf for every crossfade class


def _head_decision(n):
    reg = n // 2
    return lambda unit: oracle_lag(normalized(unit)[:reg])


def family_pitch(seed: int = 12) -> Family:
    """Joins `T H` (one word; T first after a word boundary): the head H of n samples is analysed over
    n / 2 samples at every join; T is a clean periodic unit whose lag makes the decision matter.
    Tail-side cases swap the roles: T's last samples are tuned on what the buffer will hold."""
    rng = np.random.default_rng(seed)
    cfg = H.shipped_config()
    names = Names()
    units, words, info = [], [], {"heads": [], "tails": [], "thr": [], "tie": [], "degenerate": [], "noise": []}
    tails = {}

    def tail_unit(q):
        if q not in tails:
            nm = names.take("other")
            units.append((nm, i16(periodic(rng, 5000, q, 6000) + rng.normal(0, 5, 5000))))
            tails[q] = nm
        return tails[q]

    def add_head(kind, pcm, n, group):
        nm = names.take("plosive")
        units.append((nm, pcm))
        lag = _head_decision(n)(pcm)
        t = tail_unit(tail_lag_for(lag) if lag else 150)
        words.append([[t, nm]])
        info["heads"].append(nm)
        info[kind].append((group, nm, n))

    noise_seed = rng.integers(1 << 30)
    # threshold pairs: periodic component + seeded noise, mixing weight bisected across 0.3
    for g, n in enumerate(B_HEAD_LENGTHS):
        p = int(rng.integers(60, min(n // 4, 270)))
        per = periodic(np.random.default_rng(noise_seed + g), n, p, 3000)
        for k in range(20):     # a noise whose own best score stays below 0.3
            nz = np.random.default_rng(noise_seed + 100 * k + g).normal(0, 3000, n)
            pair = bisect(lambda w: i16(w * per + nz), _head_decision(n))
            if pair is not None:
                break
        assert pair is not None, ("threshold", n)
        for pcm in pair:
            add_head("thr", pcm, n, g)
    # near-tie pairs: two periodic components, weight bisected across the arg max flip
    for g, (p1, p2, n) in enumerate(((55, 56, 420), (100, 104, 600), (150, 160, 1000), (274, 275, 1500), (55, 56, 880))):
        r = np.random.default_rng(noise_seed + 200 + g)
        c1, c2 = periodic(r, n, p1, 3000), periodic(r, n, p2, 3000)
        nz = r.normal(0, 30, n)
        pair = bisect(lambda w: i16(w * c1 + (1 - w) * c2 + nz), _head_decision(n))
        assert pair is not None, ("tie", p1, p2)
        for pcm in pair:
            add_head("tie", pcm, n, g)
    # degenerate heads: more than 64 lags score within 2e-4 of the maximum
    for g, n in enumerate((600, 880, 1500)):      # (420 samples analyse only 51 lags)
        t = np.arange(n)
        add_head("degenerate", np.full(n, 1234, np.int16), n, g)
        add_head("degenerate", i16(2000 + 300 * t / n), n, g)
        add_head("degenerate", i16(4000 * np.sin(2 * np.pi * 3.0 * t / SR + 1.3)), n, g)
    # unvoiced heads
    for g, n in enumerate(B_HEAD_LENGTHS):
        add_head("noise", i16(rng.normal(0, 2500, n)), n, g)
    # tail side: T ends in a tuned segment of reg samples, H is a long clean head of lag P
    for g, reg in enumerate((210, 280, 440, 600)):
        n_t = 3000
        p = int(rng.integers(60, min(reg // 2, 270)))
        head_n = 2 * reg      # reg = min(2 xf, count / 2, n / 2) = n / 2
        per = periodic(np.random.default_rng(noise_seed + 300 + g), n_t, p, 3000)
        body = i16(periodic(np.random.default_rng(noise_seed + 500 + g), n_t, 97, 3000))

        def make(w):
            x = body.astype(np.float64)
            x[-reg:] = w * per[-reg:] + nz[-reg:]
            return i16(x)

        # the buffer's last reg samples: T normalized, then DC-removed (T is first in its word)
        pair = None
        for k in range(20):
            nz = np.random.default_rng(noise_seed + 400 + 100 * k + g).normal(0, 3000, n_t)
            pair = bisect(make, lambda unit: oracle_lag(dc_removed(normalized(unit))[-reg:]))
            if pair is not None:
                break
        assert pair is not None, ("tail threshold", reg)
        q = tail_lag_for(p)
        hn = names.take("plosive")
        units.append((hn, i16(periodic(np.random.default_rng(noise_seed + 600 + g), head_n, q, 5000))))
        for pcm in pair:
            nm = names.take("other")
            units.append((nm, pcm))
            words.append([[nm, hn]])
            info["tails"].append((g, nm, hn, reg))
    speeds = [1.0] * len(words)
    return Family("pitch", units, words, speeds, cfg, info=info)


# ---------------------------------------------------------------------------------- C: WSOLA

C_NOISE = [0, 1, 2, 4, 8, 16, 32, 64, 128, 256]


def family_wsola(seed: int = 13) -> Family:
    rng = np.random.default_rng(seed)
    cfg = H.shipped_config()
    cfg.max_pitch_change = 0.0      # no intonation contour: it would resample the periods away
    names = Names()
    units, words, speeds = [], [], []
    info = {"noiseless": []}
    k = 0
    for period in (64, 96, 61, 99):     # multiples of 4: a coarse candidate competes; else only a fine one
        pat = rng.uniform(-5000, 5000, period)
        for amp in C_NOISE:
            n = int(rng.integers(5000, 7000))
            x = np.tile(pat, n // period + 1)[:n] + (rng.normal(0, amp, n) if amp else 0.0)
            nm = names.take(["plosive", "fricative", "other"][k % 3])
            units.append((nm, i16(x)))
            if amp == 0:
                info["noiseless"].append(nm)
            for sp in (WSOLA_SPEEDS[k % 4], WSOLA_SPEEDS[4 + k % 3]):
                words.append([[nm]])
                speeds.append(sp)
            k += 1
    for gap in ((50, 90), (80, 150), (100, 101)):      # sparse impulse trains
        n = 6000
        x = np.zeros(n)
        at = 0
        while True:
            at += int(rng.integers(gap[0], gap[1]))
            if at >= n:
                break
            x[at] = rng.choice([-1, 1]) * rng.uniform(2000, 20000)
        nm = names.take("other")
        units.append((nm, i16(x)))
        for sp in WSOLA_SPEEDS:
            words.append([[nm]])
            speeds.append(sp)
    return Family("wsola", units, words, speeds, cfg, info=info)


# ---------------------------------------------------------------------------------- D: tiny stretch

D_LENGTHS = [0, 1, 255, 511, 512, 513, 639, 640, 641, 767, 768, 769]


def family_tiny_stretch(seed: int = 14) -> Family:
    """One unit per utterance, no pause, fades or trim: the pre-stretch length is the unit's length."""
    rng = np.random.default_rng(seed)
    cfg = H.shipped_config()
    cfg.word_pause_ms = 0.0
    cfg.fade_in_ms = 0.0
    cfg.fade_out_ms = 0.0
    cfg.remove_word_silence = 0
    names = Names()
    units, words, speeds = [], [], []
    for zero in (False, True):
        for n in D_LENGTHS:
            nm = names.take("other")
            units.append((nm, np.zeros(n, np.int16) if zero else harmonic(rng, n)))
            for sp in WSOLA_SPEEDS:
                words.append([[nm]])
                speeds.append(sp)
    return Family("tiny_stretch", units, words, speeds, cfg, params={"fade_in_samples": 0})


# ---------------------------------------------------------------------------------- E: amplitude extremes

def _amplitude_units(rng):
    n = 3000
    t = np.arange(n)
    sq = np.where((t // 40) % 2 == 0, 32767, -32768).astype(np.int16)
    clipped = i16(60000 * np.sin(2 * np.pi * 150 * t / SR))
    tiny = np.zeros(n, np.int16)
    tiny[::97] = 1                                           # rms < 1: no gain
    trit = rng.choice(np.array([-1, 0, 0, 1], np.int16), n)  # values in {-1, 0, 1}, rms < 1
    g3 = np.where((t // 30) % 2 == 0, 1000, -1000).astype(np.int16)       # rms 1000: gain exactly 3.0
    g01 = np.where((t // 30) % 2 == 0, 30000, -30000).astype(np.int16)    # rms 30000: gain exactly 0.1
    over = np.where((t // 25) % 2 == 0, 200, -200).astype(np.int16)       # gain 15 -> clamped at 3.0
    under = np.where((t // 25) % 2 == 0, 32767, -32767).astype(np.int16)  # gain 0.09 -> clamped at 0.1
    neg = np.zeros(n, np.int16)
    neg[::53] = -32768                                       # only -32768 is non-zero
    dcp = i16(20000 + 3000 * np.sin(2 * np.pi * 120 * t / SR))
    dcn = i16(-20000 + 3000 * np.sin(2 * np.pi * 130 * t / SR))
    spikes = np.full(n, -20000, np.int16)
    spikes[::17] = 32767                                     # x - dc leaves int16: sub_dc saturates
    boost = np.zeros(n, np.int16)
    boost[::300] = 20000
    boost[150::300] = -20000                                 # rms 1155: gain 2.6 saturates the spikes
    return [sq, clipped, boost, tiny, trit, g3, g01, over, under, neg, dcp, dcn, spikes, harmonic(rng, 4000)]


def family_amplitude(seed: int = 15, target_rms: float = 3000.0) -> Family:
    rng = np.random.default_rng(seed)
    cfg = H.shipped_config()
    names = Names()
    units = [(names.take(["plosive", "other", "vowel"][k % 3]), pcm) for k, pcm in enumerate(_amplitude_units(rng))]
    nm = [u[0] for u in units]
    words = [[[a]] for a in nm]
    for k in range(40):   # joins between extremes (crossfade mixes clamp), several words
        words.append([list(rng.choice(nm, size=int(rng.integers(1, 4)))) for _ in range(int(rng.integers(1, 4)))])
    speeds = [1.0 if k % 3 else 1.5 for k in range(len(words))]
    return Family(f"amplitude_rms{int(target_rms)}", units, words, speeds, cfg, params={"target_rms": target_rms})


# ---------------------------------------------------------------------------------- F: trim edges

F_PEAK = 10000


TRIM_MAX_CAND = 48       # cuttable runs the trim's candidate pre-pass lists (asm_word.cuh)
SCR_WORDS = 3776         # shared scratch words of the assembly kernel (asm_common.cuh)


def trim_prepass_runs(n: int, min_sil: int) -> bool:
    """Whether the trim of an n-sample region with limit >= 0 looks for cuttable runs on the per-vector
    maxima first (asm_word.cuh: have_vm, min_sil >= 127, room for the candidate list), whatever the
    region's phase on the 8-sample grid."""
    wn = (n + 31) >> 5
    gvec = (7 + n + 7) >> 3
    have_vm = 2 * wn + (gvec + 1) // 2 + 2 <= SCR_WORDS
    sv_at = 2 * wn + (gvec + 1) // 2 + 1
    return have_vm and min_sil >= 15 + 8 * 14 and sv_at + (gvec + 31) // 32 + 2 + 2 * TRIM_MAX_CAND <= SCR_WORDS


def family_trim(seed: int = 16, negative: bool = False, min_silence_ms: float | None = None) -> Family:
    """Assembly without RMS gain, DC removal or fade-in, so the samples of a unit body reach the trim
    unchanged and the silence limit is f2s(F_PEAK * threshold).  Words [P_k S]: the preceding unit's
    length moves S's silent runs through the 8 residues of the 8-sample grid.  Words of one unit with
    47, 48, 49 and 64 cuttable runs: with short runs (min_silence_ms 10) they fit the trim's candidate
    pre-pass, which lists at most 48 runs and falls back to the full mask beyond."""
    rng = np.random.default_rng(seed)
    cfg = H.shipped_config()
    if negative:
        cfg.silence_threshold = -0.05   # limit < 0: only -32768 counts as silent
    if min_silence_ms is not None:
        cfg.min_silence_ms = min_silence_ms
    names = Names()
    fr = F.Front(H.voicedb.build_voice_db([("a", np.zeros(1, np.int16))]), cfg, H.NORM_CSV)
    prm = fr.params()
    min_sil = int(prm.min_silence_samples)
    limit = int(np.float32(F_PEAK) * np.float32(prm.silence_threshold))

    def loud(n):
        return np.where((np.arange(n) // 7) % 2 == 0, F_PEAK, -F_PEAK).astype(np.int16)

    fills = {"zero": 0, "neg": -32768, "limit": limit, "limit+1": limit + 1, "-limit": -limit}
    units, words, S = [], [], []
    for fname, v in fills.items():
        parts = [loud(600)]
        for run in (min_sil - 1, min_sil, min_sil + 1):
            parts += [np.full(run, v, np.int16), loud(100)]
        nm = names.take("plosive")
        units.append((nm, np.concatenate(parts)))
        S.append(nm)
    P = []
    for k in range(8):
        nm = names.take("other")
        units.append((nm, (loud(2000 + k) // 3).astype(np.int16)))
        P.append(nm)
    for s in S:
        for k in range(8):
            words.append([[P[k], s]])
    # 47 .. 64 cuttable runs in one word, and more than 48 in a region beyond the shared-memory window
    many = []
    for k, n_runs in enumerate((47, 48, 49, 64, 64)):
        parts = [loud(400)]
        for _ in range(n_runs):
            parts += [np.full(int(rng.integers(min_sil, min_sil + 60)), [0, -32768][k % 2], np.int16), loud(int(rng.integers(20, 60)))]
        nm = names.take("fricative")
        units.append((nm, np.concatenate(parts)))
        many.append(nm)
    words += [[[m]] for m in many[:4]]
    words.append([[P[1], many[4]], [many[2]]])
    words.append([many])
    speeds = [1.0] * len(words)
    speeds[-1] = 1.25
    name = "trim_negative" if negative else "trim" if min_silence_ms is None else "trim_short_runs"
    return Family(name, units, words, speeds, cfg,
                  params={"target_rms": 0.0, "remove_dc_offset": 0, "fade_in_samples": 0},
                  info={"limit": limit, "min_sil": min_sil, "S": S, "P": P, "many": many})


FAMILIES = {
    "short_units": family_short_units,
    "pitch": family_pitch,
    "wsola": family_wsola,
    "tiny_stretch": family_tiny_stretch,
    "amplitude_rms0": lambda: family_amplitude(target_rms=0.0),
    "amplitude_rms3000": lambda: family_amplitude(target_rms=3000.0),
    "trim": family_trim,
    "trim_short_runs": lambda: family_trim(min_silence_ms=10.0),
    "trim_negative": lambda: family_trim(negative=True),
}

_built: dict = {}


def family(name: str) -> Family:
    if name not in _built:
        _built[name] = FAMILIES[name]()
    return _built[name]
