"""tests/edge_signals.py -- stimuli at the edges of the signal range, for parity tests of the whole chain.

signals.py feeds the chain what the BASELINE workloads carry: tones at 0.05 to 0.3 of full scale with noise in every sample
(SURVEY 6.2), so IIR states never go subnormal and the kernel's guarded paths are never taken.  The builders here go where
CUDA arithmetic and x86 part ways:

  silence       digital silence long enough that every IIR state decays through the subnormals to zero, on every mode,
                blanker and ALS on and off, one-rail silence, and a SAM bucket whose warps mix silent and live lanes
  tiny          float32 planes at 1e-39 (subnormal input), 1e-30, 1e-20, and amplitude sweeps across 2^-60 for the
                envelope's |I|^2+|Q|^2 (around 1e-9) and the SAM PLL's phase-detector operands (around 1e-18)
  full_scale    int16 square waves on the rails (with -32768), input gain 10 and above, output gains 0 / 3 / 1e5 / negative,
                AGC off on some rows: |audio| >= 256, int16 pcm that wraps, the x86 "indefinite" conversion
  large_float   float32 planes up to ~1e3
  clustered     blanker bursts at the ring positions the kernel special-cases, pairs of windows 0..12 samples apart,
                bursts across block boundaries and longer than a block, thresholds that blank every sample
  setter_edges  setters outside harness.fuzz_events' ranges, changed mid-stream

Each builder is a pure, seeded function and returns (I, Q, events) like signals.make; every row's mode, blanker, ALS and AGC
setting is stated in its events.  `*_check` functions next to them show on the oracle that a case does what it says.
"""
import numpy as np

import signals as S

N_BLOCK = 128
FS = S.FS
MODES = (S.LSB, S.USB, S.CW_LSB, S.CW_USB, S.AM, S.SAM, S.WSPR)
FILTER = {S.LSB: S.AUDIO_2700, S.USB: S.AUDIO_2700, S.CW_LSB: S.AUDIO_CW, S.CW_USB: S.AUDIO_CW, S.AM: S.AUDIO_AM,
          S.SAM: S.AUDIO_AM, S.WSPR: S.AUDIO_WSPR}
FLT_MIN = float(np.finfo(np.float32).tiny)  # smallest normal float32, 2^-126
TWO_M60 = 2.0 ** -60                        # lower end of the range the kernel's fast divisions take without a fallback
RAMP_DN = np.array([0.933, 0.750, 0.500, 0.250, 0.067, 0.0, 0.0], np.float32)  # the blanker's edge (C:637-644)


def row_events(row, mode, nb=False, als=False, agc=True, nb_db=10.0):
    """Every setting a row depends on, at block 0."""
    ev = [(row, 0, "setDemodMode", mode), (row, 0, "enableNoiseBlanker" if nb else "disableNoiseBlanker"),
          (row, 0, "setNoiseBlankerThresholdDb", nb_db)]
    ev += [(row, 0, "setAGCmode", S.AGC_MEDIUM)] if agc else [(row, 0, "disableAGC")]
    ev += [(row, 0, "enableAudioFilter"), (row, 0, "setAudioFilter", FILTER[mode])]
    if als:
        ev += [(row, 0, "enableALSfilter"), (row, 0, "setALSfilterNotch" if row % 2 else "setALSfilterPeak")]
    else:
        ev += [(row, 0, "disableALSfilter")]
    return ev + [(row, 0, "setMute", 0)]


def live(mode, row, ns, amp=0.2, sigma=0.01, seed=0):
    """A channel's complex IF signal: a tone (AM-modulated carrier for AM / SAM) at `amp` of full scale plus noise."""
    t = np.arange(ns, dtype=np.float64)
    w = 2.0 * np.pi / FS
    h = S.chash(0x7E, row, 1 + seed)
    if mode in (S.AM, S.SAM):
        df = 100.0 * S._unit(h) - 50.0
        x = amp * (1.0 + 0.5 * np.cos(w * 1000.0 * t)) * np.exp(1j * w * (6890.0 + df) * t)
    else:
        fa = (700.0 if mode in (S.CW_LSB, S.CW_USB) else 1500.0 if mode == S.WSPR else 400.0 + 1800.0 * S._unit(h))
        x = amp * np.exp(1j * (w * S._audio_to_if(mode, fa) * t + 2.0 * np.pi * S._unit(h >> 7)))
    rng = np.random.Generator(np.random.Philox(key=[0xED6E0000 + seed, row]))
    n = rng.standard_normal(2 * ns)
    return x + sigma * (n[0::2] + 1j * n[1::2])


def _quantise_rows(X):
    I = np.empty(X.shape, np.int16); Q = np.empty(X.shape, np.int16)
    for r in range(X.shape[0]):
        I[r], Q[r] = S.quantise(X[r])
    return I, Q


# ---------------------------------------------------------------------------------------------------------------- silence
def silence(sam_lanes=64, before=16, silent=200, after=16, seed=1):
    """Live signal, exact zeros for `silent` blocks (starting and ending anywhere in a block), live signal again, on every
    mode x blanker on/off x ALS on/off; one-rail silence on every mode (I = 0 on even rows, Q = 0 on odd ones); and a SAM
    bucket (blanker and ALS off) of `sam_lanes` channels whose every warp mixes lanes that never see a signal, lanes that
    stay live, lanes that fall silent at different blocks and lanes that come alive at different blocks.
    Returns (I, Q, events, layout); layout: dict(full=rows, one_rail=rows, sam=rows, modes=mode of every row)."""
    nblk = before + silent + after
    ns = nblk * N_BLOCK
    rows, ev = [], []
    for m in MODES:
        for nb in (0, 1):
            for als in (0, 1):
                rows.append((m, nb, als, "both"))
    for m in MODES:
        rows.append((m, m % 2, (m // 2) % 2, "I" if m % 2 == 0 else "Q"))
    n_full, n_rail = 4 * len(MODES), len(MODES)
    nch = len(rows) + sam_lanes
    X = np.empty((nch, ns), np.complex128)
    for r, (m, nb, als, rail) in enumerate(rows):
        x = live(m, r, ns, seed=seed)
        a = before * N_BLOCK + (r * 37) % N_BLOCK          # first silent sample: anywhere in the block, row 0 at a boundary
        z = (before + silent) * N_BLOCK + (r * 53) % N_BLOCK
        if rail == "both":
            x[a:z] = 0.0
        elif rail == "I":
            x[a:z] = 1j * x[a:z].imag
        else:
            x[a:z] = x[a:z].real
        X[r] = x
        ev += row_events(r, m, nb, als)
    for k in range(sam_lanes):
        r = len(rows) + k
        x = live(S.SAM, r, ns, amp=0.3, seed=seed)
        kind = k % 4
        if kind == 1:                       # never a signal
            x[:] = 0.0
        elif kind == 2:                     # falls silent at a block of its own, mid-block
            a = (4 + (k * 7) % (nblk - 8)) * N_BLOCK + (k * 29) % N_BLOCK
            x[a:] = 0.0
        elif kind == 3:                     # silent at first, alive from a block of its own
            x[:(2 + (k * 11) % (nblk - 4)) * N_BLOCK + (k * 41) % N_BLOCK] = 0.0
        X[r] = x
        ev += row_events(r, S.SAM)
    I, Q = _quantise_rows(X)
    layout = dict(full=list(range(n_full)), one_rail=list(range(n_full, n_full + n_rail)),
                  sam=list(range(len(rows), nch)), modes=[m for m, _, _, _ in rows] + [S.SAM] * sam_lanes)
    return I, Q, ev, layout


def subnormal_rows(audio):
    """Per row: the number of non-zero subnormal audio samples."""
    a = np.abs(audio)
    return np.count_nonzero((a > 0) & (a < FLT_MIN), axis=1)


def silence_check(o, layout):
    """Every mode produces non-zero subnormal audio, and the silent rows reach exact zero as well."""
    sub = subnormal_rows(o["audio"])
    modes = np.array(layout["modes"])
    for m in MODES:
        assert sub[modes == m].sum() > 0, "mode %d: no subnormal audio" % m
    full = layout["full"]
    assert np.count_nonzero(sub[full]) >= len(full) // 2, sub[full]
    assert np.any(o["audio"][full] == 0.0)
    # the SAM bucket mixes silent and live lanes in every warp
    sam = np.array(layout["sam"])
    for g in range(0, len(sam), 32):
        rows = sam[g:g + 32]
        assert np.any(np.all(o["audio"][rows] == 0.0, axis=1)) and np.any(np.abs(o["audio"][rows]).max(axis=1) > 1e-3)
    return int(sub.sum())


# ------------------------------------------------------------------------------------------------------------------- tiny
TINY_SCALES = (1e-39, 1e-30, 1e-20, 1e-9, 1e-18)  # the last two are sweeps over +-1 decade around the value


def tiny(n_blocks=40, seed=2):
    """float32 planes: the live signal scaled by each of TINY_SCALES, on every mode (blanker on for odd rows, ALS on every
    third).  1e-39 puts subnormals into the chain's input.  The 1e-9 and 1e-18 rows sweep their amplitude over two decades,
    so that the blanker envelope's |I|^2+|Q|^2 (1e-9) and the SAM phase detector's operands (1e-18) cross 2^-60.
    Returns (I, Q, events, scale of each row)."""
    ns = n_blocks * N_BLOCK
    ev, X, scales = [], [], []
    sweep = 10.0 ** np.linspace(-1.0, 1.0, ns)
    for s in TINY_SCALES:
        for m in MODES:
            r = len(X)
            x = live(m, r, ns, amp=0.3, seed=seed) * s
            if s in (1e-9, 1e-18):
                x = x * sweep
            X.append(x)
            scales.append(s)
            ev += row_events(r, m, nb=r % 2 == 1, als=r % 3 == 0)
    X = np.array(X)
    return X.real.astype(np.float32), X.imag.astype(np.float32), ev, np.array(scales)


def step_taps(I, Q, events, row, taps=("in_i", "in_q", "if_i", "if_q")):
    """Steps one row through oracle_lib.Channel; returns {tap: [n_blocks, 128]} of the requested stage taps."""
    from oracle import oracle_lib
    ch = oracle_lib.Channel()
    mine = sorted([e for e in events if e[0] == row], key=lambda e: e[1])
    nb = I.shape[1] // N_BLOCK
    out = {t: np.empty((nb, N_BLOCK), np.float32) for t in taps}
    ei = 0
    for b in range(nb):
        while ei < len(mine) and mine[ei][1] <= b:
            ch.apply(mine[ei][2], *mine[ei][3:]); ei += 1
        ch.update(I[row, b * N_BLOCK:(b + 1) * N_BLOCK], Q[row, b * N_BLOCK:(b + 1) * N_BLOCK])
        for t in taps:
            out[t][b] = ch.taps[oracle_lib.TAPS.index(t)]
    return out


def tiny_check(I, Q, ev, scales, o):
    """1e-39 rows carry subnormal input; the envelope's squared magnitude (1e-9 rows) and the SAM PLL's input magnitude
    (1e-18 rows, the bound of |dr| and |di|) lie on both sides of 2^-60."""
    sub = (I != 0) & (np.abs(I) < FLT_MIN)
    assert sub[scales == 1e-39].mean() > 0.9
    r9 = int(np.flatnonzero(scales == 1e-9)[0])      # an odd row: blanker on, the envelope runs
    t = step_taps(I, Q, ev, r9)
    sq = t["in_i"].astype(np.float32) ** 2 + t["in_q"].astype(np.float32) ** 2
    assert np.any(sq < TWO_M60) and np.any(sq > TWO_M60)
    r18 = int(np.flatnonzero(scales == 1e-18)[MODES.index(S.SAM)])
    t = step_taps(I, Q, ev, r18)
    mag = np.hypot(t["if_i"].astype(np.float64), t["if_q"].astype(np.float64))
    assert np.any(mag < TWO_M60) and np.any(mag > 4 * TWO_M60)
    assert np.all(np.isfinite(o["audio"]))


# ------------------------------------------------------------------------------------------------------------- full scale
FULL_SCALE_ROWS = [  # (input gain, output gain, AGC on)
    (10.0, 3.0, False), (15.0, 1e5, False), (10.0, -2.0, False), (1.0, 0.0, True), (12.0, 1e5, True), (10.0, 0.5, False),
    (1.0, -3.0, True)]


def full_scale(n_blocks=30):
    """int16 square waves at full scale on both rails (+32767 / -32768, Q a quarter period behind I, periods of 5 to 8
    samples: the fundamental lands in the IF passband), every mode x FULL_SCALE_ROWS, blanker on every other row, ALS on
    every third.  Gains 10 and above (the reference clamps at 10) with the AGC off drive |audio| past 256 and the int16
    pcm through its wrap and the x86 'indefinite' conversion."""
    ns = n_blocks * N_BLOCK
    t = np.arange(ns)
    I, Q, ev = [], [], []
    for m in MODES:
        for gi, go, agc in FULL_SCALE_ROWS:
            r = len(I)
            p = 5 + r % 4
            ph = (t + r) % p
            I.append(np.where(ph < p / 2.0, 32767, -32768).astype(np.int16))
            Q.append(np.where((ph + p // 4) % p < p / 2.0, 32767, -32768).astype(np.int16))
            ev += row_events(r, m, nb=r % 2 == 1, als=r % 3 == 0, agc=agc)
            ev += [(r, 0, "setInputGain", gi), (r, 0, "setOutputGain", go)]
    return np.array(I), np.array(Q), ev


def large_float(n_blocks=30, seed=4):
    """float32 planes with amplitudes from 1 to ~1e3: the live signal scaled, and square waves, every mode, AGC off on
    every other row."""
    ns = n_blocks * N_BLOCK
    t = np.arange(ns)
    X, ev = [], []
    for m in MODES:
        for k, amp in enumerate((1.0, 30.0, 1000.0)):
            r = len(X)
            if k == 2:
                p = 5 + r % 4
                x = amp * (np.where((t % p) < p / 2.0, 1.0, -1.0) + 1j * np.where(((t + p // 4) % p) < p / 2.0, 1.0, -1.0))
            else:
                x = live(m, r, ns, amp=amp, seed=seed)
            X.append(x)
            ev += row_events(r, m, nb=r % 2 == 0, als=r % 3 == 1, agc=r % 2 == 1)
    X = np.array(X)
    return X.real.astype(np.float32), X.imag.astype(np.float32), ev


def full_scale_check(o):
    """Rows with |audio| >= 256, pcm that wraps (|g * 32767| >= 32768 but below 2^31) and samples past 2^31 (x86 gives
    the 'indefinite' 0x80000000, whose low half is 0)."""
    a = o["audio"].astype(np.float64)
    fin = np.isfinite(a)
    big = fin & (np.abs(a) >= 256.0)
    assert np.count_nonzero(big.any(axis=1)) >= 3
    scaled = np.where(fin, a, 0.0) * 32767.0
    wrap = fin & (np.abs(scaled) >= 32768.0) & (np.abs(scaled) < 2.0 ** 31)
    assert wrap.any() and np.any(wrap & (np.sign(o["pcm"]) != np.sign(scaled)))
    indefinite = fin & (np.abs(scaled) >= 2.0 ** 31)
    assert indefinite.any() and np.all(o["pcm"][indefinite] == 0)


# -------------------------------------------------------------------------------------------------------------- clustered
NB_THRESHOLDS = (None, 0.0, -1.0, 0.5, 1.0)  # None: 10 dB (setNoiseBlankerThresholdDb), else setNoiseBlankerThreshold
PAIR_BLOCKS = (16, 18, 20)
PAIR_AT = 20  # in-block position of a pair's first burst: both windows end before the positions the re-scan reaches


def pair_gaps(row):
    return tuple((row + 4 * k) % 13 for k in range(len(PAIR_BLOCKS)))


def bursts(row):
    """(first sample, length) of each burst of a row, and the blocks whose scan must detect it."""
    B = N_BLOCK
    out = [(8 * B + 0, 1), (9 * B + 1, 1), (10 * B + 9, 1), (11 * B + 10, 1), (12 * B + 76, 1),
           (13 * B + 77, 1), (13 * B + 78, 1), (13 * B + 79, 1),          # three windows on top of each other
           (14 * B + 117, 11),                                            # 117..127: the end of a block
           (22 * B + 124, 8),                                             # across a block boundary
           (24 * B + 127, 1), (25 * B + 0, 1),                            # the last and the first sample of two blocks
           (27 * B + 100, 150)]                                           # longer than a block
    for blk, g in zip(PAIR_BLOCKS, pair_gaps(row)):
        p1 = blk * B + PAIR_AT
        out += [(p1, 1), (p1 + 21 + g, 1)]                                # zero windows `g` samples apart
    return sorted(out)


# blocks whose status shows a detection at 10 dB: a burst in block k is scanned when block k is the ring's middle block,
# i.e. at the call for block k + 1 (blocks 22 / 23 and 27 / 28 carry the bursts across a boundary)
CLUSTER_DETECT = (9, 10, 11, 12, 13, 14, 15, 17, 19, 21, 23, 24, 25, 26, 28, 29)


def clustered(n_blocks=36, seed=5):
    """Blanker on, every mode x NB_THRESHOLDS, the live signal at 0.2 of full scale plus bursts of 0.9 + 0.9j (bursts())."""
    ns = n_blocks * N_BLOCK
    X, ev = [], []
    for thr in NB_THRESHOLDS:
        for m in MODES:
            r = len(X)
            x = live(m, r, ns, seed=seed)
            for a, n in bursts(r):
                x[a:a + n] = 0.9 + 0.9j
            X.append(x)
            ev += row_events(r, m, nb=True, als=r % 3 == 2)
            if thr is not None:
                ev += [(r, 0, "setNoiseBlankerThreshold", thr)]
    I, Q = _quantise_rows(np.array(X))
    return I, Q, ev


def blanker_mask(I, Q, ev, row):
    """The mask the oracle applied to each block of a row: [n_blocks - 2, 128] (block k leaves the blanker two calls later)."""
    t = step_taps(I, Q, ev, row, taps=("in_i", "in_q", "nb_i", "nb_q"))
    xi, xq = t["in_i"][:-2], t["in_q"][:-2]
    yi, yq = t["nb_i"][2:], t["nb_q"][2:]
    use_i = np.abs(xi) >= np.abs(xq)
    num, den = np.where(use_i, yi, yq), np.where(use_i, xi, xq)
    assert np.all(den != 0)
    return (num / den).astype(np.float32)


def clustered_check(I, Q, ev, block_status):
    """At 10 dB the detections come at the blocks the bursts were designed for and nowhere before them; windows closer
    together than the edge ramp get their ramp and the ones in the gap (or merge, gap 0); every sample is blanked
    at threshold <= 0; block_status: [n_blocks, BS_FIELDS, n_rows] records of the oracle."""
    import audiosdr_b200 as A
    det = A.block_status_fields(block_status)["nb_detected"]
    n10 = len(MODES)
    for r in range(n10):
        assert det[list(CLUSTER_DETECT), r].all(), (r, det[:, r].nonzero())
        assert not det[4:9, r].any(), (r, det[:, r].nonzero())
    seen = set()
    for r in range(n10):
        mask = blanker_mask(I, Q, ev, r)
        for blk, g in zip(PAIR_BLOCKS, pair_gaps(r)):
            mk = mask[blk]
            end1 = PAIR_AT + 11
            end2 = end1 + g + 21
            np.testing.assert_allclose(mk[end2 - 7:end2], RAMP_DN, atol=1e-6)
            assert np.all(mk[end2:end2 + 5] == 1.0)
            if g == 0:   # one merged window, one edge
                assert np.all(mk[PAIR_AT - 10:end2 - 7] == 0.0)
            else:
                np.testing.assert_allclose(mk[end1 - 7:end1], RAMP_DN, atol=1e-6)
                assert np.all(mk[end1:end1 + g] == 1.0) and np.all(mk[end1 + g:end2 - 7] == 0.0)
            seen.add(g)
    assert seen >= set(range(7)), seen
    for r in range(n10, 3 * n10):  # thresholds 0 and -1: every sample blanked once the rings hold signal
        mask = blanker_mask(I, Q, ev, r)
        assert np.all(mask[1:] == 0.0), r


# ------------------------------------------------------------------------------------------------------------ setter edges
SETTER_EDGES = [("setInputGain", 0.0), ("setAGCattackTime", 0.01), ("setAGCreleaseTime", 1e5), ("setAGCthreshold", 0.0),
                ("setAGCslope", 1.0), ("setNoiseBlankerThreshold", 100.0)]


def setter_edges(n_blocks=48, seed=6):
    """The live signal on every mode x SETTER_EDGES (blanker on every other row, ALS on every third); each row's setter
    comes mid-stream at a block of its own, a second row per pair gets two of them, and input gain 0 is lifted again."""
    ns = n_blocks * N_BLOCK
    X, ev = [], []
    for m in MODES:
        for k, (name, val) in enumerate(SETTER_EDGES):
            r = len(X)
            x = live(m, r, ns, seed=seed)
            x[(r * 97) % ns:(r * 97) % ns + 3] = 0.9 + 0.9j  # one impulse per row for the blanker threshold rows
            X.append(x)
            ev += row_events(r, m, nb=r % 2 == 0 or name.startswith("setNoise"), als=r % 3 == 1)
            b = 6 + (r * 5) % 20
            ev.append((r, b, name, val))
            if name == "setInputGain":
                ev.append((r, b + 9, "setInputGain", 1.0))
            if r % 2:
                o_name, o_val = SETTER_EDGES[(k + 2) % len(SETTER_EDGES)]
                ev.append((r, b + 3, o_name, o_val))
    I, Q = _quantise_rows(np.array(X))
    return I, Q, ev


CASES = ("silence", "tiny", "full_scale", "large_float", "clustered", "setter_edges")


def make(case, **kw):
    """(I, Q, events) of a case by name."""
    out = globals()[case](**kw)
    return out[:3]
