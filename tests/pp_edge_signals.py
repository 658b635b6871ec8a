"""tests/pp_edge_signals.py -- the pre-processor's image detector at its thresholds.

The detector (AudioSDRpreProcessor.cpp:81-118; the kernel's pp_fft128_stage / pp_power / pp_decide in
audiosdr_b200/csrc/sdr_aux_core.cuh) never outputs its spectrum: it is only seen through three decisions, the exact compare
max > 10 * mean in double, max / image < 10 in float, and the strict > of the arg-max scan.  Tame signals sit far from
all three, so they cannot tell two FFT networks apart that differ by a few ulp.  This module

  * restates the detector in numpy float32 for a batch of blocks (`spectrum`, `decide`), with a switch per mutation of the
    kernel's arithmetic (MUTATIONS), so that a block can be asked whether it tells the oracle apart from each mutant;
  * searches blocks one rounding away from each decision (`threshold_blocks`, `ratio_blocks`, `tie_blocks`,
    `zero_image_blocks`);
  * places a selection of them where a flipped decision changes the output samples (`build`): after 10 prepared failures,
    across the +1 -> -1 rollover of the correction, and as the block that takes successCount from 1000 to 1001.

Every builder is seeded; its selection is made against the model so that every mutation in COVERED flips at least
MIN_FLIPS decisions of its output (tests/test_emu_pp_edges.py asserts this on the oracle).

Mutations not in COVERED:
  * FMA in stage 6: its only twiddle is (1, 0), where the fused product is exact;
  * FMA in stage 5: its twiddles are (1, 0) and (6.1e-17, -1).  The product with 6.1e-17 lies some 2^-55 below the other
    term, so fusing it cannot change the rounding unless that term is zero, where both forms are the same product.
    The model confirms that no searched block flips under it; it is listed in UNREACHABLE.
"""
import os
import re

import numpy as np

N_BLOCK = 128
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, F64 = np.float32, np.float64
MIN_FLIPS = 4


def _table(name, n):
    src = open(os.path.join(ROOT, "oracle", "aux_tables.inc")).read()
    words = re.search(r"%s\[%d\] = \{([^}]*)\}" % (name, n), src).group(1).replace("u", "").split(",")
    return np.array([int(w, 16) for w in words if w.strip()], np.uint32).view(F32)


TW = _table("AUX_FFT_TW", 128)       # (cos, -sin)(2 pi k / 128), interleaved
BREV = np.array([int("{:07b}".format(i)[::-1], 2) for i in range(128)])

# ---------------------------------------------------------------- mutations of the kernel's arithmetic
STAGE_FMA = ["fma_s%d_b%d" % (s, o) for s in range(6) for o in (0, 1)]
MUTATIONS = ["argmax_ge",    # 1: v >= maximum_power in the arg-max scan
             "cross_ge",     # 2: >= at the 10 * mean compare
             "ratio_le",     # 3: imbalance_ratio <= 10
             ] + STAGE_FMA + [  # 4: b[0] = fmaf(tr, wr, -p1) / b[1] = fmaf(tr, wi, p3) in one stage
             "power_fma",    # 5: fmaf(re, re, im * im) in pp_power
             "avg_pairs",    # 6: the average as two interleaved partial sums
             "avg_recip"]    # 7: the average as sum * (1 / 118.0f)
UNREACHABLE = ["fma_s5_b0", "fma_s5_b1"]
COVERED = [m for m in MUTATIONS if m not in UNREACHABLE]


def fma32(a, b, c):
    """fmaf(a, b, c) for float32 arrays: a * b is exact in double; the sum is rounded once to float32 by resolving the
    one case where rounding through double is wrong (the double sum lands on a float32 midpoint while inexact)."""
    p = a.astype(F64) * b.astype(F64)
    c = c.astype(F64)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)   # s + err == p + c exactly (TwoSum)
    with np.errstate(over="ignore", invalid="ignore"):
        f = s.astype(F32)
        g = np.nextafter(f, np.where(s > f.astype(F64), F32(np.inf), F32(-np.inf)))
        tie = (err != 0) & (s != f.astype(F64)) & (2.0 * s == f.astype(F64) + g.astype(F64))
        toward = np.sign(err) == np.sign(g.astype(F64) - f.astype(F64))
    return np.where(tie & toward, g, f).astype(F32)


def q15(x):
    """(float)((double)(float)q / 32767.0), PP.cpp:84-85"""
    return (np.asarray(x).astype(F64) / 32767.0).astype(F32)


def spectrum(I, Q, mut=None):
    """Power of the 128-point FFT of blocks I, Q int16 [N, 128], natural bin order, float32 [N, 128]: the radix-2 DIF
    network of oracle/aux_fft128.h and pp_fft128_stage, one rounding per operation unless `mut` fuses one."""
    re, im = q15(I).copy(), q15(Q).copy()
    n = re.shape[0]
    for s in range(7):
        half = 64 >> s
        r, i = re.reshape(n, -1, 2, half), im.reshape(n, -1, 2, half)
        ar, ai, br, bi = r[:, :, 0].copy(), i[:, :, 0].copy(), r[:, :, 1].copy(), i[:, :, 1].copy()
        k = np.arange(half) << s
        wr, wi = TW[2 * k], TW[2 * k + 1]
        tr, ti = ar - br, ai - bi
        r[:, :, 0], i[:, :, 0] = ar + br, ai + bi
        p0, p1, p2, p3 = tr * wr, ti * wi, tr * wi, ti * wr
        r[:, :, 1] = fma32(tr, np.broadcast_to(wr, tr.shape), -p1) if mut == "fma_s%d_b0" % s else p0 - p1
        i[:, :, 1] = fma32(tr, np.broadcast_to(wi, tr.shape), p3) if mut == "fma_s%d_b1" % s else p2 + p3
    re, im = re[:, BREV], im[:, BREV]
    if mut == "power_fma":
        return fma32(re, re, im * im)
    return re * re + im * im


def decide(pw, mut=None):
    """The scan and compares of PP.cpp:91-104 on power spectra [N, 128].  Returns a dict of arrays: d (0 = no strong
    line, 1 = failure (image within a factor 10), 2 = success), line, mx, avg, ratio."""
    band = pw[:, 5:123]
    if mut == "avg_pairs":
        s0, s1 = np.zeros(len(pw), F32), np.zeros(len(pw), F32)
        for j in range(0, 118, 2):
            s0 = s0 + band[:, j]
            s1 = s1 + band[:, j + 1]
        tot = s0 + s1
    else:
        tot = np.zeros(len(pw), F32)
        for j in range(118):
            tot = tot + band[:, j]
    avg = tot * F32(1.0 / 118.0) if mut == "avg_recip" else tot / F32(118.0)
    mx = band.max(axis=1)
    if mut == "argmax_ge":
        line = 5 + 117 - np.argmax(band[:, ::-1], axis=1)
    else:
        line = 5 + np.argmax(band, axis=1)
    lim = 10.0 * avg.astype(F64)
    cross = mx.astype(F64) >= lim if mut == "cross_ge" else mx.astype(F64) > lim
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = mx / pw[np.arange(len(pw)), 128 - line]
    fail = ratio <= F32(10.0) if mut == "ratio_le" else ratio < F32(10.0)
    d = np.where(cross, np.where(fail, 1, 2), 0)
    return dict(d=d, line=line, mx=mx, avg=avg, ratio=ratio, cross=cross)


def decisions(I, Q, mut=None):
    return decide(spectrum(I, Q, mut), mut)["d"]


def flips(I, Q):
    """{mutation: bool [N]}: the blocks whose decision differs between the oracle's arithmetic and the mutant's."""
    base = decisions(I, Q)
    return {m: decisions(I, Q, m) != base for m in MUTATIONS}


# ---------------------------------------------------------------- the state machine over whole channels
def correct(I, Q, st):
    """pp_correct_block on blocks [C, 128] (copies) for states st [C, 6] = (autod, corr, fail, succ, saved, swap)."""
    I, Q = I.copy(), Q.copy()
    for corr, rail in ((1, I), (-1, Q)):
        m = st[:, 1] == corr
        t = rail[m, 127].copy()
        rail[m, 1:] = rail[m, :-1].copy()
        I[m, 0] = st[m, 4]
        st[m, 4] = t
    return I, Q


def apply_event(st, c, name, arg=0):
    if name == "startAutoI2SerrorDetection":
        st[c, 0], st[c, 1], st[c, 2], st[c, 3] = 1, 0, 0, 0
    elif name == "stopAutoI2SerrorDetection":
        st[c, 0], st[c, 1] = 0, 0
    elif name == "setI2SerrorCompensation":
        st[c, 1] = int(np.int16(int(arg))); st[c, 0] = 0
    elif name == "swapIQ":
        st[c, 5] = int(arg != 0)


def model_run(I, Q, events=(), mut=None, record=False):
    """The pre-processor over planes I, Q int16 [C, S] with setter events, on the model's detector: (out I, out Q,
    status [C, 6]) like oracle.aux_lib.run, plus, with record=True, the per-block states [n_blocks, C, 6] and
    decisions [n_blocks, C] (-1 where the detector is off)."""
    nch, ns = I.shape
    nb = ns // N_BLOCK
    st = np.zeros((nch, 6), np.int64)
    oi, oq = np.empty_like(I), np.empty_like(Q)
    ev = sorted(events, key=lambda e: e[1])
    states, decs = [], []
    for b in range(nb + 1):
        for e in ev:
            if (e[1] == b if b < nb else e[1] >= b):
                for c in (range(nch) if e[0] is None else [e[0]]):
                    apply_event(st, c, e[2], *(e[3:]))
        if b == nb:
            break
        z = slice(b * N_BLOCK, (b + 1) * N_BLOCK)
        bi, bq = correct(I[:, z], Q[:, z], st)
        on = st[:, 0] == 1
        dd = np.full(nch, -1)
        if on.any():
            r = decide(spectrum(bi[on], bq[on], mut), mut)
            dd[on] = r["d"]
            s, d = st[on], r["d"]
            s[:, 2] = np.where(d == 1, s[:, 2] + 1, np.where(d == 2, 0, s[:, 2]))
            turn = s[:, 2] > 10
            s[turn, 1] = np.where(s[turn, 1] < 1, s[turn, 1] + 1, -1)
            s[turn, 2] = s[turn, 3] = 0
            s[:, 3] += d != 0
            s[s[:, 3] > 1000, 0] = 0
            st[on] = s
        sw = st[:, 5] == 1
        oi[:, z] = np.where(sw[:, None], bq, bi)
        oq[:, z] = np.where(sw[:, None], bi, bq)
        if record:
            states.append(st.copy()); decs.append(dd)
    out = (oi, oq, st.astype(np.int32))
    return out + ((np.array(states), np.array(decs)) if record else ())


# ---------------------------------------------------------------- searches
def _ulp(x):
    x = np.abs(x).astype(F32)
    return (np.nextafter(x, F32(np.inf)) - x).astype(F64)


def _greedy(I, Q, objective, rng, iters, done):
    """Walks each block by +-1..3 LSB on one random sample per step, keeping a step when |objective| does not grow; a
    block stops when done(objective) holds.  I, Q int16 [N, 128] (modified in place); objective(I, Q, rows) is given the
    pool rows of the blocks it evaluates."""
    obj = objective(I, Q, np.arange(len(I)))
    for _ in range(iters):
        act = np.flatnonzero(~done(obj))
        if not len(act):
            break
        ni, nq = I[act].copy(), Q[act].copy()
        pos = rng.integers(0, 256, len(act))
        step = rng.integers(1, 4, len(act)) * rng.choice([-1, 1], len(act))
        for rail, sel in ((ni, pos < 128), (nq, pos >= 128)):
            rows, cols = np.flatnonzero(sel), pos[sel] % 128
            rail[rows, cols] = np.clip(rail[rows, cols].astype(np.int32) + step[sel], -32768, 32767)
        new = objective(ni, nq, act)
        ok = np.abs(new) <= np.abs(obj[act])
        I[act[ok]], Q[act[ok]], obj[act[ok]] = ni[ok], nq[ok], new[ok]
    return obj


def _tone(n, k, amp, phase):
    t = np.arange(N_BLOCK)
    a = 2 * np.pi * k[:, None] * t[None, :] / N_BLOCK + phase[:, None]
    return amp[:, None] * np.cos(a), amp[:, None] * np.sin(a)


def _i16(x):
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


def threshold_blocks(n, seed, recip=False):
    """Blocks with max within 1 ulp of 10 * mean: a noisy tone whose line stands about 10x the mean, walked by LSB steps.
    The objective is (max - 10 * mean) in ulp of max; blocks that end at exactly 0 decide the > vs >= mutant.
    recip=True walks on until the mean divided by 118 and the mean multiplied by 1/118 fall on either side of max / 10
    (few blocks at the threshold do: the two means differ for some sums only, by 1 ulp)."""
    rng = np.random.default_rng(seed)
    sig = rng.uniform(2000, 7000, n)
    k = rng.integers(8, 120, n)
    amp, ph = 0.42 * sig, rng.uniform(0, 2 * np.pi, n)
    nr, ni = rng.normal(0, 1, (2, n, N_BLOCK)) * sig[:, None]
    for _ in range(5):  # scale the tone until its line stands 10x the mean (line ~ amp^2, mean = (line + rest) / 118)
        re, im = _tone(n, k, amp, ph)
        I, Q = _i16(re + nr), _i16(im + ni)
        r = decide(spectrum(I, Q))
        mx = r["mx"].astype(F64)
        amp = amp * np.sqrt(np.clip(10.0 * (118.0 * r["avg"] - mx) / 108.0 / mx, 0.25, 4.0))

    def objective(i, q, rows=None):
        r = decide(spectrum(i, q))
        return (r["mx"].astype(F64) - 10.0 * r["avg"].astype(F64)) / _ulp(r["mx"])
    # a rough walk to the threshold, then on to exact equality where the average allows it (10 * avg in float32)
    obj = _greedy(I, Q, objective, rng, 400, lambda o: np.abs(o) <= 1.0)
    if recip:
        def split(i, q, rows):  # flat within 3 ulp: the walk keeps moving there until the two means fall either side
            pw = spectrum(i, q)
            r, m = decide(pw), decide(pw, "avg_recip")
            o = np.abs(r["mx"].astype(F64) - 10.0 * r["avg"].astype(F64)) / _ulp(r["mx"])
            return np.where(r["d"] != m["d"], 0.0, np.maximum(o, 3.0))
        keep = _greedy(I, Q, split, rng, 1500, lambda o: o == 0) == 0
        return I[keep], Q[keep], objective(I[keep], Q[keep])
    obj = _greedy(I, Q, objective, rng, 150, lambda o: (o == 0) | (np.abs(o) > 1.0))
    keep = np.abs(obj) <= 1.0
    return I[keep], Q[keep], obj[keep]


def ratio_blocks(n, seed):
    """Blocks whose line stands 10x its image: a tone plus an image of a third of its amplitude, with small noise, walked
    until the float32 ratio is within 1 ulp of 10.0f (both sides, and exactly 10.0f).  Objective: ratio - 10 in ulp."""
    rng = np.random.default_rng(seed)
    amp = rng.uniform(6000, 14000, n)
    k = rng.integers(6, 60, n) * rng.choice([-1, 1], n) % 128
    ph = rng.uniform(0, 2 * np.pi, n)
    re, im = _tone(n, k, amp, ph)
    re2, im2 = _tone(n, (128 - k) % 128, amp / np.sqrt(10.0), rng.uniform(0, 2 * np.pi, n))
    I = _i16(re + re2 + rng.normal(0, 20, (n, N_BLOCK)))
    Q = _i16(im + im2 + rng.normal(0, 20, (n, N_BLOCK)))
    ten_ulp = float(np.nextafter(F32(10), F32(11)) - F32(10))

    def objective(i, q, rows):
        r = decide(spectrum(i, q))
        return np.where(r["cross"], (r["ratio"].astype(F64) - 10.0) / ten_ulp, 1e9)
    obj = _greedy(I, Q, objective, rng, 300, lambda o: np.abs(o) <= 1.0)
    keep = np.abs(obj) <= 1.0
    return I[keep], Q[keep], obj[keep]


def tie_blocks(n, seed):
    """Two in-band lines with bit-identical power, the later one with a different image: line k1 < k2 of equal amplitude,
    k1 with an image at a third of its amplitude (ratio about 9: a failure), k2 without (a success), walked until the
    two powers are the same float.  Under >= the scan takes k2 and the block decides the other way."""
    rng = np.random.default_rng(seed)
    amp = rng.uniform(5000, 9000, n)
    k1 = rng.integers(6, 40, n)
    k2 = k1 + rng.integers(4, 20, n)
    a, b = _tone(n, k1, amp, rng.uniform(0, 2 * np.pi, n))
    c, d = _tone(n, k2, amp, rng.uniform(0, 2 * np.pi, n))
    e, f = _tone(n, 128 - k1, amp / 3.0, rng.uniform(0, 2 * np.pi, n))
    I = _i16(a + c + e + rng.normal(0, 8, (n, N_BLOCK)))
    Q = _i16(b + d + f + rng.normal(0, 8, (n, N_BLOCK)))

    def objective(i, q, rows):
        p = spectrum(i, q)
        x, y = p[np.arange(len(i)), k1[rows]], p[np.arange(len(i)), k2[rows]]
        return y.view(np.int32).astype(F64) - x.view(np.int32).astype(F64)  # ulps apart (same sign, same binade or next)
    obj = _greedy(I, Q, objective, rng, 600, lambda o: o == 0)
    keep = obj == 0
    return I[keep], Q[keep], np.stack([k1[keep], k2[keep]], 1)


def zero_image_blocks():
    """Blocks whose strongest line has an image of exactly zero power (ratio = inf).  A tone of period 4 leaves only
    bins 32 and 96 non-zero after stage 4 (every butterfly there subtracts equal values), and stage 5 multiplies the
    odd half by (6.1e-17, -1).  With both parts of x1 - x3 non-zero that product rounds to -i (x1 - x3) exactly, so a
    tone at 45 degrees, x = A (1 + i) i^(+-n), cancels its image bit for bit.  (With x1 - x3 on an axis the 6.1e-17
    survives and the image power is about 1e-30, not zero.)"""
    out_i, out_q = [], []
    for a in (1, 77, 9000, 32767):
        for sgn in (1, -1):
            for rot in range(4):
                z = a * (1 + 1j) * (1j ** ((sgn * np.arange(N_BLOCK) + rot) % 4))
                out_i.append(_i16(z.real)); out_q.append(_i16(z.imag))
    I, Q = np.array(out_i), np.array(out_q)
    r = decide(spectrum(I, Q))
    assert (r["cross"] & np.isinf(r["ratio"])).all()
    return I, Q


# ---------------------------------------------------------------- placement
PLACEMENTS = ("after_failures", "rollover", "finish")
SEEDS = {"after_failures": 101, "rollover": 202, "finish": 303}  # selections and phases
POOL_SEED = 1  # the searched blocks, shared by the builders
TARGET = 6  # flips per mutation the selection aims for (MIN_FLIPS is what the tests demand)
_pools = {}


def pool(seed):
    """(I, Q, kind, offset) of the searched knife-edge blocks of one seed; offset = the search's final objective (ulp
    from the threshold, 0 = exact) for "threshold" and "ratio" blocks."""
    if seed not in _pools:
        ti, tq, to = threshold_blocks(400, seed)
        ai, aq, ao = threshold_blocks(120, seed + 3, recip=True)
        ti, tq, to = np.concatenate([ti, ai]), np.concatenate([tq, aq]), np.concatenate([to, ao])
        ri, rq, ro = ratio_blocks(300, seed + 1)
        xi, xq, _ = tie_blocks(60, seed + 2)
        zi, zq = zero_image_blocks()
        _pools[seed] = (np.concatenate([ti, ri, xi, zi]), np.concatenate([tq, rq, xq, zq]),
                        np.array(["threshold"] * len(ti) + ["ratio"] * len(ri) + ["tie"] * len(xi) + ["zero_image"] * len(zi)),
                        np.concatenate([to, ro, np.zeros(len(xi) + len(zi))]))
    return _pools[seed]


def select(I, Q, kind, offset, rng):
    """Indices of pool blocks: two of each kind and side (below, at, above the threshold), then greedily the blocks that
    flip the mutations still short of TARGET."""
    F = np.array([flips(I, Q)[m] for m in COVERED]).T  # [N, M]
    pick = []
    for k, side in (("threshold", -1), ("threshold", 0), ("threshold", 1), ("ratio", -1), ("ratio", 0), ("ratio", 1),
                    ("tie", 0), ("zero_image", 0)):
        cand = np.flatnonzero((kind == k) & (np.round(offset) == side))
        pick += list(rng.permutation(cand)[:2])
    while True:
        need = np.maximum(TARGET - F[pick].sum(0), 0)
        if not need.any():
            return np.array(pick)
        gain = (F * (need > 0)).sum(1)
        gain[pick] = -1
        best = np.flatnonzero(gain == gain.max())
        assert gain.max() > 0, "no searched block flips " + str([m for m, n in zip(COVERED, need) if n])
        pick.append(int(rng.choice(best)))


def _prepared(kind, phase):
    """A block far from every threshold: "F" a real tone (line and image equal: a failure), "S" a complex tone (no
    image: a success), also when a correction shifts one rail by a sample."""
    t = np.arange(N_BLOCK)
    if kind == "F":
        return _i16(12000 * np.cos(2 * np.pi * 20 * t / N_BLOCK + phase)), np.zeros(N_BLOCK, np.int16)
    a = 2 * np.pi * 7 * t / N_BLOCK + phase
    return _i16(12000 * np.cos(a)), _i16(12000 * np.sin(a))


def build(placement, seed=None):
    """One channel per selected knife-edge block X, placed where one flipped decision moves I2Scorrection:
      after_failures  S S F x10  X  F S S       X meets failureCount 10 at correction 0;
      rollover        S S F x21  X  F S S       11 failures take the correction to +1, X meets failureCount 10 there, so
                                                a failure at X rolls it over to -1 (X is stored shifted by the +1 lag);
      finish          S x990 F x10  X  F S S    X meets successCount 1000: a strong line there stops the detector.
    The F after X separates "no strong line" from "success": it is the 11th failure only if X changed nothing.
    Returns (I, Q, events, layout) with layout = dict(block, corr, succ, kind, offset, X=(I, Q) as the detector sees it)."""
    seed = SEEDS[placement] if seed is None else seed
    rng = np.random.default_rng(seed)
    PI, PQ, kind, offset = pool(POOL_SEED)
    sel = select(PI, PQ, kind, offset, rng)
    head = {"after_failures": "SS" + "F" * 10, "rollover": "SS" + "F" * 21, "finish": "S" * 990 + "F" * 10}[placement]
    seq = head + "X" + "FSS"
    corr = 1 if placement == "rollover" else 0
    nch, nb = len(sel), len(seq)
    I, Q = np.empty((nch, nb * N_BLOCK), np.int16), np.empty((nch, nb * N_BLOCK), np.int16)
    for c, j in enumerate(sel):
        ph = rng.uniform(0, 2 * np.pi)
        for b, k in enumerate(seq):
            z = slice(b * N_BLOCK, (b + 1) * N_BLOCK)
            if k == "X":
                xi, xq = PI[j], PQ[j]
                if corr == 1:  # the detector sees I[0] = the previous block's last I sample, I[i] = I[i - 1]
                    I[c, z] = np.concatenate([xi[1:], xi[-1:]])
                    I[c, z.start - 1] = xi[0]
                else:
                    I[c, z] = xi
                Q[c, z] = xq
            else:
                I[c, z], Q[c, z] = _prepared(k, ph + 0.37 * b)
    for k, want in (("F", 1), ("S", 2)):  # the prepared blocks decide alike under every mutation, shifted or not
        bi, bq = np.array([_prepared(k, p)[0] for p in range(8)]), np.array([_prepared(k, p)[1] for p in range(8)])
        for i, q in ((bi, bq), (np.roll(bi, 1, 1), bq), (bi, np.roll(bq, 1, 1))):
            assert all((decisions(i, q, m) == want).all() for m in [None] + MUTATIONS)
    events = [(None, 0, "startAutoI2SerrorDetection")] + [(c, 0, "swapIQ", 1) for c in range(2, nch, 3)]
    layout = dict(block=seq.index("X"), corr=corr, succ={"after_failures": 12, "rollover": 11, "finish": 1000}[placement], kind=kind[sel],
                  offset=offset[sel], X=(PI[sel], PQ[sel]))
    return I, Q, events, layout
