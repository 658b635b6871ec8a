"""tests/pll_edge_signals.py -- the SAM PLL and the noise blanker one rounding away from their decisions.

The SAM PLL (C:688-749; RolePll::step in audiosdr_b200/csrc/sdr_pipeline.cuh) decides per sample between the branches of
atan2_approx, whether the phase wraps, and whether the loop is locked; the kernel adds its own decisions on top (the fast
path's range guards, float forms of the reference's double compares, the cosine index's wrap).  Noisy tones never land on
an exact tie, so none of these decisions is tested by ordinary stimuli.  This module

  * restates the chain from the blanker to the demodulator in numpy float32, one rounding per operation in the oracle's
    operand order (`Model`: nb_run, cascade_run for the IF stage, sam_run with every branch of atan2_approx, the LUT
    oscillator with the reference's double index expression, and the envelope fallback's shifter and image filter), with
    one switch per mutation of the kernel (MUTATIONS);
  * places knife-edge samples with float32 input at gain 1, where the scaled sample is the input value exactly: at a
    chosen sample the model is stopped, I[n] and Q[n] are swept (IF_I[n] depends only on I, IF_Q[n] only on Q), and the
    pair whose decision operands sit exactly on the threshold -- or one float either side -- is written into the input
    (`build`).  The blanker's knife edges are placed on the input alone: its running average depends on nothing else.

Every knife-edge row carries one placed sample, and the rows are laid out in the warps the receiver forms (WARPS), so that
on the GPU the fast-path edges meet the fast path: its warp-wide vote passes at each of them.  The rows of each target are
chosen so that every mutation in COVERED flips at least MIN_FLIPS decisions that change the demodulator output or the
block records (test_emu_pll_edges.py).

Mutations no input can observe (UNREACHABLE):
  * `wrap_gt` (the general path's `phase > 0x1.921fb6p+1f`) and `fast_wrap_gt` (the same in the fast path, with `ph2 <=`
    in the range test): they differ from the reference only at phase == 0x1.921fb6p+1 = a, the first float above pi.
    There the reference subtracts 2a, lands on -a < -pi and adds 2a back: both steps are exact, so the phase and the
    oscillator are the same as without the wrap (the `wrap_up` rows place that double wrap).
  * `fast_lo_le` (`ph0 <= -0x1.921fb4p+1f` in the fast path): at ph0 == -0x1.921fb4p+1 the mutant adds 2 pi and gets
    0x1.921fb8p+1 >= a, which fails the fast path's range test, so the general path computes the sample correctly.
Not reached (NOT_REACHED): `cos_wrap_dn`, the cosine index's bound one float down.  It differs only at ph2 ==
-0x1.921fb6p+0, which none of the searched rows reaches; its other direction, `cos_wrap_up`, is covered.

Which odd-mantissa phases a loop can reach depends on the parity its phase settles on during acquisition: filt and prev
are multiples of 2^-19 once the accumulator d0 is above 32 (a carrier at 6890 Hz), so ph0 keeps the residue of phase's
mantissa.  The targets that need a particular residue (ph0 == 0x1.921fb6p+1, ph0 == +0, ph2 on the cosine index's wrap)
are therefore searched on several rows with a 3000 Hz carrier (TRY), of which some settle on each parity.

A fast-path guard widened to |di| >= 2^-64 (div_inrange outside its stated range) is invisible on the host, whose
div_inrange is an IEEE division; the `tiny_di_dn` row (|di| one float below 2^-60) is where the GPU's division sequence
would then run, alone in its warp so that the vote passes.
"""
import os
import re

import numpy as np

N_BLOCK = 128
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, F64 = np.float32, np.float64
MIN_FLIPS = 4
PI = 3.1415926535897932384626433832795
TWO_PI = F32(2.0 * PI)
HALF_PI = F32(0.5 * PI)
PI_UP = F32(np.float32(PI))             # 0x1.921fb6p+1: the first float above pi ((double)ph >= PI <=> ph >= PI_UP)
PI_DN = np.nextafter(PI_UP, F32(0))      # 0x1.921fb4p+1: (double)ph < -PI <=> ph < -PI_DN
HALF_DN = F32(-float.fromhex("0x1.921fb4p+0"))           # the cosine index wraps for ph below this
FS = F32(44100.0)
LOCK_LO, LOCK_HI = F32(5890.0), F32(7890.0)
THR_10DB = F32(10.0 ** 0.5)              # powf(10, 10 / 20.0), correctly rounded


def _tables():
    src = open(os.path.join(ROOT, "audiosdr_b200", "csrc", "sdr_tables.inc")).read()
    out = {}
    for m in re.finditer(r"SDR_TAB_(\w+)\[(\d+)\] = \{([^}]*)\}", src):
        out[m.group(1)] = np.array([int(v.strip().rstrip("u"), 16) for v in m.group(3).split(",") if v.strip()], np.uint32).view(F32)
    return out


TAB = _tables()
SINE = TAB["SINE"]
IF_AM = TAB["IF_AM"].reshape(4, 5)
AM_IMAGE = TAB["AM_IMAGE"].reshape(4, 5)

# loop constants as the oracle's initialisers compute them (float / double promotions of H:249-284)
_wn, _zeta, _Ka = F32(0.07), F32(0.707), F32(1000.0)
_tau1, _tau2 = _Ka / (_wn * _wn), F32(2) * _zeta / _wn
B0 = F32(F64(F32(2) * _Ka / _tau1) * (1.0 + 2.0 * F64(_tau2)))
B1 = F32(F64(F32(2) * _Ka / _tau1) * (1.0 - 2.0 * F64(_tau2)))
A1 = F32(-1.0)
ALPHA = F32(0.995)
BETA = F32(1.0 - F64(ALPHA))
FCONV = FS / TWO_PI
NB_ALPHA, NB_BETA = F32(0.995), F32(1.0 - F64(F32(0.995)))

MUTATIONS = ["lock_lo_ge",      # 1: freq >= lo
             "lock_hi_le",      # 2: freq <= hi
             "wrap_gt",         # 3: general path phase > 0x1.921fb6p+1f
             "fast_wrap_gt",    # 4: fast path ph0 > ..., ph2 <= ... in the range test
             "fast_lo_le",      # 5: fast path ph0 <= -0x1.921fb4p+1f
             "fast_ge",         # 6: dr >= adi in the fast path's guard
             "atan_ge",         # 7: fabsf(x) >= fabsf(y) in atan2_approx
             "atan_ygt",        # 8: y > 0 in atan2_approx's x < 0 branch
             "cos_wrap_up",     # 9: cosine-index wrap bound one float up (-0x1.921fb2p+0f)
             "cos_wrap_dn",     # 9: ... one float down (-0x1.921fb6p+0f)
             "nb_ge"]           # 10: mag >= avg * thr in the blanker
UNREACHABLE = ["wrap_gt", "fast_wrap_gt", "fast_lo_le"]
NOT_REACHED = ["cos_wrap_dn"]
COVERED = [m for m in MUTATIONS if m not in UNREACHABLE + NOT_REACHED]


def f32(x):
    return np.asarray(x, F32)


# ---------------------------------------------------------------- reference arithmetic (arrays of any shape)
def lut_sin(ph):
    ph = f32(ph).copy()
    ph = np.where(ph >= TWO_PI, ph - TWO_PI, ph)
    ph = np.where(ph.astype(F64) < 0.0, ph + TWO_PI, ph)
    with np.errstate(invalid="ignore"):
        ip = np.trunc(ph.astype(F64) * 65535.0 / F64(TWO_PI)).astype(np.int64) & 0xFFFF
    idx, frac = ip >> 8, (ip & 0xFF).astype(F32)
    v1, v2 = SINE[idx], SINE[idx + 1]
    prod = (v2 - v1) * frac
    return (v1.astype(F64) + prod.astype(F64) / 256.0).astype(F32)


def lut_cos(ph):
    return lut_sin((f32(ph).astype(F64) + PI / 2.0).astype(F32))


def atan_poly(z):
    return (F32(0.97239411) + F32(-0.19194795) * z * z) * z


def atan2_approx(y, x, mut=()):
    """H:384-408 on arrays; every branch evaluated, the reference's choice selected."""
    y, x = f32(y), f32(x)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        z1 = y / x
        z2 = x / y
        p1, p2 = atan_poly(z1), atan_poly(z2)
        big = (np.abs(x) >= np.abs(y)) if "atan_ge" in mut else (np.abs(x) > np.abs(y))
        ypos = (y > 0) if "atan_ygt" in mut else (y >= 0)
        b1 = np.where(x > 0, p1, np.where(ypos, (p1.astype(F64) + PI).astype(F32), (p1.astype(F64) - PI).astype(F32)))
        b2 = np.where(y > 0, -p2 + HALF_PI, -p2 - HALF_PI)
        b0 = np.where(y > 0, HALF_PI, np.where(y < 0, -HALF_PI, F32(0)))
        return np.where(x != 0, np.where(big, b1, b2), b0).astype(F32)


def sqrt_hack(x):
    x = f32(x)
    u = (x.view(np.uint32) - np.uint32(1 << 23)) >> np.uint32(1)
    o = (u + np.uint32(1 << 29)).view(F32)
    with np.errstate(divide="ignore", invalid="ignore"):
        return (0.5 * (o + x / o).astype(F64)).astype(F32)


def biquad(coef, st, x):
    """One sample through a 4-stage cascade; st: [4, 4, ...] (x1, x2, y1, y2 per stage), updated in place."""
    for s in range(4):
        b0, b1, b2, a1, a2 = coef[s]
        acc = (b0 * x) + (b1 * st[s, 0]) + (b2 * st[s, 1]) + (a1 * st[s, 2]) + (a2 * st[s, 3])
        st[s, 1] = st[s, 0]; st[s, 0] = x; st[s, 3] = st[s, 2]; st[s, 2] = acc
        x = acc
    return x


def biquad_peek(coef, st, x):
    """The cascade's output for candidate inputs x (any shape) without touching its state."""
    for s in range(4):
        b0, b1, b2, a1, a2 = coef[s]
        x = (b0 * x) + (b1 * st[s, 0]) + (b2 * st[s, 1]) + (a1 * st[s, 2]) + (a2 * st[s, 3])
    return x


def sam_sample(s, xr, xi, mut=()):
    """One sample of sam_run for state dict s (arrays broadcast against xr, xi).  Returns the new state and the decision
    operands; the kernel's fast-path predicate and its decisions are reported beside them."""
    yre, yim = s["yre"], s["yim"]
    dr = xr * yre + xi * yim
    di = xi * yre - xr * yim
    err = atan2_approx(di, dr, mut)
    d1 = s["d0"]
    d0 = err - A1 * d1
    filt = B0 * d0 + B1 * d1
    ph0 = ((s["phase"].astype(F64) + (filt + s["prev"]).astype(F64) / 2.0)).astype(F32)
    # the kernel's fast path: its own guards, and the wrap it evaluates with one pass of each compare
    adi = np.abs(di)
    ok = ((dr >= adi) if "fast_ge" in mut else (dr > adi)) & (dr <= F32(2.0 ** 60)) & (adi >= F32(2.0 ** -60))
    up = (ph0 > PI_UP) if "fast_wrap_gt" in mut else (ph0 >= PI_UP)
    dn = (ph0 <= -PI_DN) if "fast_lo_le" in mut else (ph0 < -PI_DN)
    ph2 = np.where(up, ph0 - TWO_PI, ph0)
    ph2 = np.where(dn, ph2 + TWO_PI, ph2)
    top = (ph2 <= PI_UP) if "fast_wrap_gt" in mut else (ph2 < PI_UP)
    ok = ok & top & (ph2 >= -PI_DN) & (ph2 != 0)
    # the general path (the reference's `while` loops)
    ph = ph0.copy()
    for _ in range(8):
        w = (ph > PI_UP) if "wrap_gt" in mut else (ph >= PI_UP)
        if not w.any():
            break
        ph = np.where(w, ph - TWO_PI, ph)
    for _ in range(8):
        w = ph < -PI_DN
        if not w.any():
            break
        ph = np.where(w, ph + TWO_PI, ph)
    if "fast_ge" in mut:  # the mutant's fast path at dr == |di| evaluates atan_poly(di / dr)
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            tie = ok & (dr == adi)
            e2 = atan_poly(di / dr)
        err = np.where(tie, e2, err)
        d0 = np.where(tie, e2 - A1 * d1, d0)
        filt = np.where(tie, B0 * d0 + B1 * d1, filt)
        ph0 = np.where(tie, ((s["phase"].astype(F64) + (filt + s["prev"]).astype(F64) / 2.0)).astype(F32), ph0)
        ph2 = np.where(tie, np.where(ph0 >= PI_UP, ph0 - TWO_PI, np.where(ph0 < -PI_DN, ph0 + TWO_PI, ph0)), ph2)
    phase = np.where(ok, ph2, ph)
    y_re, y_im = lut_cos(phase), lut_sin(phase)
    if "cos_wrap_up" in mut or "cos_wrap_dn" in mut:  # the kernel's cosine index with the moved bound (fast path only)
        bound = F32(-float.fromhex("0x1.921fb2p+0")) if "cos_wrap_up" in mut else F32(-float.fromhex("0x1.921fb6p+0"))
        wrong = ok & ((phase < bound) != (phase < HALF_DN))
        if wrong.any():
            a = (phase.astype(F64) + PI / 2.0).astype(F32)
            a = np.where(phase < bound, a + TWO_PI, a)
            with np.errstate(invalid="ignore"):
                ip = np.trunc(np.abs(a).astype(F64) * 65535.0 / F64(TWO_PI)).astype(np.int64) & 0xFFFF
            v1, v2 = SINE[ip >> 8], SINE[(ip >> 8) + 1]
            alt = (v1.astype(F64) + ((v2 - v1) * (ip & 0xFF).astype(F32)).astype(F64) / 256.0).astype(F32)
            y_re = np.where(wrong, alt, y_re)
    freq = ALPHA * s["freq"] + BETA * (filt * FCONV)
    lo = (freq >= LOCK_LO) if "lock_lo_ge" in mut else (freq > LOCK_LO)
    hi = (freq <= LOCK_HI) if "lock_hi_le" in mut else (freq < LOCK_HI)
    new = dict(yre=y_re, yim=y_im, d0=d0, prev=filt, phase=phase, freq=freq, locked=lo & hi)
    ops = dict(dr=dr, di=di, err=err, ph0=ph0, ph2=ph2, ok=ok, freq=freq, phase=phase)
    return new, ops


# ---------------------------------------------------------------- the chain from the blanker to the demodulator
class Model:
    """R channels in SAM mode (IF = AMpre, H:744-749), stepped block by block or sample by sample."""

    def __init__(self, R, nb_on, nb_thr, mut=()):
        self.R, self.mut = R, tuple(mut)
        self.nb_on, self.nb_thr = np.asarray(nb_on, bool), f32(nb_thr)
        z = lambda: np.zeros(R, F32)
        self.if_i, self.if_q = np.zeros((4, 4, R), F32), np.zeros((4, 4, R), F32)
        self.img_i, self.img_q = np.zeros((4, 4, R), F32), np.zeros((4, 4, R), F32)
        self.s = dict(yre=z(), yim=z(), d0=z(), prev=z(), phase=z(), freq=z(), locked=np.zeros(R, bool))
        self.phase_am = z()
        self.nb_i, self.nb_q = np.zeros((R, 3 * N_BLOCK), F32), np.zeros((R, 3 * N_BLOCK), F32)
        self.nb_mask = np.ones((R, 3 * N_BLOCK), F32)
        self.nb_avg, self.nb_hit = np.full(R, F32(10.0)), np.zeros(R, bool)

    def blanker(self, I, Q):
        """nb_run (C:606-650) for the rows with the blanker on; I, Q: [R, 128], replaced in place."""
        on = self.nb_on
        for a in (self.nb_i, self.nb_q, self.nb_mask):
            a[on, :2 * N_BLOCK] = a[on, N_BLOCK:].copy()
        self.nb_i[on, 2 * N_BLOCK:], self.nb_q[on, 2 * N_BLOCK:] = I[on], Q[on]
        self.nb_mask[on, 2 * N_BLOCK:] = 1.0
        self.nb_hit[on] = False
        ge = "nb_ge" in self.mut
        for i in range(N_BLOCK - 50, 2 * N_BLOCK):
            mag = sqrt_hack(self.nb_i[:, i] * self.nb_i[:, i] + self.nb_q[:, i] * self.nb_q[:, i])
            t = self.nb_avg * self.nb_thr
            hit = on & ((mag >= t) if ge else (mag > t))
            for r in np.flatnonzero(hit):
                self.nb_mask[r, i - 10:i + 11] = 0.0
            self.nb_hit |= hit
            self.nb_avg = np.where(on, NB_ALPHA * self.nb_avg + NB_BETA * mag, self.nb_avg)
        dn = np.array([0.933, 0.750, 0.500, 0.250, 0.067, 0.0, 0.0], F32)
        for i in range(N_BLOCK, 2 * N_BLOCK):
            e = on & (self.nb_mask[:, i] == 1.0) & (self.nb_mask[:, i - 1] == 0.0)
            for r in np.flatnonzero(e):
                self.nb_mask[r, i - 7:i] = dn
        I[on] = self.nb_mask[on, :N_BLOCK] * self.nb_i[on, :N_BLOCK]
        Q[on] = self.nb_mask[on, :N_BLOCK] * self.nb_q[on, :N_BLOCK]

    def step(self, xi_in, xq_in):
        """IF stage and one PLL sample; returns the demodulator's (I, Q) for the sample before the fallback."""
        xr, xi = biquad(IF_AM, self.if_i, xi_in), biquad(IF_AM, self.if_q, xq_in)
        self.s, ops = sam_sample(self.s, xr, xi, self.mut)
        lk = self.s["locked"]
        oi = np.where(lk, xr * self.s["yre"] + xi * self.s["yim"], xr)
        oq = np.where(lk, -xr * self.s["yim"] + xi * self.s["yre"], xi)
        return xr, xi, oi, oq, ops

    def fallback(self, I, Q):
        """C:134-136 for the rows not locked at the block's end: AM shifter and image filter (I, Q: [R, 128], in place)."""
        fb = ~self.s["locked"]
        inc = F32(-6890.0) * (TWO_PI / FS)
        ph = self.phase_am.copy()
        for n in range(N_BLOCK):
            c, s = lut_cos(ph), lut_sin(ph)
            ti, tq = I[:, n].copy(), Q[:, n].copy()
            I[fb, n], Q[fb, n] = (ti * c - tq * s)[fb], (tq * c + ti * s)[fb]
            ph = ph + inc
            ph = np.where(ph > TWO_PI, ph - TWO_PI, np.where(ph.astype(F64) < 0.0, ph + TWO_PI, ph))
        self.phase_am = np.where(fb, ph, self.phase_am)
        si, sq = self.img_i.copy(), self.img_q.copy()
        for n in range(N_BLOCK):
            I[:, n] = np.where(fb, biquad(AM_IMAGE, si, I[:, n]), I[:, n])
            Q[:, n] = np.where(fb, biquad(AM_IMAGE, sq, Q[:, n]), Q[:, n])
        self.img_i[:, :, fb], self.img_q[:, :, fb] = si[:, :, fb], sq[:, :, fb]

    def block(self, I, Q, hook=None, b=0):
        """One block; hook(model, n, I, Q) may rewrite I[:, n], Q[:, n] (the blanker's output) before sample n."""
        I, Q = f32(I).copy(), f32(Q).copy()
        self.blanker(I, Q)
        taps = dict(if_i=np.empty_like(I), if_q=np.empty_like(Q), dm_i=np.empty_like(I), dm_q=np.empty_like(Q),
                    ok=np.empty(I.shape, bool))  # ok: the lane's own fast-path predicate (its vote)
        for n in range(N_BLOCK):
            if hook is not None:
                hook(self, b * N_BLOCK + n, I, Q, n)
            xr, xi, oi, oq, ops = self.step(I[:, n], Q[:, n])
            taps["if_i"][:, n], taps["if_q"][:, n], taps["dm_i"][:, n], taps["dm_q"][:, n] = xr, xi, oi, oq
            taps["ok"][:, n] = ops["ok"]
        self.fallback(taps["dm_i"], taps["dm_q"])
        return taps

    def status(self):
        return dict(pll_f=self.s["freq"].copy(), locked=self.s["locked"].copy(), nb_avg=self.nb_avg.copy(),
                    nb_hit=self.nb_hit.copy())


def model_run(I, Q, nb_on, nb_thr, mut=(), hook=None):
    """Runs the model over [R, S] planes: (taps {name: [R, S]}, status per block {name: [n_blocks, R]})."""
    R, ns = I.shape
    m = Model(R, nb_on, nb_thr, mut)
    taps, st = {}, {}
    for b in range(ns // N_BLOCK):
        z = slice(b * N_BLOCK, (b + 1) * N_BLOCK)
        t = m.block(I[:, z], Q[:, z], hook, b)
        for k, v in t.items():
            taps.setdefault(k, []).append(v)
        for k, v in m.status().items():
            st.setdefault(k, []).append(v)
    return {k: np.concatenate(v, 1) for k, v in taps.items()}, {k: np.array(v) for k, v in st.items()}


# ---------------------------------------------------------------- placing knife edges
def _nudge(x, k):
    """x moved by k floats (k an integer array)."""
    b = f32(x).view(np.int32).astype(np.int64)
    key = np.where(b < 0, -(b & 0x7FFFFFFF), b) + k
    return np.where(key < 0, (-key) | (1 << 31), key).astype(np.uint32).view(F32)


G_IF = F64(np.prod(IF_AM[:, 0].astype(F64)))  # d IF[n] / d x[n]: the cascade's direct feed-through


def _rail(st, x_now, target, K):
    """Inputs around the one that moves the IF output of this sample to `target`, and their IF outputs (unique)."""
    nat = F64(biquad_peek(IF_AM, st, f32(x_now)))
    c = F32(F64(x_now) + (F64(target) - nat) / G_IF)
    xs = _nudge(np.full(2 * K + 1, c), np.arange(-K, K + 1))
    ys = biquad_peek(IF_AM, st[..., None], xs)
    ys, first = np.unique(ys, return_index=True)
    return xs[first], ys


def _inv_poly(e):
    z = np.clip(e, -1.0, 1.0)
    for _ in range(40):
        f = (0.97239411 - 0.19194795 * z * z) * z - e
        z = z - f / (0.97239411 - 3 * 0.19194795 * z * z)
    return z


# The PLL rows, as the receiver groups them: SAM channels without blanker fill 32-lane warps in channel order, and one
# all-lanes vote per sample decides whether a warp takes the fast path.  A lane whose own guard fails sends its whole warp
# down the general path, so the rows are laid out warp by warp: the rows whose decisions are general-path ones anyway
# (dr < 0 ties, zero operands, ph0 == +0) share a warp, the fast-path edges sit in warps of live tones whose vote passes at
# every placed sample (test_emu_pll_edges.py checks it on the model), the ties that disturb their loop for a while come
# late in their warps, and the tiny-amplitude row, whose |di| is below 2^-60 on most samples, is alone in the last warp.
# Each entry: (target, signal kind, count); "fill" rows carry no placed sample.  Targets marked `try` are searched on
# several rows and need only MIN_FOUND of them: whether a loop reaches them depends on the parity its phase settles on.
WARPS = [
    [("tie_np", "tone", 2), ("tie_nn", "tone", 2), ("dr0_p", "tone", 1), ("dr0_n", "tone", 1), ("di0", "tone", 5),
     ("ph0_zero", "c3k", 8)],
    [("lo_end", "lo", 5), ("lo_end_dn", "lo", 1), ("lo_end_up", "lo", 1), ("wrap_up_dn", "tone", 1), ("tie_pp", "tone", 1)],
    [("lo_mid", "lo", 5), ("wrap_lo", "neg", 1), ("tiny_di", "small", 2), ("tie_pp", "tone", 1)],
    [("hi_end", "hi", 5), ("hi_end_dn", "hi", 1), ("hi_end_up", "hi", 1), ("big_dr", "big", 1), ("big_dr_up", "big", 1),
     ("tie_pn", "tone", 1)],
    [("hi_mid", "hi", 5), ("tie_pn", "tone", 1)],
    [("cos_wrap", "c3k", 8), ("cos_wrap_dn", "c3k", 8), ("wrap_up", "c3k", 8)],  # cos_wrap_dn: searched, not reached
    [("tiny_di_dn", "tiny", 1)],
]
TRY = {"ph0_zero": 2, "cos_wrap": 4, "cos_wrap_dn": 0, "wrap_up": 2}  # target -> MIN_FOUND
# targets whose placed sample must see the warp's other lanes pass the vote: the fast path decides them, or would under a
# mutation of its guard (dr >= |di|, dr <= 2^60, |di| >= 2^-64)
FAST = ("lo_end", "lo_end_dn", "lo_end_up", "lo_mid", "hi_end", "hi_end_dn", "hi_end_up", "hi_mid", "wrap_up_dn", "wrap_lo",
        "tiny_di", "tiny_di_dn", "big_dr", "big_dr_up", "tie_pp", "tie_pn", "cos_wrap")
LATE = ("tie_pp", "tie_pn")  # searched from block LATE_BLOCK on, after the other edges of their warp
LATE_BLOCK = 19
# the blanker's knife edges: (ring scan, in-block position, offset in floats, threshold) -- first scan: the block is B-1
# (ring positions 128..255), second scan: it is B-2 (78..127); None = 10 dB (setNoiseBlankerThresholdDb), else the
# value given to setNoiseBlankerThreshold.  Each is placed on two rows; build() fails unless every one is met on at
# least one of them (some averages are values the one-step square root cannot reach).
NB_TARGETS = [(scan, pos, off, thr) for thr in (None, 2.5)
              for scan, pos in (("first", 0), ("first", 127), ("first", 40), ("second", 78), ("second", 127), ("second", 100))
              for off in (0, 1)]
NB_COPIES = 2
EDGE_BLOCK = 12  # the knife edges sit in blocks EDGE_BLOCK .. EDGE_BLOCK + 2 (adaptive ones up to 9 blocks later)
N_BLOCKS = 24
LANES = 32
BIG = 2.0 ** 60


def _signal(kind, ns, rng):
    t = np.arange(ns, dtype=F64)
    w = 2.0 * np.pi / float(FS)
    f = {"tone": 6890.0, "neg": -6890.0, "tiny": 6890.0, "small": 6890.0, "big": 6890.0, "lo": 5890.0, "hi": 7890.0,
         "nb": 6890.0, "c3k": 3000.0}[kind]
    f += rng.uniform(-0.5, 0.5) if kind in ("lo", "hi") else rng.uniform(-20.0, 20.0)
    amp = {"tiny": 3e-18, "small": 2.0 ** -40, "big": 0.4 * BIG}.get(kind, 0.25)
    am = 0.0 if kind == "big" else 0.3  # the large rows keep dr below 2^60 on every sample
    x = amp * (1.0 + am * np.cos(w * rng.uniform(300, 900) * t)) * np.exp(1j * (w * f * t + rng.uniform(0, 2 * np.pi)))
    x = x + amp * 0.02 * (rng.standard_normal(ns) + 1j * rng.standard_normal(ns))
    return x.real.astype(F32), x.imag.astype(F32)


def _want(name, ops):
    """Boolean mask over candidate ops: the placed relation holds exactly (or one float off, as the name says)."""
    dr, di, ph0, freq = ops["dr"], ops["di"], ops["ph0"], ops["freq"]
    nx = lambda v, d: np.nextafter(F32(v), F32(np.inf) if d > 0 else F32(-np.inf))
    if name.startswith("tie_"):
        sr, si = name[4], name[5]
        return ((dr > 0) if sr == "p" else (dr < 0)) & ((di > 0) if si == "p" else (di < 0)) & (np.abs(dr) == np.abs(di))
    if name == "dr0_p":
        return (dr == 0) & ~np.signbit(dr) & (di > 0)
    if name == "dr0_n":
        return (dr == 0) & ~np.signbit(dr) & (di < 0)
    if name == "di0":
        return (di == 0) & (dr < 0)
    if name == "wrap_up":
        return ph0 == PI_UP
    if name == "wrap_up_dn":
        return (ph0 == PI_DN) & ops["ok"]
    if name == "wrap_lo":
        return ph0 == -PI_DN
    if name == "ph0_zero":
        return (ph0 == 0) & ~np.signbit(ph0)
    if name == "big_dr":
        return (dr == F32(BIG)) & ops["ok"]
    if name == "big_dr_up":
        return (dr == nx(BIG, 1)) & (dr > np.abs(di)) & (np.abs(di) >= F32(2.0 ** -60))
    if name == "cos_wrap":
        return (ops["ph2"] == HALF_DN) & ops["ok"]
    if name == "cos_wrap_dn":
        return (ops["ph2"] == nx(HALF_DN, -1)) & ops["ok"]
    if name == "tiny_di":
        return (np.abs(di) == F32(2.0 ** -60)) & (dr > np.abs(di))
    if name == "tiny_di_dn":
        return (np.abs(di) == nx(2.0 ** -60, -1)) & (dr > np.abs(di))
    if name[:3] in ("lo_", "hi_"):
        v = LOCK_LO if name.startswith("lo") else LOCK_HI
        if name.endswith("_dn"):
            v = nx(v, -1)
        elif name.endswith("_up"):
            v = nx(v, 1)
        return freq == v
    raise KeyError(name)


def _target_x(name, s, r, mag):
    """The (IF_I, IF_Q) in double that puts the operands of row r near the target, or None when this sample cannot."""
    yre, yim = F64(s["yre"][r]), F64(s["yim"][r])
    d0, prev, phase, freq = F64(s["d0"][r]), F64(s["prev"][r]), F64(s["phase"][r]), F64(s["freq"][r])
    if abs(yre) + abs(yim) < 0.5:
        return None
    def err_for_filt(filt):
        return (filt - F64(B1) * d0) / F64(B0) - d0
    if name.startswith("tie_"):
        w = {"pp": (1, 1), "pn": (1, -1), "np": (-1, 1), "nn": (-1, -1)}[name[4:6]]
        dr, di = w[0] * mag, w[1] * mag
    elif name == "dr0_p":
        dr, di = 0.0, mag
    elif name == "dr0_n":
        dr, di = 0.0, -mag
    elif name == "di0":
        dr, di = -mag, 0.0
    elif name == "tiny_di":
        dr, di = mag, 2.0 ** -60 * (1 if r % 2 else -1)
    elif name == "tiny_di_dn":
        dr, di = mag, 2.0 ** -60 * (1 if r % 2 else -1)
    elif name.startswith("big_dr"):
        dr, di = BIG, 0.1 * BIG
    else:
        if name.startswith("wrap_up"):
            ph_t = F64(PI_UP)
        elif name.startswith("wrap_lo"):
            ph_t = -F64(PI_DN)
        elif name == "ph0_zero":
            ph_t = 0.0
        elif name.startswith("cos_wrap"):
            ph_t = F64(HALF_DN)
        else:
            ph_t = None
        if ph_t is not None:
            filt = 2.0 * (ph_t - phase) - prev
        else:
            v = float(LOCK_LO if name.startswith("lo") else LOCK_HI)
            filt = (v - F64(ALPHA) * freq) / (F64(BETA) * F64(FCONV))
        e = err_for_filt(filt)
        if abs(e) > 0.7:
            return None
        z = _inv_poly(e)
        dr, di = mag, mag * z
    # x = (dr + j di) * y / |y|^2
    n2 = yre * yre + yim * yim
    return (dr * yre - di * yim) / n2, (dr * yim + di * yre) / n2


def _search(m, r, name, xi_now, xq_now, K):
    """Candidate (I[n], Q[n]) of row r for target `name` at this sample, or None."""
    s = m.s
    mag = float(np.hypot(F64(biquad_peek(IF_AM, m.if_i[..., r], f32(xi_now))), F64(biquad_peek(IF_AM, m.if_q[..., r], f32(xq_now)))))
    if name.startswith("tiny_di"):
        mag = max(mag, 4.0 * 2.0 ** -60)
    tx = _target_x(name, s, r, mag)
    if tx is None:
        return None
    xs_i, ys_i = _rail(m.if_i[..., r], xi_now, tx[0], K)
    xs_q, ys_q = _rail(m.if_q[..., r], xq_now, tx[1], K)
    # nearest 96 values of each rail
    if name[:4] in ("wrap", "cos_", "ph0_") or name[:3] in ("lo_", "hi_"):
        # the error must fall into one step of the loop filter's accumulator (~4e-6 rad): a few IF_I values, every IF_Q
        ki = np.argsort(np.abs(ys_i.astype(F64) - tx[0]))[:6]
        kq = np.arange(len(ys_q))
    else:
        ki = np.argsort(np.abs(ys_i.astype(F64) - tx[0]))[:96]
        kq = np.argsort(np.abs(ys_q.astype(F64) - tx[1]))[:96]
    XR, XI = np.meshgrid(ys_i[ki], ys_q[kq], indexing="ij")
    sr = {k: v[r] for k, v in s.items()}
    _, ops = sam_sample(sr, XR, XI)
    ok = _want(name, ops)
    if not ok.any():
        return None
    a, b = np.argwhere(ok)[0]
    return xs_i[ki[a]], xs_q[kq[b]]


def layout():
    """[(target, kind)] of the PLL rows, warp by warp, each warp but the last filled to 32 lanes with live tones."""
    rows = []
    for k, w in enumerate(WARPS):
        mine = [(name, kind) for name, kind, n in w for _ in range(n)]
        assert len(mine) <= LANES
        if k < len(WARPS) - 1:
            mine += [("fill", "tone")] * (LANES - len(mine))
        rows += mine
    return rows


def build(seed=7, n_blocks=N_BLOCKS):
    """(I, Q, events, layout) of the case: float32 planes, SAM mode; the PLL rows (layout(), blanker off) first, then the
    blanker rows.  layout: dict(rows=[target per row; "fill" / "nb"], at=[placed sample per row, -1 for none],
    nb=[NB target per row or None], nb_on, thr, warp=[warp of each PLL row])."""
    rng = np.random.default_rng(seed)
    plan = layout()
    names = [n for n, _ in plan]
    ns = n_blocks * N_BLOCK
    I, Q = [], []
    for _, kind in plan:
        i, q = _signal(kind, ns, rng)
        I.append(i); Q.append(q)
    nb_rows = [t for t in NB_TARGETS for _ in range(NB_COPIES)]
    for t in nb_rows:
        i, q = _signal("nb", ns, rng)
        I.append(i); Q.append(q)
    I, Q = np.array(I), np.array(Q)
    R, npll = len(I), len(names)
    nb_on = np.arange(R) >= npll
    thr = np.array([THR_10DB] * npll + [THR_10DB if t[3] is None else F32(t[3]) for t in nb_rows], F32)
    at = np.full(R, -1)
    # the blanker's edges first: they depend on the input alone
    for k, (scan, pos, off, _) in enumerate(nb_rows):
        r = npll + k
        for blk in range(EDGE_BLOCK + k % 3, N_BLOCKS - 3, 3):  # a block whose running average the magnitudes can meet
            try:
                at[r] = _place_nb(I, Q, r, thr[r], blk, pos, scan, off)
                break
            except RuntimeError:
                continue
    met = {t for t, a in zip(nb_rows, at[npll:]) if a >= 0}
    assert met == set(NB_TARGETS), "blanker targets met on no row: %s" % (set(NB_TARGETS) - met)
    nb_names = ["nb" if a >= 0 else "nb_fill" for a in at[npll:]]
    # the PLL's edges: one model pass, each row searched at the first suitable sample from its start
    start = np.full(R, -1)
    for r, name in enumerate(names):
        b0 = LATE_BLOCK + r % 3 if name in LATE else EDGE_BLOCK + r % 3
        if "_end" in name:
            start[r] = b0 * N_BLOCK + N_BLOCK - 1
        elif name.endswith("_mid"):
            start[r] = b0 * N_BLOCK + 40 + 7 * (r % 5)
        elif name != "fill":
            start[r] = b0 * N_BLOCK + (r * 13) % 64
    pending = {r for r in range(npll) if names[r] != "fill"}

    def hook(m, n, Ib, Qb, j):
        for r in [r for r in pending if start[r] <= n]:
            if "_end" in names[r] and j != N_BLOCK - 1:
                continue
            got = _search(m, r, names[r], Ib[r, j], Qb[r, j], 4000)
            if got is not None:
                Ib[r, j], Qb[r, j] = got
                I[r, n], Q[r, n] = got
                at[r] = n
                pending.discard(r)
            elif n > start[r] + 1200 or n == ns - 1:
                if names[r] not in TRY:
                    raise RuntimeError("no knife edge for row %d (%s)" % (r, names[r]))
                pending.discard(r)

    model_run(I, Q, nb_on, thr, hook=hook)
    for name, need in TRY.items():
        found = [r for r in range(npll) if names[r] == name and at[r] >= 0]
        assert len(found) >= need, (name, len(found))
    names = [n if (n == "fill" or at[r] >= 0) else "fill" for r, n in enumerate(names)]  # rows whose loop never got there
    ev = []
    for r in range(R):
        ev += [(r, 0, "setDemodMode", 5), (r, 0, "enableNoiseBlanker" if nb_on[r] else "disableNoiseBlanker")]
        t = nb_rows[r - npll][3] if r >= npll else None
        ev += [(r, 0, "setNoiseBlankerThresholdDb", 10.0)] if t is None else [(r, 0, "setNoiseBlankerThreshold", float(t))]
        big = r < npll and plan[r][1] == "big"
        ev += [(r, 0, "disableAGC")] if big else [(r, 0, "setAGCmode", 2)]
        ev += [(r, 0, "enableAudioFilter"), (r, 0, "setAudioFilter", 0), (r, 0, "setMute", 0)]
    lay = dict(rows=names + nb_names, at=at, nb=[None] * npll + nb_rows, nb_on=nb_on, thr=thr,
               warp=np.arange(npll) // LANES, kind=[k for _, k in plan] + ["nb"] * len(nb_rows))
    return I, Q, ev, lay


def nb_scan(I, Q, r, upto_block):
    """(call, ring position, mag, avg before) of every scan step of row r up to the call for block `upto_block`."""
    out = []
    avg = F32(10.0)
    ri, rq = np.zeros(3 * N_BLOCK, F32), np.zeros(3 * N_BLOCK, F32)
    for b in range(upto_block + 1):
        ri[:2 * N_BLOCK], rq[:2 * N_BLOCK] = ri[N_BLOCK:].copy(), rq[N_BLOCK:].copy()
        ri[2 * N_BLOCK:], rq[2 * N_BLOCK:] = I[r, b * N_BLOCK:(b + 1) * N_BLOCK], Q[r, b * N_BLOCK:(b + 1) * N_BLOCK]
        mags = sqrt_hack(ri[78:256] * ri[78:256] + rq[78:256] * rq[78:256])
        for k, mag in enumerate(mags):
            out.append((b, 78 + k, mag, avg))
            avg = NB_ALPHA * avg + NB_BETA * mag
    return out


def _place_nb(I, Q, r, thr, blk, pos, scan, off):
    """Rewrites sample (blk, pos) of row r so that its magnitude at the chosen scan equals avg * thr (off: one float above).
    The one-step square root does not reach every float, so the sample before is moved too until avg * thr is a value it
    reaches."""
    n = blk * N_BLOCK + pos
    call = blk + (1 if scan == "first" else 2)
    ring = 128 + pos if scan == "first" else pos
    prev = I[r, n - 1]
    for attempt in range(6):
        I[r, n - 1] = _nudge(prev, 997 * attempt)
        if _try_nb(I, Q, r, thr, blk, pos, scan, off, n, call, ring):
            return n
    I[r, n - 1] = prev
    raise RuntimeError("no blanker knife edge for row %d" % r)


def _try_nb(I, Q, r, thr, blk, pos, scan, off, n, call, ring):
    steps = nb_scan(I, Q, r, call)
    first = next(k for k, (b, p, _, _) in enumerate(steps) if b == blk + 1 and p == 128 + pos)
    k_at = next(k for k, (b, p, _, _) in enumerate(steps) if b == call and p == ring)
    mags = np.array([s[2] for s in steps[first:k_at]], F32)
    a0 = steps[first][3]
    phi = np.arctan2(F64(Q[r, n]), F64(I[r, n]))
    target = F64(a0) * F64(thr) * (1.2 if scan == "second" else 1.0)
    ci, cq = F32(target * np.cos(phi)), F32(target * np.sin(phi))
    for _ in range(12):
        # I swept over 4001 floats, Q over 61: the sum of squares skips magnitudes that a neighbouring Q reaches
        xs = _nudge(np.full(4001, ci), np.arange(-2000, 2001))[:, None]
        qs = _nudge(np.full(61, cq), np.arange(-30, 31))[None, :]
        mg = sqrt_hack(xs * xs + qs * qs)
        avg = np.full(mg.shape, a0, F32)
        if scan == "second":  # the running average from the first scan of this sample to its second
            avg = NB_ALPHA * avg + NB_BETA * mg
            for mv in mags[1:]:
                avg = NB_ALPHA * avg + NB_BETA * mv
        t = avg * thr
        want = np.nextafter(t, F32(np.inf)) if off else t
        hit = np.argwhere(mg == want)
        if len(hit):
            a, b = hit[len(hit) // 2]
            I[r, n], Q[r, n] = xs[a, 0], qs[0, b]
            return True
        if mg.min() <= want.max() and mg.max() >= want.min():
            return False  # the sweep spans the threshold without meeting it: this average cannot be met
        # re-centre: bisection for the I at which the magnitude (monotone in |I|) crosses the threshold
        sgn, lo, hi = F32(np.sign(ci) or 1.0), F32(0.0), F32(4.0) * np.abs(ci)
        w = F64(want[2000, 30])
        for _ in range(60):
            mid = F32((F64(lo) + F64(hi)) / 2)
            if F64(sqrt_hack(mid * mid + cq * cq)) < w:
                lo = mid
            else:
                hi = mid
        ci = sgn * hi
    return False
