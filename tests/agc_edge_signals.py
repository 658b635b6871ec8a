"""tests/agc_edge_signals.py -- the AGC one rounding away from its decisions.

The AGC (C:404-436; RoleAgc in audiosdr_b200/csrc/sdr_pipeline.cuh) decides per sample between attack (`absval >
old_absval`), hang (`hang_ctr > 0`, then `hang_ctr--`) and release, clamps its level at 1.0, and reports `AGCisActive()`,
`(double)_agc_gain < 0.99` (C:429).  The kernel restates each decision in float form, selects the table of a lane from
shared memory or, when its group holds more than four distinct tables, from global memory (SdrGroup::lut_ids,
GF_LUT_GLOBAL), and carries the hang counter from one launch to the next.  Ordinary stimuli meet none of these edges
exactly.  This module

  * restates agc_run in numpy float32 in the oracle's operand order (`model_run`): the level (2*carrier in AM mode, |v|
    otherwise), the clamp, attack / hang / release, the `(uint16_t)(int)(absval*32767.0)` index (exact in float64), the
    table interpolation, agc_active and the output clamp.  Its input is the oracle's own `audf` tap and AM carrier, so
    nothing upstream of the AGC is restated.  The tables are not restated either (the builder calls libm expf): they come
    from SdrBatch.getAGClookup of the host emulation, host code that test_tables.py compares with the oracle.  One switch
    per kernel mutation (MUTATIONS); `no_lut_global` restates the receiver's grouping (build_groups) to know which lanes
    read a table outside the four staged ones;
  * builds one case whose rows reach each edge (`build`), checked on the oracle's taps through the model:
      - attack ties: level == old exactly with the hang counter above 1, at 1 and at 0, and one float either side --
        on the AM level path (block-constant 2*carrier: attack times of 1e-4 ms give a_att = 0 and old == level after one
        attack; short non-zero attack times converge onto the level and are kept where they reach it exactly) and on
        the sample path of SSB and SAM rows (the clamp makes every |v| >= 1 an exact 1.0: old == 1.0 after an attack);
        the tie on the last sample of a block whose hang then runs out, before a falling carrier, is where a `>=`
        restarts the hang;
      - hang ends: hang counts 0, 1 and 2, and counts chosen so that the expiry sample (last attack + count + 1) falls
        on the first and the last sample of a tile for T = 8, 16 and 32, on a block boundary and on a call boundary of
        the tests' ragged chunks; disableAGC / enableAGC while the counter is 1 or 0;
      - AGCisActive: the table threshold searched so that the interpolant `l0 + (l1 - l0)*(k/256)` of index bucket
        (0, k) is exactly 0.99f, the float below and the float above; the carrier is set so that old falls into that
        bucket, and a long hang holds the gain across block ends.  Levels of exactly 1.0 (AM carriers above 0.5);
      - table staging: groups of LSB rows with exactly 4, 5 and 32 distinct tables, AGC-off lanes holding tables, and a
        threshold setter that moves a lane from a staged slot to the global path and back.
  * `long_case`: mode 3 (hang 88 200 samples) across many calls, the expiry placed on a block boundary and on the last
    sample of a 32-sample tile.

On the AM path the level changes only at block boundaries, so `one float either side` is met with the counter above 1
(converging attacks) and at 0, not at exactly 1.  SSB rows are covered by the builders that need no exact input (the clamp ties, hang ends, the 0.99 buckets through the
table staging rows and the hang rows); the Hilbert path is not restated.  The sample path's `level one float below old`
needs an exact |v| of 0x1.fffffep-1 after an attack to 1.0, which no row here places: on the sample path only the tie and
`level one float above old` (old converged to 1 - 2^-24) are reached.
"""
import ctypes
import math
import os
import subprocess

import numpy as np

N_BLOCK = 128
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, F64 = np.float32, np.float64
FS = F32(44100.0)
MIN_FLIPS = 4
ACT = F32(0.99)                                   # (double)g < 0.99  <=>  g < 0x1.fae148p-1f
ACT_DN = np.nextafter(ACT, F32(0))                # 0x1.fae146p-1
ACT_UP = np.nextafter(ACT, F32(2))
LSB, USB, AM, SAM = 0, 1, 4, 5
LANES, SLOTS = 32, 4
TINY_MS = 1e-4                                    # attack / release time whose coefficient is exactly 0

MUTATIONS = ["att_ge",         # 1: absv >= old
             "hang_gt1",       # 2: hang > 1u
             "reload_m1",      # 3: hang reloaded with hang_count - 1u
             "active_le",      # 4: gain <= 0.99f
             "active_below",   # 5: gain < 0x1.fae146p-1f
             "no_clamp",       # 6: the level clamp removed
             "no_lut_global",  # 7: GF_LUT_GLOBAL never set (lanes past the 4 staged tables read slot 0's)
             "save_no_hang"]   # 8: RoleAgc::save does not store hang (each launch starts from the initial 0)


def f32(x):
    return np.asarray(x, F32)


# ---------------------------------------------------------------- setters (C:551-566, 524-544; oracle ora_apply)
def _coef(ms):
    """(a, b) of agc_set_attack / agc_set_release: exp(log(0.1) / (FS * t / 1000.0)), FS * t a float product."""
    a = F32(math.exp(math.log(0.1) / (F64(FS * F32(ms)) / 1000.0)))
    return a, F32(1.0 - F64(a))


def hang_count(ms):
    """agc_set_hang: (uint32_t)(t * FS / 1000.0), t * FS a float product."""
    return int(F64(F32(ms) * FS) / 1000.0)


def hang_ms(n):
    """A setAGChangTime value whose count is n."""
    t = (n + 0.5) / 44.1
    assert hang_count(t) == n
    return t


class Params:
    """The AGC configuration of R channels, as the oracle's setters leave it."""

    def __init__(self, R):
        self.mode = np.full(R, LSB)
        self.on = np.ones(R, bool)
        self.nb = np.ones(R, bool)
        self.als = np.zeros(R, bool)
        self.sgain = np.full(R, F32(10.0))
        self.key = [(F32(-60.0), F32(0.1), F32(2.0))] * R
        a, b = _coef(5.0)
        self.a_att, self.b_att = np.full(R, a), np.full(R, b)
        a, b = _coef(500.0)
        self.a_rel, self.b_rel = np.full(R, a), np.full(R, b)
        self.hc = np.full(R, int(F64(FS) * (F64(F32(100.0)) / 1000.0)), np.int64)

    def apply(self, r, op, a0=0.0, *_):
        if op == "setDemodMode":
            self.mode[r] = int(a0)
        elif op == "enableAGC":
            self.on[r] = True
        elif op == "disableAGC":
            self.on[r] = False
        elif op == "enableNoiseBlanker":
            self.nb[r] = True
        elif op == "disableNoiseBlanker":
            self.nb[r] = False
        elif op == "enableALSfilter":
            self.als[r] = True
        elif op == "disableALSfilter":
            self.als[r] = False
        elif op == "setAGCattackTime":
            self.a_att[r], self.b_att[r] = _coef(a0)
        elif op == "setAGCreleaseTime":
            self.a_rel[r], self.b_rel[r] = _coef(a0)
        elif op == "setAGChangTime":
            self.hc[r] = hang_count(a0)
        elif op == "setAGCstaticGain":
            self.sgain[r] = F32(a0)
        elif op in ("setAGCthreshold", "setAGCslope", "setAGCkneeWidth"):
            k = list(self.key[r])
            k[("setAGCthreshold", "setAGCslope", "setAGCkneeWidth").index(op)] = F32(a0)
            self.key[r] = tuple(k)
        elif op == "setAGCmode":
            m = int(a0)
            if m == 0:
                self.on[r] = False
            elif m in (1, 2, 3):
                t = {1: (2.0, 100.0, 100.0), 2: (5.0, 250.0, 500.0), 3: (10.0, 500.0, 2000.0)}[m]
                self.a_att[r], self.b_att[r] = _coef(t[0])
                self.a_rel[r], self.b_rel[r] = _coef(t[1])
                self.hc[r] = hang_count(t[2])
                self.on[r] = True
        else:
            assert op in ("setMute", "enableAudioFilter", "disableAudioFilter", "setAudioFilter", "setALSfilterParams",
                          "setNoiseBlankerThresholdDb"), op


def events_by_block(ev, n_blocks):
    out = [[] for _ in range(n_blocks)]
    for e in sorted(ev, key=lambda e: e[1]):
        out[e[1]].append(e)
    return out


# ---------------------------------------------------------------- tables (host code, through the emulation library)
_emu, _luts = [], {}


def emu_lib():
    if not _emu:
        from audiosdr_b200 import api
        d = os.path.join(ROOT, "tests", "emu")
        subprocess.run(["make", "-s", "-C", d], check=True)
        _emu.append(api._bind(ctypes.CDLL(os.path.join(d, "libsdr_emu.so"))))
    return _emu[0]


def tables(keys):
    """{(thr, slope, knee): the 129-entry table of SdrBatch.getAGClookup} for every key."""
    want = sorted({k for k in keys if k not in _luts})
    if want:
        import audiosdr_b200 as A
        b = A.SdrBatch(len(want), _lib=emu_lib())
        calls = []
        for c, (t, s, k) in enumerate(want):
            calls += [(c, "setAGCthreshold", float(t)), (c, "setAGCslope", float(s)), (c, "setAGCkneeWidth", float(k))]
        b.configure(calls)
        for c, k in enumerate(want):
            _luts[k] = b.getAGClookup(c)
        b.close()
    return {k: _luts[k] for k in keys}


def groups(p, rows=None):
    """The receiver's groups (build_groups for a call over `rows`, channel order): lists of channel ids."""
    rows = range(len(p.mode)) if rows is None else rows
    order = [[LSB, USB, 2, 3, 6], [AM, SAM]]
    out = []
    for cls in (0, 1):
        for feat in range(8):
            cur = []
            for m in order[cls]:
                for r in rows:
                    rcls = 1 if p.mode[r] in (AM, SAM) else 0
                    f = (1 if p.nb[r] else 0) | (2 if p.als[r] else 0) | (4 if p.mode[r] == SAM else 0)
                    if rcls == cls and f == feat and p.mode[r] == m:
                        cur.append(r)
                        if len(cur) == LANES:
                            out.append(cur); cur = []
                if cls == 0 and cur:
                    out.append(cur); cur = []
            if cur:
                out.append(cur)
    return out


def staging(p):
    """Per channel: (slot 0's table key of its group, True when the lane reads its table from global memory)."""
    R = len(p.mode)
    first, glob = [None] * R, np.zeros(R, bool)
    for g in groups(p):
        ids = []
        for r in g:
            if p.key[r] not in ids and len(ids) < SLOTS:
                ids.append(p.key[r])
            glob[r] = p.key[r] not in ids
            first[r] = ids[0]
    return first, glob


# ---------------------------------------------------------------- the model
def lookup(lut, absv):
    """agc_lookup (C:483-494) on rows: lut [R, 129], absv [R]."""
    with np.errstate(invalid="ignore", over="ignore"):
        v = np.trunc(absv.astype(F64) * 32767.0)
    v = np.where(np.isfinite(v) & (np.abs(v) < 2.0 ** 31), v, -2.0 ** 31).astype(np.int64) & 0xFFFF
    idx = np.minimum(v >> 8, 127)
    d = (v & 0xFF).astype(F32) / F32(256.0)
    rr = np.arange(len(lut))
    l0, l1 = lut[rr, idx], lut[rr, idx + 1]
    return l0 + (l1 - l0) * d


def call_starts(ev, n_blocks, chunks):
    """The first block of each call harness.run_batch makes (a call never spans an event's block)."""
    blocks = sorted({e[1] for e in ev})
    out, pos, k = [], 0, 0
    while pos < n_blocks:
        nxt = next((b for b in blocks if b > pos), n_blocks)
        sz = min(chunks[k % len(chunks)], n_blocks - pos, max(nxt - pos, 1))
        out.append(pos)
        pos += sz
        k += 1
    return out


def model_run(audf, carrier, ev, mut=(), calls=(7, 1, 13)):
    """agc_run over [R, S] audio (the oracle's audf tap) with the AM carrier after each block ([n_blocks, R]).
    Returns (agc [R, S], per block {gain, active, old, hang} [n_blocks, R], trace {level, old, hang, att, upd} [R, S]: the
    operands of each sample's decision, before it)."""
    R, ns = audf.shape
    nb = ns // N_BLOCK
    p = Params(R)
    evb = events_by_block(ev, nb)
    starts = set(call_starts(ev, nb, calls)) if "save_no_hang" in mut else set()
    old, gain = np.zeros(R, F32), np.zeros(R, F32)
    hang, active = np.zeros(R, np.int64), np.ones(R, bool)
    out = np.empty((R, ns), F32)
    tr = dict(level=np.empty((R, ns), F32), old=np.empty((R, ns), F32), hang=np.empty((R, ns), np.int64),
              att=np.empty((R, ns), bool), upd=np.empty((R, ns), bool))
    per = {k: [] for k in ("gain", "active", "old", "hang")}
    lut = None
    for b in range(nb):
        for e in evb[b]:
            p.apply(e[0], *e[2:])
        if lut is None or evb[b]:
            keys = list(p.key)
            if "no_lut_global" in mut:
                first, glob = staging(p)
                keys = [first[r] if glob[r] else keys[r] for r in range(R)]
            t = tables(keys)
            lut = np.array([t[k] for k in keys], F32)
        if b in starts:
            hang = np.where(p.on, 0, hang)
        on = p.on
        hc = p.hc - (1 if "reload_m1" in mut else 0)
        hc = np.where(hc < 0, 0xFFFFFFFF, hc)
        for j in range(N_BLOCK):
            n = b * N_BLOCK + j
            v = audf[:, n]
            level = np.where(p.mode == AM, F32(2.0) * carrier[b], np.abs(v))
            if "no_clamp" not in mut:
                level = np.where(level > F32(1.0), F32(1.0), level)
            att = (level >= old) if "att_ge" in mut else (level > old)
            hanging = ~att & (hang > (1 if "hang_gt1" in mut else 0))
            upd = att | ~hanging
            with np.errstate(over="ignore", invalid="ignore"):
                sm = np.where(att, p.a_att * old + p.b_att * level, p.a_rel * old + p.b_rel * level)
            g = lookup(lut, sm)
            tr["level"][:, n], tr["old"][:, n], tr["hang"][:, n], tr["att"][:, n], tr["upd"][:, n] = level, old, hang, att, upd
            old = np.where(on & upd, sm, old)
            gain = np.where(on & upd, g, gain)
            hang = np.where(on, np.where(att, hc, np.where(hanging, hang - 1, hang)), hang)
            with np.errstate(over="ignore", invalid="ignore"):
                o = gain * p.sgain * v
            o = np.where(o > F32(1.0), F32(1.0), np.where(o < F32(-1.0), F32(-1.0), o))
            out[:, n] = np.where(on, o, v)
        if "active_le" in mut:
            act = gain <= ACT
        elif "active_below" in mut:
            act = gain < ACT_DN
        else:
            act = gain < ACT
        active = np.where(on, act, active)
        for k, x in (("gain", gain), ("active", active), ("old", old), ("hang", hang)):
            per[k].append(x.copy())
    return out, {k: np.array(v) for k, v in per.items()}, tr


# ---------------------------------------------------------------- the oracle's taps
def oracle_taps(I, Q, ev, rows=None):
    """Each row stepped through oracle_lib.Channel: ({audf, agc} [R, S], status vector after each block [n_blocks, R, 16])."""
    from multiprocessing.pool import ThreadPool
    from oracle import oracle_lib
    R, ns = I.shape
    rows = list(range(R)) if rows is None else list(rows)
    nb = ns // N_BLOCK
    ia, ig = oracle_lib.TAPS.index("audf"), oracle_lib.TAPS.index("agc")
    audf, agc = np.empty((len(rows), ns), F32), np.empty((len(rows), ns), F32)
    st = np.empty((nb, len(rows), oracle_lib.N_STATUS if hasattr(oracle_lib, "N_STATUS") else 16), F32)
    evs = sorted(range(len(ev)), key=lambda i: (ev[i][1], i))

    def one(k):
        r = rows[k]
        mine = [ev[i] for i in evs if ev[i][0] == r]
        ch, ei = oracle_lib.Channel(), 0
        for b in range(nb):
            while ei < len(mine) and mine[ei][1] <= b:
                ch.apply(mine[ei][2], *mine[ei][3:])
                ei += 1
            z = slice(b * N_BLOCK, (b + 1) * N_BLOCK)
            ch.update(I[r, z], Q[r, z])
            audf[k, z], agc[k, z] = ch.taps[ia], ch.taps[ig]
            st[b, k] = ch.status()

    with ThreadPool(8) as pool:
        pool.map(one, range(len(rows)))
    return dict(audf=audf, agc=agc), st


def carrier_of(st):
    return st[:, :, 6].astype(F32)


def run(I, Q, ev, mut=(), calls=(7, 1, 13)):
    taps, st = oracle_taps(I, Q, ev)
    return model_run(taps["audf"], carrier_of(st), ev, mut, calls)


# ---------------------------------------------------------------- signals
def _tone(ns, f, amp, rng, noise=0.01, env=None):
    t = np.arange(ns, dtype=F64)
    w = 2.0 * np.pi / float(FS)
    a = amp if env is None else amp * env
    x = a * np.exp(1j * (w * f * t + rng.uniform(0, 2 * np.pi)))
    x = x + amp * noise * (rng.standard_normal(ns) + 1j * rng.standard_normal(ns))
    return x.real.astype(F32), x.imag.astype(F32)


def _steps(ns, n_hi, n_lo, lo, phase):
    """Block-wise amplitude steps: n_hi blocks at 1, n_lo blocks at `lo` (rising then falling carriers)."""
    b = (np.arange(ns) // N_BLOCK + phase) % (n_hi + n_lo)
    return np.where(b < n_hi, 1.0, lo)


def _base_events(r, mode, att_ms, rel_ms, hang, thr=None, audio=None, als=False, agc_mode=None):
    ev = [(r, 0, "setDemodMode", mode), (r, 0, "disableNoiseBlanker"), (r, 0, "setMute", 0)]
    ev += [(r, 0, "enableAudioFilter"), (r, 0, "setAudioFilter", audio)] if audio is not None else [(r, 0, "disableAudioFilter")]
    if als:
        ev += [(r, 0, "enableALSfilter")]
    if agc_mode is not None:
        ev += [(r, 0, "setAGCmode", agc_mode)]
    if att_ms is not None:
        ev += [(r, 0, "setAGCattackTime", att_ms)]
    if rel_ms is not None:
        ev += [(r, 0, "setAGCreleaseTime", rel_ms)]
    if hang is not None:
        ev += [(r, 0, "setAGChangTime", hang)]
    if thr is not None:
        ev += [(r, 0, "setAGCthreshold", float(thr))]
    return ev


N_BLOCKS = 40
CHUNKS = (7, 1, 13)                       # the schedule tests' calls: the call-boundary targets are placed on them
ATT_AM = [TINY_MS, 0.01, 0.02, 0.03, 0.05]
HC_TIE = [3, 126, 127, 128]               # hang counts: a tie on the block's last sample with the counter at 0, 0, 1, 2
EXPIRY_OFFSETS = {0: "block / tile first, every T", 127: "block / tile last, every T", 31: "T=32 last", 32: "T=32 first",
                  15: "T=16 last", 48: "T=16 first", 7: "T=8 last", 8: "T=8 first"}
THRS = [F32(-72.0 + 1.5 * k) for k in range(34)]   # staging tables: distinct thresholds


def _search_thr(target, k):
    """A threshold whose table interpolates lut[0] .. lut[1] at fraction k/256 to exactly `target`."""
    d = F32(k) / F32(256.0)
    lo, hi = -80.0, -20.0
    for it in range(4):
        grid = [F32(x) for x in np.linspace(lo, hi, 801)]
        t = tables([(g, F32(0.1), F32(2.0)) for g in grid])
        gains = np.array([F32(1.0) + (t[(g, F32(0.1), F32(2.0))][1] - F32(1.0)) * d for g in grid], F32)
        hit = np.flatnonzero(gains == target)
        if len(hit):
            return grid[hit[len(hit) // 2]]
        # gains fall as the threshold rises (lut[1] grows): bracket the target
        above = np.flatnonzero(gains > target)
        below = np.flatnonzero(gains < target)
        if not len(above) or not len(below):
            raise RuntimeError("no threshold for %r at k=%d" % (target, k))
        i = above.max() if above.max() < below.min() else below.max()
        lo, hi = float(grid[max(i - 2, 0)]), float(grid[min(i + 3, 800)])
    # the bracket is a few floats wide: walk them
    x = F32(lo)
    while x <= F32(hi):
        g = F32(1.0) + (tables([(x, F32(0.1), F32(2.0))])[(x, F32(0.1), F32(2.0))][1] - F32(1.0)) * d
        if g == target:
            return x
        x = np.nextafter(x, F32(0))
    raise RuntimeError("no threshold for %r at k=%d" % (target, k))


def _scale_to(I, Q, ev, r, want_carrier, blocks=12):
    """Rescales row r so that its AM carrier settles on want_carrier (the chain is linear in the input amplitude)."""
    for _ in range(3):
        _, st = oracle_taps(I[r:r + 1, :blocks * N_BLOCK], Q[r:r + 1, :blocks * N_BLOCK], [(0,) + e[1:] for e in ev if e[0] == r])
        c = float(st[-1, 0, 6])
        I[r] = (I[r].astype(F64) * (want_carrier / c)).astype(F32)
        Q[r] = (Q[r].astype(F64) * (want_carrier / c)).astype(F32)


def layout():
    """[(kind, params)] of the case's rows, in channel order."""
    rows = []
    for att in ATT_AM:                                   # AM ties: block-constant levels, rising then falling carriers
        for hc in HC_TIE:
            for rel in (TINY_MS, 1.0):
                rows.append(("am_tie", dict(att=att, hc=hc, rel=rel)))
    for amp in (0.7, 1.2):                               # AM levels of exactly 1.0 (carrier above 0.5)
        for hc in (2, 127):
            rows.append(("am_clamp", dict(att=TINY_MS, hc=hc, rel=1.0, amp=amp)))
    for target, name in ((ACT, "act_eq"), (ACT_DN, "act_dn"), (ACT_UP, "act_up")):  # AGCisActive at 0.99
        for k in (3, 3, 5, 5):
            rows.append((name, dict(target=target, k=k)))
    for att in (TINY_MS, 0.01, 0.05):                    # sample-path ties at the clamp: SSB and SAM rows
        for hc in (0, 1, 2, 30):
            rows.append(("ssb_clamp", dict(att=att, hc=hc, rel=TINY_MS if hc % 2 else 1.0)))
    for hc in (0, 1, 2, 40):
        rows.append(("sam_clamp", dict(att=TINY_MS, hc=hc, rel=1.0)))
    for hc in (0, 0, 1, 1, 2, 2):                        # short hangs: expiries everywhere; half the rows with ALS on
        rows.append(("hang_short", dict(hc=hc)))
    for off in EXPIRY_OFFSETS:                           # long hangs, expiry placed
        for copy in range(2):
            rows.append(("hang_at", dict(off=off, copy=copy)))
    for g in range(3):                                   # table staging: groups of 4, 5 and 32 distinct tables
        for lane in range(LANES):
            rows.append(("stage", dict(group=g, lane=lane)))
    return rows


STAGE_MOVE = (0, 9, 12, 24)   # (group, lane, block to the 5th table, block back): a staged lane to the global path and back


def _stage_thr(g, lane):
    if g == 0:
        return THRS[lane % 4]
    if g == 1:
        return THRS[10 + min(lane, 4)]
    return THRS[lane]


def build(seed=11, n_blocks=N_BLOCKS):
    """(I, Q, events, layout) of the case; layout: dict(rows=[kind], params=[dict], toggles=[(row, block, hang)])."""
    rng = np.random.default_rng(seed)
    plan = layout()
    R, ns = len(plan), n_blocks * N_BLOCK
    I, Q = np.zeros((R, ns), F32), np.zeros((R, ns), F32)
    ev = []
    for r, (kind, prm) in enumerate(plan):
        if kind == "am_tie":
            env = _steps(ns, 3, 3, rng.uniform(0.5, 0.7), r % 6)
            I[r], Q[r] = _tone(ns, 6890.0 + rng.uniform(-30, 30), rng.uniform(0.05, 0.3), rng, 0.005, env)
            ev += _base_events(r, AM, prm["att"], prm["rel"], hang_ms(prm["hc"]))
        elif kind == "am_clamp":
            env = _steps(ns, 4, 4, 0.3, r % 8)
            I[r], Q[r] = _tone(ns, 6890.0, prm["amp"], rng, 0.005, env)
            ev += _base_events(r, AM, prm["att"], prm["rel"], hang_ms(prm["hc"]))
        elif kind.startswith("act_"):
            I[r], Q[r] = _tone(ns, 6890.0 + rng.uniform(-30, 30), 1e-4, rng, 0.002)
            thr = _search_thr(prm["target"], prm["k"])
            prm["thr"] = thr
            ev += _base_events(r, AM, TINY_MS, 1.0, 1000.0, thr=thr)
            _scale_to(I, Q, ev, r, (prm["k"] + rng.uniform(0.3, 0.7)) / 32767.0 / 2.0)
        elif kind == "ssb_clamp":
            env = 0.4 + 0.8 * (0.5 + 0.5 * np.sin(2 * np.pi * np.arange(ns) / rng.uniform(900, 2500)))
            I[r], Q[r] = _tone(ns, 5390.0 + rng.uniform(200, 900), 1.6, rng, 0.01, env)
            ev += _base_events(r, USB, prm["att"], prm["rel"], hang_ms(prm["hc"]))
        elif kind == "sam_clamp":
            t = np.arange(ns)
            env = 1.0 + 0.9 * np.sin(2 * np.pi * rng.uniform(300, 900) * t / float(FS))
            I[r], Q[r] = _tone(ns, 6890.0, 2.5, rng, 0.01, env)
            ev += _base_events(r, SAM, prm["att"], prm["rel"], hang_ms(prm["hc"]))
        elif kind == "hang_short":
            I[r], Q[r] = _tone(ns, 5390.0 + rng.uniform(200, 2000), 0.2, rng, 0.3)
            ev += _base_events(r, USB, 0.5, 1.0, hang_ms(prm["hc"]), audio=4, als=bool(r % 2))
        elif kind == "hang_at":
            env = np.clip((np.arange(ns) - 8 * N_BLOCK) / (4.0 * N_BLOCK), 0, 1) * (np.arange(ns) < 13 * N_BLOCK)
            env = env + 0.02
            I[r], Q[r] = _tone(ns, 5390.0 + rng.uniform(300, 1200), 0.4, rng, 0.005, env)
            ev += _base_events(r, USB, 0.2, 1.0, 1000.0)
        elif kind == "stage":
            g, lane = prm["group"], prm["lane"]
            I[r], Q[r] = _tone(ns, 7890.0 - rng.uniform(100, 1500), rng.uniform(0.05, 0.5), rng, 0.05)
            ev += _base_events(r, LSB, None, None, None, thr=_stage_thr(g, lane), agc_mode=1)
            if g == 1 and lane < 3:
                ev += [(r, 0, "disableAGC")]
            if (g, lane) == STAGE_MOVE[:2]:
                ev += [(r, STAGE_MOVE[2], "setAGCthreshold", float(THRS[33])), (r, STAGE_MOVE[3], "setAGCthreshold",
                                                                                 float(_stage_thr(g, lane)))]
    lay = dict(rows=[k for k, _ in plan], params=[p for _, p in plan], toggles=[])
    # disableAGC / enableAGC while the counter is 1 and while it is 0 (short-hang rows with counts 1 and 2)
    short = [r for r, (k, p) in enumerate(plan) if k == "hang_short" and p["hc"] >= 1]
    agc_taps, st = oracle_taps(I, Q, ev, short)
    sub_ev = [(short.index(e[0]),) + e[1:] for e in ev if e[0] in short]
    _, _, tr = model_run(agc_taps["audf"], carrier_of(st), sub_ev)
    used = set()
    for k, (r, want) in enumerate(zip(short, (1, 0, 0, 1))):
        b = next(b for b in range(12, n_blocks - 4) if tr["hang"][k, b * N_BLOCK] == want and b not in used)
        used.add(b)
        ev += [(r, b, "disableAGC"), (r, b + 2, "enableAGC")]
        lay["toggles"].append((r, b, want))
    # the placed hangs: last attack with a long hang, then the count that puts the expiry on its target
    rows_at = [r for r, (k, _) in enumerate(plan) if k == "hang_at"]
    agc_taps, st = oracle_taps(I, Q, ev, rows_at)
    sub_ev = [(rows_at.index(e[0]),) + e[1:] for e in ev if e[0] in rows_at]
    _, _, tr = model_run(agc_taps["audf"], carrier_of(st), sub_ev)
    starts = call_starts(ev, n_blocks, CHUNKS)
    for k, r in enumerate(rows_at):
        L = int(np.flatnonzero(tr["att"][k])[-1])
        off = plan[r][1]["off"]
        bl = L // N_BLOCK + 2
        if off == 0:
            bl = next(s for s in starts if s >= bl + plan[r][1]["copy"])
        E = bl * N_BLOCK + off
        plan[r][1].update(last=L, expiry=E, hc=E - L - 1)
        ev = [e for e in ev if not (e[0] == r and e[2] == "setAGChangTime")] + [(r, 0, "setAGChangTime", hang_ms(E - L - 1))]
    ev = sorted(ev, key=lambda e: e[1])
    return I, Q, ev, lay


# ---------------------------------------------------------------- mode 3 across many calls
LONG_TARGETS = [0, 0, 31, 31]   # expiry offset in its block: a block boundary, the last sample of a 32-sample tile
LONG_HC = 88200


def long_case(seed=5):
    """(I, Q, events, layout): USB rows in AGC mode 3, one burst each, the expiry of the 88 200-sample hang placed by the
    burst's start.  layout: dict(last=[last attack], expiry=[sample])."""
    rng = np.random.default_rng(seed)
    R = len(LONG_TARGETS)
    burst = 6 * N_BLOCK
    n_blocks = (burst + 2 * N_BLOCK + LONG_HC + 4 * N_BLOCK) // N_BLOCK + 4
    ns = n_blocks * N_BLOCK
    I, Q = np.zeros((R, ns), F32), np.zeros((R, ns), F32)
    from oracle import oracle_lib
    ev, last, expiry = [], [], []
    mine = _base_events(0, USB, None, None, None, agc_mode=3) + [(0, 0, "setAGCreleaseTime", 1.0)]
    shifts = np.arange(0, 512)
    z = (shifts[-1] + burst) // N_BLOCK + 3
    for r, off in enumerate(LONG_TARGETS):
        f, ph = 5390.0 + rng.uniform(300, 1200), rng.uniform(0, 2 * np.pi)
        noise = (rng.standard_normal((2, ns)) * 1e-3).astype(F32)
        t = np.arange(ns, dtype=F64)[None, :] - shifts[:, None]
        x = 0.4 * np.clip(t / burst, 0, 1) * (t < burst) * np.exp(1j * (2 * np.pi * f * t / float(FS) + ph))
        i, q = (x.real + noise[0]).astype(F32), (x.imag + noise[1]).astype(F32)
        # every start shift at once: with the AGC off the audio is 0.5 * audf exactly (out_gain 0.5)
        off_ev = [(k, 0, e[2]) + tuple(e[3:]) for k in range(len(shifts)) for e in mine] + \
                 [(k, 0, "disableAGC") for k in range(len(shifts))]
        o = oracle_lib.run(i[:, :z * N_BLOCK], q[:, :z * N_BLOCK], off_ev, threads=os.cpu_count() or 1, want_pcm=False)
        sub = [(k, 0, e[2]) + tuple(e[3:]) for k in range(len(shifts)) for e in mine]
        _, _, tr = model_run(o["audio"] * F32(2.0), np.zeros((z, len(shifts)), F32), sub)
        L = np.array([np.flatnonzero(a)[-1] for a in tr["att"]])
        hit = np.flatnonzero((L + LONG_HC + 1) % N_BLOCK == off)
        if not len(hit):
            raise RuntimeError("no burst start for expiry offset %d" % off)
        k = int(hit[r % len(hit)])
        I[r], Q[r] = i[k], q[k]
        ev += [(r,) + e[1:] for e in mine]
        last.append(int(L[k])); expiry.append(int(L[k]) + LONG_HC + 1)
    return I, Q, ev, dict(last=np.array(last), expiry=np.array(expiry))
