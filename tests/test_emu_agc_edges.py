"""CPU tier: the AGC one rounding away from its decisions (tests/agc_edge_signals.py).

  * the numpy model against the oracle: the agc tap bit for bit, and agc_gain / agc_active after every block, fed with
    the oracle's own audf tap and AM carrier;
  * the builders meet their targets: attack ties (and one float either side) in every hang state on the AM level path
    and at the clamp on the sample path, the tie before a falling carrier, expiries on tile, block and call boundaries,
    the gain on 0.99f and its neighbours across block ends, levels of exactly 1.0, groups of 4, 5 and 32 tables;
  * every covered mutation of the kernel changes the AGC output or the block records of at least MIN_FLIPS rows;
  * the host emulation of the kernel source against the oracle: audio, int16 pcm, end-of-call status and per-block
    records under several hand-over schedules, on the short-tile plans and the split ALS form, in subset calls that skip
    the knife-edge channels while their hang counter is 1 or 0, across a checkpoint moved to another handle (whose group
    it pushes past four tables), and in AGC mode 3 across many calls.
The GPU tier (test_gpu_agc_edges.py) runs the same cases on the CUDA build.
"""
import os

import numpy as np
import pytest

import agc_edge_signals as E
import audiosdr_b200 as A
import harness
from test_emu_block_status import BS, check_case, oracle_block_status
from test_emu_edge_signals import PLANS, assert_bits
from test_emu_pipeline import set_plan, set_schedule

N_BLOCK = 128
_cache = {}


def case():
    """(I, Q, events, layout, oracle result), built and run once per session."""
    if "c" not in _cache:
        I, Q, ev, lay = E.build()
        from oracle import oracle_lib
        _cache["c"] = (I, Q, ev, lay, oracle_lib.run(I, Q, ev, threads=os.cpu_count() or 1))
    return _cache["c"]


def long_case():
    if "long" not in _cache:
        I, Q, ev, lay = E.long_case()
        from oracle import oracle_lib
        _cache["long"] = (I, Q, ev, lay, oracle_lib.run(I, Q, ev, threads=os.cpu_count() or 1))
    return _cache["long"]


def taps():
    if "taps" not in _cache:
        I, Q, ev, lay, _ = case()
        _cache["taps"] = E.oracle_taps(I, Q, ev)
    return _cache["taps"]


def model(mut=()):
    key = ("model",) + tuple(mut)
    if key not in _cache:
        t, st = taps()
        _cache[key] = E.model_run(t["audf"], E.carrier_of(st), case()[2], mut)
    return _cache[key]


def rows_of(lay, *kinds):
    return np.array([r for r, k in enumerate(lay["rows"]) if k in kinds])


# ---- the model is the oracle's arithmetic
def test_model_is_the_oracles(oracle):
    t, st = taps()
    out, per, _ = model()
    assert harness.bits_equal(out, t["agc"]), harness.describe_mismatch(out, t["agc"])
    assert np.array_equal(per["gain"].view(np.uint32), st[:, :, 14].astype(np.float32).view(np.uint32))
    assert np.array_equal(per["active"], st[:, :, 2] != 0)


def test_model_is_the_oracles_in_mode_3(oracle):
    I, Q, ev, lay, _ = long_case()
    t, st = E.oracle_taps(I, Q, ev)
    out, per, tr = E.model_run(t["audf"], E.carrier_of(st), ev)
    assert harness.bits_equal(out, t["agc"]), harness.describe_mismatch(out, t["agc"])
    assert np.array_equal(per["gain"].view(np.uint32), st[:, :, 14].astype(np.float32).view(np.uint32))
    # the hang of 88 200 samples runs out where it was placed: no decision changes the gain from the last attack to it
    for r, (L, X) in enumerate(zip(lay["last"], lay["expiry"])):
        assert X == L + E.LONG_HC + 1 and X % N_BLOCK == E.LONG_TARGETS[r]
        assert not tr["upd"][r, L + 1:X].any() and tr["upd"][r, X] and not tr["att"][r, X]
        assert tr["hang"][r, X] == 0 and tr["hang"][r, X - 1] == 1


# ---- the builders meet their targets
def _census(tr, rows):
    """{(relation, hang state): count} of the samples of `rows`: relation 'eq' (level == old), 'up' (level one float above
    old), 'dn' (one float below); hang state '>1', '1', '0'."""
    lv, old, hang = tr["level"][rows], tr["old"][rows], tr["hang"][rows]
    rel = {"eq": lv == old, "up": lv == np.nextafter(old, np.float32(np.inf)),
           "dn": lv == np.nextafter(old, np.float32(-np.inf))}
    hs = {">1": hang > 1, "1": hang == 1, "0": hang == 0}
    return {(a, b): int((m & h & (old > 0)).sum()) for a, m in rel.items() for b, h in hs.items()}


def test_attack_ties_on_the_am_level_path(oracle):
    lay = case()[3]
    _, _, tr = model()
    am = rows_of(lay, "am_tie")
    c = _census(tr, am)
    assert all(c[("eq", h)] > 0 for h in (">1", "1", "0")), c
    # one float either side: the level moves only at block boundaries, so these come with the counter reloaded (> 1) by
    # the converging attacks, or run out (0) on a block-constant level that release left one float away
    assert c[("up", ">1")] > 0 and c[("up", "0")] > 0 and c[("dn", ">1")] > 0 and c[("dn", "0")] > 0, c
    # the exact ties also on rows whose attack coefficient is not 0: a fixed point of a_att*old + b_att*level
    nz = np.array([r for r in am if lay["params"][r]["att"] != E.TINY_MS])
    assert _census(tr, nz)[("eq", "1")] > 0 and _census(tr, nz)[("eq", "0")] > 0
    # the tie on a block's last sample as the hang runs out (counter 1), then a falling carrier
    last = np.arange(N_BLOCK - 1, tr["level"].shape[1] - 1, N_BLOCK)
    hit = (tr["level"][am][:, last] == tr["old"][am][:, last]) & (tr["hang"][am][:, last] == 1) & \
          (tr["level"][am][:, last + 1] < tr["old"][am][:, last + 1])
    assert hit.sum() >= E.MIN_FLIPS


def test_attack_ties_on_the_sample_path(oracle):
    lay = case()[3]
    _, _, tr = model()
    for kind in ("ssb_clamp", "sam_clamp"):
        c = _census(tr, rows_of(lay, kind))
        assert all(c[("eq", h)] > 0 for h in (">1", "1", "0")), (kind, c)
    c = _census(tr, rows_of(lay, "ssb_clamp"))  # old converged to 1 - 2^-24 below a clamped level
    assert all(c[("up", h)] > 0 for h in (">1", "1", "0")), c


def test_levels_of_exactly_one(oracle):
    lay = case()[3]
    _, _, tr = model()
    for kind in ("am_clamp", "ssb_clamp", "sam_clamp"):
        rows = rows_of(lay, kind)
        one = tr["old"][rows] == np.float32(1.0)
        assert one.any(), kind  # old == 1.0: index 32767, table row 127 at fraction 255
        assert (tr["level"][rows] == np.float32(1.0)).sum() > 100, kind
    t, st = taps()
    assert (E.carrier_of(st)[:, rows_of(lay, "am_clamp")] > 0.5).any()


def test_gain_on_the_agc_active_threshold(oracle):
    lay = case()[3]
    _, per, tr = model()
    for kind, want in (("act_eq", E.ACT), ("act_dn", E.ACT_DN), ("act_up", E.ACT_UP)):
        rows = rows_of(lay, kind)
        held = per["gain"][8:, rows] == want  # from block 8 on, at every block end and at the end of the call
        assert held.all(), (kind, per["gain"][8:, rows])
        assert (per["active"][8:, rows] == (want < E.ACT)).all()
        for r in rows:  # old sits in index bucket (0, k)
            k = lay["params"][r]["k"]
            q = int(np.float64(per["old"][-1, r]) * 32767.0)
            assert q == k, (r, q, k)


def test_hang_ends_on_tile_block_and_call_boundaries(oracle):
    I, Q, ev, lay, _ = case()
    _, _, tr = model()
    starts = E.call_starts(ev, I.shape[1] // N_BLOCK, E.CHUNKS)
    for r in rows_of(lay, "hang_at"):
        p = lay["params"][r]
        L, X = p["last"], p["expiry"]
        assert X == L + p["hc"] + 1 and X % N_BLOCK == p["off"]
        assert tr["att"][r, L] and not tr["upd"][r, L + 1:X].any() and tr["upd"][r, X] and not tr["att"][r, X]
        if p["off"] == 0:
            assert X // N_BLOCK in starts
    # short hangs (counts 0, 1, 2): expiries on the first and the last sample of tiles of every length, and on call starts
    for hc in (0, 1, 2):
        rows = [r for r in rows_of(lay, "hang_short") if lay["params"][r]["hc"] == hc]
        att = tr["att"][rows]
        rel = tr["upd"][rows] & ~att & (tr["hang"][rows] == 0)
        prev_att = np.zeros_like(att)
        prev_att[:, hc + 1:] = att[:, :att.shape[1] - hc - 1]
        between = np.ones_like(att)
        for d in range(1, hc + 1):
            between[:, hc + 1:] &= ~att[:, hc + 1 - d:att.shape[1] - d]
        exp = np.flatnonzero((rel & prev_att & between).any(0))
        for T in (8, 16, 32):
            assert (exp % T == 0).any() and (exp % T == T - 1).any(), (hc, T)
        assert (exp % N_BLOCK == 0).any() or hc == 0, hc  # (the placed hangs put expiries on call boundaries)
    for r, b, want in lay["toggles"]:
        assert tr["hang"][r, b * N_BLOCK] == want
    assert sorted(w for _, _, w in lay["toggles"]) == [0, 0, 1, 1]


def test_table_staging_groups(oracle):
    I, Q, ev, lay, _ = case()
    p = E.Params(len(I))
    for e in ev:
        if e[1] == 0:
            p.apply(e[0], *e[2:])
    stage = rows_of(lay, "stage")
    gs = [g for g in E.groups(p) if set(g) <= set(stage)]
    assert [len(g) for g in gs] == [32, 32, 32]
    assert [len({p.key[r] for r in g}) for g in gs] == [4, 5, 32]
    first, glob = E.staging(p)
    assert glob[gs[1]].sum() == 28 and glob[gs[2]].sum() == 28 and not glob[gs[0]].any()
    assert not p.on[gs[1][:3]].any() and p.on[gs[1][3:]].all()  # AGC-off lanes hold 3 of group 1's 5 tables
    g, lane, b0, b1 = E.STAGE_MOVE
    for e in ev:
        if e[1] == b0:
            p.apply(e[0], *e[2:])
    assert E.staging(p)[1][gs[g][lane]]  # the setter sends the lane to the global path, and a later one brings it back


def test_every_mutation_changes_rows(oracle):
    base, bper, _ = model()
    for m in E.MUTATIONS:
        out, per, _ = model((m,))
        differ = (out.view(np.uint32) != base.view(np.uint32)).any(1)
        differ |= (per["gain"].view(np.uint32) != bper["gain"].view(np.uint32)).any(0)
        differ |= (per["active"] != bper["active"]).any(0)
        assert differ.sum() >= E.MIN_FLIPS, (m, differ.sum())


# ---- the emulation against the oracle
@pytest.mark.parametrize("sched", ["lockstep", "consumers", "random:2/late"])
def test_emulated_agc_edges(oracle, emu_lib, monkeypatch, sched):
    set_schedule(monkeypatch, sched)
    I, Q, ev, lay, o = case()
    assert_bits(emu_lib, I, Q, ev, o, chunks=E.CHUNKS)


@pytest.mark.parametrize("plan", PLANS, ids=["tile16-x2", "tile8-merged-x3", "tile16-merged-x2"])
def test_emulated_agc_edges_short_tile_plans(oracle, emu_lib, monkeypatch, plan):
    set_schedule(monkeypatch, "random:3/late")
    set_plan(monkeypatch, *plan)
    I, Q, ev, lay, o = case()
    assert_bits(emu_lib, I, Q, ev, o, chunks=(5, 1, 17), pcm=False)


def test_emulated_agc_edges_split_als(oracle, emu_lib, monkeypatch):
    monkeypatch.setenv("SDR_ALS_SPLIT", "1")
    set_schedule(monkeypatch, "consumers")
    I, Q, ev, lay, o = case()
    assert_bits(emu_lib, I, Q, ev, o, chunks=(11, 2), pcm=False)


def test_emulated_agc_edges_block_records(oracle, emu_lib):
    I, Q, ev, lay, o = case()
    check_case(emu_lib, I, Q, ev, chunks=(9, 1, 4))


def _edge_rows(lay):
    return np.concatenate([rows_of(lay, "hang_short", "hang_at", "act_eq", "act_dn", "am_tie")])


def test_emulated_agc_edge_channels_skip_a_call(oracle, emu_lib):
    """Subset calls: the hang rows, the 0.99 rows and the AM tie rows skip three blocks while their hang counters are
    at 1 or 0 (short hangs) or running (placed hangs), then all rows continue; every row's output is the oracle's."""
    I, Q, ev, lay, o = case()
    nch, nb = I.shape[0], I.shape[1] // N_BLOCK
    assert not [e for e in ev if e[1] > 0 and e[2] not in ("disableAGC", "enableAGC", "setAGCthreshold")]
    cfg = [e for e in ev if e[1] == 0]
    skip = _edge_rows(lay).astype(np.uint32)
    allc = np.arange(nch, dtype=np.uint32)
    x = 14  # hang rows at 1 / 0 (tests above); placed hangs running from their last attack
    calls = [(allc, x), (np.setdiff1d(allc, skip).astype(np.uint32), 3), (allc, nb - x - 3), (skip, 3)]
    b = A.SdrBatch(nch, _lib=emu_lib)
    b.configure([(e[0], e[2]) + tuple(e[3:]) for e in cfg])
    pos = np.zeros(nch, np.int64)
    got = np.zeros((nch, nb * N_BLOCK), np.float32)
    pending = sorted([e for e in ev if e[1] > 0], key=lambda e: e[1])
    for ids, k in calls:
        while k > 0:
            # setters on a channel's own timeline: applied before the call that starts its block
            now = [e for e in pending if e[0] in ids and pos[e[0]] == e[1]]
            if now:
                b.configure([(e[0], e[2]) + tuple(e[3:]) for e in now])
                pending = [e for e in pending if e not in now]
            step = min([k] + [e[1] - int(pos[e[0]]) for e in pending if e[0] in ids])
            i = np.stack([I[c, pos[c] * N_BLOCK:(pos[c] + step) * N_BLOCK] for c in ids])
            q = np.stack([Q[c, pos[c] * N_BLOCK:(pos[c] + step) * N_BLOCK] for c in ids])
            out = np.empty((len(ids), step * N_BLOCK), np.float32)
            b.process_host(i, q, out, channels=ids)
            for j, c in enumerate(ids):
                got[c, pos[c] * N_BLOCK:(pos[c] + step) * N_BLOCK] = out[j]
            pos[ids] += step
            k -= step
    assert (pos == nb).all() and not pending
    assert harness.bits_equal(got, o["audio"]), harness.describe_mismatch(got, o["audio"])
    assert np.array_equal(harness.status_matrix(b), o["status"], equal_nan=True)


def test_emulated_checkpoint_at_the_hang_edges(oracle, emu_lib):
    """export_state at a block where hang counters are 1 and 0 and placed hangs are running; import into another handle,
    in an order that puts a table of group 2 into the first staging group (five tables there: the imported lane's own
    and the lanes after it go to the global path); continue there."""
    I, Q, ev, lay, o = case()
    nch, nb = I.shape[0], I.shape[1] // N_BLOCK
    x = 14
    a = A.SdrBatch(nch, _lib=emu_lib)
    evs = sorted([e for e in ev if e[1] < x], key=lambda e: e[1])
    o1, pos = np.zeros((nch, x * N_BLOCK), np.float32), 0
    for blk in sorted({e[1] for e in evs} | {x}):
        if blk > pos:
            z = slice(pos * N_BLOCK, blk * N_BLOCK)
            a.process_host(np.ascontiguousarray(I[:, z]), np.ascontiguousarray(Q[:, z]), o1[:, z])
            pos = blk
        if blk < x:
            a.configure([(e[0], e[2]) + tuple(e[3:]) for e in evs if e[1] == blk])
    blobs = a.export_state()
    stage = rows_of(lay, "stage")
    g0, g2 = list(stage[:32]), list(stage[64:])
    perm = [r for r in range(nch) if r not in stage] + g0[:6] + [g2[20]] + g0[6:] + g2[:20] + g2[21:] + list(stage[32:64])
    assert sorted(perm) == list(range(nch))
    slots = np.arange(nch, dtype=np.uint32) * 2 + 1  # every other slot of a larger handle
    b = A.SdrBatch(2 * nch + 3, _lib=emu_lib)
    b.import_state(slots, blobs[perm])
    p = E.Params(2 * nch + 3)
    for e in ev:
        if e[1] < x:
            p.apply(int(slots[perm.index(e[0])]), *e[2:])
    for r in range(2 * nch + 3):
        if r not in set(slots.tolist()):
            p.apply(r, "setDemodMode", E.AM)
    st0 = [g for g in E.groups(p, slots.tolist()) if int(slots[perm.index(g0[0])]) in g][0]
    assert len({p.key[r] for r in st0}) > E.SLOTS
    rest = nb - x
    o2 = np.zeros((nch, rest * N_BLOCK), np.float32)
    rec = np.zeros((rest, BS, nch), np.uint32)
    later = sorted([e for e in ev if e[1] >= x], key=lambda e: e[1])
    pos = x
    for blk in sorted({e[1] for e in later} | {nb}):
        if blk > pos:
            z = slice(pos * N_BLOCK, blk * N_BLOCK)
            out = np.empty((nch, (blk - pos) * N_BLOCK), np.float32)
            r2 = np.zeros((blk - pos, BS, nch), np.uint32)
            b.process_host(np.ascontiguousarray(I[perm, z]), np.ascontiguousarray(Q[perm, z]), out, block_status=r2,
                           channels=slots)
            o2[:, (pos - x) * N_BLOCK:(blk - x) * N_BLOCK] = out
            rec[pos - x:blk - x] = r2
            pos = blk
        if blk < nb:
            b.configure([(int(slots[perm.index(e[0])]), e[2]) + tuple(e[3:]) for e in later if e[1] == blk])
    got = np.concatenate([o1[perm], o2], 1)
    want = o["audio"][perm]
    assert harness.bits_equal(got, want), harness.describe_mismatch(got, want)
    assert np.array_equal(rec, oracle_block_status(I, Q, ev)[x:][:, :, perm])


def test_emulated_mode_3_across_many_calls(oracle, emu_lib):
    """The 88 200-sample hang of AGC mode 3 over about a hundred ragged calls, its expiry on a block boundary and on the
    last sample of a 32-sample tile; audio, pcm and the end-of-call status."""
    I, Q, ev, lay, o = long_case()
    assert_bits(emu_lib, I, Q, ev, o, chunks=(7, 1, 13))
