"""CPU tier: the SAM PLL and the noise blanker one rounding away from their decisions (tests/pll_edge_signals.py).

  * the numpy model against the oracle: the IF and demodulator taps bit for bit, and pll_f, locked, nb_avg and nb_hit
    after every block, so that what the builder places on is what the oracle computes;
  * the placed samples sit on their thresholds, and every covered mutation of the kernel flips decisions there that
    change the demodulator output or the block records;
  * the host emulation of the kernel source against the oracle: audio, int16 pcm, end-of-call status and per-block
    records, under several hand-over schedules, on the short-tile plans, with the general path alone, across a checkpoint
    moved to another handle just before the knife edges, and in subset calls in which the knife-edge channels skip a call.
The GPU tier (test_gpu_pll_edges.py) runs the same case on the CUDA build.
"""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import audiosdr_b200 as A
import harness
import pll_edge_signals as E
from test_emu_block_status import BS, check_case, oracle_block_status
from test_emu_edge_signals import PLANS, assert_bits
from test_emu_pipeline import set_plan, set_schedule

N_BLOCK = 128
_cache = {}


def case():
    """(I, Q, events, layout, oracle result), built and run once per session."""
    if not _cache:
        I, Q, ev, lay = E.build()
        from oracle import oracle_lib
        _cache["c"] = (I, Q, ev, lay, oracle_lib.run(I, Q, ev, threads=os.cpu_count() or 1))
    return _cache["c"]


def model(mut=()):
    key = ("model",) + tuple(mut)
    if key not in _cache:
        I, Q, ev, lay, _ = case()
        _cache[key] = E.model_run(I, Q, lay["nb_on"], lay["thr"], mut)
    return _cache[key]


def oracle_taps(I, Q, ev, rows, taps=("if_i", "if_q", "dm_i", "dm_q")):
    from oracle import oracle_lib
    out = {t: np.empty((len(rows), I.shape[1]), np.float32) for t in taps}
    for k, r in enumerate(rows):
        ch = oracle_lib.Channel()
        for e in ev:
            if e[0] == r:
                ch.apply(e[2], *e[3:])
        for b in range(I.shape[1] // N_BLOCK):
            z = slice(b * N_BLOCK, (b + 1) * N_BLOCK)
            ch.update(I[r, z], Q[r, z])
            for t in taps:
                out[t][k, z] = ch.taps[E_TAPS.index(t)]
    return out


E_TAPS = ["in_i", "in_q", "nb_i", "nb_q", "if_i", "if_q", "dm_i", "dm_q", "demod", "audf", "agc", "als"]


def model_records(st):
    """The model's status per block as record words [n_blocks, BS_FIELDS, R] (the fields it computes)."""
    return {A.BS_SAM_FREQUENCY: st["pll_f"].view(np.uint32), A.BS_SAM_LOCKED: st["locked"].astype(np.uint32),
            A.BS_NB_AVERAGE: st["nb_avg"].view(np.uint32), A.BS_NB_DETECTED: st["nb_hit"].astype(np.uint32)}


# ---- the model is the oracle's arithmetic
def test_model_taps_are_the_oracles(oracle):
    I, Q, ev, lay, _ = case()
    taps, _ = model()
    want = oracle_taps(I, Q, ev, range(len(I)))
    for t, w in want.items():
        assert harness.bits_equal(taps[t], w), (t, harness.describe_mismatch(taps[t], w))


def test_model_status_after_every_block_is_the_oracles(oracle):
    I, Q, ev, lay, _ = case()
    _, st = model()
    want = oracle_block_status(I, Q, ev)
    for f, got in model_records(st).items():
        assert np.array_equal(got, want[:, f, :]), A.BS_NAMES[f]


# ---- the placed samples do what they say
def _ops_at(lay, I, Q):
    """The decision operands of every PLL row at its placed sample, from the model."""
    out = {}

    def hook(m, n, Ib, Qb, j):
        rows = [r for r in range(len(lay["rows"])) if lay["at"][r] == n and not lay["nb_on"][r]]
        for r in rows:
            xr = E.biquad_peek(E.IF_AM, m.if_i[..., r], Ib[r, j])
            xi = E.biquad_peek(E.IF_AM, m.if_q[..., r], Qb[r, j])
            _, ops = E.sam_sample({k: v[r] for k, v in m.s.items()}, xr, xi)
            out[r] = ops

    E.model_run(I, Q, lay["nb_on"], lay["thr"], hook=hook)
    return out


def test_knife_edges_sit_on_their_thresholds(oracle):
    I, Q, ev, lay, _ = case()
    ops = _ops_at(lay, I, Q)
    names = lay["rows"]
    for r, name in enumerate(names):
        if lay["nb_on"][r] or lay["at"][r] < 0:
            continue
        assert E._want(name, ops[r]), (r, name)
    for name, _, _ in (t for w in E.WARPS for t in w):
        if name not in E.NOT_REACHED:
            assert sum(1 for r, n in enumerate(names) if n == name and lay["at"][r] >= 0) >= E.TRY.get(name, 1), name
    n_end = [r for r, n in enumerate(names) if "_end" in n]
    assert all(lay["at"][r] % N_BLOCK == N_BLOCK - 1 for r in n_end)
    assert all(lay["at"][r] % N_BLOCK != N_BLOCK - 1 for r, n in enumerate(names) if n.endswith("_mid"))
    # the blanker rows: magnitude == avg * thr at the named scan (or one float above)
    for r, t in enumerate(lay["nb"]):
        if t is None or names[r] != "nb":
            continue
        scan, pos, off, _ = t
        n = int(lay["at"][r])
        blk = n // N_BLOCK
        call, ring = (blk + 1, 128 + pos) if scan == "first" else (blk + 2, pos)
        step = next(s for s in E.nb_scan(I, Q, r, call) if s[0] == call and s[1] == ring)
        t_ = step[3] * lay["thr"][r]
        assert step[2] == (np.nextafter(t_, np.float32(np.inf)) if off else t_), (r, t)
    met = {t for r, t in enumerate(lay["nb"]) if t is not None and names[r] == "nb"}
    assert met == set(E.NB_TARGETS)  # among them the first and the last scanned ring positions, 78 and 255


def test_every_mutation_flips_knife_edge_decisions(oracle):
    """Each covered mutation of the kernel changes the demodulator output or the block records of at least MIN_FLIPS
    rows; the unreachable ones change nothing."""
    base_t, base_s = model()
    for m in E.MUTATIONS:
        t, s = model((m,))
        differ = np.zeros(len(base_t["dm_i"]), bool)
        for k in ("dm_i", "dm_q"):
            differ |= (t[k].view(np.uint32) != base_t[k].view(np.uint32)).any(1)
        for k in ("pll_f", "locked", "nb_hit"):
            differ |= (np.asarray(s[k]) != np.asarray(base_s[k])).any(0)
        if m in E.UNREACHABLE + E.NOT_REACHED:
            assert not differ.any(), m
        else:
            assert differ.sum() >= E.MIN_FLIPS, (m, differ.sum())


def test_fast_path_edges_meet_a_passing_vote(oracle):
    """On the GPU one lane whose own fast-path guard fails sends its whole warp down the general path.  At every placed
    sample of a fast-path target, every other lane of its warp (32 PLL rows in channel order, as the receiver groups SAM
    channels without blanker) passes its guard in the model, so the kernel's fast-path forms compute the edge -- or would,
    under a mutation of the guard.  cos_wrap rows are searched on loops that wander; MIN_FOUND of them must qualify."""
    I, Q, ev, lay, _ = case()
    ok = model()[0]["ok"]
    warp, names = lay["warp"], lay["rows"]
    passing = {}
    for r in range(len(warp)):
        n = int(lay["at"][r])
        if n < 0 or names[r] not in E.FAST:
            continue
        others = [x for x in range(len(warp)) if warp[x] == warp[r] and x != r]
        good = bool(ok[others, n].all())
        passing.setdefault(names[r], []).append(good)
        if names[r] != "cos_wrap":
            assert good, (r, names[r], [x for x in others if not ok[x, n]])
        if names[r] in ("wrap_up_dn", "wrap_lo", "tiny_di", "big_dr", "cos_wrap"):
            assert ok[r, n], (r, names[r])  # and the lane itself takes the fast path there
    assert sum(passing["cos_wrap"]) >= E.TRY["cos_wrap"]
    assert set(passing) == set(E.FAST)


# ---- the emulation against the oracle
@pytest.mark.parametrize("sched", ["lockstep", "consumers", "random:2/late"])
def test_emulated_knife_edges(oracle, emu_lib, monkeypatch, sched):
    set_schedule(monkeypatch, sched)
    I, Q, ev, lay, o = case()
    assert_bits(emu_lib, I, Q, ev, o)


@pytest.mark.parametrize("plan", PLANS, ids=["tile16-x2", "tile8-merged-x3", "tile16-merged-x2"])
def test_emulated_knife_edges_short_tile_plans(oracle, emu_lib, monkeypatch, plan):
    """The short-tile plans take the PLL rows (the SAM bucket without blanker)."""
    set_schedule(monkeypatch, "random:3/late")
    set_plan(monkeypatch, *plan)
    I, Q, ev, lay, o = case()
    assert_bits(emu_lib, I, Q, ev, o, chunks=(5, 1, 17), pcm=False)


def test_emulated_knife_edges_block_records(oracle, emu_lib):
    I, Q, ev, lay, o = case()
    check_case(emu_lib, I, Q, ev, chunks=(9, 1, 4))


def test_emulated_knife_edges_general_path_alone(oracle, monkeypatch):
    """Every vote of the PLL's fast path made to fail (a separate instance of the emulation library): the general path
    alone computes every sample, the fast path's own edges included."""
    from audiosdr_b200 import api
    monkeypatch.setenv("SDR_EMU_VOTE_FAILS", "1")
    emu_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
    subprocess.run(["make", "-s", "-C", emu_dir], check=True)
    with tempfile.TemporaryDirectory() as d:
        dst = os.path.join(d, "libsdr_emu_pll_general.so")
        shutil.copy(os.path.join(emu_dir, "libsdr_emu.so"), dst)
        lib = api._bind(ctypes.CDLL(dst))
        I, Q, ev, lay, o = case()
        assert_bits(lib, I, Q, ev, o, chunks=(7, 23), pcm=False)


def _first_edge_block(lay):
    return int(lay["at"][lay["at"] >= 0].min()) // N_BLOCK


def test_emulated_checkpoint_before_the_knife_edges(oracle, emu_lib):
    """export_state just before the first knife-edge block, import into other slots of a larger handle, continue there."""
    I, Q, ev, lay, o = case()
    x, nch = _first_edge_block(lay), I.shape[0]
    a = A.SdrBatch(nch, _lib=emu_lib)
    a.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
    o1 = np.empty((nch, x * N_BLOCK), np.float32)
    a.process_host(np.ascontiguousarray(I[:, :x * N_BLOCK]), np.ascontiguousarray(Q[:, :x * N_BLOCK]), o1)
    blobs = a.export_state()
    slots = (np.arange(nch)[::-1] * 2 + 3).astype(np.uint32)
    b = A.SdrBatch(int(slots.max()) + 5, _lib=emu_lib)
    b.import_state(slots, blobs)
    rest = I.shape[1] // N_BLOCK - x
    o2 = np.empty((nch, rest * N_BLOCK), np.float32)
    rec = np.zeros((rest, BS, nch), np.uint32)
    b.process_host(np.ascontiguousarray(I[:, x * N_BLOCK:]), np.ascontiguousarray(Q[:, x * N_BLOCK:]), o2, block_status=rec,
                   channels=slots)
    got = np.concatenate([o1, o2], 1)
    assert harness.bits_equal(got, o["audio"]), harness.describe_mismatch(got, o["audio"])
    assert np.array_equal(rec, oracle_block_status(I, Q, ev)[x:])


def test_emulated_knife_edge_channels_skip_a_call(oracle, emu_lib):
    """Subset calls: the knife-edge PLL rows skip the call before their knife edge (their stream pauses) while the blanker
    rows go on, then all rows continue; every row's output is the oracle's on its own stream."""
    I, Q, ev, lay, o = case()
    nch, nb = I.shape[0], I.shape[1] // N_BLOCK
    x = _first_edge_block(lay)
    pll = np.flatnonzero(~lay["nb_on"]).astype(np.uint32)
    calls = [(np.arange(nch, dtype=np.uint32), x - 3), (np.setdiff1d(np.arange(nch), pll).astype(np.uint32), 3),
             (np.arange(nch, dtype=np.uint32), nb - x), (pll, 3)]
    b = A.SdrBatch(nch, _lib=emu_lib)
    b.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev])
    pos = np.zeros(nch, np.int64)
    got = np.zeros((nch, nb * N_BLOCK), np.float32)
    for ids, k in calls:
        i = np.stack([I[c, pos[c] * N_BLOCK:(pos[c] + k) * N_BLOCK] for c in ids])
        q = np.stack([Q[c, pos[c] * N_BLOCK:(pos[c] + k) * N_BLOCK] for c in ids])
        out = np.empty((len(ids), k * N_BLOCK), np.float32)
        b.process_host(i, q, out, channels=ids)
        for j, c in enumerate(ids):
            got[c, pos[c] * N_BLOCK:(pos[c] + k) * N_BLOCK] = out[j]
        pos[ids] += k
    assert (pos == nb).all()
    assert harness.bits_equal(got, o["audio"]), harness.describe_mismatch(got, o["audio"])
    assert np.array_equal(harness.status_matrix(b), o["status"], equal_nan=True)
