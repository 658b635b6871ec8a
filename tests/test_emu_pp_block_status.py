"""CPU tier: the pre-processor's per-block status records (sdr_preproc_process_*_status, SDR_PP_BS_*).

  * the oracle's records (tests/pp_records_oracle.c, the oracle's own pre-processor code) are its status after every
    prefix of the stream (ora_aux_run, which the golden vectors and refaux pin to the unmodified reference);
  * the records instantiations run on the host (tests/emu/pp_emu_records.cpp, built from sdr_aux_core.cuh)
    against the oracle's records bit for bit: the knife-edge placements of tests/pp_edge_signals.py, a detector that steps
    its correction twice in one call, a detector that stops in the middle of a call, detector-off rows with every
    correction and swap, setters between calls, ragged call schedules;
  * every word of the record range is written and no word outside it.
The GPU tier (test_gpu_pp_block_status.py) runs the same cases on the CUDA build.
"""
import ctypes as C

import numpy as np
import pytest

import aux_signals as S
import pp_edge_signals as E
import pp_records as R
from oracle import aux_lib as A

NF = 6
SENTINEL = 0x5A5A5A5A  # no field can hold it: flags, counters up to 1 001, corrections and int16 samples
_cache = {}


@pytest.fixture(scope="module")
def emu():
    return R.emu_records()


def edge_case(placement):
    if placement not in _cache:
        I, Q, ev, lay = E.build(placement)
        _cache[placement] = (I, Q, ev, lay, R.oracle_records(I, Q, ev))
    return _cache[placement]


def emu_calls(f, I, Q, ev, ends, guard=0):
    """Calls [0, ends[0]), [ends[0], ends[1]), ... of the emulator, status carried across calls; an event at block b goes
    before the call that starts at b (setters queued between calls).  Returns (out I, out Q, records [n_blocks, 6, C],
    [status after each call]).  guard > 0: each call's record buffer is followed by `guard` sentinel words, checked intact,
    and must come back without a sentinel inside its range."""
    starts = [0] + list(ends[:-1])
    assert all(e[1] in starts for e in ev), "events must sit on call boundaries"
    nch = I.shape[0]
    oi, oq = np.empty_like(I), np.empty_like(Q)
    st = np.zeros((nch, 8), np.int32)
    recs, sts = [], []
    for pos, end in zip(starts, ends):
        blob, nev = A._pack_events("pp", [(c, 0, *rest) for c, b, *rest in ev if b == pos])
        buf = C.create_string_buffer(blob, len(blob)) if nev else None
        z = slice(pos * 128, end * 128)
        i, q = np.ascontiguousarray(I[:, z]), np.ascontiguousarray(Q[:, z])
        a, b = np.empty_like(i), np.empty_like(q)
        n = (end - pos) * NF * nch
        raw = np.full(n + guard, SENTINEL, np.int32)
        assert f(nch, end - pos, buf, nev, i.ctypes.data, q.ctypes.data, a.ctypes.data, b.ctypes.data, st.ctypes.data, raw.ctypes.data) == 0
        if guard:
            assert not (raw[:n] == SENTINEL).any() and (raw[n:] == SENTINEL).all()
        oi[:, z], oq[:, z] = a, b
        recs.append(raw[:n].reshape(end - pos, NF, nch))
        sts.append(st[:, :6].copy())
    return oi, oq, np.concatenate(recs), sts


def check_against_oracle(emu, I, Q, ev, ends, guard=0):
    want = R.oracle_records(I, Q, ev)
    oi, oq, rec, sts = emu_calls(emu, I, Q, ev, ends, guard)
    assert np.array_equal(oi, want[0]) and np.array_equal(oq, want[1])
    assert np.array_equal(rec, want[3]), np.argwhere(rec != want[3])[:5]
    for e, s in zip(ends, sts):  # the last record of a call is the status the call leaves
        assert np.array_equal(rec[e - 1].T, s), e
    return want


# ---- the oracle's records are its status after every prefix
def test_oracle_records_are_the_status_after_every_prefix():
    nch, nb = 24, 36
    I, Q = S.pp_case(nch, nb, seed=21)
    ev = S.pp_events(nch, nb)
    _, _, st, rec = R.oracle_records(I, Q, ev)
    assert np.array_equal(rec[-1].T, st[:, :6])
    for b in range(nb):
        pre = A.run("pp", (I[:, :(b + 1) * 128], Q[:, :(b + 1) * 128]), [e for e in ev if e[1] <= b])[2][:, :6]
        assert np.array_equal(rec[b].T, pre), b
    assert len(np.unique(rec[:, 1, :])) == 3 and (np.diff(rec[:, 0, :], axis=0) != 0).any()  # corrections and flags move


def test_oracle_records_pin_the_knife_edge_prefix():
    I, Q, ev, lay, want = edge_case("after_failures")
    x = lay["block"]
    for b in (0, x - 1, x, x + 1):
        pre = A.run("pp", (I[:, :(b + 1) * 128], Q[:, :(b + 1) * 128]), ev)[2][:, :6]
        assert np.array_equal(want[3][b].T, pre), b


# ---- the records instantiations on the host against the oracle
def _schedules(nb, x):
    start = 0 if nb < 100 else x - 3
    return {"ones": ([start] if start else []) + list(range(start + 1, nb + 1)), "edge": [x // 2, x + 1, nb], "all": [nb]}


@pytest.mark.parametrize("sched", ["ones", "edge", "all"])
@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_emulated_records_at_the_knife_edge(emu, placement, sched):
    I, Q, ev, lay, want = edge_case(placement)
    nb, x = I.shape[1] // 128, lay["block"]
    check_against_oracle(emu, I, Q, ev, _schedules(nb, x)[sched])
    rec = want[3]
    # the knife-edge block is where the planned state ends: every row enters it as placed, and the records of many rows
    # change at that block and not before
    assert (rec[x - 1, 0] == 1).all() and (rec[x - 1, 1] == lay["corr"]).all() and (rec[x - 1, 2] == 10).all()
    assert (rec[x - 1, 3] == lay["succ"]).all()
    moved = (rec[x, :4] != rec[x - 1, :4]).any(0)
    assert moved.sum() >= E.MIN_FLIPS and (~moved).sum() >= E.MIN_FLIPS


def test_emulated_records_detector_steps_twice_in_one_call(emu):
    """Channels whose I arrives one sample late: the detector fails eleven strong blocks in a row, steps 0 -> +1, fails
    again, steps to -1 and then succeeds, all inside one call."""
    nch, nb = 16, 48
    I, Q = S.pp_case(nch, nb, seed=9)
    ev = [(None, 0, "startAutoI2SerrorDetection")]
    want = check_against_oracle(emu, I, Q, ev, [3, nb - 2, nb])
    corr = want[3][:, 1, :]
    steps = (np.diff(corr[3:nb - 2], axis=0) != 0).sum(0)
    assert (steps >= 2).sum() >= 2
    assert set(np.unique(corr)) == {-1, 0, 1}


@pytest.mark.parametrize("ends", [[1004], [990, 1004], [998, 999, 1000, 1001, 1002, 1004]])
def test_emulated_records_detector_stops_inside_a_call(emu, ends):
    """Aligned channels succeed on every block; after 1 001 strong blocks the detector switches itself off, inside the
    call, and its rows keep running on the detector path until the call ends."""
    nch, nb = 8, 1004
    I, Q = S.pp_case(nch, nb, seed=3)
    ev = [(None, 0, "startAutoI2SerrorDetection")]
    want = check_against_oracle(emu, I, Q, ev, ends)
    auto = want[3][:, 0, :]
    stop = [int(np.argmax(auto[:, c] == 0)) for c in range(nch) if (auto[:, c] == 0).any()]
    assert len(stop) >= 2 and all(990 < s < nb - 1 for s in stop)


@pytest.mark.parametrize("ends", [[8], [1, 8], [2, 3, 8], [1, 2, 3, 4, 5, 6, 7, 8]])
def test_emulated_records_detector_off_rows(emu, ends):
    """Rows with the detector off: correction +1, -1 and 0, each with and without swap; only the saved sample moves."""
    nch = 12
    I, Q = S.pp_case(nch, 8, seed=13)
    ev = [(c, 0, "setI2SerrorCompensation", (c % 3) - 1) for c in range(nch)] + [(c, 0, "swapIQ", 1) for c in range(nch) if (c // 3) % 2]
    want = check_against_oracle(emu, I, Q, ev, ends, guard=64)
    rec = want[3]
    for c in range(nch):
        corr = (c % 3) - 1
        src = I if corr == 1 else Q
        assert (rec[:, :4, c] == [0, corr, 0, 0]).all() and (rec[:, 5, c] == (c // 3) % 2).all()
        assert np.array_equal(rec[:, 4, c], src[c, 127::128] if corr else np.zeros(8, np.int32))


@pytest.mark.parametrize("ends", [[5, 10, 15, 20, 25, 30, 36], [2, 9, 12, 18, 24, 30, 35, 36]])
def test_emulated_records_setters_between_calls(emu, ends):
    """Every public setter queued between calls: detector started and stopped, corrections set, swaps turned on, on rows
    that move between the feed-forward and the detector path from one call to the next."""
    nch, nb = 40, 36
    I, Q = S.pp_case(nch, nb, seed=5)
    starts = [0] + ends[:-1]
    ev = [(None, 0, "startAutoI2SerrorDetection")]
    rng = np.random.default_rng(11)
    names = [("stopAutoI2SerrorDetection",), ("startAutoI2SerrorDetection",), ("setI2SerrorCompensation", 1),
             ("setI2SerrorCompensation", -1), ("setI2SerrorCompensation", 0), ("swapIQ", 1), ("swapIQ", 0)]
    for pos in starts[1:]:
        for c in rng.choice(nch, 10, replace=False):
            ev.append((int(c), pos, *names[rng.integers(len(names))]))
    check_against_oracle(emu, I, Q, ev, ends, guard=32)


@pytest.mark.parametrize("ends", [list(range(1, 25)), [3, 10, 17, 24], [24], [11, 13, 24]])
def test_emulated_records_ragged_calls_mixed_rows(emu, ends):
    """Detector, manual corrections and swaps in one handle (tests/aux_signals.pp_events moved onto call boundaries),
    sentinel-filled record buffers."""
    nch, nb = 48, 24
    I, Q = S.pp_case(nch, nb, seed=17)
    starts = [0] + ends[:-1]
    ev = [(c, max(s for s in starts if s <= b), *rest) for c, b, *rest in S.pp_events(nch, nb)]
    check_against_oracle(emu, I, Q, ev, ends, guard=128)
