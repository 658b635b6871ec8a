"""The subset harness of the aux blocks (tests/aux_subset_harness.py) must not drift: fed calls on every channel (ids in
any order, ragged lengths, setters between calls), its per-channel mapping of blocks and setter events equals one plain
oracle run over the whole planes.  CPU only."""
import numpy as np

import aux_signals as S
import aux_subset_harness as H
from oracle import aux_lib as A

N = 128


def _every_channel_calls(rng, nch, sizes):
    return [(rng.permutation(nch).astype(np.uint32), nb) for nb in sizes]


def _concat(out, calls, k):
    """Channel-ordered planes from the compact rows of every call."""
    nch = len(calls[0][0])
    parts = []
    for (ids, nb), o in zip(calls, out):
        inv = np.empty(nch, np.int64)
        inv[np.asarray(ids)] = np.arange(nch)
        parts.append(o[k][inv])
    return np.concatenate(parts, 1)


def test_pp_mapping_equals_plain_run():
    nch, sizes = 12, [3, 1, 5, 2, 7, 1, 4]
    nb = sum(sizes)
    I, Q = S.pp_case(nch, nb, seed=3)
    rng = np.random.default_rng(1)
    calls = _every_channel_calls(rng, nch, sizes)
    ev0 = [(None, 0, "startAutoI2SerrorDetection")]
    setters = {2: [(5, "setI2SerrorCompensation", -1), (None, "swapIQ", 1)], 4: [(7, "stopAutoI2SerrorDetection")],
               5: [(3, "swapIQ", 0)], len(sizes): [(1, "setI2SerrorCompensation", 1)]}
    starts = np.cumsum([0] + sizes)
    plain_ev = [(None, 0, "startAutoI2SerrorDetection")]
    for j, evs in setters.items():
        plain_ev += [(e[0], int(starts[j]), e[1]) + tuple(e[2:]) for e in evs]
    want = A.run("pp", (I, Q), plain_ev)
    got = H.pp_expected(I, Q, ev0, calls, setters)
    assert np.array_equal(_concat(got, calls, 0), want[0]) and np.array_equal(_concat(got, calls, 1), want[1])
    assert np.array_equal(H.pp_final_status(I, Q, ev0, calls, setters), want[2][:, :6])
    # status after an intermediate call = the plain run over that prefix, with the setters made before that call
    j = 4
    pre = A.run("pp", (I[:, :starts[j + 1] * N], Q[:, :starts[j + 1] * N]), [e for e in plain_ev if e[1] < starts[j + 1]])
    assert np.array_equal(got[j][2], pre[2][:, :6])


def test_iq_mapping_equals_plain_run():
    nch, sizes = 9, [1, 2, 1, 3, 40, 1]
    nb = sum(sizes)
    X = S.iq_case(nch, nb, seed=5)
    calls = _every_channel_calls(np.random.default_rng(2), nch, sizes)
    setters = {1: [(2, "setGainBalance", 1.07)], 3: [(None, "setGainBalance", 0.95)]}
    starts = np.cumsum([0] + sizes)
    plain_ev = [(e[0], int(starts[j]), e[1]) + tuple(e[2:]) for j, evs in setters.items() for e in evs]
    want = A.run("iq", (X,), plain_ev)
    got = H.iq_expected(X, [], calls, setters)
    assert np.array_equal(_concat(got, calls, 0), want[0]) and np.array_equal(_concat(got, calls, 1), want[1])


def test_grab_mapping_equals_plain_run():
    nch, sizes = 7, [1, 1, 2, 3, 1]
    I, Q = S.pp_case(nch, sum(sizes), seed=8)
    calls = _every_channel_calls(np.random.default_rng(3), nch, sizes)
    got = H.grab_expected(I, Q, calls)
    p = 0
    for (ids, nb), (snap, valid, completed) in zip(calls, got):
        before = p
        p += nb
        want, flags = A.grab_run(I[:, :p * N], Q[:, :p * N])
        assert np.array_equal(snap, want) and np.array_equal(valid, flags[:, 1] != 0)
        assert (completed == (p // 2 > before // 2)).all()
