"""CPU tier: the restatement of every snapshot the grabber publishes (grabber_snapshots_oracle.grab_snapshots), checked
against the C restatement's ora_grab_run, and the expected rows of a call built on it (grab_snapshots_expected), the
authority of sdr_grabber_process_device_snapshots."""
import numpy as np

import aux_signals as S
import aux_subset_harness as H
import grabber_snapshots_oracle as G
from oracle import aux_lib as A

N = 128


def test_last_snapshot_of_every_prefix_is_grab_run():
    I, Q = S.pp_case(6, 13, seed=61)
    for n in range(14):
        snaps = G.grab_snapshots(I[:, :n * N], Q[:, :n * N])
        out, flags = A.grab_run(I[:, :n * N], Q[:, :n * N])
        assert snaps.shape == (6, n // 2, 512)
        if n >= 2:
            assert np.array_equal(snaps[:, -1].astype(np.int32), out), n
            assert (flags == 1).all()
        else:
            assert (out == -1).all() and (flags == 0).all()


def test_snapshot_m_is_blocks_2m_and_2m_plus_1_interleaved():
    rng = np.random.default_rng(62)
    I = rng.integers(-32768, 32768, (3, 11 * N)).astype(np.int16)
    Q = rng.integers(-32768, 32768, (3, 11 * N)).astype(np.int16)
    snaps = G.grab_snapshots(I, Q)
    assert snaps.shape == (3, 5, 512)
    for m in range(5):
        z = slice(2 * m * N, (2 * m + 2) * N)
        assert np.array_equal(snaps[:, m, 0::2], I[:, z]) and np.array_equal(snaps[:, m, 1::2], Q[:, z])


def test_expected_of_calls_on_every_channel_is_one_run_split_at_the_calls():
    """Ragged calls on every channel (odd lengths leave pairs open across calls): the rows of call j are the snapshots of
    one oracle run numbered [before // 2, after // 2), their power the spectrum tap's."""
    nch = 5
    I, Q = S.pp_case(nch, 44, seed=63)
    full = np.arange(nch, dtype=np.uint32)
    sizes = (1, 2, 3, 5, 8, 1, 16, 7, 1)
    calls = [(full, nb) for nb in sizes]
    want = G.grab_snapshots_expected(I, Q, calls)
    one = G.grab_snapshots(I[:, :sum(sizes) * N], Q[:, :sum(sizes) * N])
    pos = 0
    for j, nb in enumerate(sizes):
        snaps, power, counts = want[j]
        S_ = (nb + 1) // 2
        assert snaps.shape == (nch, S_, 512) and power.shape == (nch, S_, 256)
        a, b = pos // 2, (pos + nb) // 2
        assert (counts == b - a).all() and b - a in (S_, S_ - 1)
        assert np.array_equal(snaps[:, :b - a], one[:, a:b])
        for c in range(nch):
            assert np.array_equal(power[c, :b - a].view(np.uint32), A.grab_spectrum(one[c, a:b]).view(np.uint32))
        assert not snaps[:, b - a:].any() and not power[:, b - a:].any()
        pos += nb


def test_expected_of_subset_calls_follows_each_channels_own_blocks():
    nch = 9
    I, Q = S.pp_case(nch, 30, seed=64)
    rng = np.random.default_rng(65)
    calls = H.random_calls(rng, nch, 12, 24, sizes=(1, 3, 2, 1, 5))
    want = G.grab_snapshots_expected(I, Q, calls)
    pos = H.positions(nch, calls)
    for j, (ids, nb) in enumerate(calls):
        for i, c in enumerate(ids):
            own = G.grab_snapshots(I[c:c + 1, :int(pos[j + 1][c]) * N], Q[c:c + 1, :int(pos[j + 1][c]) * N])[0]
            k = int(want[j][2][i])
            assert k == int(pos[j + 1][c]) // 2 - int(pos[j][c]) // 2
            assert np.array_equal(want[j][0][i, :k], own[len(own) - k:])
