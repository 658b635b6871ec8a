"""CPU tier: the waterfall's restatement (tests/waterfall_oracle.c) against the definition of include/sdr_aux.h: K = 1 is the
spectrum oracle bit for bit, larger K is the mean of the float64 DFT power within float32 rounding, and the state carried
between calls (or moved to another channel) makes the lines independent of how the pairs are cut."""
import numpy as np
import pytest

import waterfall_oracle as W


def _pairs(n, seed):
    """int16 [n, 512] snapshots: noise plus a tone that drifts from pair to pair, and one full-scale pair"""
    rng = np.random.default_rng(seed)
    t = np.arange(256)
    s = np.empty((n, 512), np.int16)
    for j in range(n):
        ph = 2 * np.pi * (17 + 0.3 * j) * t / 256
        s[j, 0::2] = np.clip(rng.normal(0, 900, 256) + 8000 * np.cos(ph), -32768, 32767).astype(np.int16)
        s[j, 1::2] = np.clip(rng.normal(0, 900, 256) + 8000 * np.sin(ph), -32768, 32767).astype(np.int16)
    s[n // 2] = np.where(np.arange(512) % 3, 32767, -32768)
    return s


def test_k1_lines_are_the_spectrum_oracle():
    from oracle import aux_lib as A
    s = _pairs(9, 1)
    got = W.Channel(1).run(s)
    assert np.array_equal(got.view(np.uint32), A.grab_spectrum(s).view(np.uint32))


@pytest.mark.parametrize("K", [2, 3, 8, 16])
def test_lines_are_the_float64_mean_of_the_dft_power(K):
    s = _pairs(3 * K + 1, K)
    got = W.Channel(K).run(s)
    assert got.shape == (3, 256)
    x = s[:, 0::2].astype(np.float64) + 1j * s[:, 1::2].astype(np.float64)
    p = np.abs(np.fft.fft(x, axis=1)) ** 2
    want = p[:3 * K].reshape(3, K, 256).mean(axis=1)
    # float32 FFT: a few ulp of the largest line; then K float32 adds and one division
    tol = 4e-6 * want.max(axis=1, keepdims=True) * (1 + np.log2(K))
    assert (np.abs(got - want) <= tol).all(), np.abs(got - want).max() / want.max()


@pytest.mark.parametrize("K", [1, 3, 8])
def test_state_carried_across_cuts_and_channels(K):
    s = _pairs(5 * K + 2, 10 + K)
    whole = W.Channel(K).run(s)
    a = W.Channel(K)
    cut = [a.run(s[i:j]) for i, j in ((0, 1), (1, 1), (1, K + 1), (K + 1, 2 * K + 3), (2 * K + 3, 5 * K + 2))]
    assert np.array_equal(np.concatenate(cut).view(np.uint32), whole.view(np.uint32))
    # migration: the state of a channel half way through a line continues on another object
    b = W.Channel(K)
    first = b.run(s[:K + K // 2])
    c = W.Channel(K)
    c.held.value, c.acc[:] = b.held.value, b.acc
    rest = c.run(s[K + K // 2:])
    assert np.array_equal(np.concatenate([first, rest]).view(np.uint32), whole.view(np.uint32))


def test_expected_rows_follow_each_channels_own_pairs():
    """waterfall_expected over ragged subset calls equals each channel's pairs run in one piece."""
    rng = np.random.default_rng(3)
    nch, nb_total = 3, 14
    I = rng.integers(-3000, 3000, (nch, nb_total * 128)).astype(np.int16)
    Q = rng.integers(-3000, 3000, (nch, nb_total * 128)).astype(np.int16)
    calls = [([0, 1, 2], 1), ([2, 0], 3), ([1], 4), ([0, 1, 2], 2), ([2, 1], 5)]
    K = 3
    got = W.waterfall_expected(I, Q, calls, K)
    pos = W.positions(nch, calls)
    for c in range(nch):
        n = int(pos[-1][c])
        whole = W.Channel(K).run(W.grab_snapshots(I[c:c + 1, :n * 128], Q[c:c + 1, :n * 128])[0])
        mine = [lines[i, :counts[i]] for (ids, _), (lines, counts) in zip(calls, got) for i, cc in enumerate(ids) if cc == c]
        assert np.array_equal(np.concatenate(mine).view(np.uint32), whole.view(np.uint32))
    for (ids, nb), (lines, counts) in zip(calls, got):
        assert lines.shape == (len(ids), W.line_slots(K, nb), 256)
