"""GPU tier: the pre-processor's image detector one rounding away from each of its decisions (tests/pp_edge_signals.py) on
the CUDA build, exactly against the oracle.

The knife-edge blocks are selected so that a detector evaluating a different floating-point network than the oracle's
(oracle/aux_fft128.h) -- a contracted butterfly or power, a reordered or reciprocal mean, a non-strict compare -- flips
decisions, and each flip moves I2Scorrection and with it every later output sample.  Device and host planes, ragged
calls, subsets whose 32-lane CTAs mix knife-edge, idle and detector-off channels, checkpoints moved between handles right
before the knife edge, and 4 096 channels at once.  Also the I/Q generator's non-unit gain path at the gains where its
guards matter.  Integer outputs: every comparison is exact.
"""
import os

import numpy as np
import pytest

import aux_signals as S
import pp_edge_signals as E

pytestmark = pytest.mark.gpu
_cache = {}


@pytest.fixture(scope="module")
def aux():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    from audiosdr_b200 import aux as m
    assert os.path.exists(m.lib_path()), "libsdr_aux.so missing: __graft_entry__.build() must run before the GPU tier"
    m.load_library()
    return m


def case(placement):
    from oracle import aux_lib as A
    if placement not in _cache:
        I, Q, ev, lay = E.build(placement)
        _cache[placement] = (I, Q, ev, lay, A.run("pp", (I, Q), ev))
    return _cache[placement]


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _status(p, channels=None):
    return np.array([[s.auto_detect, s.correction, s.failure_count, s.success_count, s.saved_sample, s.swap]
                     for s in p.status(channels)], np.int32)


def _setters(p, ev, slots=None):
    """Setter events (all at block 0 here) on the handle; slots maps a case row to its channel of the handle."""
    for c, b, name, *arg in ev:
        assert b == 0
        ch = None if c is None else (c if slots is None else int(slots[c]))
        if c is None and slots is not None:
            ch = np.asarray(slots, np.uint32)
        getattr(p, name)(*([ch] + arg))


def _oracle_status_after(I, Q, ev, ends):
    from oracle import aux_lib as A
    return [A.run("pp", (I[:, :e * 128], Q[:, :e * 128]), ev)[2][:, :6] for e in ends]


def run_calls(p, I, Q, ends, host=False, channels=None):
    """Calls ending at the blocks in `ends`; returns (out I, out Q, [status after each call])."""
    import torch
    oi, oq = np.empty_like(I), np.empty_like(Q)
    if not host:
        dI, dQ = _dev(I), _dev(Q)
        dOi, dOq = torch.empty_like(dI), torch.empty_like(dQ)
    sts, pos = [], 0
    for end in ends:
        z = slice(pos * 128, end * 128)
        if host:
            a, b = np.empty((I.shape[0], (end - pos) * 128), np.int16), np.empty((I.shape[0], (end - pos) * 128), np.int16)
            p.process_host(np.ascontiguousarray(I[:, z]), np.ascontiguousarray(Q[:, z]), a, b, n_blocks=end - pos, channels=channels)
            oi[:, z], oq[:, z] = a, b
        else:
            p.process(dI[:, z], dQ[:, z], dOi[:, z], dOq[:, z], n_blocks=end - pos, channels=channels)
        sts.append(_status(p, channels))
        pos = end
    if not host:
        torch.cuda.synchronize()
        oi, oq = dOi.cpu().numpy(), dOq.cpu().numpy()
    return oi, oq, sts


def schedules(I, lay):
    nb, x = I.shape[1] // 128, lay["block"]
    start = 0 if nb < 100 else x - 3
    return {"ones": ([start] if start else []) + list(range(start + 1, nb + 1)), "edge": [x // 2, x + 1, nb], "all": [nb]}


# ---------------------------------------------------------------- pre-processor
@pytest.mark.parametrize("sched", ["ones", "edge", "all"])
@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_knife_edge_device_planes(aux, placement, sched):
    I, Q, ev, lay, want = case(placement)
    ends = schedules(I, lay)[sched]
    p = aux.PreProcessorBatch(I.shape[0])
    _setters(p, ev)
    oi, oq, sts = run_calls(p, I, Q, ends)
    p.close()
    assert np.array_equal(oi, want[0]) and np.array_equal(oq, want[1])
    for e, got, exp in zip(ends, sts, _oracle_status_after(I, Q, ev, ends)):
        assert np.array_equal(got, exp), e


@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_knife_edge_host_planes(aux, placement):
    I, Q, ev, lay, want = case(placement)
    ends = schedules(I, lay)["edge"]
    p = aux.PreProcessorBatch(I.shape[0])
    _setters(p, ev)
    oi, oq, sts = run_calls(p, I, Q, ends, host=True)
    p.close()
    assert np.array_equal(oi, want[0]) and np.array_equal(oq, want[1])
    assert np.array_equal(sts[-1], want[2][:, :6])


@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_knife_edge_subsets_share_ctas_with_idle_and_feed_forward_lanes(aux, placement):
    """A handle of 131 channels; each call lists the knife-edge channels interleaved with detector-off channels (corrected
    and swapped, on the feed-forward path) in shuffled slots, so that the detector's 32-lane CTAs hold knife-edge lanes
    next to lanes of no listed channel, and the list (not a multiple of 32) ends in a partial CTA.  Unlisted channels
    keep their state."""
    from oracle import aux_lib as A
    I, Q, ev, lay, want = case(placement)
    nk, nb = I.shape[0], I.shape[1] // 128
    n_off, n_total = 23, 131
    oI, oQ = S.pp_case(n_off, nb, seed=61)
    rows_I, rows_Q = np.concatenate([I, oI]), np.concatenate([Q, oQ])
    rng = np.random.default_rng(7)
    order = rng.permutation(nk + n_off)                       # row r of the call planes carries case row order[r]
    slots = rng.choice(n_total, nk + n_off, replace=False)   # ... on channel slots[r] of the handle
    off_ev = [(nk + k, 0, "setI2SerrorCompensation", (k % 3) - 1) for k in range(n_off)] + [(nk + k, 0, "swapIQ", 1) for k in range(0, n_off, 2)]
    case_ev = [(c, b, n, *a) for c, b, n, *a in ev if c is not None] + [(c, 0, "startAutoI2SerrorDetection") for c in range(nk)]
    w = A.run("pp", (rows_I, rows_Q), case_ev + off_ev)
    inv = np.argsort(order)
    p = aux.PreProcessorBatch(n_total)
    _setters(p, case_ev + off_ev, slots=slots[inv])
    ends = schedules(I, lay)["edge"]
    oi, oq, sts = run_calls(p, rows_I[order], rows_Q[order], ends, channels=slots)
    assert np.array_equal(oi, w[0][order]) and np.array_equal(oq, w[1][order])
    assert np.array_equal(sts[-1], w[2][order, :6])
    unlisted = np.setdiff1d(np.arange(n_total), slots)
    assert not _status(p, unlisted).any()
    p.close()


@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_knife_edge_checkpoint_moves_to_another_handle(aux, placement):
    """export_state just before the knife-edge block, import into other slots of a larger handle, continue there."""
    I, Q, ev, lay, want = case(placement)
    nk, nb, x = I.shape[0], I.shape[1] // 128, lay["block"]
    a = aux.PreProcessorBatch(nk)
    _setters(a, ev)
    oi1, oq1, _ = run_calls(a, I[:, :x * 128], Q[:, :x * 128], [x])
    blobs = a.export_state()
    a.close()
    slots = (np.arange(nk)[::-1] * 3 + 5).astype(np.uint32)
    b = aux.PreProcessorBatch(int(slots.max()) + 9)
    b.import_state(slots, blobs)
    oi2, oq2, sts = run_calls(b, I[:, x * 128:], Q[:, x * 128:], [1, 2, nb - x], channels=slots)
    b.close()
    assert np.array_equal(np.concatenate([oi1, oi2], 1), want[0]) and np.array_equal(np.concatenate([oq1, oq2], 1), want[1])
    assert np.array_equal(sts[-1], want[2][:, :6])


def test_knife_edge_many_channels(aux):
    """4 096 channels in one call: the 44 knife-edge channels of each short case spread over many CTAs among channels
    running the tame signals; every knife-edge row and a sample of the rest against the oracle."""
    import torch
    from oracle import aux_lib as A
    nch = 4096
    I0, Q0, ev0, lay0, want0 = case("after_failures")
    nb = I0.shape[1] // 128
    bI, bQ = S.pp_case(64, nb, seed=33)
    I, Q = np.tile(bI, (nch // 64, 1)), np.tile(bQ, (nch // 64, 1))
    knife = np.linspace(3, nch - 2, I0.shape[0]).astype(int)
    I[knife], Q[knife] = I0, Q0
    swap = [knife[c] for c, b, n, *a in ev0 if n == "swapIQ"]
    p = aux.PreProcessorBatch(nch)
    p.startAutoI2SerrorDetection()
    p.swapIQ(np.array(swap, np.uint32), True)
    dI, dQ = _dev(I), _dev(Q)
    dOi, dOq = torch.empty_like(dI), torch.empty_like(dQ)
    p.process(dI, dQ, dOi, dOq)
    torch.cuda.synchronize()
    oi, oq = dOi.cpu().numpy(), dOq.cpu().numpy()
    st = _status(p)
    p.close()
    assert np.array_equal(oi[knife], want0[0]) and np.array_equal(oq[knife], want0[1]) and np.array_equal(st[knife], want0[2][:, :6])
    rest = np.random.default_rng(3).choice(np.setdiff1d(np.arange(nch), knife), 64, replace=False)
    w = A.run("pp", (I[rest], Q[rest]), [(None, 0, "startAutoI2SerrorDetection")])
    assert np.array_equal(oi[rest], w[0]) and np.array_equal(oq[rest], w[1]) and np.array_equal(st[rest], w[2][:, :6])


# ---------------------------------------------------------------- I/Q generator: the non-unit gain path
def _edge_gains():
    """Gains at the guards of aux_to_pcm: zero, negative zero, a subnormal (its reciprocal, gainQ, overflows to inf), inf,
    NaN, negative; then gains around 2^31 / 32767 and -(2^31 + 1) / 32767, which put the full-scale sample's
    v * 32767 * g (v = 1) a few float steps below and above the limits of the 32-bit truncation."""
    g = [0.0, -0.0, 1e-40, -1e-40, np.inf, -np.inf, np.nan, -1.0, -1.5]
    for lim, sign in ((2147483648.0, 1.0), (2147483649.0, -1.0)):
        near = [np.float32(lim / 32767.0)]
        for _ in range(2):
            near = [np.nextafter(near[0], np.float32(0))] + near + [np.nextafter(near[-1], np.float32(np.inf))]
        g += [sign * float(x) for x in near]
    return g


def test_generator_gain_edges(aux):
    import torch
    from oracle import aux_lib as A
    gains = _edge_gains()
    nch, nb = len(gains), 6
    X = S.iq_case(nch, nb, seed=17)
    X[:, 5 * 128 - 40] = 32767        # a full-scale sample in every row, 128 samples before the last block's outputs
    X[:, 3 * 128 + 9] = -32768
    ev = [(c, 0, "setGainBalance", g) for c, g in enumerate(gains)]
    want = A.run("iq", (X,), ev)
    # the near-2^31 gains really land either side of the limits (I rail: the input delayed by 128, times 32767 * g)
    d = 1.0 * 32767.0 * np.array([float(np.float32(g)) for g in gains[9:]])
    assert ((d >= 2147483648.0) & (d < 2147484000.0)).any() and ((d < 2147483648.0) & (d > 2147483000.0)).any()
    assert ((d <= -2147483649.0) & (d > -2147484000.0)).any() and ((d > -2147483649.0) & (d < -2147483000.0)).any()
    assert (want[0][:, 6 * 128 - 40] == 0).any() and (want[0][:, 6 * 128 - 40] != 0).any()  # 0x80000000 -> 0, or not
    for host in (False, True):
        g = aux.IQGeneratorBatch(nch)
        for c, gain in enumerate(gains):
            g.setGainBalance(c, gain)
        if host:
            oi, oq = np.empty_like(X), np.empty_like(X)
            for lo, hi in ((0, 1), (1, 4), (4, nb)):
                a, b = np.empty((nch, (hi - lo) * 128), np.int16), np.empty((nch, (hi - lo) * 128), np.int16)
                g.process_host(np.ascontiguousarray(X[:, lo * 128:hi * 128]), a, b, n_blocks=hi - lo)
                oi[:, lo * 128:hi * 128], oq[:, lo * 128:hi * 128] = a, b
        else:
            dX = _dev(X)
            dOi, dOq = torch.empty_like(dX), torch.empty_like(dX)
            g.process(dX[:, :128], dOi[:, :128], dOq[:, :128], n_blocks=1)
            g.process(dX[:, 128:], dOi[:, 128:], dOq[:, 128:], n_blocks=nb - 1)
            torch.cuda.synchronize()
            oi, oq = dOi.cpu().numpy(), dOq.cpu().numpy()
        g.close()
        for c in range(nch):
            assert np.array_equal(oi[c], want[0][c]) and np.array_equal(oq[c], want[1][c]), (host, gains[c])
