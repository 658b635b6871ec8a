"""GPU tier: every snapshot a grabber process call publishes and its power spectrum (sdr_grabber_process_device_snapshots)
on the CUDA library, exactly against the oracle (grabber_snapshots_oracle.grab_snapshots_expected, ora_grab_spectrum).  Output
buffers sit between guard bands filled with a sentinel, and slots a call must not write keep the sentinel too."""
import os

import numpy as np
import pytest

import aux_signals as S
import aux_subset_harness as H
import grabber_snapshots_oracle as G

pytestmark = pytest.mark.gpu
N = 128
GUARD = 256          # elements of sentinel either side of each output
RAW_SENT = 0x5A5A
POW_SENT = 0x7FC0DEAD  # a NaN no spectrum produces


@pytest.fixture(scope="module")
def aux():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    from audiosdr_b200 import aux as m
    assert os.path.exists(m.lib_path()), "libsdr_aux.so missing: __graft_entry__.build() must run before the GPU tier"
    m.load_library()
    return m


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


class Out:
    """A CUDA output [rows, S, width] inside a flat buffer with sentinel guard bands."""

    def __init__(self, rows, S, width, kind):
        import torch
        self.shape = (rows, S, width)
        n = rows * S * width
        if kind == "raw":
            self.buf = torch.full((n + 2 * GUARD,), RAW_SENT, dtype=torch.int16, device="cuda:0")
        else:
            self.buf = torch.full((n + 2 * GUARD,), POW_SENT, dtype=torch.int32, device="cuda:0").view(torch.float32)
        self.t = self.buf[GUARD:GUARD + n].view(self.shape)
        self.kind = kind

    def bits(self):
        """(the output as raw bits, whether both guard bands are intact)"""
        import torch
        torch.cuda.synchronize()
        a = self.buf.cpu().numpy().view(np.uint16 if self.kind == "raw" else np.uint32)
        s = RAW_SENT if self.kind == "raw" else POW_SENT
        return a[GUARD:-GUARD].reshape(self.shape), bool((a[:GUARD] == s).all() and (a[-GUARD:] == s).all())


def run_call(g, I, Q, nb, channels=None, raw=True, power=True):
    rows = I.shape[0]
    S_ = (nb + 1) // 2
    o_raw = Out(rows, S_, 512, "raw") if raw else None
    o_pow = Out(rows, S_, 256, "pow") if power else None
    counts = g.process(I, Q, n_blocks=nb, channels=channels, snapshots=o_raw.t if raw else None, power=o_pow.t if power else None)
    return o_raw, o_pow, counts


def check_slots(j, o_raw, o_pow, want):
    """Slots < counts equal the oracle bit for bit, later slots and the guard bands keep the sentinel."""
    snaps, power, counts = want
    for o, w, sent, view in ((o_raw, snaps, RAW_SENT, np.uint16), (o_pow, power, POW_SENT, np.uint32)):
        if o is None:
            continue
        got, guards = o.bits()
        assert guards, "call %d: a guard band was written" % j
        for i, k in enumerate(counts):
            if not np.array_equal(got[i, :k], w[i, :k].view(view)):
                bad = np.argwhere(got[i, :k] != w[i, :k].view(view))
                raise AssertionError("call %d row %d (%s): %d words differ, first slot %d word %d" % (j, i, o.kind, len(bad), bad[0][0], bad[0][1]))
            assert (got[i, k:] == sent).all(), "call %d row %d: slot past counts written" % (j, i)


def state_of(g):
    import torch
    torch.cuda.synchronize()
    return g.export_state()


# ---------------------------------------------------------------- calls on every channel
def test_ragged_plain_calls_match_oracle_and_leave_the_plain_calls_state(aux):
    """Ragged n_blocks on every channel: raw slots, power slots, counts and unwritten trailing slots against the oracle; after
    each call grab, newDataAvailable, spectrum and the state blobs equal a twin handle driven by the plain call."""
    nch = 19
    sizes = (1, 2, 3, 5, 8, 1, 16, 7, 1, 1, 4, 9)
    I, Q = S.pp_case(nch, sum(sizes), seed=71)
    full = np.arange(nch, dtype=np.uint32)
    calls = [(full, nb) for nb in sizes]
    want = G.grab_snapshots_expected(I, Q, calls)
    g, twin = aux.GrabberBatch(nch), aux.GrabberBatch(nch)
    pos = np.zeros(nch, np.int64)
    for j, (ids, nb) in enumerate(calls):
        di, dq = _dev(H.gather_rows(I, ids, pos, nb)), _dev(H.gather_rows(Q, ids, pos, nb))
        pos[ids] += nb
        o_raw, o_pow, counts = run_call(g, di, dq, nb)
        twin.process(di, dq, n_blocks=nb)
        assert np.array_equal(counts, want[j][2]), j
        check_slots(j, o_raw, o_pow, want[j])
        assert np.array_equal(state_of(g), state_of(twin)), j
        assert [g.newDataAvailable(c) for c in range(nch)] == [twin.newDataAvailable(c) for c in range(nch)]
        a, b = g.spectrum(), twin.spectrum()
        assert (a is None) == (b is None) and (a is None or np.array_equal(a.view(np.uint32), b.view(np.uint32)))
        if j % 2:
            a, b = g.grab(), twin.grab()
            assert (a is None) == (b is None) and (a is None or np.array_equal(a, b))
            if counts.any():  # the last slot is the snapshot grab() hands out after the call
                got, _ = o_raw.bits()
                assert np.array_equal(got[:, counts[0] - 1].view(np.int16), a)
    g.close(); twin.close()


# ---------------------------------------------------------------- subsets, channels out of phase
def test_subset_calls_out_of_phase(aux):
    """Random subsets with ragged lengths leave the channels' pair phases apart: compact rows, slot 0 starting with the
    carried half, rows with counts == 0 (a 1-block call at even phase), and the same state as the subset call."""
    nch = 41
    I, Q = S.pp_case(nch, 40, seed=72)
    rng = np.random.default_rng(73)
    calls = H.random_calls(rng, nch, 24, 36, sizes=(1, 3, 1, 2, 5, 1, 4, 7))
    want = G.grab_snapshots_expected(I, Q, calls)
    g, twin = aux.GrabberBatch(nch), aux.GrabberBatch(nch)
    pos = np.zeros(nch, np.int64)
    seen_zero = seen_carried = 0
    for j, (ids, nb) in enumerate(calls):
        before = pos.copy()
        di, dq = _dev(H.gather_rows(I, ids, pos, nb)), _dev(H.gather_rows(Q, ids, pos, nb))
        pos[ids] += nb
        o_raw, o_pow, counts = run_call(g, di, dq, nb, channels=ids)
        twin.process(di, dq, n_blocks=nb, channels=ids)
        assert np.array_equal(counts, want[j][2]), j
        check_slots(j, o_raw, o_pow, want[j])
        assert np.array_equal(state_of(g), state_of(twin)), j
        seen_zero += int((counts == 0).sum())
        seen_carried += int(((before[ids] % 2) == 1).sum())
    assert seen_zero > 0 and seen_carried > 0
    g.close(); twin.close()


def test_outputs_one_at_a_time_together_and_none(aux):
    """snapshots only, power only, both, and all NULL (through the C entry point): the same slots, and with all NULL the
    state, grab and spectrum of the plain call."""
    nch = 12
    I, Q = S.pp_case(nch, 9, seed=74)
    full = np.arange(nch, dtype=np.uint32)
    calls = [(full, 3), (full, 1), (full, 5)]
    want = G.grab_snapshots_expected(I, Q, calls)
    hs = {m: aux.GrabberBatch(nch) for m in ("raw", "pow", "both", "null", "plain")}
    pos = 0
    for j, (ids, nb) in enumerate(calls):
        di, dq = _dev(I[:, pos * N:(pos + nb) * N]), _dev(Q[:, pos * N:(pos + nb) * N])
        pos += nb
        for m, h in hs.items():
            if m == "plain":
                h.process(di, dq, n_blocks=nb)
            elif m == "null":
                assert h.L.sdr_grabber_process_device_snapshots(h.h, None, nch, di.data_ptr(), dq.data_ptr(), di.stride(0), nb, None, None, None, None) == 0
            else:
                o_raw, o_pow, counts = run_call(h, di, dq, nb, raw=m != "pow", power=m != "raw")
                assert np.array_equal(counts, want[j][2])
                check_slots(j, o_raw, o_pow, want[j])
    ref = hs["plain"]
    want_state, want_spec = state_of(ref), ref.spectrum()
    for m, h in hs.items():  # states first: grab() clears the new-data flag the blobs carry
        assert np.array_equal(state_of(h), want_state), m
        assert np.array_equal(h.spectrum().view(np.uint32), want_spec.view(np.uint32)), m
    grabs = {m: h.grab() for m, h in hs.items()}
    for m, h in hs.items():
        assert np.array_equal(grabs[m], grabs["plain"]), m
        h.close()


# ---------------------------------------------------------------- full size
def test_full_size_4096_channels_256_blocks(aux):
    """One call of bench.py's receiver size: every raw row against numpy, power against the oracle on 512 sampled rows."""
    import torch
    from oracle import aux_lib as A
    nch, nb = 4096, 256
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(75)
    I = torch.randint(-32768, 32768, (nch, nb * N), generator=gen, device="cuda:0", dtype=torch.int32).to(torch.int16)
    Q = torch.randint(-32768, 32768, (nch, nb * N), generator=gen, device="cuda:0", dtype=torch.int32).to(torch.int16)
    g = aux.GrabberBatch(nch)
    o_raw, o_pow, counts = run_call(g, I, Q, nb)
    assert (counts == nb // 2).all()
    raw, ok = o_raw.bits()
    assert ok
    hI, hQ = I.cpu().numpy(), Q.cpu().numpy()
    want = np.empty((nch, nb // 2, 512), np.int16)
    want[:, :, 0::2] = hI.reshape(nch, nb // 2, 256)
    want[:, :, 1::2] = hQ.reshape(nch, nb // 2, 256)
    assert np.array_equal(raw.view(np.int16), want)
    pw, ok = o_pow.bits()
    assert ok
    pick = np.random.default_rng(76).permutation(nch)[:512]
    for c in pick:
        assert np.array_equal(pw[c], A.grab_spectrum(want[c]).view(np.uint32)), c
    g.close()


# ---------------------------------------------------------------- edge values
def test_edge_values_power_bit_exact(aux):
    """Zeros, full-scale square waves (+-32768 on both rails), single impulses of -32768 and 32767: power bit for bit,
    exact zeros included."""
    nch, nb = 8, 6
    ns = nb * N
    I, Q = np.zeros((nch, ns), np.int16), np.zeros((nch, ns), np.int16)
    t = np.arange(ns)
    I[1] = np.where(t % 16 < 8, 32767, -32768); Q[1] = np.where(t % 32 < 16, -32768, 32767)
    I[2] = np.where(t % 2 == 0, -32768, 32767); Q[2] = -32768
    I[3, 5] = -32768
    Q[4, 300] = 32767
    I[5, 128 * 3 + 77] = -32768; Q[5, 128 * 3 + 77] = -32768
    I[6] = -32768; Q[6] = -32768
    I[7, ::256] = 32767
    want = G.grab_snapshots_expected(I, Q, [(np.arange(nch, dtype=np.uint32), nb)])[0]
    assert (want[1][0] == 0).any() and (want[1][3] == 0).any()
    g = aux.GrabberBatch(nch)
    o_raw, o_pow, counts = run_call(g, _dev(I), _dev(Q), nb)
    check_slots(0, o_raw, o_pow, want)
    g.close()


# ---------------------------------------------------------------- checkpoints
def test_odd_phase_export_import_carried_half(aux):
    """A channel exported at odd phase (a block carried) and imported into another handle and slot: the next call's slot
    0 there starts with the blob's carried half, as the oracle over the channel's whole stream says."""
    I, Q = S.pp_case(6, 12, seed=77)
    src = aux.GrabberBatch(6)
    src.process(_dev(I[:, :3 * N]), _dev(Q[:, :3 * N]))
    blob = src.export_state([4])
    dst = aux.GrabberBatch(10)
    dst.process(_dev(np.zeros((10, 2 * N), np.int16)), _dev(np.ones((10, 2 * N), np.int16)))  # even phase everywhere
    dst.import_state([7], blob)
    o_raw, o_pow, counts = run_call(dst, _dev(I[4:5, 3 * N:8 * N]), _dev(Q[4:5, 3 * N:8 * N]), 5, channels=[7])
    want = G.grab_snapshots_expected(I[4:5, :8 * N], Q[4:5, :8 * N], [(np.array([0], np.uint32), 3), (np.array([0], np.uint32), 5)])[1]
    assert list(counts) == [3] and list(want[2]) == [3]
    check_slots(0, o_raw, o_pow, want)
    raw, _ = o_raw.bits()
    assert np.array_equal(raw[0, 0, :256].view(np.int16)[0::2], I[4, 2 * N:3 * N])
    src.close(); dst.close()


# ---------------------------------------------------------------- the graph
def test_preprocessor_subset_then_grabber_snapshots(aux):
    """I2S in -> pre-processor -> grabber, both advanced with the same id list on device planes: each row's snapshots are the
    oracle grabber run over the channel's own pre-processor output stream."""
    import torch
    nch = 20
    I, Q = S.pp_case(nch, 30, seed=78)
    rng = np.random.default_rng(79)
    calls = H.random_calls(rng, nch, 12, 26, sizes=(1, 3, 2, 5, 1))
    ev0 = [(None, 0, "startAutoI2SerrorDetection")]
    want_pp = H.pp_expected(I, Q, ev0, calls)
    pos = H.positions(nch, calls)
    PI, PQ = np.zeros_like(I), np.zeros_like(Q)
    for j, (ids, nb) in enumerate(calls):
        for i, c in enumerate(ids):
            z = slice(int(pos[j][c]) * N, int(pos[j + 1][c]) * N)
            PI[c, z], PQ[c, z] = want_pp[j][0][i], want_pp[j][1][i]
    want = G.grab_snapshots_expected(PI, PQ, calls)
    p, g = aux.PreProcessorBatch(nch), aux.GrabberBatch(nch)
    p.startAutoI2SerrorDetection()
    own = np.zeros(nch, np.int64)
    for j, (ids, nb) in enumerate(calls):
        di, dq = _dev(H.gather_rows(I, ids, own, nb)), _dev(H.gather_rows(Q, ids, own, nb))
        own[ids] += nb
        oi, oq = torch.empty_like(di), torch.empty_like(dq)
        p.process(di, dq, oi, oq, n_blocks=nb, channels=ids)
        o_raw, o_pow, counts = run_call(g, oi, oq, nb, channels=ids)
        assert np.array_equal(counts, want[j][2]), j
        check_slots(j, o_raw, o_pow, want[j])
    p.close(); g.close()


# ---------------------------------------------------------------- rejection
def test_rejected_arguments_change_nothing(aux):
    """Misaligned outputs, duplicate and out-of-range ids, a NULL list with the wrong count: EINVAL, outputs and guards
    untouched, state blobs and flags unchanged."""
    nch = 10
    I, Q = S.pp_case(nch, 4, seed=80)
    g = aux.GrabberBatch(nch)
    g.process(_dev(I[:, :N]), _dev(Q[:, :N]))  # odd phase: a carried half
    before = state_of(g)
    x, y = _dev(I[:3, N:3 * N]), _dev(Q[:3, N:3 * N])
    o_raw, o_pow = Out(3, 1, 512, "raw"), Out(3, 1, 256, "pow")
    ok_ids = np.array([1, 4, 7], np.uint32)
    L, rp, pp = g.L, o_raw.t.data_ptr(), o_pow.t.data_ptr()
    counts = np.full(3, 99, np.uint32)
    bad = [(ok_ids, 3, rp + 2, pp), (ok_ids, 3, rp, pp + 4), (ok_ids, 3, rp + 8, None), (ok_ids, 3, None, pp + 8),
           (np.array([1, 1, 2], np.uint32), 3, rp, pp), (np.array([1, nch, 2], np.uint32), 3, rp, pp), (None, 3, rp, pp)]
    for ids, n, r, p in bad:
        ptr = ids.ctypes.data if ids is not None else None
        assert L.sdr_grabber_process_device_snapshots(g.h, ptr, n, x.data_ptr(), y.data_ptr(), x.stride(0), 2, r, p, counts.ctypes.data, None) == -1
    assert (counts == 99).all()
    for o in (o_raw, o_pow):
        got, guards = o.bits()
        assert guards and (got == (RAW_SENT if o.kind == "raw" else POW_SENT)).all()
    assert np.array_equal(state_of(g), before)
    g.close()
