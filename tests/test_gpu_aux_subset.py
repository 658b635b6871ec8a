"""GPU tier: calls on chosen subsets of the channels of the pre-processor, the I/Q generator and the grabber
(sdr_*_process_*_subset), and checkpoints of their channels (sdr_*_export_state / import_state), on the CUDA library
against the oracle stepped over each channel's own blocks (tests/aux_subset_harness.py).  Integer outputs: every
comparison is exact."""
import os

import numpy as np
import pytest

import aux_signals as S
import aux_subset_harness as H

pytestmark = pytest.mark.gpu
N = 128


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


def _status(p, channels=None):
    return np.array([[s.auto_detect, s.correction, s.failure_count, s.success_count, s.saved_sample, s.swap] for s in p.status(channels)], np.int32)


def _apply(obj, e):
    getattr(obj, e[1])(*([e[0]] + list(e[2:])))


def drive_pp(p, I, Q, calls, setters=None, plain=(), path="device", pos=None, id_map=None):
    """Runs the calls on PreProcessorBatch p; returns [(I_out, Q_out, status of every channel after the call)].
    plain: call indices run with channels=None (their ids must be arange); id_map: channel -> slot of p (a moved channel)."""
    import torch
    setters = setters or {}
    nch = I.shape[0]
    pos = np.zeros(nch, np.int64) if pos is None else pos
    out = []
    for j, (ids, nb) in enumerate(calls):
        for e in setters.get(j, []):
            _apply(p, e if id_map is None or e[0] is None else (id_map[e[0]],) + tuple(e[1:]))
        i, q = H.gather_rows(I, ids, pos, nb), H.gather_rows(Q, ids, pos, nb)
        pos[ids] += nb
        ch = None if j in plain else (ids if id_map is None else id_map[ids])
        if path == "host":
            oi, oq = np.full_like(i, 0x5A5A), np.full_like(q, 0x5A5A)
            p.process_host(i, q, oi, oq, n_blocks=nb, channels=ch)
        else:
            di, dq = _dev(i), _dev(q)
            doi, doq = torch.empty_like(di), torch.empty_like(dq)
            p.process(di, dq, doi, doq, n_blocks=nb, channels=ch)
            oi, oq = doi.cpu().numpy(), doq.cpu().numpy()
        out.append((oi, oq, _status(p) if id_map is None else None))
    return out


def drive_iq(g, X, calls, setters=None, plain=(), path="device", pos=None, id_map=None):
    import torch
    setters = setters or {}
    pos = np.zeros(X.shape[0], np.int64) if pos is None else pos
    out = []
    for j, (ids, nb) in enumerate(calls):
        for e in setters.get(j, []):
            g.setGainBalance(e[0] if id_map is None or e[0] is None else id_map[e[0]], e[2])
        x = H.gather_rows(X, ids, pos, nb)
        pos[ids] += nb
        ch = None if j in plain else (ids if id_map is None else id_map[ids])
        if path == "host":
            oi, oq = np.full_like(x, 0x5A5A), np.full_like(x, 0x5A5A)
            g.process_host(x, oi, oq, n_blocks=nb, channels=ch)
        else:
            dx = _dev(x)
            doi, doq = torch.empty_like(dx), torch.empty_like(dx)
            g.process(dx, doi, doq, n_blocks=nb, channels=ch)
            oi, oq = doi.cpu().numpy(), doq.cpu().numpy()
        out.append((oi, oq))
    return out


def assert_rows(j, got, want, what):
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)
        raise AssertionError("call %d: %s differs in %d samples, first row %d sample %d" % (j, what, len(bad), bad[0][0], bad[0][1]))


# ---------------------------------------------------------------- pre-processor
def _pp_setup(nch, seed):
    rng = np.random.default_rng(seed)
    calls = H.random_calls(rng, nch, 16, 40)
    full = np.arange(nch, dtype=np.uint32)
    calls.insert(3, (full, 1))
    calls.insert(8, (full, 2))
    calls.insert(9, (calls[2][0], 1))  # a 1-block call right after a full call
    setters = {}
    for j in (2, 5, 7, 10, 13):
        unlisted = np.setdiff1d(np.arange(nch), calls[j][0])
        if len(unlisted) == 0:
            continue
        c = int(unlisted[rng.integers(len(unlisted))])
        setters[j] = [(c, "swapIQ", int(j % 2)), (int(unlisted[-1]), "setI2SerrorCompensation", (j % 3) - 1)]
    setters.setdefault(11, []).append((6, "startAutoI2SerrorDetection"))
    return calls, setters, {3, 8}


@pytest.mark.parametrize("path", ["device", "host"])
def test_preprocessor_random_subsets(aux, path):
    """Detector running on every channel; channels skip random calls, setters hit unlisted channels, 1-block calls and
    full calls alternate.  Every call's rows and every channel's status after every call equal the oracle."""
    nch = 48
    I, Q = S.pp_case(nch, 50, seed=19)
    calls, setters, plain = _pp_setup(nch, 4)
    ev0 = [(None, 0, "startAutoI2SerrorDetection")]
    want = H.pp_expected(I, Q, ev0, calls, setters)
    p = aux.PreProcessorBatch(nch)
    p.startAutoI2SerrorDetection()
    got = drive_pp(p, I, Q, calls, setters, plain, path=path)
    for j, (g, w) in enumerate(zip(got, want)):
        assert_rows(j, g[0], w[0], "I_out")
        assert_rows(j, g[1], w[1], "Q_out")
        assert np.array_equal(g[2], w[2]), (j, np.argwhere(g[2] != w[2])[:4])
    # the walking channels (I one sample late) really change correction while they skip calls
    walked = [c for c in range(2, nch, 4) if len(set(w[2][c, 1] for w in want)) >= 3]
    assert walked, "no channel walked +1 -> -1"
    p.close()


# ---------------------------------------------------------------- I/Q generator
@pytest.mark.parametrize("path", ["device", "host"])
def test_generator_subsets_in_place_history(aux, path):
    """Back-to-back 1- and 2-block calls on the same channels (the history is rewritten in place), calls shorter than the
    256-sample history, calls across the 4096-sample segments, alternation with full calls (which flip the handle's
    history buffers), gain balance set on unlisted channels."""
    nch = 40
    X = S.iq_case(nch, 120, seed=23)
    rng = np.random.default_rng(6)
    full = np.arange(nch, dtype=np.uint32)
    a, b = rng.permutation(nch)[:13].astype(np.uint32), rng.permutation(nch)[:27].astype(np.uint32)
    calls = [(a, 1), (a, 1), (a, 2), (a, 1), (full, 1), (b, 2), (a, 1), (full, 3), (b, 1), (b, 1), (a, 36), (b, 2), (full, 2), (a, 1)]
    calls += H.random_calls(rng, nch, 8, 30)
    plain = {4, 7, 12}
    ev0 = [(c, 0, "setGainBalance", 1.0 + 0.01 * c) for c in range(0, nch, 3)]
    setters = {}
    for j in (1, 5, 9, 15):
        unlisted = np.setdiff1d(np.arange(nch), calls[j][0])
        if len(unlisted):
            setters[j] = [(int(unlisted[0]), "setGainBalance", 0.9 + 0.01 * j)]
    want = H.iq_expected(X, ev0, calls, setters)
    g = aux.IQGeneratorBatch(nch)
    for e in ev0:
        g.setGainBalance(e[0], e[3])
    got = drive_iq(g, X, calls, setters, plain, path=path)
    for j, (gg, w) in enumerate(zip(got, want)):
        assert_rows(j, gg[0], w[0], "I_out")
        assert_rows(j, gg[1], w[1], "Q_out")
    g.close()


# ---------------------------------------------------------------- grabber
def _grab_device(g, nch, sentinel):
    import torch
    out = torch.full((nch, 512), sentinel, dtype=torch.int16, device="cuda:0")
    r = g.L.sdr_grabber_grab_device(g.h, out.data_ptr(), None)
    torch.cuda.synchronize()
    return r, out.cpu().numpy()


def _spectrum_device(g, nch, ids=None):
    import torch
    n = nch if ids is None else len(ids)
    out = torch.full((n, 256), 12345.0, dtype=torch.float32, device="cuda:0")
    if ids is None:
        r = g.L.sdr_grabber_spectrum_device(g.h, None, 0, out.data_ptr(), None)
    else:
        d = torch.from_numpy(np.asarray(ids, np.int32)).to("cuda:0")
        r = g.L.sdr_grabber_spectrum_device(g.h, d.data_ptr(), n, out.data_ptr(), None)
    torch.cuda.synchronize()
    return r, out.cpu().numpy()


def check_grabber(aux, g, nch, snap, valid, fresh, j, rng):
    """Every reader of the grabber against the oracle's snapshots in the (possibly mixed) state; rows of channels without a
    snapshot must keep a sentinel."""
    from oracle import aux_lib as A
    assert [g.newDataAvailable(c) for c in range(nch)] == list(fresh.f), j
    spec = np.zeros((nch, 256), np.float32)
    if valid.any():
        spec[valid] = A.grab_spectrum(snap[valid].astype(np.int16))
    pick = rng.permutation(nch)[:max(1, nch // 2)]
    o = np.full((len(pick), 256), 777.0, np.float32)
    r = g.spectrum(pick, out=o)
    assert (r is None) == (not valid[pick].any())
    assert np.array_equal(o[valid[pick]].view(np.uint32), spec[pick][valid[pick]].view(np.uint32)) and (o[~valid[pick]] == 777.0).all()
    r, o = _spectrum_device(g, nch)
    assert r == int(valid.any())
    assert np.array_equal(o[valid].view(np.uint32), spec[valid].view(np.uint32)) and (o[~valid] == 12345.0).all()
    r, o = _spectrum_device(g, nch, pick)
    assert r == int(valid[pick].any())
    assert np.array_equal(o[valid[pick]].view(np.uint32), spec[pick][valid[pick]].view(np.uint32)) and (o[~valid[pick]] == 12345.0).all()
    assert [g.newDataAvailable(c) for c in range(nch)] == list(fresh.f), "a spectrum is not a grab()"
    if j % 3 == 1:
        r, o = _grab_device(g, nch, 0x5A5A)
        fresh.grab(None)
        assert r == int(valid.any())
        assert np.array_equal(o[valid].astype(np.int32), snap[valid]) and (o[~valid] == 0x5A5A).all()
    elif j % 2 == 0:
        o = np.full((len(pick), 512), 0x5A5A, np.int16)
        r = g.grab(pick, out=o)
        fresh.grab(pick)
        assert (r is None) == (not valid[pick].any())
        assert np.array_equal(o[valid[pick]].astype(np.int32), snap[pick][valid[pick]]) and (o[~valid[pick]] == 0x5A5A).all()
    assert [g.newDataAvailable(c) for c in range(nch)] == list(fresh.f), j


def drive_grab(g, I, Q, calls, pos=None, id_map=None, plain=()):
    import torch
    pos = np.zeros(I.shape[0], np.int64) if pos is None else pos
    for j, (ids, nb) in enumerate(calls):
        i, q = H.gather_rows(I, ids, pos, nb), H.gather_rows(Q, ids, pos, nb)
        pos[ids] += nb
        g.process(_dev(i), _dev(q), n_blocks=nb, channels=None if j in plain else (ids if id_map is None else id_map[ids]))
        torch.cuda.synchronize()
        yield j


def test_grabber_out_of_phase_subsets(aux):
    """1-block subset calls leave the channels' pair phases apart; channels 0 and 1 are never processed.  After every call:
    newDataAvailable, grab (rows with a sentinel where no snapshot exists), the host and device spectra, grab_device."""
    nch = 37
    I, Q = S.pp_case(nch, 30, seed=29)
    rng = np.random.default_rng(8)
    calls = [(ids + 2, nb) for ids, nb in H.random_calls(rng, nch - 2, 18, 20, sizes=(1, 1, 2, 1, 3, 1))]
    want = H.grab_expected(I, Q, calls)
    g = aux.GrabberBatch(nch)
    fresh = H.FreshModel(nch)
    for j in drive_grab(g, I, Q, calls):
        snap, valid, completed = want[j]
        fresh.after_call(completed)
        check_grabber(aux, g, nch, snap, valid, fresh, j, rng)
    assert not want[-1][1][:2].any() and want[-1][1][2:].any()
    g.close()


# ---------------------------------------------------------------- checkpoints
def test_export_import_moves_channels_bit_for_bit(aux):
    """Each block's channels, exported from a 48-channel handle after a subset sequence, go to other slots of an
    80-channel handle that has run an odd number of blocks (other history buffer, other grabber parity); then both handles
    run on.  Both equal the oracle over each channel's concatenated stream."""
    import torch
    nch, big = 48, 80
    I, Q = S.pp_case(nch, 60, seed=31)
    X = S.iq_case(nch, 60, seed=32)
    rng = np.random.default_rng(10)
    first = H.random_calls(rng, nch, 9, 25, sizes=(1, 3, 2, 1, 5))
    cont = H.random_calls(rng, nch, 8, 25, sizes=(2, 1, 4, 1))
    calls = first + cont
    slot = rng.permutation(big)[:nch]  # channel c of the small handles -> slot[c] of the big ones
    k = len(first)
    pp_set = {2: [(5, "swapIQ", 1)], k: [(9, "setI2SerrorCompensation", 1), (13, "swapIQ", 1)]}
    ev0 = [(None, 0, "startAutoI2SerrorDetection")]
    iq_ev0 = [(c, 0, "setGainBalance", 1.03) for c in range(1, nch, 4)]
    iq_set = {k: [(7, "setGainBalance", 0.96)]}
    want_pp = H.pp_expected(I, Q, ev0, calls, pp_set)
    want_iq = H.iq_expected(X, iq_ev0, calls, iq_set)
    want_gr = H.grab_expected(I, Q, calls)

    def junk(n, nb):
        return torch.from_numpy(np.random.default_rng(n).integers(-9000, 9000, (n, nb * N)).astype(np.int16)).to("cuda:0")

    # the small handles run the first calls
    p, g, r = aux.PreProcessorBatch(nch), aux.IQGeneratorBatch(nch), aux.GrabberBatch(nch)
    p.startAutoI2SerrorDetection()
    for e in iq_ev0:
        g.setGainBalance(e[0], e[3])
    pos_p, pos_g, pos_r = (np.zeros(nch, np.int64) for _ in range(3))
    drive_pp(p, I, Q, first, pp_set, pos=pos_p)
    drive_iq(g, X, first, iq_set, pos=pos_g)
    list(drive_grab(r, I, Q, first, pos=pos_r))
    blobs = (p.export_state(), g.export_state(), r.export_state())
    assert [b.shape for b in blobs] == [(nch, p.state_bytes), (nch, g.state_bytes), (nch, r.state_bytes)]
    # the big handles: 3 blocks of other input first (odd: the other history buffer, the other grabber parity)
    P, G, R = aux.PreProcessorBatch(big), aux.IQGeneratorBatch(big), aux.GrabberBatch(big)
    P.setI2SerrorCompensation(None, -1)
    G.setGainBalance(None, 1.2)
    z, z2 = junk(big, 3), junk(big, 3)
    P.process(z, z2, torch.empty_like(z), torch.empty_like(z2))
    G.process(z, torch.empty_like(z), torch.empty_like(z2))
    R.process(z, z2)
    P.import_state(slot, blobs[0])
    G.import_state(slot, blobs[1])
    R.import_state(slot, blobs[2])
    for side, (pp, gg, rr, idm) in enumerate(((p, g, r, None), (P, G, R, slot))):
        got_pp = drive_pp(pp, I, Q, cont, {0: pp_set[k]}, pos=pos_p.copy(), id_map=idm)
        got_iq = drive_iq(gg, X, cont, {0: iq_set[k]}, pos=pos_g.copy(), id_map=idm)
        for j in range(len(cont)):
            assert_rows(j, got_pp[j][0], want_pp[k + j][0], "pp I_out side %d" % side)
            assert_rows(j, got_pp[j][1], want_pp[k + j][1], "pp Q_out side %d" % side)
            assert_rows(j, got_iq[j][0], want_iq[k + j][0], "iq I_out side %d" % side)
            assert_rows(j, got_iq[j][1], want_iq[k + j][1], "iq Q_out side %d" % side)
        chans = np.arange(nch) if idm is None else slot
        assert np.array_equal(_status(pp, chans), want_pp[-1][2]), side
        fresh = [rr.newDataAvailable(int(c)) for c in chans]
        for j in drive_grab(rr, I, Q, cont, pos=pos_r.copy(), id_map=idm):
            snap, valid, completed = want_gr[k + j]
            o = np.full((nch, 512), 0x5A5A, np.int16)
            rr.grab(chans, out=o)
            assert np.array_equal(o[valid].astype(np.int32), snap[valid]) and (o[~valid] == 0x5A5A).all(), (side, j)
        assert any(fresh)
    for h in (p, g, r, P, G, R):
        h.close()


def test_import_running_detector_into_fresh_handle(aux):
    """A blob whose detector is running (non-zero counters) imported into a handle that never saw
    startAutoI2SerrorDetection: the detector must keep running there (channel 6 of this case has correction +1 and
    failures counted after 14 blocks, and walks on to -1 after the move)."""
    import torch
    I, Q = S.pp_case(8, 40, seed=41)
    src = aux.PreProcessorBatch(8)
    src.startAutoI2SerrorDetection()
    h = 14 * N
    dI, dQ = _dev(I[:, :h]), _dev(Q[:, :h])
    src.process(dI, dQ, torch.empty_like(dI), torch.empty_like(dQ))
    blob = src.export_state([6])
    st = src.status([6])[0]
    assert st.auto_detect and st.correction == 1 and st.failure_count > 0 and st.success_count > 0
    dst = aux.PreProcessorBatch(6)
    dst.import_state([4], blob)
    x, y = _dev(I[6:7, h:]), _dev(Q[6:7, h:])
    oi, oq = torch.empty_like(x), torch.empty_like(y)
    dst.process(x, y, oi, oq, channels=[4])
    from oracle import aux_lib as A
    want = A.run("pp", (I[6:7], Q[6:7]), [(None, 0, "startAutoI2SerrorDetection")])
    assert want[2][0, 1] == -1
    assert np.array_equal(oi.cpu().numpy(), want[0][:, h:]) and np.array_equal(oq.cpu().numpy(), want[1][:, h:])
    assert np.array_equal(_status(dst, [4]), want[2][:, :6])
    src.close(); dst.close()


# ---------------------------------------------------------------- the graph
def test_preprocessor_then_receiver_on_the_same_ids(aux):
    """I2S in -> pre-processor -> receiver, both advanced with the same id list on device int16 planes: each channel equals
    the oracle chain (oracle pre-processor, then oracle receiver) over its own blocks."""
    import torch
    import audiosdr_b200 as A
    import signals as RS
    from subset_harness import oracle_calls
    nch = 24
    I, Q = S.pp_case(nch, 30, seed=43)
    rng = np.random.default_rng(12)
    calls = H.random_calls(rng, nch, 10, 24)
    ev0 = [(None, 0, "startAutoI2SerrorDetection")]
    want_pp = H.pp_expected(I, Q, ev0, calls)
    pos = H.positions(nch, calls)
    PI, PQ = np.zeros_like(I), np.zeros_like(Q)  # each channel's own pre-processor output stream
    for j, (ids, nb) in enumerate(calls):
        for i, c in enumerate(ids):
            z = slice(int(pos[j][c]) * N, int(pos[j + 1][c]) * N)
            PI[c, z], PQ[c, z] = want_pp[j][0][i], want_pp[j][1][i]
    _, _, rx_ev = RS.make(4, list(range(nch)), 1)
    want_rx = oracle_calls(PI, PQ, rx_ev, calls)
    p = aux.PreProcessorBatch(nch)
    p.startAutoI2SerrorDetection()
    rx = A.SdrBatch(nch)
    rx.configure([(None if e[0] == 0xFFFFFFFF else e[0], e[2]) + tuple(e[3:]) for e in rx_ev])
    own = np.zeros(nch, np.int64)
    for j, (ids, nb) in enumerate(calls):
        di, dq = _dev(H.gather_rows(I, ids, own, nb)), _dev(H.gather_rows(Q, ids, own, nb))
        own[ids] += nb
        oi, oq = torch.empty_like(di), torch.empty_like(dq)
        p.process(di, dq, oi, oq, n_blocks=nb, channels=ids)
        audio = torch.empty((len(ids), nb * N), dtype=torch.float32, device="cuda:0")
        rx.process(oi, oq, audio, n_blocks=nb, channels=ids)
        got = audio.cpu().numpy()
        assert np.array_equal(got.view(np.uint32), want_rx[j][0].view(np.uint32)), j
    p.close(); rx.close()


# ---------------------------------------------------------------- identity and rejection
def test_identity_ids_and_null_equal_the_plain_call(aux):
    import torch
    nch = 20
    I, Q = S.pp_case(nch, 12, seed=47)
    X = S.iq_case(nch, 12, seed=48)
    ar = np.arange(nch, dtype=np.uint32)
    outs = []
    for mode in ("plain", "arange", "null"):
        p, g, r = aux.PreProcessorBatch(nch), aux.IQGeneratorBatch(nch), aux.GrabberBatch(nch)
        p.startAutoI2SerrorDetection([c for c in range(nch) if c % 2])
        p.setI2SerrorCompensation([c for c in range(nch) if c % 2 == 0], 1)
        res = []
        for a, b in ((0, 3), (3, 4), (4, 9), (9, 12)):
            z = slice(a * N, b * N)
            di, dq, dx = _dev(I[:, z]), _dev(Q[:, z]), _dev(X[:, z])
            oi, oq, xi, xq = (torch.empty_like(di) for _ in range(4))
            if mode == "plain":
                p.process(di, dq, oi, oq); g.process(dx, xi, xq); r.process(di, dq)
            elif mode == "arange":
                p.process(di, dq, oi, oq, channels=ar); g.process(dx, xi, xq, channels=ar); r.process(di, dq, channels=ar)
            else:
                L, nb, s = p.L, b - a, None
                assert L.sdr_preproc_process_device_subset(p.h, None, nch, di.data_ptr(), dq.data_ptr(), di.stride(0), oi.data_ptr(), oq.data_ptr(), oi.stride(0), nb, s) == 0
                assert L.sdr_iqgen_process_device_subset(g.h, None, nch, dx.data_ptr(), dx.stride(0), xi.data_ptr(), xq.data_ptr(), xi.stride(0), nb, s) == 0
                assert L.sdr_grabber_process_device_subset(r.h, None, nch, di.data_ptr(), dq.data_ptr(), di.stride(0), nb, s) == 0
            res += [t.cpu().numpy() for t in (oi, oq, xi, xq)] + [r.grab(), _status(p)]
        outs.append(res)
        for h in (p, g, r):
            h.close()
    for other in outs[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(outs[0], other))


def test_rejected_id_lists_change_nothing(aux):
    import torch
    nch = 10
    I, Q = S.pp_case(nch, 4, seed=53)
    ref_p, ref_g, ref_r = aux.PreProcessorBatch(nch), aux.IQGeneratorBatch(nch), aux.GrabberBatch(nch)
    p, g, r = aux.PreProcessorBatch(nch), aux.IQGeneratorBatch(nch), aux.GrabberBatch(nch)
    for h in (ref_p, p):
        h.startAutoI2SerrorDetection()
    dI, dQ = _dev(I[:, :2 * N]), _dev(Q[:, :2 * N])
    for pp, gg, rr in ((ref_p, ref_g, ref_r), (p, g, r)):
        pp.process(dI, dQ, torch.empty_like(dI), torch.empty_like(dQ)); gg.process(dI, torch.empty_like(dI), torch.empty_like(dI)); rr.process(dI[:, :N], dQ[:, :N])
    p.swapIQ(3, True)  # pending: a rejected call must not apply it either
    ref_p.swapIQ(3, True)
    x, y = _dev(I[:2, 2 * N:3 * N]), _dev(Q[:2, 2 * N:3 * N])
    oi, oq = torch.full_like(x, 0x5A5A), torch.full_like(y, 0x5A5A)
    bad = [(np.array([1, 1], np.uint32), 2), (np.array([1, nch], np.uint32), 2), (np.array([0], np.uint32), 0), (None, nch - 1), (None, 2)]
    for ids, n in bad:
        ptr = ids.ctypes.data if ids is not None else None
        assert p.L.sdr_preproc_process_device_subset(p.h, ptr, n, x.data_ptr(), y.data_ptr(), x.stride(0), oi.data_ptr(), oq.data_ptr(), oi.stride(0), 1, None) == -1
        assert g.L.sdr_iqgen_process_device_subset(g.h, ptr, n, x.data_ptr(), x.stride(0), oi.data_ptr(), oq.data_ptr(), oi.stride(0), 1, None) == -1
        assert r.L.sdr_grabber_process_device_subset(r.h, ptr, n, x.data_ptr(), y.data_ptr(), x.stride(0), 1, None) == -1
        ho, hq = np.full((2, N), 0x5A5A, np.int16), np.full((2, N), 0x5A5A, np.int16)
        hi, hqi = np.ascontiguousarray(I[:2, :N]), np.ascontiguousarray(Q[:2, :N])
        assert p.L.sdr_preproc_process_host_subset(p.h, ptr, n, hi.ctypes.data, hqi.ctypes.data, N, ho.ctypes.data, hq.ctypes.data, N, 1) == -1
        assert g.L.sdr_iqgen_process_host_subset(g.h, ptr, n, hi.ctypes.data, N, ho.ctypes.data, hq.ctypes.data, N, 1) == -1
        assert (ho == 0x5A5A).all() and (hq == 0x5A5A).all()
    torch.cuda.synchronize()
    assert (oi.cpu().numpy() == 0x5A5A).all() and (oq.cpu().numpy() == 0x5A5A).all()
    with pytest.raises(aux.AuxError):
        p.import_state([0], np.zeros((1, p.state_bytes), np.uint8))  # not a blob
    # nothing moved: the next call equals the handles that never saw the rejected calls
    dI, dQ = _dev(I[:, 2 * N:]), _dev(Q[:, 2 * N:])
    res = []
    for pp, gg, rr in ((ref_p, ref_g, ref_r), (p, g, r)):
        oi, oq, xi, xq = (torch.empty_like(dI) for _ in range(4))
        pp.process(dI, dQ, oi, oq); gg.process(dI, xi, xq); rr.process(dI[:, :N], dQ[:, :N])
        res.append([t.cpu().numpy() for t in (oi, oq, xi, xq)] + [_status(pp), rr.grab(), [rr.newDataAvailable(c) for c in range(nch)]])
    assert all(np.array_equal(a, b) for a, b in zip(res[0], res[1]))
    for h in (ref_p, ref_g, ref_r, p, g, r):
        h.close()
