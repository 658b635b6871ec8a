"""GPU tier: the pre-processor's per-block status records (sdr_preproc_process_device_status / _host_status, SDR_PP_BS_*)
on the CUDA build, bit for bit against the oracle's records (tests/pp_records.py), and the calls with records against twin
handles running the plain calls.  The CPU tier (test_emu_pp_block_status.py) runs the same cases on the host emulation."""
import os

import numpy as np
import pytest

import aux_signals as S
import pp_edge_signals as E
import pp_records as R

pytestmark = pytest.mark.gpu
NF = 6
SENTINEL = 0x5A5A5A5A
_cache = {}


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
    return np.array([[s.auto_detect, s.correction, s.failure_count, s.success_count, s.saved_sample, s.swap]
                     for s in p.status(channels)], np.int32)


def _set(p, c, name, *arg):
    getattr(p, name)(*([None if c is None else np.atleast_1d(np.asarray(c, np.uint32))] + list(arg)))


def edge_case(placement):
    if placement not in _cache:
        I, Q, ev, lay = E.build(placement)
        _cache[placement] = (I, Q, ev, lay, R.oracle_records(I, Q, ev))
    return _cache[placement]


def run_calls(p, I, Q, ev, ends, host=False, channels=None, guard=64, plain=None):
    """Calls [0, ends[0]), [ends[0], ends[1]), ... with records; an event (row, block, setter, *arg) at block b is queued
    before the call that starts at b, on channel channels[row] (channels None: row).  Every record buffer is followed by
    `guard` sentinel words that must stay intact, and comes back without a sentinel in range.  plain: a twin handle that
    runs the same calls without records; its outputs and state must equal p's.  Returns (out I, out Q, records
    [n_blocks, 6, rows], [status of the listed channels after each call])."""
    import torch
    starts = [0] + list(ends[:-1])
    assert all(e[1] in starts for e in ev)
    rows = I.shape[0]
    slot = (lambda c: c) if channels is None else (lambda c: None if c is None else channels[c])
    oi, oq = np.empty_like(I), np.empty_like(Q)
    recs, sts = [], []
    for pos, end in zip(starts, ends):
        for h in (p, plain) if plain is not None else (p,):
            for c, b, name, *arg in ev:
                if b == pos:
                    _set(h, slot(c) if c is not None else (None if channels is None else channels), name, *arg)
        nb, z = end - pos, slice(pos * 128, end * 128)
        n = nb * NF * rows
        if host:
            raw = np.full(n + guard, SENTINEL, np.int32)
            a, b = np.empty((rows, nb * 128), np.int16), np.empty((rows, nb * 128), np.int16)
            p.process_host(np.ascontiguousarray(I[:, z]), np.ascontiguousarray(Q[:, z]), a, b, n_blocks=nb, channels=channels,
                           block_status=raw[:n].reshape(nb, NF, rows))
            if plain is not None:
                a2, b2 = np.empty_like(a), np.empty_like(b)
                plain.process_host(np.ascontiguousarray(I[:, z]), np.ascontiguousarray(Q[:, z]), a2, b2, n_blocks=nb, channels=channels)
                assert np.array_equal(a, a2) and np.array_equal(b, b2)
        else:
            dI, dQ = _dev(I[:, z]), _dev(Q[:, z])
            dOi, dOq = torch.empty_like(dI), torch.empty_like(dQ)
            draw = torch.full((n + guard,), SENTINEL, dtype=torch.int32, device="cuda:0")
            p.process(dI, dQ, dOi, dOq, n_blocks=nb, channels=channels, block_status=draw[:n].view(nb, NF, rows))
            if plain is not None:
                dOi2, dOq2 = torch.empty_like(dI), torch.empty_like(dQ)
                plain.process(dI, dQ, dOi2, dOq2, n_blocks=nb, channels=channels)
                assert torch.equal(dOi, dOi2) and torch.equal(dOq, dOq2)
            torch.cuda.synchronize()
            a, b, raw = dOi.cpu().numpy(), dOq.cpu().numpy(), draw.cpu().numpy()
        assert not (raw[:n] == SENTINEL).any() and (raw[n:] == SENTINEL).all()
        oi[:, z], oq[:, z] = a, b
        recs.append(raw[:n].reshape(nb, NF, rows))
        st = _status(p, channels)
        assert np.array_equal(recs[-1][-1].T, st)  # the last record is get_status after the call
        if plain is not None:
            assert np.array_equal(_status(plain, channels), st)
        sts.append(st)
    return oi, oq, np.concatenate(recs), sts


def check(aux, I, Q, ev, ends, host=False):
    want = R.oracle_records(I, Q, ev)
    p, t = aux.PreProcessorBatch(I.shape[0]), aux.PreProcessorBatch(I.shape[0])
    oi, oq, rec, _ = run_calls(p, I, Q, ev, ends, host=host, plain=t)
    p.close(); t.close()
    assert np.array_equal(oi, want[0]) and np.array_equal(oq, want[1])
    assert np.array_equal(rec, want[3]), np.argwhere(rec != want[3])[:5]
    return want


def _schedules(nb, x):
    start = 0 if nb < 100 else x - 3
    return {"ones": ([start] if start else []) + list(range(start + 1, nb + 1)), "edge": [x // 2, x + 1, nb], "all": [nb]}


# ---------------------------------------------------------------- the cases of the CPU tier, device and host forms
@pytest.mark.parametrize("sched", ["ones", "edge", "all"])
@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_records_at_the_knife_edge(aux, placement, sched):
    I, Q, ev, lay, want = edge_case(placement)
    nb, x = I.shape[1] // 128, lay["block"]
    check(aux, I, Q, ev, _schedules(nb, x)[sched])
    if sched == "edge":
        check(aux, I, Q, ev, _schedules(nb, x)[sched], host=True)


def _cases():
    steps = S.pp_case(16, 48, seed=9) + ([(None, 0, "startAutoI2SerrorDetection")], [3, 46, 48])
    stops = S.pp_case(8, 1004, seed=3) + ([(None, 0, "startAutoI2SerrorDetection")], [990, 1004])
    off_ev = [(c, 0, "setI2SerrorCompensation", (c % 3) - 1) for c in range(12)] + [(c, 0, "swapIQ", 1) for c in range(12) if (c // 3) % 2]
    off = S.pp_case(12, 8, seed=13) + (off_ev, [1, 3, 8])
    ends = [5, 10, 15, 20, 25, 30, 36]
    rng = np.random.default_rng(11)
    names = [("stopAutoI2SerrorDetection",), ("startAutoI2SerrorDetection",), ("setI2SerrorCompensation", 1),
             ("setI2SerrorCompensation", -1), ("setI2SerrorCompensation", 0), ("swapIQ", 1), ("swapIQ", 0)]
    sev = [(None, 0, "startAutoI2SerrorDetection")] + [(int(c), pos, *names[rng.integers(len(names))])
                                                        for pos in ends[:-1] for c in rng.choice(40, 10, replace=False)]
    setters = S.pp_case(40, 36, seed=5) + (sev, ends)
    rends = [3, 4, 11, 17, 24]
    starts = [0] + rends[:-1]
    rev = [(c, max(s for s in starts if s <= b), *rest) for c, b, *rest in S.pp_events(48, 24)]
    ragged = S.pp_case(48, 24, seed=17) + (rev, rends)
    return dict(steps_twice=steps, stops_inside=stops, detector_off=off, setters_between_calls=setters, ragged=ragged)


@pytest.mark.parametrize("host", [False, True])
@pytest.mark.parametrize("name", ["steps_twice", "stops_inside", "detector_off", "setters_between_calls", "ragged"])
def test_records_cases(aux, name, host):
    I, Q, ev, ends = _cases()[name]
    check(aux, I, Q, ev, ends, host=host)


def test_records_one_block_calls(aux):
    I, Q = S.pp_case(48, 24, seed=17)
    ev = [(c, 0, *rest) for c, b, *rest in S.pp_events(48, 24)]
    check(aux, I, Q, ev, list(range(1, 25)))


# ---------------------------------------------------------------- subsets
@pytest.mark.parametrize("host", [False, True])
def test_records_on_random_subsets(aux, host):
    """A handle of 173 channels; each round lists a random half of them, then the other half, in random order, so that
    every channel advances by the round's blocks.  Columns map to ids, unlisted channels keep their state during the other
    half's call, every record equals the oracle's for that channel's own stream."""
    n, rounds = 173, [3, 1, 7, 2, 5]
    nb = sum(rounds)
    I, Q = S.pp_case(n, nb, seed=29)
    ev = [(c, 0, "setI2SerrorCompensation", (c % 3) - 1) for c in range(n) if c % 4 == 1] + [(c, 0, "swapIQ", 1) for c in range(0, n, 5)]
    ev += [(c, 0, "startAutoI2SerrorDetection") for c in range(n) if c % 4 in (0, 2)]
    want = R.oracle_records(I, Q, ev)
    p = aux.PreProcessorBatch(n)
    for c, b, name, *arg in ev:
        _set(p, c, name, *arg)
    rng = np.random.default_rng(4)
    pos = 0
    for nbr in rounds:
        perm = rng.permutation(n).astype(np.uint32)
        k = int(rng.integers(1, n))
        for ids, other in ((perm[:k], perm[k:]), (perm[k:], perm[:k])):
            before = _status(p, other)
            z = slice(pos * 128, (pos + nbr) * 128)
            _, _, rec, _ = run_calls(p, I[ids][:, z], Q[ids][:, z], [], [nbr], host=host, channels=ids, guard=n * NF)
            assert np.array_equal(rec, want[3][pos:pos + nbr][:, :, ids])
            assert np.array_equal(_status(p, other), before)
        pos += nbr
    assert np.array_equal(_status(p), want[2][:, :6])
    p.close()


# ---------------------------------------------------------------- full size
def test_records_full_size(aux):
    """4 096 channels x 256 blocks, rows interleaved: detector, +1, -1, 0.  Sampled channels against the oracle, every row
    against a twin handle running the plain call."""
    import torch
    nch, nb = 4096, 256
    bI, bQ = S.pp_case(64, nb, seed=41)
    I, Q = np.tile(bI, (nch // 64, 1)), np.tile(bQ, (nch // 64, 1))
    def setup(h):
        for k, corr in ((1, 1), (2, -1), (3, 0)):
            h.setI2SerrorCompensation(np.arange(k, nch, 4, dtype=np.uint32), corr)
        h.startAutoI2SerrorDetection(np.arange(0, nch, 4, dtype=np.uint32))
        h.swapIQ(np.arange(0, nch, 8, dtype=np.uint32), True)
    p, t = aux.PreProcessorBatch(nch), aux.PreProcessorBatch(nch)
    setup(p); setup(t)
    dI, dQ = _dev(I), _dev(Q)
    o = [torch.empty_like(dI) for _ in range(4)]
    rec = torch.full((nb, NF, nch), SENTINEL, dtype=torch.int32, device="cuda:0")
    p.process(dI, dQ, o[0], o[1], block_status=rec)
    t.process(dI, dQ, o[2], o[3])
    torch.cuda.synchronize()
    assert torch.equal(o[0], o[2]) and torch.equal(o[1], o[3])
    r = rec.cpu().numpy()
    st = _status(p)
    assert np.array_equal(st, _status(t)) and np.array_equal(r[-1].T, st) and not (r == SENTINEL).any()
    sample = np.sort(np.random.default_rng(2).choice(nch, 48, replace=False))
    ev = []
    for i, c in enumerate(sample):
        if c % 4:
            ev.append((i, 0, "setI2SerrorCompensation", {1: 1, 2: -1, 3: 0}[c % 4]))
        else:
            ev.append((i, 0, "startAutoI2SerrorDetection"))
        if c % 8 == 0:
            ev.append((i, 0, "swapIQ", 1))
    want = R.oracle_records(I[sample], Q[sample], ev)
    assert np.array_equal(r[:, :, sample], want[3])
    assert np.array_equal(o[0].cpu().numpy()[sample], want[0]) and np.array_equal(o[1].cpu().numpy()[sample], want[1])
    p.close(); t.close()


# ---------------------------------------------------------------- checkpoint
def test_records_continue_across_a_checkpoint(aux):
    """A running detector exported just before the knife edge and imported into other slots of a fresh, larger handle
    continues its records bit for bit."""
    I, Q, ev, lay, want = edge_case("rollover")
    nk, nb, x = I.shape[0], I.shape[1] // 128, lay["block"]
    a = aux.PreProcessorBatch(nk)
    _, _, r1, _ = run_calls(a, I[:, :x * 128], Q[:, :x * 128], ev, [x - 2, x])
    blobs = a.export_state()
    a.close()
    slots = (np.arange(nk)[::-1] * 3 + 5).astype(np.uint32)
    b = aux.PreProcessorBatch(int(slots.max()) + 9)
    b.import_state(slots, blobs)
    _, _, r2, _ = run_calls(b, I[:, x * 128:], Q[:, x * 128:], [], [1, 2, nb - x], channels=slots)
    b.close()
    assert np.array_equal(np.concatenate([r1, r2]), want[3])


# ---------------------------------------------------------------- rejected calls
def test_rejected_calls_change_nothing(aux):
    import torch
    n, nb = 40, 4
    I, Q = S.pp_case(n, nb, seed=23)
    p = aux.PreProcessorBatch(n)
    p.startAutoI2SerrorDetection(np.arange(0, n, 2, dtype=np.uint32))
    p.setI2SerrorCompensation(np.arange(1, n, 2, dtype=np.uint32), 1)
    dI, dQ = _dev(I), _dev(Q)
    p.process(dI, dQ, torch.empty_like(dI), torch.empty_like(dQ), n_blocks=1)
    torch.cuda.synchronize()
    st, launches = _status(p), p.launch_count
    oi, oq = torch.full_like(dI, 7), torch.full_like(dQ, 7)
    flat = torch.full((nb * NF * n + 4,), SENTINEL, dtype=torch.int32, device="cuda:0")
    L = p.L
    args = (dI.data_ptr(), dQ.data_ptr(), dI.stride(0), oi.data_ptr(), oq.data_ptr(), oi.stride(0), nb)
    EINVAL = -1  # SDR_AUX_EINVAL
    assert L.sdr_preproc_process_device_status(p.h, None, n, *args, flat.data_ptr() + 4, None) == EINVAL
    bad = [np.array([1, 2, 1], np.uint32), np.array([n], np.uint32), np.zeros(1, np.uint32)[:0]]
    for ids in bad:
        assert L.sdr_preproc_process_device_status(p.h, ids.ctypes.data, len(ids), *args, flat.data_ptr(), None) == EINVAL
    hI, hQ = np.ascontiguousarray(I), np.ascontiguousarray(Q)
    ho, hq = np.full_like(hI, 7), np.full_like(hQ, 7)
    hraw = np.full(nb * NF * n + 4, SENTINEL, np.int32)
    assert L.sdr_preproc_process_host_status(p.h, None, n, hI.ctypes.data, hQ.ctypes.data, hI.shape[1], ho.ctypes.data, hq.ctypes.data,
                                             ho.shape[1], nb, hraw.ctypes.data + 4) == EINVAL
    assert L.sdr_preproc_process_host_status(p.h, bad[0].ctypes.data, 3, hI.ctypes.data, hQ.ctypes.data, hI.shape[1], ho.ctypes.data,
                                             hq.ctypes.data, ho.shape[1], nb, hraw.ctypes.data) == EINVAL
    torch.cuda.synchronize()
    assert p.launch_count == launches and np.array_equal(_status(p), st)
    assert (oi == 7).all() and (oq == 7).all() and (flat == SENTINEL).all() and (ho == 7).all() and (hq == 7).all() and (hraw == SENTINEL).all()
    with pytest.raises(aux.AuxError):
        p.process(dI[:2], dQ[:2], oi[:2], oq[:2], channels=[3, 3], block_status=torch.empty((nb, NF, 2), dtype=torch.int32, device="cuda:0"))
    assert p.launch_count == launches and np.array_equal(_status(p), st) and (oi == 7).all()
    p.close()


# ---------------------------------------------------------------- the whole graph
def test_preprocessor_and_receiver_records_on_one_id_list(aux):
    """I2S in -> pre-processor -> receiver on one id list and one stream, both with records: the pre-processor's records
    are the oracle's, and the receiver's records and audio are those of a twin receiver fed the oracle's pre-processor
    output with the same calls."""
    import torch
    import audiosdr_b200 as rxlib
    import signals as RS
    n, rounds = 24, [4, 9, 3]
    nb = sum(rounds)
    I, Q = S.pp_case(n, nb, seed=37)
    ev = [(None, 0, "startAutoI2SerrorDetection")]
    want = R.oracle_records(I, Q, ev)
    _, _, rev = RS.make(4, list(range(n)), 1)
    pp = aux.PreProcessorBatch(n)
    pp.startAutoI2SerrorDetection()
    rx, twin = rxlib.SdrBatch(n), rxlib.SdrBatch(n)
    for h in (rx, twin):
        h.configure([(e[0], e[2]) + tuple(e[3:]) for e in rev])
    stream = torch.cuda.Stream()
    rng = np.random.default_rng(8)
    pos = 0
    for nbr in rounds:
        perm = rng.permutation(n).astype(np.uint32)
        for ids in (perm[:n // 3], perm[n // 3:]):
            z = slice(pos * 128, (pos + nbr) * 128)
            k = len(ids)
            with torch.cuda.stream(stream):
                dI, dQ = _dev(I[ids][:, z]), _dev(Q[ids][:, z])
                oI, oQ = torch.empty_like(dI), torch.empty_like(dQ)
                prec = torch.empty((nbr, NF, k), dtype=torch.int32, device="cuda:0")
                audio = torch.empty((k, nbr * 128), dtype=torch.float32, device="cuda:0")
                rrec = torch.empty((nbr, rxlib.BS_FIELDS, k), dtype=torch.int32, device="cuda:0")
                pp.process(dI, dQ, oI, oQ, n_blocks=nbr, stream=stream, channels=ids, block_status=prec)
                rx.process(oI, oQ, audio, n_blocks=nbr, stream=stream, channels=ids, block_status=rrec)
            stream.synchronize()
            assert np.array_equal(prec.cpu().numpy(), want[3][pos:pos + nbr][:, :, ids])
            assert np.array_equal(oI.cpu().numpy(), want[0][ids][:, z]) and np.array_equal(oQ.cpu().numpy(), want[1][ids][:, z])
            tI, tQ = _dev(want[0][ids][:, z]), _dev(want[1][ids][:, z])
            taudio = torch.empty_like(audio)
            trec = torch.empty_like(rrec)
            twin.process(tI, tQ, taudio, n_blocks=nbr, channels=ids, block_status=trec)
            torch.cuda.synchronize()
            assert torch.equal(audio.view(torch.int32), taudio.view(torch.int32)) and torch.equal(rrec, trec)
        pos += nbr
    pp.close(); rx.close(); twin.close()
