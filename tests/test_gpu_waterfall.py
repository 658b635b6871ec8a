"""GPU tier: averaged waterfall lines (sdr_waterfall_*, sdr_grabber_process_device_waterfall, the graph's _waterfall calls)
on the CUDA libraries, bit for bit against the oracle (tests/waterfall_oracle.py), against the per-pair spectra, across call
cuts, migrations and graph chunkings.  Line buffers are filled with a sentinel: slots a call must not write keep it."""
import os
import subprocess
import sys

import numpy as np
import pytest

import waterfall_oracle as W

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENT = np.uint32(0x7FC0BEEF)  # a NaN no line produces
NCH = 6
# ragged calls: 1-block calls, odd lengths, calls shorter than K pairs, channels skipping calls with different phases
CALLS = [(list(range(NCH)), 1), ([2, 0, 5], 3), ([1, 3], 7), (list(range(NCH)), 2), ([4, 5, 0], 5), ([3], 1), (list(range(NCH)), 1),
         ([5, 1], 9), (list(range(NCH)), 33), ([0, 2, 4], 16), ([1], 2), (list(range(NCH)), 40), ([3, 5], 3)]


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


def _planes(nch, nb, seed):
    """int16 I, Q [nch, 128 nb]: noise, a drifting tone per channel, a few full-scale blocks"""
    rng = np.random.default_rng(seed)
    t = np.arange(nb * 128)
    I = rng.normal(0, 700, (nch, nb * 128))
    Q = rng.normal(0, 700, (nch, nb * 128))
    for c in range(nch):
        f = (5 + 11 * c + 0.001 * t) / 256
        I[c] += 9000 * np.cos(2 * np.pi * f * t)
        Q[c] += 9000 * np.sin(2 * np.pi * f * t)
    I[:, 128 * 5:128 * 6] = 32767
    Q[:, 128 * 6:128 * 7] = -32768
    return np.clip(I, -32768, 32767).astype(np.int16), np.clip(Q, -32768, 32767).astype(np.int16)


def _lines(rows, slots):
    import torch
    return torch.full((rows, slots, 256), int(SENT.view(np.int32)), dtype=torch.int32, device="cuda:0").view(torch.float32)


def _bits(t):
    import torch
    torch.cuda.synchronize()
    return t.view(torch.int32).cpu().numpy().view(np.uint32)


def _gather(I, Q, pos, ids, nb):
    sel = np.asarray(ids)
    cols = [np.arange(pos[c] * 128, (pos[c] + nb) * 128) for c in ids]
    return _dev(np.stack([I[c, k] for c, k in zip(sel, cols)])), _dev(np.stack([Q[c, k] for c, k in zip(sel, cols)]))


def run_calls(aux, gr, wf, I, Q, calls, pos=None):
    """Each call's (lines bits [rows, Lmax, 256], counts) from the device; pos (advanced in place): blocks per channel so far"""
    pos = pos if pos is not None else np.zeros(I.shape[0], np.int64)
    out = []
    for ids, nb in calls:
        dI, dQ = _gather(I, Q, pos, ids, nb)
        t = _lines(len(ids), wf.line_slots(nb))
        ch = None if list(ids) == list(range(gr.n_channels)) else ids
        counts = gr.process(dI, dQ, n_blocks=nb, channels=ch, waterfall=wf, lines=t)
        out.append((_bits(t), counts))
        pos[np.asarray(ids)] += nb
    return out


def check(got, want, what=""):
    for j, ((bits, counts), (lines, wc)) in enumerate(zip(got, want)):
        assert np.array_equal(counts, wc), "%s call %d: counts %s, want %s" % (what, j, counts, wc)
        for i, k in enumerate(counts):
            if not np.array_equal(bits[i, :k], lines[i, :k].view(np.uint32)):
                bad = np.argwhere(bits[i, :k] != lines[i, :k].view(np.uint32))
                raise AssertionError("%s call %d row %d: %d words differ, first at %s" % (what, j, i, len(bad), bad[0]))
            assert (bits[i, k:] == SENT).all(), "%s call %d row %d: a slot past counts was written" % (what, j, i)


@pytest.mark.parametrize("K", [1, 2, 3, 8, 16])
def test_ragged_calls_equal_the_oracle(aux, K):
    total = sum(nb for _, nb in CALLS)
    I, Q = _planes(NCH, total, K)
    gr, wf, twin = aux.GrabberBatch(NCH), aux.WaterfallBatch(NCH, K), aux.GrabberBatch(NCH)
    got = run_calls(aux, gr, wf, I, Q, CALLS)
    check(got, W.waterfall_expected(I, Q, CALLS, K), "K=%d" % K)
    assert sum(int(c.sum()) for _, c in got) > 0
    # the grabber's state is that of plain subset calls
    pos = np.zeros(NCH, np.int64)
    for ids, nb in CALLS:
        dI, dQ = _gather(I, Q, pos, ids, nb)
        twin.process(dI, dQ, n_blocks=nb, channels=ids)
        pos[np.asarray(ids)] += nb
    assert np.array_equal(gr.export_state(), twin.export_state())


def test_k1_lines_are_the_snapshot_spectra(aux):
    I, Q = _planes(NCH, 80, 21)
    calls = [(list(range(NCH)), 3), ([1, 4], 5), (list(range(NCH)), 24), ([0, 5, 2], 1), (list(range(NCH)), 47)]
    gr, wf, twin = aux.GrabberBatch(NCH), aux.WaterfallBatch(NCH, 1), aux.GrabberBatch(NCH)
    got = run_calls(aux, gr, wf, I, Q, calls)
    pos = np.zeros(NCH, np.int64)
    import torch
    for (ids, nb), (bits, counts) in zip(calls, got):
        dI, dQ = _gather(I, Q, pos, ids, nb)
        power = torch.zeros((len(ids), (nb + 1) // 2, 256), dtype=torch.float32, device="cuda:0")
        c2 = twin.process(dI, dQ, n_blocks=nb, channels=ids, power=power)
        pos[np.asarray(ids)] += nb
        assert np.array_equal(counts, c2)
        p = _bits(power)
        for i, k in enumerate(counts):
            assert np.array_equal(bits[i, :k], p[i, :k])


def _grab_blob(gr):
    """The grabber's blobs without the carried block of channels with no pair open (byte 8: the phase; bytes 16-527: the
    carried block): those bytes are never read, and hold the last open pair's first block, which depends on the cuts."""
    b = gr.export_state()
    b[b[:, 8] == 0, 16:528] = 0
    return b


@pytest.mark.parametrize("K", [3, 8])
def test_one_long_call_equals_many_short_ones(aux, K):
    I, Q = _planes(NCH, 120, 30 + K)
    ids = list(range(NCH))
    long_gr, long_wf = aux.GrabberBatch(NCH), aux.WaterfallBatch(NCH, K)
    (bits, counts), = run_calls(aux, long_gr, long_wf, I, Q, [(ids, 120)])
    cuts = [1, 1, 3, 2, 7, 1, 16, 5, 33, 2, 49]
    assert sum(cuts) == 120
    gr, wf = aux.GrabberBatch(NCH), aux.WaterfallBatch(NCH, K)
    parts = run_calls(aux, gr, wf, I, Q, [(ids, nb) for nb in cuts])
    for i in range(NCH):
        short = np.concatenate([b[i, :c[i]] for b, c in parts])
        assert np.array_equal(short, bits[i, :counts[i]])
    assert np.array_equal(_grab_blob(gr), _grab_blob(long_gr))
    assert np.array_equal(wf.export_state(), long_wf.export_state())


@pytest.mark.parametrize("K", [2, 8])
def test_migration_continues_the_lines(aux, K):
    """A channel exported half way through a line with an odd pair phase and imported into another channel of other handles
    (which have run other blocks) continues bit for bit."""
    I, Q = _planes(NCH, 100, 40 + K)
    a_gr, a_wf = aux.GrabberBatch(NCH), aux.WaterfallBatch(NCH, K)
    run_calls(aux, a_gr, a_wf, I, Q, [([0], 2 * K + 3)])  # K + 1 pairs held: K > 1 leaves 1 pair held, phase 1
    gb, wb = a_gr.export_state([0]), a_wf.export_state([0])
    b_gr, b_wf = aux.GrabberBatch(NCH + 2), aux.WaterfallBatch(NCH + 2, K)
    I2, Q2 = _planes(NCH + 2, 100, 99)
    run_calls(aux, b_gr, b_wf, I2, Q2, [(list(range(NCH + 2)), 7), ([3, 1], 4)])
    b_gr.import_state([5], gb)
    b_wf.import_state([5], wb)
    rest = I[0:1, (2 * K + 3) * 128:], Q[0:1, (2 * K + 3) * 128:]
    got_a = run_calls(aux, a_gr, a_wf, I, Q, [([0], 9), ([0], 30)], pos=np.array([2 * K + 3] + [0] * (NCH - 1)))
    ib, qb = np.zeros((NCH + 2, rest[0].shape[1]), np.int16), np.zeros((NCH + 2, rest[0].shape[1]), np.int16)
    ib[5], qb[5] = rest[0][0], rest[1][0]
    got_b = run_calls(aux, b_gr, b_wf, ib, qb, [([5], 9), ([5], 30)])
    for (ba, ca), (bb, cb) in zip(got_a, got_b):
        assert np.array_equal(ca, cb) and np.array_equal(ba, bb)
    assert sum(int(c[0]) for _, c in got_a) > 0
    # and the continuation is the oracle's: the channel's whole stream from the start
    want = W.waterfall_expected(I[:1], Q[:1], [([0], 2 * K + 3), ([0], 9), ([0], 30)], K)[1:]
    check(got_a, want, "migrated")


def test_bad_arguments_change_nothing(aux):
    import torch
    K = 3
    I, Q = _planes(4, 9, 5)
    gr, wf = aux.GrabberBatch(4), aux.WaterfallBatch(4, K)
    run_calls(aux, gr, wf, I, Q, [([1, 3], 3)])  # some state to keep
    g0, w0 = gr.export_state(), wf.export_state()
    dI, dQ = _dev(I[:, :6 * 128]), _dev(Q[:, :6 * 128])
    L = aux.load_library()
    buf = _lines(4 * 4 + 1, 1)  # room for a misaligned view
    good = buf[:4 * 3].view(4, 3, 256)
    def call(g=gr.h, w=wf.h, ids=None, n=4, lines=good.data_ptr()):
        p = np.ascontiguousarray(ids, np.uint32) if ids is not None else None
        counts = np.full(4, 77, np.uint32)
        rc = L.sdr_grabber_process_device_waterfall(g, w, p.ctypes.data if p is not None else None, n, dI.data_ptr(), dQ.data_ptr(),
                                                    dI.stride(0), 6, lines, counts.ctypes.data, None)
        return rc, counts
    other = aux.WaterfallBatch(5, K)
    for kw in ({"lines": good.data_ptr() + 4}, {"lines": None}, {"w": other.h}, {"w": None}, {"ids": [1, 1], "n": 2},
               {"ids": [0, 4], "n": 2}, {"ids": [], "n": 0}):
        rc, counts = call(**kw)
        assert rc == -1, kw
        assert (counts == 77).all()
    torch.cuda.synchronize()
    assert (_bits(buf) == SENT).all()
    assert np.array_equal(gr.export_state(), g0) and np.array_equal(wf.export_state(), w0)
    # a blob of another K does not import
    with pytest.raises(aux.AuxError):
        aux.WaterfallBatch(4, K + 1).import_state([0], w0[:1])
    # the line slots a call must not write keep the sentinel (odd n_blocks, phase 0, K = 1)
    g1, w1 = aux.GrabberBatch(2), aux.WaterfallBatch(2, 1)
    (bits, counts), = run_calls(aux, g1, w1, I[:2], Q[:2], [([0, 1], 5)])
    assert list(counts) == [2, 2] and (bits[:, 2:] == SENT).all() and not (bits[:, :2] == SENT).any()


# ---------------------------------------------------------------- graph
GN = 24
GCALLS = [(None, 17), (None, 64), ("sub", 1), (None, 255), ("sub", 16), (None, 3), (None, 40)]


def _graph_plan(alt):
    """[(ids | None, n_blocks)]: alt first runs the odd channels for 3 blocks, so that rows alternate pair phase and held pairs"""
    rng = np.random.default_rng(8)
    calls = [(np.arange(1, GN, 2, dtype=np.uint32), 3)] if alt else []
    for ids, nb in GCALLS:
        calls.append((rng.permutation(GN)[:GN // 2 + 1].astype(np.uint32) if ids else None, nb))
    return calls


def _inputs(calls):
    import graph_harness as GH
    return GH.inputs("pp", GN, [(i, nb, None) for i, nb in calls])


def graph_run(K, alt):
    """The calls through a GraphBatch with a waterfall: {"lines_j", "counts_j", "gr", "wf"}"""
    import graph_harness as GH
    from audiosdr_b200 import aux, graph
    calls = _graph_plan(alt)
    I, Q = _inputs(calls)
    h = GH.make_handles("pp", GN)
    wf = aux.WaterfallBatch(GN, K)
    g = graph.GraphBatch(h["rx"], preproc=h["pp"], grabber=h["gr"], waterfall=wf)
    out, pos, keep, tickets = {}, 0, [], []
    for j, (ids, nb) in enumerate(calls):
        rows = GN if ids is None else len(ids)
        sel = slice(None) if ids is None else ids.astype(np.int64)
        hI = np.ascontiguousarray(I[sel, pos * 128:(pos + nb) * 128])
        hQ = np.ascontiguousarray(Q[sel, pos * 128:(pos + nb) * 128])
        audio = np.empty((rows, nb * 128), np.int16)
        lines = np.full((rows, wf.line_slots(nb), 256), SENT, np.uint32).view(np.float32)
        t, counts = g.submit_host(hI, hQ, audio, n_blocks=nb, channels=ids, lines=lines)
        keep.append((hI, hQ, audio))
        tickets.append(t)
        if len(tickets) >= 2:
            g.wait_host(tickets[-2])
        out["lines_%d" % j], out["counts_%d" % j] = lines, counts
        pos += nb
    g.wait_host()
    g.close()
    out["gr"], out["wf"] = h["gr"].export_state(), wf.export_state()
    return {k: (v.view(np.uint32) if v.dtype == np.float32 else v) for k, v in out.items()}


def device_run(K, alt):
    """The same calls as the blocks' device calls: pre-processor, then the grabber with the waterfall"""
    import torch
    import graph_harness as GH
    from audiosdr_b200 import aux
    calls = _graph_plan(alt)
    I, Q = _inputs(calls)
    h = GH.make_handles("pp", GN)
    wf = aux.WaterfallBatch(GN, K)
    out, pos = {}, 0
    for j, (ids, nb) in enumerate(calls):
        rows = GN if ids is None else len(ids)
        sel = slice(None) if ids is None else ids.astype(np.int64)
        dI, dQ = _dev(I[sel, pos * 128:(pos + nb) * 128]), _dev(Q[sel, pos * 128:(pos + nb) * 128])
        oI, oQ = torch.empty_like(dI), torch.empty_like(dQ)
        h["pp"].process(dI, dQ, oI, oQ, n_blocks=nb, channels=ids)
        t = _lines(rows, wf.line_slots(nb))
        counts = h["gr"].process(oI, oQ, n_blocks=nb, channels=ids, waterfall=wf, lines=t)
        out["lines_%d" % j], out["counts_%d" % j] = _bits(t), counts
        pos += nb
    out["gr"], out["wf"] = h["gr"].export_state(), wf.export_state()
    return out


CHILD = """
import sys
sys.path[:0] = [%(root)r, %(tests)r]
import numpy as np
import test_gpu_waterfall as T
np.savez(%(path)r, **T.graph_run(%(K)d, %(alt)d))
"""


@pytest.mark.parametrize("K,alt", [(1, 0), (8, 0), (3, 1), (8, 1), (16, 1)])
def test_graph_lines_equal_the_device_call_under_any_chunking(aux, tmp_path, K, alt):
    want = device_run(K, alt)
    assert sum(int(want[k].sum()) for k in want if k.startswith("counts_")) > 0
    for chunks, min_chunk in ((1, 16), (3, 2), (12, 2)):
        path = str(tmp_path / ("c%d.npz" % chunks))
        env = dict(os.environ, SDR_HOST_CHUNKS=str(chunks), SDR_HOST_MIN_CHUNK=str(min_chunk))
        r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT, "tests": os.path.join(ROOT, "tests"), "path": path, "K": K, "alt": alt}],
                           env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        z = np.load(path)
        for k, v in want.items():
            if k == "gr":  # the carried block of a channel with no pair open may differ (sdr_graph.h); everything else is exact
                continue
            assert np.array_equal(z[k], v), (chunks, k)


def test_graph_rejects_plain_calls_and_missing_lines(aux):
    import graph_harness as GH
    from audiosdr_b200 import graph
    h = GH.make_handles("pp", GN)
    wf = aux.WaterfallBatch(GN, 2)
    g = graph.GraphBatch(h["rx"], preproc=h["pp"], grabber=h["gr"], waterfall=wf)
    I = np.zeros((GN, 256), np.int16)
    audio = np.zeros((GN, 256), np.int16)
    L = graph.load_library()
    assert L.sdr_graph_submit_host(g.h, None, GN, I.ctypes.data, I.ctypes.data, 256, audio.ctypes.data, 256, 0, 2, None) != 0
    assert L.sdr_graph_submit_host_waterfall(g.h, None, GN, I.ctypes.data, I.ctypes.data, 256, audio.ctypes.data, 256, 0, 2, None, None, None) != 0
    lines = np.full((GN, 1, 256), SENT, np.uint32)
    assert L.sdr_graph_submit_host_waterfall(g.h, None, GN, I.ctypes.data, I.ctypes.data, 256, audio.ctypes.data, 256, 0, 2, None,
                                             lines.ctypes.data + 4, None) != 0
    assert (lines == SENT).all()
    assert np.array_equal(wf.export_state()[:, 12:16], np.zeros((GN, 4), np.uint8))  # no pair held: nothing ran
    g.close()
