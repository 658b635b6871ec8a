"""GPU tier: the streamed receiver graph (include/sdr_graph.h) equals the composition of the blocks' device calls bit for bit
-- audio, both kinds of records, spectra, snapshots, counts and every member's final state -- with each front, with calls
kept in flight, under every chunking, and end to end against the oracle; bad arguments change nothing."""
import os
import subprocess
import sys

import numpy as np
import pytest

import graph_harness as H

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 64


@pytest.fixture(scope="module")
def libs():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test running without a CUDA device"
    from audiosdr_b200 import graph
    assert os.path.exists(graph.lib_path()), "libsdr_graph.so missing: __graft_entry__.build() must run before the GPU tier"
    return graph.load_library()


def _equal_runs(front, n=N, lengths=H.LENGTHS, grabber=True):
    calls = H.plan(n, lengths)
    I, Q = H.inputs(front, n, calls)
    a, b = H.make_handles(front, n, grabber), H.make_handles(front, n, grabber)
    got = H.run_graph(a, calls, I, Q)
    want = H.run_device(b, calls, I, Q)
    assert not H.mismatches(got, want), H.mismatches(got, want)
    sa, sb = H.states(a), H.states(b)
    assert sorted(sa) == sorted(sb)
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), "%s state differs after the sequence" % k
    return got


@pytest.mark.parametrize("front", ["pp", "gen", "none"])
def test_graph_equals_the_device_composition(libs, front):
    got = _equal_runs(front)
    # the sequence does exercise what it claims: both pair phases in one call, the detector deciding, slots left unwritten
    assert any(o["counts"].min() != o["counts"].max() for o in got)
    assert any((o["power"] == H.POWER_SENTINEL).all(axis=2).any() for o in got)
    if front == "pp":
        from audiosdr_b200 import aux
        last = got[-1]["pp_status"]
        assert (last[:, aux.PP_BS_CORRECTION] != 0).any()


def test_graph_equals_the_composition_with_the_two_launch_als_form(libs, monkeypatch):
    monkeypatch.setenv("SDR_ALS_SPLIT", "1")
    _equal_runs("pp", lengths=[3, 17, 64])


def test_graph_without_the_grabber(libs):
    _equal_runs("pp", lengths=[2, 17], grabber=False)


CHILD = """
import sys
sys.path[:0] = [%(root)r, %(tests)r]
import numpy as np
import graph_harness as H
calls = H.plan(%(n)d)
I, Q = H.inputs("pp", %(n)d, calls)
h = H.make_handles("pp", %(n)d)
got = H.run_graph(h, calls, I, Q, in_flight=2, pinned=False)
out = {"%%d_%%s" %% (j, k): np.ascontiguousarray(v) for j, o in enumerate(got) for k, v in o.items()}
out.update({"state_" + k: v for k, v in H.states(h).items()})
np.savez(%(path)r, **out)
"""


def test_chunking_is_invisible(libs, tmp_path):
    """SDR_HOST_CHUNKS / SDR_HOST_MIN_CHUNK (read once per process) cut the same calls into 1, 3 and 12 chunks, odd last
    chunks and mixed pair phases included: the bytes are those of the device composition every time."""
    calls = H.plan(N)
    I, Q = H.inputs("pp", N, calls)
    ref = H.make_handles("pp", N)
    want = H.run_device(ref, calls, I, Q)
    want_states = H.states(ref)
    for chunks, min_chunk in ((1, 16), (3, 2), (12, 2)):
        path = str(tmp_path / ("c%d.npz" % chunks))
        env = dict(os.environ, SDR_HOST_CHUNKS=str(chunks), SDR_HOST_MIN_CHUNK=str(min_chunk))
        r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT, "tests": os.path.join(ROOT, "tests"), "n": N, "path": path}],
                           env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        z = np.load(path)
        got = [{k: z["%d_%s" % (j, k)] for k in o} for j, o in enumerate(want)]
        assert not H.mismatches(got, want), (chunks, H.mismatches(got, want))
        for k, v in want_states.items():
            assert np.array_equal(z["state_" + k], v), (chunks, k)


def test_oracle_spot_check(libs):
    """A few channels end to end: the pre-processor oracle, then the receiver oracle on its output."""
    import aux_signals as AS
    import signals as S
    from audiosdr_b200 import api, aux, graph
    from oracle import aux_lib, oracle_lib
    n, lengths = 8, [7, 16, 17]
    total = sum(lengths)
    I, Q, ev = S.make(4, list(range(n)), total)
    pev = [(c, 0, "startAutoI2SerrorDetection") for c in range(0, n, 2)] + [(1, 0, "setI2SerrorCompensation", 1),
                                                                            (3, 0, "setI2SerrorCompensation", -1), (5, 0, "swapIQ", 1)]
    wI, wQ, _ = aux_lib.run("pp", (I, Q), pev)
    want = oracle_lib.run(wI, wQ, ev, threads=4)["audio"]
    rx, pp = api.SdrBatch(n), aux.PreProcessorBatch(n)
    rx.configure([(e[0],) + tuple(e[2:]) for e in ev])
    for e in pev:
        getattr(pp, e[2])(*([e[0]] + list(e[3:])))
    g = graph.GraphBatch(rx, preproc=pp)
    got, pos = [], 0
    for nb in lengths:
        a, _ = g.process_host(np.ascontiguousarray(I[:, pos * 128:(pos + nb) * 128]), np.ascontiguousarray(Q[:, pos * 128:(pos + nb) * 128]),
                              out_fmt=api.FMT_F32)
        got.append(a)
        pos += nb
    g.close()
    got = np.concatenate(got, 1)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_bad_arguments_change_nothing(libs):
    from audiosdr_b200 import api, aux, graph
    n, nb = 16, 5
    h = H.make_handles("pp", n)
    g = graph.GraphBatch(h["rx"], preproc=h["pp"], grabber=h["gr"])
    L = g.L
    I = np.ones((n, nb * 128 + 8), np.int16); Q = I.copy()
    before = H.states(h)

    def call(ids=None, n_ids=n, i=I, q=Q, in_pitch=nb * 128 + 8, out_pitch=nb * 128, fmt=api.FMT_I16, n_blocks=nb, misalign=None):
        audio = np.full((n_ids, out_pitch), 0x1111, np.int16)
        S_ = (n_blocks + 1) // 2
        bufs = {"rx_status": np.full(n_blocks * api.BS_FIELDS * n_ids + 8, 0x2222, np.uint32),
                "pp_status": np.full(n_blocks * aux.PP_BS_FIELDS * n_ids + 8, 0x3333, np.int32),
                "power": np.full(n_ids * S_ * 256 + 8, -3.0, np.float32), "snapshots": np.full(n_ids * S_ * 512 + 8, 0x4444, np.int16)}
        counts = np.full(n_ids, 99, np.uint32)
        o = graph.GraphOutputs()
        for k, a in bufs.items():
            base = a.ctypes.data
            off = (-base) % 16
            setattr(o, k, base + off + (a.itemsize if k == misalign else 0))
        o.counts = counts.ctypes.data
        keep = [np.full_like(a, a.flat[0]) for a in bufs.values()]
        ida = None if ids is None else np.asarray(ids, np.uint32)
        rc = L.sdr_graph_process_host(g.h, None if ida is None else ida.ctypes.data, n_ids, i.ctypes.data, None if q is None else q.ctypes.data,
                                     in_pitch, audio.ctypes.data, out_pitch, fmt, n_blocks, o)
        untouched = (audio == 0x1111).all() and (counts == 99).all() and all(np.array_equal(a, k) for a, k in zip(bufs.values(), keep))
        return rc, untouched

    assert call()[0] == 0  # the well-formed call (it advances every member by nb blocks)
    g.wait_host()
    before = H.states(h)
    for kw in (dict(ids=[1, 2, 2], n_ids=3), dict(ids=[0, n], n_ids=2), dict(ids=None, n_ids=n - 1), dict(misalign="rx_status"),
               dict(misalign="pp_status"), dict(misalign="power"), dict(misalign="snapshots"), dict(in_pitch=nb * 128 - 8),
               dict(out_pitch=nb * 128 - 8), dict(q=None), dict(fmt=7), dict(n_blocks=0)):
        if "n_ids" in kw and kw["n_ids"] != n:
            kw["i"] = np.ones((kw["n_ids"], nb * 128 + 8), np.int16); kw["q"] = kw["i"].copy()
        rc, untouched = call(**kw)
        assert rc == -1 and untouched, kw
    g.wait_host()
    after = H.states(h)
    for k in before:
        assert np.array_equal(before[k], after[k]), k
    g.close()
    # the generator front takes no Q plane
    gen = aux.IQGeneratorBatch(n)
    g2 = graph.GraphBatch(h["rx"], iqgen=gen)
    blob = gen.export_state()
    audio = np.full((n, nb * 128), 0x1111, np.int16)
    rc = g2.L.sdr_graph_submit_host(g2.h, None, n, I.ctypes.data, Q.ctypes.data, nb * 128 + 8, audio.ctypes.data, nb * 128, api.FMT_I16, nb, None)
    assert rc == -1 and (audio == 0x1111).all() and np.array_equal(gen.export_state(), blob)
    g2.close()
    # create refuses members of another channel count, and two fronts
    with pytest.raises(graph.GraphError):
        graph.GraphBatch(h["rx"], grabber=aux.GrabberBatch(n + 1))
    with pytest.raises(graph.GraphError):
        graph.GraphBatch(h["rx"], preproc=aux.PreProcessorBatch(n + 1))
    with pytest.raises(graph.GraphError):
        graph.GraphBatch(h["rx"], preproc=h["pp"], iqgen=gen)
