"""CPU tier: the pre-processor's image detector one rounding away from each of its decisions (tests/pp_edge_signals.py).

  * the numpy model of the detector against the oracle: power spectra bit for bit (ora_aux_power128) and the status
    after every block (ora_aux_run), so that what the builders select on is what the oracle computes;
  * the builders do what they say: the knife-edge blocks sit where they were placed, in the state they were placed in,
    and every covered mutation of the kernel's arithmetic flips at least MIN_FLIPS of their decisions and changes the
    output samples;
  * the kernel's detector path run on the host (tests/emu/pp_emu.cpp, built from sdr_aux_core.cuh) against the oracle in
    ragged calls: outputs and all six status fields after every call.
The GPU tier (test_gpu_pp_edges.py) runs the same cases on the CUDA build.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import pp_edge_signals as E
from oracle import aux_lib as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_cache = {}


def case(placement):
    if placement not in _cache:
        I, Q, ev, lay = E.build(placement)
        _cache[placement] = (I, Q, ev, lay, A.run("pp", (I, Q), ev))
    return _cache[placement]


def schedules(placement):
    """{name: call ends}: 1-block calls (around the knife edge only for the long case), calls that end on the knife-edge
    block, one call for everything."""
    I, _, _, lay, _ = case(placement)
    nb, x = I.shape[1] // 128, lay["block"]
    start = 0 if nb < 100 else x - 3
    return {"ones": ([start] if start else []) + list(range(start + 1, nb + 1)),
            "edge": [x // 2, x + 1, nb],
            "all": [nb]}


def oracle_status_after(I, Q, ev, ends):
    return [A.run("pp", (I[:, :e * 128], Q[:, :e * 128]), [x for x in ev if x[1] < e])[2][:, :6] for e in ends]


def run_calls(fn, I, Q, ev, ends):
    """Calls [0, ends[0]), [ends[0], ends[1]), ... of fn (the signature of ora_aux_run, status carried across calls);
    events (all at block 0 here) go with the first call.  Returns (out I, out Q, [status after each call])."""
    assert all(e[1] == 0 for e in ev)
    blob, nev = A._pack_events("pp", ev)
    nch = I.shape[0]
    oi, oq = np.empty_like(I), np.empty_like(Q)
    st = np.zeros((nch, 8), np.int32)
    out, pos = [], 0
    for k, end in enumerate(ends):
        z = slice(pos * 128, end * 128)
        i, q = np.ascontiguousarray(I[:, z]), np.ascontiguousarray(Q[:, z])
        a, b = np.empty_like(i), np.empty_like(q)
        buf = C.create_string_buffer(blob, len(blob)) if (nev and k == 0) else None
        assert fn(1, nch, end - pos, buf, nev if k == 0 else 0, i.ctypes.data, q.ctypes.data, a.ctypes.data, b.ctypes.data,
                  st.ctypes.data, 1) == 0
        oi[:, z], oq[:, z] = a, b
        out.append(st[:, :6].copy())
        pos = end
    return oi, oq, out


@pytest.fixture(scope="module")
def pp_emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("pp_emu") / "libpp_emu.so")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-std=gnu++17", "-Wno-unused-function", "-shared", "-fPIC",
                    os.path.join(ROOT, "tests", "emu", "pp_emu.cpp"), "-o", so], check=True)
    f = C.CDLL(so).pp_emu_run
    f.restype = C.c_int
    f.argtypes = [C.c_int, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32] + [C.c_void_p] * 5 + [C.c_int]
    return f


# ---- the model is the oracle's arithmetic
def test_model_spectrum_is_the_oracles():
    rng = np.random.default_rng(5)
    I = rng.integers(-32768, 32768, (40, 128)).astype(np.int16)
    Q = rng.integers(-32768, 32768, (40, 128)).astype(np.int16)
    for p in E.PLACEMENTS:
        XI, XQ = case(p)[3]["X"]
        I, Q = np.concatenate([I, XI]), np.concatenate([Q, XQ])
    got = E.spectrum(I, Q)
    for k in range(len(I)):
        assert np.array_equal(got[k].view(np.uint32), A.power128(I[k], Q[k]).view(np.uint32)), k


@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_model_status_after_every_block_is_the_oracles(placement):
    I, Q, ev, lay, want = case(placement)
    oi, oq, st, states, _ = E.model_run(I, Q, ev, record=True)
    assert np.array_equal(oi, want[0]) and np.array_equal(oq, want[1]) and np.array_equal(st, want[2][:, :6])
    nb, x = I.shape[1] // 128, lay["block"]
    ends = range(1, nb + 1) if nb < 100 else [1, 2, 500, 990, 995] + list(range(x - 2, nb + 1))
    for e, s in zip(ends, oracle_status_after(I, Q, ev, ends)):
        assert np.array_equal(states[e - 1], s), e


# ---- the builders do what they say (oracle arithmetic)
@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_knife_edge_blocks_meet_the_planned_state(placement):
    I, Q, ev, lay, _ = case(placement)
    x = lay["block"]
    before = E.model_run(I[:, :x * 128], Q[:, :x * 128], ev)[2]
    assert (before[:, 0] == 1).all() and (before[:, 1] == lay["corr"]).all()
    assert (before[:, 2] == 10).all() and (before[:, 3] == lay["succ"]).all()
    seen = E.correct(I[:, x * 128:(x + 1) * 128], Q[:, x * 128:(x + 1) * 128], before.astype(np.int64).copy())
    assert np.array_equal(seen[0], lay["X"][0]) and np.array_equal(seen[1], lay["X"][1])


@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_knife_edge_blocks_sit_on_their_thresholds(placement):
    XI, XQ = case(placement)[3]["X"]
    kind = case(placement)[3]["kind"]
    pw = E.spectrum(XI, XQ)
    r = E.decide(pw)
    t = kind == "threshold"
    gap = (r["mx"][t].astype(np.float64) - 10.0 * r["avg"][t].astype(np.float64)) / E._ulp(r["mx"][t])
    assert np.abs(gap).max() <= 1.0 and (gap < 0).sum() >= 2 and (gap > 0).sum() >= 2
    assert (gap == 0).sum() >= 2                                    # exact equality: > and >= decide apart
    ra = r["ratio"][kind == "ratio"]
    ten = np.float32(10.0)
    assert (ra == ten).sum() >= 2 and (ra == np.nextafter(ten, np.float32(0))).sum() >= 1 and (ra == np.nextafter(ten, np.float32(11))).sum() >= 1
    tie = np.flatnonzero(kind == "tie")
    assert len(tie) >= 2
    for k in tie:                                                   # two in-band lines with the same float power
        band = pw[k, 5:123]
        lines = 5 + np.flatnonzero(band == band.max())
        assert len(lines) == 2 and pw[k, 128 - lines[0]] != pw[k, 128 - lines[1]]
    z = kind == "zero_image"
    assert z.sum() >= 2 and np.isinf(r["ratio"][z]).all() and r["cross"][z].all()


@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_every_mutation_flips_knife_edge_decisions(placement):
    XI, XQ = case(placement)[3]["X"]
    f = E.flips(XI, XQ)
    for m in E.COVERED:
        assert f[m].sum() >= E.MIN_FLIPS, m
    for m in E.UNREACHABLE:  # stage 5's twiddles (1, 0) and (6.1e-17, -1): fusing changes no rounding
        assert not f[m].any(), m


@pytest.mark.parametrize("placement", ["after_failures", "rollover"])
def test_every_mutation_changes_the_output_samples(placement):
    """A flipped decision at the knife edge moves I2Scorrection, so the mutant's output differs on as many channels."""
    I, Q, ev, lay, want = case(placement)
    for m in E.COVERED:
        oi, oq, st = E.model_run(I, Q, ev, mut=m)
        differ = (oi != want[0]).any(1) | (oq != want[1]).any(1)
        assert differ.sum() >= E.MIN_FLIPS, m


# ---- the kernel's detector path on the host
@pytest.mark.parametrize("sched", ["ones", "edge", "all"])
@pytest.mark.parametrize("placement", E.PLACEMENTS)
def test_emulated_detector_matches_oracle(pp_emu, placement, sched):
    I, Q, ev, lay, want = case(placement)
    ends = schedules(placement)[sched]
    oi, oq, sts = run_calls(pp_emu, I, Q, ev, ends)
    assert np.array_equal(oi, want[0]) and np.array_equal(oq, want[1])
    for e, got, exp in zip(ends, sts, oracle_status_after(I, Q, ev, ends)):
        assert np.array_equal(got, exp), e


def test_emulated_feed_forward_path_after_the_detector_stops(pp_emu):
    """The finish case's channels whose detector stopped at the knife edge continue on the feed-forward path in the next
    calls, the others on the detector path, against the oracle over the longer stream."""
    I, Q, ev, lay, want = case("finish")
    more = 9
    I2 = np.concatenate([I, I[:, -more * 128:]], 1)
    Q2 = np.concatenate([Q, Q[:, -more * 128:]], 1)
    nb = I.shape[1] // 128
    stopped = want[2][:, 0] == 0
    assert stopped.sum() >= 4 and (~stopped).sum() >= 4
    ends = [nb, nb + 2, nb + more]
    oi, oq, sts = run_calls(pp_emu, I2, Q2, ev, ends)
    w = A.run("pp", (I2, Q2), ev)
    assert np.array_equal(oi, w[0]) and np.array_equal(oq, w[1])
    for got, exp in zip(sts, oracle_status_after(I2, Q2, ev, ends)):
        assert np.array_equal(got, exp)
