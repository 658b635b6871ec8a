"""GPU tier: the AGC one rounding away from its decisions (tests/agc_edge_signals.py) on the CUDA build, bit for bit
against the oracle.

Attack ties on the AM level path and at the clamp, hang expiries on tile, block and call boundaries, the gain on 0.99f and
its neighbours, and groups of 4, 5 and 32 AGC tables (the global-memory look-up): every plan on device planes,
process_host and submit_host / wait_host with ragged calls, int16 pcm, per-block records, one edge in all 32 lanes of a
warp, 4 096 channels in one call, and AGC mode 3 across many calls.  test_emu_agc_edges.py shows on the CPU that each row
reaches the edge it was built for.
"""
import os

import numpy as np
import pytest

import agc_edge_signals as E
import harness
from test_emu_pipeline import set_plan
from test_gpu_block_status import check_device
from test_gpu_edge_signals import PLANS, PLAN_IDS, check, run_submitted

pytestmark = pytest.mark.gpu
N_BLOCK = 128
_cache = {}


@pytest.fixture(scope="module")
def dev(cuda_lib):
    import torch
    return torch.device("cuda:0")


def case(name="c"):
    if name not in _cache:
        I, Q, ev, lay = E.build() if name == "c" else E.long_case()
        from oracle import oracle_lib
        _cache[name] = (I, Q, ev, lay, oracle_lib.run(I, Q, ev, threads=os.cpu_count() or 1))
    return _cache[name]


@pytest.mark.parametrize("plan", PLANS, ids=PLAN_IDS)
def test_cuda_agc_edges_on_device(cuda_lib, oracle, dev, monkeypatch, plan):
    if plan == "als-split":
        monkeypatch.setenv("SDR_ALS_SPLIT", "1")
    elif plan:
        set_plan(monkeypatch, *plan)
    I, Q, ev, lay, o = case()
    a, b = harness.run_batch(cuda_lib, I, Q, ev, chunks=E.CHUNKS, device=dev, return_batch=True)
    p = harness.run_batch(cuda_lib, I, Q, ev, chunks=(1, 64, 9), out_dtype=np.int16, device=dev)
    check(a, b, o, p)


def test_cuda_agc_edges_host_paths(cuda_lib, oracle):
    I, Q, ev, lay, o = case()
    a, b = harness.run_batch(cuda_lib, I, Q, ev, chunks=(1, 13, 5), return_batch=True)
    check(a, b, o)
    p, _ = run_submitted(cuda_lib, I, Q, ev, (9, 1, 30), np.int16)
    assert np.array_equal(p, o["pcm"]), harness.describe_mismatch(p.astype(np.float32), o["pcm"].astype(np.float32))
    a, b = run_submitted(cuda_lib, I, Q, ev, E.CHUNKS, np.float32)
    check(a, b, o)


def test_cuda_agc_edges_block_records(cuda_lib, oracle, dev):
    I, Q, ev, lay, o = case()
    check_device(cuda_lib, dev, I, Q, ev, chunks=(7, 1, 13))


def test_cuda_agc_mode_3_across_many_calls(cuda_lib, oracle, dev):
    I, Q, ev, lay, o = case("long")
    a, b = harness.run_batch(cuda_lib, I, Q, ev, chunks=(7, 1, 13), device=dev, return_batch=True)
    check(a, b, o)
    p, _ = run_submitted(cuda_lib, I, Q, ev, (40, 1, 3), np.int16)
    assert np.array_equal(p, o["pcm"]), harness.describe_mismatch(p.astype(np.float32), o["pcm"].astype(np.float32))


def _copies(src_kind):
    """32 copies of the first row of one kind, alone in a handle: one group, every lane on the same edge at the same
    sample.  Returns (I, Q, events, source row of each row)."""
    I0, Q0, ev0, lay, o = case()
    src = lay["rows"].index(src_kind)
    order = [src] * E.LANES
    ev = [(k,) + tuple(e[1:]) for k in range(E.LANES) for e in ev0 if e[0] == src]
    return I0[order], Q0[order], ev, np.array(order)


@pytest.mark.parametrize("kind", ["act_eq", "act_dn", "am_tie", "ssb_clamp", "hang_at"])
def test_cuda_agc_one_edge_in_every_lane(cuda_lib, oracle, dev, kind):
    I, Q, ev, order = _copies(kind)
    o = case()[4]
    a, b = harness.run_batch(cuda_lib, I, Q, ev, chunks=(5, 11), device=dev, return_batch=True)
    assert harness.bits_equal(a, o["audio"][order]), harness.describe_mismatch(a, o["audio"][order])
    assert np.array_equal(harness.status_matrix(b), o["status"][order], equal_nan=True)


def test_cuda_agc_edges_many_channels(cuda_lib, oracle, dev):
    """4 096 channels: the case over and over in one call (each full copy's 96 staging rows make three LSB groups of their
    own, with 4, 5 and 32 tables)."""
    I0, Q0, ev0, lay, o = case()
    order = (list(range(len(I0))) * (4096 // len(I0) + 1))[:4096]
    mine = {}
    for e in ev0:
        mine.setdefault(e[0], []).append(e)
    ev = [(k,) + tuple(e[1:]) for k, r in enumerate(order) for e in mine[r]]
    a = harness.run_batch(cuda_lib, I0[order], Q0[order], ev, chunks=(40,), device=dev)
    want = o["audio"][order]
    assert harness.bits_equal(a, want), harness.describe_mismatch(a, want)
