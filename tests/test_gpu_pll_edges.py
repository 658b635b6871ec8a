"""GPU tier: the SAM PLL and the noise blanker one rounding away from their decisions (tests/pll_edge_signals.py) on the
CUDA build, bit for bit against the oracle.

On the GPU the fast path's forms meet these edges: the FMA select of the phase wrap, the cosine index, the vote behind the
table look-ups, the division without its range check.  The case's PLL rows fill the receiver's 32-lane warps so that the
vote passes at every fast-path edge (test_emu_pll_edges.py checks it on the model): knife-edge lanes beside live tracking
lanes, and a last warp with one lane and 31 idle ones.  Device planes on every plan, process_host and submit_host /
wait_host, per-block records, a warp whose 32 lanes hit the same edge at the same sample, and 4 096 channels in one call.
"""
import os

import numpy as np
import pytest

import harness
import pll_edge_signals as E
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


def case():
    if not _cache:
        I, Q, ev, lay = E.build()
        from oracle import oracle_lib
        _cache["c"] = (I, Q, ev, lay, oracle_lib.run(I, Q, ev, threads=os.cpu_count() or 1))
    return _cache["c"]


@pytest.mark.parametrize("plan", PLANS, ids=PLAN_IDS)
def test_cuda_knife_edges_on_device(cuda_lib, oracle, dev, monkeypatch, plan):
    if plan == "als-split":
        monkeypatch.setenv("SDR_ALS_SPLIT", "1")
    elif plan:
        set_plan(monkeypatch, *plan)
    I, Q, ev, lay, o = case()
    a, b = harness.run_batch(cuda_lib, I, Q, ev, chunks=(17, 1, 40, 2), device=dev, return_batch=True)
    p = harness.run_batch(cuda_lib, I, Q, ev, chunks=(1, 64, 9), out_dtype=np.int16, device=dev)
    check(a, b, o, p)


def test_cuda_knife_edges_host_paths(cuda_lib, oracle):
    I, Q, ev, lay, o = case()
    a, b = harness.run_batch(cuda_lib, I, Q, ev, chunks=(1, 13, 5), return_batch=True)
    check(a, b, o)
    p, _ = run_submitted(cuda_lib, I, Q, ev, (9, 1, 30), np.int16)
    assert np.array_equal(p, o["pcm"]), harness.describe_mismatch(p.astype(np.float32), o["pcm"].astype(np.float32))


def test_cuda_knife_edges_block_records(cuda_lib, oracle, dev):
    I, Q, ev, lay, o = case()
    check_device(cuda_lib, dev, I, Q, ev, chunks=(7, 1, 13))


def _aligned_copies(src_name="lo_end"):
    """The case with 32 copies of one knife-edge row inserted after the first six PLL warps, so that they fill one warp of
    their own: every lane hits the same edge at the same sample.  Returns (I, Q, events, source row of each row)."""
    I0, Q0, ev0, lay, _ = case()
    cut = 6 * E.LANES
    assert not lay["nb_on"][:cut].any() and (lay["warp"][:cut] < 6).all()
    src = next(r for r, n in enumerate(lay["rows"]) if n == src_name)
    order = list(range(cut)) + [src] * E.LANES + list(range(cut, len(I0)))
    ev = [(k,) + tuple(e[1:]) for k, r in enumerate(order) for e in ev0 if e[0] == r]
    return I0[order], Q0[order], ev, np.array(order)


def test_cuda_knife_edges_one_edge_in_every_lane(cuda_lib, oracle, dev):
    I, Q, ev, order = _aligned_copies()
    o = case()[4]
    a, b = harness.run_batch(cuda_lib, I, Q, ev, chunks=(5, 11), device=dev, return_batch=True)
    assert harness.bits_equal(a, o["audio"][order]), harness.describe_mismatch(a, o["audio"][order])
    assert np.array_equal(harness.status_matrix(b), o["status"][order], equal_nan=True)


@pytest.mark.parametrize("plan", [None, (8, 3, 1)], ids=["default", "tile8-merged-x3"])
def test_cuda_knife_edges_many_channels(cuda_lib, oracle, dev, monkeypatch, plan):
    """4 096 channels: the case's six full PLL warps 21 times over (each copy keeps its warp alignment), the one-lane warp,
    and the blanker rows.  The SAM-only bucket's merged 8-sample plan takes over by itself only beyond 2 groups per SM
    (9 472 channels on 148 SMs); the second run forces it through SDR_TILE_ENV / SDR_CTAS_PER_SM / SDR_NO_MERGE."""
    if plan:
        set_plan(monkeypatch, *plan)
    I0, Q0, ev0, lay, o = case()
    cut = 6 * E.LANES
    order = list(range(cut)) * 21 + list(range(cut, len(I0)))
    order += list(range(cut + 1, cut + 1 + 4096 - len(order)))  # blanker rows again, to 4 096
    assert len(order) == 4096 and all(lay["nb_on"][r] for r in order[21 * cut + len(I0) - cut:])
    ev = [(k,) + tuple(e[1:]) for k, r in enumerate(order) for e in ev0 if e[0] == r]
    a = harness.run_batch(cuda_lib, I0[order], Q0[order], ev, chunks=(24,), device=dev)
    want = o["audio"][order]
    assert harness.bits_equal(a, want), harness.describe_mismatch(a, want)
