"""CPU tier: the chain at the edges of the signal (tests/edge_signals.py) through the host emulation of the kernel source.

Digital silence that decays through the subnormals, tiny and full-scale input, clustered blanker bursts and setters outside
the fuzzer's ranges: float32 audio, int16 pcm, end-of-call status and per-block records bit for bit against the oracle,
under several hand-over schedules, on the short-tile plans and with the split ALS form.  The "does what it says" tests pin
each stimulus to the edge it was built for, so that a builder drifting back to tame input fails here.  The GPU tier
(test_gpu_edge_signals.py) runs the same cases on the CUDA build.
"""
import os

import numpy as np
import pytest

import edge_signals as E
import harness
from test_emu_block_status import check_case, oracle_block_status
from test_emu_pipeline import set_plan, set_schedule

SCHEDULES = ["lockstep", "consumers", "random:2/late"]
PLANS = [(16, 2, 0), (8, 3, 1), (16, 2, 1)]
_cache = {}


def case(name):
    """(I, Q, events, oracle result) of a case, built and run once per session."""
    if name not in _cache:
        I, Q, ev = E.make(name)
        from oracle import oracle_lib
        _cache[name] = (I, Q, ev, oracle_lib.run(I, Q, ev, threads=os.cpu_count() or 1))
    return _cache[name]


def assert_bits(lib, I, Q, ev, o, chunks=(7, 1, 13), pcm=True):
    a, b = harness.run_batch(lib, I, Q, ev, chunks=chunks, return_batch=True)
    assert harness.bits_equal(a, o["audio"]), harness.describe_mismatch(a, o["audio"])
    assert np.array_equal(harness.status_matrix(b), o["status"], equal_nan=True)
    if not pcm:
        return
    p = harness.run_batch(lib, I, Q, ev, chunks=(3, 11), out_dtype=np.int16)
    assert np.array_equal(p, o["pcm"]), harness.describe_mismatch(p.astype(np.float32), o["pcm"].astype(np.float32))


# ---- the cases do what they say (oracle only)
def test_silence_case_decays_through_subnormals(oracle):
    I, Q, ev, layout = E.silence()
    o = case("silence")[3]
    assert E.silence_check(o, layout) > 100000


def test_tiny_case_straddles_the_fast_path_ranges(oracle):
    I, Q, ev, scales = E.tiny()
    E.tiny_check(I, Q, ev, scales, case("tiny")[3])


def test_full_scale_case_reaches_the_fp64_pcm_branch(oracle):
    E.full_scale_check(case("full_scale")[3])
    a = case("large_float")[3]["audio"]
    assert np.any(np.isfinite(a) & (np.abs(a) >= 256.0))


def test_clustered_case_detects_at_the_designed_blocks(oracle):
    I, Q, ev, _ = case("clustered")
    E.clustered_check(I, Q, ev, oracle_block_status(I, Q, ev))


def test_setter_edges_case_takes_effect(oracle):
    """Input gain 0 lets a row's filters ring down until the gain is lifted; some rows run away to NaN, as in the
    reference, and every row has finite audio before that."""
    I, Q, ev, o = case("setter_edges")
    for r in range(0, I.shape[0], len(E.SETTER_EDGES)):  # the setInputGain rows
        b = next(e[1] for e in ev if e[0] == r and e[2] == "setInputGain" and e[3] == 0.0)
        a = o["audio"][r].reshape(-1, 128)
        assert np.abs(a[b + 8]).max() < 0.1 * np.abs(a[b - 1]).max(), r
        assert np.abs(a[b + 12:]).max() > 1e-2 * np.abs(a[b - 1]).max(), r
    assert np.isnan(o["audio"]).any() and np.isfinite(o["audio"]).any(axis=1).all()


# ---- the emulation against the oracle
@pytest.mark.parametrize("sched", SCHEDULES)
@pytest.mark.parametrize("name", E.CASES)
def test_emulated_edge_case(oracle, emu_lib, monkeypatch, name, sched):
    set_schedule(monkeypatch, sched)
    I, Q, ev, o = case(name)
    assert_bits(emu_lib, I, Q, ev, o)


@pytest.mark.parametrize("plan", PLANS, ids=["tile16-x2", "tile8-merged-x3", "tile16-merged-x2"])
@pytest.mark.parametrize("name", ["silence", "tiny", "setter_edges"])
def test_emulated_edge_case_short_tile_plans(oracle, emu_lib, monkeypatch, name, plan):
    """The short-tile plans run the buckets without blanker and ALS (among them the SAM mixed-warp bucket)."""
    set_schedule(monkeypatch, "random:3/late")
    set_plan(monkeypatch, *plan)
    I, Q, ev, o = case(name)
    assert_bits(emu_lib, I, Q, ev, o, chunks=(5, 1, 17), pcm=False)  # the output format is the schedules' test


@pytest.mark.parametrize("name", E.CASES)
def test_emulated_edge_case_split_als(oracle, emu_lib, monkeypatch, name):
    monkeypatch.setenv("SDR_ALS_SPLIT", "1")
    set_schedule(monkeypatch, "consumers")
    I, Q, ev, o = case(name)
    assert_bits(emu_lib, I, Q, ev, o, chunks=(11, 2), pcm=False)


@pytest.mark.parametrize("name", E.CASES)
def test_emulated_edge_case_block_records(oracle, emu_lib, name):
    I, Q, ev, o = case(name)
    if name == "silence":  # the records of the long case on its first 64 blocks: silence starts in block 16
        I, Q = I[:, :64 * 128], Q[:, :64 * 128]
    check_case(emu_lib, I, Q, ev, chunks=(9, 1, 4))
