"""GPU tier: the CUDA library on the edge-of-signal cases of tests/edge_signals.py, bit for bit against the oracle.

These inputs take the kernel's guarded paths and fallbacks, where CUDA arithmetic differs from x86: packed FP32 on
subnormal operands (IIR states decaying through the subnormals in digital silence, subnormal input), the range guards of
the envelope's and the SAM PLL's fast divisions (exact zeros, |I|^2+|Q|^2 and phase-detector operands around 2^-60, warps
mixing silent and live SAM lanes), the FP64 branch of the int16 output (|audio| >= 256, wrap, x86 'indefinite'), the
blanker's window and edge bookkeeping (clustered bursts) and setters outside the fuzzer's ranges.  Every plan, the split
ALS form, the device and both host entry points, and the per-block records.  test_emu_edge_signals.py shows on the CPU that
each case reaches the edge it was built for.
"""
import os

import numpy as np
import pytest

import audiosdr_b200 as A
import edge_signals as E
import harness
from test_emu_pipeline import set_plan
from test_gpu_block_status import check_device
from test_gpu_parity import assert_same

pytestmark = pytest.mark.gpu
N_BLOCK = 128
GPU_KW = {"silence": dict(sam_lanes=160)}  # 5 groups of the SAM bucket, every warp mixing silent and live lanes
PLANS = [None, (16, 2, 0), (8, 3, 1), (16, 2, 1), "als-split"]
PLAN_IDS = ["default", "tile16-x2", "tile8-merged-x3", "tile16-merged-x2", "als-split"]
_cache = {}


@pytest.fixture(scope="module")
def dev(cuda_lib):
    import torch
    return torch.device("cuda:0")


def case(name):
    """(I, Q, events, oracle result) of a case, built and run once per session."""
    if name not in _cache:
        I, Q, ev = E.make(name, **GPU_KW.get(name, {}))
        from oracle import oracle_lib
        _cache[name] = (I, Q, ev, oracle_lib.run(I, Q, ev, threads=os.cpu_count() or 1))
    return _cache[name]


def check(a, b, o, pcm=None):
    assert_same(a, o["audio"])
    assert np.array_equal(harness.status_matrix(b), o["status"], equal_nan=True)
    if pcm is not None:
        assert np.array_equal(pcm, o["pcm"]), harness.describe_mismatch(pcm.astype(np.float32), o["pcm"].astype(np.float32))


@pytest.mark.parametrize("plan", PLANS, ids=PLAN_IDS)
@pytest.mark.parametrize("name", E.CASES)
def test_cuda_edge_case_on_device(cuda_lib, oracle, dev, monkeypatch, name, plan):
    """process() on device planes, ragged calls with 1-block calls among them, float32 audio and int16 pcm."""
    if plan == "als-split":
        monkeypatch.setenv("SDR_ALS_SPLIT", "1")
    elif plan:
        set_plan(monkeypatch, *plan)
    I, Q, ev, o = case(name)
    a, b = harness.run_batch(cuda_lib, I, Q, ev, chunks=(17, 1, 40, 2), device=dev, return_batch=True)
    p = harness.run_batch(cuda_lib, I, Q, ev, chunks=(1, 64, 9), out_dtype=np.int16, device=dev)
    check(a, b, o, p)


def run_submitted(lib, I, Q, events, chunks, out_dtype):
    """harness.run_batch through submit_host: pinned host planes, calls queued back to back, setters configured between
    two submits, one wait_host at the end."""
    import torch
    nch, ns = I.shape
    b = A.SdrBatch(nch, _lib=lib)
    hI, hQ = torch.from_numpy(np.ascontiguousarray(I)).pin_memory(), torch.from_numpy(np.ascontiguousarray(Q)).pin_memory()
    hO = torch.zeros((nch, ns), dtype=torch.float32 if out_dtype == np.float32 else torch.int16).pin_memory()
    nI, nQ, nO = hI.numpy(), hQ.numpy(), hO.numpy()
    ev = sorted(events, key=lambda e: e[1])
    nb_total, pos, ei, k, t = ns // N_BLOCK, 0, 0, 0, 0
    while pos < nb_total:
        calls = []
        while ei < len(ev) and ev[ei][1] <= pos:
            e = ev[ei]
            calls.append((None if e[0] == 0xFFFFFFFF else e[0], e[2]) + tuple(e[3:]))
            ei += 1
        if calls:
            b.configure(calls)
        nxt = ev[ei][1] if ei < len(ev) else nb_total
        sz = min(chunks[k % len(chunks)], nb_total - pos, max(nxt - pos, 1))
        k += 1
        a, z = pos * N_BLOCK, (pos + sz) * N_BLOCK
        t = b.submit_host(nI[:, a:z], nQ[:, a:z], nO[:, a:z])
        pos += sz
    b.wait_host(ticket=t)
    return nO.copy(), b


@pytest.mark.parametrize("name", E.CASES)
def test_cuda_edge_case_host_paths(cuda_lib, oracle, name):
    """process_host (float32 audio, ragged calls with 1-block calls) and submit_host / wait_host (int16 pcm, then float32)."""
    I, Q, ev, o = case(name)
    a, b = harness.run_batch(cuda_lib, I, Q, ev, chunks=(1, 13, 5), return_batch=True)
    check(a, b, o)
    p, _ = run_submitted(cuda_lib, I, Q, ev, (9, 1, 30), np.int16)
    assert np.array_equal(p, o["pcm"]), harness.describe_mismatch(p.astype(np.float32), o["pcm"].astype(np.float32))
    a, b = run_submitted(cuda_lib, I, Q, ev, (40, 1, 3), np.float32)
    check(a, b, o)


@pytest.mark.parametrize("name", E.CASES)
def test_cuda_edge_case_block_records(cuda_lib, oracle, dev, name):
    I, Q, ev, o = case(name)
    check_device(cuda_lib, dev, I, Q, ev, chunks=(7, 1, 13))


def test_cuda_contracting_build_on_silence(cuda_lib, oracle, dev):
    """The opt-in contracting build through silence and back: the exact build's NaN pattern, and outside NaN the error
    profile test_gpu_long pins for it on the BASELINE configurations."""
    I, Q, ev, o = case("silence")
    exact = harness.run_batch(cuda_lib, I, Q, ev, chunks=(100, 1, 131), device=dev)
    a = harness.run_batch(cuda_lib, I, Q, ev, chunks=(100, 1, 131), device=dev, contract=True)
    nan = np.isnan(a)
    assert np.array_equal(nan, np.isnan(exact))
    err = np.abs(a[~nan].astype(np.float64) - o["audio"][~nan])
    assert float(np.sqrt(np.mean(err ** 2))) < 5e-6
    assert float(np.mean(err > 1e-4)) < 1e-4 and float(err.max()) < 1e-2, "max %g, share above 1e-4: %g" % (err.max(), np.mean(err > 1e-4))
