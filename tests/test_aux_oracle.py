"""CPU tier for the blocks either side of the receiver chain (SURVEY 8f rows 2, 4): AudioSDRpreProcessor and AudioIQgenerator.

  * the C restatement (oracle/sdr_aux_oracle.c) against the committed golden outputs of the unmodified reference
    (tests/golden/aux_*.npz, tools/gen_golden_aux.py) and, where oracle/_ref/refaux exists, against the reference itself;
  * the per-lane source of the CUDA kernels (audiosdr_b200/csrc/sdr_aux_core.cuh) compiled for the host against the oracle
    (tests/emu/aux_emu.cpp), including the exhaustive check of the divide-free Q15 conversion;
  * the detector's decisions against a float64 DFT (the FFT's rounding is the one unpinned piece, oracle/aux_fft128.h);
  * the C ABI of include/sdr_aux.h: every declared symbol exported, setter ids consistent, no CPU fallback."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import aux_signals as S
from oracle import aux_lib as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def test_preprocessor_oracle_matches_golden():
    g = np.load(os.path.join(GOLD, "aux_pp.npz"))
    nch, nb = int(g["n_channels"]), int(g["n_blocks"])
    I, Q = S.pp_case(nch, nb)
    o0, o1, st = A.run("pp", (I, Q), S.pp_events(nch, nb))
    assert np.array_equal(S.block_crcs(o0, o1), g["crc"])
    assert np.array_equal(o0[:, :32 * 128], g["I_head"]) and np.array_equal(o1[:, :32 * 128], g["Q_head"])
    assert np.array_equal(st, g["status"])
    # the fixture really exercises the detector: finished, found +1 and -1, still searching, swapped
    assert (st[:, 3] == 1001).sum() >= 4 and (st[:, 1] == 1).any() and (st[:, 1] == -1).any() and (st[:, 0] == 1).any() and (st[:, 5] == 1).any()


def test_generator_oracle_matches_golden():
    g = np.load(os.path.join(GOLD, "aux_iq.npz"))
    nch, nb = int(g["n_channels"]), int(g["n_blocks"])
    X = S.iq_case(nch, nb)
    o0, o1, _ = A.run("iq", (X,), S.iq_events(nch, nb))
    assert np.array_equal(o0, g["I_out"]) and np.array_equal(o1, g["Q_out"])
    # I is the input delayed by 128 samples and requantised: within 1 LSB where the balance is 1
    assert np.max(np.abs(o0[0, 128:].astype(int) - X[0, :-128].astype(int))) <= 1


@pytest.mark.skipif(not A.ref_available(), reason="oracle/_ref/refaux not built (needs the reference tree)")
def test_oracle_matches_reference_binary():
    I, Q = S.pp_case(12, 300, seed=99)
    ev = S.pp_events(12, 300) + [(3, 10, "setI2SerrorCompensation", 1), (3, 11, "setI2SerrorCompensation", -1), (3, 12, "swapIQ", 1),
                                 (2, 299, "stopAutoI2SerrorDetection"), (1, 300, "swapIQ", 1)]
    for a, b in zip(A.run("pp", (I, Q), ev), A.ref_run("pp", (I, Q), ev)):
        assert np.array_equal(a, b)
    X = S.iq_case(9, 33, seed=5)
    ev = S.iq_events(9, 33) + [(0, 7, "setGainBalance", 40000.0), (4, 3, "setGainBalance", -1.5)]
    for a, b in zip(A.run("iq", (X,), ev)[:2], A.ref_run("iq", (X,), ev)[:2]):
        assert np.array_equal(a, b)


def test_kernel_lane_source_matches_oracle_on_host(tmp_path):
    exe = str(tmp_path / "aux_emu")
    obj = str(tmp_path / "aux_oracle.o")
    subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-std=c11", "-c", os.path.join(ROOT, "oracle", "sdr_aux_oracle.c"),
                    "-o", obj], check=True)
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-std=gnu++17", "-Wno-unused-function",
                    os.path.join(ROOT, "tests", "emu", "aux_emu.cpp"), obj, "-lpthread", "-lm", "-o", exe], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "total mismatches 0" in r.stdout


def test_detector_decisions_do_not_hinge_on_fft_rounding():
    """PARITY UNPINNED piece (oracle/aux_fft128.h): the FFT is a restatement of CMSIS-DSP.  Its float32 power spectrum must
    agree with a float64 DFT to float32 accuracy, and the quantities the detector thresholds (strongest line vs 10 x mean,
    line vs image vs 10) must sit far from their thresholds on the test signals, so any correct float32 FFT decides alike."""
    I, Q = S.pp_case(8, 40, seed=3)
    worst, margins = 0.0, []
    for c in range(8):
        for b in range(0, 40, 7):
            z = slice(b * 128, (b + 1) * 128)
            p = A.power128(I[c, z], Q[c, z]).astype(np.float64)
            x = (I[c, z].astype(np.float32) / np.float32(32767.0)).astype(np.float64) + 1j * (Q[c, z].astype(np.float32) / np.float32(32767.0)).astype(np.float64)
            want = np.abs(np.fft.fft(x)) ** 2
            worst = max(worst, float(np.max(np.abs(p - want)) / np.max(want)))
            band = want[5:123]
            line = 5 + int(np.argmax(band))
            strong = band.max() / (10.0 * band.mean())
            margins.append(abs(np.log10(strong)))
            if strong > 1.0:
                margins.append(abs(np.log10(band.max() / want[128 - line] / 10.0)))
    assert worst < 2e-6
    assert min(margins) > 1e-3  # decisions at least 0.2 % away from a threshold vs 2e-6 of FFT rounding


def test_grabber_oracle_matches_reference_binary():
    """SURVEY 8f row 3 (no arithmetic): the restatement against the unmodified AudioGrabberComplex256 for 1..9 blocks."""
    if not A.ref_available():
        pytest.skip("oracle/_ref/refaux not built (needs the reference tree)")
    for nb in (1, 2, 3, 4, 9):
        I, Q = S.pp_case(6, nb, seed=40 + nb)
        o, f = A.grab_run(I, Q)
        ro, rf = A.ref_grab_run(I, Q)
        assert np.array_equal(o, ro) and np.array_equal(f, rf)
        if nb >= 2:
            last = (nb // 2) * 2   # blocks [last-2, last) form the snapshot
            assert np.array_equal(o[:, 0::2], I[:, (last - 2) * 128: last * 128]) and np.array_equal(o[:, 1::2], Q[:, (last - 2) * 128: last * 128])


def test_spectrum_oracle_is_the_dft():
    """The spectrum tap's oracle (radix-2 network in float32, oracle/aux_fft128.h) against the float64 DFT of numpy: the
    restatement is the mathematically defined transform up to float32 rounding, bins in natural order."""
    rng = np.random.default_rng(11)
    snap = rng.integers(-30000, 30000, (16, 512)).astype(np.int16)
    t = np.arange(256)
    snap[0, 0::2] = np.round(20000 * np.cos(2 * np.pi * 5 * t / 256)); snap[0, 1::2] = np.round(20000 * np.sin(2 * np.pi * 5 * t / 256))      # +5 bins
    snap[1, 0::2] = np.round(20000 * np.cos(2 * np.pi * 5 * t / 256)); snap[1, 1::2] = np.round(-20000 * np.sin(2 * np.pi * 5 * t / 256))     # -5 bins
    p = A.grab_spectrum(snap)
    x = snap[:, 0::2].astype(np.float64) + 1j * snap[:, 1::2].astype(np.float64)
    ref = np.abs(np.fft.fft(x, axis=1)) ** 2
    assert np.max(np.abs(p - ref) / ref.max(axis=1, keepdims=True)) < 2e-6
    assert int(np.argmax(p[0])) == 5 and int(np.argmax(p[1])) == 251
    z = A.grab_spectrum(np.zeros((1, 512), np.int16))
    assert not z.any()


def declared(prefixes=("sdr_preproc_", "sdr_iqgen_", "sdr_grabber_", "sdr_aux_")):
    src = open(os.path.join(ROOT, "include", "sdr_aux.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(n for n in re.findall(r"\b(sdr_\w+)\s*\(", src) if n.startswith(prefixes)))


def test_aux_library_exports_every_declared_symbol():
    from audiosdr_b200 import aux, build
    lib = ctypes.CDLL(build.build_aux_library())  # nvcc cross-compiles sm_100a without a GPU
    names = declared()
    assert "sdr_preproc_process_device" in names and "sdr_iqgen_process_device" in names
    for n in names:
        assert hasattr(lib, n), n
    assert set(aux.EXPORTS) == set(names)
    assert b"sm_100a" in ctypes.cast(lib.sdr_aux_version, ctypes.CFUNCTYPE(ctypes.c_char_p))()
    src = open(os.path.join(ROOT, "include", "sdr_aux.h")).read()
    ids = {m.group(1): int(m.group(2)) for m in re.finditer(r"SDR_PP_(\w+)\s*=\s*(\d+)", src)}
    assert ids == aux.PP_SETTERS == A.OPS["pp"]


NO_DEVICE_CHILD = """
import os, sys
sys.path.insert(0, %(root)r)
from audiosdr_b200 import aux
aux.load_library()  # the built library loads: the batches below fail for want of a device, not of the library
for make in (lambda: aux.PreProcessorBatch(4), lambda: aux.IQGeneratorBatch(4),
             lambda: aux.load_library(os.path.join(%(root)r, "audiosdr_b200", "no_such_library.so"))):
    try:
        make()
    except aux.AuxError:
        continue
    sys.exit("no AuxError")
print("NO_FALLBACK_OK")
"""


def test_aux_has_no_cpu_fallback():
    """Without a CUDA device the batches raise instead of computing on the CPU.  The devices are hidden from a child process,
    so that a machine with a GPU checks this too."""
    from audiosdr_b200 import build
    build.build_aux_library()  # nvcc cross-compiles sm_100a without a GPU
    r = subprocess.run([sys.executable, "-c", NO_DEVICE_CHILD % {"root": ROOT}], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "NO_FALLBACK_OK" in r.stdout, r.stdout + r.stderr


def test_aux_tables_are_current():
    if not os.path.exists("/root/reference/SRC/AudioSDRlib/AudioIQgenerator.h"):
        pytest.skip("reference tree not present")
    r = subprocess.run(["python", os.path.join(ROOT, "tools", "gen_aux_tables.py"), "--check"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout


def test_iq_generator_taps_keep_the_tap_41_sign():
    """The generator's tap table is NOT the receiver's: tap 41 is positive in AudioIQgenerator.h, negative in AudioSDR.h."""
    for path in (os.path.join(ROOT, "oracle", "aux_tables.inc"), os.path.join(ROOT, "audiosdr_b200", "csrc", "aux_tables.inc")):
        a = open(path).read()
        taps = re.search(r"AUX_IQ_HILBERT\[64\] = \{([^}]*)\}", a).group(1).replace("u", "").split(",")
        v = np.array([int(t, 16) for t in taps if t.strip()], np.uint32).view(np.float32)
        assert v[41] > 0 and (np.delete(v, 41) < 0).all(), path
