"""tools/bench_grabber_snapshots.py -- what it costs to get every snapshot a grabber process call publishes, and its spectrum
(sdr_grabber_process_device_snapshots), against the path that existed before: 2-block process calls, each followed by
sdr_grabber_spectrum_device.

All in one process, every step between its own CUDA events on one stream, the arms of a comparison alternated step by step
(who goes first rotates); inputs of 512 MB (> 126 MB L2) per workload:
  snapshots  power-only, raw-only and both, at 4 096 channels x 256 blocks and 16 384 channels x 64 blocks (4 096 x 32 768
             samples x 2 rails and 16 384 x 8 192 x 2: 512 MB each).  Snapshots/s, and the share of two bounds computed here
             from shapes: HBM (1 KB read per snapshot, + 1 KB of power, + 1 KB of raw snapshot) and FP32 issue (11 008 unfused
             operations per spectrum: 1 024 butterflies x 10 + 256 x 3), against the live FMUL+FADD microbenchmark of
             libsdr_batch.so.
  gate       power-only against the old path run on the parent build (--parent-lib) on the same planes; the power of both
             must be bit-identical.
  tap        the spectrum tap (sdr_grabber_spectrum_device, bench_aux.py's grabber_spectrum workload: 65 536 channels) on this
             build's warp FFT core against the parent build's CTA-per-channel kernel, bit-identical power.
  plain      the plain process call (no outputs) of this build against the parent build's at 4 096 x 256, with the state
             blobs of both handles compared byte for byte.
The GPU's name and power limit are read in the same run.

    python tools/bench_grabber_snapshots.py --parent-lib build/parent/libsdr_aux.so --out profiles/r06_grabber_snapshots_bench.json
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

N_BLOCK = 128
WORKLOADS = ((4096, 256), (16384, 64))
FLOP_PER_SPECTRUM = 1024 * 10 + 256 * 3
READ_B, POWER_B, RAW_B = 1024, 1024, 1024


def planes(nch, nb, seed, dev):
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    mk = lambda: (torch.randn((nch, nb * N_BLOCK), generator=g, device=dev) * 3000.0).round().clamp(-32768, 32767).to(torch.int16)
    return mk(), mk()


def snapshots_part(aux, args, dev, parent, hbm, fp32):
    import torch
    from bench_aux_subset import alternate, stats
    stream = torch.cuda.current_stream()
    out = []
    for nch, nb in WORKLOADS:
        I, Q = planes(nch, nb, 11, dev)
        S = (nb + 1) // 2
        items = nch * S
        raw = torch.empty((nch, S, 512), dtype=torch.int16, device=dev)
        pw = torch.empty((nch, S, 256), dtype=torch.float32, device=dev)
        hs = {k: aux.GrabberBatch(nch) for k in ("power", "raw", "both")}
        arms = {"power": lambda: hs["power"].process(I, Q, n_blocks=nb, stream=stream, power=pw),
                "raw": lambda: hs["raw"].process(I, Q, n_blocks=nb, stream=stream, snapshots=raw),
                "both": lambda: hs["both"].process(I, Q, n_blocks=nb, stream=stream, snapshots=raw, power=pw)}
        # the old path on the parent build: 2-block calls, each followed by the spectrum tap into slot k (slot-major buffer)
        old = aux.GrabberBatch(nch, _lib=parent)
        old_pw = torch.empty((S, nch, 256), dtype=torch.float32, device=dev)

        def old_path():
            for k in range(S):
                old.process(I[:, 2 * k * N_BLOCK:(2 * k + 2) * N_BLOCK], Q[:, 2 * k * N_BLOCK:(2 * k + 2) * N_BLOCK], n_blocks=2, stream=stream)
                old.spectrum_device(old_pw[k], stream=stream)
        arms["old_path_parent"] = old_path
        arms["power"]()
        old_path()
        torch.cuda.synchronize()
        identical = bool(torch.equal(pw.view(torch.int32), old_pw.transpose(0, 1).contiguous().view(torch.int32)))
        ms = alternate(args.steps, args.warmup, arms)
        torch.cuda.synchronize()
        r = dict(channels=nch, blocks=nb, snapshots_per_call=items, input_mb=2 * I.numel() * 2 / 1e6,
                 gate=dict(power_bit_identical_to_old_path=identical))
        for k, per in (("power", READ_B + POWER_B), ("raw", READ_B + RAW_B), ("both", READ_B + POWER_B + RAW_B)):
            st = stats(ms[k])
            s = st["ms_median"] * 1e-3
            st["snapshots_per_s"] = items / s
            st["hbm_bound_share"] = (items * per / (hbm * 1e9)) / s
            if k != "raw":
                st["fp32_issue_bound_share"] = (items * FLOP_PER_SPECTRUM / fp32) / s if fp32 else None
            st["bytes_per_snapshot"] = per
            r[k] = st
        r["old_path_parent"] = stats(ms["old_path_parent"])
        r["old_path_parent"]["launches_per_call"] = 2 * S
        r["gate"]["power_speedup_vs_old_path"] = r["old_path_parent"]["ms_median"] / r["power"]["ms_median"]
        r["gate"]["faster"] = r["power"]["ms_median"] < r["old_path_parent"]["ms_median"]
        print(json.dumps(r), flush=True)
        out.append(r)
        for h in list(hs.values()) + [old]:
            h.close()
        del I, Q, raw, pw, old_pw
        torch.cuda.empty_cache()
    return out


def tap_part(aux, args, dev, parent):
    """bench_aux.py's grabber_spectrum workload on this build and on the parent build."""
    import torch
    from bench_aux_subset import alternate, stats
    stream = torch.cuda.current_stream()
    nch = 65536
    g = torch.Generator(device=dev); g.manual_seed(99)
    I = (torch.randn((nch, 256), generator=g, device=dev) * 3000.0).round().clamp(-32768, 32767).to(torch.int16)
    Q = (torch.randn((nch, 256), generator=g, device=dev) * 3000.0).round().clamp(-32768, 32767).to(torch.int16)
    t = torch.arange(256, device=dev, dtype=torch.float32)
    I += (8000.0 * torch.cos(2 * np.pi * 37.0 / 256.0 * t)).round().to(torch.int16)[None, :]
    Q += (8000.0 * torch.sin(2 * np.pi * 37.0 / 256.0 * t)).round().to(torch.int16)[None, :]
    hs = {"new": aux.GrabberBatch(nch), "parent": aux.GrabberBatch(nch, _lib=parent)}
    pw = {k: torch.empty((nch, 256), dtype=torch.float32, device=dev) for k in hs}
    for k, h in hs.items():
        h.process(I, Q, n_blocks=2, stream=stream)
        assert h.spectrum_device(pw[k], stream=stream)
    torch.cuda.synchronize()
    identical = bool(torch.equal(pw["new"].view(torch.int32), pw["parent"].view(torch.int32)))
    ms = alternate(args.steps, args.warmup, {k: (lambda k=k: hs[k].spectrum_device(pw[k], stream=stream)) for k in hs})
    r = dict(channels=nch, power_bit_identical=identical)
    for k in hs:
        r[k] = stats(ms[k])
        r[k]["spectra_per_s"] = nch / (r[k]["ms_median"] * 1e-3)
        hs[k].close()
    r["new_vs_parent"] = r["new"]["ms_median"] / r["parent"]["ms_median"] - 1.0
    print(json.dumps(r), flush=True)
    return r


def plain_part(aux, args, dev, parent):
    import torch
    from bench_aux_subset import alternate, stats
    stream = torch.cuda.current_stream()
    nch, nb = WORKLOADS[0]
    sets = [planes(nch, nb, 20 + s, dev) for s in range(2)]
    hs = {"new": aux.GrabberBatch(nch), "parent": aux.GrabberBatch(nch, _lib=parent)}
    it = {k: 0 for k in hs}

    def step(k):
        I, Q = sets[it[k] % 2]
        it[k] += 1
        hs[k].process(I, Q, n_blocks=nb - 1, stream=stream)  # odd: the phase and the carried half change every call
    ms = alternate(args.steps, args.warmup, {k: (lambda k=k: step(k)) for k in hs})
    torch.cuda.synchronize()
    same_calls = it["new"] == it["parent"]
    identical = same_calls and bool(np.array_equal(hs["new"].export_state(), hs["parent"].export_state()))
    r = dict(channels=nch, blocks=nb - 1, state_bit_identical=identical, new=stats(ms["new"]), parent=stats(ms["parent"]))
    r["new_vs_parent"] = r["new"]["ms_median"] / r["parent"]["ms_median"] - 1.0
    for h in hs.values():
        h.close()
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--parent-lib", default=os.path.join(ROOT, "build", "parent", "libsdr_aux.so"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--parts", default="snapshots,tap,plain")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    from bench_block_status import gpu_info
    from bench_aux import fp32_issue_rate, measured_hbm
    from audiosdr_b200 import aux
    dev = torch.device("cuda:0")
    hbm, hbm_src = measured_hbm()
    fp32 = fp32_issue_rate()
    parent = aux.load_library(path=args.parent_lib)
    out = dict(tool="tools/bench_grabber_snapshots.py", gpu=gpu_info(), version=aux.load_library().sdr_aux_version().decode(),
               parent_lib=os.path.relpath(args.parent_lib, ROOT), hbm_gbs=hbm, hbm_source=hbm_src, fp32_issue_per_s=fp32,
               fp32_issue_source="measured live: unfused FMUL+FADD microbenchmark of libsdr_batch.so",
               flop_per_spectrum=FLOP_PER_SPECTRUM, steps=args.steps, warmup=max(args.warmup, 3))
    parts = args.parts.split(",")
    if "snapshots" in parts:
        out["snapshots"] = snapshots_part(aux, args, dev, parent, hbm, fp32)
    if "tap" in parts:
        out["tap"] = tap_part(aux, args, dev, parent)
    if "plain" in parts:
        out["plain"] = plain_part(aux, args, dev, parent)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
