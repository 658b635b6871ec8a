"""tools/bench_aux_subset.py -- what calls on a subset of the channels cost for the pre-processor and the I/Q generator
(sdr_preproc_process_device_subset, sdr_iqgen_process_device_subset), at bench_aux.py's sizes: 4 096 channels x 256 blocks.

Three measurements in one process, each step between its own CUDA events on one stream, the variants alternated step by
step (who goes first rotates):
  plain   the plain process() of this build against another build of libsdr_aux.so (--parent-lib, e.g. the parent
          commit's), for iqgen, preproc_static (correction +1 everywhere) and preproc_detect (detector running everywhere,
          noise input that never reaches a verdict, as in bench_aux.py), and whether their outputs of the same call are
          bit-identical.  Inputs 256 MB per plane (> 126 MB L2).
  subset  a 4 096-channel handle running subsets of 1 024, 2 048 and 3 072 random ids (compact planes), against a handle of
          exactly that many channels running plain calls on the same planes.  Each variant rotates over 3 input sets, so that
          a step does not find its input in L2.
  host    host time of one 1-block subset call listing 65 536 ids in random order on a 65 536-channel handle (the id list
          check and upload; the kernels are asynchronous and synchronised outside the timed region).
The GPU's name and power limit are read in the same run.

    python tools/bench_aux_subset.py --parent-lib build/parent/libsdr_aux.so --out profiles/r05_aux_subset_bench.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

N_BLOCK = 128
NCH, NBLK = 4096, 256
PATHS = ("iqgen", "preproc_static", "preproc_detect")


def stats(a):
    a = np.asarray(a, dtype=np.float64)
    return dict(ms_median=float(np.median(a)), ms_min=float(a.min()), ms_max=float(a.max()))


def alternate(steps, warmup, fns):
    """Runs each fn once per step, rotating who goes first; returns {name: [ms per step]}."""
    import torch
    st = torch.cuda.current_stream()
    names = list(fns)
    for _ in range(max(warmup, 3)):
        for k in names:
            fns[k]()
    torch.cuda.synchronize()
    ms = {k: [] for k in names}
    for s in range(steps):
        seq = names[s % len(names):] + names[:s % len(names)]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(seq) + 1)]
        ev[0].record(st)
        for i, k in enumerate(seq):
            fns[k]()
            ev[i + 1].record(st)
        ev[-1].synchronize()
        for i, k in enumerate(seq):
            ms[k].append(ev[i].elapsed_time(ev[i + 1]))
    return ms


def inputs(path, rows, seed, dev):
    """int16 planes [rows, NBLK * 128] on the device: X for iqgen, (I, Q) for the pre-processor (bench_aux.py's signals)."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    noise = lambda: (torch.randn((rows, NBLK * N_BLOCK), generator=g, device=dev) * 3000.0).round().clamp(-32768, 32767).to(torch.int16)
    if path == "iqgen":
        return (noise(),)
    I, Q = noise(), noise()
    if path == "preproc_detect":  # a flat spectrum: no line is ever strong, the detector keeps running (bench_aux.py)
        I, Q = (I.float() / 100.0).round().to(torch.int16), (Q.float() / 100.0).round().to(torch.int16)
        I[:, ::128] = 20000
        Q[:, ::128] = 20000
    return I, Q


def make(aux, path, n, lib=None):
    if path == "iqgen":
        return aux.IQGeneratorBatch(n, _lib=lib)
    h = aux.PreProcessorBatch(n, _lib=lib)
    if path == "preproc_static":
        h.setI2SerrorCompensation(None, 1)
    else:
        h.startAutoI2SerrorDetection()
    return h


def call(h, path, planes, outs, stream, channels=None):
    if path == "iqgen":
        h.process(planes[0], outs[0], outs[1], n_blocks=NBLK, stream=stream, channels=channels)
    else:
        h.process(planes[0], planes[1], outs[0], outs[1], n_blocks=NBLK, stream=stream, channels=channels)


def plain_vs_parent(aux, path, args, dev, parent_lib):
    import torch
    stream = torch.cuda.current_stream()
    planes = inputs(path, NCH, 1234, dev)
    new, par = make(aux, path, NCH), make(aux, path, NCH, lib=parent_lib)
    o_new = [torch.empty_like(planes[0]) for _ in range(2)]
    o_par = [torch.empty_like(planes[0]) for _ in range(2)]
    # the first call of both handles on the same state: outputs must agree bit for bit
    call(new, path, planes, o_new, stream)
    call(par, path, planes, o_par, stream)
    torch.cuda.synchronize()
    identical = all(bool(torch.equal(a, b)) for a, b in zip(o_new, o_par))
    ms = alternate(args.steps, args.warmup, {"new": lambda: call(new, path, planes, o_new, stream),
                                             "parent": lambda: call(par, path, planes, o_par, stream)})
    torch.cuda.synchronize()
    r = dict(path=path, channels=NCH, blocks_per_step=NBLK, new=stats(ms["new"]), parent=stats(ms["parent"]), outputs_bit_identical=identical)
    r["new_vs_parent"] = r["new"]["ms_median"] / r["parent"]["ms_median"] - 1.0
    new.close(); par.close()
    del planes, o_new, o_par
    torch.cuda.empty_cache()
    return r


def subset_vs_handle(aux, path, args, dev):
    import torch
    stream = torch.cuda.current_stream()
    rng = np.random.default_rng(7)
    out = []
    for k in (1024, 2048, 3072):
        ids = rng.permutation(NCH)[:k].astype(np.uint32)
        big, small = make(aux, path, NCH), make(aux, path, k)
        sets = [inputs(path, k, 100 + s, dev) for s in range(3)]
        o1 = [torch.empty_like(sets[0][0]) for _ in range(2)]
        o2 = [torch.empty_like(sets[0][0]) for _ in range(2)]
        it = {"a": 0, "b": 0}

        def sub():
            call(big, path, sets[it["a"] % 3], o1, stream, channels=ids)
            it["a"] += 1

        def hnd():
            call(small, path, sets[it["b"] % 3], o2, stream)
            it["b"] += 1
        ms = alternate(args.steps, args.warmup, {"subset_of_4096": sub, "handle_of_k": hnd})
        torch.cuda.synchronize()
        r = dict(path=path, k=k, blocks_per_step=NBLK, subset_of_4096=stats(ms["subset_of_4096"]), handle_of_k=stats(ms["handle_of_k"]),
                 input_mb_per_step=sum(t.numel() * 2 for t in sets[0]) / 1e6)
        r["subset_vs_handle"] = r["subset_of_4096"]["ms_median"] / r["handle_of_k"]["ms_median"] - 1.0
        r["msps_subset"] = k * NBLK * N_BLOCK / (r["subset_of_4096"]["ms_median"] * 1e-3) / 1e6
        print(json.dumps(r), flush=True)
        out.append(r)
        big.close(); small.close()
        del sets, o1, o2
        torch.cuda.empty_cache()
    return out


def host_time(aux, args, dev):
    import torch
    n = 65536
    rng = np.random.default_rng(3)
    res = {}
    for path in ("iqgen", "preproc_static"):
        h = make(aux, path, n)
        z = torch.zeros((n, N_BLOCK), dtype=torch.int16, device=dev)
        o = [torch.empty_like(z) for _ in range(2)]
        t = []
        for s in range(args.host_calls + 2):
            ids = rng.permutation(n).astype(np.uint32)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if path == "iqgen":
                h.process(z, o[0], o[1], n_blocks=1, channels=ids)
            else:
                h.process(z, z, o[0], o[1], n_blocks=1, channels=ids)
            t1 = time.perf_counter()
            if s >= 2:
                t.append((t1 - t0) * 1e3)
        torch.cuda.synchronize()
        res[path] = stats(t)
        h.close()
    return dict(channels=n, ids=n, calls=args.host_calls, host_ms_per_call=res)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--parent-lib", default=os.path.join(ROOT, "build", "parent", "libsdr_aux.so"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-calls", type=int, default=20)
    ap.add_argument("--parts", default="plain,subset,host")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    from bench_block_status import gpu_info
    from audiosdr_b200 import aux
    dev = torch.device("cuda:0")
    out = dict(tool="tools/bench_aux_subset.py", gpu=gpu_info(), version=aux.load_library().sdr_aux_version().decode())
    parts = args.parts.split(",")
    if "plain" in parts:
        parent = aux.load_library(path=args.parent_lib)
        out["parent_lib"] = os.path.relpath(args.parent_lib, ROOT)
        out["plain"] = []
        for path in PATHS:
            r = plain_vs_parent(aux, path, args, dev, parent)
            out["plain"].append(r)
            print(json.dumps(r), flush=True)
    if "subset" in parts:
        out["subset"] = [r for path in PATHS for r in subset_vs_handle(aux, path, args, dev)]
    if "host" in parts:
        out["host"] = host_time(aux, args, dev)
        print(json.dumps(out["host"]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
