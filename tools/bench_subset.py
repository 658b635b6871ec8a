"""tools/bench_subset.py -- what calls on a subset of the channels (sdr_batch_process_device_subset) cost on the GPU.

Three measurements in one process, each step between its own CUDA events on one stream:
  plain    BASELINE configs 2-5 at the benchmark's sizes (bench.py's Workload): this build's plain process() against another
           build of the library (--parent-lib, e.g. the parent commit's), alternated step by step, and whether their audio of
           the last step is bit-identical.
  subset   a 16 384-channel handle of config 4's mix running subsets of 1 024, 4 096 and 8 192 channels, against a handle of
           exactly that many channels (the same channels' configuration) running plain calls, alternated step by step.  Two
           histories: "aligned" (the subset's channels have all run the same calls: one oscillator phase per mode, no slot
           turns) and "random" (before timing, random subsets ran for random lengths, so the subset's channels lag the clock
           by different amounts: RoleNco's per-lane path and the slot turns of the reset kernel).
  host     host time of one subset call (1 block) on a 65 536-channel handle listing all 65 536 ids in a random order: the
           id list repeated (grouping reused) and a new order at every call (grouping built again), time from the call to
           its return (the launches are asynchronous; the device work is synchronised outside the timed region).
The GPU's name and power limit are read in the same run.

    python tools/bench_subset.py --parent-lib build/parent/libsdr_batch.so --out profiles/r04_subset_bench.json
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


def stats(a):
    a = np.asarray(a, dtype=np.float64)
    return dict(ms_median=float(np.median(a)), ms_min=float(a.min()), ms_max=float(a.max()))


def alternate(steps, warmup, fns):
    """Runs each fn once per step, rotating who goes first; returns {name: [ms per step]}."""
    import torch
    st = torch.cuda.current_stream()
    names = list(fns)
    for _ in range(warmup):
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


def plain_vs_parent(cfg, args, dev, new_lib, parent_lib):
    import torch
    import audiosdr_b200 as A
    import bench
    w = bench.Workload(cfg, 0, 1, 0, dev)
    par = A.SdrBatch(w.nch, _lib=parent_lib)
    par.configure(w.calls)
    out_p = torch.empty_like(w.out)
    ms = alternate(args.steps, args.warmup, {
        "new": lambda: w.b.process(w.If, w.Qf, w.out, n_blocks=w.nblk),
        "parent": lambda: par.process(w.If, w.Qf, out_p, n_blocks=w.nblk)})
    torch.cuda.synchronize()
    res = dict(config=cfg, channels=w.nch, blocks_per_step=w.nblk, new=stats(ms["new"]), parent=stats(ms["parent"]),
               launches_per_step=dict(new=None, parent=None))
    res["new_vs_parent"] = res["new"]["ms_median"] / res["parent"]["ms_median"] - 1.0
    res["audio_bit_identical"] = bool(np.array_equal(w.out.cpu().numpy().view(np.uint32), out_p.cpu().numpy().view(np.uint32)))
    n0, p0 = w.b.launch_count, par.launch_count
    w.b.process(w.If, w.Qf, w.out, n_blocks=w.nblk)
    par.process(w.If, w.Qf, out_p, n_blocks=w.nblk)
    res["launches_per_step"] = dict(new=w.b.launch_count - n0, parent=par.launch_count - p0)
    par.close()
    w.free()
    torch.cuda.empty_cache()
    return res


def subset_vs_handle(args, dev, lib):
    import torch
    import audiosdr_b200 as A
    import signals as S
    nch, nb = 16384, args.subset_blocks
    _, _, ev = S.make(4, list(range(nch)), 1)
    calls = [(e[0], e[2]) + tuple(e[3:]) for e in ev]
    T_I, T_Q, _ = S.make(4, list(range(256)), nb)
    rng = np.random.default_rng(7)
    out = []
    for history in ("aligned", "random"):
        big = A.SdrBatch(nch, _lib=lib)
        big.configure(calls)
        if history == "random":  # random subsets for random lengths: the channels' clocks and oscillator phases spread
            for _ in range(12):
                ids = rng.permutation(nch)[:int(nch * rng.uniform(0.2, 0.8))].astype(np.uint32)
                n = int(rng.integers(1, 9))
                z = torch.zeros((len(ids), n * N_BLOCK), dtype=torch.int16, device=dev)
                big.process(z, z, torch.empty((len(ids), n * N_BLOCK), dtype=torch.float32, device=dev), n_blocks=n, channels=ids)
        for k in (1024, 4096, 8192):
            ids = np.sort(rng.permutation(nch)[:k]).astype(np.uint32)
            small = A.SdrBatch(k, _lib=lib)  # the same channels' configuration: channel i is configured as channel ids[i]
            _, _, ev_k = S.make(4, ids.tolist(), 1)
            small.configure([(e[0], e[2]) + tuple(e[3:]) for e in ev_k])
            I = torch.from_numpy(np.ascontiguousarray(T_I[ids % 256])).to(dev)
            Q = torch.from_numpy(np.ascontiguousarray(T_Q[ids % 256])).to(dev)
            o1, o2 = torch.empty((k, nb * N_BLOCK), dtype=torch.float32, device=dev), torch.empty((k, nb * N_BLOCK), dtype=torch.float32, device=dev)
            ms = alternate(args.steps, args.warmup, {
                "subset_of_16384": lambda: big.process(I, Q, o1, n_blocks=nb, channels=ids),
                "handle_of_k": lambda: small.process(I, Q, o2, n_blocks=nb)})
            torch.cuda.synchronize()
            r = dict(history=history, k=k, blocks_per_step=nb, subset_of_16384=stats(ms["subset_of_16384"]), handle_of_k=stats(ms["handle_of_k"]))
            r["subset_vs_handle"] = r["subset_of_16384"]["ms_median"] / r["handle_of_k"]["ms_median"] - 1.0
            r["msps_subset"] = k * nb * N_BLOCK / (r["subset_of_16384"]["ms_median"] * 1e-3) / 1e6
            out.append(r)
            print(json.dumps(r), flush=True)
            small.close()
        big.close()
        torch.cuda.empty_cache()
    return out


def host_time(args, dev, lib):
    import torch
    import audiosdr_b200 as A
    nch = 65536
    b = A.SdrBatch(nch, _lib=lib)
    z = torch.zeros((nch, N_BLOCK), dtype=torch.int16, device=dev)
    o = torch.empty((nch, N_BLOCK), dtype=torch.float32, device=dev)
    rng = np.random.default_rng(3)
    res = {}
    for form in ("same_list", "new_list"):
        ids = rng.permutation(nch).astype(np.uint32)
        t = []
        for s in range(args.host_calls + 2):
            if form == "new_list":
                ids = rng.permutation(nch).astype(np.uint32)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            b.process(z, z, o, n_blocks=1, channels=ids)
            t1 = time.perf_counter()
            if s >= 2:
                t.append((t1 - t0) * 1e3)
        torch.cuda.synchronize()
        res[form] = stats(t)
    b.close()
    return dict(channels=nch, ids=nch, calls=args.host_calls, host_ms_per_call=res)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--parent-lib", default=os.path.join(ROOT, "build", "parent", "libsdr_batch.so"))
    ap.add_argument("--configs", default="2,3,4,5")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--subset-blocks", type=int, default=64)
    ap.add_argument("--host-calls", type=int, default=20)
    ap.add_argument("--parts", default="plain,subset,host")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    from bench_block_status import gpu_info
    os.environ.pop("SDR_LIB", None)
    from audiosdr_b200 import api
    lib = api.load_library()
    dev = torch.device("cuda:0")
    out = dict(tool="tools/bench_subset.py", gpu=gpu_info(), version=lib.sdr_batch_version().decode())
    parts = args.parts.split(",")
    if "plain" in parts:
        parent = api.load_library(path=args.parent_lib)
        out["parent_lib"] = os.path.relpath(args.parent_lib, ROOT)
        out["plain"] = []
        for cfg in [int(c) for c in args.configs.split(",")]:
            r = plain_vs_parent(cfg, args, dev, lib, parent)
            out["plain"].append(r)
            print(json.dumps(r), flush=True)
    if "subset" in parts:
        out["subset"] = subset_vs_handle(args, dev, lib)
    if "host" in parts:
        out["host"] = host_time(args, dev, lib)
        print(json.dumps(out["host"]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
