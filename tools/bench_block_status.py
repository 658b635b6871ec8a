"""tools/bench_block_status.py -- cost of the per-block status records, and the path without them against another build.

For BASELINE configs 2-5 at the benchmark's sizes (bench.py's Workload: same planes, setters and step), three handles on the
same input run in one process, alternated step by step on one stream, each step between its own CUDA events:
    off     this build, process() without records
    on      this build, process() with records ([blocks, 7, channels] int32 on the device)
    parent  another build of the library (--parent-lib, e.g. the parent commit's), process() without records
Reported per config: ms per step (median, min, max) and Msps (channel-samples/s) for each, the records' overhead (on / off),
off against parent, and whether the three audio planes of the last step are bit-identical.  The GPU's name and power limit
are read in the same run.

    python tools/bench_block_status.py --parent-lib build/parent/libsdr_batch.so --out profiles/r03_block_status.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def gpu_info():
    import torch
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except Exception as e:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = "not read: %s" % e
    return info


def run_config(cfg, args, dev, new_lib, parent_lib):
    import torch
    import audiosdr_b200 as A
    import bench
    w = bench.Workload(cfg, 0, 1, 0, dev, nblk=args.blocks or None)
    handles = {"off": w.b, "on": A.SdrBatch(w.nch, _lib=new_lib), "parent": A.SdrBatch(w.nch, _lib=parent_lib)}
    for k in ("on", "parent"):
        handles[k].configure(w.calls)
    outs = {k: torch.empty_like(w.out) for k in handles}
    rec = torch.empty((w.nblk, A.BS_FIELDS, w.nch), dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream()

    def step(k):
        handles[k].process(w.If, w.Qf, outs[k], n_blocks=w.nblk, stream=st, block_status=rec if k == "on" else None)

    order = ["off", "on", "parent"]
    for _ in range(args.warmup):
        for k in order:
            step(k)
    torch.cuda.synchronize()
    ms = {k: [] for k in order}
    for s in range(args.steps):
        seq = order[s % 3:] + order[:s % 3]  # rotate who goes first
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record(st)
        for i, k in enumerate(seq):
            step(k)
            ev[i + 1].record(st)
        ev[-1].synchronize()
        for i, k in enumerate(seq):
            ms[k].append(ev[i].elapsed_time(ev[i + 1]))
    torch.cuda.synchronize()
    samples = float(w.nch) * w.ns
    res = dict(config=cfg, channels=w.nch, blocks_per_step=w.nblk, steps=args.steps, warmup=args.warmup)
    for k in order:
        a = np.array(ms[k])
        res[k] = dict(ms_median=float(np.median(a)), ms_min=float(a.min()), ms_max=float(a.max()),
                      msps_median=samples / (np.median(a) * 1e-3) / 1e6)
    res["records_overhead"] = res["on"]["ms_median"] / res["off"]["ms_median"] - 1.0
    res["off_vs_parent"] = res["off"]["ms_median"] / res["parent"]["ms_median"] - 1.0
    a_off = outs["off"].cpu().numpy()
    res["audio_bit_identical"] = dict(on_vs_off=bool(np.array_equal(outs["on"].cpu().numpy().view(np.uint32), a_off.view(np.uint32))),
                                      parent_vs_off=bool(np.array_equal(outs["parent"].cpu().numpy().view(np.uint32), a_off.view(np.uint32))))
    r = rec.cpu().numpy().view(np.uint32)
    res["records"] = dict(bytes_per_step=int(r.nbytes), nb_detected_blocks=int(A.block_status_fields(r)["nb_detected"].sum()),
                          sam_locked_blocks=int(A.block_status_fields(r)["sam_locked"].sum()))
    for h in handles.values():
        h.close()
    w.free()
    del outs, rec
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--parent-lib", default=os.environ.get("SDR_LIB") or os.path.join(ROOT, "build", "parent", "libsdr_batch.so"),
                    help="the other build the path without records is compared with (default: $SDR_LIB, else build/parent/)")
    ap.add_argument("--configs", default="2,3,4,5")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--blocks", type=int, default=0, help="blocks per step (default: the benchmark's per config)")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    os.environ.pop("SDR_LIB", None)  # this build is loaded from the package directory, the other one by path
    from audiosdr_b200 import api
    new_lib = api.load_library()
    parent_lib = api.load_library(path=args.parent_lib)
    dev = torch.device("cuda:0")
    out = dict(tool="tools/bench_block_status.py", gpu=gpu_info(), parent_lib=os.path.relpath(args.parent_lib, ROOT),
               new_version=new_lib.sdr_batch_version().decode(), results=[])
    for cfg in [int(c) for c in args.configs.split(",")]:
        r = run_config(cfg, args, dev, new_lib, parent_lib)
        out["results"].append(r)
        print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(dict(gpu=out["gpu"], summary={r["config"]: dict(off_msps=round(r["off"]["msps_median"]), on_msps=round(r["on"]["msps_median"]),
                                                                    parent_msps=round(r["parent"]["msps_median"]),
                                                                    overhead=round(r["records_overhead"], 4), off_vs_parent=round(r["off_vs_parent"], 4))
                                                   for r in out["results"]})))


if __name__ == "__main__":
    main()
