"""tools/bench_pp_block_status.py -- what the pre-processor's per-block status records cost (sdr_preproc_process_device_status),
at bench_aux.py's sizes: 4 096 channels x 256 blocks, inputs 256 MB per plane (> the 126 MB L2).

Each step runs between its own CUDA events on one stream, the variants alternated step by step (who goes first rotates):
  records  plain call against the call with records on two handles in the same state, for preproc_static (correction +1
           everywhere: the feed-forward path, records from pp_finish_kernel<.., true>) and preproc_detect (detector running
           everywhere on noise that never reaches a verdict, as in bench_aux.py: records from pp_detect_kernel<.., true>);
           outputs of the first call of both compared bit for bit.
  parent   the plain call of this build against another build of libsdr_aux.so (--parent-lib, e.g. the parent commit's),
           and the run-to-run spread: the same build against itself in the same alternation.
The GPU's name and power limit are read in the same run.

    python tools/bench_pp_block_status.py --parent-lib build/parent/libsdr_aux.so --out profiles/r08_pp_block_status_bench.json
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from bench_aux_subset import NBLK, NCH, alternate, inputs, make, stats  # noqa: E402

PATHS = ("preproc_static", "preproc_detect")


def records_vs_plain(aux, path, args, dev):
    import torch
    stream = torch.cuda.current_stream()
    planes = inputs(path, NCH, 1234, dev)
    rec, plain = make(aux, path, NCH), make(aux, path, NCH)
    o_rec = [torch.empty_like(planes[0]) for _ in range(2)]
    o_plain = [torch.empty_like(planes[0]) for _ in range(2)]
    status = torch.empty((NBLK, aux.PP_BS_FIELDS, NCH), dtype=torch.int32, device=dev)
    run_rec = lambda: rec.process(planes[0], planes[1], o_rec[0], o_rec[1], n_blocks=NBLK, stream=stream, block_status=status)
    run_plain = lambda: plain.process(planes[0], planes[1], o_plain[0], o_plain[1], n_blocks=NBLK, stream=stream)
    run_rec(); run_plain()
    torch.cuda.synchronize()
    identical = all(bool(torch.equal(a, b)) for a, b in zip(o_rec, o_plain))
    ms = alternate(args.steps, args.warmup, {"records": run_rec, "plain": run_plain})
    torch.cuda.synchronize()
    r = dict(path=path, channels=NCH, blocks_per_step=NBLK, plain=stats(ms["plain"]), records=stats(ms["records"]),
             outputs_bit_identical=identical, record_mb_per_step=status.numel() * 4 / 1e6,
             plane_mb_per_step=4 * planes[0].numel() * 2 / 1e6)
    r["records_vs_plain"] = r["records"]["ms_median"] / r["plain"]["ms_median"] - 1.0
    rec.close(); plain.close()
    del planes, o_rec, o_plain, status
    torch.cuda.empty_cache()
    return r


def plain_vs_lib(aux, path, args, dev, other_lib, label):
    import torch
    stream = torch.cuda.current_stream()
    planes = inputs(path, NCH, 1234, dev)
    new, other = make(aux, path, NCH), make(aux, path, NCH, lib=other_lib)
    o_new = [torch.empty_like(planes[0]) for _ in range(2)]
    o_other = [torch.empty_like(planes[0]) for _ in range(2)]
    run_new = lambda: new.process(planes[0], planes[1], o_new[0], o_new[1], n_blocks=NBLK, stream=stream)
    run_other = lambda: other.process(planes[0], planes[1], o_other[0], o_other[1], n_blocks=NBLK, stream=stream)
    run_new(); run_other()
    torch.cuda.synchronize()
    identical = all(bool(torch.equal(a, b)) for a, b in zip(o_new, o_other))
    ms = alternate(args.steps, args.warmup, {"new": run_new, label: run_other})
    torch.cuda.synchronize()
    r = dict(path=path, new=stats(ms["new"]), outputs_bit_identical=identical)
    r[label] = stats(ms[label])
    r["new_vs_" + label] = r["new"]["ms_median"] / r[label]["ms_median"] - 1.0
    new.close(); other.close()
    del planes, o_new, o_other
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--parent-lib", default=os.path.join(ROOT, "build", "parent", "libsdr_aux.so"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    from bench_block_status import gpu_info
    from audiosdr_b200 import aux
    dev = torch.device("cuda:0")
    out = dict(tool="tools/bench_pp_block_status.py", gpu=gpu_info(), version=aux.load_library().sdr_aux_version().decode())
    out["records"] = []
    for path in PATHS:
        r = records_vs_plain(aux, path, args, dev)
        out["records"].append(r)
        print(json.dumps(r), flush=True)
    parent = aux.load_library(path=args.parent_lib)
    out["parent_lib"] = os.path.relpath(args.parent_lib, ROOT)
    out["parent"], out["spread"] = [], []
    for path in PATHS:
        r = plain_vs_lib(aux, path, args, dev, parent, "parent")
        out["parent"].append(r)
        print(json.dumps(r), flush=True)
        r = plain_vs_lib(aux, path, args, dev, None, "same")
        out["spread"].append(r)
        print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
