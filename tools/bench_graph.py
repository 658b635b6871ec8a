"""tools/bench_graph.py -- the receiver graph streamed from host memory (include/sdr_graph.h) against the composition of the
blocks' host calls, and both against the host link.

Workload: BASELINE config 2's receiver mix (bench.py's planes and setters), 4 096 channels, 256 blocks per call, pinned
int16 host planes, pre-processor front; three cases: detector off (correction +1 on every channel) with the grabber tap off
and on (the tap's spectra come down too: float32 [S][256] per row), and the detector started on every channel.  Per case,
end to end in channel-samples per second (Msps), each a host clock around `--calls` calls submitted back to back and
waited for, the best of `--reps` repetitions, the variants alternated:
  graph        sdr_graph_submit_host, two calls in flight (6 B per sample over the link; 10 with the tap's spectra)
  composition  sdr_preproc_process_host, then sdr_batch_submit_host on the corrected planes (14 B per sample); no host form
               of the grabber exists, so the tap-on case has none
  link_bound   the graph's own bytes copied up and down at once on two streams, nothing computed (as bench.py's
               e2e.link_bound)
  compute      the same blocks' device calls on device-resident planes, nothing copied: if the graph falls short of the
               link bound and this is below it, the compute stream is the exposed one
The GPU's name and power limit are read in the same run.

    python tools/bench_graph.py --out profiles/r09_graph_bench.json
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

NCH, NBLK = 4096, 256


def run_case(name, detector, tap, args, dev, I16, Q16, calls):
    import torch
    from audiosdr_b200 import api, aux, graph
    ns = NBLK * 128
    S = (NBLK + 1) // 2

    def members():
        rx = api.SdrBatch(NCH)
        rx.configure(calls)
        pp = aux.PreProcessorBatch(NCH)
        if detector:
            pp.startAutoI2SerrorDetection()
        else:
            pp.setI2SerrorCompensation(None, 1)
        return rx, pp

    pin = lambda t: t.pin_memory().numpy()
    hI, hQ = pin(I16.cpu()), pin(Q16.cpu())
    hO = [pin(torch.empty((NCH, ns), dtype=torch.int16)) for _ in range(2)]
    hP = [pin(torch.empty((NCH, S, 256), dtype=torch.float32)) for _ in range(2)] if tap else None
    hM = [(pin(torch.empty((NCH, ns), dtype=torch.int16)), pin(torch.empty((NCH, ns), dtype=torch.int16))) for _ in range(2)]

    rx_g, pp_g = members()
    gr = aux.GrabberBatch(NCH) if tap else None
    g = graph.GraphBatch(rx_g, preproc=pp_g, grabber=gr)

    def run_graph():
        t = []
        for k in range(args.calls):
            t.append(g.submit_host(hI, hQ, hO[k & 1], n_blocks=NBLK, power=hP[k & 1] if tap else None)[0])
            if k >= 1:
                g.wait_host(t[k - 1])
        g.wait_host()

    rx_c, pp_c = members()

    def run_composition():
        t = []
        for k in range(args.calls):
            if k >= 2:
                rx_c.wait_host(t[k - 2])  # the receiver's call k - 2 has read the corrected planes set k & 1
            mI, mQ = hM[k & 1]
            pp_c.process_host(hI, hQ, mI, mQ, n_blocks=NBLK)
            t.append(rx_c.submit_host(mI, mQ, hO[k & 1], n_blocks=NBLK))
        rx_c.wait_host()

    dI, dQ = I16, Q16
    dO = torch.empty((NCH, ns), dtype=torch.int16, device=dev)
    dP = torch.empty((NCH, S, 256), dtype=torch.float32, device=dev) if tap else None
    s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def run_link():
        for k in range(args.calls):
            with torch.cuda.stream(s_up):
                dI.copy_(torch.from_numpy(hI), non_blocking=True); dQ.copy_(torch.from_numpy(hQ), non_blocking=True)
            with torch.cuda.stream(s_dn):
                torch.from_numpy(hO[k & 1]).copy_(dO, non_blocking=True)
                if tap:
                    torch.from_numpy(hP[k & 1]).copy_(dP, non_blocking=True)
        torch.cuda.synchronize()

    rx_d, pp_d = members()
    gr_d = aux.GrabberBatch(NCH) if tap else None
    mI, mQ = torch.empty_like(dI), torch.empty_like(dQ)
    dO2 = torch.empty_like(dO)

    def run_compute():
        for _ in range(args.calls):
            pp_d.process(dI, dQ, mI, mQ, n_blocks=NBLK)
            if tap:
                gr_d.process(mI, mQ, n_blocks=NBLK, power=dP)
            rx_d.process(mI, mQ, dO2, n_blocks=NBLK)
        torch.cuda.synchronize()

    variants = {"graph": run_graph, "link_bound": run_link, "compute": run_compute}
    if not tap:
        variants["composition"] = run_composition
    for f in variants.values():  # warm-up: staging allocated, modules loaded
        f()
    best = {k: None for k in variants}
    for rep in range(args.reps):
        order = list(variants)
        order = order[rep % len(order):] + order[:rep % len(order)]
        for k in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            variants[k]()
            dt = time.perf_counter() - t0
            best[k] = dt if best[k] is None else min(best[k], dt)
    samples = float(NCH) * ns * args.calls
    r = dict(case=name, detector_on_all_channels=detector, grabber_tap=tap, channels=NCH, blocks_per_call=NBLK, calls=args.calls,
             link_bytes_per_sample=dict(graph=6 + (4 if tap else 0), composition=None if tap else 14))
    for k, dt in best.items():
        r[k + "_msps"] = samples / dt / 1e6
    r["graph_vs_link_bound"] = r["graph_msps"] / r["link_bound_msps"]
    if not tap:
        r["graph_vs_composition"] = r["graph_msps"] / r["composition_msps"]
    r["exposed"] = ("link" if r["link_bound_msps"] <= r["compute_msps"] else "compute") + \
        " (the slower of the copy-only and compute-only rates)"
    g.close()
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--calls", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    import bench
    from bench_block_status import gpu_info
    from audiosdr_b200 import graph
    dev = torch.device("cuda:0")
    I16, Q16, calls = bench.synth_planes(dev, 0, NCH, NBLK * 128, 1234, config_id=2)
    out = dict(tool="tools/bench_graph.py", gpu=gpu_info(), version=graph.load_library().sdr_graph_version().decode(),
               wall_clock="host clock around the calls of a variant, ended by a device synchronise; best of --reps", cases=[])
    for name, detector, tap in (("detector_off_tap_off", False, False), ("detector_off_tap_on", False, True), ("detector_on", True, False)):
        r = run_case(name, detector, tap, args, dev, I16, Q16, calls)
        out["cases"].append(r)
        print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
