"""tools/bench_waterfall.py -- averaged waterfall lines (sdr_grabber_process_device_waterfall, the graph's _waterfall calls)
against what they replace.

Workload: 4 096 channels x 256 blocks per call (128 pairs per row), BASELINE config 2's planes and receiver mix (bench.py).
  device   per call, device-resident planes, CUDA events around `--iters` calls, best of `--reps`: the grabber's power-only
           snapshot call (every pair's spectrum written, 1 KB per pair) against the waterfall call at K = 1, 8 and 16 (the
           same 128 FFTs per row; 1 KB per K pairs written).  Rate in snapshots (pairs) per second.
  graph    sdr_graph_submit_host with the pre-processor front (correction +1), two calls in flight, host clock around `--calls`
           calls, best of `--reps`, variants alternated: no tap; tap with power-only spectra (float32 [S][256] down); tap
           with a waterfall at K = 1, 8, 16 on rows in one accumulation state, and K = 8 on rows that alternate (odd channels
           one pair ahead, so the rows' line slots differ from call to call).  Each case beside its copy-only bound measured in
           the same run: the case's own bytes copied up and down at once on two streams, nothing computed.
The GPU's name and power limit are read in the same run.

    python tools/bench_waterfall.py --out profiles/r10_waterfall_bench.json
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


def device_cases(args, dev, mI, mQ):
    import torch
    from audiosdr_b200 import aux
    S = (NBLK + 1) // 2
    power = torch.empty((NCH, S, 256), dtype=torch.float32, device=dev)
    gr = aux.GrabberBatch(NCH)
    fns = {"snapshots_power_only": lambda: gr.process(mI, mQ, n_blocks=NBLK, power=power)}
    for K in (1, 8, 16):
        wf, g = aux.WaterfallBatch(NCH, K), aux.GrabberBatch(NCH)
        lines = torch.empty((NCH, wf.line_slots(NBLK), 256), dtype=torch.float32, device=dev)
        fns["waterfall_k%d" % K] = (lambda g=g, wf=wf, lines=lines: g.process(mI, mQ, n_blocks=NBLK, waterfall=wf, lines=lines))
        fns["waterfall_k%d" % K].keep = (wf, g, lines)
    best = {k: None for k in fns}
    for f in fns.values():
        f()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for rep in range(args.reps):
        for k, f in fns.items():
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.iters):
                f()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1) / args.iters
            best[k] = ms if best[k] is None else min(best[k], ms)
    pairs = float(NCH) * S
    out = {k: dict(ms_per_call=ms, gsnapshots_per_s=pairs / ms / 1e6) for k, ms in best.items()}
    for k in out:
        out[k]["vs_power_only"] = best["snapshots_power_only"] / best[k]
    return out


def graph_cases(args, dev, I16, Q16, calls):
    import torch
    from audiosdr_b200 import api, aux, graph
    ns, S = NBLK * 128, (NBLK + 1) // 2
    pin = lambda t: t.pin_memory().numpy()
    hI, hQ = pin(I16.cpu()), pin(Q16.cpu())
    hO = [pin(torch.empty((NCH, ns), dtype=torch.int16)) for _ in range(2)]
    dI, dQ, dO = I16, Q16, torch.empty((NCH, ns), dtype=torch.int16, device=dev)
    s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    odd = [c for c in range(NCH) if c % 2]

    def make(case):
        rx = api.SdrBatch(NCH)
        rx.configure(calls)
        pp = aux.PreProcessorBatch(NCH)
        pp.setI2SerrorCompensation(None, 1)
        kind, K, alt = case
        gr = aux.GrabberBatch(NCH) if kind != "none" else None
        wf = aux.WaterfallBatch(NCH, K) if kind == "waterfall" else None
        g = graph.GraphBatch(rx, preproc=pp, grabber=gr, waterfall=wf)
        if alt:  # odd channels one pair (and one block of phase) ahead
            x = pin(torch.zeros((len(odd), 3 * 128), dtype=torch.int16))
            a = pin(torch.zeros((len(odd), 3 * 128), dtype=torch.int16))
            g.process_host(x, x, a, n_blocks=3, channels=odd, lines=pin(torch.zeros((len(odd), wf.line_slots(3), 256))))
        down = None
        if kind == "power":
            down = [pin(torch.empty((NCH, S, 256), dtype=torch.float32)) for _ in range(2)]
        elif kind == "waterfall":
            down = [pin(torch.empty((NCH, wf.line_slots(NBLK), 256), dtype=torch.float32)) for _ in range(2)]
        dD = torch.empty(down[0].shape, dtype=torch.float32, device=dev) if down is not None else None

        def run_graph():
            t = []
            for k in range(args.calls):
                kw = {"power": down[k & 1]} if kind == "power" else {"lines": down[k & 1]} if kind == "waterfall" else {}
                t.append(g.submit_host(hI, hQ, hO[k & 1], n_blocks=NBLK, **kw)[0])
                if k >= 1:
                    g.wait_host(t[k - 1])
            g.wait_host()

        def run_link():
            for k in range(args.calls):
                with torch.cuda.stream(s_up):
                    dI.copy_(torch.from_numpy(hI), non_blocking=True); dQ.copy_(torch.from_numpy(hQ), non_blocking=True)
                with torch.cuda.stream(s_dn):
                    torch.from_numpy(hO[k & 1]).copy_(dO, non_blocking=True)
                    if down is not None:
                        torch.from_numpy(down[k & 1]).copy_(dD, non_blocking=True)
            torch.cuda.synchronize()
        extra = 0.0 if down is None else down[0].nbytes / float(NCH * ns)
        return dict(graph=run_graph, link_bound=run_link, keep=(rx, pp, gr, wf, g), bytes_per_sample=6 + extra)

    cases = {"no_tap": ("none", 0, 0), "tap_power": ("power", 0, 0), "waterfall_k1": ("waterfall", 1, 0),
             "waterfall_k8": ("waterfall", 8, 0), "waterfall_k16": ("waterfall", 16, 0), "waterfall_k8_alternating": ("waterfall", 8, 1)}
    made = {name: make(c) for name, c in cases.items()}
    for m in made.values():  # warm-up
        m["graph"](); m["link_bound"]()
    best = {(n, v): None for n in made for v in ("graph", "link_bound")}
    keys = list(best)
    for rep in range(args.reps):
        order = keys[rep % len(keys):] + keys[:rep % len(keys)]
        for n, v in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            made[n][v]()
            dt = time.perf_counter() - t0
            best[(n, v)] = dt if best[(n, v)] is None else min(best[(n, v)], dt)
    samples = float(NCH) * ns * args.calls
    out = {}
    for n, m in made.items():
        r = dict(link_bytes_per_sample=m["bytes_per_sample"], graph_gsps=samples / best[(n, "graph")] / 1e9,
                 link_bound_gsps=samples / best[(n, "link_bound")] / 1e9)
        r["graph_vs_link_bound"] = r["graph_gsps"] / r["link_bound_gsps"]
        out[n] = r
        m["keep"][4].close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--calls", type=int, default=12)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    import bench
    from bench_block_status import gpu_info
    from audiosdr_b200 import aux
    dev = torch.device("cuda:0")
    I16, Q16, calls = bench.synth_planes(dev, 0, NCH, NBLK * 128, 1234, config_id=2)
    out = dict(tool="tools/bench_waterfall.py", gpu=gpu_info(), version=aux.load_library().sdr_aux_version().decode(),
               channels=NCH, blocks_per_call=NBLK, device=device_cases(args, dev, I16, Q16))
    print(json.dumps(out["device"]), flush=True)
    out["graph"] = graph_cases(args, dev, I16, Q16, calls)
    print(json.dumps(out["graph"]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
