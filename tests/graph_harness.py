"""tests/graph_harness.py -- one deterministic sequence of receiver-graph calls, run two ways: through the streamed graph
(audiosdr_b200.graph, host planes) and as the composition of the blocks' device calls on torch tensors (the definition the
graph must equal bit for bit).

Workload: config 4's receiver mix (all seven modes, blanker, AGC, ALS), a pre-processor whose detector runs on a third of
the channels with correction -1 / +1 and swap on others (or an I/Q generator with gain balances, or no front), the grabber
tap, call lengths 1, 2, 3, 16, 17, 64 and 255 blocks on shuffled subsets alternating with calls on every channel, audio
alternating int16 / float32, and setters on every member between two calls."""
import numpy as np

import aux_signals as AS
import signals as S
from audiosdr_b200 import api, aux
from audiosdr_b200 import graph as G

N_BLOCK = 128
LENGTHS = [1, 2, 3, 16, 17, 64, 255]
POWER_SENTINEL, SNAP_SENTINEL = -7.0, 0x2A2A


def plan(n, lengths=LENGTHS, seed=5):
    """[(ids uint32 array | None, n_blocks, out dtype)]: a shuffled subset, then a call on every channel, per length."""
    rng = np.random.default_rng(seed)
    calls = []
    for k, nb in enumerate(lengths):
        ids = rng.permutation(n)[:max(1, n // 2 + 3 * k)].astype(np.uint32)
        calls.append((ids, nb, np.int16 if k % 2 == 0 else np.float32))
        calls.append((None, lengths[(k + 3) % len(lengths)], np.float32 if k % 2 == 0 else np.int16))
    return calls


def inputs(front, n, calls):
    """The input planes of the whole sequence, int16 [n, 128 * total blocks]: (I, Q), or (X, None) for the generator."""
    total = sum(nb for _, nb, _ in calls)
    if front == "gen":
        return AS.iq_case(n, total), None
    I, Q, _ = S.make(4, list(range(n)), total)
    return I, Q


def make_handles(front, n, grabber=True):
    rx = api.SdrBatch(n)
    rx.configure([(c,) + tuple(e[2:]) for c in range(n) for e in S.channel_events(4, c, c)])
    h = {"rx": rx, "pp": None, "gen": None, "gr": aux.GrabberBatch(n) if grabber else None}
    if front == "pp":
        pp = h["pp"] = aux.PreProcessorBatch(n)
        pp.startAutoI2SerrorDetection([c for c in range(n) if c % 3 == 0])
        pp.setI2SerrorCompensation([c for c in range(n) if c % 3 == 1], -1)
        pp.setI2SerrorCompensation([c for c in range(n) if c % 3 == 2], 1)
        pp.swapIQ([c for c in range(n) if c % 5 == 2], True)
    elif front == "gen":
        gen = h["gen"] = aux.IQGeneratorBatch(n)
        for c in range(n):
            if c % 3 == 1:
                gen.setGainBalance(c, 1.0 + 0.01 * (c % 10 + 1))
    return h


def setters_between(h, j):
    """Setters on every member before call j (j >= 1): they take effect at that block boundary."""
    if j == 3:
        h["rx"].setDemodMode([3, 10], S.SAM)
        h["rx"].setAGCmode(7, api.AGC_FAST)
        if h["pp"] is not None:
            h["pp"].setI2SerrorCompensation([4, 5], 1)
            h["pp"].startAutoI2SerrorDetection([1])
        if h["gen"] is not None:
            h["gen"].setGainBalance([5, 6], 0.95)
    if j == 8:
        h["rx"].disableNoiseBlanker([0, 1, 2])
        if h["pp"] is not None:
            h["pp"].swapIQ([0, 9], True)


def _alloc(shape, dtype, pinned, fill=0):
    if pinned:
        import torch
        a = torch.empty(shape, dtype={np.int16: torch.int16, np.float32: torch.float32, np.uint32: torch.int32, np.int32: torch.int32}[dtype],
                        pin_memory=True).numpy()
        a = a.view(dtype)
    else:
        a = np.empty(shape, dtype)
    a[...] = fill
    return a


def run_graph(h, calls, I, Q, in_flight=3, pinned=True, want=("rx_status", "pp_status", "power", "snapshots")):
    """Submits the sequence through a GraphBatch over the handles h with up to `in_flight` calls queued; returns one dict
    of outputs per call."""
    g = G.GraphBatch(h["rx"], preproc=h["pp"], iqgen=h["gen"], grabber=h["gr"])
    res, tickets, pos = [], [], 0
    for j, (ids, nb, dt) in enumerate(calls):
        if j:
            setters_between(h, j)
        rows = h["rx"].n_channels if ids is None else len(ids)
        sel = slice(None) if ids is None else ids.astype(np.int64)
        ns, S_ = nb * N_BLOCK, (nb + 1) // 2
        # inputs with a wider pitch than the call: 8 spare samples per row
        hI = _alloc((rows, ns + 8), np.int16, pinned)
        hI[:, :ns] = I[sel, pos * N_BLOCK:pos * N_BLOCK + ns]
        hQ = None
        if Q is not None:
            hQ = _alloc((rows, ns + 8), np.int16, pinned)
            hQ[:, :ns] = Q[sel, pos * N_BLOCK:pos * N_BLOCK + ns]
        o = {"audio": _alloc((rows, ns), dt, pinned)}
        kw = {}
        if "rx_status" in want:
            o["rx_status"] = kw["block_status"] = _alloc((nb, api.BS_FIELDS, rows), np.uint32, pinned)
        if h["pp"] is not None and "pp_status" in want:
            o["pp_status"] = kw["pp_block_status"] = _alloc((nb, aux.PP_BS_FIELDS, rows), np.int32, pinned)
        if h["gr"] is not None:
            if "power" in want:
                o["power"] = kw["power"] = _alloc((rows, S_, 256), np.float32, pinned, POWER_SENTINEL)
            if "snapshots" in want:
                o["snapshots"] = kw["snapshots"] = _alloc((rows, S_, 512), np.int16, pinned, SNAP_SENTINEL)
        t, counts = g.submit_host(hI[:, :ns], None if hQ is None else hQ[:, :ns], o["audio"], n_blocks=nb, channels=ids, **kw)
        if counts is not None:
            o["counts"] = counts
        o["_keep"] = (hI, hQ)
        res.append(o)
        tickets.append(t)
        if len(tickets) >= in_flight:
            g.wait_host(tickets[-in_flight])
        pos += nb
    g.wait_host()
    g.close()
    for o in res:
        del o["_keep"]
    return res


def run_device(h, calls, I, Q, want=("rx_status", "pp_status", "power", "snapshots")):
    """The same sequence as the composition of the blocks' device calls on torch tensors (current stream)."""
    import torch
    dev = torch.device("cuda:0")
    td = {np.int16: torch.int16, np.float32: torch.float32}
    res, pos = [], 0
    for j, (ids, nb, dt) in enumerate(calls):
        if j:
            setters_between(h, j)
        rows = h["rx"].n_channels if ids is None else len(ids)
        sel = slice(None) if ids is None else ids.astype(np.int64)
        ns, S_ = nb * N_BLOCK, (nb + 1) // 2
        dI = torch.from_numpy(np.ascontiguousarray(I[sel, pos * N_BLOCK:pos * N_BLOCK + ns])).to(dev)
        dQ = None if Q is None else torch.from_numpy(np.ascontiguousarray(Q[sel, pos * N_BLOCK:pos * N_BLOCK + ns])).to(dev)
        o = {}
        if h["pp"] is not None:
            mI, mQ = torch.empty_like(dI), torch.empty_like(dI)
            rec = torch.zeros((nb, aux.PP_BS_FIELDS, rows), dtype=torch.int32, device=dev) if "pp_status" in want else None
            h["pp"].process(dI, dQ, mI, mQ, n_blocks=nb, channels=ids, block_status=rec)
            if rec is not None:
                o["pp_status"] = rec
        elif h["gen"] is not None:
            mI, mQ = torch.empty_like(dI), torch.empty_like(dI)
            h["gen"].process(dI, mI, mQ, n_blocks=nb, channels=ids)
        else:
            mI, mQ = dI, dQ
        if h["gr"] is not None:
            pw = torch.full((rows, S_, 256), POWER_SENTINEL, dtype=torch.float32, device=dev) if "power" in want else None
            sn = torch.full((rows, S_, 512), SNAP_SENTINEL, dtype=torch.int16, device=dev) if "snapshots" in want else None
            o["counts"] = h["gr"].process(mI, mQ, n_blocks=nb, channels=ids, snapshots=sn, power=pw)
            if pw is not None:
                o["power"] = pw
            if sn is not None:
                o["snapshots"] = sn
        audio = torch.empty((rows, ns), dtype=td[dt], device=dev)
        rrec = torch.zeros((nb, api.BS_FIELDS, rows), dtype=torch.int32, device=dev) if "rx_status" in want else None
        h["rx"].process(mI, mQ, audio, n_blocks=nb, channels=ids, block_status=rrec)
        o["audio"] = audio
        if rrec is not None:
            o["rx_status"] = rrec
        res.append(o)
        pos += nb
    torch.cuda.synchronize()
    return [{k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in o.items()} for o in res]


def states(h):
    """Every member's export_state blobs.  The grabber's carried block (bytes 16..527 of its blob) is state only while a pair
    is open (phase byte 8 == 1): a call that closes the pair leaves whatever the last open pair carried, so a call cut into
    chunks leaves other bytes there than the whole call.  They are never read; they are zeroed here."""
    out = {k: v.export_state() for k, v in h.items() if v is not None}
    if "gr" in out:
        out["gr"][out["gr"][:, 8] == 0, 16:16 + 512] = 0
    return out


def mismatches(got, want):
    """[(call, output)] that differ in any bit (outputs compared as raw bytes)."""
    bad = []
    assert len(got) == len(want)
    for j, (a, b) in enumerate(zip(got, want)):
        if set(a) != set(b):
            bad.append((j, "keys %s vs %s" % (sorted(a), sorted(b))))
            continue
        for k in a:
            x, y = np.ascontiguousarray(a[k]), np.ascontiguousarray(b[k])
            if x.shape != y.shape or x.tobytes() != y.tobytes():
                bad.append((j, k))
    return bad
