#!/usr/bin/env python3
"""bench.py -- headline benchmark of the batched receiver chain (contract: one JSON line on rank 0).

Workload (BASELINE.json configs[1], the configuration the metric is quoted on, one GPU's worth per rank):
4 096 independent channels in mixed CW_LSB/CW_USB/LSB/USB modes, noise blanker (10 dB) + AGC (medium) + audio
band-pass on, synthetic two-tone / keyed-carrier IF signals with impulse noise.  A "step" is one
sdr_batch_process call advancing every channel by --blocks-per-step 128-sample blocks (state carries from step
to step).  `value` is whole-job channel-samples/s with the float32 I/Q planes already resident in HBM;
`e2e` is the same through sdr_batch_process_host with pinned HOST int16 planes (the reference's audio_block_t
wire format), copies inside the timed region.

  python bench.py [--gpus N --steps K --warmup W]          our CUDA path
  python bench.py ... --dump-outputs DIR                    also save the audio of each workload's last timed step (DIR/config<N>.npy)
  python bench.py --impl reference ...                      the reference's own CPU update() on all host cores
Under torchrun every rank drives its own GPU and its own 4 096 channels (weak scaling); there is no data-path
collective, NCCL only reduces the counters (samples, elapsed time, parity error, status counters).

The JSON line's headline keys are the config-2 workload.  The other BASELINE configurations are timed in the same run and
reported under "workloads": config 3 (65 536 SAM channels, STRONG-scaled: the channels are sharded over the ranks),
config 4 (16 384 channels per GPU, all seven modes, blanker + AGC + ALS) and config 5 (32 768 WSPR channels per GPU),
each with its own ms_per_step, FP32 roofline (with that chain's flop count) and parity probe; "sustained" repeats the
headline workload for a timed region of at least two seconds with the clock record.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "channel_samples_per_s"
UNIT = "Msps"
CHANNELS_PER_GPU = 4096
CONFIG_ID = 2
FLOP_PER_SAMPLE = 364.0     # SURVEY 8a: SSB/CW core 345 + noise blanker 19 (algorithmic flop per channel-sample)
INSTR_PER_SAMPLE = 364.0    # the same operations issued unfused (parity forbids FMA contraction)
# SURVEY 8a cost table per workload (flop = unfused FP32 instructions per channel-sample):
#   config 3: SAM locked 183 (288 while the envelope fallback runs);  config 5: WSPR core 345;
#   config 4: blanker 19 + ALS 152 on top of each mode's chain: SSB/CW/WSPR 516 (5 modes of 7), AM 402, SAM 354 -> mean 476.6
WORKLOADS = {
    2: dict(channels=CHANNELS_PER_GPU, scaling="weak", blocks=256, flop=364.0,
            name="BASELINE configs[1]: 4096 channels/GPU, mixed CW_LSB/CW_USB/LSB/USB, NB(10 dB)+AGC(medium)+audio BPF"),
    3: dict(channels=65536, scaling="strong", blocks=64, flop=183.0,
            name="BASELINE configs[2]: 65536 SAM channels (sharded over the GPUs) with carrier PLL + AGC, +-50 Hz carrier offsets"),
    4: dict(channels=16384, scaling="weak", blocks=64, flop=(5 * 516.0 + 402.0 + 354.0) / 7.0,
            name="BASELINE configs[3]: 16384 channels/GPU, all seven modes mixed per channel, NB + AGC + ALS auto-notch/peak, tone + impulse interference"),
    5: dict(channels=32768, scaling="weak", blocks=64, flop=345.0,
            name="BASELINE configs[4]: 32768 WSPR-mode channels/GPU (262144 over 8 GPUs), BareBonesWSPR setter sequence"),
}
BYTES_PER_SAMPLE = 12.0     # SURVEY 8d: 8 B in (f32 I + f32 Q) + 4 B out per channel-sample
HBM_FALLBACK_GBS = 6650.0
DUMP_BYTES = 32 << 20       # --dump-outputs: the headline step's audio is 512 MB, a fixed sample of its rows is kept
DUMP_BYTES_SIDE = 8 << 20   # the same for each of configs 3, 4 and 5: 56 MB in all


def shard_range(total, rank, world):
    """Contiguous channel range of `rank` (SURVEY 8e)."""
    return total * rank // world, total * (rank + 1) // world


def reduce_counters(sums, maxs, world, device):
    """All-reduce of two small vectors over the ranks (SUM / MAX): the only inter-rank traffic of the whole job."""
    import torch
    import torch.distributed as dist
    if world > 1 and dist.is_initialized():
        t = torch.tensor(list(sums), dtype=torch.float64, device=device if device is not None else "cpu")
        m = torch.tensor(list(maxs), dtype=torch.float64, device=device if device is not None else "cpu")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        dist.all_reduce(m, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()], [float(v) for v in m.tolist()]
    return [float(v) for v in sums], [float(v) for v in maxs]


def gather_counters(samples, ms, world, device):
    """Sum of samples and max of elapsed ms over ranks."""
    s, m = reduce_counters([samples], [ms], world, device)
    return dict(samples=s[0], max_ms=m[0])


def gather_parity(parity, status, world, device):
    """Parity probe and status counters of every rank folded into one record (SURVEY 8e): channels and counters summed,
    max_abs_err is the maximum, bit_exact holds only if it holds on every rank."""
    keys = sorted(status)
    s, m = reduce_counters([parity["channels"], parity["samples"]] + [status[k] for k in keys],
                           [parity["max_abs_err"], 0.0 if parity["bit_exact"] else 1.0], world, device)
    out = dict(channels=int(s[0]), samples=int(s[1]), bit_exact=m[1] == 0.0, max_abs_err=m[0], ranks=world)
    return out, {k: int(v) for k, v in zip(keys, s[2:])}


def pin_to_gpu_numa_node(local):
    """Run this rank on the cores of the NUMA node its GPU hangs off (pinned host planes are then allocated there too)."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else local
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return dict(numa_node=None, note="the platform reports no NUMA node for the GPU")
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return dict(numa_node=node, cpus=len(allowed), nodes=len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")]))
    except Exception as e:
        return dict(numa_node=None, note="not pinned: %s" % e)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": HBM_FALLBACK_GBS}, "fallback"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe).  The timed region is a few tens of
    milliseconds, so the samples come from NVML polled by a thread every ~2 ms; nvidia-smi (one sample per 100 ms at
    best) is the fallback when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.p, self.t, self.stop_flag = index, [], None, None, False
        self.sm, self.mx, self.reasons = [], [], set()

    def _nvml_loop(self, nv, h):
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))); self.mx.append(mx)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.t = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True); self.t.start()
            # the first NVML queries of a process take tens of milliseconds -- longer than a short timed region: wait for the
            # loop to deliver, then start counting from here
            t_end = time.time() + 1.0
            while not self.sm and time.time() < t_end:
                time.sleep(0.001)
            self.pre = (self.sm[-1], self.mx[-1]) if self.sm else None
            self.sm, self.mx = [], []
            return
        except Exception:
            self.t = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.p = None

    def _pump(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.t is not None:
            self.stop_flag = True; self.t.join(timeout=1.0)
            if not self.sm:
                if getattr(self, "pre", None):
                    return {"sm_mhz": self.pre[0], "sm_max_mhz": self.pre[1], "reasons": sorted(self.reasons), "samples": 0,
                            "source": "nvml: no poll fell inside the timed region; the value is the sample taken right before it"}
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "nvml"}
            return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": float(max(self.mx)), "reasons": sorted(self.reasons),
                    "samples": len(self.sm), "source": "nvml, polled every 2 ms inside the timed region"}
        if self.p:
            self.p.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "nvidia-smi"}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


def synth_planes(dev, first_channel, n_channels, n_samples, seed, config_id=CONFIG_ID):
    """IF signals of BASELINE config 2 (headline), 3, 4 or 5, generated on the device (int16 I/Q + setter lists).
    Up to three complex tones per channel (wanted pair or carrier + side band, interferer), optional keying and impulses."""
    import torch
    import signals as S
    f = np.zeros((n_channels, 3)); amp = np.zeros((n_channels, 3)); keyed = np.zeros(n_channels, bool); off = np.full(n_channels, -10**9, np.int64)
    calls = []
    for r in range(n_channels):
        c = first_channel + r
        m = S.channel_mode(config_id, c)
        if config_id == 3 or (config_id == 4 and m in (S.AM, S.SAM)):
            df = 100.0 * S._unit(S.chash(config_id, c, 4)) - 50.0
            f[r, :2] = [6890.0 + df, 6890.0 + df + 1000.0]; amp[r, :2] = [0.3, 0.075]
        elif config_id == 5:
            f[r, 0] = S._audio_to_if(S.WSPR, 1500.0); amp[r, 0] = 0.05
        elif m == S.WSPR:
            f[r, 0] = S._audio_to_if(S.WSPR, 1500.0); amp[r, 0] = 0.2
        elif m in (S.LSB, S.USB):
            f1 = 300.0 + 900.0 * S._unit(S.chash(config_id, c, 2)); f2 = 1300.0 + 1200.0 * S._unit(S.chash(config_id, c, 3))
            f[r, :2] = [S._audio_to_if(m, f1), S._audio_to_if(m, f2)]; amp[r, :2] = [0.2, 0.2]
        else:
            f[r, 0] = S._audio_to_if(m, 700.0); amp[r, 0] = 0.3; keyed[r] = True
        if config_id == 4:  # steady interferer at audio 1 kHz
            f[r, 2] = S._audio_to_if(m, 1000.0); amp[r, 2] = 0.1
        if config_id in (2, 4):
            off[r] = S.chash(config_id, c, 5) % 11025
        calls += [(r,) + tuple(e[2:]) for e in S.channel_events(config_id, c, 0)]
    sigma = 0.05 if config_id == 5 else 0.01
    g = torch.Generator(device=dev); g.manual_seed(seed)
    I = torch.empty((n_channels, n_samples), dtype=torch.int16, device=dev)
    Q = torch.empty_like(I)
    t = torch.arange(n_samples, device=dev, dtype=torch.float64)
    for a in range(0, n_channels, 256):
        z = slice(a, min(a + 256, n_channels))
        fz = torch.tensor(f[z], device=dev); az = torch.tensor(amp[z], device=dev)
        ph0 = 2.0 * np.pi / 44100.0 * fz[:, 0:1] * t[None, :]
        ph1 = 2.0 * np.pi / 44100.0 * fz[:, 1:2] * t[None, :]
        key = torch.where(torch.tensor(keyed[z], device=dev)[:, None], ((t[None, :] // (44100.0 / 40.0)).long() & 1) == 0, True)
        re = az[:, 0:1] * torch.cos(ph0) * key + az[:, 1:2] * torch.cos(ph1)
        im = az[:, 0:1] * torch.sin(ph0) * key + az[:, 1:2] * torch.sin(ph1)
        if config_id == 4:
            ph2 = 2.0 * np.pi / 44100.0 * fz[:, 2:3] * t[None, :]
            re = re + az[:, 2:3] * torch.cos(ph2); im = im + az[:, 2:3] * torch.sin(ph2)
        re = re + sigma * torch.randn(re.shape, generator=g, device=dev, dtype=torch.float64)
        im = im + sigma * torch.randn(im.shape, generator=g, device=dev, dtype=torch.float64)
        burst = ((t[None, :].long() - torch.tensor(off[z], device=dev)[:, None]) % 11025) < 3
        re = torch.where(burst, 0.9, re); im = torch.where(burst, 0.9, im)
        I[z] = torch.round(re.clamp(-1, 1) * 32767.0).to(torch.int16)
        Q[z] = torch.round(im.clamp(-1, 1) * 32767.0).to(torch.int16)
    return I, Q, calls


def cpu_reference_rate(seconds, cores):
    """The reference's own CPU update() (oracle/_ref, unmodified source) or, if absent, the oracle port, on `cores` workers."""
    import signals as S
    from oracle import ref_client as rc
    chans = S.sample_channels(CONFIG_ID, CHANNELS_PER_GPU, max(cores, 8))[:max(cores, 1)]
    I, Q, ev = S.make(CONFIG_ID, chans, 64)
    sample = "%d sampled config-2 channels x 64 blocks streamed round-robin for %.0f s, one channel per worker" % (len(chans), seconds)
    if rc.available():
        r = rc.bench(I, Q, ev, seconds, cores)
        return dict(value=r["sps_update_only"] / 1e6, unit=UNIT, cores=cores, kind="reference", sample=sample,
                    wall_msps=r["sps_wall"] / 1e6)
    from oracle import oracle_lib
    oracle_lib.build()
    reps, total, t0 = 0, 0.0, time.perf_counter()
    Ir, Qr = np.tile(I, (1, 4)), np.tile(Q, (1, 4))
    Ir = np.repeat(Ir, max(1, cores // len(chans) + 1), 0)[:cores]; Qr = np.repeat(Qr, max(1, cores // len(chans) + 1), 0)[:cores]
    evr = []
    for w in range(cores):
        evr += [(w,) + tuple(e[1:]) for e in ev if e[0] == w % len(chans)]
    busy = 0.0
    while time.perf_counter() - t0 < seconds:
        busy += oracle_lib.run(Ir, Qr, evr, threads=cores, want_pcm=False)["seconds"]
        total += Ir.size; reps += 1
    return dict(value=total / busy / 1e6, unit=UNIT, cores=cores, kind="port", sample=sample)


WORKLOAD = WORKLOADS[CONFIG_ID]["name"]


def config_dict(nch, nblk, cfg_id=None, variant=None):
    ns = nblk * 128
    wl = WORKLOADS[cfg_id or CONFIG_ID]["name"]
    if cfg_id not in (None, CONFIG_ID):
        wl = "NOT the headline metric: " + wl
    if variant:
        wl = "DIAGNOSTIC (not the headline): " + wl + " with switches [%s]" % variant
    return dict(workload=wl, channels_per_gpu=nch, blocks_per_step=nblk, samples_per_step=int(nch) * ns,
                planes="float32 channel-major in HBM",
                l2="inputs per step %.0f MB >> 126 MB L2, no flush needed" % (2 * nch * ns * 4 / 1e6),
                parallelism="channels sharded, no collective")


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = 2.0
    vals, t_steps = [], []
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = cpu_reference_rate(per_step, cores)
        if s >= args.warmup:
            vals.append(r["value"]); t_steps.append((time.perf_counter() - t0) * 1e3)
    v = float(np.mean(vals))
    r["value"] = v
    line = dict(metric=METRIC, value=v, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=float(np.mean(t_steps)), higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(config_dict(CHANNELS_PER_GPU, args.blocks_per_step),
                            reference_arm="unmodified reference update() on the host CPU, %d workers, each step = %.0f s of streaming over "
                                          "sampled channels of this workload" % (r["cores"], per_step)),
                cpu_baseline=r, e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def fp32_peaks(lib):
    """FP32 pipe microbenchmarks of the library (MEASURED_PEAKS.json has no FP32 entry): lane-instructions/s."""
    import ctypes as C
    ips = C.c_double(); ms = C.c_float()
    lib.sdrk_fp32_peak.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]
    res = {}
    for kind, name in ((0, "ffma"), (1, "fmul_fadd")):
        if lib.sdrk_fp32_peak(kind, 4096, C.byref(ips), C.byref(ms)) == 0:
            res[name] = ips.value
    return res


def fp32_roofline(peaks32, flop, samples_per_launch, launch_s):
    ach = flop * samples_per_launch / launch_s
    return dict(bound="fp32", achieved=ach / 1e12, peak=2.0 * peaks32["ffma"] / 1e12, unit="TFLOP/s", frac=ach / (2.0 * peaks32["ffma"]),
                peak_source="measured live: dependent-FFMA microbenchmark, 2 flop/instr",
                issue_frac=ach / peaks32["fmul_fadd"], issue_peak_ginstr_s=peaks32["fmul_fadd"] / 1e9,
                note="issue_frac = algorithmic unfused FP32 instructions / measured FMUL+FADD issue rate (parity forbids FMA contraction)",
                algorithmic_flop_per_sample=flop)


class Workload:
    """One BASELINE configuration on this rank's GPU: planes resident in HBM, a configured handle, timing and parity."""

    def __init__(self, cfg_id, rank, world, local, dev, nblk=None, variant=(), contract=False):
        import torch
        import audiosdr_b200 as A
        import signals as S
        w = WORKLOADS[cfg_id]
        self.cfg_id, self.rank, self.world, self.dev = cfg_id, rank, world, dev
        if w["scaling"] == "strong":
            # diagnostics: SDR_BENCH_WORLD=n on one GPU measures the shard rank 0 of n ranks would get (plan choice per shard size)
            emu_world = int(os.environ.get("SDR_BENCH_WORLD", "0") or 0)
            self.first, end = shard_range(w["channels"], rank, emu_world if (emu_world > 0 and world == 1) else world); self.nch = end - self.first
        else:
            self.nch = w["channels"]; self.first = rank * self.nch
        self.nblk = nblk or w["blocks"]; self.ns = self.nblk * 128
        self.I16, self.Q16, calls = synth_planes(dev, self.first, self.nch, self.ns, 0x5D120000 + cfg_id + rank, cfg_id)
        self.If = (self.I16.to(torch.float32) / 32767.0).contiguous(); self.Qf = (self.Q16.to(torch.float32) / 32767.0).contiguous()
        self.out = torch.empty((self.nch, self.ns), dtype=torch.float32, device=dev)
        self.b = A.SdrBatch(self.nch, device=local, contract=contract)
        self.b.configure(calls)
        self.calls = calls
        if "nonb" in variant: self.b.disableNoiseBlanker(None)
        if "noagc" in variant: self.b.disableAGC(None)
        if "noaud" in variant: self.b.disableAudioFilter(None)
        if "als" in variant: self.b.enableALSfilter(None)
        self.variant = variant
        self.stream = torch.cuda.current_stream()
        self.S = S

    def step(self):
        self.b.process(self.If, self.Qf, self.out, n_blocks=self.nblk, stream=self.stream)

    def warm_up(self, n):
        """n untimed steps; after the first one, sampled channels are compared with the oracle and the status getters counted."""
        import torch
        from oracle import oracle_lib
        S = self.S
        picks = sorted(set(S.sample_channels(self.cfg_id, self.nch, 12, n_shards=2)))
        parity = status = None
        for w in range(n):
            self.step()
            if w == 0 and not self.variant:
                torch.cuda.synchronize()
                got = self.out[picks].cpu().numpy()
                hi, hq = self.If[picks].cpu().numpy(), self.Qf[picks].cpu().numpy()
                ev = []
                for row, c in enumerate(picks):
                    ev += S.channel_events(self.cfg_id, self.first + c, row)
                want = oracle_lib.run(hi, hq, ev, threads=os.cpu_count() or 1, want_pcm=False)["audio"]
                fin = np.isfinite(got) & np.isfinite(want)
                parity = dict(channels=len(picks), samples=int(want.size),
                              bit_exact=bool(np.array_equal(got.view(np.uint32), want.view(np.uint32))),
                              max_abs_err=float(np.max(np.abs(got[fin].astype(np.float64) - want[fin]))) if fin.any() else 0.0)
                st = self.b.status()
                status = dict(channels=len(st), sam_locked=sum(int(x.sam_locked) for x in st), agc_active=sum(int(x.agc_active) for x in st),
                              nb_detected=sum(int(x.nb_detected) for x in st))
        torch.cuda.synchronize()
        if parity is not None:
            parity, status = gather_parity(parity, status, self.world, self.dev)
        return parity, status

    def timed(self, steps, barrier):
        """`steps` launches, each between its own CUDA event pair on the launching stream; max over ranks."""
        import torch
        ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        l0 = self.b.launch_count
        barrier()
        ev0[0].record(self.stream)
        for k in range(steps):
            self.step()
            ev0[k + 1].record(self.stream)
        barrier()
        total_ms = ev0[0].elapsed_time(ev0[-1])
        per = [ev0[k].elapsed_time(ev0[k + 1]) for k in range(steps)]
        cnt = gather_counters(float(self.nch) * self.ns * steps, total_ms, self.world, self.dev)
        return dict(value=cnt["samples"] / (cnt["max_ms"] * 1e-3) / 1e6, ms_per_step=cnt["max_ms"] / steps, per_launch_ms=per,
                    launches=int(self.b.launch_count - l0), samples=cnt["samples"])

    def dump(self, path, budget):
        """The audio plane of the last step, as a caller of process() receives it, saved as path/config<N>.npy (float32
        [rows, samples]): the same seeded sample of channel rows in every run, at most `budget` bytes, so that two builds can
        be compared output for output."""
        import torch
        n = min(self.nch, max(1, budget // (4 * self.ns)))
        rows = np.sort(np.random.default_rng(0).choice(self.nch, n, replace=False))
        torch.cuda.synchronize()
        audio = self.out[torch.from_numpy(rows).to(self.dev), :budget // (4 * n)].cpu().numpy()
        os.makedirs(path, exist_ok=True)
        np.save(os.path.join(path, "config%d.npy" % self.cfg_id), audio)

    def free(self):
        import torch
        del self.b, self.I16, self.Q16, self.If, self.Qf, self.out
        torch.cuda.empty_cache()


def side_workload(cfg_id, args, rank, world, local, dev, barrier, peaks32):
    """One of the non-headline BASELINE configurations: device-resident rate, FP32 roofline with its own flop count, parity."""
    w = Workload(cfg_id, rank, world, local, dev)
    parity, status = w.warm_up(3)
    steps = args.steps
    t = w.timed(steps, barrier)
    if args.dump_outputs and rank == 0:
        w.dump(args.dump_outputs, DUMP_BYTES_SIDE)
    launch_s = float(np.mean(t["per_launch_ms"])) * 1e-3
    rec = dict(workload=WORKLOADS[cfg_id]["name"], metric=METRIC, unit=UNIT, value=t["value"], n_gpus=world, scaling=WORKLOADS[cfg_id]["scaling"],
               channels_this_rank=w.nch, blocks_per_step=w.nblk, steps=steps, warmup=3, ms_per_step=t["ms_per_step"], gpu_launches=t["launches"],
               roofline_fp32=fp32_roofline(peaks32, WORKLOADS[cfg_id]["flop"], float(w.nch) * w.ns, launch_s) if peaks32 else None,
               hbm_gbs=BYTES_PER_SAMPLE * float(w.nch) * w.ns / launch_s / 1e9, parity=parity, status=status)
    w.free()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--blocks-per-step", type=int, default=256)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", type=int, default=CONFIG_ID, choices=[2, 3, 4, 5],
                    help="diagnostics only: make BASELINE config 3 / 4 / 5 the line's workload instead of the headline config 2")
    ap.add_argument("--only-headline", action="store_true", help="skip the config 3 / 4 / 5 workloads and the sustained run")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--no-aux", action="store_true", help="skip the bench_aux.py summary (aux_blocks)")
    ap.add_argument("--variant", default="", help="diagnostics only: comma list of nonb,noagc,noaud,als (changes the workload!)")
    ap.add_argument("--role-profile", action="store_true", help="per-stage busy fractions (adds clock reads; not for headline numbers)")
    ap.add_argument("--contract", action="store_true", help="diagnostics only: the opt-in contracting build (not bit-exact) as the line's workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="save the audio of each workload's last timed step as DIR/config<N>.npy "
                                                            "(float32, a fixed sample of channel rows: at most 32 MB for the "
                                                            "line's workload, 8 MB for each of configs 3-5; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves what the CUDA path computed: it needs --impl ours")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import audiosdr_b200 as A
    from audiosdr_b200 import api
    A.build_library()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU path"
    affinity = pin_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = api.load_library()
    cfg_id = args.workload
    diagnostic = cfg_id != CONFIG_ID or bool(args.variant) or args.role_profile or args.contract
    if args.role_profile:
        os.environ["SDR_ROLE_PROFILE"] = "1"
    variant = tuple(v for v in args.variant.split(",") if v)
    W = Workload(cfg_id, rank, world, local, dev, nblk=args.blocks_per_step if cfg_id == CONFIG_ID else None, variant=variant, contract=args.contract)
    nch, nblk, ns, b, I16, Q16 = W.nch, W.nblk, W.ns, W.b, W.I16, W.Q16
    parity, status = W.warm_up(max(args.warmup, 3))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: K launches, each timed with its own CUDA event pair on the launching stream
    clk = ClockSampler(local); clk.start()
    T = W.timed(args.steps, barrier)
    clocks = clk.stop()
    if args.dump_outputs and rank == 0:
        W.dump(args.dump_outputs, DUMP_BYTES)  # before the sustained and e2e runs below advance the same handle
    launches, per_launch_ms, value = T["launches"], T["per_launch_ms"], T["value"]
    role_profile = b.role_profile() if args.role_profile else None  # before the chunked e2e launches dilute the per-launch average

    # ---- the same workload for a timed region of seconds: sustained clocks (config 5 streams for 120 s per channel)
    sustained = None
    if not diagnostic and not args.only_headline and args.sustained_seconds > 0:
        n_sus = max(args.steps, int(np.ceil(args.sustained_seconds * 1e3 / max(T["ms_per_step"], 1e-3))))
        clk2 = ClockSampler(local); clk2.start()
        Ts = W.timed(n_sus, barrier)
        sustained = dict(value=Ts["value"], unit=UNIT, steps=n_sus, ms_per_step=Ts["ms_per_step"], seconds=Ts["ms_per_step"] * n_sus * 1e-3,
                         clocks=clk2.stop())

    # ---- the opt-in contracting build on the same planes: what bit-exactness costs (a second number beside the exact one)
    contracting = None
    if not diagnostic and not args.only_headline:
        try:
            Wc = Workload.__new__(Workload)
            Wc.__dict__.update({k: v for k, v in W.__dict__.items() if k != "b"})
            Wc.b = A.SdrBatch(nch, device=local, contract=True)
            Wc.b.configure(W.calls)
            Wc.out = torch.empty_like(W.out)
            for _ in range(3):
                Wc.step()
            torch.cuda.synchronize()
            Tc = Wc.timed(args.steps, barrier)
            contracting = dict(value=Tc["value"], unit=UNIT, ms_per_step=Tc["ms_per_step"], flag="SDR_BATCH_CONTRACT",
                               note="fused multiply-adds + history-first sums in cascades / Hilbert / NCO; NOT bit-exact: see tests/test_gpu_long.py for the error profile")
            del Wc.b, Wc.out
        except Exception as e:
            contracting = dict(error="%s: %s" % (type(e).__name__, e))

    # ---- end to end through the C ABI with HOST buffers (pinned int16 in, int16 out), copies inside the timed region
    hI = torch.empty((nch, ns), dtype=torch.int16).pin_memory(); hQ = torch.empty_like(hI).pin_memory()
    hO = torch.empty((nch, ns), dtype=torch.int16).pin_memory()
    hI.copy_(I16); hQ.copy_(Q16)
    nI, nQ, nO = hI.numpy(), hQ.numpy(), hO.numpy()
    b.process_host(nI, nQ, nO, n_blocks=nblk)  # warm-up (allocates staging)
    # (a) one synchronous call per step: every call pays its own start-up (first copy-in) and drain (last kernel + copy-out)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.e2e_steps):
        b.process_host(nI, nQ, nO, n_blocks=nblk)
    torch.cuda.synchronize()
    sync_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    scnt = gather_counters(float(nch) * ns * args.e2e_steps, sync_ms, world, dev)
    # (b) the streaming form (the reference's update() is an endless stream of blocks): the steps are submitted back to back
    # and waited for once; every step still copies its own inputs up and its own result down inside the timed region
    b.submit_host(nI, nQ, nO, n_blocks=nblk); b.wait_host()  # warm-up of the streamed form (its chunks are longer: staging grows once)
    hO.zero_()
    barrier()
    t0 = time.perf_counter()
    for k in range(args.e2e_steps):
        b.submit_host(nI, nQ, nO, n_blocks=nblk)
    b.wait_host()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    ecnt = gather_counters(float(nch) * ns * args.e2e_steps, e2e_ms, world, dev)
    e2e = dict(value=ecnt["samples"] / (ecnt["max_ms"] * 1e-3) / 1e6, unit=UNIT, h2d_bytes_per_step=int(2 * nch * ns * 2),
               d2h_bytes_per_step=int(nch * ns * 2), steps=args.e2e_steps, wire_format="int16 in / int16 out, pinned host memory",
               api="sdr_batch_submit_host x steps + sdr_batch_wait_host (streamed calls; host planes copied up and the result copied down every step)",
               per_call_sync=dict(value=scnt["samples"] / (scnt["max_ms"] * 1e-3) / 1e6, unit=UNIT, api="sdr_batch_process_host, one synchronous call per step"),
               result_nonzero=bool(hO[0].any().item() or hO[-1].any().item()))

    # ---- what the host link allows: the same planes copied both ways at once, nothing computed (bounds e2e from above)
    try:
        dI, dQ = torch.empty_like(I16), torch.empty_like(Q16)
        dO = torch.zeros((nch, ns), dtype=torch.int16, device=dev)
        s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        torch.cuda.synchronize()
        best = None
        for rep in range(3):
            barrier()
            t0 = time.perf_counter()
            with torch.cuda.stream(s_up):
                dI.copy_(hI, non_blocking=True); dQ.copy_(hQ, non_blocking=True)
            with torch.cuda.stream(s_dn):
                hO.copy_(dO, non_blocking=True)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        e2e["link_bound"] = dict(value=float(nch) * ns * world / best / 1e6, unit=UNIT, h2d_gbs=4.0 * nch * ns / best / 1e9,
                                 note="both host planes up and one down concurrently with no kernel: the host-link ceiling of e2e per GPU x n_gpus")
        e2e["link_frac"] = e2e["value"] / e2e["link_bound"]["value"]
        del dI, dQ, dO
    except Exception as e:
        e2e["link_bound"] = dict(error=str(e))

    # ---- rooflines of the dominant kernel (sdr_pipeline_kernel: one launch per step)
    peaks, peak_src = measured_peaks()
    launch_s = float(np.mean(per_launch_ms)) * 1e-3
    samples_per_launch = float(nch) * ns
    hbm_gbs = BYTES_PER_SAMPLE * samples_per_launch / launch_s / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch_default_bench")
        except Exception:
            traffic = None
    roofline = dict(bound="hbm", achieved=hbm_gbs, peak=float(peaks["hbm_gbs"]), unit="GB/s", frac=hbm_gbs / float(peaks["hbm_gbs"]),
                    traffic=traffic, peak_source=peak_src + " (MEASURED_PEAKS.json hbm_gbs)" if peak_src == "measured" else "fallback",
                    kernel="sdr_pipeline_kernel", algorithmic_bytes_per_sample=BYTES_PER_SAMPLE,
                    note="BASELINE.json quotes % of HBM roofline; the binding roofline of this chain is the FP32 pipe, see roofline_fp32")
    flop = WORKLOADS[cfg_id]["flop"] + (152.0 if "als" in variant else 0.0) - (19.0 if "nonb" in variant and cfg_id == 2 else 0.0)
    peaks32 = None
    try:
        peaks32 = fp32_peaks(lib)
        fp32 = fp32_roofline(peaks32, flop, samples_per_launch, launch_s)
    except Exception as e:  # the microbenchmark is evidence, not the product
        fp32 = dict(error=str(e)); peaks32 = None

    # ---- free the headline planes, then the other BASELINE configurations (each sized for one GPU)
    del hI, hQ, hO, nI, nQ, nO
    W.free()
    workloads = None
    if not diagnostic and not args.only_headline:
        workloads = {}
        for other in (3, 4, 5):
            try:
                workloads["config%d" % other] = side_workload(other, args, rank, world, local, dev, barrier, peaks32)
            except Exception as e:  # a side workload must not take the headline line down with it
                workloads["config%d" % other] = dict(error="%s: %s" % (type(e).__name__, e))

    # ---- the blocks either side of the chain (SURVEY 8f rows 2-4: I/Q generator, pre-processor, grabber spectrum tap), measured by
    # bench_aux.py in a process of its own and summarised here so that the one line the driver keeps carries them
    aux_blocks = None
    if rank == 0 and world == 1 and not diagnostic and not args.only_headline and not args.no_aux:
        aux_blocks = {}
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "bench_aux.py"), "--no-cpu-baseline", "--steps", str(args.steps),
                                "--warmup", str(args.warmup), "--e2e-steps", "1"],
                               capture_output=True, text=True, timeout=240)
            for ln in r.stdout.splitlines():
                if not ln.startswith("{"):
                    continue
                a = json.loads(ln)
                aux_blocks[a.get("path", "?")] = {k: a.get(k) for k in ("value", "unit", "ms_per_step", "parity", "roofline", "roofline_fp32_issue", "spectra_per_s", "e2e", "gpu_launches") if a.get(k) is not None}
            if not aux_blocks:
                aux_blocks = dict(error=(r.stderr or "no output")[-300:])
        except Exception as e:
            aux_blocks = dict(error="%s: %s" % (type(e).__name__, e))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_rate(args.cpu_seconds, os.cpu_count() or 1)

    if rank == 0:
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=T["ms_per_step"], higher_is_better=True, scaling=WORKLOADS[cfg_id]["scaling"], vs_baseline=None, dtype="f32",
                    data="synthetic",
                    config=config_dict(nch, nblk, cfg_id, args.variant or None),
                    e2e=e2e, gpu_launches=int(launches), clocks=clocks, roofline=roofline, roofline_fp32=fp32, cpu_baseline=cpu,
                    role_profile=role_profile, variant=args.variant or None,
                    diagnostic_workload=(None if cfg_id == CONFIG_ID else "BASELINE configs[%d], %d channels/GPU: NOT the headline metric" % (cfg_id - 1, nch)),
                    parity=parity, status=status, host_affinity=affinity, sustained=sustained, contracting_build=contracting, workloads=workloads,
                    aux_blocks=aux_blocks,
                    per_launch_ms=dict(mean=float(np.mean(per_launch_ms)), min=float(np.min(per_launch_ms)), max=float(np.max(per_launch_ms))))
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
