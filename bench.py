#!/usr/bin/env python
"""bench.py -- channel-samples/s of the fused G.711 decode -> meter -> mix -> encode
path on N B200s (BASELINE.json metric), with its HBM roofline, the end-to-end
number through the C ABI with host buffers, and the CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--cfg4] [--dump-outputs DIR]

One "step" = one pass of the fused kernel over one resident batch of
BASELINE config 3: 4096 channels (1024 bridges x 4 legs) x 1640 frames of
20 ms (1.07 GB of G.711 codes per GPU, >> the 126 MB L2).  N > 1: one rank per
GPU (torchrun), every rank owns its own 1024 bridges (weak scaling, no
collective on the data path); the per-channel event summaries are gathered to
rank 0 over NCCL once, outside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "channel-samples/s G.711 dec+meter+mix+enc"
UNIT = "channel-samples/s"
B, G, F = 1024, 4, 1640                 # bridges, legs per bridge, frames per step (per GPU)
C = B * G
FRAME = 160
# SURVEY.md 8(d): algorithmic bytes per bridge-frame (G=4, 16 B meter record per leg)
BYTES_PER_BF = G * FRAME + 2 * FRAME + FRAME + G * 16      # 1184
WORKLOAD = (f"cfg3: {C} channels ({B} bridges x {G} legs, A-law/u-law alternating) x {F} frames of 20 ms, "
            "noise+tone, gates 2-of-4 open at gain 2.0")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(algorithmic_bytes_per_launch):
    """dram bytes per launch of the fused kernel from the committed ncu capture -- only for the launch shape the
    capture was taken on (same algorithmic bytes per launch); any other shape reports null."""
    p = os.path.join(ROOT, "profiles", "fused_traffic.json")
    if os.path.exists(p):
        try:
            t = json.load(open(p))
            if int(t.get("algorithmic_bytes_per_launch", -1)) == int(algorithmic_bytes_per_launch):
                return t.get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def pin_to_gpu_numa_node(gpu_index):
    """Binds this process to the CPUs NVML reports as local to the GPU, so that the pinned host
    buffers of the e2e leg are allocated (first touch) on the GPU's own NUMA node.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cpus local to gpu {gpu_index}"
    except Exception as e:                      # no NVML / not permitted: keep the default placement
        return f"default ({type(e).__name__})"
    return "default"


def oracle_lib():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_py as O   # bench.py's cpu_baseline / --impl reference legs: the oracle is timed, never shipped
    return O


def seeded_codes_host(nf, ch0=0):
    """The bench workload's input codes for frames [0, nf) generated on the host: the same seeded noise+tone
    family as the GPU arm (synth.pcm_noise_tone), encoded by the oracle (used by --impl reference, which must
    not touch the GPU path; the ours arm hands its own device-generated codes to the CPU leg instead)."""
    import numpy as np
    from igate4xsoftphonedsp_b200 import synth
    O = oracle_lib()
    law = synth.laws(C, ch0)
    codes = np.empty((nf, C, FRAME), np.uint8)
    step = 512
    for c0 in range(0, C, step):
        pcm = synth.pcm_noise_tone(nf, min(step, C - c0), ch0=ch0 + c0)
        for k in range(pcm.shape[1]):
            codes[:, c0 + k] = O.g711_encode(pcm[:, k], int(law[c0 + k]))
    return codes


def cpu_sample(seconds_target=12.0, threads=None, codes=None, gpu_out=None):
    """Times the CPU oracle (reference-faithful scalar port, -O2) with all host threads on a bounded sample of
    the SAME workload: the seeded noise+tone codes and the 2-of-4 gate pattern of the GPU arm (frames [0, nf)).
    codes: host copy of the GPU arm's input codes (ours arm) or None (generated on the host).
    gpu_out: the GPU arm's outputs for the same frames -> the CPU outputs are byte-compared with them.
    Returns (channel-samples/s, cores, description, outputs_equal or None)."""
    import numpy as np
    from igate4xsoftphonedsp_b200 import synth
    O = oracle_lib()
    cores = threads or os.cpu_count() or 1
    law, out_law = synth.laws(C), synth.out_laws(B)
    if codes is None:
        codes = seeded_codes_host(min(F, 256))

    def run(nf, out=None):
        t0 = time.perf_counter()
        res = O.process_batch(codes[:nf], law, synth.gains(nf, B, G), out_law, G, threads=cores, out=out)
        return time.perf_counter() - t0, res

    t, _ = run(8)                                # calibration (also warms the thread pool / pages)
    nf = int(max(8, min(codes.shape[0], 8 * seconds_target / max(t, 1e-6))))
    outs = O.alloc_outputs(nf, C, G)             # pre-faulted output buffers, reused by every pass
    passes, dt = 0, 0.0
    while dt < seconds_target and passes < 4096:   # bounded: repeat the sample until ~seconds_target of CPU work
        d, _ = run(nf, out=outs)
        dt += d
        passes += 1
    equal = None
    if gpu_out is not None:
        equal = bool(np.array_equal(outs[0], gpu_out["mix"][:nf]) and np.array_equal(outs[1], gpu_out["enc"][:nf]) and
                     np.array_equal(outs[2].view(np.uint32).reshape(nf, C, 4)[..., :2],
                                    gpu_out["meter"][:nf].view(np.uint32).reshape(nf, C, 4)[..., :2]) and
                     outs[3].tobytes() == gpu_out["bmeter"][:nf].tobytes())
    return (C * nf * FRAME * passes / dt, cores,
            f"{C} channels x frames [0,{nf}) of the seeded noise+tone workload x {passes} passes, {cores} threads, {dt:.1f} s",
            equal)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference cannot be
    built here (Qt/PJSIP/Boost absent, DESIGN.md) so this is the oracle port, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    desc, cores = "", 1
    codes = seeded_codes_host(min(F, 256))
    for i in range(args.warmup + args.steps):
        v, cores, desc, _ = cpu_sample(seconds_target=max(2.0, 60.0 / max(1, args.warmup + args.steps)), codes=codes)
        if i >= args.warmup:
            vals.append(v)
    value = sum(vals) / len(vals)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8/int16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": desc},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


DUMP_LIMIT = 64 << 20      # bytes of .npy data --dump-outputs writes at most


def dump_frames(F, framed, fixed=()):
    """--dump-outputs: a fixed, seeded sample of frame indices of the per-frame outputs `framed` (tensors with the
    frame on axis 0) small enough that the whole dump stays under DUMP_LIMIT: they and the arrays `fixed` take at
    most 4 bytes of float per byte of output, and 1 MB is set aside for frames.npy and the .npy headers."""
    import numpy as np
    per_frame = 4 * sum(t[0].numel() * t.element_size() for t in framed)
    n = min(F, (DUMP_LIMIT - (1 << 20) - 4 * sum(t.numel() * t.element_size() for t in fixed)) // per_frame)
    if n < 1:
        raise SystemExit("--dump-outputs: one frame of the outputs is larger than the 64 MB dump")
    return np.sort(np.random.default_rng(0).choice(F, size=n, replace=False))


def write_dump(d, arrays):
    """--dump-outputs: d/<name>.npy for every array, d/<name>_<field>.npy for every field of a record array
    (padding fields skipped), in float32 or, for 32- and 64-bit integers, float64: every value exactly."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        fields = [(name, a)] if a.dtype.names is None else \
            [(f"{name}_{f}", a[f]) for f in a.dtype.names if not f.startswith("reserved")]
        for n, v in fields:
            wide = v.dtype.itemsize == 8 or (v.dtype.kind in "iu" and v.dtype.itemsize == 4)
            np.save(os.path.join(d, n + ".npy"), v.astype(np.float64 if wide else np.float32))


def run_chain(args):
    print(json.dumps(measure_chain(args, dump=args.dump_outputs)))


def measure_chain(args, vp=None, dump=None):
    """--chain (and the "chain" object of the default line): SURVEY 8(d) "with RTP" accounting -- raw 180-byte ED-137 packets of every leg in, finished ED-137
    packets of every bridge out, through igd_gateway_process (receive-side walk = liveness + gate arbitration, sender
    walk on a side stream, fused decode -> meter -> mix -> encode -> packet kernel), device resident.
    1284 algorithmic bytes per bridge-frame (4 x 180 in, 180 + 320 + 4 x 16 out).
    dump: directory for --dump-outputs, or None."""
    import numpy as np
    import torch
    import igate4xsoftphonedsp_b200 as ig
    from igate4xsoftphonedsp_b200 import _native as N
    from igate4xsoftphonedsp_b200 import synth
    args.warmup = max(args.warmup, 3)
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    own_vp = vp is None
    if own_vp:
        vp = ig.VoicePath(dev.index)
    vp.use_torch_stream()
    Bc = args.chain_bridges
    Fc = args.chain_frames
    Cc = Bc * G
    law_np, out_law_np = synth.laws(Cc), synth.out_laws(Bc)
    law = torch.from_numpy(law_np).to(dev)
    out_law = torch.from_numpy(out_law_np).to(dev)
    codes = vp.g711_encode(synth.pcm_noise_tone_torch(Fc, Cc, dev), law)
    gate = torch.from_numpy(synth.gates(Fc, Bc, G).reshape(Fc, Cc).astype(np.uint8)).to(dev)
    pk = torch.zeros((Fc, Cc, 180), dtype=torch.uint8, device=dev)
    pk[..., 0] = 0x90
    pk[..., 1] = torch.where(law == 0, 8, 0).to(torch.uint8).view(1, Cc)            # PT 8 = PCMA, 0 = PCMU
    f_idx = torch.arange(Fc, device=dev).view(Fc, 1)
    pk[..., 2] = ((f_idx >> 8) & 255).to(torch.uint8)
    pk[..., 3] = (f_idx & 255).to(torch.uint8)
    pk[..., 12], pk[..., 13], pk[..., 15] = 0x01, 0x67, 0x01
    prio = (1 + torch.arange(Cc, device=dev) % G % 4).view(1, Cc)                   # PTT type = 1 + g % 4 while the gate is open
    pk[..., 16] = (gate.to(torch.int64) * (prio << 5)).to(torch.uint8)              # bits 31-29 of the big-endian word
    pk[..., 20:] = codes
    del codes
    rtp12_np = synth.rtp12(Fc, Bc, np.where(out_law_np == 0, 8, 0).astype(np.uint8))
    rtp12 = torch.from_numpy(rtp12_np).to(dev)
    ctl_np = np.zeros((Fc, Bc), dtype=N.CTL_DT)
    ctl_np["pttstatus"] = 1
    ctl_np["pttpriority"] = 1
    ctl = torch.from_numpy(ctl_np.view(np.int32).reshape(Fc, Bc, 2)).to(dev)
    now0 = 1_000_000
    tx0 = ig.make_state(Bc, now_ms=now0)

    def fresh():
        return (torch.zeros((Cc, 4), dtype=torch.int32, device=dev), torch.zeros((Cc, 2), dtype=torch.int32, device=dev),
                torch.zeros((Bc, 4), dtype=torch.int32, device=dev),
                torch.from_numpy(tx0.copy().view(np.int32).reshape(Bc, 10)).to(dev))

    outs = None
    walk_flags = N.F_WALK_SERIAL if args.serial_walks else 0      # A/B: the thread-per-channel walks

    def step(st, now):
        nonlocal outs
        outs = vp.gateway_process(pk, law, out_law, st[0], st[1], st[2], rtp12, st[3], tx_ctl=ctl, mode=N.ARB_CLIENT_PTT,
                                  now_ms0=now, want=("meter", "bmeter", "mix"), out=outs, flags=walk_flags)

    # ---- parity: a fresh run, two bridges recomputed by the oracle from the raw packets (outside the timed region)
    st = fresh()
    outs = None
    step(st, now0)
    torch.cuda.synchronize()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import rx_arb_cases as R
    import tx_scenarios as T
    O = oracle_lib()
    ok = True
    for b in (0, Bc - 1):
        chs = slice(b * G, b * G + G)
        pkb = pk[:, chs].cpu().numpy()
        szb = np.full((Fc, G), 180, np.uint32)
        ev, _ = R.oracle_rx_walk(pkb, szb, np.ones((Fc, G), np.uint8), now0=now0)
        g, _, _ = R.oracle_arb_walk(np.ascontiguousarray(ev["word"]), G, N.ARB_CLIENT_PTT)
        g = np.where((ev["flags"] & N.RXE_FRAME) == 0, g | N.GAIN_NO_AUDIO, g).astype(np.uint16)
        mix, enc, _, _ = O.process_batch(np.ascontiguousarray(pkb[:, :, 20:]), law_np[chs], g, out_law_np[b:b + 1], G)
        s_ = dict(name="chain", legs=[dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200, slave=None)], F=Fc,
                  ctl=ctl_np[:, b:b + 1], tick_ms=20, now0=now0, payload=enc, rtp12=rtp12_np[:, b:b + 1])
        wpk, wsz, _, _ = T.run_oracle(s_)
        wpk, _ = T.clean_expectation(s_, wpk, wsz)
        ok = ok and np.array_equal(outs["mix"][:, b].cpu().numpy(), mix[:, 0])
        ok = ok and np.array_equal(outs["tx_pkts"][:, b].cpu().numpy(), wpk[:, 0])
        ok = ok and np.array_equal(outs["tx_sizes"][:, b].cpu().numpy().view(np.uint32), wsz[:, 0])
    parity = bool(ok)

    for i in range(args.warmup):
        step(st, now0 + (i + 1) * Fc * 20)
    torch.cuda.synchronize()
    l0 = vp.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step(st, now0 + (args.warmup + i + 1) * Fc * 20)
    e1.record()
    torch.cuda.synchronize()
    launches = vp.launch_count() - l0
    ms = e0.elapsed_time(e1) / args.steps
    if dump:                    # what the last timed step returned and left in the four state arrays
        fs = dump_frames(Fc, list(outs.values()), fixed=st)
        h = {k: v[torch.from_numpy(fs).to(dev)].cpu().numpy() for k, v in outs.items()}
        write_dump(dump, {"frames": fs, "tx_pkts": h["tx_pkts"], "tx_sizes": h["tx_sizes"].view(np.uint32),
                          "meter": h["meter"].view(ig.METER_DT)[..., 0], "bmeter": h["bmeter"].view(ig.BRIDGE_DT),
                          "mix": h["mix"], "rx_state": st[0].cpu().numpy().view(N.RX_STATE_DT)[:, 0],
                          "arb_legs": st[1].cpu().numpy().view(N.ARB_LEG_DT)[:, 0],
                          "arb_bridges": st[2].cpu().numpy().view(N.ARB_BRIDGE_DT)[:, 0],
                          "tx_state": st[3].cpu().numpy().view(N.STATE_DT)[:, 0]})
    sampler = ClockSampler(dev.index)
    sampler.start()
    t_end = time.perf_counter() + 1.5
    k = 0
    while time.perf_counter() < t_end:
        for _ in range(20):
            k += 1
            step(st, now0 + (args.warmup + args.steps + k) * Fc * 20)
        torch.cuda.synchronize()
    clocks = sampler.stop()
    # ---- stage breakdown through the separate entry points (same kernels; the two-kernel pack instead of the fused packet output)
    fields, _ = vp.ed137_parse(pk.view(Fc * Cc, 180), want_payload=False)
    dummy_enc = torch.zeros((Fc, Bc, FRAME), dtype=torch.uint8, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    s2 = fresh()
    for rep in range(args.steps):
        ev[0].record()
        fields, _ = vp.ed137_parse(pk.view(Fc * Cc, 180), want_payload=False)
        ev[1].record()
        events = vp.rx_track(fields.view(Fc, Cc, 4), s2[0], now_ms0=now0 + rep * Fc * 20)
        ev[2].record()
        gain = vp.gate_arbitrate(events, s2[1], s2[2], G, N.ARB_CLIENT_PTT, silence=True)
        ev[3].record()
        vp.ed137_pack(rtp12, dummy_enc, s2[3], ctl, now_ms0=now0 + rep * Fc * 20)
        ev[4].record()
        torch.cuda.synchronize()
    stage = {"fields": ev[0].elapsed_time(ev[1]), "rx_track": ev[1].elapsed_time(ev[2]), "gate_arbitrate": ev[2].elapsed_time(ev[3]),
             "plan+assemble (separate call; the gateway runs the plan walk only)": ev[3].elapsed_time(ev[4])}
    # ---- end to end: the same call with pinned HOST buffers -- packets, RTP headers and setter values copied in, the
    # finished packets, their sizes and the meter records copied out, the four state arrays round-tripped, every step
    e2e = None
    if not args.no_e2e:
        affinity0 = os.sched_getaffinity(0)
        numa = pin_to_gpu_numa_node(dev.index)

        def pinned(t):
            h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            h.copy_(t)
            return h

        h_pk, h_rtp, h_ctl = pinned(pk), pinned(rtp12), pinned(ctl)
        h_out_t = {"tx_pkts": torch.empty((Fc, Bc, 180), dtype=torch.uint8, pin_memory=True),
                   "tx_sizes": torch.empty((Fc, Bc), dtype=torch.int32, pin_memory=True),
                   "meter": torch.empty((Fc, Cc, 4), dtype=torch.int32, pin_memory=True),
                   "bmeter": torch.empty((Fc, Bc), dtype=torch.int32, pin_memory=True)}
        for t in h_out_t.values():
            t.zero_()
        os.sched_setaffinity(0, affinity0)
        h_out = {"tx_pkts": h_out_t["tx_pkts"].numpy(), "tx_sizes": h_out_t["tx_sizes"].numpy().view(np.uint32),
                 "meter": h_out_t["meter"].numpy().view(ig.METER_DT).reshape(Fc, Cc),
                 "bmeter": h_out_t["bmeter"].numpy().view(ig.BRIDGE_DT).reshape(Fc, Bc)}
        h_state = (np.zeros(Cc, N.RX_STATE_DT), np.zeros(Cc, N.ARB_LEG_DT), np.zeros(Bc, N.ARB_BRIDGE_DT), tx0.copy())
        h_ctl_np = h_ctl.numpy().view(N.CTL_DT).reshape(Fc, Bc)

        def host_step(now):
            vp.gateway_process(h_pk.numpy(), law_np, out_law_np, h_state[0], h_state[1], h_state[2], h_rtp.numpy(), h_state[3],
                               tx_ctl=h_ctl_np, mode=N.ARB_CLIENT_PTT, now_ms0=now, want=("meter", "bmeter"), out=h_out, flags=walk_flags)

        host_step(now0)                         # a fresh run from the same start state as the device-resident parity run
        st_d = fresh()
        outs = None
        step(st_d, now0)
        torch.cuda.synchronize()
        ok_e2e = bool(torch.equal(h_out_t["tx_pkts"], outs["tx_pkts"].cpu()) and torch.equal(h_out_t["bmeter"], outs["bmeter"].cpu()))
        esteps = args.steps
        host_step(now0 + Fc * 20)
        t0 = time.perf_counter()
        for i in range(esteps):
            host_step(now0 + (i + 2) * Fc * 20)
        dt = time.perf_counter() - t0
        h2d = h_pk.numel() + h_rtp.numel() + h_ctl.numel() * 4 + law_np.nbytes + out_law_np.nbytes + sum(a.nbytes for a in h_state)
        d2h = sum(v.nbytes for v in h_out.values()) + sum(a.nbytes for a in h_state)
        e2e = {"value": Cc * Fc * FRAME * esteps / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "steps": esteps, "outputs": ["tx_pkts", "tx_sizes", "meter", "bmeter", "state arrays"], "matches_device_path": ok_e2e,
               "host_buffers": numa, "note": "PCIe-bound on the packets in (h2d_bytes_per_step)"}
    alg = 1284 * Bc * Fc
    peak, peak_src = peaks()
    value = Cc * Fc * FRAME / (ms * 1e-3)
    if own_vp:
        vp.close()
    return ({
        "metric": METRIC + " (packets in -> packets out)", "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/int16", "data": "synthetic",
        "config": {"workload": f"chain: {Cc} channels ({Bc} bridges x {G} legs) x {Fc} ticks, raw 180-byte ED-137 packets of every leg in, "
                               f"one finished ED-137 packet per bridge and tick out (igd_gateway_process, CLIENT arbitration, silence marking)",
                   "l2": "inputs larger than L2" if Cc * Fc * 180 > (256 << 20) else "inputs may be L2 resident"},
        "roofline": {"bound": "hbm", "achieved": alg / ms / 1e6, "peak": peak, "unit": "GB/s", "frac": alg / ms / 1e6 / peak,
                     "traffic": None, "kernel": ("igd_gateway_process: k_rx_track<packets> + k_gate_arbitrate + k_ed137_plan (side stream) + "
                                if args.serial_walks else "igd_gateway_process: k_rxarb_walk (liveness walk + arbitration, warp per bridge, "
                                "ticks across the lanes) + k_plan_walk (side stream) + " if Cc < 65536 and Fc >= 8 else
                                "igd_gateway_process: k_rxarb_bridge (liveness walk + arbitration, one thread per bridge) + sender walk (side stream) + ") + "k_fused_q<4, packets in, packets out>", "peak_source": peak_src,
                     "algorithmic_bytes_per_step": alg, "bytes_per_bridge_frame": 1284, "stage_ms": stage},
        "cpu_baseline": None, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "parity_vs_oracle_on_two_bridges": parity,
    })


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=F, help="frames per step (default: the config-3 value)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer end-to-end leg")
    ap.add_argument("--cfg4", action="store_true",
                    help="BASELINE config 4 instead of config 3: 1 M channel-seconds (1024 bridges x 4 legs x 12207 frames "
                         "= 5.0e7 channel-frames) as ONE fixed job whose bridges are split over the ranks (strong scaling); "
                         "device-resident legs only")
    ap.add_argument("--cfg5", action="store_true",
                    help="BASELINE config 5: one mixed-codec batch of 65536 channels (16384 bridges x 4 legs, A-law / u-law "
                         "alternating) x 100 frames, bridges split over the ranks (strong scaling), per-channel dBFS "
                         "summaries gathered to rank 0 over NCCL and checked against the oracle; device-resident legs only")
    ap.add_argument("--chain", action="store_true", help="packets in -> packets out (SURVEY 8d 'with RTP' accounting, 1284 B per "
                    "bridge-frame) through igd_gateway_process, device resident, 1 GPU")
    ap.add_argument("--no-chain", action="store_true", help="skip the packets-in -> packets-out measurement of the default line")
    ap.add_argument("--serial-walks", action="store_true", help="--chain: IGD_F_WALK_SERIAL, the thread-per-channel walks (A/B)")
    ap.add_argument("--chain-bridges", type=int, default=B)
    ap.add_argument("--chain-frames", type=int, default=F)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's outputs; a fixed, seeded "
                         "sample of frames, at most 64 MB) to DIR/<name>.npy as float32 / float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.chain:
        return run_chain(args)
    if args.cfg5:
        world_ = int(os.environ.get("WORLD_SIZE", "1"))
        if 16384 % world_:
            raise SystemExit("--cfg5 needs a rank count that divides 16384 bridges")
        globals()["B"] = 16384 // world_
        globals()["C"] = globals()["B"] * G
        globals()["F"] = 100
        globals()["WORKLOAD"] = (f"cfg5: mixed-codec batch of 65536 channels (16384 bridges x {G} legs, A-law/u-law alternating) x 100 "
                                 f"frames of 20 ms, bridges split over {world_} rank(s) ({globals()['B']} bridges each), noise+tone, "
                                 "gates 2-of-4 open at gain 2.0, per-channel summaries gathered to rank 0")
        args.no_e2e = args.no_cpu = True
    if args.cfg4:
        world_ = int(os.environ.get("WORLD_SIZE", "1"))
        if 1024 % world_:
            raise SystemExit("--cfg4 needs a rank count that divides 1024 bridges")
        globals()["B"] = 1024 // world_
        globals()["C"] = globals()["B"] * G
        globals()["F"] = 12207
        globals()["WORKLOAD"] = (f"cfg4: 1 M channel-seconds = 4096 channels (1024 bridges x {G} legs) x 12207 frames of 20 ms, "
                                 f"bridges split over {world_} rank(s) ({globals()['B']} bridges each), noise+tone, gates 2-of-4 open at gain 2.0")
        args.no_e2e = args.no_cpu = True
    if not args.cfg4 and not args.cfg5 and args.frames != F:
        globals()["F"] = args.frames
        globals()["WORKLOAD"] = WORKLOAD.replace("x 1640 frames", f"x {args.frames} frames (non-default)")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import torch.distributed as dist
    import igate4xsoftphonedsp_b200 as ig
    from igate4xsoftphonedsp_b200 import sharding, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    vp = ig.VoicePath(local)                    # raises if libigate_dsp.so / an sm_100 GPU is missing
    vp.use_torch_stream()
    # ---- resident inputs: this rank's bridges [rank*B, (rank+1)*B) of a world*B-bridge system
    ch0 = rank * C
    law = torch.from_numpy(synth.laws(C, ch0)).to(dev)
    out_law = torch.from_numpy(synth.out_laws(B, rank * B)).to(dev)
    gain_np = synth.gains(F, B, G)
    gain = torch.from_numpy(gain_np.view(np.int16)).to(dev)
    pcm = synth.pcm_noise_tone_torch(F, C, dev, ch0=ch0)
    codes = vp.g711_encode(pcm, law)            # inputs are G.711 codes, produced by the GPU encoder
    del pcm
    out = vp.alloc_outputs(F, B, G)
    torch.cuda.synchronize()

    def step():
        vp.process_batch(codes, law, gain, out_law, G, out=out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    l0 = vp.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for i in range(args.steps):
        step()
        ev[i + 1].record()
    barrier()
    launches = vp.launch_count() - l0
    total_ms = ev[0].elapsed_time(ev[-1])
    if args.dump_outputs and rank == 0:
        fs = dump_frames(F, list(out.values()))
        h = {k: v[torch.from_numpy(fs).to(dev)].cpu().numpy() for k, v in out.items()}
        write_dump(args.dump_outputs, {"frames": fs, "mix": h["mix"], "enc": h["enc"],
                                       "meter": h["meter"].view(ig.METER_DT)[..., 0], "bmeter": h["bmeter"].view(ig.BRIDGE_DT)})
    # clocks / throttle reasons under the same load: the K timed steps last only milliseconds, so the
    # nvidia-smi sampler (100 ms period) runs over a ~1.5 s loop of the identical kernel right after them
    clocks = None
    if rank == 0:
        sampler = ClockSampler(local)
        sampler.start()
    t_end = time.perf_counter() + 1.5
    while time.perf_counter() < t_end:
        for _ in range(50):
            step()
        torch.cuda.synchronize()
    if rank == 0:
        clocks = sampler.stop()
    per_launch_ms = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps))
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    samples_per_step = world * C * F * FRAME
    value = samples_per_step * args.steps / (total_ms_max * 1e-3)

    # ---- roofline of the dominant (only) kernel: algorithmic bytes / avg launch duration
    peak, peak_src = peaks()
    avg_launch_s = (total_ms / args.steps) * 1e-3
    achieved = BYTES_PER_BF * B * F / avg_launch_s / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(BYTES_PER_BF * B * F), "kernel": "k_fused_q<G=4, 24 autonomous warps/SM, 8 bridge-frames per per-warp TMA slot, 4 lanes per bridge-frame>", "peak_source": peak_src,
                "algorithmic_bytes_per_launch": BYTES_PER_BF * B * F,
                "launch_ms": {"avg": total_ms / args.steps, "min": per_launch_ms[0], "max": per_launch_ms[-1]}}

    # ---- parity spot check on the timed outputs (oracle as checker, outside the timed region)
    parity, parity_frames = None, 0
    if rank == 0:
        O = oracle_lib()
        fs = sorted({0, F - 1} | {int(x) for x in np.random.default_rng(args.steps).choice(F, size=min(F, 64), replace=False)})
        sel = torch.tensor(fs, device=dev)
        want = O.process_batch(codes[sel].cpu().numpy(), law.cpu().numpy(), gain_np[fs], out_law.cpu().numpy(), G,
                               threads=os.cpu_count() or 1)
        parity = bool(np.array_equal(out["mix"][sel].cpu().numpy(), want[0]) and
                      np.array_equal(out["enc"][sel].cpu().numpy(), want[1]) and
                      np.array_equal(out["meter"][sel].cpu().numpy().view(np.uint32)[..., :2].reshape(len(fs), C, 2),
                                     want[2].view(np.uint32).reshape(len(fs), C, 4)[..., :2]) and
                      out["bmeter"][sel].cpu().numpy().tobytes() == want[3].tobytes())
        parity_frames = len(fs)

    # ---- per-channel summaries gathered to rank 0 (the only collective; outside the timed region)
    summ, _ = vp.event_summary(out["meter"], gain, want_db=False)
    torch.cuda.synchronize()
    gathered = sharding.gather_records(summ, world * B, G) if world > 1 else summ
    n_summaries = int(gathered.shape[0]) if rank == 0 else None
    # content check of the gathered records ON HARDWARE: rank 0 regenerates two bridges of EVERY rank from the seed
    # (GPU encoder for the codes, as the ranks did), runs the oracle on them and compares the records that came
    # over NCCL bit for bit
    summaries_parity = None
    if rank == 0:
        O = oracle_lib()
        gath = gathered.cpu().numpy().view(np.uint8).reshape(-1, 32).copy().view(O.SUMMARY_DT).reshape(-1)
        ok = True
        for r in range(world):
            for b_off in (0, B - 1):
                chs = (r * B + b_off) * G
                p_ = synth.pcm_noise_tone_torch(F, G, dev, ch0=chs)
                lw = synth.laws(G, chs)
                cd = vp.g711_encode(p_, torch.from_numpy(lw).to(dev)).cpu().numpy()
                gn = synth.gains(F, 1, G)
                _, _, mt, _ = O.process_batch(cd, lw, gn, synth.out_laws(1, r * B + b_off), G)
                want_s = O.event_summary(mt, gn)
                ok = ok and gath[chs:chs + G].tobytes() == want_s.tobytes()
        summaries_parity = bool(ok)

    # ---- end to end through the C ABI with HOST buffers (pinned), H2D + kernel + D2H every step.
    # Headline form: what a gateway takes back -- the encoded bridge output (packet payloads), the per-leg meter
    # records and the bridge records; the int16 mix stays on the device (igd_batch_desc.mix = NULL).  The form with
    # every output, r01's, is reported beside it.
    e2e = None
    h_codes = None
    if not args.no_e2e:
        affinity0 = os.sched_getaffinity(0)
        numa = pin_to_gpu_numa_node(local)      # the pinned buffers are first-touched on the GPU's own NUMA node
        h_codes = torch.empty((F, C, FRAME), dtype=torch.uint8, pin_memory=True)
        h_codes.copy_(codes)
        h_in = {"codes": h_codes.numpy(), "law": law.cpu().numpy(), "gain": gain_np, "out_law": out_law.cpu().numpy()}
        h_out_t = {"mix": torch.empty((F, B, FRAME), dtype=torch.int16, pin_memory=True),
                   "enc": torch.empty((F, B, FRAME), dtype=torch.uint8, pin_memory=True),
                   "meter": torch.empty((F, C, 4), dtype=torch.int32, pin_memory=True),
                   "bmeter": torch.empty((F, B), dtype=torch.int32, pin_memory=True)}
        h_out = {"mix": h_out_t["mix"].numpy(), "enc": h_out_t["enc"].numpy(),
                 "meter": h_out_t["meter"].numpy().view(ig.METER_DT).reshape(F, C),
                 "bmeter": h_out_t["bmeter"].numpy().view(ig.BRIDGE_DT).reshape(F, B)}
        for t in h_out_t.values():
            t.zero_()                           # first touch while bound
        os.sched_setaffinity(0, affinity0)      # the CPU legs below use every host core again
        esteps = args.steps
        h2d = h_in["codes"].nbytes + h_in["gain"].nbytes + h_in["law"].nbytes + h_in["out_law"].nbytes

        def e2e_leg(names):
            o = {k: h_out[k] for k in names}
            for _ in range(2):
                vp.process_batch(h_in["codes"], h_in["law"], h_in["gain"], h_in["out_law"], G, out=o)
            barrier()
            t0 = time.perf_counter()
            for _ in range(esteps):
                vp.process_batch(h_in["codes"], h_in["law"], h_in["gain"], h_in["out_law"], G, out=o)
            barrier()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            return samples_per_step * esteps / float(dt.item()), sum(v.nbytes for v in o.values())

        v_all, d2h_all = e2e_leg(("mix", "enc", "meter", "bmeter"))
        ok_all = bool(torch.equal(h_out_t["mix"], out["mix"].cpu()) and torch.equal(h_out_t["enc"], out["enc"].cpu()))
        for k in ("enc", "meter", "bmeter"):
            h_out_t[k].zero_()
        v_gw, d2h_gw = e2e_leg(("enc", "meter", "bmeter"))
        ok_gw = bool(torch.equal(h_out_t["enc"], out["enc"].cpu()) and torch.equal(h_out_t["meter"], out["meter"].cpu()) and
                     torch.equal(h_out_t["bmeter"], out["bmeter"].cpu()))
        e2e = {"value": v_gw, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_gw, "steps": esteps,
               "outputs": ["enc", "meter", "bmeter"], "matches_device_path": ok_gw, "host_buffers": numa,
               "all_outputs": {"value": v_all, "d2h_bytes_per_step": d2h_all, "outputs": ["mix", "enc", "meter", "bmeter"],
                               "matches_device_path": ok_all},
               "note": "PCIe-bound: the input codes alone are h2d_bytes_per_step; profiles/tools/pcie_probe.py gives the box's copy rates"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # same inputs as the GPU arm (its own device-generated codes, copied to the host), outputs byte-compared
        host_codes = h_codes.numpy() if h_codes is not None else codes.cpu().numpy()
        gpu_out = {"mix": out["mix"].cpu().numpy(), "enc": out["enc"].cpu().numpy(),
                   "meter": out["meter"].cpu().numpy(), "bmeter": out["bmeter"].cpu().numpy()}
        v, cores, desc, equal = cpu_sample(codes=host_codes, gpu_out=gpu_out)
        v1, _, desc1, _ = cpu_sample(seconds_target=3.0, threads=1, codes=host_codes)   # SURVEY 8(d): also the single-thread figure
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc,
               "outputs_equal_gpu": equal, "single_thread": {"value": v1, "sample": desc1}}

    # ---- the same hot path with its callers on either side (SURVEY 8d "with RTP"): packets in -> packets out through
    # igd_gateway_process at the bench shape, device resident -- a compact copy of what `--chain` prints in full
    chain = None
    if rank == 0 and world == 1 and not (args.cfg4 or args.cfg5 or args.no_chain) and args.frames == 1640:
        import copy
        a2 = copy.copy(args)
        a2.no_e2e, a2.steps, a2.warmup, a2.serial_walks, a2.chain_bridges, a2.chain_frames = True, args.steps, 3, False, B, F
        try:
            full = measure_chain(a2, vp=vp)
            chain = {"workload": full["config"]["workload"], "value": full["value"], "unit": full["unit"],
                     "ms_per_step": full["ms_per_step"], "vs_fused_kernel_ms": full["ms_per_step"] / (total_ms / args.steps),
                     "roofline": {k: full["roofline"][k] for k in ("bound", "achieved", "peak", "unit", "frac", "bytes_per_bridge_frame", "kernel")},
                     "gpu_launches_per_step": full["gpu_launches"] // a2.steps,
                     "parity_vs_oracle_on_two_bridges": full["parity_vs_oracle_on_two_bridges"]}
        except Exception as e:      # the headline line must not depend on the extra measurement
            chain = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong" if (args.cfg4 or args.cfg5) else "weak", "vs_baseline": None, "dtype": "u8/int16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "per_gpu_codes_bytes": C * F * FRAME, "l2": "inputs larger than L2",
                       "parallelism": f"bridges sharded over {world} GPU(s), no data-path collective",
                       "summaries_gathered_to_rank0": n_summaries, "summaries_parity_vs_oracle": summaries_parity,
                       "parity_frames_checked": parity_frames},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clocks, "parity_vs_oracle_on_timed_output": parity, "chain": chain,
        }))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    vp.close()


if __name__ == "__main__":
    main()
