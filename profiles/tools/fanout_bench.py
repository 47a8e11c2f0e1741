#!/usr/bin/env python
"""Gateway fan-out (igd_gateway_fanout): one PCM frame per bridge and tick in, a finished ED-137 packet for every leg
out.  Device-resident buffers; per shape: ms per call of the fan-out, of its assembly kernel (k_fanout_tile) alone and
of the composed path it replaces (igd_g711_encode_ch over the replicated PCM, prepared outside the timed region, then
igd_ed137_pack), the two forms alternated call by call in the same process; algorithmic bytes and the fraction of the
HBM peak; oracle parity of 64 sampled bridge-frames of the timed output.  Then the one-tick call replayed as a CUDA
graph: p50 / p99 over 1000 replays.  One GPU command:
    python profiles/tools/fanout_bench.py --out profiles/fanout_r03.json
Without --out the result is printed and no file is written."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import igate4xsoftphonedsp_b200 as ig                      # noqa: E402
from igate4xsoftphonedsp_b200 import _native as N          # noqa: E402
from igate4xsoftphonedsp_b200 import synth                 # noqa: E402
from bench import peaks                                    # noqa: E402  (the HBM peak exactly as bench.py finds it)
import oracle_py as O                                      # noqa: E402  (checker only)
import tx_scenarios as T                                   # noqa: E402

THROUGHPUT = [(1024, 4, 1640), (16384, 4, 100), (128, 32, 1640)]      # (B, G, F)
TICK = [(1024, 4), (16384, 4)]                                          # (B, G) at F = 1
NOW0 = 1_000_000


def alg_bytes(F, B, G):
    """PCM in + RTP headers in + packets out; the sender plan, sizes and levels are not counted"""
    return F * B * (2 * N.FRAME + G * 12 + G * N.PKT_MAX)


def inputs(B, G, F, dev):
    Cn = B * G
    law = np.array([i % 2 for i in range(Cn)], np.uint8)                # A-law / u-law alternating, mixed in a bridge
    legs = [dict(radiocall=1, callIn=(c // 3) % 2, calltype=T.CALLTYPES[c % len(T.CALLTYPES)],
                 keepalive=(40, 200)[(c // 2) % 2], slave=None) for c in range(Cn)]
    st0 = T.gpu_inputs(dict(legs=legs, now0=NOW0))
    ctl = synth.ed137_ctl(F, B, G, N.CTL_DT)                             # 2 of 4 legs keyed, the rest with squelch
    rtp12 = synth.rtp12(F, Cn, np.where(law == 0, 8, 0))
    pcm = synth.pcm_noise_tone_torch(F, B, dev)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return dict(law=law, legs=legs, st0=st0, ctl=ctl, rtp12=rtp12, pcm=pcm, law_t=t(law), st0_t=t(st0.view(np.uint8)),
                ctl_t=t(ctl.view(np.uint8)), rtp_t=t(rtp12))


def kernel_ms(fn, names, n):
    """device time per call of the kernels whose name contains one of `names`, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    tot = {}
    for e in prof.key_averages():
        for k in names:
            if k in e.key:
                tot[k] = tot.get(k, 0.0) + e.device_time_total / 1e3
    return {k: v / n for k, v in tot.items()}


def parity(x, got, B, G, F, rng):
    """64 sampled (tick, bridge) pairs of the timed output, the last one among them, against the oracle"""
    pairs = [(int(rng.integers(0, F)), int(rng.integers(0, B))) for _ in range(63)] + [(F - 1, B - 1)]
    pcm = x["pcm"]
    ok = True
    for f, b in pairs:
        cs = slice(b * G, (b + 1) * G)
        enc = [O.g711_encode(pcm[:f + 1, b].cpu().numpy(), lw) for lw in (N.LAW_ALAW, N.LAW_ULAW)]
        payload = np.stack([enc[int(x["law"][c] != 0)] for c in range(b * G, (b + 1) * G)], axis=1)
        s = dict(name="fanout", legs=x["legs"][cs], F=f + 1, ctl=x["ctl"][:f + 1, cs], tick_ms=20, now0=NOW0,
                 payload=payload, rtp12=x["rtp12"][:f + 1, cs])
        pk, sz, _, _ = T.run_oracle(s)
        pk, bm = T.clean_expectation(s, pk, sz)
        ok &= np.array_equal(got["tx_pkts"][f, cs].cpu().numpy(), pk[f])
        ok &= np.array_equal(got["tx_sizes"][f, cs].cpu().numpy().view(np.uint32), sz[f])
        ok &= np.array_equal(got["tx_level"][f, cs].cpu().numpy(), bm[f])
    return bool(ok)


def throughput(vp, B, G, F, peak, steps, rng, dev):
    x = inputs(B, G, F, dev)
    st = x["st0_t"].clone()
    rep = x["pcm"].repeat_interleave(G, dim=1).contiguous()             # the composed path's input, built untimed
    out = None

    def fan():
        nonlocal out
        out = vp.gateway_fanout(x["pcm"], x["law_t"], x["rtp_t"], st, tx_ctl=x["ctl_t"], now_ms0=NOW0, out=out)

    def comp():
        codes = vp.g711_encode(rep, x["law_t"])
        return vp.ed137_pack(x["rtp_t"], codes, st, ctl=x["ctl_t"], now_ms0=NOW0)

    for _ in range(3):
        st.copy_(x["st0_t"]); fan()
        st.copy_(x["st0_t"]); comp()
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(2 * steps)]
    for i in range(steps):           # alternate: fan-out, composed, fan-out, ... each timed alone, state reset untimed
        for j, fn in enumerate((fan, comp)):
            st.copy_(x["st0_t"])
            a, b = ev[2 * i + j]
            a.record(); fn(); b.record()
    torch.cuda.synchronize()
    fan_ms = [ev[2 * i][0].elapsed_time(ev[2 * i][1]) for i in range(steps)]
    comp_ms = [ev[2 * i + 1][0].elapsed_time(ev[2 * i + 1][1]) for i in range(steps)]
    # the timed fan-out output (state from st0) against the composed path's, whole, and the oracle, sampled
    st.copy_(x["st0_t"]); fan()
    st.copy_(x["st0_t"]); pk, sz, bm = comp()
    torch.cuda.synchronize()
    same = bool(torch.equal(out["tx_pkts"], pk) and torch.equal(out["tx_sizes"], sz) and torch.equal(out["tx_level"], bm))
    sizes = {str(k): int(v) for k, v in zip(*np.unique(out["tx_sizes"].cpu().numpy(), return_counts=True))}
    par = parity(x, out, B, G, F, rng)
    # kernel times in a profiled phase of their own
    kt = kernel_ms(lambda: (st.copy_(x["st0_t"]), fan()), ["k_fanout_tile", "k_plan_walk", "k_ed137_plan"], steps)
    ab = alg_bytes(F, B, G)
    fan_med, comp_med, asm = float(np.median(fan_ms)), float(np.median(comp_ms)), kt.get("k_fanout_tile")
    del rep, out, pk, sz, bm
    torch.cuda.empty_cache()
    return {
        "shape": {"B": B, "G": G, "F": F, "legs": B * G},
        "sizes_histogram": sizes,
        "ms_per_call": {"fanout": fan_med, "fanout_min": min(fan_ms), "composed": comp_med, "composed_min": min(comp_ms),
                        "speedup": comp_med / fan_med, "timed_calls_each": steps},
        "kernel_ms_per_call": kt,
        "algorithmic_bytes": {"total": ab, "per_bridge_frame": ab // (F * B)},
        "hbm": {"assembly_kernel_GBps": ab / asm / 1e6 if asm else None,
                "assembly_kernel_frac": ab / asm / 1e6 / peak if asm else None,
                "fanout_call_GBps": ab / fan_med / 1e6, "fanout_call_frac": ab / fan_med / 1e6 / peak},
        "equal_to_composed": same,
        "oracle_parity_64_bridge_frames": par,
    }


def tick_latency(vp, B, G, replays, dev):
    x = inputs(B, G, 1, dev)
    st = x["st0_t"].clone()
    args = (x["pcm"], x["law_t"], x["rtp_t"], st)
    kw = dict(tx_ctl=x["ctl_t"], now_ms0=NOW0)
    out = vp.gateway_fanout(*args, **kw)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        vp.use_torch_stream()
        for _ in range(5):
            vp.gateway_fanout(*args, out=out, **kw)
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        vp.use_torch_stream()
        vp.gateway_fanout(*args, out=out, **kw)
    vp.use_torch_stream()
    for _ in range(50):
        gr.replay()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(replays)]
    for a, b in ev:
        a.record(); gr.replay(); b.record()
    torch.cuda.synchronize()
    us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
    return {"shape": {"B": B, "G": G, "F": 1, "legs": B * G}, "replays": replays,
            "graph_replay_us": {"p50": float(np.percentile(us, 50)), "p99": float(np.percentile(us, 99)),
                                "min": float(us.min())}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the result as JSON to this file (default: print it only)")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--replays", type=int, default=1000)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fanout_bench.py needs the GPU: nothing is measured without one")
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True)
    peak, peak_src = peaks()
    # for reference beside the peak: a device-to-device copy of 4 GiB on this card, read + write bytes over time
    src = torch.empty(1 << 32, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(10):
        dst.copy_(src)
    a1.record()
    torch.cuda.synchronize()
    copy_gbps = 2 * 10 * src.numel() / (a0.elapsed_time(a1) * 1e6)
    del src, dst
    torch.cuda.empty_cache()
    vp = ig.VoicePath(0)
    vp.use_torch_stream()
    rng = np.random.default_rng(3)
    res = {
        "device": torch.cuda.get_device_name(0),
        "nvidia_smi": smi.stdout.strip() if smi.returncode == 0 else smi.stderr.strip(),
        "hbm_peak_GBps": peak, "hbm_peak_source": peak_src, "d2d_copy_4GiB_GBps_measured_in_this_run": copy_gbps,
        "algorithmic_bytes_note": "per bridge-frame: 320 B PCM in + G*12 B RTP headers in + G*180 B packets out; the "
                                  "sender plan (written and read once), tx_sizes and tx_level are not counted",
        "timing": "CUDA events around each call, medians; the fan-out and the composed path alternate call by call; "
                  "sender state reset outside the timed region; kernel times from torch.profiler in a separate phase",
        "throughput": [], "tick": [],
    }
    for B, G, F in THROUGHPUT:
        r = throughput(vp, B, G, F, peak, a.steps, rng, dev)
        print(json.dumps(r), flush=True)
        res["throughput"].append(r)
    for B, G in TICK:
        r = tick_latency(vp, B, G, a.replays, dev)
        print(json.dumps(r), flush=True)
        res["tick"].append(r)
    vp.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps({"written": a.out}))
    else:
        print(json.dumps(res))


if __name__ == "__main__":
    main()
