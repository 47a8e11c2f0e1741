#!/usr/bin/env python
"""Gateway fan-out from packets (igd_gateway_fanout_packets): the console call's received ED-137 packets in, a finished
ED-137 packet for every leg out.  Device-resident buffers larger than L2; per shape: ms per call of the new call, of
the four-step composition it replaces (igd_ed137_parse -> igd_g711_decode_ch -> PCM 0 on the ticks without a whole
frame -> igd_gateway_fanout) and of igd_gateway_fanout on PCM (reference point; its PCM is built outside the timed
region), the three alternated call by call in the same process; kernel times of k_fanout_pkt_tile and k_fanout_tile
from torch.profiler in a separate phase; algorithmic bytes and the fraction of the HBM peak; the new call's output
against the composition's, whole, and 64 sampled bridge-frames against the oracle.  Then one full-duplex tick
(igd_gateway_process + igd_gateway_fanout_packets) replayed as a CUDA graph: p50 / p99 over 1000 replays.
One GPU command:
    python profiles/tools/fanout_packets_bench.py --out profiles/fanout_packets_r03.json
Without --out the result is printed and no file is written."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

TOOLS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(TOOLS))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), TOOLS]
import igate4xsoftphonedsp_b200 as ig                      # noqa: E402
from igate4xsoftphonedsp_b200 import _native as N          # noqa: E402
from igate4xsoftphonedsp_b200 import synth                 # noqa: E402
from bench import peaks                                    # noqa: E402  (the HBM peak exactly as bench.py finds it)
import fanout_bench as FB                                  # noqa: E402  (legs, setters, headers, kernel_ms)
import oracle_py as O                                      # noqa: E402  (checker only)
import tx_scenarios as T                                   # noqa: E402
from test_gpu_fanout_packets import console_frames         # noqa: E402  (checker only: the frame rule on the oracle)

THROUGHPUT = [(1024, 4, 1640), (16384, 4, 100), (128, 32, 1640)]      # (B, G, F)
TICK = [(1024, 4), (16384, 4)]                                          # (B, G) at F = 1
NOW0 = 1_000_000


def alg_bytes(F, B, G, pcm=False):
    """console packets (or PCM) in + RTP headers in + packets out; the sender plan, sizes and levels are not counted"""
    return F * B * ((2 * N.FRAME if pcm else N.PKT_MAX) + G * 12 + G * N.PKT_MAX)


def console_packets(vp, pcm, in_law_t):
    """the console call's packets from the bridges' PCM: G.711 in the call's law, PT 8 / 0; every tenth tick of a bridge
    a 20-byte keep-alive (PT 123, zero past 20 bytes) -- rx_pkts [F][B][180], rx_sizes [F][B]"""
    F, B, _ = pcm.shape
    dev = pcm.device
    rx = torch.zeros((F, B, N.PKT_MAX), dtype=torch.uint8, device=dev)
    ka = (torch.arange(F, device=dev)[:, None] + torch.arange(B, device=dev)[None, :]) % 10 == 0
    rx[..., 0] = 0x90
    rx[..., 1] = torch.where(ka, 123, torch.where(in_law_t == 0, 8, 0)[None, :]).to(torch.uint8)
    rx[..., 12:16] = torch.tensor([0x01, 0x67, 0x00, 0x01], dtype=torch.uint8, device=dev)
    rx[..., 20:] = vp.g711_encode(pcm, in_law_t)
    rx[..., 20:].masked_fill_(ka[..., None], 0)
    sizes = torch.where(ka, 20, 180).to(torch.int32)
    return rx, sizes


def composed(vp, x, st, out):
    F, B = x["rx"].shape[:2]
    fields, pay = vp.ed137_parse(x["rx"].view(F * B, N.PKT_MAX), x["rsz"].view(-1))
    pcm = vp.g711_decode(pay.view(F, B, N.FRAME), x["in_law_t"])
    plen, pt, fl = (fields[:, 1] >> 16) & 0xFFFF, fields[:, 2] & 0xFF, (fields[:, 3] >> 24) & 0xFF
    frame = ((pt == 0) | (pt == 8)) & (plen == 160) & ((fl & 0x10) == 0)
    pcm.mul_(frame.view(F, B, 1))                                     # PCM 0 on the ticks without a whole frame
    return vp.gateway_fanout(pcm, x["law_t"], x["rtp_t"], st, tx_ctl=x["ctl_t"], now_ms0=NOW0, out=out)


def parity(x, got, B, G, F, rng):
    """64 sampled (tick, bridge) pairs of the timed output, the last one among them, against the oracle"""
    pairs = [(int(rng.integers(0, F)), int(rng.integers(0, B))) for _ in range(63)] + [(F - 1, B - 1)]
    ok = True
    for f, b in pairs:
        cs = slice(b * G, (b + 1) * G)
        frames = console_frames(x["rx"][:f + 1, b:b + 1].cpu().numpy(),
                                x["rsz"][:f + 1, b:b + 1].cpu().numpy().view(np.uint32), x["in_law"][b:b + 1])
        enc = [O.g711_encode(frames, lw) for lw in (N.LAW_ALAW, N.LAW_ULAW)]
        payload = np.concatenate([enc[int(x["law"][c] != 0)] for c in range(b * G, (b + 1) * G)], axis=1)
        s = dict(name="fanout_packets", legs=x["legs"][cs], F=f + 1, ctl=x["ctl"][:f + 1, cs], tick_ms=20, now0=NOW0,
                 payload=payload, rtp12=x["rtp12"][:f + 1, cs])
        pk, sz, _, _ = T.run_oracle(s)
        pk, bm = T.clean_expectation(s, pk, sz)
        ok &= np.array_equal(got["tx_pkts"][f, cs].cpu().numpy(), pk[f])
        ok &= np.array_equal(got["tx_sizes"][f, cs].cpu().numpy().view(np.uint32), sz[f])
        ok &= np.array_equal(got["tx_level"][f, cs].cpu().numpy(), bm[f])
    return bool(ok)


def throughput(vp, B, G, F, peak, steps, rng, dev):
    x = FB.inputs(B, G, F, dev)
    x["in_law"] = np.array([b % 2 for b in range(B)], np.uint8)        # the legs alternate A / u: both same and other law
    x["in_law_t"] = torch.from_numpy(x["in_law"]).to(dev)
    x["rx"], x["rsz"] = console_packets(vp, x["pcm"], x["in_law_t"])
    # igd_gateway_fanout's input: the console frames, built untimed
    pcm = vp.g711_decode(x["rx"][..., 20:].contiguous(), x["in_law_t"])
    pcm.masked_fill_((x["rsz"] != 180)[..., None], 0)
    del x["pcm"]
    torch.cuda.empty_cache()
    st = x["st0_t"].clone()
    outs = {"packets": None, "composed": None, "pcm": None}

    def pkt():
        outs["packets"] = vp.gateway_fanout_packets(x["rx"], x["in_law_t"], x["law_t"], x["rtp_t"], st, rx_sizes=x["rsz"],
                                                    tx_ctl=x["ctl_t"], now_ms0=NOW0, out=outs["packets"])

    def comp():
        outs["composed"] = composed(vp, x, st, outs["composed"])

    def pcmf():
        outs["pcm"] = vp.gateway_fanout(pcm, x["law_t"], x["rtp_t"], st, tx_ctl=x["ctl_t"], now_ms0=NOW0, out=outs["pcm"])

    fns = (("packets", pkt), ("composed", comp), ("pcm", pcmf))
    for _ in range(3):
        for _, fn in fns:
            st.copy_(x["st0_t"]); fn()
    torch.cuda.synchronize()
    ev = {k: [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(steps)] for k, _ in fns}
    for i in range(steps):           # alternate: packets, composed, pcm, packets, ... each timed alone, state reset untimed
        for k, fn in fns:
            st.copy_(x["st0_t"])
            a, b = ev[k][i]
            a.record(); fn(); b.record()
    torch.cuda.synchronize()
    ms = {k: [a.elapsed_time(b) for a, b in ev[k]] for k, _ in fns}
    # each output from st0: the new call against the composition (whole) and against the PCM form, and the oracle
    res_out = {}
    for k, fn in fns:
        st.copy_(x["st0_t"]); fn()
        torch.cuda.synchronize()
        res_out[k] = {n: v.clone() for n, v in outs[k].items()}
    same = all(torch.equal(res_out["packets"][n], res_out["composed"][n]) for n in ("tx_pkts", "tx_sizes", "tx_level"))
    same_pcm = all(torch.equal(res_out["packets"][n], res_out["pcm"][n]) for n in ("tx_pkts", "tx_sizes", "tx_level"))
    got = res_out["packets"]
    sizes = {str(k): int(v) for k, v in zip(*np.unique(got["tx_sizes"].cpu().numpy(), return_counts=True))}
    par = parity(x, got, B, G, F, rng)
    del res_out, got
    torch.cuda.empty_cache()
    kt = FB.kernel_ms(lambda: (st.copy_(x["st0_t"]), pkt(), st.copy_(x["st0_t"]), pcmf()),
                      ["k_fanout_pkt_tile", "k_fanout_tile", "k_plan_walk", "k_ed137_plan"], steps)
    ab, abp = alg_bytes(F, B, G), alg_bytes(F, B, G, pcm=True)
    med = {k: float(np.median(v)) for k, v in ms.items()}
    kp, kf = kt.get("k_fanout_pkt_tile"), kt.get("k_fanout_tile")
    del pcm, outs
    torch.cuda.empty_cache()
    return {
        "shape": {"B": B, "G": G, "F": F, "legs": B * G},
        "sizes_histogram": sizes,
        "ms_per_call": {"packets": med["packets"], "packets_min": min(ms["packets"]), "composed": med["composed"],
                        "composed_min": min(ms["composed"]), "pcm_fanout": med["pcm"], "pcm_fanout_min": min(ms["pcm"]),
                        "speedup_vs_composed": med["composed"] / med["packets"], "timed_calls_each": steps},
        "kernel_ms_per_call": kt,
        "algorithmic_bytes": {"packets": ab, "packets_per_bridge_frame": ab // (F * B), "pcm_fanout": abp,
                              "pcm_fanout_per_bridge_frame": abp // (F * B)},
        "hbm": {"k_fanout_pkt_tile_GBps": ab / kp / 1e6 if kp else None,
                "k_fanout_pkt_tile_frac": ab / kp / 1e6 / peak if kp else None,
                "k_fanout_tile_GBps": abp / kf / 1e6 if kf else None,
                "k_fanout_tile_frac": abp / kf / 1e6 / peak if kf else None,
                "packets_call_GBps": ab / med["packets"] / 1e6, "packets_call_frac": ab / med["packets"] / 1e6 / peak},
        "equal_to_composed": same,
        "equal_to_pcm_fanout_on_the_same_frames": same_pcm,
        "oracle_parity_64_bridge_frames": par,
    }


def tick_latency(vp, B, G, replays, dev):
    """one full-duplex tick: igd_gateway_process (radios -> console, G = 4) and igd_gateway_fanout_packets (console ->
    radios, its input the console call's received packets), captured together"""
    Cn = B * G
    x = FB.inputs(B, G, 1, dev)
    in_law = torch.from_numpy(synth.out_laws(B)).to(dev)
    rx_con, rsz_con = console_packets(vp, x["pcm"], in_law)
    gen = torch.Generator(device=dev).manual_seed(1)
    rx_rad = torch.randint(0, 256, (1, Cn, N.PKT_MAX), dtype=torch.uint8, device=dev, generator=gen)
    rx_rad[..., 0] = 0x90
    rx_rad[..., 1] = 8
    rad_law = torch.from_numpy(synth.laws(Cn)).to(dev)
    con_rtp = torch.from_numpy(synth.rtp12(1, B, [8] * B)).to(dev)
    gst = (torch.zeros((Cn, 4), dtype=torch.int32, device=dev), torch.zeros((Cn, 2), dtype=torch.int32, device=dev),
           torch.zeros((B, 4), dtype=torch.int32, device=dev),
           torch.from_numpy(ig.make_state(B, now_ms=0).view(np.int32).reshape(B, 10)).to(dev))
    st = x["st0_t"].clone()
    outs = [None, None]

    def tick():
        outs[0] = vp.gateway_process(rx_rad, rad_law, in_law, gst[0], gst[1], gst[2], con_rtp, gst[3],
                                     mode=N.ARB_CLIENT_PTT, now_ms0=NOW0, want=("bmeter",), out=outs[0])
        outs[1] = vp.gateway_fanout_packets(rx_con, in_law, x["law_t"], x["rtp_t"], st, rx_sizes=rsz_con,
                                            tx_ctl=x["ctl_t"], now_ms0=NOW0, out=outs[1])

    tick()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        vp.use_torch_stream()
        for _ in range(5):
            tick()
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        vp.use_torch_stream()
        tick()
    vp.use_torch_stream()
    for _ in range(50):
        gr.replay()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(replays)]
    for a, b in ev:
        a.record(); gr.replay(); b.record()
    torch.cuda.synchronize()
    us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
    return {"shape": {"B": B, "G": G, "F": 1, "radio_legs": Cn}, "replays": replays,
            "full_duplex_tick_graph_replay_us": {"p50": float(np.percentile(us, 50)), "p99": float(np.percentile(us, 99)),
                                                 "min": float(us.min())}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the result as JSON to this file (default: print it only)")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--replays", type=int, default=1000)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fanout_packets_bench.py needs the GPU: nothing is measured without one")
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True)
    peak, peak_src = peaks()
    src = torch.empty(1 << 32, dtype=torch.uint8, device=dev)      # beside the peak: a 4 GiB device-to-device copy
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
        "algorithmic_bytes_note": "per bridge-frame: 180 B console packet in (igd_gateway_fanout: 320 B PCM) + G*12 B RTP "
                                  "headers in + G*180 B packets out; the sender plan, rx_sizes, tx_sizes and tx_level "
                                  "are not counted",
        "inputs": "console packets: the bridges' PCM (noise + tone) G.711-encoded in the call's law (A / u alternating "
                  "by bridge), every tenth tick a keep-alive; leg laws alternate A / u inside a bridge",
        "timing": "CUDA events around each call, medians; the new call, the four-step composition and igd_gateway_fanout "
                  "alternate call by call; sender state reset outside the timed region; kernel times from torch.profiler "
                  "in a separate phase",
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
