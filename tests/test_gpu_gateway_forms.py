"""igd_gateway_process against the oracle in every form the call takes: the three receive walks (warp per bridge with
the tick axis across its lanes, thread per bridge, IGD_F_WALK_SERIAL's thread-per-channel kernels pipelined over chunks
of ticks), both fused kernels (default and IGD_F_KERNEL_W), both char signs, host and device buffers, with and without
rx_sizes / tx_ctl / active, every watchdog period, a non-zero frame0, a non-default tick and state carried across split
calls.  Everything the call returns is recomputed by the oracle from the raw packets: the receive walk
(transport_rtp_cb + the R2S watchdog), checkEvents' gate decisions with silent no-audio ticks, decode -> meter -> mix ->
encode, and the sender (transport_send_rtp, clean mode).  Also: the host form's chunked pipeline equals the device
form byte for byte, packet arrays beyond 2^32 bytes, outputs that stay inside their buffers, argument errors that
launch nothing, and host-form calls that wait for device-form work already queued on the same context."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle_py as O
import rx_arb_cases as R
import test_gpu_fanout as FO
import test_gpu_fanout_packets as FP
import test_gpu_packets_fused as PF
import tx_scenarios as T
import igate4xsoftphonedsp_b200 as ig
from igate4xsoftphonedsp_b200 import _native as N
from igate4xsoftphonedsp_b200 import synth
from test_gpu_fused import check
from test_gpu_gateway import G, make_case, tx_state_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WANT = ("rx_events", "gain_q7", "meter", "bmeter", "mix", "enc")
# numpy record type and per-call shape of every output ([F][B] or [F][B*4] leading axes)
OUT_DT = {"tx_pkts": np.uint8, "tx_sizes": np.uint32, "rx_events": N.RX_EVENT_DT, "gain_q7": np.uint16,
          "meter": N.METER_DT, "bmeter": N.BRIDGE_DT, "mix": np.int16, "enc": np.uint8}
PER_LEG = ("rx_events", "gain_q7", "meter")
STATE_DT = (N.RX_STATE_DT, N.ARB_LEG_DT, N.ARB_BRIDGE_DT, N.STATE_DT)


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def host_out(k, x, F, B):
    """a device output as the host form returns it"""
    a = np.ascontiguousarray(x.cpu().numpy()).view(OUT_DT[k])
    lead = (F, 4 * B) if k in PER_LEG else (F, B)
    return a.reshape(lead + a.shape[len(lead):]) if k in ("tx_pkts", "mix", "enc") else a.reshape(lead)


def states0(c):
    Cn = 4 * c["B"]
    return [np.zeros(Cn, N.RX_STATE_DT), np.zeros(Cn, N.ARB_LEG_DT), np.zeros(c["B"], N.ARB_BRIDGE_DT), tx_state_of(c)]


def dev_states(st):
    return [t(s.view(np.int32).reshape(len(s), -1)) for s in st]


def host_states(dst):
    return [np.ascontiguousarray(x.cpu().numpy()).view(dt).reshape(-1) for x, dt in zip(dst, STATE_DT)]


def call(vp, c, st, flags, f0=0, want=WANT, out=None, **x):
    """one igd_gateway_process call on the ticks in x (pk, sizes, rtp12, ctl: numpy or torch), scalars from c"""
    return vp.gateway_process(x["pk"], c["law_x"], c["out_law_x"], st[0], st[1], st[2], x["rtp12"], st[3],
                              rx_sizes=x["sizes"], tx_ctl=x["ctl"], active=c["active_x"], mode=c["mode"],
                              now_ms0=c["now0"] + c["tick"] * f0, tick_ms=c["tick"], wd_ticks=c["wd"],
                              frame0=c["frame0"] + f0, flags=flags, want=want, out=out)


def run(vp, c, flags, device, cuts=None, want=WANT):
    """the case through the call, its ticks split at `cuts` (state carried by the arrays and frame0); -> (outputs as
    numpy [F]..., final states as numpy)"""
    F, B = c["F"], c["B"]
    cuts = cuts or (0, F)
    st = states0(c)

    def conv(a, as_dev=lambda a: a):
        return None if a is None else t(as_dev(a)) if device else np.ascontiguousarray(a)

    c = dict(c, law_x=conv(c["law"]), out_law_x=conv(c["out_law"]), active_x=conv(c["active"]))
    if device:
        st = dev_states(st)
    parts = []
    for f0, f1 in zip(cuts[:-1], cuts[1:]):
        sl = slice(f0, f1)
        x = dict(pk=conv(c["pk"][sl]), rtp12=conv(c["rtp12"][sl]),
                 sizes=conv(None if c["sizes"] is None else c["sizes"][sl], lambda a: a.view(np.int32)),
                 ctl=conv(None if c["ctl"] is None else c["ctl"][sl], lambda a: a.view(np.int32).reshape(f1 - f0, B, 2)))
        if device:
            torch.cuda.synchronize()
        o = call(vp, c, st, flags, f0=f0, want=want, **x)
        if device:
            torch.cuda.synchronize()
            o = {k: host_out(k, v, f1 - f0, B) for k, v in o.items()}
        parts.append(o)
    out = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    return out, host_states(st) if device else st


def oracle(c, signed_char=0):
    """everything the call returns, recomputed by the oracle from the raw packets"""
    F, B = c["F"], c["B"]
    Cn = 4 * B
    sizes = np.full((F, Cn), 180, np.uint32) if c["sizes"] is None else c["sizes"]
    ev, rx_st = R.oracle_rx_walk(c["pk"], sizes, (sizes != 0).astype(np.uint8), now0=c["now0"], tick=c["tick"],
                                 wd_ticks=c["wd"], frame0=c["frame0"])
    g, lg, br = R.oracle_arb_walk(np.ascontiguousarray(ev["word"]), G, c["mode"], active=c["active"])
    g = np.where((ev["flags"] & N.RXE_FRAME) == 0, g | N.GAIN_NO_AUDIO, g).astype(np.uint16)
    payload = np.zeros((F, Cn, 160), np.uint8)
    full = sizes >= 180
    payload[full] = c["pk"][full][:, 20:180]         # only whole frames are heard (the others carry GAIN_NO_AUDIO)
    mix, enc, meter, bmeter = O.process_batch(payload, c["law"], g, c["out_law"], G, signed_char=signed_char)
    s = dict(name="gw", legs=c["legs"], F=F, ctl=c["ctl"], tick_ms=c["tick"], now0=c["now0"], payload=enc,
             rtp12=c["rtp12"])
    pk, sz, _, ads = T.run_oracle(s, signed_char)        # the reference-exact sender (quirks included) ...
    pk, _ = T.clean_expectation(s, pk, sz, signed_char)  # ... with this tick's payload in every audio packet (Q2 off)
    return dict(tx_pkts=pk, tx_sizes=sz, rx_events=ev, gain_q7=g, mix=mix, enc=enc, meter=meter, bmeter=bmeter,
                states=(rx_st, lg, br), ads=ads, payload=enc)


def compare(vp, got, st, c, want, signed_char=0, where=""):
    assert np.array_equal(got["tx_sizes"], want["tx_sizes"]), where
    assert np.array_equal(got["tx_pkts"], want["tx_pkts"]), where           # all 180 bytes of every slot
    assert got["rx_events"].tobytes() == want["rx_events"].tobytes(), where
    assert np.array_equal(got["gain_q7"], want["gain_q7"]), where
    check(got, (want["mix"], want["enc"], want["meter"], want["bmeter"]))     # integer meters, dB within 1e-4
    for name, a, b in zip(("rx_state", "arb_legs", "arb_bridges"), st[:3], want["states"]):
        assert a.tobytes() == b.tobytes(), (where, name)
    for b, a in enumerate(want["ads"]):
        for name in FO.STATE_FIELDS:
            assert int(st[3][name][b]) == int(getattr(a, name)), (where, b, name)
    # the whole sender record against the verified sender walk on the oracle's payload (rtpFalse, never read by the
    # reference, is not maintained by the gateway call)
    st_p = tx_state_of(c)
    vp.ed137_pack(c["rtp12"], want["payload"], st_p, ctl=c["ctl"], now_ms0=c["now0"], tick_ms=c["tick"],
                  flags=N.F_SIGNED_CHAR if signed_char else 0)
    assert FO.masked(st[3]) == FO.masked(st_p), where


def small_case(F, B, seed, mode, sizes=True, ctl=True, active=False, wd=2, frame0=0, tick=20):
    c = make_case(F, B, seed, mode)
    rng = np.random.default_rng(seed + 7)
    c.update(F=F, B=B, mode=mode, tick=tick, wd=wd, frame0=frame0,
             sizes=c["sizes"] if sizes else None, ctl=c["ctl"] if ctl else None,
             active=(rng.random(4 * B) < 0.75).astype(np.uint8) if active else None)
    return c


# ---------------------------------------------------------------- (a) the oracle matrix at small shapes
FORMS = ("lanes", "bridge", "serial")
MATRIX = [(form, kern, sc, device) for form in FORMS for kern in (0, N.F_KERNEL_W) for sc in (0, 1)
          for device in (False, True)]


def matrix_case(i, form):
    """the options case i of the matrix runs with, spread over the eight cases of its form (i % 8 enumerates kernel,
    char sign and memory form within it; shifted per form): within every form each option below takes each of its
    values, wd every one of 0..3"""
    j = (i + 3 * FORMS.index(form)) % 8
    F = {"lanes": 17 + (7 * i) % 48,                     # >= 8 ticks per call, also when split in two
         "bridge": 1 + i % 7,                            # < 8 ticks: one thread per bridge
         "serial": (3 + i % 5) if j % 2 else 24 + (5 * i) % 40}[form]
    B = 1 + (5 * i) % 16
    opts = dict(sizes=j % 3 != 0, ctl=j % 3 != 1, active=(j // 2) % 2 == 1, wd=j % 4, frame0=0 if j == 0 else 3 + 11 * j,
                tick=(20, 20, 30 if j % 2 else 10)[j % 3])
    mode = N.ARB_SERVER_BEST if (j + (j >> 2)) % 2 else N.ARB_CLIENT_PTT
    cuts = (0, F // 2 + (j & 1), F) if j % 4 in (1, 2) and F >= 2 else None
    return small_case(F, B, 300 + i, mode, **opts), cuts


@pytest.mark.parametrize("form,kern,signed_char,device", MATRIX,
                         ids=[f"{f}-{'w' if k else 'q'}-{'signed' if s else 'unsigned'}-{'dev' if d else 'host'}"
                              for f, k, s, d in MATRIX])
def test_gateway_against_the_oracle_in_every_form(vp, form, kern, signed_char, device):
    i = MATRIX.index((form, kern, signed_char, device))
    c, cuts = matrix_case(i, form)
    flags = kern | (N.F_SIGNED_CHAR if signed_char else 0) | (N.F_WALK_SERIAL if form == "serial" else 0)
    got, st = run(vp, c, flags, device, cuts)
    compare(vp, got, st, c, oracle(c, signed_char), signed_char)


# ---------------------------------------------------------------- (b) the device-form pipeline of IGD_F_WALK_SERIAL
def test_walk_serial_pipeline_in_device_form_against_the_oracle(vp):
    """96 ticks of 160 channels: six chunks of 16 ticks, liveness walk / arbitration / fused kernel on three streams
    with the sender walk beside them, every stage carrying its state from chunk to chunk"""
    c = small_case(96, 40, 501, N.ARB_SERVER_BEST, active=True, wd=3, frame0=5)
    n0 = vp.launch_count()
    got, st = run(vp, c, N.F_WALK_SERIAL, device=True)
    # per chunk: header view + liveness walk (2), sender walk (1), fused kernel (2)
    assert vp.launch_count() - n0 == 6 * 5
    compare(vp, got, st, c, oracle(c))


def test_walk_serial_pipeline_is_cuda_graph_capturable(vp):
    """64 ticks of 1200 channels with IGD_F_WALK_SERIAL = 4 chunks: liveness walk, arbitration and fused kernel on three
    streams of the library and the sender walk on a fourth, forked from and joined back to the caller's stream by
    events.  The whole call captures into one CUDA graph and replays with the bytes of the eager call, which equal
    those of the lane walk (one chunk)."""
    F, B, mode = 64, 300, N.ARB_CLIENT_PTT
    case = make_case(F, B, 31, mode)
    st0 = dev_states(states0(dict(case, B=B)))
    st = [s.clone() for s in st0]
    args = (t(case["pk"]), t(case["law"]), t(case["out_law"]), *st[:3], t(case["rtp12"]), st[3])
    kw = dict(rx_sizes=t(case["sizes"].view(np.int32)), tx_ctl=t(case["ctl"].view(np.int32).reshape(F, B, 2)), mode=mode,
              now_ms0=case["now0"], want=("bmeter", "meter", "enc", "gain_q7"))

    def reset():
        for a, b in zip(st, st0):
            a.copy_(b)

    def snapshot(out):
        torch.cuda.synchronize()
        return {k: v.cpu().numpy().copy() for k, v in out.items()}, [s.cpu().numpy().copy() for s in st]

    torch.cuda.synchronize()
    vp.use_torch_stream()
    lanes = snapshot(vp.gateway_process(*args, **kw))
    reset()
    n0 = vp.launch_count()
    eager = vp.gateway_process(*args, flags=N.F_WALK_SERIAL, **kw)
    assert vp.launch_count() - n0 == 4 * 5        # per chunk: header view + liveness walk, sender walk, fused kernel
    want = snapshot(eager)
    for k in want[0]:
        assert np.array_equal(want[0][k], lanes[0][k]), k
    for a, b in zip(want[1], lanes[1]):
        assert np.array_equal(a, b)
    reset()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        vp.use_torch_stream()
        vp.gateway_process(*args, flags=N.F_WALK_SERIAL, out=eager, **kw)     # warm-up on a side stream: sizes the scratch
    torch.cuda.synchronize()
    reset()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        vp.use_torch_stream()
        vp.gateway_process(*args, flags=N.F_WALK_SERIAL, out=eager, **kw)
    vp.use_torch_stream()
    for rep in range(2):
        reset()
        for v in eager.values():
            v.zero_()
        gr.replay()
        torch.cuda.synchronize()
        got = snapshot(eager)
        for k in want[0]:
            assert np.array_equal(got[0][k], want[0][k]), (rep, k)
        for a, b in zip(got[1], want[1]):
            assert np.array_equal(a, b), rep


# ---------------------------------------------------------------- closed-form inputs for the large shapes
def _h(x):
    """a 32-bit integer hash, elementwise on int64 tensors"""
    x = x & 0xFFFFFFFF
    x = (((x >> 16) ^ x) * 0x45D9F3B) & 0xFFFFFFFF
    x = (((x >> 16) ^ x) * 0x45D9F3B) & 0xFFFFFFFF
    return (x >> 16) ^ x


ODD_SIZES = [0, 7, 12, 19, 20, 21, 100, 179, 180, 1043, 1044, 4000]


def device_case(F, B, seed, mode, active=False, ctl=True):
    """received packets built on the device without a per-channel loop: per leg, runs of audio (PT 8 / 0, some PT 18),
    keep-alives, gaps and odd packets (short, truncated, oversized, unaccepted PT, no header extension), with PTT /
    squelch words in bursts that overlap between the legs of a bridge"""
    Cn = 4 * B
    gen = torch.Generator(device=DEV).manual_seed(seed)
    pk = torch.randint(0, 256, (F, Cn, 180), dtype=torch.uint8, device=DEV, generator=gen)
    f = torch.arange(F, device=DEV, dtype=torch.int64)[:, None]
    ch = torch.arange(Cn, device=DEV, dtype=torch.int64)[None, :]
    s = seed * 7919
    rl = 3 + _h(ch + s) % 37
    blk = (f + _h(ch + s + 1) % rl) // rl
    h = _h(blk * 1000003 + ch * 31 + s + 2)
    kind = torch.where(ch % 6 == 0, 0, h % 20)          # 0-8 audio, 9-13 keep-alive, 14-16 gap, 17-19 odd
    del blk, rl
    hf = _h(f * 65599 + ch * 131 + s + 3)                # per packet
    pt = torch.tensor([8, 0, 8, 0, 18], device=DEV)[(h >> 5) % 5]
    pt = torch.where(kind >= 9, 123, pt)
    pt = torch.where(kind >= 17, hf % 128, pt)
    size = torch.full_like(kind, 180)
    size = torch.where(kind >= 9, 20, size)
    size = torch.where(kind >= 14, 0, size)
    size = torch.where(kind >= 17, torch.tensor(ODD_SIZES, device=DEV)[(hf >> 8) % len(ODD_SIZES)], size)
    # one leg in eleven falls silent for 40..199 ticks: the watchdog reports it late and hangs it up
    g0 = _h(ch + s + 7) % max(F - 40, 1)
    size = torch.where((ch % 11 == 5) & (f >= g0) & (f < g0 + 40 + _h(ch + s + 8) % 160), 0, size)
    b0 = torch.where((kind >= 17) & ((hf >> 12) % 3 == 0), 0x80, 0x90)
    b1 = pt | torch.where((hf >> 14) % 16 == 0, 0x80, 0)
    del h, kind
    rl = 2 + _h(ch + s + 4) % 29
    wblk = (f + _h(ch + s + 5) % rl) // rl
    hw = _h(wblk * 1000033 + ch * 17 + s + 6)
    if mode == N.ARB_CLIENT_PTT:
        word = (torch.tensor([0, 0, 1, 1, 2, 3, 4], device=DEV)[hw % 7] << 29) | (((hw >> 4) % 64) << 22)
    else:
        word = (((hw >> 4) % 2) << 28) | (((hw >> 6) % 32) << 3) | 0x00013100
    del wblk, rl, hw, hf
    hdr = torch.empty((F, Cn, 20), dtype=torch.uint8, device=DEV)
    fb = lambda v, sh: ((v >> sh) & 0xFF).to(torch.uint8)
    hdr[..., 0] = b0.to(torch.uint8)
    hdr[..., 1] = b1.to(torch.uint8)
    for k, (v, nb) in enumerate(((f & 0xFFFF, 2), (160 * f, 4), (ch, 4), (torch.tensor(0x0167, device=DEV), 2),
                                 (torch.tensor(1, device=DEV), 2), (word, 4))):
        o = (2, 4, 8, 12, 14, 16)[k]
        for q in range(nb):
            hdr[..., o + q] = fb(v, 8 * (nb - 1 - q))
    pk[..., :20] = hdr
    del hdr, word, b0, b1, pt
    sizes = size.to(torch.int32)
    rng = np.random.default_rng(seed)
    law = rng.integers(0, 2, Cn).astype(np.uint8)
    out_law = rng.integers(0, 2, B).astype(np.uint8)
    legs = [dict(radiocall=1, callIn=b % 2, calltype=T.CALLTYPES[(b // 2) % 4], keepalive=(40, 200)[(b // 8) % 2],
                 slave=None) for b in range(B)]
    ctl = T._random_ctl(F, B, seed + 2, p_hold=0.9) if ctl else None
    rtp12 = synth.rtp12(F, B, np.where(out_law == 0, 8, 0))
    c = dict(F=F, B=B, mode=mode, tick=20, wd=2, frame0=0, now0=1_000_000, legs=legs, law=law, out_law=out_law,
             active=(rng.random(Cn) < 0.8).astype(np.uint8) if active else None, ctl=ctl, rtp12=rtp12)
    x = dict(pk=pk, sizes=sizes, rtp12=t(rtp12), ctl=None if ctl is None else t(ctl.view(np.int32).reshape(F, B, 2)))
    c.update(law_x=t(law), out_law_x=t(out_law), active_x=None if c["active"] is None else t(c["active"]))
    return c, x


def sub_case(c, x, bridges):
    """the bridges `bridges` of a device case as a host case of their own (bridges are independent in every stage)"""
    bl = torch.tensor(bridges, device=DEV)
    chl = (bl[:, None] * 4 + torch.arange(4, device=DEV)[None, :]).reshape(-1)
    chn, bn = chl.cpu().numpy(), np.asarray(bridges)
    return dict(F=c["F"], B=len(bridges), mode=c["mode"], tick=c["tick"], wd=c["wd"], frame0=c["frame0"], now0=c["now0"],
                legs=[c["legs"][b] for b in bridges], law=c["law"][chn], out_law=c["out_law"][bn],
                active=None if c["active"] is None else c["active"][chn], ctl=None if c["ctl"] is None else c["ctl"][:, bn], rtp12=c["rtp12"][:, bn],
                pk=x["pk"].index_select(1, chl).cpu().numpy(),
                sizes=x["sizes"].index_select(1, chl).cpu().numpy().view(np.uint32)), chl, bl


def compare_bridges(vp, c, x, got, dst, bridges, signed_char=0):
    """the call's results on a sample of bridges against the oracle run on those bridges alone"""
    cs, chl, bl = sub_case(c, x, bridges)
    F, Bs = c["F"], len(bridges)
    g = {k: host_out(k, v.index_select(1, chl if k in PER_LEG else bl), F, Bs) for k, v in got.items()}
    st = [s.index_select(0, i) for s, i in zip(dst, (chl, chl, bl, bl))]
    compare(vp, g, host_states(st), cs, oracle(cs, signed_char), signed_char, where=bridges)


def run_dev(vp, c, x, flags, want=WANT):
    st = dev_states(states0(c))
    torch.cuda.synchronize()
    got = call(vp, c, st, flags, want=want, **x)
    torch.cuda.synchronize()
    return got, st


# ---------------------------------------------------------------- (c) host form = device form where the host form chunks
@pytest.mark.parametrize("flags", [0, N.F_WALK_SERIAL], ids=["lanes", "walk_serial"])
def test_chunked_host_form_equals_device_form(vp, flags):
    """120 ticks of 4096 channels = 88 MB of packets: the host form copies them in two chunks beside the kernels (with
    IGD_F_WALK_SERIAL through the field-record scratch), the device form runs one chunk (lanes) or seven (serial)"""
    F, B = 120, 1024
    c, x = device_case(F, B, 601 + flags, N.ARB_CLIENT_PTT, active=True)
    dev_t, dst = run_dev(vp, c, x, flags)
    dev = {k: host_out(k, v, F, B) for k, v in dev_t.items()}
    h = dict(c, law_x=c["law"], out_law_x=c["out_law"], active_x=c["active"])
    st = states0(c)
    n0 = vp.launch_count()
    host = call(vp, h, st, flags, pk=x["pk"].cpu().numpy(), sizes=x["sizes"].cpu().numpy().view(np.uint32),
                rtp12=c["rtp12"], ctl=c["ctl"])
    assert vp.launch_count() - n0 == 2 * (4 if flags == 0 else 5)          # two chunks
    for k in dev:
        assert host[k].tobytes() == dev[k].tobytes(), k
    for a, b in zip(st, host_states(dst)):
        assert a.tobytes() == b.tobytes()
    assert (host["tx_sizes"] == 180).any() and (host["tx_sizes"] == 20).any()
    compare_bridges(vp, c, x, dev_t, dst, [0, 517, B - 1])


# ---------------------------------------------------------------- (d) packet arrays beyond 4 GiB
def straddlers(total_items):
    """the item whose 180-byte slot straddles byte 2^32 of an array of such slots, and its two neighbours"""
    i = (1 << 32) // 180
    return [j for j in (i - 1, i, i + 1) if 0 <= j < total_items]


def test_packet_array_beyond_4_gib_lane_walk_and_serial_walks(vp):
    """16 383 bridges = 65 532 channels (the largest lane-walk call) x 400 ticks: 4.7 GB of received packets.  The lane
    walk and IGD_F_WALK_SERIAL (k_rx_track reading the packets: >= 32 768 channels) agree byte for byte; six bridges
    (the first, the last, three in between and the one whose packets straddle byte 2^32 of rx_pkts) against the
    oracle"""
    F, B = 400, 16383
    free, _ = torch.cuda.mem_get_info()
    if free < 40 << 30:
        pytest.skip("needs 40 GB of free device memory")
    c, x = device_case(F, B, 701, N.ARB_CLIENT_PTT)
    assert x["pk"].numel() > 2 ** 32
    lanes, st_l = run_dev(vp, c, x, 0)
    serial, st_s = run_dev(vp, c, x, N.F_WALK_SERIAL)
    for k in lanes:
        assert torch.equal(lanes[k], serial[k]), k
    for a, b in zip(st_l, st_s):
        assert torch.equal(a, b)
    del serial, st_s
    rx_b = sorted({i % (4 * B) // 4 for i in straddlers(F * 4 * B)})
    bridges = sorted({0, B - 1, 5000, 8191, 12001} | set(rx_b))
    compare_bridges(vp, c, x, lanes, st_l, bridges)


def test_packet_array_beyond_4_gib_thread_per_bridge_walk(vp):
    """65 536 bridges x 370 ticks: 17.5 GB of received packets and 4.37 GB of sent ones, both beyond 2^32 bytes, one
    thread per bridge walking liveness + arbitration; nine bridges (the first, the last, three in between and those
    whose packets straddle byte 2^32 of rx_pkts and of tx_pkts) against the oracle"""
    F, B = 370, 65536
    free, _ = torch.cuda.mem_get_info()
    if free < 64 << 30:
        pytest.skip("needs 64 GB of free device memory")
    c, x = device_case(F, B, 801, N.ARB_SERVER_BEST, active=True)
    assert x["pk"].numel() > 2 ** 32
    got, dst = run_dev(vp, c, x, 0)
    assert got["tx_pkts"].numel() > 2 ** 32
    rx_b = {i % (4 * B) // 4 for i in straddlers(F * 4 * B)}
    tx_b = {i % B for i in straddlers(F * B)}
    bridges = sorted({0, B - 1, 20000, 32768, 40000} | rx_b | tx_b)
    compare_bridges(vp, c, x, got, dst, bridges)


# ---------------------------------------------------------------- (e) outputs stay inside their buffers
GUARD = 4096


def guarded(nbytes, fill):
    a = torch.full((GUARD + nbytes + (-nbytes) % 32 + GUARD,), fill, dtype=torch.uint8, device=DEV)
    return a, a[GUARD:GUARD + nbytes]


@pytest.mark.parametrize("form,F,B", [("lanes", 37, 11), ("bridge", 5, 53), ("serial", 29, 17)])
def test_outputs_and_states_stay_inside_their_buffers(vp, form, F, B):
    """F*B off a multiple of the fused kernel's 184 bridge-frame tiles (23 warps x 8): every output and every in/out
    state array sits between two guard bands and the call writes all of it and nothing around it; the packets it
    reads sit between guard bands of bytes that would change the results"""
    assert (F * B) % 184 and F * B > 184
    c = small_case(F, B, 900 + F, N.ARB_CLIENT_PTT, active=True, wd=3)
    Cn = 4 * B
    arenas = {}

    def put(name, nbytes, dtype, shape, init=None):
        a, inner = guarded(nbytes, 0xA5)
        if init is not None:
            inner.copy_(t(np.ascontiguousarray(init).view(np.uint8).reshape(-1)))
        arenas[name] = (a, nbytes)
        return inner.view(dtype).reshape(shape)

    out = {k: put(k, F * n * sz, dt, (F, n) + tail) for k, n, sz, dt, tail in (
        ("tx_pkts", B, 180, torch.uint8, (180,)), ("tx_sizes", B, 4, torch.int32, ()),
        ("rx_events", Cn, 8, torch.int32, (2,)), ("gain_q7", Cn, 2, torch.int16, ()),
        ("meter", Cn, 16, torch.int32, (4,)), ("bmeter", B, 4, torch.int32, ()),
        ("mix", B, 320, torch.int16, (160,)), ("enc", B, 160, torch.uint8, (160,)))}
    st = [put(f"state{i}", s.nbytes, torch.int32, (len(s), s.itemsize // 4), s) for i, s in enumerate(states0(c))]
    _, pk_in = guarded(c["pk"].nbytes, 0x5A)
    pk_in.copy_(t(c["pk"].reshape(-1)))
    x = dict(pk=pk_in.view(F, Cn, 180), sizes=t(c["sizes"].view(np.int32)), rtp12=t(c["rtp12"]),
             ctl=t(c["ctl"].view(np.int32).reshape(F, B, 2)))
    cx = dict(c, law_x=t(c["law"]), out_law_x=t(c["out_law"]), active_x=t(c["active"]))
    flags = N.F_WALK_SERIAL if form == "serial" else 0
    torch.cuda.synchronize()
    got = call(vp, cx, st, flags, out=out, **x)
    torch.cuda.synchronize()
    for k, (a, nbytes) in arenas.items():
        assert bool((a[:GUARD] == 0xA5).all()) and bool((a[GUARD + nbytes:] == 0xA5).all()), f"{k}: wrote outside"
    compare(vp, {k: host_out(k, v, F, B) for k, v in got.items()}, host_states(st), c, oracle(c))


# ---------------------------------------------------------------- (f) argument errors launch nothing
def test_argument_errors_launch_nothing(vp):
    F, B = 2, 3
    Cn = 4 * B
    z = lambda n: torch.zeros(n + 64, dtype=torch.uint8, device=DEV)   # room for the misaligned pointers below
    buf = dict(rx_pkts=z(F * Cn * 180), rx_sizes=z(F * Cn * 4), law=z(Cn), active=z(Cn), rx_state=z(Cn * 16),
               arb_legs=z(Cn * 8), arb_bridges=z(B * 16), out_law=z(B), tx_rtp12=z(F * B * 12), tx_ctl=z(F * B * 8),
               tx_state=t(ig.make_state(B).view(np.uint8)), tx_pkts=z(F * B * 180), tx_sizes=z(F * B * 4),
               rx_events=z(F * Cn * 8), gain_q7=z(F * Cn * 2), meter=z(F * Cn * 16), bmeter=z(F * B * 4),
               mix=z(F * B * 320), enc=z(F * B * 160))
    p = {k: v.data_ptr() for k, v in buf.items()}
    vp.use_torch_stream()

    def call_(**over):
        d = dict(struct_size=C.sizeof(N.GatewayDesc), mem=N.MEM_DEVICE, F=F, B=B, G=4, flags=0,
                 arb_mode=N.ARB_CLIENT_PTT, tick_ms=20, r2s_period_ms=200, wd_ticks=2, frame0=0, reserved=0, now_ms0=0, **p)
        d.update(over)
        return vp._lib.igd_gateway_process(vp._h, C.byref(N.GatewayDesc(**d)))

    n0 = vp.launch_count()
    assert call_() == 0 and vp.launch_count() > n0
    for flags in (N.F_SIGNED_CHAR, N.F_KERNEL_W, N.F_WALK_SERIAL, N.F_SIGNED_CHAR | N.F_KERNEL_W | N.F_WALK_SERIAL):
        assert call_(flags=flags) == 0, flags
    assert call_(frame0=7, wd_ticks=0) == 0
    required = ("rx_pkts", "law", "rx_state", "arb_legs", "arb_bridges", "out_law", "tx_rtp12", "tx_state", "tx_pkts",
                "tx_sizes")
    misaligned = dict(rx_pkts=4, rx_sizes=2, law=2, rx_state=8, arb_legs=4, arb_bridges=2, tx_rtp12=2, tx_ctl=4,
                      tx_state=4, tx_pkts=2, tx_sizes=2, rx_events=4, gain_q7=4, meter=8, bmeter=2, mix=16, enc=8)
    bad = [dict(G=3), dict(G=8), dict(G=0), dict(arb_mode=2), dict(arb_mode=-1), dict(F=-1), dict(B=-1), dict(wd_ticks=-1),
           dict(frame0=-1), dict(frame0=-(1 << 31)), dict(struct_size=C.sizeof(N.GatewayDesc) - 8),
           dict(struct_size=C.sizeof(N.GatewayDesc) + 8), dict(flags=N.F_REF_QUIRKS), dict(flags=N.F_GENERIC_KERNEL),
           dict(flags=0x100), dict(flags=N.F_SIGNED_CHAR | 0x80000000)]
    bad += [{k: None} for k in required]
    bad += [{k: p[k] + off} for k, off in misaligned.items()]
    for over in bad:
        n = vp.launch_count()
        assert call_(**over) == -22, over
        assert vp.launch_count() == n, over
    for over in (dict(F=0), dict(B=0), dict(F=0, rx_pkts=None)):
        n = vp.launch_count()
        assert call_(**over) == 0 and vp.launch_count() == n, over
    torch.cuda.synchronize()


def test_rx_track_rejects_a_negative_frame0(vp):
    F, Cn = 3, 8
    fields = torch.zeros(F * Cn * 16, dtype=torch.uint8, device=DEV)
    state = torch.zeros(Cn * 16, dtype=torch.uint8, device=DEV)
    events = torch.zeros(F * Cn * 8, dtype=torch.uint8, device=DEV)
    vp.use_torch_stream()

    def call_(**over):
        d = dict(struct_size=C.sizeof(N.RxTrackDesc), mem=N.MEM_DEVICE, F=F, C=Cn, tick_ms=20, r2s_period_ms=200,
                 wd_ticks=2, frame0=0, now_ms0=0, fields=fields.data_ptr(), present=None, state=state.data_ptr(),
                 events=events.data_ptr(), sizes=None)
        d.update(over)
        return vp._lib.igd_rx_track(vp._h, C.byref(N.RxTrackDesc(**d)))

    n0 = vp.launch_count()
    assert call_(frame0=5) == 0 and vp.launch_count() == n0 + 1
    for over in (dict(frame0=-1), dict(frame0=-(1 << 31)), dict(wd_ticks=-1), dict(F=-1)):
        n = vp.launch_count()
        assert call_(**over) == -22, over
        assert vp.launch_count() == n, over
    torch.cuda.synchronize()


# ---------------------------------------------------------------- (g) calls on one context are ordered
def _process_packets_case(vp):
    """a host-form igd_process_packets (G = 4) whose field records fit the scratch the device-form call before it
    already sized; its expectation is computed, and its scratch sized, before that call is queued"""
    pk, sizes, law, gain, out_law = PF.make(40, 64, 1101, True)
    fields, want = PF.want_of(vp, pk, sizes, law, gain, out_law)
    check(vp.process_packets(pk, fields, law, gain, out_law), want)
    return (pk, fields, law, gain, out_law), want


def test_host_form_process_packets_waits_for_a_queued_device_form_gateway_call(vp):
    """igd_gateway_process keeps its gains in scratch slot 8 when gain_q7 is not wanted; a host-form process_packets
    right after it stages its field records there.  Both must come out as if run one after the other.  The gateway
    call is long and narrow (50 000 ticks of 128 bridges): its receive walk writes the first ticks' gains at once and
    runs for milliseconds before the fused kernel reads them."""
    F, B = 50000, 128
    c, x = device_case(F, B, 1201, N.ARB_CLIENT_PTT)
    want_gw, st_w = run_dev(vp, c, x, 0, want=("bmeter", "enc"))
    args, want_pp = _process_packets_case(vp)
    st = dev_states(states0(c))
    torch.cuda.synchronize()
    got_gw = call(vp, c, st, 0, want=("bmeter", "enc"), **x)  # queued, not waited for
    got_pp = vp.process_packets(*args)
    torch.cuda.synchronize()
    check(got_pp, want_pp)
    for k in want_gw:
        assert torch.equal(got_gw[k], want_gw[k]), k
    for a, b in zip(st, st_w):
        assert torch.equal(a, b)


def test_host_form_process_packets_waits_for_a_queued_device_form_fanout(vp):
    """the same with igd_gateway_fanout_packets, which keeps its sender plan in slot 8"""
    F, B, Gf = 1640, 4096, 4
    case = FP.make_case(40, 8, Gf, seed=1301)            # console packets and legs of 8 bridges, repeated below
    ticks = torch.arange(F, device=DEV) % 40
    rx = t(case["rx_pkts"])[ticks].repeat(1, B // 8, 1).contiguous()
    rsz = t(case["rx_sizes"].view(np.int32))[ticks].repeat(1, B // 8).contiguous()
    in_law, law = t(np.tile(case["in_law"], B // 8)), t(np.tile(case["law"], B // 8))
    rtp = t(synth.rtp12(F, B * Gf, np.where(np.tile(case["law"], B // 8) == 0, 8, 0)))
    st0 = t(np.tile(T.gpu_inputs(case), B // 8).view(np.uint8))
    args_f = (rx, in_law, law, rtp)

    def fanout(st):
        return vp.gateway_fanout_packets(*args_f, st, rx_sizes=rsz, now_ms0=case["now0"])

    st_w = st0.clone()
    torch.cuda.synchronize()
    want_f = fanout(st_w)
    torch.cuda.synchronize()
    args, want_pp = _process_packets_case(vp)
    st = st0.clone()
    torch.cuda.synchronize()
    got_f = fanout(st)                                   # queued, not waited for
    got_pp = vp.process_packets(*args)
    torch.cuda.synchronize()
    check(got_pp, want_pp)
    for k in want_f:
        assert torch.equal(got_f[k], want_f[k]), k
    assert torch.equal(st, st_w)
