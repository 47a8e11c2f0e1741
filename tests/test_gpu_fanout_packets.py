"""igd_gateway_fanout_packets: the console call's received ED-137 packets in (conference slot 0 of every bridge), a
finished ED-137 packet for every leg of the bridge out.  Checked (1) against the oracle end to end: the console frame
is the oracle's G.711 decode of the packet's payload in the call's law when the packet is a whole audio frame
(rx_arb_cases.frame_flag, the IGD_RXE_FRAME rule), digital silence otherwise, then the oracle path of
test_gpu_fanout.py (compressor per leg law, reference-pinned sender); (2) against the composition of the verified calls
it replaces (ed137_parse -> g711_decode -> silence on non-frames -> gateway_fanout) at a wide and a tall shape; (3) the
same-law identities; (4) state carry across calls, host form = device form, CUDA-graph capture together with
igd_gateway_process, a packet array beyond 2^32 bytes and argument errors."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle_py as O
import test_gpu_fanout as FO
import test_gpu_gateway as GW
import tx_scenarios as T
import igate4xsoftphonedsp_b200 as ig
from igate4xsoftphonedsp_b200 import _native as N
from igate4xsoftphonedsp_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
t = FO.t

# console packet kinds: PCMA, PCMU, keep-alive, absent, PT 18, short audio, unaccepted PT, 1043 bytes (still a whole
# frame), 1044 bytes (dropped)
KIND_P = [0.24, 0.24, 0.12, 0.08, 0.06, 0.06, 0.08, 0.06, 0.06]
KIND_PT = [8, 0, 123, 8, 18, 0, -1, 8, 0]
KIND_SIZE = [180, 180, 20, 0, 180, 100, 180, 1043, 1044]


def console_packets(F, B, rng):
    """rx_pkts u8 [F][B][180] (zero past each size), rx_sizes u32 [F][B]"""
    kind = rng.choice(len(KIND_P), (F, B), p=KIND_P)
    pt = np.asarray(KIND_PT)[kind]
    pt = np.where(pt < 0, rng.choice([3, 9, 96, 127], (F, B)), pt)
    sizes = np.asarray(KIND_SIZE, np.uint32)[kind]
    pk = rng.integers(0, 256, (F, B, 180), dtype=np.uint8)
    pk[..., 0] = 0x90                                            # v = 2, x = 1
    pk[..., 1] = pt | (rng.integers(0, 2, (F, B)) << 7)           # marker set at random
    pk[..., 12:16] = [0x01, 0x67, 0x00, 0x01]
    pk[np.arange(180)[None, None, :] >= sizes[..., None]] = 0
    return pk, sizes


def console_frames(pk, sizes, in_law):
    """the frame each bridge's legs send: the oracle's decode in the call's law, or PCM 0 without a whole frame"""
    sz = np.full(pk.shape[:2], 180, np.uint32) if sizes is None else sizes
    pt = pk[..., 1] & 0x7F
    frame = ((pt == 0) | (pt == 8)) & (sz >= 180) & (sz < 1044)           # rx_arb_cases.frame_flag, vectorised
    dec = [O.g711_decode(pk[..., 20:], lw) for lw in (N.LAW_ALAW, N.LAW_ULAW)]
    pcm = np.where((in_law != 0)[None, :, None], dec[1], dec[0])
    return np.where(frame[..., None], pcm, 0).astype(np.int16)


def make_case(F, B, G, seed, sizes=True):
    case = FO.make_case(F, B, G, seed)                 # leg laws, RTP headers, setter values, every call type
    rng = np.random.default_rng(seed + 1000)
    pk, sz = console_packets(F, B, rng)
    case.update(rx_pkts=pk, rx_sizes=sz if sizes else None, in_law=rng.integers(0, 2, B).astype(np.uint8))
    case["pcm"] = console_frames(pk, case["rx_sizes"], case["in_law"])   # what the oracle path of FO encodes
    return case


def fanout_pkts(vp, case, **kw):
    st = T.gpu_inputs(case)
    got = vp.gateway_fanout_packets(case["rx_pkts"], case["in_law"], case["law"], case["rtp12"], st,
                                    rx_sizes=case["rx_sizes"], tx_ctl=case["ctl"], now_ms0=case["now0"],
                                    tick_ms=case["tick_ms"], **kw)
    return got, st


# B per (G, F): F = 1 with an odd B leaves the packet array's size off a multiple of 16 (the last tile's window stops
# short of it); G = 7 starts tiles at every residue of bf0*180 mod 16; the last tile is partial wherever the shape
# allows it (not at G = 32 with an even F)
B_OF = {1: {1: 301, 8: 37, 60: 7}, 2: {1: 151, 8: 19, 60: 5}, 3: {1: 101, 8: 13, 60: 3}, 4: {1: 75, 8: 9, 60: 3},
        7: {1: 43, 8: 6, 60: 2}, 32: {1: 9, 8: 3, 60: 1}}


@pytest.mark.parametrize("G", [1, 2, 3, 4, 7, 32])
@pytest.mark.parametrize("F", [1, 8, 60])
@pytest.mark.parametrize("signed_char", [0, 1])
def test_fanout_packets_against_the_oracle(vp, G, F, signed_char):
    B = B_OF[G][F]
    assert (F * B * G) % 64 != 0 or (F * G) % 64 == 0      # G = 32 with an even F: every B gives whole tiles
    case = make_case(F, B, G, seed=10 * G + F, sizes=(G + F) % 3 != 0)
    flags = N.F_SIGNED_CHAR if signed_char else 0
    want_pk, want_sz, want_bm, ads = FO.oracle(case, signed_char)
    got, st = fanout_pkts(vp, case, flags=flags)
    assert np.array_equal(got["tx_sizes"], want_sz)
    assert np.array_equal(got["tx_pkts"], want_pk)            # all 180 bytes of every slot
    assert np.array_equal(got["tx_level"], want_bm)
    for c, a in enumerate(ads):
        for name in FO.STATE_FIELDS:
            assert int(st[name][c]) == int(getattr(a, name)), (c, name)
    _, _, _, st2 = FO.composed_host(vp, case, flags=flags)   # the whole state record (rtpFalse masked)
    assert FO.masked(st) == FO.masked(st2)


def composed_device(vp, x, st):
    """ed137_parse -> g711_decode in the console call's law -> PCM 0 where the packet is not a whole frame ->
    gateway_fanout: the host-side steps the call replaces"""
    F, B = x["rx"].shape[:2]
    fields, pay = vp.ed137_parse(x["rx"].reshape(F * B, 180), None if x["rsz"] is None else x["rsz"].reshape(-1))
    pcm = vp.g711_decode(pay.reshape(F, B, 160), x["in_law"])
    plen, pt, fl = (fields[:, 1] >> 16) & 0xFFFF, fields[:, 2] & 0xFF, (fields[:, 3] >> 24) & 0xFF
    frame = ((pt == 0) | (pt == 8)) & (plen == 160) & ((fl & 0x10) == 0)      # igd_fields_no_audio, negated
    pcm = torch.where(frame.view(F, B, 1), pcm, torch.zeros((), dtype=torch.int16, device=pcm.device)).contiguous()
    return vp.gateway_fanout(pcm, x["law"], x["rtp"], st, tx_ctl=x["ctl"], now_ms0=x["now0"])


def device_case(case):
    return dict(rx=t(case["rx_pkts"]), rsz=None if case["rx_sizes"] is None else t(case["rx_sizes"].view(np.int32)),
                in_law=t(case["in_law"]), law=t(case["law"]), rtp=t(case["rtp12"]), ctl=t(case["ctl"].view(np.uint8)),
                st0=t(T.gpu_inputs(case).view(np.uint8)), now0=case["now0"])


@pytest.mark.parametrize("B,G,F,sizes", [(16384, 4, 20, True), (16385, 4, 21, False), (1024, 4, 400, True),
                                         (333, 7, 401, True)])
def test_fanout_packets_equals_the_composition(vp, B, G, F, sizes):
    case = make_case(F, B, G, seed=B + G + F, sizes=sizes)
    x = device_case(case)
    st_a, st_b = x["st0"].clone(), x["st0"].clone()
    got = vp.gateway_fanout_packets(x["rx"], x["in_law"], x["law"], x["rtp"], st_a, rx_sizes=x["rsz"], tx_ctl=x["ctl"],
                                    now_ms0=x["now0"])
    want = composed_device(vp, x, st_b)
    torch.cuda.synchronize()
    for k in ("tx_sizes", "tx_pkts", "tx_level"):
        assert torch.equal(got[k], want[k]), k
    assert FO.masked(st_a.cpu().numpy().view(N.STATE_DT)) == FO.masked(st_b.cpu().numpy().view(N.STATE_DT))
    szn = got["tx_sizes"].cpu().numpy()
    assert (szn == 20).any() and (szn == 180).any()
    if F >= 37:                  # long enough for the keep-alive throttle to suppress packets
        assert (szn == 0).any()


def test_same_law_legs_carry_the_console_payload(vp):
    """every console packet a whole frame; every leg in its console call's law: an A-law leg's payload is the console
    payload, a u-law leg's too but for 0x7F (-0) -> 0xFF (+0)"""
    F, B, G = 40, 64, 4
    case = make_case(F, B, G, seed=77)
    rng = np.random.default_rng(78)
    case["in_law"] = (np.arange(B) % 2).astype(np.uint8)
    case["law"] = np.repeat(case["in_law"], G)
    pk = rng.integers(0, 256, (F, B, 180), dtype=np.uint8)
    pk[..., 0], pk[..., 1] = 0x90, np.where(case["in_law"] == 0, 8, 0)[None, :]
    pk[:, :, 20:40] = 0x7F                                         # -0 in every frame
    case["rx_pkts"], case["rx_sizes"] = pk, None
    got, _ = fanout_pkts(vp, case)
    sent = got["tx_sizes"] == 180
    cons = np.repeat(pk[..., 20:], G, axis=1)                      # [F][B*G][160] the console payload per leg
    ulaw = np.repeat(case["in_law"] == 1, G)
    assert sent[:, ulaw].any() and sent[:, ~ulaw].any()
    for c in range(B * G):
        rows = sent[:, c]
        want = cons[rows, c]
        if ulaw[c]:
            want = np.where(want == 0x7F, 0xFF, want)
        assert np.array_equal(got["tx_pkts"][rows, c, 20:], want), c


def test_state_carries_across_calls(vp):
    F, B, G = 60, 20, 4
    case = make_case(F, B, G, seed=41)
    whole, st_whole = fanout_pkts(vp, case)
    st = T.gpu_inputs(case)
    parts = {k: [] for k in whole}
    f0 = 0
    for nf in (1, 3, 8, 5, F - 17):  # both sides of the lane-walk switch
        sl = slice(f0, f0 + nf)
        got = vp.gateway_fanout_packets(case["rx_pkts"][sl], case["in_law"], case["law"], case["rtp12"][sl], st,
                                        rx_sizes=case["rx_sizes"][sl], tx_ctl=case["ctl"][sl],
                                        now_ms0=case["now0"] + f0 * case["tick_ms"])
        for k in parts:
            parts[k].append(got[k])
        f0 += nf
    assert f0 == F
    for k in parts:
        assert np.array_equal(np.concatenate(parts[k]), whole[k]), k
    assert st.tobytes() == st_whole.tobytes()


def test_host_form_equals_device_form_two_launches_per_call(vp):
    F, B, G = 40, 50, 4
    case = make_case(F, B, G, seed=51)
    n0 = vp.launch_count()
    host, st_h = fanout_pkts(vp, case)
    assert vp.launch_count() == n0 + 2
    x = device_case(case)
    st_d = x["st0"].clone()
    n1 = vp.launch_count()
    dev = vp.gateway_fanout_packets(x["rx"], x["in_law"], x["law"], x["rtp"], st_d, rx_sizes=x["rsz"], tx_ctl=x["ctl"],
                                    now_ms0=x["now0"])
    torch.cuda.synchronize()
    assert vp.launch_count() == n1 + 2
    assert np.array_equal(dev["tx_pkts"].cpu().numpy(), host["tx_pkts"])
    assert np.array_equal(dev["tx_sizes"].cpu().numpy().view(np.uint32), host["tx_sizes"])
    assert np.array_equal(dev["tx_level"].cpu().numpy(), host["tx_level"])
    assert st_d.cpu().numpy().tobytes() == st_h.tobytes()
    no_level, _ = fanout_pkts(vp, case, level=False)
    assert set(no_level) == {"tx_pkts", "tx_sizes"} and np.array_equal(no_level["tx_pkts"], host["tx_pkts"])


def test_full_duplex_tick_in_one_cuda_graph(vp):
    """igd_gateway_process (radios -> console) and igd_gateway_fanout_packets (console -> radios, its input the console
    call's received packets) captured into one graph for one tick; replayed over ticks whose packets change, it
    produces what the eager calls do, states carried.  (The graph holds the captured now_ms0: the eager calls use it.)"""
    T_TICKS, B, G = 6, 300, 4
    Cn = B * G
    gw = GW.make_case(T_TICKS, B, 91, N.ARB_CLIENT_PTT)
    fo = make_case(T_TICKS, B, G, seed=92)
    fo["in_law"] = gw["out_law"]                        # the console call has one codec in both directions
    now0 = gw["now0"]
    # per-tick inputs on the device, and the one-tick buffers the graph reads
    src = dict(g_pk=t(gw["pk"]), g_sz=t(gw["sizes"].view(np.int32)), g_rtp=t(gw["rtp12"]),
               g_ctl=t(gw["ctl"].view(np.int32).reshape(T_TICKS, B, 2)), f_pk=t(fo["rx_pkts"]),
               f_sz=t(fo["rx_sizes"].view(np.int32)), f_rtp=t(fo["rtp12"]), f_ctl=t(fo["ctl"].view(np.int32).reshape(T_TICKS, Cn, 2)))
    cur = {k: v[:1].clone() for k, v in src.items()}
    law, out_law, leg_law = t(gw["law"]), t(gw["out_law"]), t(fo["law"])
    g_tx0 = GW.tx_state_of(gw).view(np.int32).reshape(B, 10)
    f_tx0 = T.gpu_inputs(fo).view(np.int32).reshape(Cn, 10)
    rx_state, legs, bridges = t(np.zeros((Cn, 4), np.int32)), t(np.zeros((Cn, 2), np.int32)), t(np.zeros((B, 4), np.int32))
    g_tx, f_tx = t(g_tx0), t(f_tx0)

    def reset():
        rx_state.zero_(); legs.zero_(); bridges.zero_(); g_tx.copy_(t(g_tx0)); f_tx.copy_(t(f_tx0))

    def tick(g_out=None, f_out=None):
        g = vp.gateway_process(cur["g_pk"], law, out_law, rx_state, legs, bridges, cur["g_rtp"], g_tx, rx_sizes=cur["g_sz"],
                               tx_ctl=cur["g_ctl"], now_ms0=now0, want=("bmeter",), out=g_out)
        f = vp.gateway_fanout_packets(cur["f_pk"], out_law, leg_law, cur["f_rtp"], f_tx, rx_sizes=cur["f_sz"],
                                      tx_ctl=cur["f_ctl"], now_ms0=now0, out=f_out)
        return g, f

    def load(k):
        for name, v in src.items():
            cur[name].copy_(v[k:k + 1])

    vp.use_torch_stream()
    want = []
    for k in range(T_TICKS):         # eager; the first tick also sizes the scratch of both calls
        load(k)
        g, f = tick()
        torch.cuda.synchronize()
        want.append(({n: v.cpu().numpy().copy() for n, v in g.items()}, {n: v.cpu().numpy().copy() for n, v in f.items()}))
    want_states = [s.cpu().numpy().copy() for s in (rx_state, legs, bridges, g_tx, f_tx)]
    reset()
    load(0)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        vp.use_torch_stream()
        g_out, f_out = tick()        # warm-up on the side stream
    torch.cuda.synchronize()
    reset()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        vp.use_torch_stream()
        tick(g_out, f_out)
    vp.use_torch_stream()
    reset()
    for k in range(T_TICKS):
        load(k)
        for v in list(g_out.values()) + list(f_out.values()):
            v.zero_()
        gr.replay()
        torch.cuda.synchronize()
        for n, v in g_out.items():
            assert np.array_equal(v.cpu().numpy(), want[k][0][n]), (k, "process", n)
        for n, v in f_out.items():
            assert np.array_equal(v.cpu().numpy(), want[k][1][n]), (k, "fanout", n)
    for got_s, want_s in zip((rx_state, legs, bridges, g_tx, f_tx), want_states):
        assert np.array_equal(got_s.cpu().numpy(), want_s)
    assert (np.concatenate([w[1]["tx_sizes"] for w in want]) == 180).any()


def test_packet_array_beyond_4_gib(vp):
    """F = 1640 ticks of 4096 bridges x 4 legs: 4.8 GB of packets out of 1.2 GB of console packets; 64 bridges (the
    last among them) checked against the oracle over every tick"""
    F, B, G = 1640, 4096, 4
    Cn = B * G
    rng = np.random.default_rng(81)
    gen = torch.Generator(device=DEV).manual_seed(81)
    rx = torch.randint(0, 256, (F, B, 180), dtype=torch.uint8, device=DEV, generator=gen)
    pts = torch.tensor([8, 0, 123, 18, 96], dtype=torch.uint8, device=DEV)
    kind = torch.randint(0, 5, (F, B), device=DEV, generator=gen)
    rx[..., 0] = 0x90
    rx[..., 1] = pts[kind]
    rsz = torch.where(kind == 2, 20, 180).to(torch.int32)
    rsz = torch.where(torch.rand((F, B), device=DEV, generator=gen) < 0.05, torch.zeros_like(rsz), rsz)
    in_law = rng.integers(0, 2, B).astype(np.uint8)
    law = rng.integers(0, 2, Cn).astype(np.uint8)
    rtp12 = synth.rtp12(F, Cn, np.where(law == 0, 8, 0))
    ctl = T._random_ctl(F, Cn, 82, p_hold=0.95)
    legs = FO.make_legs(Cn, 83)
    now0 = 1_000_000
    st = t(T.gpu_inputs(dict(legs=legs, now0=now0)).view(np.uint8))
    got = vp.gateway_fanout_packets(rx, t(in_law), t(law), t(rtp12), st, rx_sizes=rsz, tx_ctl=t(ctl.view(np.uint8)),
                                    now_ms0=now0)
    torch.cuda.synchronize()
    assert got["tx_pkts"].numel() > 2 ** 32
    st_np = st.cpu().numpy().view(N.STATE_DT)
    for b in sorted(set(rng.choice(B - 1, 63, replace=False).tolist()) | {B - 1}):
        cs = slice(b * G, (b + 1) * G)
        pk_b, sz_b = rx[:, b:b + 1].cpu().numpy(), rsz[:, b:b + 1].cpu().numpy().view(np.uint32)
        case = dict(F=F, B=1, G=G, pcm=console_frames(pk_b, sz_b, in_law[b:b + 1]), law=law[cs], rtp12=rtp12[:, cs],
                    ctl=ctl[:, cs], legs=legs[cs], now0=now0, tick_ms=20)
        want_pk, want_sz, want_bm, ads = FO.oracle(case)
        assert np.array_equal(got["tx_sizes"][:, cs].cpu().numpy().view(np.uint32), want_sz), b
        assert np.array_equal(got["tx_pkts"][:, cs].cpu().numpy(), want_pk), b
        assert np.array_equal(got["tx_level"][:, cs].cpu().numpy(), want_bm), b
        for g, a in enumerate(ads):
            for name in FO.STATE_FIELDS:
                assert int(st_np[name][b * G + g]) == int(getattr(a, name)), (b, g, name)


def test_argument_errors_launch_nothing(vp):
    F, B, G = 2, 3, 4
    Cn = B * G
    rx = torch.zeros((F * B * 180 + 16,), dtype=torch.uint8, device=DEV)
    rsz = torch.zeros((F * B + 1,), dtype=torch.int32, device=DEV)
    in_law = torch.zeros(B, dtype=torch.uint8, device=DEV)
    law = torch.zeros(Cn, dtype=torch.uint8, device=DEV)
    rtp = torch.zeros((F, Cn, 12), dtype=torch.uint8, device=DEV)
    st = t(ig.make_state(Cn).view(np.uint8))
    pk = torch.zeros((F, Cn, 180), dtype=torch.uint8, device=DEV)
    sz = torch.zeros((F, Cn), dtype=torch.int32, device=DEV)
    vp.use_torch_stream()

    def call(**over):
        d = dict(struct_size=C.sizeof(N.FanoutPktDesc), mem=N.MEM_DEVICE, F=F, B=B, G=G, flags=0, tick_ms=20, reserved=0,
                 now_ms0=0, rx_pkts=rx.data_ptr(), rx_sizes=rsz.data_ptr(), in_law=in_law.data_ptr(), law=law.data_ptr(),
                 tx_rtp12=rtp.data_ptr(), tx_ctl=None, tx_state=st.data_ptr(), tx_pkts=pk.data_ptr(),
                 tx_sizes=sz.data_ptr(), tx_level=None)
        d.update(over)
        return vp._lib.igd_gateway_fanout_packets(vp._h, C.byref(N.FanoutPktDesc(**d)))

    n0 = vp.launch_count()
    assert call() == 0 and vp.launch_count() == n0 + 2
    assert call(rx_sizes=None) == 0 and vp.launch_count() == n0 + 4
    for over in (dict(G=0), dict(G=33), dict(flags=N.F_REF_QUIRKS), dict(flags=N.F_WALK_SERIAL), dict(flags=0x100),
                 dict(rx_pkts=None), dict(in_law=None), dict(law=None), dict(tx_pkts=None), dict(tx_state=None),
                 dict(tx_sizes=None), dict(tx_rtp12=None),
                 dict(rx_pkts=rx.data_ptr() + 4), dict(tx_pkts=pk.data_ptr() + 4), dict(tx_state=st.data_ptr() + 4),
                 dict(tx_ctl=st.data_ptr() + 4), dict(tx_rtp12=rtp.data_ptr() + 2), dict(tx_sizes=sz.data_ptr() + 2),
                 dict(rx_sizes=rsz.data_ptr() + 2), dict(F=-1), dict(B=-1), dict(B=1 << 26, G=32),
                 dict(struct_size=C.sizeof(N.FanoutPktDesc) - 8)):
        n = vp.launch_count()
        assert call(**over) == -22, over
        assert vp.launch_count() == n, over
    for over in (dict(F=0), dict(B=0)):
        n = vp.launch_count()
        assert call(**over) == 0 and vp.launch_count() == n, over
    torch.cuda.synchronize()
