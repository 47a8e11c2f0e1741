"""igd_gateway_fanout: one PCM frame per bridge and tick in (conference slot 0), a finished ED-137 packet for every leg of
the bridge out, each in its leg's law and with its leg's sender state.  Checked (1) against the oracle end to end: the
G.711 compressor on each bridge frame in each leg's law, then the reference-pinned sender (transport_send_rtp, clean
mode); (2) against the composition of the verified calls it replaces (igd_g711_encode_ch over the replicated PCM, then
igd_ed137_pack); (3) for state carry across calls, host form = device form, two launches per call, CUDA-graph capture,
a packet array beyond 2^32 bytes and argument errors."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle_py as O
import tx_scenarios as T
import igate4xsoftphonedsp_b200 as ig
from igate4xsoftphonedsp_b200 import _native as N
from igate4xsoftphonedsp_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SLAVES = [None, (1, 0), (0, 1), (1, 1)]
# sender fields the oracle's adapter shares with igd_ed137_state (rtpFalse is not maintained by the fan-out)
STATE_FIELDS = ("packetCnt", "firstR2SPacket", "trxSlaveEnableChangedCount", "r2sSendtime", "rxSlaveEnable",
                "txSlaveEnable", "pttstatus", "sqlstatus")


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def make_legs(Cn, seed):
    """every call type, both call directions, keep-alive periods of 40 and 200 ms, slave-enable changes"""
    rng = np.random.default_rng(seed)
    return [dict(radiocall=1, callIn=(c // 3) % 2, calltype=T.CALLTYPES[(c + seed) % len(T.CALLTYPES)],
                 keepalive=(40, 200)[(c // 2) % 2], slave=SLAVES[int(rng.integers(0, 4))]) for c in range(Cn)]


def make_case(F, B, G, seed, ctl=True):
    rng = np.random.default_rng(seed)
    Cn = B * G
    pcm = rng.integers(-32768, 32768, (F, B, 160), dtype=np.int16)
    pcm[:, ::5] //= 64                       # quieter frames
    pcm[::4, ::3] = 0                        # digital silence
    law = rng.integers(0, 2, Cn).astype(np.uint8)        # laws mixed inside a bridge
    return dict(F=F, B=B, G=G, pcm=pcm, law=law, rtp12=synth.rtp12(F, Cn, np.where(law == 0, 8, 0)),
                ctl=T._random_ctl(F, Cn, seed + 1, p_hold=0.85) if ctl else None, legs=make_legs(Cn, seed),
                now0=1_000_000, tick_ms=20)


def oracle(case, signed_char=0):
    """(pkts [F][C][180], sizes [F][C], levels [F][C], adapters): O.g711_encode of each bridge frame in each leg's law,
    through the reference-pinned sender and its clean (no Q2 / Q3) expectation"""
    G = case["G"]
    Cn = case["law"].size
    enc = [O.g711_encode(case["pcm"], lw) for lw in (N.LAW_ALAW, N.LAW_ULAW)]
    leg_b = np.arange(Cn) // G
    payload = np.where((case["law"] == 0)[None, :, None], enc[0][:, leg_b], enc[1][:, leg_b])
    s = dict(name="fanout", legs=case["legs"], F=case["F"], ctl=case["ctl"], tick_ms=case["tick_ms"], now0=case["now0"],
             payload=payload, rtp12=case["rtp12"])
    pk, sz, _, ads = T.run_oracle(s, signed_char)
    pk, bm = T.clean_expectation(s, pk, sz, signed_char)
    return pk, sz, bm, ads


def masked(st):
    st = st.copy()
    st["rtpFalse"] = 0
    return st.tobytes()


def fanout(vp, case, **kw):
    st = T.gpu_inputs(case)
    got = vp.gateway_fanout(case["pcm"], case["law"], case["rtp12"], st, tx_ctl=case["ctl"], now_ms0=case["now0"],
                            tick_ms=case["tick_ms"], **kw)
    return got, st


def composed_host(vp, case, flags=0):
    codes = vp.g711_encode(np.repeat(case["pcm"], case["G"], axis=1), case["law"])
    st = T.gpu_inputs(case)
    pk, sz, bm = vp.ed137_pack(case["rtp12"], codes, st, ctl=case["ctl"], now_ms0=case["now0"], tick_ms=case["tick_ms"],
                               flags=flags)
    return pk, sz, bm, st


@pytest.mark.parametrize("G,B,F,seed", [(1, 16, 60, 1), (2, 9, 7, 2), (4, 6, 8, 3), (4, 10, 1, 4), (7, 3, 60, 5),
                                        (32, 2, 1, 6), (32, 2, 60, 7), (7, 4, 8, 8)])
@pytest.mark.parametrize("signed_char", [0, 1])
def test_fanout_against_the_oracle(vp, G, B, F, seed, signed_char):
    case = make_case(F, B, G, seed)
    want_pk, want_sz, want_bm, ads = oracle(case, signed_char)
    got, st = fanout(vp, case, flags=N.F_SIGNED_CHAR if signed_char else 0)
    assert np.array_equal(got["tx_sizes"], want_sz)
    assert np.array_equal(got["tx_pkts"], want_pk)            # all 180 bytes of every slot
    assert np.array_equal(got["tx_level"], want_bm)
    for c, a in enumerate(ads):
        for name in STATE_FIELDS:
            assert int(st[name][c]) == int(getattr(a, name)), (c, name)
    # the whole state record against the composition of the verified calls (rtpFalse masked)
    _, _, _, st2 = composed_host(vp, case, flags=N.F_SIGNED_CHAR if signed_char else 0)
    assert masked(st) == masked(st2)


@pytest.mark.parametrize("B,G,F", [(8192, 4, 37), (300, 32, 40), (1024, 4, 200), (50, 3, 5)])
def test_fanout_equals_encode_then_pack(vp, B, G, F):
    case = make_case(F, B, G, seed=B + G + F)
    st0 = T.gpu_inputs(case)
    pcm, law, rtp, ctl = t(case["pcm"]), t(case["law"]), t(case["rtp12"]), t(case["ctl"].view(np.uint8))
    st_a, st_b = t(st0.view(np.uint8)), t(st0.view(np.uint8))
    got = vp.gateway_fanout(pcm, law, rtp, st_a, tx_ctl=ctl, now_ms0=case["now0"])
    codes = vp.g711_encode(pcm.repeat_interleave(G, dim=1).contiguous(), law)
    pk, sz, bm = vp.ed137_pack(rtp, codes, st_b, ctl=ctl, now_ms0=case["now0"])
    torch.cuda.synchronize()
    assert torch.equal(got["tx_sizes"], sz)
    assert torch.equal(got["tx_pkts"], pk)
    assert torch.equal(got["tx_level"], bm)
    a = st_a.cpu().numpy().view(N.STATE_DT)
    b = st_b.cpu().numpy().view(N.STATE_DT)
    assert masked(a) == masked(b)
    if F >= 37:                  # suppressed, keep-alive and audio packets all occur
        szn = sz.cpu().numpy()
        assert (szn == 0).any() and (szn == 20).any() and (szn == 180).any()


def test_state_carries_across_calls(vp):
    F, B, G = 60, 20, 4
    case = make_case(F, B, G, seed=41)
    whole, st_whole = fanout(vp, case)
    st = T.gpu_inputs(case)
    parts = {k: [] for k in whole}
    f0 = 0
    for nf in (1, 3, 8, F - 12):     # both sides of the lane-walk switch
        sl = slice(f0, f0 + nf)
        got = vp.gateway_fanout(case["pcm"][sl], case["law"], case["rtp12"][sl], st, tx_ctl=case["ctl"][sl],
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
    host, st_h = fanout(vp, case)
    assert vp.launch_count() == n0 + 2
    st_d = t(T.gpu_inputs(case).view(np.uint8))
    n1 = vp.launch_count()
    dev = vp.gateway_fanout(t(case["pcm"]), t(case["law"]), t(case["rtp12"]), st_d, tx_ctl=t(case["ctl"].view(np.uint8)),
                            now_ms0=case["now0"])
    torch.cuda.synchronize()
    assert vp.launch_count() == n1 + 2
    assert np.array_equal(dev["tx_pkts"].cpu().numpy(), host["tx_pkts"])
    assert np.array_equal(dev["tx_sizes"].cpu().numpy().view(np.uint32), host["tx_sizes"])
    assert np.array_equal(dev["tx_level"].cpu().numpy(), host["tx_level"])
    assert st_d.cpu().numpy().tobytes() == st_h.tobytes()
    # without the level output
    no_level, _ = fanout(vp, case, level=False)
    assert set(no_level) == {"tx_pkts", "tx_sizes"} and np.array_equal(no_level["tx_pkts"], host["tx_pkts"])


@pytest.mark.parametrize("F", [1, 24])
def test_fanout_call_is_cuda_graph_capturable(vp, F):
    B, G = 300, 4
    case = make_case(F, B, G, seed=61 + F)
    st0 = t(T.gpu_inputs(case).view(np.uint8))
    st = st0.clone()
    args = (t(case["pcm"]), t(case["law"]), t(case["rtp12"]), st)
    kw = dict(tx_ctl=t(case["ctl"].view(np.uint8)), now_ms0=case["now0"])

    vp.use_torch_stream()
    eager = vp.gateway_fanout(*args, **kw)
    torch.cuda.synchronize()
    want = {k: v.cpu().numpy().copy() for k, v in eager.items()}
    want_st = st.cpu().numpy().copy()
    st.copy_(st0)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        vp.use_torch_stream()
        vp.gateway_fanout(*args, out=eager, **kw)       # warm-up on a side stream: sizes the scratch
    torch.cuda.synchronize()
    st.copy_(st0)
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        vp.use_torch_stream()
        vp.gateway_fanout(*args, out=eager, **kw)
    vp.use_torch_stream()
    for rep in range(2):
        st.copy_(st0)
        for v in eager.values():
            v.zero_()
        gr.replay()
        torch.cuda.synchronize()
        for k in want:
            assert np.array_equal(eager[k].cpu().numpy(), want[k]), (rep, k)
        assert np.array_equal(st.cpu().numpy(), want_st), rep


def test_packet_array_beyond_4_gib(vp):
    """F = 1640 ticks of 4096 bridges x 4 legs: 4.8 GB of packets; 64 bridges (the last among them) checked against
    the oracle over every tick"""
    F, B, G = 1640, 4096, 4
    Cn = B * G
    rng = np.random.default_rng(71)
    gen = torch.Generator(device=DEV).manual_seed(71)
    pcm = torch.randint(-32768, 32768, (F, B, 160), dtype=torch.int16, device=DEV, generator=gen)
    law = rng.integers(0, 2, Cn).astype(np.uint8)
    rtp12 = synth.rtp12(F, Cn, np.where(law == 0, 8, 0))
    ctl = T._random_ctl(F, Cn, 72, p_hold=0.95)
    legs = make_legs(Cn, 73)
    now0 = 1_000_000
    st = t(T.gpu_inputs(dict(legs=legs, now0=now0)).view(np.uint8))
    got = vp.gateway_fanout(pcm, t(law), t(rtp12), st, tx_ctl=t(ctl.view(np.uint8)), now_ms0=now0)
    torch.cuda.synchronize()
    assert got["tx_pkts"].numel() > 2 ** 32
    st_np = st.cpu().numpy().view(N.STATE_DT)
    for b in sorted(set(rng.choice(B - 1, 63, replace=False).tolist()) | {B - 1}):
        cs = slice(b * G, (b + 1) * G)
        case = dict(F=F, B=1, G=G, pcm=pcm[:, b:b + 1].cpu().numpy(), law=law[cs], rtp12=rtp12[:, cs], ctl=ctl[:, cs],
                    legs=legs[cs], now0=now0, tick_ms=20)
        want_pk, want_sz, want_bm, ads = oracle(case)
        assert np.array_equal(got["tx_sizes"][:, cs].cpu().numpy().view(np.uint32), want_sz), b
        assert np.array_equal(got["tx_pkts"][:, cs].cpu().numpy(), want_pk), b
        assert np.array_equal(got["tx_level"][:, cs].cpu().numpy(), want_bm), b
        for g, a in enumerate(ads):
            for name in STATE_FIELDS:
                assert int(st_np[name][b * G + g]) == int(getattr(a, name)), (b, g, name)


def test_argument_errors_launch_nothing(vp):
    F, B, G = 2, 3, 4
    Cn = B * G
    pcm = torch.zeros((F * B * 160 + 8,), dtype=torch.int16, device=DEV)
    law = torch.zeros(Cn, dtype=torch.uint8, device=DEV)
    rtp = torch.zeros((F, Cn, 12), dtype=torch.uint8, device=DEV)
    st = t(ig.make_state(Cn).view(np.uint8))
    pk = torch.zeros((F, Cn, 180), dtype=torch.uint8, device=DEV)
    sz = torch.zeros((F, Cn), dtype=torch.int32, device=DEV)
    vp.use_torch_stream()

    def call(**over):
        d = dict(struct_size=C.sizeof(N.FanoutDesc), mem=N.MEM_DEVICE, F=F, B=B, G=G, flags=0, tick_ms=20, reserved=0,
                 now_ms0=0, pcm=pcm.data_ptr(), law=law.data_ptr(), tx_rtp12=rtp.data_ptr(), tx_ctl=None,
                 tx_state=st.data_ptr(), tx_pkts=pk.data_ptr(), tx_sizes=sz.data_ptr(), tx_level=None)
        d.update(over)
        return vp._lib.igd_gateway_fanout(vp._h, C.byref(N.FanoutDesc(**d)))

    n0 = vp.launch_count()
    assert call() == 0 and vp.launch_count() == n0 + 2
    for over in (dict(G=0), dict(G=33), dict(flags=N.F_REF_QUIRKS), dict(flags=N.F_WALK_SERIAL), dict(tx_pkts=None),
                 dict(pcm=pcm.data_ptr() + 2), dict(tx_pkts=pk.data_ptr() + 4), dict(tx_state=st.data_ptr() + 4),
                 dict(F=-1), dict(B=1 << 26, G=32), dict(struct_size=C.sizeof(N.FanoutDesc) - 8)):
        n = vp.launch_count()
        assert call(**over) == -22, over
        assert vp.launch_count() == n, over
    for over in (dict(F=0), dict(B=0)):
        n = vp.launch_count()
        assert call(**over) == 0 and vp.launch_count() == n, over
    torch.cuda.synchronize()
