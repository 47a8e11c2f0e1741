"""The product shim is a real `pjmedia_transport`: a PJSIP-role driver (tests/host_cpp/vtable_driver.cpp) creates
adapters through the reference's factory signature and drives them ONLY through `tp->op->...`, the RTP callback
registered with the slave transport, and the reference's public functions -- the same moves
oracle/ref_harness.cpp makes on the REFERENCE'S OWN adapter (TransportAdapter.cpp compiled from
/root/reference).  Packets, forwarded stream packets, latched words, levels and events must be equal.
Where oracle/_ref is absent the oracle (pinned to the reference by tests/test_ref_pins.py) stands in."""
import ctypes as C

import numpy as np
import pytest

import keepalive_cases as K
import oracle_py as O
import ref_py as RP
import rx_arb_cases as R
import shim_py as SP
import tx_scenarios as T
import igate4xsoftphonedsp_b200 as ig
from igate4xsoftphonedsp_b200 import _native as N


def test_vtable_driver_builds_and_refuses_without_gpu_or_opens_with_one():
    S = SP.lib()
    bank = S.shimta_open(0, 4)
    if bank:                      # GPU box
        S.shimta_close(bank)
    else:                         # no sm_100 device: no bank, no fallback
        assert S.shimta_create(1, 0, b"TRx", 1, b"i", b"TRx", 200, 1, 0, 1) is None


def reference_tx(s):
    if RP.available():
        pk, sz, bm, _ = RP.run_tx(s)
        return pk, sz, bm, "reference"
    pk, sz, bm, _ = T.run_oracle(s)
    return pk, sz, bm, "oracle"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["trx_out_gated", "rx_in_sql", "rxonly_out", "tx_in_recorder", "idle_in", "nonradio",
                                  "slave_switch", "keepalive_fast_tick", "no_ctl_idle_keepalive", "fuzz64"])
def test_send_path_through_vtable_equals_reference(name):
    s = [x for x in T.SCENARIOS if x["name"] == name][0]
    pk, sz, level = SP.run_tx(s, ig.F_REF_QUIRKS)
    wpk, wsz, wbm, _ = reference_tx(s)
    assert np.array_equal(sz, wsz)
    assert np.array_equal(pk, wpk)
    # trx->OutgoingRTP keeps its last value between audio packets (roip_ed137.cpp:6519-6534)
    F, Cn = sz.shape
    for c in range(Cn):
        last = 0
        for f in range(F):
            if wsz[f, c] and (wpk[f, c, 1] & 0x7F) != 123:
                last = int(wbm[f, c])
            assert level[f, c] == last, (f, c)


@pytest.mark.gpu
def test_receive_path_through_vtable_equals_reference():
    """slave transport -> registered RTP callback -> (tick) -> stream callback, latched word, r2sPacket, edges"""
    S = SP.lib()
    pkts, sizes, present = R.make_rx_stream(120, 12, seed=6)
    sizes = R.ref_comparable_sizes(sizes)
    F, Cn = sizes.shape
    now0, tick = 1000, 20
    want_ev, want_st = (RP.run_rx if RP.available() else R.oracle_rx_walk)(pkts, sizes, present, now0=now0, tick=tick,
                                                                           wd_ticks=2)
    bank = S.shimta_open(0, Cn)
    assert bank
    leg = dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200)
    hs = [SP.create(S, leg, 0, call_id=c) for c in range(Cn)]
    word = C.c_uint32()
    fsize = C.c_size_t()
    fwd = np.zeros(512, np.uint8)
    for f in range(F):
        now = now0 + f * tick
        S.shimta_set_clock(now)
        for c in range(Cn):
            if present[f, c]:
                n = int(sizes[f, c])
                p = np.zeros(max(n, 180), np.uint8)
                p[:180] = pkts[f, c]
                assert S.shimta_rx(hs[c], p.ctypes.data, n) == 0
        assert S.shimta_flush_rx(bank) == int(present[f].sum())
        if f % 2 == 1:
            assert S.shimta_watchdog(bank, 200) >= 0
        for c in range(Cn):
            fl = int(want_ev["flags"][f, c])
            nf = S.shimta_take_stream(hs[c], fwd.ctypes.data, C.byref(fsize))
            assert nf == (1 if fl & N.RXE_AUDIO else 0), (f, c)
            if nf:                                      # the stream gets the packet as received (:301)
                n = min(int(sizes[f, c]), 180)
                assert fsize.value == n and np.array_equal(fwd[:n], pkts[f, c, :n])
            ev = S.shimta_take_events(hs[c], C.byref(word))
            assert bool(ev & N.RXE_EDGE) == bool(fl & N.RXE_EDGE), (f, c)
            assert bool(ev & N.RXE_HANGUP) == bool(fl & N.RXE_HANGUP), (f, c)
            assert S.shimta_get_ed137_value(hs[c]) == int(want_ev["word"][f, c]), (f, c)
    for c in range(Cn):
        assert S.shimta_getR2SStatus(hs[c]) == int(want_st["r2sPacket"][c])
        S.shimta_destroy(hs[c])
    S.shimta_set_clock(777000)
    assert S.shimta_getR2SStatus(None) == 777000 - 3000          # TransportAdapter.cpp:324
    assert S.shimta_get_ed137_value(None) == 0                   # :345
    S.shimta_close(bank)


@pytest.mark.gpu
def test_two_packets_between_ticks_are_both_processed():
    """a jitter burst: the reference handles each packet in its callback; the shim queues and runs two rounds"""
    S = SP.lib()
    bank = S.shimta_open(0, 2)
    h = SP.create(S, dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200), 0, call_id=0)
    L = O.lib()
    a = np.zeros(180, np.uint8)
    b = np.zeros(20, np.uint8)
    L.orc_hdr_write(a.ctypes.data, 2, 0, 1, 0, 0, 8, 1, 160, 9, 0x0167, 1, 0x20013100)
    a[20:] = 0xD5
    L.orc_hdr_write(b.ctypes.data, 2, 0, 1, 0, 0, 123, 2, 320, 9, 0x0167, 1, 0x00413100)
    S.shimta_set_clock(5000)
    S.shimta_rx(h, a.ctypes.data, 180)
    S.shimta_rx(h, b.ctypes.data, 20)
    assert S.shimta_flush_rx(bank) == 2
    assert S.shimta_take_stream(h, None, None) == 1                       # only the audio packet is forwarded
    assert S.shimta_get_ed137_value(h) == 0x00413100                      # the later packet's word
    assert S.shimta_take_events(h, None) & N.RXE_EDGE                      # audio -> keep-alive edge
    lv = (C.c_int * 7)()
    S.shimta_levels(h, lv)
    assert lv[0] == 0xD5
    S.shimta_destroy(h)
    S.shimta_close(bank)


@pytest.mark.gpu
def test_sendR2SStatus_through_shim_equals_reference():
    """the reference signature `void sendR2SStatus(pjmedia_transport*)` (TransportAdapter.h:38): per adapter and
    as one bank-wide launch; state left behind by earlier transport_send_rtp calls included"""
    S = SP.lib()
    legs, hdr, ctl = K.make(24, 60, seed=5)
    now0, tick = 10_000, 40
    # history: three send_rtp ticks first (they leave the stamped header in the send buffer), then keep-alives
    s = dict(legs=[dict(l, slave=l["slave"]) for l in legs], F=3, ctl=ctl[:3], tick_ms=20, now0=now0 - 60,
             payload=np.random.default_rng(1).integers(0, 256, (3, 24, 160), dtype=np.uint8),
             rtp12=__import__("igate4xsoftphonedsp_b200").synth.rtp12(3, 24, [8] * 24), name="hist")
    if RP.available():
        Rf = RP.lib(0)
        want = np.zeros((60, 24, 20), np.uint8)
        wsz = np.zeros((60, 24), np.uint32)
        out = np.zeros(512, np.uint8)
        for c, leg in enumerate(legs):
            Rf.refapp_reset(RP.SERVER, 1)
            h = RP.create(Rf, leg, s["now0"], call_id=7)
            if leg["slave"] is not None:
                Rf.refta_setTxRxSlaveEnable(h, leg["slave"][0], leg["slave"][1])
            for f in range(3):
                k = ctl[f, c]
                Rf.refta_setAdapterPtt(h, int(k["pttstatus"]), int(k["pttpriority"]), int(k["callRecorder"]))
                Rf.refta_setAdapterQslOn(h, int(k["sqlstatus"]), 0, int(k["ed137_bssi"]))
                Rf.refta_setAdapterPttId(h, int(k["pttid"]))
                pkt = np.concatenate([s["rtp12"][f, c], s["payload"][f, c]])
                Rf.refta_set_clock(s["now0"] + f * 20)
                Rf.refta_send_rtp(h, pkt.ctypes.data, pkt.size, out.ctypes.data, None)
            for t in range(60):
                k = ctl[t, c]
                Rf.refta_setAdapterPtt(h, int(k["pttstatus"]), int(k["pttpriority"]), int(k["callRecorder"]))
                Rf.refta_setAdapterQslOn(h, int(k["sqlstatus"]), 0, int(k["ed137_bssi"]))
                Rf.refta_setAdapterPttId(h, int(k["pttid"]))
                Rf.refta_set_clock(now0 + t * tick)
                n = Rf.refta_sendR2SStatus(h, out.ctypes.data)
                wsz[t, c] = n
                want[t, c, :n] = out[:n]
            Rf.refta_destroy(h)
    else:                                                        # the same moves on the oracle's adapters
        L = O.lib()
        _, _, _, ads = T.run_oracle(s)                           # the three send_rtp ticks of the history
        want = np.zeros((60, 24, 20), np.uint8)
        wsz = np.zeros((60, 24), np.uint32)
        out = np.zeros(512, np.uint8)
        for c, a in enumerate(ads):
            for t in range(60):
                k = ctl[t, c]
                L.orc_setAdapterPtt(C.byref(a), int(k["pttstatus"]), int(k["pttpriority"]), int(k["callRecorder"]))
                L.orc_setAdapterQslOn(C.byref(a), int(k["sqlstatus"]), 0, int(k["ed137_bssi"]))
                L.orc_setAdapterPttId(C.byref(a), int(k["pttid"]))
                n = L.orc_sendR2SStatus(C.byref(a), now0 + t * tick, out.ctypes.data)
                wsz[t, c] = n
                want[t, c, :n] = out[:n]
    for bankwide in (False, True):
        bank = S.shimta_open(0, 24)
        hs = []
        for c, leg in enumerate(legs):
            hs.append(SP.create(S, leg, s["now0"], call_id=c))
            if leg["slave"] is not None:
                S.shimta_setTxRxSlaveEnable(hs[c], leg["slave"][0], leg["slave"][1])
        out = np.zeros(512, np.uint8)

        def setters(c, k):
            S.shimta_setAdapterPtt(hs[c], int(k["pttstatus"]), int(k["pttpriority"]), int(k["callRecorder"]))
            S.shimta_setAdapterQslOn(hs[c], int(k["sqlstatus"]), 0, int(k["ed137_bssi"]))
            S.shimta_setAdapterPttId(hs[c], int(k["pttid"]))
        for f in range(3):
            S.shimta_set_clock(s["now0"] + f * 20)
            for c in range(24):
                setters(c, ctl[f, c])
                pkt = np.concatenate([s["rtp12"][f, c], s["payload"][f, c]])
                S.shimta_send_rtp(hs[c], pkt.ctypes.data, pkt.size)
            S.shimta_flush_tx(bank, ig.F_REF_QUIRKS)
            for c in range(24):
                S.shimta_take_sent(hs[c], out.ctypes.data)
        for t in range(60):
            S.shimta_set_clock(now0 + t * tick)
            for c in range(24):
                setters(c, ctl[t, c])
                if not bankwide:
                    S.shimta_sendR2SStatus(hs[c])
            if bankwide:
                assert S.shimta_bank_keepalive(bank) == int((wsz[t] > 0).sum())
            for c in range(24):
                n = S.shimta_take_sent(hs[c], out.ctypes.data)
                assert n == wsz[t, c], (t, c, bankwide)
                assert np.array_equal(out[:n], want[t, c, :n]), (t, c, bankwide)
        for h in hs:
            S.shimta_destroy(h)
        S.shimta_close(bank)
    assert (wsz == 20).sum() > 200


@pytest.mark.gpu
def test_vtable_layout_passthrough_sdp_and_channel_reuse():
    S = SP.lib()
    bank = S.shimta_open(0, 2)
    h = SP.create(S, dict(radiocall=1, callIn=0, calltype="Rxonly", keepalive=150), 0, call_id=2)
    assert S.shimta_transport_type(h) == 4                       # PJMEDIA_TRANSPORT_TYPE_USER + 1 (:101-102)
    bits = S.shimta_vtable_passthrough(h)
    buf = C.create_string_buffer(1024)
    S.shimta_encode_sdp(h, buf, 1024)
    sdp_rxonly = buf.value.decode()
    S.shimta_setCallType(h, b"TRx")
    S.shimta_encode_sdp(h, buf, 1024)
    sdp_trx = buf.value.decode()
    cnt = (C.c_int * 16)()
    S.shimta_counters(h, cnt)
    if RP.available():                                           # the same moves on the reference's adapter
        Rf = RP.lib(0)
        Rf.refapp_reset(RP.SERVER, 1)
        rh = RP.create(Rf, dict(radiocall=1, callIn=0, calltype="Rxonly", keepalive=150), 0, call_id=2)
        assert bits == Rf.refta_vtable_passthrough(rh)
        Rf.refta_encode_sdp(rh, buf, 1024)
        assert sdp_rxonly == buf.value.decode()
        Rf.refta_setCallType(rh, b"TRx")
        Rf.refta_encode_sdp(rh, buf, 1024)
        assert sdp_trx == buf.value.decode()
        rcnt = (C.c_int * 16)()
        Rf.refta_counters(rh, rcnt)
        assert list(cnt) == list(rcnt)
        Rf.refta_destroy(rh)
    assert sdp_rxonly == RP.SDP_RXONLY_150
    assert cnt[RP.COUNTERS_ATTACH] == 1 and cnt[RP.COUNTERS_ENCODE_SDP] == 2
    assert bits == 0b0111_0111_0001
    assert "ptt-id:1\n" in sdp_trx and "ptt-id" not in sdp_rxonly and "R2S-KeepAlivePeriod:150\n" in sdp_rxonly
    rtcp = np.zeros(8, np.uint8)
    assert S.shimta_rtcp(h, rtcp.ctypes.data, 8) == 1            # RTCP goes straight to the stream (:327-335)
    # destroy gives the channel back: a bank of 2 can host more than 2 adapters over time
    h2 = SP.create(S, dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200), 0, call_id=3)
    assert S.shimta_create(1, 0, b"TRx", 4, b"i", b"TRx", 200, 1, 0, 1) is None      # bank full
    S.shimta_destroy(h)                                          # closes the slave too (del_base)
    h3 = SP.create(S, dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200), 0, call_id=5)
    S.shimta_destroy(h2)
    S.shimta_destroy(h3)
    S.shimta_close(bank)
