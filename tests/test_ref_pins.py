"""oracle == REFERENCE, for the in-repo state machines of the hot path.

The reference's own TransportAdapter.cpp (whole file) and the hot-path members of RoIP_ED137 (line ranges of
roip_ed137.cpp / Functions.cpp) are compiled from /root/reference under stub Qt/PJSIP headers into
oracle/_ref/libigd_ref_ta{,_sc}.so (oracle/Makefile, oracle/ref_harness.cpp) and driven the way PJSIP drives
them: tp->op->send_rtp, the RTP callback registered in tp->op->attach, the public setters.

  *_live tests   replay the shared seeded cases through that library and through oracle/igd_oracle.c and
                 compare arrays (they run wherever oracle/_ref/ is present: the build container and, since
                 the .so travels with gpurun, the GPU box);
  golden tests   compare the oracle with tests/golden/ref_pins.json, which tests/golden/make_golden.py
                 wrote FROM THE REFERENCE RUN (they need nothing but the oracle), and with
                 tests/golden/live_cases.json: the oracle's side of the remaining *_live comparisons, recorded
                 where they pass, so that a change to the oracle or to the shared cases is caught without the
                 reference build.
"""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import keepalive_cases as K
import oracle_py as O
import ref_py as RP
import rx_arb_cases as R
import tx_scenarios as T
from igate4xsoftphonedsp_b200 import _native as N

live = pytest.mark.skipif(not RP.available(), reason="oracle/_ref/libigd_ref_ta.so not built (no /root/reference here)")
L = O.lib()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def radio_mask(legs):
    return np.array([bool(l["radiocall"]) for l in legs])


# ----------------------------------------------------------------------------- transport_send_rtp
@live
@pytest.mark.parametrize("s", T.SCENARIOS, ids=[s["name"] for s in T.SCENARIOS])
def test_send_rtp_oracle_equals_reference_live(s):
    """packets, sizes, setOutgoingRTP level and the adapter state after the last frame: identical to what the
    reference's transport_send_rtp (TransportAdapter.cpp:635-874) hands its slave transport."""
    pk, sz, bm, ads = T.run_oracle(s)
    rpk, rsz, rbm, fin = RP.run_tx(s)
    assert np.array_equal(sz, rsz)
    assert np.array_equal(pk, rpk)
    assert np.array_equal(bm, rbm)
    assert sz.sum() > 0 or not radio_mask(s["legs"]).any()
    for a, r, leg in zip(ads, fin, s["legs"]):
        if not leg["radiocall"]:
            continue      # the reference's non-radio branch has no return statement (ref_harness.cpp: not executed)
        for f in RP.TX_STATE_FIELDS:
            assert getattr(a, f) == getattr(r, f), f
        assert bytes(a.send_pkt_buff) == bytes(r.send_pkt_buff)
        assert bytes(a.tmp_payload_buf) == bytes(r.tmp_payload_buf)
        assert a.send_payload_bufSize == r.send_payload_bufSize


@live
def test_send_rtp_signed_char_build_live():
    """quirk Q4: the x86 (`char` signed) build of the reference gives the signed byte-mean"""
    assert RP.lib(1).refta_char_is_signed() == 1 and RP.lib(0).refta_char_is_signed() == 0
    s = T.SCENARIOS[0]
    for sc in (0, 1):
        pk, sz, bm, _ = T.run_oracle(s, signed_char=sc)
        rpk, rsz, rbm, _ = RP.run_tx(s, signed_char=sc)
        assert np.array_equal(pk, rpk) and np.array_equal(sz, rsz) and np.array_equal(bm, rbm)
    assert not np.array_equal(T.run_oracle(s, 0)[2], T.run_oracle(s, 1)[2])


@live
def test_send_rtp_csrc_extension_padding_live():
    """pjmedia_rtp_decode_rtp's payload offset (CSRC list, header extension, padding: RFC 3550 5.1) as the
    sender uses it (TransportAdapter.cpp:651-654)."""
    Rf = RP.lib(0)
    rng = np.random.default_rng(4)
    leg = dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200)
    out, rout = np.zeros(512, np.uint8), np.zeros(512, np.uint8)
    for cc, x, extw in ((0, 0, 0), (2, 0, 0), (0, 1, 1), (1, 1, 2), (3, 0, 0)):
        pkt = np.zeros(12 + 4 * cc + (4 + 4 * extw if x else 0) + 160, np.uint8)
        pkt[:] = rng.integers(0, 256, pkt.size)
        pkt[0] = 0x80 | (x << 4) | cc
        pkt[1] = 8
        if x:
            pkt[12 + 4 * cc + 2] = 0
            pkt[12 + 4 * cc + 3] = extw
        a = O.Adapter()
        L.orc_adapter_init(C.byref(a), 1, 0, b"TRx", 200, 5000)
        L.orc_setAdapterPtt(C.byref(a), 1, 3, 0)
        Rf.refapp_reset(RP.SERVER, 1)
        h = RP.create(Rf, leg, 5000, call_id=7)
        Rf.refapp_server_bind(0, 7, 1, b"TRx")
        Rf.refta_setAdapterPtt(h, 1, 3, 0)
        n = L.orc_transport_send_rtp(C.byref(a), pkt.ctypes.data, pkt.size, 5000, out.ctypes.data, 1, 0)
        rn = Rf.refta_send_rtp(h, pkt.ctypes.data, pkt.size, rout.ctypes.data, None)
        assert n == rn and n == 20 + 160 and np.array_equal(out[:n], rout[:n])
        leg_rec = RP.Leg()
        Rf.refapp_get_leg(0, C.byref(leg_rec))
        assert leg_rec.OutgoingRTP == a.OutgoingRTP
        Rf.refta_destroy(h)


# ----------------------------------------------------------------------------- sendR2SStatus
@live
def test_sendR2SStatus_oracle_equals_reference_live():
    legs, hdr, ctl = K.make(40, 120, seed=2)
    pk, sz, hf = K.oracle_walk(legs, hdr, ctl)
    rpk, rsz, rhf = RP.run_keepalive(legs, hdr, ctl)
    assert np.array_equal(sz, rsz) and np.array_equal(pk, rpk) and np.array_equal(hf, rhf)
    assert (sz == 20).sum() > 1000


# ----------------------------------------------------------------------------- transport_rtp_cb
@live
def test_rtp_cb_walk_oracle_equals_reference_live():
    """latch, PT demux, drop rule, audio<->keep-alive edges (setIncomingED137Value -> checkEvents), r2sPacket
    stamps and the watchdog counts: the reference's callback (TransportAdapter.cpp:240-316) vs the oracle."""
    pkts, sizes, present = R.make_rx_stream(300, 24, seed=3)
    sizes = R.ref_comparable_sizes(sizes)
    ev, st = R.oracle_rx_walk(pkts, sizes, present)
    rev, rst = RP.run_rx(pkts, sizes, present)
    assert np.array_equal(ev, rev) and np.array_equal(st, rst)
    fl = ev["flags"]
    assert ((fl & N.RXE_EDGE) != 0).sum() > 50 and ((fl & N.RXE_DROPPED) != 0).sum() > 5
    assert ((fl & N.RXE_HANGUP) != 0).sum() > 0


@live
def test_rtp_cb_state_carry_live():
    pkts, sizes, present = R.make_rx_stream(120, 8, seed=9)
    sizes = R.ref_comparable_sizes(sizes)
    _, st_full = R.oracle_rx_walk(pkts, sizes, present)
    ev1, st1 = RP.run_rx(pkts[:50], sizes[:50], present[:50])
    ev2, st2 = RP.run_rx(pkts[50:], sizes[50:], present[50:], now0=1000 + 50 * 20, frame0=50, state0=st1)
    assert np.array_equal(st2, st_full)


@live
@pytest.mark.parametrize("signed_char", [0, 1])
def test_setIncomingRTP_bytemean_live(signed_char):
    """the reference's own setIncomingRTP (roip_ed137.cpp:6541-6587, SERVER mode) on payloads of several
    lengths incl. the 164 / 24 byte ones its dead `i = 4` skips name; payload as copied by the callback"""
    Rf = RP.lib(signed_char)
    rng = np.random.default_rng(21)
    leg = dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200)
    Rf.refapp_reset(RP.SERVER, 1)
    h = RP.create(Rf, leg, 0, call_id=5)
    Rf.refapp_server_bind(2, 5, 1, b"TRx")         # trx2->radio1
    a = O.Adapter()
    L.orc_adapter_init(C.byref(a), 1, 0, b"TRx", 200, 0)
    rec = RP.Leg()
    hdr = np.zeros(20, np.uint8)
    for n in (160, 164, 24, 1, 80, 256, 200):
        pkt = rng.integers(0, 256, 20 + n, dtype=np.uint8)
        if n == 80:
            pkt[20:] = rng.integers(128, 256, n)    # all "negative" chars
        L.orc_hdr_write(hdr.ctypes.data, 2, 0, 1, 0, 0, 8, 1, 160, 9, 0x0167, 1, 0x10013178)
        pkt[:20] = hdr
        assert L.orc_transport_rtp_cb(C.byref(a), pkt.ctypes.data, pkt.size, 40, 1, signed_char) == 1
        assert Rf.refta_rx(h, pkt.ctypes.data, pkt.size, pkt.size) == 1
        Rf.refapp_get_leg(2, C.byref(rec))
        assert rec.IncomingRTP == a.IncomingRTP, n
        assert rec.IncomingRTP == L.orc_bytemean(pkt[20:].ctypes.data, n, signed_char)
        s = RP.state(Rf, h)
        assert bytes(s.payload_buff)[:n] == bytes(a.payload_buff)[:n] and s.payload_bufSize == a.payload_bufSize == n
    Rf.refta_destroy(h)


@live
def test_non_radio_rtp_cb_live():
    """non-radio call: 12-byte header, nothing latched (TransportAdapter.cpp:267-275); forwarded to the stream"""
    Rf = RP.lib(0)
    leg = dict(radiocall=0, callIn=0, calltype="", keepalive=200)
    radio = dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200)
    Rf.refapp_reset(RP.CLIENT, 1)
    hr = RP.create(Rf, radio, 0, call_id=1)
    h = RP.create(Rf, leg, 0, call_id=2)
    rng = np.random.default_rng(2)
    pkt = rng.integers(0, 256, 172, dtype=np.uint8)
    pkt[0], pkt[1] = 0x80, 8
    # the reference tests the PT through a file-static pointer that only radio calls assign (:76, :246-262, :298):
    # give it a radio packet first so that the pointer is valid, as it is in a running gateway
    rp = rng.integers(0, 256, 180, dtype=np.uint8)
    rp[0], rp[1] = 0x90, 8
    assert Rf.refta_rx(hr, rp.ctypes.data, 180, 180) == 1
    assert Rf.refta_rx(h, pkt.ctypes.data, 172, 172) == 1
    a = O.Adapter()
    L.orc_adapter_init(C.byref(a), 0, 0, b"", 200, 0)
    assert L.orc_transport_rtp_cb(C.byref(a), pkt.ctypes.data, 172, 0, 0, 0) == 1
    s = RP.state(Rf, h)
    assert s.payload_bufSize == a.payload_bufSize == 160
    assert bytes(s.payload_buff)[:160] == bytes(a.payload_buff)[:160] == pkt[12:].tobytes()
    assert s.ed137_value == 0 == a.ed137_value and Rf.refta_get_ed137_value(h) == 0
    Rf.refta_destroy(h)
    Rf.refta_destroy(hr)


# ----------------------------------------------------------------------------- getters / setters by call id
@live
def test_field_getters_oracle_equals_reference_live():
    """get_IPRadioBss / PttStatus / PttId / Squelch / Status (Functions.cpp:1001-1179) and get_ed137_value
    (TransportAdapter.cpp:337-346) on the word the reference's callback latched from a wire packet"""
    Rf = RP.lib(0)
    rng = np.random.default_rng(8)
    leg = dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200)
    Rf.refapp_reset(RP.SERVER, 1)
    h = RP.create(Rf, leg, 0, call_id=4)
    Rf.refapp_server_bind(1, 4, 1, b"TRx")
    words = [0, 1, 0x00013100, 0x000131C0, 0x00013140, 0x00013180, 0x00413100, 0x104131F8, 0xE0013100,
             0x10013178, 0xFFFFFFFF] + [int(x) for x in rng.integers(0, 2**32, 200)]
    hdr = np.zeros(20, np.uint8)
    got = (C.c_int * 5)()
    f = O.Fields()
    for w in words:
        L.orc_hdr_write(hdr.ctypes.data, 2, 0, 1, 0, 0, 123, 7, 1120, 4, 0x0167, 1, w)
        assert Rf.refta_rx(h, hdr.ctypes.data, 20, 20) == 0
        assert Rf.refta_get_ed137_value(h) == w
        Rf.refapp_fields(4, got)
        L.orc_ed137_fields_from_word(w, C.byref(f))
        assert list(got) == [f.bss, f.ptt_type, f.ptt_id, f.squelch, f.active], hex(w)
    assert Rf.refta_get_ed137_value(None) == 0                       # NULL adapter (:345)
    RP.lib(0).refta_set_clock(123456)
    assert Rf.refta_getR2SStatus(None) == 123456 - 3000              # NULL adapter (:324)
    assert Rf.refapp_get_R2SStatus(99) == 123456 - 3000              # unknown call (Functions.cpp:1037)
    Rf.refta_destroy(h)


@live
def test_setters_by_call_id_live():
    """setRadioPttbyCallID / setRadioSqlOnbyCallID (rssi >> 6, default 15) / setSlaveEnable
    (Functions.cpp:909-999) land in the adapter exactly as the oracle's setters"""
    Rf = RP.lib(0)
    leg = dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200)
    Rf.refapp_reset(RP.SERVER, 1)
    h = RP.create(Rf, leg, 0, call_id=6)
    a = O.Adapter()
    L.orc_adapter_init(C.byref(a), 1, 0, b"TRx", 200, 0)
    Rf.refapp_setRadioPttbyCallID(1, 6, 3, 1)
    L.orc_setAdapterPtt(C.byref(a), 1, 3, 1)
    Rf.refapp_setRadioSqlOnbyCallID(1, 6, 2, 1000)
    L.orc_setAdapterQslOn(C.byref(a), 1, 2, 1000 >> 6)
    Rf.refapp_setSlaveEnable(6, 1, 0)
    L.orc_setTxRxSlaveEnable(C.byref(a), 1, 0)
    s = RP.state(Rf, h)
    for f in ("pttstatus", "pttpriority", "callRecorder", "sqlstatus", "sqlpriority", "ed137_bssi",
              "rxSlaveEnableChanged", "txSlaveEnableChanged", "trxSlaveEnableChangedCount"):
        assert getattr(s, f) == getattr(a, f), f
    assert s.ed137_bssi == 15
    Rf.refapp_setRadioSqlOnbyCallID(0, 6, 0, -1)      # the 3-argument overload: bssi 15 (Functions.cpp:976)
    assert RP.state(Rf, h).ed137_bssi == 15 and RP.state(Rf, h).sqlstatus == 0
    Rf.refta_destroy(h)


# ----------------------------------------------------------------------------- checkEvents
@live
@pytest.mark.parametrize("mode,G,seed", [(N.ARB_CLIENT_PTT, 4, 4), (N.ARB_SERVER_BEST, 4, 4), (N.ARB_CLIENT_PTT, 7, 1),
                                         (N.ARB_CLIENT_PTT, 32, 2), (N.ARB_SERVER_BEST, 2, 3), (N.ARB_SERVER_BEST, 3, 5)])
def test_gate_arbitration_oracle_equals_reference_live(mode, G, seed):
    """the reference's own checkEvents() (roip_ed137.cpp:5609-6348) with setvolume / setSlotVolume down to the
    level given to pjsua_conf_adjust_rx_level, tick by tick, vs orc_arb_*_tick"""
    w = R.make_arb_words(200, 6, G, mode, seed=seed)
    g, lg, br = R.oracle_arb_walk(w, G, mode)
    rg, rl, rb = RP.run_arb(w, G, mode)
    assert np.array_equal(g, rg)
    assert np.array_equal(lg, rl)
    assert np.array_equal(br, rb)
    assert (g == 256).sum() > 100


@live
def test_gate_arbitration_inactive_legs_live():
    rng = np.random.default_rng(12)
    for mode in (N.ARB_CLIENT_PTT, N.ARB_SERVER_BEST):
        w = R.make_arb_words(150, 5, 4, mode, seed=17)
        active = (rng.random(20) < 0.7).astype(np.uint8)
        g, lg, br = R.oracle_arb_walk(w, 4, mode, active=active)
        rg, rl, rb = RP.run_arb(w, 4, mode, active=active)
        assert np.array_equal(g, rg) and np.array_equal(lg, rl) and np.array_equal(br, rb)


# ----------------------------------------------------------------------------- event logger
def _event_case(seed, F=400):
    rng = np.random.default_rng(seed)
    meter = np.zeros((F, 1), O.METER_DT)
    s = rng.integers(0, 160 * 32768**2 // 4, F, dtype=np.int64).astype(np.uint64)
    bm = rng.integers(0, 256, F).astype(np.uint32)
    meter["sumsq_lo"][:, 0] = (s & 0xFFFFFFFF).astype(np.uint32)
    meter["hi"][:, 0] = ((s >> 32) & 0xFF).astype(np.uint32) | (bm << 8)
    gain = (rng.random((F, 1)) < 0.8).astype(np.uint16) * 256
    return meter, gain, s, bm


def _oracle_event_message(meter, gain, url, sp):
    rec = O.event_summary(meter, gain)[0]
    av, mx, mn, bmav = O.summary_db(rec)
    buf = C.create_string_buffer(2048)
    n = L.orc_ptt_event_json(buf, 2048, sp, b"pptTest_released", av, mx, mn, url, bmav, int(rec["bm_max"]),
                             int(rec["bm_min"]))
    return buf.raw[:n].decode(), rec


@live
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_event_logger_oracle_equals_reference_live(seed):
    """keeplogAudioLevel + createPTTEventDataLogger (Functions.cpp:2126-2230), the reference's own code and
    format string, vs orc_event_summary -> orc_summary_db -> orc_ptt_event_json"""
    Rf = RP.lib(0)
    meter, gain, s, bm = _event_case(seed)
    want, rec = _oracle_event_message(meter, gain, b"sip:radio1@10.0.0.5", 3)
    Rf.refapp_reset(RP.SERVER, 1)
    buf = C.create_string_buffer(2048)
    assert Rf.refapp_ptt_event(0, b"pptTest_pressed", 4.0, b"sip:radio1@10.0.0.5", 3, buf, 2048) > 0
    assert b'"Ptt"                          :"pptTest_pressed"' in buf.value
    assert Rf.refapp_ptt_event(0, b"pptTest_pressed", 4.0, b"sip:radio1@10.0.0.5", 3, buf, 2048) == 0   # already on
    for f in range(meter.shape[0]):
        if gain[f, 0]:
            Rf.refapp_keeplog(0, float(s[f]) / 160.0, int(bm[f]))
    n = Rf.refapp_ptt_event(0, b"pptTest_released", 0.0, b"sip:radio1@10.0.0.5", 3, buf, 2048)
    assert n > 0 and buf.value.decode() == want
    assert rec["count"] == int((gain != 0).sum()) > 256      # the u16 OutgoingRTPSum has wrapped
    assert Rf.refapp_ptt_event(0, b"pptTest_released", 0.0, b"x", 3, buf, 2048) == 0             # already off


# ----------------------------------------------------------------------------- the adapter as PJSIP sees it
@live
def test_reference_vtable_and_sdp_live():
    """what a drop-in has to reproduce at the plugin boundary: `base` first, 12-entry op table, pass-through of
    the non-RTP entries to the slave transport, the SDP attributes (TransportAdapter.cpp:59-133, 941-1044)"""
    Rf = RP.lib(0)
    assert Rf.refta_offsetof_base() == 0
    Rf.refapp_reset(RP.SERVER, 1)
    h = RP.create(Rf, dict(radiocall=1, callIn=0, calltype="Rxonly", keepalive=150), 0, call_id=2)
    assert Rf.refta_vtable_passthrough(h) == 0b0111_0111_0001
    buf = C.create_string_buffer(1024)
    Rf.refta_encode_sdp(h, buf, 1024)
    assert buf.value.decode() == RP.SDP_RXONLY_150
    Rf.refta_setCallType(h, b"TRx")
    Rf.refta_encode_sdp(h, buf, 1024)
    assert "ptt-id:1\n" in buf.value.decode()
    cnt = (C.c_int * 16)()
    Rf.refta_counters(h, cnt)
    assert cnt[RP.COUNTERS_ATTACH] == 1 and cnt[RP.COUNTERS_ENCODE_SDP] == 2    # attach once, encode_sdp twice
    Rf.refta_destroy(h)


# ----------------------------------------------------------------------------- goldens written from the reference
def _oracle_digest():
    """everything tests/golden/make_golden.py's ref_pins() hashes, computed here with the ORACLE"""
    out = {"tx": {}}
    for s in T.SCENARIOS:
        pk, sz, bm, _ = T.run_oracle(s)
        out["tx"][s["name"]] = {"packets": sha(pk), "sizes": sha(sz), "bytemean": sha(bm), "bytes": int(sz.sum())}
    pk, sz, bm, _ = T.run_oracle(T.SCENARIOS[0], signed_char=1)
    out["tx_signed_char"] = {"packets": sha(pk), "bytemean": sha(bm)}
    legs, hdr, ctl = K.make(40, 120, seed=2)
    pk, sz, hf = K.oracle_walk(legs, hdr, ctl)
    out["keepalive"] = {"packets": sha(pk), "sizes": sha(sz), "final_headers": sha(hf)}
    pkts, sizes, present = R.make_rx_stream(300, 24, seed=3)
    ev, st = R.oracle_rx_walk(pkts, R.ref_comparable_sizes(sizes), present)
    out["rx_walk"] = {"events": sha(ev), "state": sha(st)}
    for name, mode, G in (("client_ptt", N.ARB_CLIENT_PTT, 4), ("server_best", N.ARB_SERVER_BEST, 4)):
        w = R.make_arb_words(200, 9, G, mode, seed=G)
        g, lg, br = R.oracle_arb_walk(w, G, mode)
        out[name] = {"gain": sha(g), "legs": sha(lg), "bridges": sha(br)}
    out["event_messages"] = [_oracle_event_message(*_event_case(seed)[:2], b"sip:radio1@10.0.0.5", 3)[0]
                             for seed in (1, 2, 3)]
    return out


def _live_case_digest():
    """the oracle's side of every *_live comparison above that ref_pins.json does not already pin, on the same cases
    (tests/golden/make_golden.py live_cases -> live_cases.json)"""
    out = {"tx_final_state": {}}
    for s in T.SCENARIOS:
        _, _, _, ads = T.run_oracle(s)
        out["tx_final_state"][s["name"]] = [
            {**{f: int(getattr(a, f)) for f in RP.TX_STATE_FIELDS}, "send_pkt_buff": sha(np.frombuffer(bytes(a.send_pkt_buff), np.uint8)),
             "tmp_payload_buf": sha(np.frombuffer(bytes(a.tmp_payload_buf), np.uint8)), "send_payload_bufSize": int(a.send_payload_bufSize)}
            for a, leg in zip(ads, s["legs"]) if leg["radiocall"]]
    pk, sz, bm, _ = T.run_oracle(T.SCENARIOS[0], signed_char=1)
    out["tx_signed_char_sizes"] = sha(sz)
    rng = np.random.default_rng(4)                  # test_send_rtp_csrc_extension_padding_live
    out["csrc"] = []
    o = np.zeros(512, np.uint8)
    for cc, x, extw in ((0, 0, 0), (2, 0, 0), (0, 1, 1), (1, 1, 2), (3, 0, 0)):
        pkt = np.zeros(12 + 4 * cc + (4 + 4 * extw if x else 0) + 160, np.uint8)
        pkt[:] = rng.integers(0, 256, pkt.size)
        pkt[0] = 0x80 | (x << 4) | cc
        pkt[1] = 8
        if x:
            pkt[12 + 4 * cc + 2] = 0
            pkt[12 + 4 * cc + 3] = extw
        a = O.Adapter()
        L.orc_adapter_init(C.byref(a), 1, 0, b"TRx", 200, 5000)
        L.orc_setAdapterPtt(C.byref(a), 1, 3, 0)
        n = L.orc_transport_send_rtp(C.byref(a), pkt.ctypes.data, pkt.size, 5000, o.ctypes.data, 1, 0)
        out["csrc"].append({"size": int(n), "packet": sha(o[:n]), "OutgoingRTP": int(a.OutgoingRTP)})
    pkts, sizes, present = R.make_rx_stream(120, 8, seed=9)    # test_rtp_cb_state_carry_live
    out["rx_state_carry"] = sha(R.oracle_rx_walk(pkts, R.ref_comparable_sizes(sizes), present)[1])
    out["setIncomingRTP"] = {}
    for signed_char in (0, 1):                      # test_setIncomingRTP_bytemean_live
        rng = np.random.default_rng(21)
        a = O.Adapter()
        L.orc_adapter_init(C.byref(a), 1, 0, b"TRx", 200, 0)
        hdr = np.zeros(20, np.uint8)
        res = []
        for n in (160, 164, 24, 1, 80, 256, 200):
            pkt = rng.integers(0, 256, 20 + n, dtype=np.uint8)
            if n == 80:
                pkt[20:] = rng.integers(128, 256, n)
            L.orc_hdr_write(hdr.ctypes.data, 2, 0, 1, 0, 0, 8, 1, 160, 9, 0x0167, 1, 0x10013178)
            pkt[:20] = hdr
            r = L.orc_transport_rtp_cb(C.byref(a), pkt.ctypes.data, pkt.size, 40, 1, signed_char)
            res.append({"n": n, "forwarded": int(r), "IncomingRTP": int(a.IncomingRTP), "payload_bufSize": int(a.payload_bufSize),
                        "payload": sha(np.frombuffer(bytes(a.payload_buff), np.uint8)[:n])})
        out["setIncomingRTP"][str(signed_char)] = res
    rng = np.random.default_rng(2)                  # test_non_radio_rtp_cb_live
    pkt = rng.integers(0, 256, 172, dtype=np.uint8)
    pkt[0], pkt[1] = 0x80, 8
    a = O.Adapter()
    L.orc_adapter_init(C.byref(a), 0, 0, b"", 200, 0)
    r = L.orc_transport_rtp_cb(C.byref(a), pkt.ctypes.data, 172, 0, 0, 0)
    out["non_radio"] = {"forwarded": int(r), "payload_bufSize": int(a.payload_bufSize), "ed137_value": int(a.ed137_value),
                        "payload": sha(np.frombuffer(bytes(a.payload_buff), np.uint8)[:160])}
    rng = np.random.default_rng(8)                  # test_field_getters_oracle_equals_reference_live
    words = [0, 1, 0x00013100, 0x000131C0, 0x00013140, 0x00013180, 0x00413100, 0x104131F8, 0xE0013100,
             0x10013178, 0xFFFFFFFF] + [int(x) for x in rng.integers(0, 2**32, 200)]
    f = O.Fields()
    got = []
    for w in words:
        L.orc_ed137_fields_from_word(w, C.byref(f))
        got.append([f.bss, f.ptt_type, f.ptt_id, f.squelch, f.active])
    out["field_getters"] = sha(np.array(got, np.int64))
    a = O.Adapter()                                 # test_setters_by_call_id_live
    L.orc_adapter_init(C.byref(a), 1, 0, b"TRx", 200, 0)
    L.orc_setAdapterPtt(C.byref(a), 1, 3, 1)
    L.orc_setAdapterQslOn(C.byref(a), 1, 2, 1000 >> 6)
    L.orc_setTxRxSlaveEnable(C.byref(a), 1, 0)
    out["setters"] = {f: int(getattr(a, f)) for f in ("pttstatus", "pttpriority", "callRecorder", "sqlstatus", "sqlpriority",
                                                       "ed137_bssi", "rxSlaveEnableChanged", "txSlaveEnableChanged",
                                                       "trxSlaveEnableChangedCount")}
    out["arbitration"] = {}
    for mode, G, seed in ((N.ARB_CLIENT_PTT, 4, 4), (N.ARB_SERVER_BEST, 4, 4), (N.ARB_CLIENT_PTT, 7, 1),
                          (N.ARB_CLIENT_PTT, 32, 2), (N.ARB_SERVER_BEST, 2, 3), (N.ARB_SERVER_BEST, 3, 5)):
        g, lg, br = R.oracle_arb_walk(R.make_arb_words(200, 6, G, mode, seed=seed), G, mode)
        out["arbitration"][f"mode{mode}_G{G}_seed{seed}"] = {"gain": sha(g), "legs": sha(lg), "bridges": sha(br)}
    rng = np.random.default_rng(12)                 # test_gate_arbitration_inactive_legs_live
    for mode in (N.ARB_CLIENT_PTT, N.ARB_SERVER_BEST):
        active = (rng.random(20) < 0.7).astype(np.uint8)
        g, lg, br = R.oracle_arb_walk(R.make_arb_words(150, 5, 4, mode, seed=17), 4, mode, active=active)
        out["arbitration"][f"mode{mode}_inactive"] = {"gain": sha(g), "legs": sha(lg), "bridges": sha(br)}
    return out


def test_oracle_matches_the_live_cases_pins(golden_dir):
    """every *_live comparison on a machine without the reference build: the oracle against what it computed on the
    same cases where the *_live tests showed it equal to the reference"""
    g = json.load(open(os.path.join(golden_dir, "live_cases.json")))
    got = _live_case_digest()
    for k in got:
        assert got[k] == g[k], k


def test_oracle_matches_goldens_generated_from_the_reference(golden_dir):
    g = json.load(open(os.path.join(golden_dir, "ref_pins.json")))
    assert g["generated_from"] == "reference"
    got = _oracle_digest()
    for k in got:
        assert got[k] == g[k], k
