"""ctypes binding of the REFERENCE-backed harness oracle/_ref/libigd_ref_ta{,_sc}.so: the reference's
own TransportAdapter.cpp + the line-range extracts of its RoIP_ED137 members, compiled from
/root/reference by oracle/Makefile (oracle/ref_harness.cpp documents the API).

TEST INFRASTRUCTURE ONLY.  The walks below replay the shared seeded cases (tx_scenarios.py,
keepalive_cases.py, rx_arb_cases.py) through the reference exactly as the oracle walks replay them
through oracle/igd_oracle.c, so that `oracle == reference` is an array comparison.
"""
import ctypes as C
import os

import numpy as np

from igate4xsoftphonedsp_b200 import _native as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_DIR = os.path.join(ROOT, "oracle", "_ref")

SERVER, CLIENT = 1, 2

# what the reference's encode_sdp (TransportAdapter.cpp:941-1044) wrote for a radio call of type "Rxonly" and
# keep-alive period 150, and its slave-transport counters after attach + two encode_sdp calls
SDP_RXONLY_150 = ("rtphe:1\ntype:Rxonly\ntxrxmode:TRx\nbss:RSSI\nsigtime:1\nptt_rep:0\n"
                  "R2S-KeepAlivePeriod:150\nR2S-KeepAliveMultiplier:10\n")
COUNTERS_ATTACH, COUNTERS_ENCODE_SDP = 4 + 1, 4 + 7


class State(C.Structure):
    _fields_ = [("radiostatus", C.c_int), ("pttstatus", C.c_int), ("sqlstatus", C.c_int),
                ("callIn", C.c_int), ("callRecorder", C.c_int),
                ("pttpriority", C.c_int), ("sqlpriority", C.c_int), ("ed137_bssi", C.c_int), ("pttid", C.c_int),
                ("rxSlaveEnable", C.c_int), ("txSlaveEnable", C.c_int),
                ("rxSlaveEnableChanged", C.c_int), ("txSlaveEnableChanged", C.c_int),
                ("trxSlaveEnableChangedCount", C.c_int),
                ("firstR2SPacket", C.c_int), ("packetCnt", C.c_int),
                ("keepAlivePeroid", C.c_int), ("rtpFalse", C.c_int), ("rtpAudio", C.c_int),
                ("r2sSendtime", C.c_longlong), ("r2sPacket", C.c_longlong),
                ("ed137_value", C.c_uint32), ("payloadsize", C.c_uint32),
                ("calltype", C.c_char * 64),
                ("send_pkt_buff", C.c_uint8 * 256), ("tmp_payload_buf", C.c_uint8 * 256),
                ("payload_buff", C.c_uint8 * 256),
                ("payload_bufSize", C.c_uint64), ("send_payload_bufSize", C.c_uint64)]


class Leg(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("lastRx", "lastTx", "lastRxmsec", "lastTxmsec", "audioSQLOn", "rssi",
                                       "m_PttPressed", "pttLevel", "SQLOn", "IncomingRTP", "OutgoingRTP")]


def path(signed_char=0):
    return os.path.join(_DIR, "libigd_ref_ta_sc.so" if signed_char else "libigd_ref_ta.so")


def available():
    return os.path.exists(path(0)) and os.path.exists(path(1))


_libs = {}


def lib(signed_char=0):
    if signed_char not in _libs:
        R = C.CDLL(path(signed_char))
        R.refta_create.restype = C.c_void_p
        R.refta_create.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_char_p, C.c_int, C.c_int,
                                   C.c_int, C.c_int]
        R.refta_destroy.argtypes = [C.c_void_p]
        R.refta_set_clock.argtypes = [C.c_longlong]
        R.refta_send_rtp.restype = C.c_size_t
        R.refta_send_rtp.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_int)]
        R.refta_sendR2SStatus.restype = C.c_size_t
        R.refta_sendR2SStatus.argtypes = [C.c_void_p, C.c_void_p]
        R.refta_rx.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
        R.refta_rtcp.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        R.refta_setAdapterPtt.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        R.refta_setTxRxSlaveEnable.argtypes = [C.c_void_p, C.c_int, C.c_int]
        R.refta_setAdapterQslOn.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint32]
        R.refta_setAdapterPttId.argtypes = [C.c_void_p, C.c_int]
        R.refta_setcallRecorder.argtypes = [C.c_void_p, C.c_int]
        R.refta_setCallType.argtypes = [C.c_void_p, C.c_char_p]
        R.refta_setAdapterRadioModeAndType.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
        R.refta_get_ed137_value.restype = C.c_uint32
        R.refta_get_ed137_value.argtypes = [C.c_void_p]
        R.refta_getR2SStatus.restype = C.c_longlong
        R.refta_getR2SStatus.argtypes = [C.c_void_p]
        R.refta_get_state.argtypes = [C.c_void_p, C.POINTER(State)]
        R.refta_poke_send_hdr.argtypes = [C.c_void_p, C.c_void_p]
        R.refta_poke_word.argtypes = [C.c_void_p, C.c_uint32]
        R.refta_poke_rx.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_uint32, C.c_uint32]
        R.refta_counters.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        R.refta_vtable_passthrough.argtypes = [C.c_void_p]
        R.refta_encode_sdp.restype = C.c_size_t
        R.refta_encode_sdp.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t]
        R.refapp_reset.argtypes = [C.c_int, C.c_int]
        R.refapp_server_bind.argtypes = [C.c_int, C.c_int, C.c_int, C.c_char_p]
        R.refapp_client_add.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_char_p]
        R.refapp_rx_level.restype = C.c_float
        R.refapp_rx_level.argtypes = [C.c_int]
        R.refapp_get_leg.argtypes = [C.c_int, C.POINTER(Leg)]
        R.refapp_set_leg.argtypes = [C.c_int, C.POINTER(Leg)]
        R.refapp_get_bridge.argtypes = [C.POINTER(C.c_int)]
        R.refapp_set_bridge.argtypes = [C.c_int, C.c_int, C.c_int]
        R.refapp_fields.argtypes = [C.c_int, C.POINTER(C.c_int)]
        R.refapp_setRadioPttbyCallID.argtypes = [C.c_int] * 4
        R.refapp_setRadioSqlOnbyCallID.argtypes = [C.c_int] * 4
        R.refapp_setSlaveEnable.argtypes = [C.c_int] * 3
        R.refapp_get_R2SStatus.restype = C.c_longlong
        R.refapp_get_R2SStatus.argtypes = [C.c_int]
        R.refapp_keeplog.argtypes = [C.c_int, C.c_double, C.c_int]
        R.refapp_ptt_event.restype = C.c_size_t
        R.refapp_ptt_event.argtypes = [C.c_int, C.c_char_p, C.c_double, C.c_char_p, C.c_int, C.c_char_p, C.c_size_t]
        _libs[signed_char] = R
    return _libs[signed_char]


def create(R, leg, now, call_id=-1, attach=1):
    R.refta_set_clock(now)
    h = R.refta_create(leg["radiocall"], leg["callIn"], leg["calltype"].encode(), call_id, b"idx", b"TRx",
                       leg["keepalive"], 1, 0, attach)
    assert h
    return h


def state(R, h):
    s = State()
    R.refta_get_state(h, C.byref(s))
    return s


# ------------------------------------------------------------------ transport_send_rtp
def run_tx(s, signed_char=0):
    """tx_scenarios.run_oracle, through the reference's tp->op->send_rtp (TransportAdapter.cpp:635-874) and its
    own setOutgoingRTP (roip_ed137.cpp:6500-6536): -> pkts, sizes, bytemean, final adapter states."""
    R = lib(signed_char)
    F, Cn = s["F"], len(s["legs"])
    pk = np.zeros((F, Cn, 180), np.uint8)
    sizes = np.zeros((F, Cn), np.uint32)
    bm = np.zeros((F, Cn), np.uint8)
    finals = []
    out = np.zeros(512, np.uint8)
    leg_rec = Leg()
    for c, leg in enumerate(s["legs"]):
        R.refapp_reset(SERVER, 1)
        h = create(R, leg, s["now0"], call_id=7)
        R.refapp_server_bind(0, 7, 1, b"TRx")       # trx1->radio1 is this call: OutgoingRTP lands there
        if leg["slave"] is not None:
            R.refta_setTxRxSlaveEnable(h, leg["slave"][0], leg["slave"][1])
        for f in range(F):
            if s["ctl"] is not None:
                k = s["ctl"][f, c]
                R.refta_setAdapterPtt(h, int(k["pttstatus"]), int(k["pttpriority"]), int(k["callRecorder"]))
                R.refta_setAdapterQslOn(h, int(k["sqlstatus"]), 0, int(k["ed137_bssi"]))
                R.refta_setAdapterPttId(h, int(k["pttid"]))
            pkt = np.concatenate([s["rtp12"][f, c], s["payload"][f, c]])
            R.refta_set_clock(s["now0"] + f * s["tick_ms"])
            n = R.refta_send_rtp(h, pkt.ctypes.data, pkt.size, out.ctypes.data, None)
            sizes[f, c] = n
            pk[f, c, :n] = out[:n]
            if n and (out[1] & 0x7F) != 123:
                R.refapp_get_leg(0, C.byref(leg_rec))
                bm[f, c] = leg_rec.OutgoingRTP
        finals.append(state(R, h))
        R.refta_destroy(h)
    return pk, sizes, bm, finals


TX_STATE_FIELDS = ("pttstatus", "sqlstatus", "callRecorder", "pttpriority", "sqlpriority", "ed137_bssi", "pttid",
                   "rxSlaveEnable", "txSlaveEnable", "rxSlaveEnableChanged", "txSlaveEnableChanged",
                   "trxSlaveEnableChangedCount", "firstR2SPacket", "packetCnt", "rtpFalse", "r2sSendtime")


# ------------------------------------------------------------------ sendR2SStatus
def run_keepalive(legs, hdr, ctl, now0=10_000, tick=40):
    """keepalive_cases.oracle_walk through the reference's sendR2SStatus (TransportAdapter.cpp:422-633)."""
    R = lib(0)
    T, Cn = ctl.shape
    pk = np.zeros((T, Cn, 20), np.uint8)
    sizes = np.zeros((T, Cn), np.uint32)
    hfin = np.zeros((Cn, 20), np.uint8)
    out = np.zeros(512, np.uint8)
    for c, leg in enumerate(legs):
        R.refapp_reset(SERVER, 1)
        h = create(R, leg, now0)
        if leg["slave"] is not None:
            R.refta_setTxRxSlaveEnable(h, leg["slave"][0], leg["slave"][1])
        hd = np.ascontiguousarray(hdr[c])
        R.refta_poke_send_hdr(h, hd.ctypes.data)
        for t in range(T):
            k = ctl[t, c]
            R.refta_setAdapterPtt(h, int(k["pttstatus"]), int(k["pttpriority"]), int(k["callRecorder"]))
            R.refta_setAdapterQslOn(h, int(k["sqlstatus"]), 0, int(k["ed137_bssi"]))
            R.refta_setAdapterPttId(h, int(k["pttid"]))
            R.refta_set_clock(now0 + t * tick)
            n = R.refta_sendR2SStatus(h, out.ctypes.data)
            sizes[t, c] = n
            pk[t, c, :n] = out[:n]
        hfin[c] = np.frombuffer(bytes(state(R, h).send_pkt_buff)[:20], np.uint8)
        R.refta_destroy(h)
    return pk, sizes, hfin


# ------------------------------------------------------------------ transport_rtp_cb + watchdog
def ref_safe_rx_size(n):
    """Sizes the reference can be fed without corrupting itself: a radio packet with 256 < size-20 < 1024
    is copied past the 256-byte payload_buff (TransportAdapter.cpp:286-287, latent overflow, SURVEY 8b) and
    then sizes a stack array from the overwritten length (roip_ed137.cpp:6553)."""
    return not (276 < n < 1044)


def run_rx(pkts, sizes, present, now0=1000, tick=20, period=200, wd_ticks=2, frame0=0, state0=None):
    """rx_arb_cases.oracle_rx_walk through the callback the reference adapter registers with its slave transport
    (transport_rtp_cb, TransportAdapter.cpp:240-316).  The watchdog arithmetic of
    RoIP_ED137::detectR2SPacketAndReconn (roip_ed137.cpp:1767-1777) is replayed here on the r2sPacket stamp the
    REFERENCE produced (getR2SStatus), since that function is reconnect logic around three lines of arithmetic."""
    R = lib(0)
    F, Cn = sizes.shape
    ev = np.zeros((F, Cn), N.RX_EVENT_DT)
    st = np.zeros(Cn, N.RX_STATE_DT) if state0 is None else state0.copy()
    leg = dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200)
    for c in range(Cn):
        R.refapp_reset(CLIENT, 1)                   # inviteServer = 0 in the oracle walk: no byte-mean
        h = create(R, leg, 0, call_id=3)
        R.refta_poke_rx(h, int(st["r2sPacket"][c]), int(st["rtpAudio"][c]), int(st["ed137_value"][c]),
                        int(st["payloadsize"][c]))
        cnt = int(st["r2sCount"][c])
        for f in range(F):
            now = now0 + f * tick
            flags = 0
            if present[f, c]:
                flags |= N.RXE_PACKET
                n = int(sizes[f, c])
                assert ref_safe_rx_size(n)
                p = np.ascontiguousarray(pkts[f, c])
                calls = R.refapp_checkEvents_calls()
                before = state(R, h)
                R.refta_set_clock(now)
                fwd = R.refta_rx(h, p.ctypes.data, n, p.size)
                after = state(R, h)
                if fwd == 1:
                    from rx_arb_cases import frame_flag
                    flags |= N.RXE_AUDIO | frame_flag(pkts[f, c], n)
                elif after.rtpAudio == before.rtpAudio and (n < 20 or n - 20 >= 1024):
                    flags |= N.RXE_DROPPED          # :289-290: stamped r2sPacket and returned
                if R.refapp_checkEvents_calls() != calls:
                    flags |= N.RXE_EDGE
            if wd_ticks > 0 and (frame0 + f) % wd_ticks == wd_ticks - 1:
                r2s = R.refta_getR2SStatus(h)
                if now - r2s > period * 3:          # roip_ed137.cpp:1769
                    flags |= N.RXE_LATE
                    if cnt == 5:                    # :1771
                        flags |= N.RXE_HANGUP
                    cnt += 1                        # :1776
                else:
                    cnt = 0                         # :1779
            ev[f, c] = (R.refta_get_ed137_value(h), flags, min(cnt, 255), 0)
        s = state(R, h)
        st[c] = (s.r2sPacket, R.refta_get_ed137_value(h), s.payloadsize & 0xFFFF, s.rtpAudio, min(cnt, 255))
        R.refta_destroy(h)
    return ev, st


# ------------------------------------------------------------------ checkEvents (gate arbitration)
def _q7(level):
    """pjsua_conf_adjust_rx_level(level) -> the Q7 gain (SURVEY Appendix D); -1 = never set = 0"""
    return 0 if level < 0 else int((level - 1.0) * 128) + 128


def run_arb(words, G, mode, active=None):
    """rx_arb_cases.oracle_arb_walk through the reference's own checkEvents() (roip_ed137.cpp:5609-6348):
    one call per tick per bridge; the latched word of every leg is placed in its adapter, the gain is what the
    reference last handed to pjsua_conf_adjust_rx_level for that call."""
    R = lib(0)
    F, Cn = words.shape
    B = Cn // G
    gain = np.zeros((F, Cn), np.uint16)
    legs = np.zeros(Cn, N.ARB_LEG_DT)
    bridges = np.zeros(B, N.ARB_BRIDGE_DT)
    leg = dict(radiocall=1, callIn=0, calltype="TRx", keepalive=200)
    rec = Leg()
    br = (C.c_int * 3)()
    for b in range(B):
        server = mode != N.ARB_CLIENT_PTT
        R.refapp_reset(SERVER if server else CLIENT, 1)
        hs = []
        for g in range(G):
            act = 1 if active is None else int(active[b * G + g])
            hs.append(create(R, leg, 0, call_id=10 + g))
            if server:
                R.refapp_server_bind(g, 10 + g, act, b"TRx")
            else:
                R.refapp_client_add(10 + g, act, b"TRx", ("call%d" % g).encode())
        for f in range(F):
            for g in range(G):
                R.refta_poke_word(hs[g], int(words[f, b * G + g]))
            R.refapp_checkEvents()
            for g in range(G):
                gain[f, b * G + g] = _q7(R.refapp_rx_level(10 + g))
        for g in range(G):
            R.refapp_get_leg(g, C.byref(rec))
            if server:
                legs[b * G + g] = (rec.lastRx, rec.lastRxmsec, rec.audioSQLOn, rec.rssi, gain[F - 1, b * G + g], 0)
            else:
                legs[b * G + g] = (rec.lastTx, rec.lastTxmsec, rec.m_PttPressed, 0, gain[F - 1, b * G + g], 0)
        R.refapp_get_bridge(br)
        bridges[b] = (br[0], br[1], br[2], [0] * 7) if False else bridges[b]
        bridges["ptt_level"][b], bridges["sqlStatusCount"][b], bridges["sqlStatusOn"][b] = br[0], br[1], br[2]
        for h in hs:
            R.refta_destroy(h)
    return gain, legs, bridges
