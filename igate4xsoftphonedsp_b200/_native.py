"""ctypes binding of include/igate_dsp.h (libigate_dsp.so).

The library is the product; this file only declares its C ABI to Python.
There is no fallback: if the shared object is missing or no sm_100 GPU is
present, loading / context creation raises.
"""
import ctypes as C
import os

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# IGD_LIB_PATH: developer knob to load an experimental build of the same library
LIB_PATH = os.environ.get("IGD_LIB_PATH") or os.path.join(PKG_DIR, "libigate_dsp.so")

FRAME = 160
PKT_HDR = 20
PKT_MAX = 180
LAW_ALAW, LAW_ULAW = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1
F_SIGNED_CHAR, F_REF_QUIRKS, F_GENERIC_KERNEL, F_KERNEL_W, F_WALK_SERIAL = 0x1, 0x2, 0x4, 0x8, 0x10
CT_IDLE, CT_RXONLY, CT_TXISH = 0x1, 0x2, 0x4
EDF_ACTIVE, EDF_RRC, EDF_MAIN_TX, EDF_MAIN_RX, EDF_DROPPED = 0x01, 0x02, 0x04, 0x08, 0x10

ERRORS = {-22: "IGD_EINVAL", -12: "IGD_ENOMEM", -19: "IGD_ENODEV", -5: "IGD_ECUDA"}

# numpy views of the C records (include/igate_dsp.h)
METER_DT = np.dtype([("sumsq_lo", "<u4"), ("hi", "<u4"), ("rms_dbfs", "<f4"), ("peak_dbfs", "<f4")])
BRIDGE_DT = np.dtype([("bytemean_out", "u1"), ("n_open", "u1"), ("mix_peak", "<u2")])
SUMMARY_DT = np.dtype([("count", "<u4"), ("bm_sum", "<u2"), ("bm_max", "u1"), ("bm_min", "u1"),
                       ("sum_s", "<u8"), ("max_s", "<u8"), ("min_s", "<u8")])
SUMMARY_DB_DT = np.dtype([("level_av_db", "<f4"), ("level_max_db", "<f4"), ("level_min_db", "<f4"),
                          ("bm_av", "<u4")])
FIELDS_DT = np.dtype([("word", "<u4"), ("length_raw", "<u2"), ("payload_len", "<u2"), ("pt", "u1"),
                      ("accepted", "u1"), ("keepalive", "u1"), ("ptt_type", "u1"), ("ptt_id", "u1"),
                      ("squelch", "u1"), ("bss", "u1"), ("flags", "u1")])
STATE_DT = np.dtype([("radiostatus", "u1"), ("pttstatus", "u1"), ("sqlstatus", "u1"), ("callIn", "u1"),
                     ("callRecorder", "u1"), ("pttpriority", "u1"), ("pttid", "u1"), ("ed137_bssi", "u1"),
                     ("rxSlaveEnable", "u1"), ("txSlaveEnable", "u1"), ("rxSlaveEnableChanged", "u1"),
                     ("txSlaveEnableChanged", "u1"), ("trxSlaveEnableChangedCount", "u1"),
                     ("firstR2SPacket", "u1"), ("calltype_flags", "u1"), ("sqlpriority", "u1"),
                     ("packetCnt", "<i4"), ("keepAlivePeroid", "<i4"), ("r2sSendtime", "<i8"),
                     ("rtpFalse", "<i4"), ("reserved", "<i4")])
CTL_DT = np.dtype([("pttstatus", "u1"), ("sqlstatus", "u1"), ("pttpriority", "u1"), ("ed137_bssi", "u1"),
                   ("pttid", "u1"), ("callRecorder", "u1"), ("reserved", "u1", (2,))])
assert METER_DT.itemsize == 16 and BRIDGE_DT.itemsize == 4 and SUMMARY_DT.itemsize == 32
assert SUMMARY_DB_DT.itemsize == 16 and FIELDS_DT.itemsize == 16 and STATE_DT.itemsize == 40
RX_STATE_DT = np.dtype([("r2sPacket", "<i8"), ("ed137_value", "<u4"), ("payloadsize", "<u2"), ("rtpAudio", "u1"),
                        ("r2sCount", "u1")])
RX_EVENT_DT = np.dtype([("word", "<u4"), ("flags", "u1"), ("r2sCount", "u1"), ("reserved", "<u2")])
ARB_LEG_DT = np.dtype([("last", "u1"), ("msec", "u1"), ("on", "u1"), ("rssi", "i1"), ("gain_q7", "<u2"),
                       ("reserved", "<u2")])
ARB_BRIDGE_DT = np.dtype([("ptt_level", "<i4"), ("sqlStatusCount", "<i4"), ("sqlStatusOn", "u1"),
                          ("reserved", "u1", (7,))])
RXE_PACKET, RXE_AUDIO, RXE_EDGE, RXE_DROPPED, RXE_LATE, RXE_HANGUP, RXE_FRAME = 0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40
ARB_CLIENT_PTT, ARB_SERVER_BEST = 0, 1
ARB_F_SILENCE = 0x1
GAIN_NO_AUDIO = 0x8000
assert CTL_DT.itemsize == 8 and RX_STATE_DT.itemsize == 16 and RX_EVENT_DT.itemsize == 8
assert ARB_LEG_DT.itemsize == 8 and ARB_BRIDGE_DT.itemsize == 16


class DevInfo(C.Structure):
    _fields_ = [("device", C.c_int), ("sm_count", C.c_int), ("cc_major", C.c_int), ("cc_minor", C.c_int),
                ("total_mem", C.c_size_t), ("name", C.c_char * 64)]


class BatchDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mem", C.c_int32), ("F", C.c_int32), ("B", C.c_int32),
                ("G", C.c_int32), ("flags", C.c_uint32),
                ("codes", C.c_void_p), ("law", C.c_void_p), ("gain_q7", C.c_void_p), ("out_law", C.c_void_p),
                ("mix", C.c_void_p), ("enc", C.c_void_p), ("meter", C.c_void_p), ("bmeter", C.c_void_p)]


class PacketsDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mem", C.c_int32), ("F", C.c_int32), ("B", C.c_int32),
                ("G", C.c_int32), ("flags", C.c_uint32),
                ("pkts", C.c_void_p), ("fields", C.c_void_p), ("law", C.c_void_p), ("gain_q7", C.c_void_p),
                ("out_law", C.c_void_p),
                ("mix", C.c_void_p), ("enc", C.c_void_p), ("meter", C.c_void_p), ("bmeter", C.c_void_p)]


class PackDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mem", C.c_int32), ("F", C.c_int32), ("C", C.c_int32),
                ("flags", C.c_uint32), ("payload_len", C.c_uint32), ("out_stride", C.c_uint32),
                ("tick_ms", C.c_int32), ("now_ms0", C.c_int64),
                ("rtp12", C.c_void_p), ("payload", C.c_void_p), ("ctl", C.c_void_p), ("state", C.c_void_p),
                ("pkts", C.c_void_p), ("sizes", C.c_void_p), ("bytemean_out", C.c_void_p),
                ("stale_payload", C.c_void_p)]


class RxTrackDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mem", C.c_int32), ("F", C.c_int32), ("C", C.c_int32),
                ("tick_ms", C.c_int32), ("r2s_period_ms", C.c_int32), ("wd_ticks", C.c_int32),
                ("frame0", C.c_int32), ("now_ms0", C.c_int64),
                ("fields", C.c_void_p), ("present", C.c_void_p), ("state", C.c_void_p), ("events", C.c_void_p),
                ("sizes", C.c_void_p)]


class GatewayDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mem", C.c_int32), ("F", C.c_int32), ("B", C.c_int32), ("G", C.c_int32),
                ("flags", C.c_uint32), ("arb_mode", C.c_int32), ("tick_ms", C.c_int32), ("r2s_period_ms", C.c_int32),
                ("wd_ticks", C.c_int32), ("frame0", C.c_int32), ("reserved", C.c_int32), ("now_ms0", C.c_int64),
                ("rx_pkts", C.c_void_p), ("rx_sizes", C.c_void_p), ("law", C.c_void_p), ("active", C.c_void_p),
                ("rx_state", C.c_void_p), ("arb_legs", C.c_void_p), ("arb_bridges", C.c_void_p),
                ("out_law", C.c_void_p), ("tx_rtp12", C.c_void_p), ("tx_ctl", C.c_void_p), ("tx_state", C.c_void_p),
                ("tx_pkts", C.c_void_p), ("tx_sizes", C.c_void_p), ("rx_events", C.c_void_p), ("gain_q7", C.c_void_p),
                ("meter", C.c_void_p), ("bmeter", C.c_void_p), ("mix", C.c_void_p), ("enc", C.c_void_p)]


class FanoutDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mem", C.c_int32), ("F", C.c_int32), ("B", C.c_int32), ("G", C.c_int32),
                ("flags", C.c_uint32), ("tick_ms", C.c_int32), ("reserved", C.c_int32), ("now_ms0", C.c_int64),
                ("pcm", C.c_void_p), ("law", C.c_void_p), ("tx_rtp12", C.c_void_p), ("tx_ctl", C.c_void_p),
                ("tx_state", C.c_void_p), ("tx_pkts", C.c_void_p), ("tx_sizes", C.c_void_p), ("tx_level", C.c_void_p)]


class FanoutPktDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mem", C.c_int32), ("F", C.c_int32), ("B", C.c_int32), ("G", C.c_int32),
                ("flags", C.c_uint32), ("tick_ms", C.c_int32), ("reserved", C.c_int32), ("now_ms0", C.c_int64),
                ("rx_pkts", C.c_void_p), ("rx_sizes", C.c_void_p), ("in_law", C.c_void_p), ("law", C.c_void_p),
                ("tx_rtp12", C.c_void_p), ("tx_ctl", C.c_void_p), ("tx_state", C.c_void_p), ("tx_pkts", C.c_void_p),
                ("tx_sizes", C.c_void_p), ("tx_level", C.c_void_p)]


class ArbDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mem", C.c_int32), ("F", C.c_int32), ("B", C.c_int32),
                ("G", C.c_int32), ("mode", C.c_int32), ("word_stride", C.c_uint32), ("flags", C.c_uint32),
                ("words", C.c_void_p), ("active", C.c_void_p), ("legs", C.c_void_p), ("bridges", C.c_void_p),
                ("gain_q7", C.c_void_p)]


# every symbol include/igate_dsp.h declares: name -> (restype, argtypes)
_vp, _sz, _i = C.c_void_p, C.c_size_t, C.c_int
SYMBOLS = {
    "igd_abi_version": (_i, []),
    "igd_init": (_i, [_i, C.POINTER(_vp)]),
    "igd_shutdown": (_i, [_vp]),
    "igd_set_stream": (_i, [_vp, _vp]),
    "igd_use_own_stream": (_i, [_vp]),
    "igd_sync": (_i, [_vp]),
    "igd_last_error": (C.c_char_p, [_vp]),
    "igd_device_info": (_i, [_vp, C.POINTER(DevInfo)]),
    "igd_launch_count": (C.c_uint64, [_vp]),
    "igd_host_alloc": (_vp, [_sz]),
    "igd_host_free": (None, [_vp]),
    "igd_dev_alloc": (_vp, [_vp, _sz]),
    "igd_dev_free": (None, [_vp, _vp]),
    "igd_copy_to_device": (_i, [_vp, _vp, _vp, _sz]),
    "igd_copy_to_host": (_i, [_vp, _vp, _vp, _sz]),
    "igd_g711_decode": (_i, [_vp, _vp, _vp, _sz, _i, _i]),
    "igd_g711_encode": (_i, [_vp, _vp, _vp, _sz, _i, _i]),
    "igd_g711_decode_ch": (_i, [_vp, _vp, _vp, _vp, _sz, _sz, _i]),
    "igd_g711_encode_ch": (_i, [_vp, _vp, _vp, _vp, _sz, _sz, _i]),
    "igd_frame_meter": (_i, [_vp, _vp, _sz, _vp, _i]),
    "igd_bytemean": (_i, [_vp, _vp, _sz, _sz, _sz, C.c_uint, _vp, _i]),
    "igd_level_percent": (_i, [_vp, _vp, _sz, _vp, _i]),
    "igd_gain_q7": (_i, [C.c_float]),
    "igd_mix": (_i, [_vp, _vp, _vp, _sz, _sz, _i, _vp, _i]),
    "igd_process_batch": (_i, [_vp, C.POINTER(BatchDesc)]),
    "igd_process_packets": (_i, [_vp, C.POINTER(PacketsDesc)]),
    "igd_event_summary": (_i, [_vp, _vp, _vp, _sz, _sz, _vp, _vp, _i]),
    "igd_ed137_parse": (_i, [_vp, _vp, _vp, _sz, _sz, _vp, _vp, _i]),
    "igd_calltype_flags": (C.c_uint, [C.c_char_p]),
    "igd_ed137_state_init": (None, [_vp, _i, _i, C.c_char_p, _i, C.c_int64]),
    "igd_ed137_pack": (_i, [_vp, C.POINTER(PackDesc)]),
    "igd_ed137_keepalive": (_i, [_vp, _vp, _vp, _sz, C.c_int64, _vp, _i]),
    "igd_rx_track": (_i, [_vp, C.POINTER(RxTrackDesc)]),
    "igd_gate_arbitrate": (_i, [_vp, C.POINTER(ArbDesc)]),
    "igd_gateway_process": (_i, [_vp, C.POINTER(GatewayDesc)]),
    "igd_gateway_fanout": (_i, [_vp, C.POINTER(FanoutDesc)]),
    "igd_gateway_fanout_packets": (_i, [_vp, C.POINTER(FanoutPktDesc)]),
    "igd_wav_size": (_sz, [_sz, _i]),
    "igd_wav_image": (_i, [_vp, _vp, _sz, _i, _i, _i, _vp, C.POINTER(_sz), _i]),
    "igd_wav_images": (_i, [_vp, _vp, _sz, _sz, _vp, _sz, _vp, _i, _i, _vp, _sz, _i]),
}

_lib = None


class NativeLibraryMissing(RuntimeError):
    pass


def load():
    """Loads libigate_dsp.so and binds every declared symbol; raises if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C igate4xsoftphonedsp_b200/csrc`). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            if os.environ.get("IGD_LIB_PATH") and not hasattr(lib, name):
                continue              # developer knob only: an older experimental build may lack newer entry points
            fn = getattr(lib, name)   # AttributeError = ABI drift, fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
