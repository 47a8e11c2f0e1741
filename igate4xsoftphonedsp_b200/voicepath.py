"""Host-side mirror of the reference's voice-path interface over the C ABI.

`VoicePath` is what a user of the reference switches to for the hot path:
G.711 (PJSIP PCMA/PCMU, roip_ed137.cpp:3546-3574), the per-packet level meter
(RoIP_ED137::setIncomingRTP/setOutgoingRTP, roip_ed137.cpp:6500-6587), the
conference-bridge gain + mix (roip_ed137.cpp:4907-4920, 5221), the ED-137 RTP
header extension (TransportAdapter.cpp:240-316, 635-874; Functions.cpp:
1001-1179), the PTT event summary (Functions.cpp:2126-2230) and the WavWriter
sink (WavWriter.cpp:63-156) -- batched over channels x 20 ms frames.

Arguments are numpy arrays (host memory: the library stages them through the
GPU) or torch CUDA tensors (used in place; results are torch CUDA tensors).
Either way all arithmetic happens in the CUDA kernels of libigate_dsp.so.
"""
import ctypes as C

import numpy as np

from . import _native as N

try:  # torch is plumbing only (device memory + streams)
    import torch
except Exception:  # pragma: no cover
    torch = None


class IgdError(RuntimeError):
    pass


def _is_torch(x):
    return torch is not None and isinstance(x, torch.Tensor)


def gain_q7(level):
    """pjsua_conf_adjust_rx_level(level) -> Q7 multiplier (2.0->256, 0.1->13)."""
    return N.load().igd_gain_q7(float(level))


def calltype_flags(calltype):
    return N.load().igd_calltype_flags(calltype.encode())


def make_state(n, radiocall=True, callIn=False, calltype="TRx", keepAlivePeroid=200, now_ms=0):
    """n sender states initialised like pjmedia_custom_tp_adapter_create."""
    lib = N.load()
    st = np.zeros(n, dtype=N.STATE_DT)
    one = np.zeros(1, dtype=N.STATE_DT)
    lib.igd_ed137_state_init(one.ctypes.data, int(radiocall), int(callIn), calltype.encode(),
                             int(keepAlivePeroid), int(now_ms))
    st[:] = one[0]
    return st


class VoicePath:
    def __init__(self, device=0):
        self._lib = N.load()
        h = C.c_void_p()
        rc = self._lib.igd_init(int(device), C.byref(h))
        if rc != 0:
            raise IgdError(f"igd_init(device={device}) failed: {N.ERRORS.get(rc, rc)} "
                           "(an sm_100 CUDA device is required; there is no CPU fallback)")
        self._h = h
        self.device = int(device)

    # ------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None):
            self._lib.igd_shutdown(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _chk(self, rc):
        if rc != 0:
            msg = self._lib.igd_last_error(self._h)
            raise IgdError(f"{N.ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")

    def use_torch_stream(self, stream=None):
        """Launch on a torch stream (default: torch's current stream on this device)."""
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        self._chk(self._lib.igd_set_stream(self._h, C.c_void_p(s.cuda_stream)))

    def use_own_stream(self):
        self._chk(self._lib.igd_use_own_stream(self._h))

    def sync(self):
        self._chk(self._lib.igd_sync(self._h))

    def launch_count(self):
        return int(self._lib.igd_launch_count(self._h))

    def device_info(self):
        d = N.DevInfo()
        self._chk(self._lib.igd_device_info(self._h, C.byref(d)))
        return {"device": d.device, "sm_count": d.sm_count, "cc": (d.cc_major, d.cc_minor),
                "total_mem": d.total_mem, "name": d.name.decode()}

    @staticmethod
    def _ptr(x):
        if x is None:
            return None
        if _is_torch(x):
            return C.c_void_p(x.data_ptr())
        return C.c_void_p(x.ctypes.data)

    def _mode(self, *arrays):
        kinds = {_is_torch(a) for a in arrays if a is not None}
        if len(kinds) != 1:
            raise IgdError("all buffers of one call must be numpy arrays or all torch CUDA tensors")
        dev = kinds.pop()
        if dev:
            for a in arrays:
                if a is not None and (not a.is_cuda or not a.is_contiguous()):
                    raise IgdError("torch arguments must be contiguous CUDA tensors")
            self.use_torch_stream()      # device buffers are ordered on torch's current stream
        return N.MEM_DEVICE if dev else N.MEM_HOST

    def _empty(self, like_torch, shape, np_dtype):
        """uninitialised output: torch byte tensor viewed as records, or numpy."""
        if like_torch:
            nbytes = int(np.prod(shape)) * np.dtype(np_dtype).itemsize
            return torch.empty(max(nbytes, 1), dtype=torch.uint8, device=f"cuda:{self.device}")
        return np.empty(shape, dtype=np_dtype)

    @staticmethod
    def _tview(t, tdtype, shape):
        return t.view(tdtype).reshape(shape)

    # ------------------------------------------------------------ G.711
    def g711_decode(self, codes, law):
        """codes u8 [...] -> PCM int16 [...]. `law`: LAW_* or a [nch] array for
        codes laid out [frames][nch][160]."""
        per_ch = not np.isscalar(law)
        mem = self._mode(codes, law if per_ch else None)
        if mem == N.MEM_DEVICE:
            out = torch.empty(codes.shape, dtype=torch.int16, device=codes.device)
            n = codes.numel()
        else:
            codes = np.ascontiguousarray(codes, dtype=np.uint8)
            out = np.empty(codes.shape, dtype=np.int16)
            n = codes.size
            if per_ch:
                law = np.ascontiguousarray(law, dtype=np.uint8)
        if per_ch:
            nch = law.numel() if _is_torch(law) else law.size
            if codes.shape[-1] != N.FRAME or n % (nch * N.FRAME):
                raise IgdError("per-channel law needs codes shaped [frames][nch][160]")
            self._chk(self._lib.igd_g711_decode_ch(self._h, self._ptr(codes), self._ptr(law), self._ptr(out),
                                                   n // (nch * N.FRAME), nch, mem))
        else:
            self._chk(self._lib.igd_g711_decode(self._h, self._ptr(codes), self._ptr(out), n, int(law), mem))
        return out

    def g711_encode(self, pcm, law):
        per_ch = not np.isscalar(law)
        mem = self._mode(pcm, law if per_ch else None)
        if mem == N.MEM_DEVICE:
            out = torch.empty(pcm.shape, dtype=torch.uint8, device=pcm.device)
            n = pcm.numel()
        else:
            pcm = np.ascontiguousarray(pcm, dtype=np.int16)
            out = np.empty(pcm.shape, dtype=np.uint8)
            n = pcm.size
            if per_ch:
                law = np.ascontiguousarray(law, dtype=np.uint8)
        if per_ch:
            nch = law.numel() if _is_torch(law) else law.size
            if pcm.shape[-1] != N.FRAME or n % (nch * N.FRAME):
                raise IgdError("per-channel law needs pcm shaped [frames][nch][160]")
            self._chk(self._lib.igd_g711_encode_ch(self._h, self._ptr(pcm), self._ptr(law), self._ptr(out),
                                                   n // (nch * N.FRAME), nch, mem))
        else:
            self._chk(self._lib.igd_g711_encode(self._h, self._ptr(pcm), self._ptr(out), n, int(law), mem))
        return out

    # ------------------------------------------------------------ meters
    def frame_meter(self, pcm):
        """pcm int16 [..., 160] -> igd_meter_rec per frame (numpy structured /
        torch int32 [..., 4] raw words)."""
        mem = self._mode(pcm)
        if pcm.shape[-1] != N.FRAME:
            raise IgdError("pcm must be shaped [..., 160]")
        lead = tuple(pcm.shape[:-1])
        nfr = int(np.prod(lead)) if lead else 1
        if mem == N.MEM_DEVICE:
            raw = self._empty(True, (nfr,), N.METER_DT)
            self._chk(self._lib.igd_frame_meter(self._h, self._ptr(pcm), nfr, self._ptr(raw), mem))
            return self._tview(raw[: nfr * 16], torch.int32, lead + (4,))
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        out = np.empty(lead, dtype=N.METER_DT)
        self._chk(self._lib.igd_frame_meter(self._h, self._ptr(pcm), nfr, self._ptr(out), mem))
        return out

    def bytemean(self, payloads, length=None, flags=0):
        """payloads u8 [n][stride] -> reference per-packet level u8 [n]."""
        mem = self._mode(payloads)
        n, stride = payloads.shape
        length = stride if length is None else int(length)
        if mem == N.MEM_DEVICE:
            out = torch.empty(n, dtype=torch.uint8, device=payloads.device)
        else:
            payloads = np.ascontiguousarray(payloads, dtype=np.uint8)
            out = np.empty(n, dtype=np.uint8)
        self._chk(self._lib.igd_bytemean(self._h, self._ptr(payloads), n, length, stride, flags,
                                         self._ptr(out), mem))
        return out

    def level_percent(self, v):
        """AudioMeter scale: int(float(v*100.0/30000.0)) (audiometer.cpp:30-31)."""
        mem = self._mode(v)
        if mem == N.MEM_DEVICE:
            out = torch.empty_like(v)
            n = v.numel()
        else:
            v = np.ascontiguousarray(v, dtype=np.int32)
            out = np.empty(v.shape, dtype=np.int32)
            n = v.size
        self._chk(self._lib.igd_level_percent(self._h, self._ptr(v), n, self._ptr(out), mem))
        return out

    # ------------------------------------------------------------ mix
    def mix(self, pcm, gain, legs):
        """pcm int16 [F][B*legs][160], gain u16 [F][B*legs] -> mix int16 [F][B][160]."""
        mem = self._mode(pcm, gain)
        F, Cn, n = pcm.shape
        if n != N.FRAME or Cn % legs:
            raise IgdError("pcm must be [F][B*legs][160]")
        B = Cn // legs
        if mem == N.MEM_DEVICE:
            out = torch.empty((F, B, N.FRAME), dtype=torch.int16, device=pcm.device)
        else:
            pcm = np.ascontiguousarray(pcm, dtype=np.int16)
            gain = np.ascontiguousarray(gain, dtype=np.uint16)
            out = np.empty((F, B, N.FRAME), dtype=np.int16)
        self._chk(self._lib.igd_mix(self._h, self._ptr(pcm), self._ptr(gain), F, B, legs, self._ptr(out), mem))
        return out

    # ------------------------------------------------------------ fused path
    OUTPUTS = ("mix", "enc", "meter", "bmeter")

    def alloc_outputs(self, F, B, G, want=OUTPUTS):
        """Device output buffers for process_batch (torch); `want` selects which outputs exist."""
        dev = f"cuda:{self.device}"
        o = {
            "mix": lambda: torch.empty((F, B, N.FRAME), dtype=torch.int16, device=dev),
            "enc": lambda: torch.empty((F, B, N.FRAME), dtype=torch.uint8, device=dev),
            "meter": lambda: torch.empty((F, B * G, 4), dtype=torch.int32, device=dev),
            "bmeter": lambda: torch.empty((F, B), dtype=torch.int32, device=dev),
        }
        return {k: o[k]() for k in want}

    @staticmethod
    def _host_outputs(F, B, Cn, want):
        o = {
            "mix": lambda: np.empty((F, B, N.FRAME), dtype=np.int16),
            "enc": lambda: np.empty((F, B, N.FRAME), dtype=np.uint8),
            "meter": lambda: np.empty((F, Cn), dtype=N.METER_DT),
            "bmeter": lambda: np.empty((F, B), dtype=N.BRIDGE_DT),
        }
        return {k: o[k]() for k in want}

    def process_batch(self, codes, law, gain_q7, out_law, legs, flags=0, out=None, want=OUTPUTS):
        """decode -> meter -> gate/gain -> mix -> encode in one pass.

        codes u8 [F][B*legs][160]; law u8 [B*legs]; gain_q7 u16 [F][B*legs]
        (0 = gate shut, bit 15 = GAIN_NO_AUDIO); out_law u8 [B].  Returns dict(mix, enc, meter, bmeter);
        `want` (or the keys of `out`) selects a subset: an output that is not asked for is neither
        stored nor copied back (the int16 mix is 57 % of the result bytes).
        """
        mem = self._mode(codes, law, gain_q7, out_law)
        F, Cn, n = codes.shape
        if n != N.FRAME or Cn % legs:
            raise IgdError("codes must be [F][B*legs][160]")
        B = Cn // legs
        if mem == N.MEM_DEVICE:
            if codes.dtype != torch.uint8 or law.dtype != torch.uint8 or out_law.dtype != torch.uint8:
                raise IgdError("codes/law/out_law must be uint8")
            if gain_q7.dtype not in (torch.int16, torch.uint16):
                raise IgdError("gain_q7 must be a 16-bit tensor")
            o = out if out is not None else self.alloc_outputs(F, B, legs, want)
        else:
            codes = np.ascontiguousarray(codes, dtype=np.uint8)
            law = np.ascontiguousarray(law, dtype=np.uint8)
            gain_q7 = np.ascontiguousarray(gain_q7, dtype=np.uint16)
            out_law = np.ascontiguousarray(out_law, dtype=np.uint8)
            o = out if out is not None else self._host_outputs(F, B, Cn, want)
        if law.shape[0] != Cn or out_law.shape[0] != B or tuple(gain_q7.shape) != (F, Cn):
            raise IgdError("law / out_law / gain_q7 shapes do not match codes")
        d = N.BatchDesc(C.sizeof(N.BatchDesc), mem, F, B, legs, flags,
                        self._ptr(codes), self._ptr(law), self._ptr(gain_q7), self._ptr(out_law),
                        self._ptr(o.get("mix")), self._ptr(o.get("enc")), self._ptr(o.get("meter")),
                        self._ptr(o.get("bmeter")))
        self._chk(self._lib.igd_process_batch(self._h, C.byref(d)))
        return o

    def process_packets(self, pkts, fields, law, gain_q7, out_law, legs=4, flags=0, out=None, want=OUTPUTS):
        """process_batch with the codes read straight out of the raw ED-137 packets.

        pkts u8 [F][B*legs][180] as received; fields [F][B*legs] from ed137_parse; the rest as
        process_batch.  A leg-frame whose packet is not a whole G.711 audio frame (keep-alive,
        truncated, dropped, absent) is silent (GAIN_NO_AUDIO); otherwise identical results to
        ed137_parse(...)[1] fed to process_batch.  legs = 4 runs one kernel; other leg counts
        extract the payloads inside the library first.
        """
        mem = self._mode(pkts, fields, law, gain_q7, out_law)
        F, Cn, n = pkts.shape
        if n != N.PKT_MAX or Cn % legs:
            raise IgdError("pkts must be [F][B*legs][180]")
        B = Cn // legs
        if mem == N.MEM_DEVICE:
            if pkts.dtype != torch.uint8 or law.dtype != torch.uint8 or out_law.dtype != torch.uint8:
                raise IgdError("pkts/law/out_law must be uint8")
            o = out if out is not None else self.alloc_outputs(F, B, legs, want)
        else:
            pkts = np.ascontiguousarray(pkts, dtype=np.uint8)
            fields = np.ascontiguousarray(fields, dtype=N.FIELDS_DT)
            law = np.ascontiguousarray(law, dtype=np.uint8)
            gain_q7 = np.ascontiguousarray(gain_q7, dtype=np.uint16)
            out_law = np.ascontiguousarray(out_law, dtype=np.uint8)
            o = out if out is not None else self._host_outputs(F, B, Cn, want)
        if law.shape[0] != Cn or out_law.shape[0] != B or tuple(gain_q7.shape) != (F, Cn):
            raise IgdError("law / out_law / gain_q7 shapes do not match pkts")
        d = N.PacketsDesc(C.sizeof(N.PacketsDesc), mem, F, B, legs, flags,
                          self._ptr(pkts), self._ptr(fields), self._ptr(law), self._ptr(gain_q7), self._ptr(out_law),
                          self._ptr(o.get("mix")), self._ptr(o.get("enc")), self._ptr(o.get("meter")),
                          self._ptr(o.get("bmeter")))
        self._chk(self._lib.igd_process_packets(self._h, C.byref(d)))
        return o

    # ------------------------------------------------------------ summary
    def event_summary(self, meter, gain_q7, want_db=True):
        """meter [F][C] records, gain_q7 [F][C] -> (summary [C], db [C])."""
        mem = self._mode(meter, gain_q7)
        if mem == N.MEM_DEVICE:
            F, Cn = gain_q7.shape
            out = torch.empty((Cn, 8), dtype=torch.int32, device=gain_q7.device)
            db = torch.empty((Cn, 4), dtype=torch.int32, device=gain_q7.device) if want_db else None
        else:
            meter = np.ascontiguousarray(meter, dtype=N.METER_DT)
            gain_q7 = np.ascontiguousarray(gain_q7, dtype=np.uint16)
            F, Cn = gain_q7.shape
            out = np.empty(Cn, dtype=N.SUMMARY_DT)
            db = np.empty(Cn, dtype=N.SUMMARY_DB_DT) if want_db else None
        self._chk(self._lib.igd_event_summary(self._h, self._ptr(meter), self._ptr(gain_q7), F, Cn,
                                              self._ptr(out), self._ptr(db), mem))
        return out, db

    # ------------------------------------------------------------ ED-137
    def ed137_parse(self, pkts, sizes=None, want_payload=True):
        """pkts u8 [n][stride] (+ sizes u32 [n]) -> (fields [n], payload u8 [n][160])."""
        mem = self._mode(pkts, sizes)
        n, stride = pkts.shape
        if mem == N.MEM_DEVICE:
            fields = torch.empty((n, 4), dtype=torch.int32, device=pkts.device)
            pay = torch.empty((n, N.FRAME), dtype=torch.uint8, device=pkts.device) if want_payload else None
        else:
            pkts = np.ascontiguousarray(pkts, dtype=np.uint8)
            if sizes is not None:
                sizes = np.ascontiguousarray(sizes, dtype=np.uint32)
            fields = np.empty(n, dtype=N.FIELDS_DT)
            pay = np.empty((n, N.FRAME), dtype=np.uint8) if want_payload else None
        self._chk(self._lib.igd_ed137_parse(self._h, self._ptr(pkts), self._ptr(sizes), n, stride,
                                            self._ptr(fields), self._ptr(pay), mem))
        return fields, pay

    def ed137_pack(self, rtp12, payload, state, ctl=None, now_ms0=0, tick_ms=20, payload_len=N.FRAME,
                   out_stride=N.PKT_MAX, flags=0, stale_payload=None):
        """Batched transport_send_rtp.  rtp12 u8 [F][C][12], payload u8 [F][C][160],
        state [C] (updated in place), ctl [F][C] or None.
        Returns (pkts u8 [F][C][out_stride], sizes u32 [F][C], bytemean_out u8 [F][C])."""
        mem = self._mode(rtp12, payload, state, ctl, stale_payload)
        F, Cn = rtp12.shape[0], rtp12.shape[1]
        if mem == N.MEM_DEVICE:
            dev = rtp12.device
            pkts = torch.empty((F, Cn, out_stride), dtype=torch.uint8, device=dev)   # the kernels define every byte
            sizes = torch.empty((F, Cn), dtype=torch.int32, device=dev)
            bm = torch.empty((F, Cn), dtype=torch.uint8, device=dev)
        else:
            rtp12 = np.ascontiguousarray(rtp12, dtype=np.uint8)
            payload = np.ascontiguousarray(payload, dtype=np.uint8)
            if state.dtype != N.STATE_DT or not state.flags.c_contiguous:
                raise IgdError("state must be a contiguous STATE_DT array (updated in place)")
            if ctl is not None:
                ctl = np.ascontiguousarray(ctl, dtype=N.CTL_DT)
            pkts = np.zeros((F, Cn, out_stride), dtype=np.uint8)
            sizes = np.empty((F, Cn), dtype=np.uint32)
            bm = np.empty((F, Cn), dtype=np.uint8)
        d = N.PackDesc(C.sizeof(N.PackDesc), mem, F, Cn, flags, payload_len, out_stride, tick_ms, now_ms0,
                       self._ptr(rtp12), self._ptr(payload), self._ptr(ctl), self._ptr(state),
                       self._ptr(pkts), self._ptr(sizes), self._ptr(bm), self._ptr(stale_payload))
        self._chk(self._lib.igd_ed137_pack(self._h, C.byref(d)))
        return pkts, sizes, bm

    def ed137_keepalive(self, hdr20, state, now_ms):
        """Batched sendR2SStatus: hdr20 u8 [C][20] (each adapter's send-buffer header, in/out), state [C]
        (in/out) -> sizes [C] (20 where a keep-alive leaves, else 0)."""
        mem = self._mode(hdr20, state)
        Cn = hdr20.shape[0]
        sizes = torch.empty((Cn,), dtype=torch.int32, device=hdr20.device) if mem == N.MEM_DEVICE else np.empty(Cn, np.uint32)
        self._chk(self._lib.igd_ed137_keepalive(self._h, self._ptr(hdr20), self._ptr(state), Cn, int(now_ms),
                                                self._ptr(sizes), mem))
        return sizes

    # ------------------------------------------------------------ RX liveness, gate arbitration
    def rx_track(self, fields, state, present=None, now_ms0=0, tick_ms=20, r2s_period_ms=200, wd_ticks=2,
                 frame0=0):
        """Batched receive-side state of transport_rtp_cb + the R2S watchdog.
        fields [F][C] (from ed137_parse), state [C] (RX_STATE_DT, updated in place),
        present u8 [F][C] or None.  Returns events [F][C] (RX_EVENT_DT)."""
        mem = self._mode(fields, state, present)
        F, Cn = fields.shape[0], fields.shape[1]
        if mem == N.MEM_DEVICE:
            events = torch.empty((F, Cn, 2), dtype=torch.int32, device=fields.device)
        else:
            fields = np.ascontiguousarray(fields, dtype=N.FIELDS_DT)
            if present is not None:
                present = np.ascontiguousarray(present, dtype=np.uint8)
            events = np.empty((F, Cn), dtype=N.RX_EVENT_DT)
        d = N.RxTrackDesc(C.sizeof(N.RxTrackDesc), mem, F, Cn, int(tick_ms), int(r2s_period_ms), int(wd_ticks),
                          int(frame0), int(now_ms0), self._ptr(fields), self._ptr(present), self._ptr(state),
                          self._ptr(events), None)
        self._chk(self._lib.igd_rx_track(self._h, C.byref(d)))
        return events

    def gate_arbitrate(self, words, legs, bridges, G, mode=N.ARB_CLIENT_PTT, active=None, silence=False):
        """checkEvents() gate decisions.  words: u32 [F][B*G] or an RX_EVENT_DT array [F][B*G]
        (its .word is read in place); legs [B*G] (ARB_LEG_DT) and bridges [B] (ARB_BRIDGE_DT)
        are updated in place.  Returns gain_q7 u16 [F][B*G] for process_batch.
        silence=True (words must be rx_track events): ticks without a whole audio frame
        (no RXE_FRAME) carry GAIN_NO_AUDIO, i.e. the leg is silent while keep-alives arrive."""
        mem = self._mode(words, legs, bridges, active)
        F, Cn = words.shape[0], words.shape[1]
        B = Cn // G
        if mem == N.MEM_DEVICE:
            stride = 8 if (words.dim() == 3 and words.shape[2] == 2) else 4
            gain = torch.empty((F, Cn), dtype=torch.int16, device=words.device)
        else:
            stride = 8 if words.dtype == N.RX_EVENT_DT else 4
            words = np.ascontiguousarray(words) if stride == 8 else np.ascontiguousarray(words, dtype=np.uint32)
            if active is not None:
                active = np.ascontiguousarray(active, dtype=np.uint8)
            gain = np.empty((F, Cn), dtype=np.uint16)
        if silence and stride != 8:
            raise ValueError("silence=True needs the rx_track events as `words`")
        d = N.ArbDesc(C.sizeof(N.ArbDesc), mem, F, B, int(G), int(mode), stride, N.ARB_F_SILENCE if silence else 0,
                      self._ptr(words),
                      self._ptr(active), self._ptr(legs), self._ptr(bridges), self._ptr(gain))
        self._chk(self._lib.igd_gate_arbitrate(self._h, C.byref(d)))
        return gain

    # ------------------------------------------------------------ gateway: packets in, packets out
    def gateway_process(self, rx_pkts, law, out_law, rx_state, arb_legs, arb_bridges, tx_rtp12, tx_state, rx_sizes=None,
                        tx_ctl=None, active=None, mode=N.ARB_CLIENT_PTT, now_ms0=0, tick_ms=20, r2s_period_ms=200,
                        wd_ticks=2, frame0=0, flags=0, want=("meter", "bmeter"), out=None):
        """The whole per-tick voice path in one call (igd_gateway_process): received ED-137 packets of every leg
        in, finished ED-137 packets of every bridge out.  rx_pkts u8 [F][B*4][180]; rx_sizes u32 [F][B*4] or None;
        tx_rtp12 u8 [F][B][12]; states (rx_state RX_STATE_DT [B*4], arb_legs ARB_LEG_DT [B*4], arb_bridges
        ARB_BRIDGE_DT [B], tx_state STATE_DT [B]) are updated in place.  Returns dict(tx_pkts [F][B][180],
        tx_sizes [F][B]) plus the optional outputs named in `want` (rx_events, gain_q7, meter, bmeter, mix, enc)."""
        mem = self._mode(rx_pkts, law, out_law, rx_state, arb_legs, arb_bridges, tx_rtp12, tx_state, rx_sizes, tx_ctl, active)
        F, Cn, n = rx_pkts.shape
        if n != N.PKT_MAX or Cn % 4:
            raise IgdError("rx_pkts must be [F][B*4][180]")
        B = Cn // 4
        if out is not None:
            o = out
        elif mem == N.MEM_DEVICE:
            dev = rx_pkts.device
            mk = {"tx_pkts": lambda: torch.empty((F, B, N.PKT_MAX), dtype=torch.uint8, device=dev),
                  "tx_sizes": lambda: torch.empty((F, B), dtype=torch.int32, device=dev),
                  "rx_events": lambda: torch.empty((F, Cn, 2), dtype=torch.int32, device=dev),
                  "gain_q7": lambda: torch.empty((F, Cn), dtype=torch.int16, device=dev),
                  "meter": lambda: torch.empty((F, Cn, 4), dtype=torch.int32, device=dev),
                  "bmeter": lambda: torch.empty((F, B), dtype=torch.int32, device=dev),
                  "mix": lambda: torch.empty((F, B, N.FRAME), dtype=torch.int16, device=dev),
                  "enc": lambda: torch.empty((F, B, N.FRAME), dtype=torch.uint8, device=dev)}
            o = {k: mk[k]() for k in ("tx_pkts", "tx_sizes") + tuple(want)}
        else:
            rx_pkts = np.ascontiguousarray(rx_pkts, dtype=np.uint8)
            if rx_sizes is not None:
                rx_sizes = np.ascontiguousarray(rx_sizes, dtype=np.uint32)
            law = np.ascontiguousarray(law, dtype=np.uint8)
            out_law = np.ascontiguousarray(out_law, dtype=np.uint8)
            tx_rtp12 = np.ascontiguousarray(tx_rtp12, dtype=np.uint8)
            mk = {"tx_pkts": lambda: np.empty((F, B, N.PKT_MAX), np.uint8), "tx_sizes": lambda: np.empty((F, B), np.uint32),
                  "rx_events": lambda: np.empty((F, Cn), N.RX_EVENT_DT), "gain_q7": lambda: np.empty((F, Cn), np.uint16),
                  "meter": lambda: np.empty((F, Cn), N.METER_DT), "bmeter": lambda: np.empty((F, B), N.BRIDGE_DT),
                  "mix": lambda: np.empty((F, B, N.FRAME), np.int16), "enc": lambda: np.empty((F, B, N.FRAME), np.uint8)}
            o = {k: mk[k]() for k in ("tx_pkts", "tx_sizes") + tuple(want)}
        d = N.GatewayDesc(C.sizeof(N.GatewayDesc), mem, F, B, 4, int(flags), int(mode), int(tick_ms), int(r2s_period_ms),
                          int(wd_ticks), int(frame0), 0, int(now_ms0),
                          self._ptr(rx_pkts), self._ptr(rx_sizes), self._ptr(law), self._ptr(active), self._ptr(rx_state),
                          self._ptr(arb_legs), self._ptr(arb_bridges), self._ptr(out_law), self._ptr(tx_rtp12),
                          self._ptr(tx_ctl), self._ptr(tx_state), self._ptr(o["tx_pkts"]), self._ptr(o["tx_sizes"]),
                          self._ptr(o.get("rx_events")), self._ptr(o.get("gain_q7")), self._ptr(o.get("meter")),
                          self._ptr(o.get("bmeter")), self._ptr(o.get("mix")), self._ptr(o.get("enc")))
        self._chk(self._lib.igd_gateway_process(self._h, C.byref(d)))
        return o

    def gateway_fanout(self, pcm, law, tx_rtp12, tx_state, tx_ctl=None, now_ms0=0, tick_ms=20, flags=0, level=True,
                       out=None):
        """The other direction of a bridge (igd_gateway_fanout): one PCM frame per bridge and tick in, a finished
        ED-137 packet for every leg of the bridge out, each encoded in its leg's law and sent with its leg's sender
        state.  pcm int16 [F][B][160]; law u8 [B*G]; tx_rtp12 u8 [F][B*G][12]; tx_ctl [F][B*G] or None; tx_state
        STATE_DT [B*G] is updated in place.  Returns dict(tx_pkts [F][B*G][180], tx_sizes [F][B*G]) plus tx_level
        [F][B*G] when `level`; `out` (such a dict) is written instead of fresh buffers, e.g. inside a CUDA graph."""
        mem = self._mode(pcm, law, tx_rtp12, tx_state, tx_ctl)
        F, B, n = pcm.shape
        Cn = law.numel() if _is_torch(law) else np.size(law)
        if n != N.FRAME or B == 0 or Cn % B:
            raise IgdError("pcm must be [F][B][160] and law [B*G]")
        G = Cn // B
        if tuple(tx_rtp12.shape[:2]) != (F, Cn):
            raise IgdError("tx_rtp12 must be [F][B*G][12]")
        keys = ("tx_pkts", "tx_sizes") + (("tx_level",) if level else ())
        if mem == N.MEM_DEVICE:
            dev = pcm.device
            mk = {"tx_pkts": lambda: torch.empty((F, Cn, N.PKT_MAX), dtype=torch.uint8, device=dev),
                  "tx_sizes": lambda: torch.empty((F, Cn), dtype=torch.int32, device=dev),
                  "tx_level": lambda: torch.empty((F, Cn), dtype=torch.uint8, device=dev)}
        else:
            pcm = np.ascontiguousarray(pcm, dtype=np.int16)
            law = np.ascontiguousarray(law, dtype=np.uint8)
            tx_rtp12 = np.ascontiguousarray(tx_rtp12, dtype=np.uint8)
            if tx_state.dtype != N.STATE_DT or not tx_state.flags.c_contiguous:
                raise IgdError("tx_state must be a contiguous STATE_DT array (updated in place)")
            if tx_ctl is not None:
                tx_ctl = np.ascontiguousarray(tx_ctl, dtype=N.CTL_DT)
            mk = {"tx_pkts": lambda: np.empty((F, Cn, N.PKT_MAX), np.uint8), "tx_sizes": lambda: np.empty((F, Cn), np.uint32),
                  "tx_level": lambda: np.empty((F, Cn), np.uint8)}
        o = out if out is not None else {k: mk[k]() for k in keys}
        d = N.FanoutDesc(C.sizeof(N.FanoutDesc), mem, F, B, G, int(flags), int(tick_ms), 0, int(now_ms0),
                         self._ptr(pcm), self._ptr(law), self._ptr(tx_rtp12), self._ptr(tx_ctl), self._ptr(tx_state),
                         self._ptr(o["tx_pkts"]), self._ptr(o["tx_sizes"]), self._ptr(o.get("tx_level")))
        self._chk(self._lib.igd_gateway_fanout(self._h, C.byref(d)))
        return o

    def gateway_fanout_packets(self, rx_pkts, in_law, law, tx_rtp12, tx_state, rx_sizes=None, tx_ctl=None, now_ms0=0,
                               tick_ms=20, flags=0, level=True, out=None):
        """gateway_fanout with slot 0 as received from the console call (igd_gateway_fanout_packets): the console's
        ED-137 packets in, a finished packet for every leg of the bridge out.  rx_pkts u8 [F][B][180] as received;
        rx_sizes u32 [F][B] or None (all 180); in_law u8 [B] the console call's law; law u8 [B*G]; tx_rtp12 u8
        [F][B*G][12]; tx_ctl [F][B*G] or None; tx_state STATE_DT [B*G] is updated in place.  Every leg of bridge b
        sends the G.711 frame of rx_pkts[f][b] decoded in in_law[b], or digital silence where that packet is not a
        whole audio frame.  Returns dict(tx_pkts [F][B*G][180], tx_sizes [F][B*G]) plus tx_level [F][B*G] when
        `level`; `out` (such a dict) is written instead of fresh buffers, e.g. inside a CUDA graph."""
        mem = self._mode(rx_pkts, in_law, law, tx_rtp12, tx_state, rx_sizes, tx_ctl)
        F, B, n = rx_pkts.shape
        Cn = law.numel() if _is_torch(law) else np.size(law)
        nin = in_law.numel() if _is_torch(in_law) else np.size(in_law)
        if n != N.PKT_MAX or B == 0 or Cn % B or nin != B:
            raise IgdError("rx_pkts must be [F][B][180], in_law [B] and law [B*G]")
        G = Cn // B
        if tuple(tx_rtp12.shape[:2]) != (F, Cn):
            raise IgdError("tx_rtp12 must be [F][B*G][12]")
        keys = ("tx_pkts", "tx_sizes") + (("tx_level",) if level else ())
        if mem == N.MEM_DEVICE:
            dev = rx_pkts.device
            mk = {"tx_pkts": lambda: torch.empty((F, Cn, N.PKT_MAX), dtype=torch.uint8, device=dev),
                  "tx_sizes": lambda: torch.empty((F, Cn), dtype=torch.int32, device=dev),
                  "tx_level": lambda: torch.empty((F, Cn), dtype=torch.uint8, device=dev)}
        else:
            rx_pkts = np.ascontiguousarray(rx_pkts, dtype=np.uint8)
            if rx_sizes is not None:
                rx_sizes = np.ascontiguousarray(rx_sizes, dtype=np.uint32)
            in_law = np.ascontiguousarray(in_law, dtype=np.uint8)
            law = np.ascontiguousarray(law, dtype=np.uint8)
            tx_rtp12 = np.ascontiguousarray(tx_rtp12, dtype=np.uint8)
            if tx_state.dtype != N.STATE_DT or not tx_state.flags.c_contiguous:
                raise IgdError("tx_state must be a contiguous STATE_DT array (updated in place)")
            if tx_ctl is not None:
                tx_ctl = np.ascontiguousarray(tx_ctl, dtype=N.CTL_DT)
            mk = {"tx_pkts": lambda: np.empty((F, Cn, N.PKT_MAX), np.uint8), "tx_sizes": lambda: np.empty((F, Cn), np.uint32),
                  "tx_level": lambda: np.empty((F, Cn), np.uint8)}
        o = out if out is not None else {k: mk[k]() for k in keys}
        d = N.FanoutPktDesc(C.sizeof(N.FanoutPktDesc), mem, F, B, G, int(flags), int(tick_ms), 0, int(now_ms0),
                            self._ptr(rx_pkts), self._ptr(rx_sizes), self._ptr(in_law), self._ptr(law),
                            self._ptr(tx_rtp12), self._ptr(tx_ctl), self._ptr(tx_state), self._ptr(o["tx_pkts"]),
                            self._ptr(o["tx_sizes"]), self._ptr(o.get("tx_level")))
        self._chk(self._lib.igd_gateway_fanout_packets(self._h, C.byref(d)))
        return o

    # ------------------------------------------------------------ recorder
    def wav_image(self, payload, rate=8000, law=N.LAW_ULAW, ref_quirks=False):
        """WavWriter file image (header + body) built on the GPU."""
        mem = self._mode(payload)
        n = payload.numel() if mem == N.MEM_DEVICE else payload.size
        total = self._lib.igd_wav_size(n, int(ref_quirks))
        if mem == N.MEM_DEVICE:
            out = torch.empty(total, dtype=torch.uint8, device=payload.device)
        else:
            payload = np.ascontiguousarray(payload, dtype=np.uint8)
            out = np.empty(total, dtype=np.uint8)
        ln = C.c_size_t()
        self._chk(self._lib.igd_wav_image(self._h, self._ptr(payload), n, rate, law, int(ref_quirks),
                                          self._ptr(out), C.byref(ln), mem))
        return out

    def wav_images(self, codes, chans=None, law=None, rate=8000, ref_quirks=False):
        """WavWriter file images of many channels at once, gathered from codes u8 [F][C][160].
        chans: u32 channel indices (None = every channel); law u8 [C] (None = u-law).
        Returns u8 [len(chans)][image bytes]."""
        mem = self._mode(codes, chans, law)
        F, Cn = codes.shape[0], codes.shape[1]
        nch = Cn if chans is None else (chans.numel() if mem == N.MEM_DEVICE else len(chans))
        size = self._lib.igd_wav_size(F * N.FRAME, int(ref_quirks))
        stride = (size + 3) & ~3
        if mem == N.MEM_DEVICE:
            out = torch.zeros((nch, stride), dtype=torch.uint8, device=codes.device)
        else:
            codes = np.ascontiguousarray(codes, dtype=np.uint8)
            chans = None if chans is None else np.ascontiguousarray(chans, dtype=np.uint32)
            law = None if law is None else np.ascontiguousarray(law, dtype=np.uint8)
            out = np.zeros((nch, stride), dtype=np.uint8)
        self._chk(self._lib.igd_wav_images(self._h, self._ptr(codes), F, Cn, self._ptr(chans), nch, self._ptr(law),
                                           int(rate), int(ref_quirks), self._ptr(out), stride, mem))
        return out[:, :size]
