#!/usr/bin/env python
"""Generates the committed fixtures under tests/golden/.

Run in the BUILD container (needs /root/reference for the reference-backed
probe oracle/_ref/libigd_ref.so):   python tests/golden/make_golden.py

  ed137_ref_headers.json  20-byte headers produced THROUGH THE REFERENCE'S OWN
                          struct custom_rtp_hdr (ed137_rtp.h:22-47) with the
                          byte-order calls of TransportAdapter.cpp:725-727,800
  wavwriter_ref.bin       file written by the reference's own WavWriter.cpp
                          (start/wav_write/stop) for wavwriter_payload.bin
  g711_pins.json          SHA-256 of the four G.711 tables (SURVEY Appendix B)
                          + ITU known answers
  ed137_tx_scenarios.json sender scenarios and the packets the REFERENCE'S OWN
                          transport_send_rtp emits (TransportAdapter.cpp compiled from
                          /root/reference into oracle/_ref/libigd_ref_ta.so, driven through
                          tp->op->send_rtp by tests/ref_py.run_tx)
  ref_pins.json           SHA-256 digests of the REFERENCE run (same library) on every
                          shared seeded case: sender scenarios (both `char` signs), sendR2SStatus,
                          the transport_rtp_cb walk, checkEvents gate arbitration (CLIENT / SERVER
                          best signal) and the PTTEventDataLogger messages; the oracle has to
                          reproduce them (tests/test_ref_pins.py)
  fused_cfg2.npz          BASELINE config 2 (4 legs, 2 u-law + 2 A-law), 75
                          frames: inputs + oracle outputs
  rx_arb_keepalive.json   SHA-256 of the oracle's receive-side walk (transport_rtp_cb
                          + R2S watchdog), gate arbitration (CLIENT PTT priority,
                          SERVER best signal), sendR2SStatus and the
                          PTTEventDataLogger message on the seeded cases of
                          tests/rx_arb_cases.py / keepalive_cases.py
  live_cases.json         the oracle's side of every *_live comparison of
                          tests/test_ref_pins.py that ref_pins.json does not pin (final
                          sender state, CSRC / extension offsets, setIncomingRTP,
                          non-radio callback, field getters, setters, arbitration at
                          G = 2 / 3 / 7 / 32 and with inactive legs, split-run receive
                          state), so that they are compared without the reference build.
                          Written by `python tests/golden/make_golden.py live_cases`, and
                          only where those *_live tests pass against the reference
"""
import ctypes as C
import glob
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)
import oracle_py as O  # noqa: E402
from igate4xsoftphonedsp_b200 import synth  # noqa: E402
from tx_scenarios import SCENARIOS, run_oracle  # noqa: E402
import ref_py as RP  # noqa: E402


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def ref_headers():
    R = O.ref()
    rng = np.random.default_rng(137)
    cases = []
    words = [0x00000000, 0x00013100, 0x000131C0, 0x00013140, 0x00013180, 0x00413100, 0x104131F8,
             0x20013100, 0xE0013100, 0x10013178, 0xFFFFFFFF]
    for w in words:
        for pt in (8, 0, 18, 123, 96):
            m = int(rng.integers(0, 2))
            seq, ts, ssrc = int(rng.integers(0, 65536)), int(rng.integers(0, 2**32)), int(rng.integers(0, 2**32))
            buf = np.zeros(20, np.uint8)
            R.ref_hdr_build(buf.ctypes.data, 2, 0, 1, 0, m, pt, seq, ts, ssrc, 0x0167, 1, w)
            f = (C.c_uint * 12)()
            R.ref_hdr_parse(buf.ctypes.data, f)
            cases.append({"v": 2, "p": 0, "x": 1, "cc": 0, "m": m, "pt": pt, "seq": seq, "ts": ts, "ssrc": ssrc,
                          "profile": 0x0167, "length": 1, "word": w, "hex": buf.tobytes().hex(),
                          "parsed_by_ref": [int(v) for v in f]})
    # stamping an existing PJSIP header the way transport_send_rtp does
    stamps = []
    for w, m, ptov in ((0x00413100, 1, -1), (0x10013178, 0, 123), (0x600131C0, 0, -1)):
        base = synth.rtp12(1, 1, [8])[0, 0]
        buf = np.zeros(20, np.uint8)
        buf[:12] = base
        buf[12:] = [0xAA] * 8
        before = buf.tobytes().hex()
        R.ref_hdr_stamp(buf.ctypes.data, m, w, ptov)
        stamps.append({"before": before, "m": m, "word": w, "pt_override": ptov, "after": buf.tobytes().hex()})
    return {"sizeof": R.ref_hdr_sizeof(), "cases": cases, "stamps": stamps}


def wavwriter():
    R = O.ref()
    rng = np.random.default_rng(7)
    payload = rng.integers(0, 256, 480, dtype=np.uint8)
    with tempfile.TemporaryDirectory() as d:
        prefix = os.path.join(d, "ref_").encode()
        assert R.ref_wavwriter_run(prefix, 8000, payload.ctypes.data, payload.size, 160) == 0
        files = glob.glob(os.path.join(d, "ref_*.wav"))
        assert len(files) == 1
        data = open(files[0], "rb").read()
    payload.tofile(os.path.join(HERE, "wavwriter_payload.bin"))
    open(os.path.join(HERE, "wavwriter_ref.bin"), "wb").write(data)
    return len(data)


def g711_pins():
    L = O.lib()
    return {
        "sha256": {"alaw_decode": sha(O.decode_table(0)), "ulaw_decode": sha(O.decode_table(1)),
                   "alaw_encode": sha(O.encode_table(0)), "ulaw_encode": sha(O.encode_table(1))},
        "known_answers": {"alaw": {str(v): L.orc_lin2alaw(v) for v in (0, -1, 32767, -32768, 8, -8, 255, 256)},
                          "ulaw": {str(v): L.orc_lin2ulaw(v) for v in (0, -1, 32767, -32768, 4, -4, 123, -124)}},
    }


def fused_cfg2():
    F, B, G = 75, 1, 4
    # channels 64..67: the A=16000 amplitude class, so two open legs at gain 2.0 saturate
    pcm = synth.pcm_noise_tone(F, B * G, ch0=64)
    law = synth.laws(B * G, ch0=64)
    codes = np.stack([O.g711_encode(pcm[:, c], int(law[c])) for c in range(B * G)], axis=1)
    gain = synth.gains(F, B, G)
    out_law = synth.out_laws(B)
    mix, enc, meter, bmeter = O.process_batch(codes, law, gain, out_law, G)
    np.savez_compressed(os.path.join(HERE, "fused_cfg2.npz"), codes=codes, law=law, gain=gain, out_law=out_law,
                        mix=mix, enc=enc, meter=meter.view(np.uint32).reshape(F, B * G, 4),
                        bmeter=bmeter.view(np.uint32).reshape(F, B))
    return sha(mix), sha(enc)


def rx_arb_keepalive():
    import keepalive_cases as K
    import rx_arb_cases as R
    from igate4xsoftphonedsp_b200 import _native as N
    out = {}
    pkts, sizes, present = R.make_rx_stream(300, 24, seed=3)
    ev, st = R.oracle_rx_walk(pkts, sizes, present)
    out["rx_walk"] = {"inputs": sha(pkts) + sha(sizes) + sha(present), "events": sha(ev), "state": sha(st),
                      "edges": int(((ev["flags"] & N.RXE_EDGE) != 0).sum()),
                      "hangups": int(((ev["flags"] & N.RXE_HANGUP) != 0).sum())}
    for name, mode, G in (("client_ptt", N.ARB_CLIENT_PTT, 4), ("server_best", N.ARB_SERVER_BEST, 4)):
        w = R.make_arb_words(200, 9, G, mode, seed=G)
        gain, legs, br = R.oracle_arb_walk(w, G, mode)
        out[name] = {"inputs": sha(w), "gain": sha(gain), "legs": sha(legs), "bridges": sha(br),
                     "open_leg_frames": int((gain == 256).sum())}
    legs, hdr, ctl = K.make(40, 120, seed=2)
    pk, sz, hfin = K.oracle_walk(legs, hdr, ctl)
    out["keepalive"] = {"packets": sha(pk), "sizes": sha(sz), "final_headers": sha(hfin), "sent": int((sz == 20).sum())}
    buf = C.create_string_buffer(1024)
    n = O.lib().orc_ptt_event_json(buf, 1024, 3, b"pptTest_released", 61.25, 70.5, 12.0412, b"sip:radio1@10.0.0.5", 133, 201, 17)
    out["ptt_event_json"] = buf.raw[:n].decode()
    return out


def ref_pins():
    """the digest tests/test_ref_pins._oracle_digest computes with the oracle, computed with the REFERENCE"""
    import keepalive_cases as K
    import rx_arb_cases as R
    from igate4xsoftphonedsp_b200 import _native as N
    out = {"generated_from": "reference",
           "how": "oracle/_ref/libigd_ref_ta{,_sc}.so = /root/reference/TransportAdapter.cpp + line-range extracts of "
                  "roip_ed137.cpp / Functions.cpp (oracle/ref_extract.sh), driven by tests/ref_py.py",
           "tx": {}}
    for s in SCENARIOS:
        pk, sz, bm, _ = RP.run_tx(s)
        out["tx"][s["name"]] = {"packets": sha(pk), "sizes": sha(sz), "bytemean": sha(bm), "bytes": int(sz.sum())}
    pk, sz, bm, _ = RP.run_tx(SCENARIOS[0], signed_char=1)
    out["tx_signed_char"] = {"packets": sha(pk), "bytemean": sha(bm)}
    legs, hdr, ctl = K.make(40, 120, seed=2)
    pk, sz, hf = RP.run_keepalive(legs, hdr, ctl)
    out["keepalive"] = {"packets": sha(pk), "sizes": sha(sz), "final_headers": sha(hf)}
    pkts, sizes, present = R.make_rx_stream(300, 24, seed=3)
    ev, st = RP.run_rx(pkts, R.ref_comparable_sizes(sizes), present)
    out["rx_walk"] = {"events": sha(ev), "state": sha(st)}
    for name, mode, G in (("client_ptt", N.ARB_CLIENT_PTT, 4), ("server_best", N.ARB_SERVER_BEST, 4)):
        w = R.make_arb_words(200, 9, G, mode, seed=G)
        g, lg, br = RP.run_arb(w, G, mode)
        out[name] = {"gain": sha(g), "legs": sha(lg), "bridges": sha(br)}
    import test_ref_pins as TP
    msgs = []
    Rf = RP.lib(0)
    for seed in (1, 2, 3):
        meter, gain, s, bm = TP._event_case(seed)
        Rf.refapp_reset(RP.SERVER, 1)
        buf = C.create_string_buffer(2048)
        Rf.refapp_ptt_event(0, b"pptTest_pressed", 4.0, b"sip:radio1@10.0.0.5", 3, buf, 2048)
        for f in range(meter.shape[0]):
            if gain[f, 0]:
                Rf.refapp_keeplog(0, float(s[f]) / 160.0, int(bm[f]))
        Rf.refapp_ptt_event(0, b"pptTest_released", 0.0, b"sip:radio1@10.0.0.5", 3, buf, 2048)
        msgs.append(buf.value.decode())
    out["event_messages"] = msgs
    return out


def main():
    if not O.ref_available() or not RP.available():
        sys.exit("oracle/_ref/libigd_ref*.so missing: run `make -C oracle` where /root/reference exists")
    json.dump(ref_headers(), open(os.path.join(HERE, "ed137_ref_headers.json"), "w"), indent=1)
    print("wavwriter_ref.bin", wavwriter(), "bytes")
    json.dump(g711_pins(), open(os.path.join(HERE, "g711_pins.json"), "w"), indent=1)
    scen = []
    for s in SCENARIOS:
        pk, sizes, bm, st = RP.run_tx(s)          # the reference's own transport_send_rtp
        opk, osz, obm, _ = run_oracle(s)
        assert np.array_equal(pk, opk) and np.array_equal(sizes, osz) and np.array_equal(bm, obm), s["name"]
        scen.append({"name": s["name"], "sha256_packets": sha(pk), "sizes": sizes.tolist(),
                     "bytemean": bm.tolist(), "first_packets_hex": [pk[f, 0, :sizes[f, 0]].tobytes().hex()
                                                                    for f in range(min(4, pk.shape[0]))]})
    json.dump(scen, open(os.path.join(HERE, "ed137_tx_scenarios.json"), "w"), indent=1)
    print("fused_cfg2", fused_cfg2())
    json.dump(rx_arb_keepalive(), open(os.path.join(HERE, "rx_arb_keepalive.json"), "w"), indent=1)
    json.dump(ref_pins(), open(os.path.join(HERE, "ref_pins.json"), "w"), indent=1)


def live_cases():
    import test_ref_pins as TP
    return TP._live_case_digest()


if __name__ == "__main__":
    if sys.argv[1:] == ["live_cases"]:
        json.dump(live_cases(), open(os.path.join(HERE, "live_cases.json"), "w"), indent=1)
    else:
        main()
