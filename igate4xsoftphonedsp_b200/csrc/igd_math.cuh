// igd_math.cuh -- scalar building blocks of the voice-path kernels.
//
// Everything here is __host__ __device__ so that tests/ can compile this very
// file with g++ (-DIGD_HOST_EMUL) and check the integer/bit tricks against the
// oracle on the CPU before a GPU run.  The product only ever runs them inside
// the CUDA kernels of igd_fused.cu / igd_codec.cu / igd_packet.cu.
#pragma once
#include <stdint.h>

#ifdef IGD_HOST_EMUL
#define IGD_UNROLL
#include <math.h>
#include <string.h>
#define IGD_HD inline
static inline int igd_f2i(float f) { int i; memcpy(&i, &f, 4); return i; }
static inline float igd_i2f(int i) { float f; memcpy(&f, &i, 4); return f; }
static inline float igd_log2(float x) { return log2f(x); }
static inline int igd_max(int a, int b) { return a > b ? a : b; }
static inline int igd_min(int a, int b) { return a < b ? a : b; }
#else
#define IGD_UNROLL _Pragma("unroll")
#define IGD_HD __device__ __forceinline__
__device__ __forceinline__ int igd_f2i(float f) { return __float_as_int(f); }
__device__ __forceinline__ float igd_i2f(int i) { return __int_as_float(i); }
// arguments are integers converted to float (0 or >= 1): never denormal, so the bare SFU op
// (no denormal pre-scaling) is exact enough; lg2(0) = -inf
__device__ __forceinline__ float igd_log2(float x)
{
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ int igd_max(int a, int b) { return max(a, b); }
__device__ __forceinline__ int igd_min(int a, int b) { return min(a, b); }
#endif

// ---------------------------------------------------------------- G.711 decode
// ITU-T G.711 expansion (SURVEY.md Appendix B); used to fill the shared-memory
// decode table once per CTA.
IGD_HD int igd_alaw2lin(uint32_t code)
{
    uint32_t a = code ^ 0x55u;
    int t = (int)((a & 0x0Fu) << 4);
    int seg = (int)((a >> 4) & 7u);
    t = (seg == 0) ? t + 8 : ((t + 0x108) << (seg - 1));
    return (a & 0x80u) ? t : -t;
}

IGD_HD int igd_ulaw2lin(uint32_t code)
{
    uint32_t u = ~code & 0xFFu;
    int t = (int)(((u & 0x0Fu) << 3) + 0x84u) << ((u >> 4) & 7u);
    return (u & 0x80u) ? (0x84 - t) : (t - 0x84);
}

// ---------------------------------------------------------------- G.711 encode
// Branch-free compressor for both laws.  With s = x>>31 and t = x^s
// (= |x| for x>=0, |x|-1 for x<0) the Sun g711.c pre-bias is
//      A-law : p = x            (x>=0)      p = max(-x-8, 0) = max(t-7, 0)  (x<0)
//      u-law : p = x+0x84       (x>=0)      p = 0x84-x       = t+133        (x<0)
// and, after p = min(p, 0x7FFF) (u-law clip; no-op for A-law), both laws are
// "4 mantissa bits below the leading one, 3-bit segment = position of it":
// P = p + max(p, thr) moves A-law's linear segment 0 (p<256, thr=256) onto a
// leading one at bit 8 and doubles everything else (thr=0 for u-law), so the
// segment is e(P)-8 for every input.  The float (8388608+P) * 2^-7 - 65536 has
// exponent field 120+e(P) == segment (mod 16) and the mantissa's top 4 bits are
// the quantisation bits, so bits[26:19] of that float ARE seg<<4|mant.
struct igd_enc_law {
    int bpos, bneg;       // pre-bias for x>=0 / x<0 (applied to t)
    int thr;              // 256 (A-law) or 0 (u-law)
    uint32_t mpos, mneg;  // output XOR mask for x>=0 / x<0
};

IGD_HD igd_enc_law igd_enc_law_make(int law)
{
    igd_enc_law L;
    if (law == 0) { L.bpos = 0;    L.bneg = -7;  L.thr = 256; L.mpos = 0xD5u; L.mneg = 0x55u; }
    else          { L.bpos = 0x84; L.bneg = 133; L.thr = 0;   L.mpos = 0xFFu; L.mneg = 0x7Fu; }
    return L;
}

// x must already be clamped to int16.  Returns the 8-bit code.
IGD_HD uint32_t igd_g711_enc1(int x, const igd_enc_law &L)
{
    int s = x >> 31;
    int t = x ^ s;
    int p = t + (s ? L.bneg : L.bpos);
    p = igd_min(igd_max(p, 0), 0x7FFF);
    int P = p + igd_max(p, L.thr);
    float g = fmaf(igd_i2f(0x4B000000 | P), 0.0078125f, -65536.0f);
    uint32_t code = ((uint32_t)igd_f2i(g) >> 19) & 0xFFu;
    return code ^ (s ? L.mneg : L.mpos);
}

// ---------------------------------------------------------------- G.711 transcode
// The code that a G.711 code of in_law becomes once decoded and encoded again in out_law (0 = A-law, else u-law):
// enc_out(dec_in(code)).  A-law -> A-law is the identity, u-law -> u-law the identity but for 0x7F (-0) -> 0xFF (+0).
// k_fanout_pkt_tile builds its 2 x 2 x 256 code table from this.
IGD_HD uint32_t igd_g711_transcode1(uint32_t code, int in_law, int out_law)
{
    const int x = in_law ? igd_ulaw2lin(code) : igd_alaw2lin(code);
    return igd_g711_enc1(x, igd_enc_law_make(out_law));
}

// ---------------------------------------------------------------- meters
// rms_dbfs = 10 log10(S/160) - 20 log10(32768); peak_dbfs = 20 log10(P/32768).
// log2 through the SFU (abs error ~2^-22) and the affine map in fp32: total
// error < 2e-5 dB, inside the 1e-4 dB contract (tests/test_meter*.py).
IGD_HD float igd_rms_dbfs(uint64_t sumsq)
{
    // 10*log10(2) * (log2(S) - log2(160)) - 20*log10(32768)
    float l2 = igd_log2((float)sumsq);
    return fmaf(l2, 3.0102999566398120f, -112.35019852575360f);
}

IGD_HD float igd_peak_dbfs(uint32_t peak)
{
    float l2 = igd_log2((float)peak);
    return fmaf(l2, 6.0205999132796240f, -90.308998699194360f);
}

// reference per-packet level: (uint8_t)(sum/len) with C truncating division
// (roip_ed137.cpp:6564-6568); `sum` may be negative under IGD_F_SIGNED_CHAR.
IGD_HD uint32_t igd_bytemean_from_sum(int sum, int len)
{
    return len > 0 ? (uint32_t)(sum / len) & 0xFFu : 0u;
}

// ---------------------------------------------------------------- ED-137 word
// RX field extraction (Functions.cpp:1018-1020, 1087-1090, 1136-1178).
struct igd_edf {
    uint32_t ptt_type, ptt_id, squelch, bss, flags;
};

IGD_HD igd_edf igd_ed137_fields_of(uint32_t w)
{
    igd_edf f;
    f.ptt_type = (w & 0xe0000000u) >> 29;
    f.ptt_id = (w & 0x0fc00000u) >> 22;
    f.squelch = (w & 0x10000000u) >> 28;
    f.bss = (w & 0x000000f8u) >> 3;
    f.flags = (w > 0 ? 1u : 0u) | (((w & 0x00013100u) == 0x00013100u) ? 2u : 0u) |
              (((w & 0x80u) == 0x80u) ? 0u : 4u) | (((w & 0x40u) == 0x40u) ? 0u : 8u);
    return f;
}

// TX: one step of the sender state machine = transport_send_rtp
// (TransportAdapter.cpp:675-855) without the byte copies.  `S` is any struct
// with the igd_ed137_state field names.
struct igd_tx_plan {
    uint32_t word;      // host-order ED-137 word (to be stored big-endian)
    uint32_t size;      // 0 = suppressed, 20, or 20+payload_len
    uint8_t pt123;      // force PT to 123
    uint8_t marker;     // M bit
    uint8_t copy_payload;  // payload bytes are refreshed (:680-684)
};

template <class S>
IGD_HD igd_tx_plan igd_ed137_tx_step(S &a, uint32_t payload_len, long long now)
{
    igd_tx_plan r;
    r.word = 0; r.size = 0; r.pt123 = 0; r.marker = 0; r.copy_payload = 0;
    if (!a.radiostatus) return r;                                      // :641
    const bool idle = a.calltype_flags & 1u, rxonly = a.calltype_flags & 2u,
               txish = a.calltype_flags & 4u;
    if (idle && a.callIn) { a.sqlstatus = 0; a.pttstatus = 0; }         // :675-679
    const bool ptt = a.pttstatus != 0, sql = a.sqlstatus != 0, in = a.callIn != 0;
    if ((ptt && !in) || (sql && in)) {                                  // :680-684
        r.copy_payload = 1;
    } else {                                                            // :685-706
        unsigned long long since = (unsigned long long)now - (unsigned long long)a.r2sSendtime;
        unsigned long long ka = (unsigned long long)(long long)a.keepAlivePeroid;
        if (since < ka && !a.firstR2SPacket) return r;                  // suppressed
        if (since >= ka) a.r2sSendtime = now;
    }
    r.marker = (a.firstR2SPacket && a.packetCnt == 0) ? 1 : 0;          // :715-723
    uint32_t w;
    const bool stable = (a.txSlaveEnable == a.txSlaveEnableChanged) &&
                        (a.rxSlaveEnable == a.rxSlaveEnableChanged) &&
                        (a.trxSlaveEnableChangedCount >= 5);            // :728
    if (!stable) {                                                      // :744-747
        a.txSlaveEnable = a.txSlaveEnableChanged;
        a.rxSlaveEnable = a.rxSlaveEnableChanged;
        a.trxSlaveEnableChangedCount =
            (uint8_t)(a.trxSlaveEnableChangedCount + 1 >= 5 ? 5 : a.trxSlaveEnableChangedCount + 1);
    }
    {
        const uint32_t rx = a.rxSlaveEnable, tx = a.txSlaveEnable;
        if (rx == 0 && tx == 0)      w = stable ? 0x00000000u : 0x00013100u;
        else if (rx == 1 && tx == 1) w = 0x000131c0u;
        else if (rx == 1 && tx == 0) w = 0x00013140u;
        else if (rx == 0 && tx == 1) w = 0x00013180u;
        else                         w = 0x00000000u;
    }
    if (sql) {                                                          // :763-778
        a.sqlpriority = 0;
        w |= 0x10000000u;
        w |= 0x000000f8u & ((uint32_t)a.ed137_bssi << 3);
    } else if (!ptt) {                                                  // :779-784
        w |= 0x0fc00000u & (1u << 22);
    }
    if (ptt) {                                                          // :786-796
        w |= 0x0fc00000u & ((uint32_t)a.pttid << 22);
        w |= 0xe0000000u & ((uint32_t)a.pttpriority << 29);
    }
    r.word = w;
    if (rxonly && !in) r.pt123 = 1;                                     // :801-804
    if (!ptt && !sql)               { r.pt123 = 1; r.size = 20; }       // :811-815
    else if (rxonly && !sql)        { r.pt123 = 1; r.size = 20; }       // :821-825
    else if (txish && !ptt && !sql) { r.pt123 = 1; r.size = 20; }       // :826-829
    else if (txish && ptt && in) {                                      // :830-841
        if (a.callRecorder || sql) r.size = 20 + payload_len;
        else { r.pt123 = 1; r.size = 20; }
    } else r.size = 20 + payload_len;                                   // :842-845
    if (a.firstR2SPacket && a.packetCnt < 30) a.packetCnt++;            // :849-855
    else if (a.packetCnt >= 30) a.firstR2SPacket = 0;
    return r;
}

// Plan of one outgoing packet, produced by the per-channel sender walk and
// consumed by the packet assembly kernel.
struct igd_tx_plan_rec {
    uint32_t word;        // host-order ED-137 word
    uint16_t size;        // 0 = suppressed
    uint8_t flags;        // bit0 pt123, bit1 marker, bit2 copy_payload
    uint8_t reserved;
    int32_t src_frame;    // frame whose payload the packet carries (-1: none yet)
};

// Timer-driven keep-alive: sendR2SStatus (TransportAdapter.cpp:422-633), the twin of the step above.
// It differs where the reference differs: no payload, the slave-enable "changed" values are NOT latched
// (:513-516 vs :744-745), an extra Idle&&callIn branch (:585-589), and a packet only leaves when the PT
// ends up 123 (:617-630).  The header it stamps lives in the adapter's send buffer, so whatever the
// last call left in bytes 0..11 (incl. the PT in byte 1) is reused: `stale_pt` is that PT.
// plan.size: 0 = nothing sent, 20 = keep-alive; plan.copy_payload is reused as "header fields were
// written into the send buffer" (they persist even when nothing is sent).
template <class S>
IGD_HD igd_tx_plan igd_ed137_r2s_step(S &a, long long now, uint32_t stale_pt)
{
    igd_tx_plan r;
    r.word = 0; r.size = 0; r.pt123 = 0; r.marker = 0; r.copy_payload = 0;
    if (!a.radiostatus) return r;                                      // :429
    const bool idle = a.calltype_flags & 1u, rxonly = a.calltype_flags & 2u,
               txish = a.calltype_flags & 4u;
    if (idle && a.callIn) { a.sqlstatus = 0; a.pttstatus = 0; }         // :444-448
    const bool ptt = a.pttstatus != 0, sql = a.sqlstatus != 0, in = a.callIn != 0;
    if ((ptt && !in) || (sql && in)) return r;                          // :449-454 audio is flowing
    {
        unsigned long long since = (unsigned long long)now - (unsigned long long)a.r2sSendtime;
        unsigned long long ka = (unsigned long long)(long long)a.keepAlivePeroid;
        if (since < ka && !a.firstR2SPacket) return r;                  // :457-460
        if (since >= ka) a.r2sSendtime = now;                           // :463-473
    }
    r.copy_payload = 1;                                                 // header fields get written from here on
    r.marker = (a.firstR2SPacket && a.packetCnt == 0) ? 1 : 0;          // :485-493
    uint32_t w;
    const bool stable = (a.txSlaveEnable == a.txSlaveEnableChanged) &&
                        (a.rxSlaveEnable == a.rxSlaveEnableChanged) &&
                        (a.trxSlaveEnableChangedCount >= 5);            // :499
    if (!stable)                                                        // :513-516: count only, no latch
        a.trxSlaveEnableChangedCount =
            (uint8_t)(a.trxSlaveEnableChangedCount + 1 >= 5 ? 5 : a.trxSlaveEnableChangedCount + 1);
    {
        const uint32_t rx = a.rxSlaveEnable, tx = a.txSlaveEnable;
        if (rx == 0 && tx == 0)      w = stable ? 0x00000000u : 0x00013100u;
        else if (rx == 1 && tx == 1) w = 0x000131c0u;
        else if (rx == 1 && tx == 0) w = 0x00013140u;
        else if (rx == 0 && tx == 1) w = 0x00013180u;
        else                         w = 0x00000000u;
    }
    if (sql) {                                                          // :531-546
        a.sqlpriority = 0;
        w |= 0x10000000u;
        w |= 0x000000f8u & ((uint32_t)a.ed137_bssi << 3);
    } else if (!ptt) {                                                  // :547-552
        w |= 0x0fc00000u & (1u << 22);
    }
    if (ptt) {                                                          // :554-564
        w |= 0x0fc00000u & ((uint32_t)a.pttid << 22);
        w |= 0xe0000000u & ((uint32_t)a.pttpriority << 29);
    }
    r.word = w;
    bool pt123 = false, leaves;
    if (rxonly && !in) pt123 = true;                                    // :570-573
    if (!ptt && !sql)               pt123 = true;                       // :580-584
    else if (idle && in)            pt123 = true;                       // :585-589
    else if (rxonly && !sql)        pt123 = true;                       // :590-594
    else if (txish && !ptt && !sql) pt123 = true;                       // :595-598
    else if (txish && ptt && in) {                                      // :599-610
        if (!(a.callRecorder || sql)) pt123 = true;
    }
    r.pt123 = pt123 ? 1 : 0;
    leaves = pt123 || stale_pt == 123;                                  // :617
    if (!leaves) return r;
    r.size = 20;
    if (a.firstR2SPacket && a.packetCnt < 30) a.packetCnt++;            // :622-629
    else if (a.packetCnt >= 30) a.firstR2SPacket = 0;
    return r;
}

// ---------------------------------------------------------------- RX liveness
// One tick of the receive side of one radio call: the state the reference keeps in
// struct tp_adapter across transport_rtp_cb calls (TransportAdapter.cpp:240-316) plus the
// R2S keep-alive watchdog of RoIP_ED137::detectR2SPacketAndReconn (roip_ed137.cpp:1767-1780).
// `S` has the igd_rx_state field names, `FL` the igd_ed137_fields ones.  Returns IGD_RXE_* bits.
template <class S, class FL>
IGD_HD uint32_t igd_rx_step(S &a, const FL &f, bool present, bool run_watchdog, long long now, int r2s_period)
{
    uint32_t ev = 0;
    if (present) {
        ev |= 0x01u;                                                  // IGD_RXE_PACKET
        if (f.accepted) {
            a.ed137_value = f.word;                                   // :252-256 (kept in host order)
            a.payloadsize = f.length_raw;
        }
        if (f.flags & 0x10u) {                                        // :286-291 oversized / truncated packet
            a.r2sPacket = now;
            ev |= 0x08u;                                              // IGD_RXE_DROPPED
        } else if (f.pt != 123) {                                     // :298-307
            a.r2sPacket = now;
            ev |= 0x02u;                                              // IGD_RXE_AUDIO
            if ((f.pt == 0 || f.pt == 8) && f.payload_len == 160) ev |= 0x40u;   // IGD_RXE_FRAME: a whole G.711 frame
            if (!a.rtpAudio) ev |= 0x04u;                             // IGD_RXE_EDGE -> setIncomingED137Value
            a.rtpAudio = 1;
        } else {                                                      // :308-315
            a.r2sPacket = now;
            if (a.rtpAudio) ev |= 0x04u;
            a.rtpAudio = 0;
        }
    }
    if (run_watchdog) {                                               // roip_ed137.cpp:1767-1780
        const long long secDiff = now - a.r2sPacket;
        if (secDiff > (long long)r2s_period * 3) {
            ev |= 0x10u;                                              // IGD_RXE_LATE
            if (a.r2sCount == 5) ev |= 0x20u;                         // IGD_RXE_HANGUP (WG-67 cause 2001)
            if (a.r2sCount < 255) a.r2sCount++;
        } else {
            a.r2sCount = 0;
        }
    }
    return ev;
}

// A leg-frame the fused path must not decode: its packet (igd_ed137_fields words 1..3) is not a whole G.711
// audio frame -- pt other than 0 / 8, payload_len != 160, dropped, or absent (size 0 parses as payload_len 0).
// The same rule as IGD_RXE_FRAME above.
IGD_HD bool igd_fields_no_audio(uint32_t w1, uint32_t w2, uint32_t w3)
{
    const uint32_t plen = w1 >> 16, pt = w2 & 0xFFu, flags = w3 >> 24;
    return !(pt == 0u || pt == 8u) || plen != 160u || (flags & 0x10u) != 0u;
}

// ---------------------------------------------------------------- gate arbitration
// a leg count known at compile time (loops unroll, leg state stays in registers)
template <int N> struct igd_const_int {
#ifdef IGD_HOST_EMUL
    constexpr operator int() const { return N; }
#else
    __host__ __device__ constexpr operator int() const { return N; }
#endif
};
// One checkEvents() pass over the G legs of one bridge.  `L` has the igd_arb_leg field names,
// `BR` the igd_arb_bridge ones; `word(g)` returns leg g's latched ED-137 word (host order),
// `active(g)` whether the leg takes part (callState, and trxmode != RX for CLIENT / != TX for SERVER).
// CLIENT mode: highest ptt_type wins, winner gets SLOT_VOLUME 2.0 (256), pressed losers 0
// (roip_ed137.cpp:6124-6231); a released PTT is held for five more ticks (:6140-6153).
template <class BR, class L, class GI, class W, class A>
IGD_HD void igd_arb_client_tick(BR &b, L *legs, GI G, W word, A active)
{
    IGD_UNROLL
    for (int i = 0; i < G; i++) {
        if (!active(i)) continue;
        int ptt = (int)((word(i) & 0xe0000000u) >> 29);
        if (ptt != legs[i].last) {
            if (ptt == 0) {
                legs[i].msec++;
                if (legs[i].msec < 6) ptt = 1;
            }
        } else {
            legs[i].msec = 0;
        }
        legs[i].last = (uint8_t)ptt;
        if (ptt && ptt > b.ptt_level) {
            b.ptt_level = ptt;
            legs[i].gain_q7 = 256;
            IGD_UNROLL
            for (int j = 0; j < G; j++)
                if (legs[j].on && j != i) legs[j].gain_q7 = 0;
        }
        if (ptt > 0 && !legs[i].on) {
            legs[i].on = 1;
        } else if (ptt == 0 && legs[i].on) {
            legs[i].on = 0;
            legs[i].gain_q7 = 0;
            b.ptt_level = ptt;
        }
    }
}

// SERVER mode with rxBestSignalEnable: per-radio squelch bookkeeping (roip_ed137.cpp:5627-5719 and
// its three twins), then after five consecutive ticks of squelch only the radio with the best BSS
// quality index is unmuted (:5985-6121).
template <class BR, class L, class GI, class W, class A>
IGD_HD void igd_arb_server_best_tick(BR &b, L *legs, GI G, W word, A active)
{
    IGD_UNROLL
    for (int i = 0; i < G; i++) {
        if (!active(i)) continue;
        const uint32_t w = word(i);
        int sqlon = (int)((w & 0x10000000u) >> 28);
        legs[i].rssi = (int8_t)((w & 0xf8u) >> 3);
        if (sqlon != legs[i].last) {
            if (sqlon == 0) {
                legs[i].msec++;
                if (legs[i].msec < 1) sqlon = 1;
            }
        } else {
            legs[i].msec = 0;
        }
        if (legs[i].last != sqlon) {
            legs[i].last = (uint8_t)sqlon;
            if (!sqlon) legs[i].gain_q7 = 0;
        }
    }
    bool any = false;
    IGD_UNROLL
    for (int i = 0; i < G; i++) {
        if (!active(i) || legs[i].last == 0) {
            if (legs[i].on) { b.sqlStatusCount = 0; b.sqlStatusOn = 0; }
            legs[i].on = 0;
            legs[i].rssi = -1;
        }
        any = any || legs[i].last > 0;
    }
    if (any) {
        b.sqlStatusCount++;
        if (b.sqlStatusCount >= 5 && !b.sqlStatusOn) {
            IGD_UNROLL
    for (int i = 0; i < G; i++)
                if (legs[i].last > 0) legs[i].gain_q7 = 0;
            b.sqlStatusOn = 1;
            // the first radio nobody beats (:6060-6121); found first, applied after, so that every leg index below is
            // a compile-time constant once the loops unroll (a `break` out of the search made the compiler keep the
            // leg array in local memory behind a run-time index)
            int best_i = -1;
            IGD_UNROLL
            for (int i = 0; i < G; i++) {
                bool best = legs[i].last != 0;
                IGD_UNROLL
                for (int j = 0; j < G; j++)
                    if (best && j != i && legs[i].rssi < legs[j].rssi) best = false;
                if (best && best_i < 0) best_i = i;
            }
            if (best_i >= 0) {
                IGD_UNROLL
                for (int j = 0; j < G; j++) {
                    legs[j].on = (uint8_t)(j == best_i);
                    if (j == best_i && active(j)) legs[j].gain_q7 = 256;
                }
            }
        }
    } else {
        b.sqlStatusCount = 0;
        b.sqlStatusOn = 0;
        IGD_UNROLL
    for (int i = 0; i < G; i++) legs[i].on = 0;
    }
}
