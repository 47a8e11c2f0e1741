/*
 * igate_dsp.h -- C ABI of libigate_dsp.so: the B200 (sm_100a) implementation of
 * the per-frame voice path of the iGate4x ED-137 RoIP softphone/gateway.
 *
 * Plain C types only (no CUDA / torch types): pointers are either host
 * pointers (IGD_MEM_HOST; the library stages them through the GPU itself) or
 * CUDA device pointers (IGD_MEM_DEVICE; e.g. from igd_dev_alloc()).  Every
 * arithmetic entry point runs on the GPU; there is no CPU fallback -- when no
 * usable device exists igd_init() fails with IGD_ENODEV and nothing else can
 * be called.
 *
 * Reference = piyanon108/iGate4xSoftphoneDSP; "replaces" cites the reference
 * interface (file:line) each entry point takes over.  The Qt/PJSIP-side
 * binding a maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions (reference: pj_status_t, PJ_SUCCESS==0, setters never fail --
 * TransportAdapter.cpp:135-223): every function returns 0 on success or a
 * negative errno-style code; nothing aborts; the caller owns every buffer it
 * passes; one igd_ctx = one CUDA stream, calls on one ctx are serialised by
 * the caller, different ctxs are independent (re-entrant, unlike the
 * reference's file-static scratch pointers, TransportAdapter.cpp:76-79).
 */
#ifndef IGATE_DSP_H
#define IGATE_DSP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define IGD_ABI_VERSION 2
#define IGD_FRAME 160            /* 20 ms @ 8 kHz: roip_ed137.h:112-115           */
#define IGD_PKT_HDR 20           /* sizeof(custom_rtp_hdr): ed137_rtp.h:22-47     */
#define IGD_PKT_MAX 180          /* 20 + 160: TransportAdapter.cpp:814,844        */
#define IGD_MAX_LEGS 32          /* legs per bridge (reference: 4 radios + calls) */

enum { IGD_LAW_ALAW = 0,         /* PCMA, RTP PT 8 (roip_ed137.cpp:3563)          */
       IGD_LAW_ULAW = 1 };       /* PCMU, RTP PT 0 (roip_ed137.cpp:3564)          */
enum { IGD_MEM_HOST = 0, IGD_MEM_DEVICE = 1 };

enum {
    IGD_OK = 0,
    IGD_EINVAL = -22,            /* bad argument / misaligned device pointer      */
    IGD_ENOMEM = -12,
    IGD_ENODEV = -19,            /* no CUDA device / not sm_100                    */
    IGD_ECUDA = -5               /* CUDA runtime error; see igd_last_error()      */
};

/* flags (igd_batch_desc.flags and the `flags` arguments below) */
#define IGD_F_SIGNED_CHAR 0x1u   /* quirk Q4: x86 `char` signedness in the byte-mean
                                    (roip_ed137.cpp:6566); default = unsigned, the
                                    aarch64 production target                     */
#define IGD_F_REF_QUIRKS 0x2u    /* quirks Q2/Q3 of SURVEY.md Appendix A in the
                                    packet path (stale payload; outgoing byte-mean
                                    over header+payload)                          */
#define IGD_F_KERNEL_W 0x8u       /* diagnostics (A/B runs, tests): the previous generation of the fused kernel -- k_fused_w
                                     instead of k_fused_q (G <= 4, codes and packet forms), k_fused_g instead of
                                     k_fused_h (G = 8).  Same results, bit for bit. */
#define IGD_F_WALK_SERIAL 0x10u    /* diagnostics (A/B runs, tests; igd_gateway_process, igd_ed137_pack): walk the per-call
                                     state machines with separate thread-per-channel / -bridge / -sender kernels
                                     (k_rx_track, k_gate_arbitrate, k_ed137_plan) instead of k_rxarb_walk / k_plan_walk
                                     (one warp per bridge / sender, tick axis across its lanes) or k_rxarb_bridge.
                                     Same results, bit for bit. */
#define IGD_F_GENERIC_KERNEL 0x4u /* diagnostic (igd_process_batch): run the block-cooperative kernel that
                                    serves batches beyond 32-bit indices instead of the warp-autonomous
                                    ones; same results, slower                                       */

typedef struct igd_ctx igd_ctx;

/* ------------------------------------------------------------------ runtime */
int igd_abi_version(void);
/* Creates a context on CUDA device `device` with its own stream.              */
int igd_init(int device, igd_ctx **ctx);
int igd_shutdown(igd_ctx *ctx);
/* Run on an existing CUDA stream: cudaStream_t cast to void*; NULL is CUDA's
 * legacy default stream (what torch.cuda.current_stream() is by default).     */
int igd_set_stream(igd_ctx *ctx, void *cuda_stream);
/* Back to the context's own (non-blocking) stream.                            */
int igd_use_own_stream(igd_ctx *ctx);
int igd_sync(igd_ctx *ctx);
const char *igd_last_error(igd_ctx *ctx);
typedef struct {
    int device, sm_count, cc_major, cc_minor;
    size_t total_mem;
    char name[64];
} igd_devinfo;
int igd_device_info(igd_ctx *ctx, igd_devinfo *out);
/* number of kernels this ctx has launched so far (bench.py "gpu_launches")    */
uint64_t igd_launch_count(igd_ctx *ctx);
/* memory helpers so a host without the CUDA toolkit can own device buffers     */
void *igd_host_alloc(size_t bytes);              /* pinned host memory          */
void igd_host_free(void *p);
void *igd_dev_alloc(igd_ctx *ctx, size_t bytes);
void igd_dev_free(igd_ctx *ctx, void *p);
int igd_copy_to_device(igd_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
int igd_copy_to_host(igd_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);

/* --------------------------------------------------------------------- G.711
 * replaces: PJSIP's PCMA/PCMU codec selected at roip_ed137.cpp:3546-3574
 * (pjmedia alaw_ulaw.c, un-vendored; SURVEY.md Appendix B is the contract).    */
int igd_g711_decode(igd_ctx *ctx, const uint8_t *codes, int16_t *pcm, size_t n, int law, int mem);
int igd_g711_encode(igd_ctx *ctx, const int16_t *pcm, uint8_t *codes, size_t n, int law, int mem);
/* per-channel law: codes/pcm are [nframes][nch][160], law is [nch]             */
int igd_g711_decode_ch(igd_ctx *ctx, const uint8_t *codes, const uint8_t *law, int16_t *pcm,
                       size_t nframes, size_t nch, int mem);
int igd_g711_encode_ch(igd_ctx *ctx, const int16_t *pcm, const uint8_t *law, uint8_t *codes,
                       size_t nframes, size_t nch, int mem);

/* -------------------------------------------------------------------- meters
 * One 16-byte record per (frame, channel).
 *   bytemean : reference per-packet level, RoIP_ED137::setIncomingRTP
 *              (roip_ed137.cpp:6541-6587): (uint8_t)(sum(payload bytes)/len)
 *   sumsq/peak/rms_dbfs/peak_dbfs : per-frame RMS / peak dBFS (north_star; the
 *              reference's audiometer.cpp only rescales a pre-computed level)  */
typedef struct {
    uint32_t sumsq_lo;           /* low 32 bits of sum(x^2) over the frame        */
    uint32_t hi;                 /* [7:0] sumsq bits 39:32, [15:8] bytemean,
                                    [31:16] peak = max|x| (0..32768)              */
    float rms_dbfs;              /* 10log10(S/160) - 20log10(32768); -inf if S==0 */
    float peak_dbfs;             /* 20log10(peak/32768);            -inf if 0     */
} igd_meter_rec;
#define IGD_METER_SUMSQ(r) ((uint64_t)(r).sumsq_lo | ((uint64_t)((r).hi & 0xFFu) << 32))
#define IGD_METER_BYTEMEAN(r) (((r).hi >> 8) & 0xFFu)
#define IGD_METER_PEAK(r) ((r).hi >> 16)

typedef struct {
    uint8_t bytemean_out;        /* RoIP_ED137::setOutgoingRTP level of the encoded
                                    mix (roip_ed137.cpp:6500-6536)                */
    uint8_t n_open;              /* legs with a non-zero gain in this frame       */
    uint16_t mix_peak;           /* max|mix| (0..32768)                           */
} igd_bridge_rec;

/* PCM frames in -> records out (bytemean field = 0).  pcm is [nframes][160].    */
int igd_frame_meter(igd_ctx *ctx, const int16_t *pcm, size_t nframes, igd_meter_rec *out, int mem);
/* replaces: setIncomingRTP/setOutgoingRTP byte-mean (roip_ed137.cpp:6500-6587).
 * payload i = base + i*stride, `len` bytes each.                               */
int igd_bytemean(igd_ctx *ctx, const uint8_t *payloads, size_t npayloads, size_t len,
                 size_t stride, unsigned flags, uint8_t *out, int mem);
/* replaces: AudioMeter::getAudioLevel scale (audiometer.cpp:30-31):
 * out[i] = int(float(v[i]*100.0/30000.0))                                      */
int igd_level_percent(igd_ctx *ctx, const int32_t *v, size_t n, int32_t *out, int mem);

/* ----------------------------------------------------------------- gain, mix
 * replaces: pjsua_conf_adjust_rx_level() per call (roip_ed137.cpp:5221, policy
 * Functions.cpp:1664-1705) + the PJSIP conference bridge into slot 0
 * (roip_ed137.cpp:4907-4920).  SURVEY.md Appendix D:
 *   adj = (int)((level-1)*128)+128;  y = clamp16((x*adj)>>7);
 *   mix = clamp16(sum over legs with adj != 0 of y)                            */
int igd_gain_q7(float level);                    /* host helper: level -> adj    */
/* pcm [nframes][nbridges*legs][160], gain_q7 [nframes][nbridges*legs],
 * mix [nframes][nbridges][160]                                                  */
int igd_mix(igd_ctx *ctx, const int16_t *pcm, const uint16_t *gain_q7, size_t nframes,
            size_t nbridges, int legs, int16_t *mix, int mem);

/* ------------------------------------------------------- fused voice path
 * decode -> meter -> gate/gain -> saturating mix -> encode, one pass over HBM.
 * Layout (frame-major = arrival order of one 20 ms tick):
 *   codes   [F][B*G][160] u8     G.711 payloads of every leg
 *   law     [B*G] u8             IGD_LAW_* per leg
 *   gain_q7 [F][B*G] u16         adj per leg and frame; 0 = gate shut.  Bit 15
 *                                (IGD_GAIN_NO_AUDIO) = no audio frame arrived for this
 *                                leg on this tick (keep-alive, lost / truncated packet):
 *                                the reference never hands such a packet to the stream
 *                                (TransportAdapter.cpp:298-315), so its bridge hears the
 *                                stream's silence.  The leg adds nothing to the mix
 *                                whatever the low bits say, is not counted in n_open, its
 *                                meter record is digital silence (sum 0, peak 0, byte-mean
 *                                0, -inf dB) and igd_event_summary skips the frame.  The
 *                                code bytes of such a leg-frame are not interpreted.
 *   out_law [B] u8               law the bridge output is encoded with
 *   mix     [F][B][160] i16      bridge output PCM
 *   enc     [F][B][160] u8       bridge output, G.711
 *   meter   [F][B*G] igd_meter_rec
 *   bmeter  [F][B]   igd_bridge_rec
 * Any of the four outputs may be NULL (not all): it is then neither stored nor, for
 * host buffers, copied back -- a gateway that only forwards packets and levels leaves
 * mix NULL and moves 43 % of the result bytes.
 * Device pointers must be 16-byte aligned (32 for mix).  Host buffers (ideally from
 * igd_host_alloc) are staged in frame chunks: the H2D copy of chunk k+1, the kernel of
 * chunk k and the D2H copy of chunk k-1 overlap; the call returns when all is done.  */
#define IGD_GAIN_NO_AUDIO 0x8000u
typedef struct {
    uint32_t struct_size;        /* = sizeof(igd_batch_desc)                      */
    int32_t mem;                 /* IGD_MEM_HOST or IGD_MEM_DEVICE (all pointers) */
    int32_t F, B, G;
    uint32_t flags;              /* IGD_F_*                                       */
    const uint8_t *codes;
    const uint8_t *law;
    const uint16_t *gain_q7;
    const uint8_t *out_law;
    int16_t *mix;
    uint8_t *enc;
    igd_meter_rec *meter;
    igd_bridge_rec *bmeter;
} igd_batch_desc;
int igd_process_batch(igd_ctx *ctx, const igd_batch_desc *d);

/* ------------------------------------------------------------ event summary
 * replaces: keeplogAudioLevel / createPTTEventDataLogger
 * (Functions.cpp:2126-2145, 2148-2230): per channel, over the frames whose
 * gate is open: count, sum/max/min of the level and of the byte-mean, then
 * 10*log10 of av/max/min.  "level" = frame mean square S/160, carried as the
 * exact integer S.                                                              */
typedef struct {
    uint32_t count;              /* level_in_count                                */
    uint16_t bm_sum;             /* OutgoingRTPSum (uint16_t, wraps: roip_ed137.h:742) */
    uint8_t bm_max;              /* init 0                                        */
    uint8_t bm_min;              /* init 255                                      */
    uint64_t sum_s;
    uint64_t max_s;              /* init 0                                        */
    uint64_t min_s;              /* init 255*160 (reference inits min level to 255) */
} igd_summary_rec;
typedef struct {
    float level_av_db;           /* 10*log10(sum/count)   Functions.cpp:2196      */
    float level_max_db;          /* 10*log10(max)         Functions.cpp:2197      */
    float level_min_db;          /* 10*log10(min)         Functions.cpp:2198      */
    uint32_t bm_av;              /* OutgoingRTPSum/count  Functions.cpp:2200      */
} igd_summary_db;
/* meter [F][C], gain_q7 [F][C] -> out [C], db [C] (db may be NULL)              */
int igd_event_summary(igd_ctx *ctx, const igd_meter_rec *meter, const uint16_t *gain_q7,
                      size_t F, size_t C, igd_summary_rec *out, igd_summary_db *db, int mem);

/* ----------------------------------------------- ED-137 RTP header extension
 * replaces: transport_rtp_cb (TransportAdapter.cpp:240-316), get_ed137_value
 * (:337-346), the RoIP_ED137::get_IPRadio* parsers (Functions.cpp:1001-1179),
 * transport_send_rtp (:635-874) and sendR2SStatus (:422-633).                   */
typedef struct {
    uint32_t word;               /* ntohl(hdr->ed137), only latched when accepted */
    uint16_t length_raw;         /* hdr->length as stored, un-swapped (:255)      */
    uint16_t payload_len;        /* size-20 (radio) ; 0 when dropped              */
    uint8_t pt;                  /* payload type                                  */
    uint8_t accepted;            /* PT in {8,0,18,123}              (:252)        */
    uint8_t keepalive;           /* PT == 123                       (:298)        */
    uint8_t ptt_type;            /* (w&0xE0000000)>>29  Functions.cpp:1136-1138   */
    uint8_t ptt_id;              /* (w&0x0FC00000)>>22  Functions.cpp:1148-1150   */
    uint8_t squelch;             /* (w&0x10000000)>>28  Functions.cpp:1160-1162   */
    uint8_t bss;                 /* (w&0xF8)>>3         Functions.cpp:1018-1020   */
    uint8_t flags;               /* bit0 active (w>0, :1172-1178), bit1 RRC present
                                    ((w&0x13100)==0x13100, :1087), bit2 mainTxUsed
                                    (:1089), bit3 mainRxUsed (:1090), bit4 dropped
                                    (payload_len>=1024 or size<20, :286-291)      */
} igd_ed137_fields;
#define IGD_EDF_ACTIVE 0x01u
#define IGD_EDF_RRC 0x02u
#define IGD_EDF_MAIN_TX 0x04u
#define IGD_EDF_MAIN_RX 0x08u
#define IGD_EDF_DROPPED 0x10u

/* pkts: npkts packets, packet i at pkts + i*stride, sizes[i] bytes long
 * (sizes==NULL: every packet is `stride` bytes).  payload_out (optional):
 * [npkts][160] payload bytes (zero-filled past payload_len).                    */
int igd_ed137_parse(igd_ctx *ctx, const uint8_t *pkts, const uint32_t *sizes, size_t npkts,
                    size_t stride, igd_ed137_fields *fields, uint8_t *payload_out, int mem);

/* call-type classification = the QString tests of TransportAdapter.cpp:675,801,
 * 821,826,830 evaluated once instead of per packet                              */
#define IGD_CT_IDLE 0x1u         /* contains "Idle"                               */
#define IGD_CT_RXONLY 0x2u       /* contains "Rxonly" or == "Rx"                  */
#define IGD_CT_TXISH 0x4u        /* contains "Tx" or "TRx"                        */
unsigned igd_calltype_flags(const char *calltype);

/* Per-channel sender state = the fields of struct tp_adapter
 * (TransportAdapter.h:40-93) that transport_send_rtp reads and writes.          */
typedef struct {
    uint8_t radiostatus, pttstatus, sqlstatus, callIn;
    uint8_t callRecorder, pttpriority, pttid, ed137_bssi;
    uint8_t rxSlaveEnable, txSlaveEnable, rxSlaveEnableChanged, txSlaveEnableChanged;
    uint8_t trxSlaveEnableChangedCount, firstR2SPacket, calltype_flags, sqlpriority;
    int32_t packetCnt;
    int32_t keepAlivePeroid;     /* ms, default 200 (TransportAdapter.h:78)       */
    int64_t r2sSendtime;         /* ms                                            */
    int32_t rtpFalse;            /* stuck-audio counter (:657-673)                */
    int32_t reserved;
} igd_ed137_state;               /* 40 bytes                                      */
/* = pjmedia_custom_tp_adapter_create field init (TransportAdapter.cpp:97-128)   */
void igd_ed137_state_init(igd_ed137_state *s, int radiocall, int callIn, const char *calltype,
                          int keepAlivePeroid, int64_t now_ms);

/* Per-(frame,channel) control inputs = what the setters (setAdapterPtt,
 * setAdapterQslOn, setcallRecorder, setAdapterPttId; TransportAdapter.cpp:
 * 135-213) would have written before that frame's packet is sent.               */
typedef struct {
    uint8_t pttstatus, sqlstatus, pttpriority, ed137_bssi;
    uint8_t pttid, callRecorder, reserved[2];
} igd_ed137_ctl;                 /* 8 bytes                                       */

/* Batched transport_send_rtp: for every channel c and frame f (in frame order,
 * the per-channel state is carried from frame to frame and written back):
 *   in : rtp12   [F][C][12]   the PJSIP-built RTP header of the packet
 *        payload [F][C][160]  its G.711 payload (payload_len bytes each)
 *        ctl     [F][C]       (NULL = keep the state's own flags)
 *        now_ms0, tick_ms     currenttime of frame f = now_ms0 + f*tick_ms
 *   out: pkts    [F][C][out_stride]  packet bytes (out_stride >= 180); the bytes of a slot past
 *                             sizes[f][c] are written as zero
 *        sizes   [F][C]       0 = suppressed by the keep-alive throttle,
 *                             20 = header only, 20+payload_len = with payload
 *        bytemean_out [F][C]  setOutgoingRTP level (roip_ed137.cpp:6500-6536) of
 *                             packets sent with PT != 123, 0 otherwise
 *   state [C] is updated in place.                                              */
typedef struct {
    uint32_t struct_size;
    int32_t mem;
    int32_t F, C;
    uint32_t flags;              /* IGD_F_REF_QUIRKS, IGD_F_SIGNED_CHAR            */
    uint32_t payload_len;        /* <= 160                                        */
    uint32_t out_stride;         /* >= 20 + payload_len, multiple of 4            */
    int32_t tick_ms;             /* 20                                            */
    int64_t now_ms0;
    const uint8_t *rtp12;
    const uint8_t *payload;
    const igd_ed137_ctl *ctl;
    igd_ed137_state *state;
    uint8_t *pkts;
    uint32_t *sizes;
    uint8_t *bytemean_out;
    uint8_t *stale_payload;      /* optional [C][160], in/out: the payload bytes last copied
                                    into each adapter's send buffer (send_pkt_buff+20,
                                    TransportAdapter.cpp:683).  Only used with
                                    IGD_F_REF_QUIRKS: carries quirk Q2 across calls.
                                    NULL = zero-filled at the start of every call.  */
} igd_ed137_pack_desc;
int igd_ed137_pack(igd_ctx *ctx, const igd_ed137_pack_desc *d);

/* Batched sendR2SStatus (TransportAdapter.cpp:422-633), the timer-driven keep-alive: one call at
 * time now_ms for every channel.  hdr20 [C][20] is the header region of each adapter's send buffer
 * (send_pkt_buff): read (the reference re-stamps whatever the last packet left there, PT included)
 * and updated in place; sizes [C] = 20 where a keep-alive leaves (copy hdr20[c] to the wire), else 0. */
int igd_ed137_keepalive(igd_ctx *ctx, uint8_t *hdr20, igd_ed137_state *state, size_t C, int64_t now_ms,
                        uint32_t *sizes, int mem);

/* ------------------------------------------- fused voice path, packets in
 * The same computation as igd_process_batch with the codes read straight out
 * of the raw ED-137 packets: pkts [F][B*G][IGD_PKT_MAX] as received
 * (transport_rtp_cb, TransportAdapter.cpp:240-316: payload = bytes 20..size),
 * fields [F][B*G] from igd_ed137_parse.  A leg-frame whose packet is not a whole
 * G.711 audio frame -- pt other than 0 / 8 (the R2S keep-alive is pt 123), fewer
 * than 160 payload bytes, dropped, or absent (size 0) -- is silent exactly as if
 * its gain carried IGD_GAIN_NO_AUDIO (the same rule as IGD_RXE_FRAME): the reference
 * never gives such a packet's bytes to the decoder.  Otherwise the results are
 * identical to igd_ed137_parse(payload_out) followed by igd_process_batch on that
 * payload with those gains; the payload array is never materialised.
 * G = 4 (the reference's four radios per softphone, roip_ed137.cpp:130-139) runs ONE
 * kernel that reads the codes out of the packets; any other leg count (e.g. the 32
 * inbound call slots of a CLIENT-mode softphone, :141-150) extracts the payloads into
 * the context's scratch first and runs the codes-form kernels -- same results, one
 * more pass over the packets.  Device pointers: pkts 16-byte aligned, the rest as for
 * igd_process_batch.                                                             */
typedef struct {
    uint32_t struct_size;        /* = sizeof(igd_packets_desc)                    */
    int32_t mem;
    int32_t F, B, G;
    uint32_t flags;              /* IGD_F_SIGNED_CHAR                             */
    const uint8_t *pkts;
    const igd_ed137_fields *fields;
    const uint8_t *law;
    const uint16_t *gain_q7;
    const uint8_t *out_law;
    int16_t *mix;
    uint8_t *enc;
    igd_meter_rec *meter;
    igd_bridge_rec *bmeter;
} igd_packets_desc;
int igd_process_packets(igd_ctx *ctx, const igd_packets_desc *d);

/* -------------------------------------------------- RX liveness / call events
 * replaces: the receive-side state transport_rtp_cb keeps per call
 * (TransportAdapter.cpp:240-316: ed137_value / payloadsize latch :252-256,
 * r2sPacket stamp :289,302,311, rtpAudio edge -> setIncomingED137Value ->
 * checkEvents() :304-306,312-314), getR2SStatus (:317-325) and the R2S
 * keep-alive watchdog RoIP_ED137::detectR2SPacketAndReconn
 * (roip_ed137.cpp:1756-1780: no packet for more than 3*r2sPeriod on five
 * consecutive 40 ms timer ticks -> hang up with "WG-67 ;cause=2001").
 * Together with igd_ed137_parse this is the batched RX front-end.             */
typedef struct {
    int64_t r2sPacket;           /* ms of the last packet (getR2SStatus)          */
    uint32_t ed137_value;        /* latched word in HOST order (get_ed137_value)  */
    uint16_t payloadsize;        /* hdr->length as stored                          */
    uint8_t rtpAudio;            /* last packet carried audio (pt != 123)          */
    uint8_t r2sCount;            /* watchdog strikes                               */
} igd_rx_state;                  /* 16 bytes; zero-init + r2sPacket = call start   */
typedef struct {
    uint32_t word;               /* get_ed137_value() after this tick              */
    uint8_t flags;               /* IGD_RXE_*                                      */
    uint8_t r2sCount;
    uint16_t reserved;
} igd_rx_event;                  /* 8 bytes                                        */
#define IGD_RXE_PACKET 0x01u     /* a packet arrived on this tick                  */
#define IGD_RXE_AUDIO 0x02u      /* forwarded to the stream (pt != 123)            */
#define IGD_RXE_EDGE 0x04u       /* audio <-> keep-alive edge: setIncomingED137Value(word) */
#define IGD_RXE_DROPPED 0x08u    /* oversized / truncated packet (:286-291)        */
#define IGD_RXE_LATE 0x10u       /* watchdog: now - r2sPacket > 3*r2s_period       */
#define IGD_RXE_HANGUP 0x20u     /* watchdog: sixth late tick in a row, hang up    */
#define IGD_RXE_FRAME 0x40u      /* a whole G.711 audio frame arrived: forwarded (pt 0 / 8) with at
                                    least 160 payload bytes (fields.payload_len == 160) -- what the
                                    fused path may decode; without it the leg is silent on this
                                    tick (IGD_GAIN_NO_AUDIO)                                       */
typedef struct {
    uint32_t struct_size;
    int32_t mem;
    int32_t F, C;
    int32_t tick_ms;             /* 20: packet time of frame f = now_ms0 + f*tick_ms */
    int32_t r2s_period_ms;       /* radio->r2sPeriod, default 200 (roip_ed137.h:685) */
    int32_t wd_ticks;            /* the watchdog runs on every wd_ticks-th frame
                                    (40 ms timer / 20 ms frames = 2); 0 = never    */
    int32_t frame0;              /* index of this call's first frame (watchdog phase),
                                    >= 0 (negative: IGD_EINVAL)                    */
    int64_t now_ms0;
    const igd_ed137_fields *fields;   /* [F][C] from igd_ed137_parse               */
    const uint8_t *present;      /* [F][C] 0 = no packet on that tick; NULL = all  */
    igd_rx_state *state;         /* [C], updated in place                          */
    igd_rx_event *events;        /* [F][C] out                                     */
    const uint32_t *sizes;       /* [F][C] optional, used when present == NULL: a packet arrived
                                    iff sizes[f][c] != 0 (the sizes igd_ed137_parse was given)   */
} igd_rx_track_desc;
int igd_rx_track(igd_ctx *ctx, const igd_rx_track_desc *d);

/* ---------------------------------------------------------- gate arbitration
 * replaces: the gate decisions of RoIP_ED137::checkEvents() that end in
 * setSlotVolume (roip_ed137.cpp:5190-5234) -- the only inputs are the legs'
 * latched ED-137 words, the output is the gain_q7 array igd_process_batch
 * consumes:
 *   IGD_ARB_CLIENT_PTT  highest ptt_type wins: winner SLOT_VOLUME 2.0, pressed
 *                       losers 0.0, five-tick release hold (roip_ed137.cpp:6124-6231)
 *   IGD_ARB_SERVER_BEST per-radio squelch gate (:5627-5719) + best-signal
 *                       selection: after five ticks of squelch only the radio with
 *                       the best BSS quality index is unmuted (:5985-6121)
 * MUTE/UNMUTE are taken as gain 0 / 256 (Functions.cpp:1664-1705 with its
 * sidetone / group-mute side conditions left to the host).                     */
enum { IGD_ARB_CLIENT_PTT = 0, IGD_ARB_SERVER_BEST = 1 };
/* words are igd_rx_event records read in place (word_stride 8): every gain written for a tick whose
 * event lacks IGD_RXE_FRAME carries IGD_GAIN_NO_AUDIO, i.e. the leg is silent on ticks on which no
 * whole audio frame arrived (the PTT hold-off keeps a gate open for five ticks while the radio already
 * sends 20-byte keep-alives, roip_ed137.cpp:6140-6147; the reference's bridge hears stream silence
 * then).  The arbitration state itself is unaffected.                                              */
#define IGD_ARB_F_SILENCE 0x1u
typedef struct {
    uint8_t last;                /* lastTx (CLIENT) / lastRx (SERVER)             */
    uint8_t msec;                /* lastTxmsec / lastRxmsec                       */
    uint8_t on;                  /* m_PttPressed (CLIENT) / audioSQLOn (SERVER)   */
    int8_t rssi;                 /* radio->rssi, -1 while not receiving           */
    uint16_t gain_q7;            /* the slot volume the leg currently has         */
    uint16_t reserved;
} igd_arb_leg;                   /* 8 bytes                                       */
typedef struct {
    int32_t ptt_level;           /* CLIENT                                        */
    int32_t sqlStatusCount;      /* SERVER                                        */
    uint8_t sqlStatusOn;         /* SERVER                                        */
    uint8_t reserved[7];
} igd_arb_bridge;                /* 16 bytes                                      */
typedef struct {
    uint32_t struct_size;
    int32_t mem;
    int32_t F, B, G;             /* G <= IGD_MAX_LEGS                             */
    int32_t mode;                /* IGD_ARB_*                                     */
    uint32_t word_stride;        /* bytes between consecutive words: 4 for a plain
                                    u32 array, 8 to read igd_rx_event.word in place */
    uint32_t flags;              /* IGD_ARB_F_*                                   */
    const void *words;           /* [F][B*G] latched ED-137 words, host order     */
    const uint8_t *active;       /* [B*G] leg takes part (callState...); NULL = all */
    igd_arb_leg *legs;           /* [B*G], updated in place                       */
    igd_arb_bridge *bridges;     /* [B], updated in place                         */
    uint16_t *gain_q7;           /* [F][B*G] out                                  */
} igd_arb_desc;
int igd_gate_arbitrate(igd_ctx *ctx, const igd_arb_desc *d);

/* ------------------------------------------------- gateway: packets in, packets out
 * One call = the whole per-tick voice path of a RoIP gateway for F ticks of B bridges x 4 legs,
 * everything on the device: the receive callback's header work on every leg's packet
 * (transport_rtp_cb, TransportAdapter.cpp:240-316) and the liveness / edge walk (igd_rx_track, reading the
 * header words straight out of the packets), checkEvents()'s gate decisions with silent no-audio ticks
 * (igd_gate_arbitrate + IGD_ARB_F_SILENCE), the sender walk of the call each bridge's output leaves
 * on (transport_send_rtp, :635-874) and the fused decode -> meter -> mix -> encode kernel, which
 * reads the codes straight out of the received packets and writes FINISHED 180-byte ED-137 packets
 * (header from the sender walk + the PJSIP RTP header, payload = this tick's encoded mix; the bytes of
 * a slot past tx_sizes are zero) -- the bytes igd_ed137_pack produces without IGD_F_REF_QUIRKS.
 * Three kernels: the receive-side walk (liveness + arbitration in one launch, header words straight out of the
 * packets: one bridge per warp with the tick axis across its lanes for calls of >= 8 ticks below 65 536 channels,
 * one bridge per thread otherwise), the sender walk (on a side stream) and the fused kernel.  IGD_F_WALK_SERIAL:
 * header view + liveness walk, arbitration and sender walk as separate thread-per-channel kernels.  No payload, code or plan array exists between
 * them, nothing but packets and state crosses the API.  (tx_state.rtpFalse, the
 * reference's never-read stuck-audio diagnostic counter, is not maintained here: the payload it
 * looks at is produced after the sender walk.)
 * Algorithmic bytes per bridge-frame (SURVEY 8d "with RTP"): 4*180 in + 180 + 320 (optional mix) + 4*16
 * = 1284.  rx_events / gain_q7 / meter / bmeter / mix / enc are optional outputs (NULL = not wanted;
 * rx_events and gain_q7 then live in the context's scratch).  G must be 4.                            */
typedef struct {
    uint32_t struct_size;        /* = sizeof(igd_gateway_desc)                    */
    int32_t mem;                 /* IGD_MEM_DEVICE or IGD_MEM_HOST (all pointers) */
    int32_t F, B, G;
    uint32_t flags;              /* IGD_F_SIGNED_CHAR, IGD_F_KERNEL_W, IGD_F_WALK_SERIAL; any other
                                    bit (IGD_F_REF_QUIRKS included) is IGD_EINVAL  */
    int32_t arb_mode;            /* IGD_ARB_*                                     */
    int32_t tick_ms;             /* 20                                            */
    int32_t r2s_period_ms;       /* 200                                           */
    int32_t wd_ticks;            /* watchdog every wd_ticks ticks, 0 = never      */
    int32_t frame0;              /* index of this call's first tick (watchdog phase), >= 0 */
    int32_t reserved;
    int64_t now_ms0;
    /* receive side */
    const uint8_t *rx_pkts;      /* [F][B*G][180] as received (zero padded)       */
    const uint32_t *rx_sizes;    /* [F][B*G] received sizes, 0 = nothing arrived; NULL = all 180 */
    const uint8_t *law;          /* [B*G]                                         */
    const uint8_t *active;       /* [B*G] or NULL                                 */
    igd_rx_state *rx_state;      /* [B*G] in/out                                  */
    igd_arb_leg *arb_legs;       /* [B*G] in/out                                  */
    igd_arb_bridge *arb_bridges; /* [B] in/out                                    */
    /* send side: the call each bridge's output goes out on */
    const uint8_t *out_law;      /* [B]                                           */
    const uint8_t *tx_rtp12;     /* [F][B][12] PJSIP-built RTP headers            */
    const igd_ed137_ctl *tx_ctl; /* [F][B] setter values per tick, or NULL        */
    igd_ed137_state *tx_state;   /* [B] in/out                                    */
    /* outputs */
    uint8_t *tx_pkts;            /* [F][B][180]                                   */
    uint32_t *tx_sizes;          /* [F][B] 0 = suppressed, 20 = keep-alive, 180   */
    igd_rx_event *rx_events;     /* [F][B*G] optional                             */
    uint16_t *gain_q7;           /* [F][B*G] optional                             */
    igd_meter_rec *meter;        /* [F][B*G] optional                             */
    igd_bridge_rec *bmeter;      /* [F][B] optional (bytemean_out = the level of the outgoing payload) */
    int16_t *mix;                /* [F][B][160] optional                          */
    uint8_t *enc;                /* [F][B][160] optional                          */
} igd_gateway_desc;
int igd_gateway_process(igd_ctx *ctx, const igd_gateway_desc *d);

/* ------------------------------------------------- gateway fan-out: one frame per bridge in, a packet per leg out
 * The other direction of a bridge.  In the reference every call port is connected to conference slot 0
 * (roip_ed137.cpp:4907-4920), so on each 20 ms tick every call of the bridge sends the same slot-0 frame (the
 * sound-device capture), G.711-encoded in that call's own codec and sent through transport_send_rtp
 * (TransportAdapter.cpp:635-874) with that call's own ED-137 sender state (PTT, squelch, keep-alive throttle, marker,
 * RRC word).  One call does this for F ticks of B bridges x G legs, leg c = b*G + g:
 *   in : pcm      [F][B][160]    the frame every leg of bridge b sends on tick f
 *        law      [B*G]          IGD_LAW_* of each leg's call
 *        tx_rtp12 [F][B*G][12]   PJSIP-built RTP headers; tx_ctl [F][B*G] setter values or NULL
 *   out: tx_pkts  [F][B*G][180]  the bytes of a slot past tx_sizes are zero
 *        tx_sizes [F][B*G]       0 = suppressed by the keep-alive throttle, 20 = keep-alive, 180 = audio
 *        tx_level [F][B*G]       optional: setOutgoingRTP level (roip_ed137.cpp:6500-6536), 0 for PT 123 / nothing sent
 *   tx_state [B*G] is updated in place.
 * The results are byte for byte those of igd_g711_encode_ch over pcm with each bridge's frame copied to its G legs,
 * followed by igd_ed137_pack (payload_len 160, out_stride 180, stale_payload NULL, flags & IGD_F_SIGNED_CHAR) --
 * except tx_state.rtpFalse, the reference's never-read stuck-audio counter, which is not maintained here (as in
 * igd_gateway_process: the payload it looks at is encoded after the sender walk).  Quirks Q2 / Q3 are not offered:
 * flags other than IGD_F_SIGNED_CHAR are IGD_EINVAL.  Two kernels: the sender walk and one that stages the PCM,
 * encodes each bridge-frame once per law among its legs and assembles the packets; no code array exists between
 * them.  Device pointers: pcm and tx_pkts 16-byte aligned, tx_state and tx_ctl 8, tx_rtp12 and tx_sizes 4.  The
 * device form only enqueues work on the context's stream and, once an earlier call of the same or a larger shape has
 * sized the scratch, allocates nothing: it can be captured into a CUDA graph.
 * Algorithmic bytes per bridge-frame: 320 + G*12 + G*180 (G = 4: 1088).                                      */
typedef struct {
    uint32_t struct_size;        /* = sizeof(igd_fanout_desc)                     */
    int32_t mem;                 /* IGD_MEM_DEVICE or IGD_MEM_HOST (all pointers) */
    int32_t F, B, G;             /* 1 <= G <= IGD_MAX_LEGS; leg c = b*G + g        */
    uint32_t flags;              /* IGD_F_SIGNED_CHAR only                        */
    int32_t tick_ms;             /* 20                                            */
    int32_t reserved;
    int64_t now_ms0;             /* currenttime of tick f = now_ms0 + f*tick_ms    */
    const int16_t *pcm;          /* [F][B][160] the frame every leg of bridge b sends (conference slot 0) */
    const uint8_t *law;          /* [B*G] IGD_LAW_* of each leg's call            */
    const uint8_t *tx_rtp12;     /* [F][B*G][12] PJSIP-built RTP headers          */
    const igd_ed137_ctl *tx_ctl; /* [F][B*G] setter values per tick, or NULL      */
    igd_ed137_state *tx_state;   /* [B*G] in/out                                  */
    uint8_t *tx_pkts;            /* [F][B*G][180]; bytes past tx_sizes are zero   */
    uint32_t *tx_sizes;          /* [F][B*G] 0 = suppressed, 20 = keep-alive, 180 */
    uint8_t *tx_level;           /* [F][B*G] optional: setOutgoingRTP level, 0 for PT 123 / nothing sent */
} igd_fanout_desc;
int igd_gateway_fanout(igd_ctx *ctx, const igd_fanout_desc *d);

/* ------------------------------------------------- gateway fan-out from packets: the console call's packets in, a packet per leg out
 * igd_gateway_fanout with slot 0 taken from where a gateway without a sound card has it: the remote console, whose
 * audio arrives as ED-137 packets on the same call that igd_gateway_process sends the bridge's mix out on (a call has
 * one codec in both directions, so in_law is igd_gateway_process's out_law).  One call does F ticks of B bridges x G
 * legs, leg c = b*G + g:
 *   in : rx_pkts  [F][B][180]    the console call's packets as received, zero padded
 *        rx_sizes [F][B]         received sizes, 0 = nothing arrived; NULL = all 180
 *        in_law   [B]            IGD_LAW_* of the console call
 *        law, tx_rtp12, tx_ctl   as in igd_fanout_desc
 *   out: tx_pkts, tx_sizes, tx_level, tx_state as in igd_fanout_desc
 * The frame every leg of bridge b sends on tick f is igd_g711_decode of bytes 20..179 of rx_pkts[f][b] in in_law[b]
 * when that packet carries a whole G.711 audio frame -- accepted PT 0 or 8, payload_len 160, not dropped (the
 * IGD_RXE_FRAME rule; the decode law is in_law, not the packet's PT, as in igd_process_packets) -- and digital silence
 * (PCM 0) otherwise: a keep-alive, a lost, short or PT 18 packet, an unaccepted PT.  The results are byte for byte
 * those of igd_ed137_parse (payload_out) -> igd_g711_decode_ch in in_law -> PCM 0 on the ticks without a whole frame
 * -> igd_gateway_fanout with that PCM: packets, sizes, levels and tx_state, except tx_state.rtpFalse, which is not
 * maintained (as in igd_gateway_fanout).  No PCM exists in between: each payload byte is mapped through a 256-entry
 * code table of the (in law, leg law) pair.  1 <= G <= 32; flags other than IGD_F_SIGNED_CHAR are IGD_EINVAL;
 * B*G <= 2^31.  Two kernels: the sender walk and one that stages the console packets, maps each bridge-frame once per
 * law among its legs and assembles the packets.  Device pointers: rx_pkts and tx_pkts 16-byte aligned, tx_state and
 * tx_ctl 8, tx_rtp12, tx_sizes and rx_sizes 4.  The device form only enqueues work on the context's stream and, once
 * an earlier call of the same or a larger shape has sized the scratch, allocates nothing: it can be captured into a
 * CUDA graph together with igd_gateway_process.
 * Algorithmic bytes per bridge-frame: 180 + G*12 + G*180 (G = 4: 948, against 1088 for igd_gateway_fanout).     */
typedef struct {
    uint32_t struct_size;        /* = sizeof(igd_fanout_pkt_desc)                 */
    int32_t mem;                 /* IGD_MEM_DEVICE or IGD_MEM_HOST (all pointers) */
    int32_t F, B, G;             /* 1 <= G <= IGD_MAX_LEGS; leg c = b*G + g        */
    uint32_t flags;              /* IGD_F_SIGNED_CHAR only                        */
    int32_t tick_ms;             /* 20                                            */
    int32_t reserved;
    int64_t now_ms0;             /* currenttime of tick f = now_ms0 + f*tick_ms    */
    const uint8_t *rx_pkts;      /* [F][B][180] the console call's packets as received (zero padded) */
    const uint32_t *rx_sizes;    /* [F][B] received sizes, 0 = nothing arrived; NULL = all 180 */
    const uint8_t *in_law;       /* [B] IGD_LAW_* of the console call             */
    const uint8_t *law;          /* [B*G] IGD_LAW_* of each leg's call            */
    const uint8_t *tx_rtp12;     /* [F][B*G][12] PJSIP-built RTP headers          */
    const igd_ed137_ctl *tx_ctl; /* [F][B*G] setter values per tick, or NULL      */
    igd_ed137_state *tx_state;   /* [B*G] in/out                                  */
    uint8_t *tx_pkts;            /* [F][B*G][180]; bytes past tx_sizes are zero   */
    uint32_t *tx_sizes;          /* [F][B*G] 0 = suppressed, 20 = keep-alive, 180 */
    uint8_t *tx_level;           /* [F][B*G] optional: setOutgoingRTP level, 0 for PT 123 / nothing sent */
} igd_fanout_pkt_desc;
int igd_gateway_fanout_packets(igd_ctx *ctx, const igd_fanout_pkt_desc *d);

/* ------------------------------------------------------------ recorder sink
 * replaces: WavWriter::start/wav_write/stop (WavWriter.cpp:63-156).
 * Builds the complete file image on the GPU: 44-byte header + body.
 * ref_quirks!=0 reproduces the reference byte for byte (format tag 7 with
 * 2 channels x 16 bit, every payload byte b written as {b,0x00}); otherwise a
 * valid 8-bit mono WAVE_FORMAT_ALAW(6)/MULAW(7) file (Codecs.h:33-34).
 * Returns the file size through *out_len; `out` needs igd_wav_size() bytes.     */
size_t igd_wav_size(size_t payload_bytes, int ref_quirks);
int igd_wav_image(igd_ctx *ctx, const uint8_t *payload, size_t payload_bytes, int rate, int law,
                  int ref_quirks, uint8_t *out, size_t *out_len, int mem);

/* The same sink for many calls at once, straight from the batch layout: image k is the WAV file of channel
 * chans[k] (NULL: channel k) over all F frames of codes [F][C][160]; law [C] picks the format tag of the
 * valid (non-quirk) header (NULL: u-law).  Image k starts at out + k*image_stride; image_stride must be a
 * multiple of 4 and >= igd_wav_size(F*160, ref_quirks).  (Per-recording avg/max level as stored by
 * Database::updateAudioRec, database.cpp:471-490, is igd_event_summary's output for that channel.)       */
int igd_wav_images(igd_ctx *ctx, const uint8_t *codes, size_t F, size_t C, const uint32_t *chans, size_t nchan,
                   const uint8_t *law, int rate, int ref_quirks, uint8_t *out, size_t image_stride, int mem);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* IGATE_DSP_H */
