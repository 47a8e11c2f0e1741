// igd_packet.cu -- ED-137 RTP parse / pack / keep-alive, RX liveness walk, gate arbitration, recorder sink
// (hand-written sm_100a kernels of the iGate4x voice path; design notes in igd_fused.cu and DESIGN.md)
#include "igd_device.cuh"
#include "igd_walks.cuh"      // igd_rxarb_args

namespace {

// ============================================================ ED-137 parse
// transport_rtp_cb (TransportAdapter.cpp:240-316) + field getters
// (Functions.cpp:1001-1179).  One warp per packet: lanes 0..4 fetch the five
// header words, every lane copies payload words.
__device__ __forceinline__ uint32_t bswap32(uint32_t v) { return __byte_perm(v, 0, 0x0123); }

// Tile form of the receive parse for the wire stride (180 B): a CTA stages 64 packets
// (11 520 contiguous bytes) in shared memory with 16-byte loads, 64 threads extract the fields,
// all threads write the 64 x 160 payload bytes with 16-byte stores.  Same results as
// k_ed137_parse below (which keeps serving other strides / unaligned buffers).
constexpr int kPktTile = 64, kPktWords = IGD_PKT_MAX / 4;      // 45 words per packet
__global__ void __launch_bounds__(256) k_ed137_parse_tile(const uint8_t *__restrict__ pkts,
                                                          const uint32_t *__restrict__ sizes, size_t npkts,
                                                          igd_ed137_fields *__restrict__ fields,
                                                          uint8_t *__restrict__ payload_out)
{
    __shared__ __align__(128) uint32_t img[kPktTile * kPktWords];
    __shared__ uint32_t plen_s[kPktTile];
    const size_t first = (size_t)blockIdx.x * kPktTile;
    const uint32_t np = (uint32_t)min((size_t)kPktTile, npkts - first);
    const uint4 *src = reinterpret_cast<const uint4 *>(pkts + first * IGD_PKT_MAX);
    const uint32_t tile_bytes = np * IGD_PKT_MAX;
    if ((tile_bytes & 15u) == 0) {
        // full tiles (and any tail whose size is a multiple of 16): ONE bulk async copy (TMA) stages the
        // tile, completion on the CTA's mbarrier -- no registers, no LSU issue slots
        __shared__ uint64_t bar;
        const uint32_t bar_s = shared_addr(&bar);
        if (threadIdx.x == 0) {
            mbar_init(bar_s, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            mbar_expect_tx(bar_s, tile_bytes);
            bulk_g2s(shared_addr(img), src, tile_bytes, bar_s);
        }
        __syncthreads();                 // the barrier is initialised before anyone polls it
        mbar_wait(bar_s, 0);
    } else {
        const uint32_t nvec = (tile_bytes + 15) / 16;
        for (uint32_t j = threadIdx.x; j < nvec; j += blockDim.x) {
            uint4 v;
            if ((j + 1) * 16 <= tile_bytes) v = __ldcs(src + j);
            else {                                               // ragged tail of the whole buffer: word loads
                const uint32_t *w = reinterpret_cast<const uint32_t *>(src + j);
                const uint32_t left = (tile_bytes - j * 16) / 4;
                v.x = left > 0 ? w[0] : 0u; v.y = left > 1 ? w[1] : 0u; v.z = left > 2 ? w[2] : 0u; v.w = 0u;
            }
            reinterpret_cast<uint4 *>(img)[j] = v;
        }
        __syncthreads();
    }
    if (threadIdx.x < np) {
        const uint32_t p = threadIdx.x;
        const size_t i = first + p;
        const uint32_t size = sizes ? sizes[i] : (uint32_t)IGD_PKT_MAX;
        const uint32_t navail = min(size, (uint32_t)IGD_PKT_MAX) / 4;
        const uint32_t *hw = img + p * kPktWords;
        const uint32_t w0 = navail > 0 ? hw[0] : 0u, w3 = navail > 3 ? hw[3] : 0u, w4 = navail > 4 ? hw[4] : 0u;
        const uint32_t pt = (w0 >> 8) & 0x7Fu;
        const bool too_short = size < IGD_PKT_HDR;
        const uint32_t plen_raw = size - IGD_PKT_HDR;
        const bool dropped = too_short || plen_raw >= 1024u;
        const bool accepted = !too_short && (pt == 8 || pt == 0 || pt == 18 || pt == 123);
        const uint32_t plen = dropped ? 0u : min(plen_raw, (uint32_t)IGD_FRAME);
        plen_s[p] = plen;
        igd_ed137_fields f;
        const uint32_t word = accepted ? bswap32(w4) : 0u;
        const igd_edf e = igd_ed137_fields_of(word);
        f.word = word;
        f.length_raw = accepted ? (uint16_t)(w3 >> 16) : (uint16_t)0;
        f.payload_len = (uint16_t)plen;
        f.pt = (uint8_t)pt;
        f.accepted = accepted;
        f.keepalive = (!too_short && pt == 123);
        f.ptt_type = (uint8_t)e.ptt_type;
        f.ptt_id = (uint8_t)e.ptt_id;
        f.squelch = (uint8_t)e.squelch;
        f.bss = (uint8_t)e.bss;
        f.flags = (uint8_t)(e.flags | (dropped ? IGD_EDF_DROPPED : 0u));
        *reinterpret_cast<uint4 *>(fields + i) = *reinterpret_cast<const uint4 *>(&f);
    }
    if (!payload_out) return;
    __syncthreads();
    uint4 *dst = reinterpret_cast<uint4 *>(payload_out + first * IGD_FRAME);
    for (uint32_t j = threadIdx.x; j < np * kChunks; j += blockDim.x) {
        const uint32_t p = j / kChunks, ch = j - p * kChunks;
        const uint32_t plen = plen_s[p], b0 = ch * 16;
        const uint32_t *w = img + p * kPktWords + 5 + ch * 4;
        uint32_t v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t b = b0 + 4 * k;
            v[k] = b < plen ? w[k] : 0u;
            if (b < plen && plen - b < 4) v[k] &= (1u << (8 * (plen - b))) - 1u;
        }
        __stcs(dst + j, make_uint4(v[0], v[1], v[2], v[3]));
    }
}

// transport_rtp_cb's view of a packet header (TransportAdapter.cpp:248-292) from its words 0, 3, 4 and its size
__device__ __forceinline__ igd_ed137_fields fields_of_header(uint32_t w0, uint32_t w3, uint32_t w4, uint32_t size)
{
    const uint32_t pt = (w0 >> 8) & 0x7Fu;
    const bool too_short = size < IGD_PKT_HDR;
    const uint32_t plen_raw = size - IGD_PKT_HDR;
    const bool dropped = too_short || plen_raw >= 1024u;
    const bool accepted = !too_short && (pt == 8 || pt == 0 || pt == 18 || pt == 123);
    igd_ed137_fields f;
    const uint32_t word = accepted ? bswap32(w4) : 0u;
    const igd_edf e = igd_ed137_fields_of(word);
    f.word = word;
    f.length_raw = accepted ? (uint16_t)(w3 >> 16) : (uint16_t)0;
    f.payload_len = (uint16_t)(dropped ? 0u : min(plen_raw, (uint32_t)IGD_FRAME));
    f.pt = (uint8_t)pt;
    f.accepted = accepted;
    f.keepalive = (!too_short && pt == 123);
    f.ptt_type = (uint8_t)e.ptt_type;
    f.ptt_id = (uint8_t)e.ptt_id;
    f.squelch = (uint8_t)e.squelch;
    f.bss = (uint8_t)e.bss;
    f.flags = (uint8_t)(e.flags | (dropped ? IGD_EDF_DROPPED : 0u));
    return f;
}

// Fields only (no payload wanted, e.g. the RX front-end feeding k_rx_track): one thread per packet
// reads the three header words it needs -- 1-2 DRAM sectors per packet instead of the whole packet.
__global__ void __launch_bounds__(256) k_ed137_fields(const uint8_t *__restrict__ pkts,
                                                      const uint32_t *__restrict__ sizes, size_t npkts,
                                                      size_t stride, igd_ed137_fields *__restrict__ fields)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npkts) return;
    const uint32_t *pw = reinterpret_cast<const uint32_t *>(pkts + i * stride);
    const uint32_t size = sizes ? sizes[i] : (uint32_t)stride;
    const uint32_t navail = min(size, (uint32_t)stride) / 4;
    const uint32_t w0 = navail > 0 ? __ldg(pw) : 0u, w3 = navail > 3 ? __ldg(pw + 3) : 0u, w4 = navail > 4 ? __ldg(pw + 4) : 0u;
    const igd_ed137_fields f = fields_of_header(w0, w3, w4, size);
    *reinterpret_cast<uint4 *>(fields + i) = *reinterpret_cast<const uint4 *>(&f);
}

__global__ void __launch_bounds__(256) k_ed137_parse(const uint8_t *__restrict__ pkts,
                                                     const uint32_t *__restrict__ sizes, size_t npkts,
                                                     size_t stride, igd_ed137_fields *__restrict__ fields,
                                                     uint8_t *__restrict__ payload_out)
{
    const uint32_t lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t i = warp; i < npkts; i += nwarps) {
        const uint32_t *pw = reinterpret_cast<const uint32_t *>(pkts + i * stride);
        const uint32_t size = sizes ? sizes[i] : (uint32_t)stride;
        const uint32_t navail = min(size, (uint32_t)stride) / 4;
        const uint32_t hw = (lane < 5 && lane < navail) ? __ldcs(pw + lane) : 0u;
        const uint32_t w0 = __shfl_sync(0xffffffffu, hw, 0);
        const uint32_t w3 = __shfl_sync(0xffffffffu, hw, 3);
        const uint32_t w4 = __shfl_sync(0xffffffffu, hw, 4);
        const uint32_t pt = (w0 >> 8) & 0x7Fu;                           // byte 1, low 7 bits
        const bool too_short = size < IGD_PKT_HDR;
        const uint32_t plen_raw = size - IGD_PKT_HDR;                     // unsigned wrap (:279)
        const bool dropped = too_short || plen_raw >= 1024u;              // :286-291
        const bool accepted = !too_short && (pt == 8 || pt == 0 || pt == 18 || pt == 123);   // :252
        const uint32_t plen = dropped ? 0u : min(plen_raw, (uint32_t)IGD_FRAME);
        if (lane == 0) {
            igd_ed137_fields f;
            const uint32_t word = accepted ? bswap32(w4) : 0u;            // ntohl (:342)
            const igd_edf e = igd_ed137_fields_of(word);
            f.word = word;
            f.length_raw = accepted ? (uint16_t)(w3 >> 16) : (uint16_t)0; // bytes 14..15 as stored
            f.payload_len = (uint16_t)plen;
            f.pt = (uint8_t)pt;
            f.accepted = accepted;
            f.keepalive = (!too_short && pt == 123);
            f.ptt_type = (uint8_t)e.ptt_type;
            f.ptt_id = (uint8_t)e.ptt_id;
            f.squelch = (uint8_t)e.squelch;
            f.bss = (uint8_t)e.bss;
            f.flags = (uint8_t)(e.flags | (dropped ? IGD_EDF_DROPPED : 0u));
            *reinterpret_cast<uint4 *>(fields + i) = *reinterpret_cast<const uint4 *>(&f);
        }
        if (payload_out) {
            uint32_t *dst = reinterpret_cast<uint32_t *>(payload_out + i * IGD_FRAME);
            for (uint32_t k = lane; k < IGD_FRAME / 4; k += 32) {
                uint32_t v = 0;
                if (k * 4 < plen) {
                    v = __ldcs(pw + 5 + k);
                    const uint32_t rem = plen - k * 4;
                    if (rem < 4) v &= (1u << (8 * rem)) - 1u;
                }
                dst[k] = v;
            }
        }
    }
}

// ============================================================ ED-137 pack
// ============================================================ RX liveness walk
// One thread per channel walks its frames through the receive-side state of
// transport_rtp_cb (TransportAdapter.cpp:240-316) and the R2S watchdog
// (roip_ed137.cpp:1767-1780).  Consecutive threads read consecutive 16-byte field
// records and write consecutive 8-byte events: coalesced, latency-bound.
// kPres: 0 = a packet on every tick, 1 = d.present[], 2 = d.sizes[] != 0 (resolved at launch: a per-element
// choice between the three inside the prefetch loop cost 2.6x on the walk)
//        3 = gateway form: d.fields is NULL, the header words are read straight out of the received packets
//            (pkts [F][C][180], sizes optional) -- no field array between the header pass and the walk
template <int kPres>
__global__ void __launch_bounds__(128) k_rx_track(const igd_rx_track_desc d, const uint8_t *__restrict__ pkts = nullptr)
{
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d.C) return;
    igd_rx_state s = d.state[c];
    // The walk is sequential, its inputs are not: the fields of the NEXT run of 8 frames are in flight
    // while this run is walked (with a few thousand channels there is one warp per SM and nothing
    // else to hide the latency behind).
#ifndef IGD_RX_AHEAD
#define IGD_RX_AHEAD 8
#endif
    constexpr int kAhead = IGD_RX_AHEAD;
    uint4 raw[kAhead], nraw[kAhead];
    uint8_t pres[kAhead], npres[kAhead];
    auto fetch = [&](int f0, uint4 (&r)[kAhead], uint8_t (&p)[kAhead]) {
#pragma unroll
        for (int u = 0; u < kAhead; u++) {
            const int f = f0 + u;
            if (f < d.F) {
                const size_t i = (size_t)f * d.C + c;
                if (kPres == 3) {
                    const uint32_t size = d.sizes ? __ldg(d.sizes + i) : (uint32_t)IGD_PKT_MAX;
                    const uint32_t navail = min(size, (uint32_t)IGD_PKT_MAX) / 4;
                    const uint32_t *pw = reinterpret_cast<const uint32_t *>(pkts + i * IGD_PKT_MAX);
                    // raw header words now, the field record when the tick is walked (keeps the loads in flight)
                    r[u] = make_uint4(navail > 0 ? __ldg(pw) : 0u, navail > 3 ? __ldg(pw + 3) : 0u, navail > 4 ? __ldg(pw + 4) : 0u, size);
                    p[u] = (uint8_t)(size != 0u);
                } else {
                    r[u] = __ldg(reinterpret_cast<const uint4 *>(d.fields + i));
                    p[u] = kPres == 1 ? d.present[i] : kPres == 2 ? (uint8_t)(__ldg(d.sizes + i) != 0u) : (uint8_t)1;
                }
            }
        }
    };
    fetch(0, nraw, npres);
    const int wd_ticks = d.wd_ticks;
    int wd_phase = wd_ticks > 0 ? (int)(d.frame0 % wd_ticks) : 0;
    long long now = d.now_ms0;
    for (int f0 = 0; f0 < d.F; f0 += kAhead) {
#pragma unroll
        for (int u = 0; u < kAhead; u++) { raw[u] = nraw[u]; pres[u] = npres[u]; }
        fetch(f0 + kAhead, nraw, npres);
#pragma unroll
        for (int u = 0; u < kAhead; u++) {
            const int f = f0 + u;
            if (f >= d.F) break;
            const size_t i = (size_t)f * d.C + c;
            const igd_ed137_fields fl = kPres == 3 ? fields_of_header(raw[u].x, raw[u].y, raw[u].z, raw[u].w)
                                                   : *reinterpret_cast<const igd_ed137_fields *>(&raw[u]);
            // watchdog phase and clock as running values: a modulo and a 64-bit multiply per tick are a fifth of the
            // walk's dependent instruction chain (4096 channels x 1640 ticks: 0.40 -> 0.28 ms)
            const bool wd = wd_ticks > 0 && wd_phase == wd_ticks - 1;
            wd_phase = wd_phase + 1 == wd_ticks ? 0 : wd_phase + 1;
            const uint32_t ev = igd_rx_step(s, fl, pres[u] != 0, wd, now, d.r2s_period_ms);
            now += d.tick_ms;
            igd_rx_event e;
            e.word = s.ed137_value;
            e.flags = (uint8_t)ev;
            e.r2sCount = s.r2sCount;
            e.reserved = 0;
            *reinterpret_cast<uint2 *>(d.events + i) = *reinterpret_cast<const uint2 *>(&e);
        }
    }
    d.state[c] = s;
}

// ============================================================ gate arbitration
// One thread per bridge walks its frames through checkEvents()'s gate decisions
// (igd_math.cuh: igd_arb_client_tick / igd_arb_server_best_tick); the leg state of
// the block's bridges lives in registers (G in {1,2,4}) or shared memory for the walk.
// A block owns `bpb` <= 64 bridges (the launcher shrinks bpb until the grid covers the
// SMs several times: the walk over F is sequential per bridge, so few bridges x many
// frames must not sit on a handful of SMs); all 64 threads stage the words / gains of
// a run of ticks through shared memory with coalesced rows.
// the leg state as one integer, built from the fields (taking the struct's address would push the
// register-resident leg array of the compile-time-G kernels into local memory)
__device__ __forceinline__ uint64_t arb_leg_bits(const igd_arb_leg &l)
{
    return (uint64_t)l.last | ((uint64_t)l.msec << 8) | ((uint64_t)l.on << 16) | ((uint64_t)(uint8_t)l.rssi << 24) |
           ((uint64_t)l.gain_q7 << 32);
}
#ifndef IGD_ARB_THREADS
#define IGD_ARB_THREADS 128
#endif
constexpr int kArbThreads = IGD_ARB_THREADS;   // staging threads per block; the first bpb (<= kArbMaxBpb) of them walk a bridge each
constexpr int kArbMaxBpb = 64;
constexpr int kArbStageWords = 4096;     // words (and gains) of a run of ticks staged per block
template <int kG> struct arb_legs {      // compile-time leg count: the leg state lives in registers
    igd_arb_leg v[kG > 0 ? kG : 1];
};
template <int kG>
__global__ void __launch_bounds__(kArbThreads) k_gate_arbitrate(const igd_arb_desc d, const int bpb)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const int G = kG > 0 ? kG : d.G;
    uint32_t *words_s = reinterpret_cast<uint32_t *>(smem);             // [T][bpb*G]
    uint16_t *gain_s = reinterpret_cast<uint16_t *>(words_s + kArbStageWords);   // [T][bpb*G]
    uint8_t *frame_s = reinterpret_cast<uint8_t *>(gain_s + kArbStageWords);      // [T][bpb*G] IGD_RXE_FRAME of the tick's event (wide rows)
    igd_arb_leg *legs_s = reinterpret_cast<igd_arb_leg *>(frame_s + kArbStageWords);   // [bpb][G] (runtime G only)
    const int b0 = blockIdx.x * bpb;
    const int b = b0 + threadIdx.x;
    const int nb = min(bpb, d.B - b0);
    const bool owner = (int)threadIdx.x < nb;                            // this thread walks bridge b
    const int row = nb * G;                                             // words of this block per tick
    const int T = max(1, kArbStageWords / (bpb * G));                   // ticks per staged run
    const size_t Cn = (size_t)d.B * G;
    arb_legs<kG> lr;
    igd_arb_leg *legs;
    if (kG > 0) {
        legs = lr.v;
        if (owner) {
#pragma unroll
            for (int g = 0; g < (kG > 0 ? kG : 1); g++) lr.v[g] = d.legs[(size_t)b * G + g];
        }
    } else {
        for (int k = threadIdx.x; k < row; k += kArbThreads) legs_s[k] = d.legs[(size_t)b0 * G + k];
        legs = legs_s + (owner ? threadIdx.x : 0) * G;
    }
    igd_arb_bridge br;
    if (owner) br = d.bridges[b];
    const uint8_t *act = d.active ? d.active + (size_t)b * G : nullptr;
    uint32_t act_mask = 0xFFFFFFFFu;                                    // G <= 32 legs
    if (act && owner) {
        act_mask = 0;
        for (int g = 0; g < G; g++) act_mask |= (act[g] != 0 ? 1u : 0u) << g;
    }
    // steady-state skip (see the walk below): the words of the last full pass and whether it moved the state
    uint32_t prevw[kG > 0 ? kG : 1];
    uint64_t snap[kG > 0 ? kG : 1];
    // runtime leg count: snapshots [bpb][G] u64 and last words [bpb][G] u32 follow the leg state in shared memory
    uint64_t *snap_s = reinterpret_cast<uint64_t *>(legs_s + (size_t)bpb * G) + (owner ? threadIdx.x : 0) * G;
    uint32_t *prev_s = reinterpret_cast<uint32_t *>(reinterpret_cast<uint64_t *>(legs_s + (size_t)bpb * G) + (size_t)bpb * G) +
                       (owner ? threadIdx.x : 0) * G;
    bool have_prev = false, steady = false, counting = false;
    for (int f0 = 0; f0 < d.F; f0 += T) {
        const int nt = min(T, d.F - f0);
        __syncthreads();
        // coalesced (a tick's words are contiguous), eight independent loads in flight per thread: the walk
        // below is short once the steady-state skip engages, so the staging latency is what is left
        const bool mark = (d.flags & IGD_ARB_F_SILENCE) != 0u && d.word_stride >= 8u;
        // a wide row (tens of bridges per block: many channels, few ticks per stage): thread = column, loop over the
        // ticks -- no index division on the staging path, and the event's flags byte comes in with the word so that the
        // write-out below only stores (65 536 channels x 100 ticks: 0.088 -> 0.061 ms).  A narrow row (a few bridges per
        // block, hundreds of ticks per stage) keeps the flattened loop: all threads busy.
        const bool wide = row * 2 >= kArbThreads;
        if (wide) {
            const size_t tick_bytes = Cn * d.word_stride;
            for (int j = threadIdx.x; j < row; j += kArbThreads) {
                const uint8_t *col = reinterpret_cast<const uint8_t *>(d.words) + ((size_t)f0 * Cn + (size_t)b0 * G + j) * d.word_stride;
                for (int t0 = 0; t0 < nt; t0 += 8) {
                    uint32_t v[8], fl[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        fl[u] = IGD_RXE_FRAME;
                        if (t0 + u < nt) {
                            const uint8_t *p = col + (size_t)(t0 + u) * tick_bytes;
                            v[u] = __ldg(reinterpret_cast<const uint32_t *>(p));
                            if (mark) fl[u] = __ldg(p + 4);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        if (t0 + u < nt) {
                            words_s[(t0 + u) * row + j] = v[u];
                            frame_s[(t0 + u) * row + j] = (uint8_t)(fl[u] & IGD_RXE_FRAME);
                        }
                    }
                }
            }
        } else
        for (int k0 = threadIdx.x; k0 < nt * row; k0 += kArbThreads * 8) {
            uint32_t v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int k = k0 + u * kArbThreads;
                if (k < nt * row) {
                    const int t = k / row, j = k - t * row;
                    const uint8_t *wrow = reinterpret_cast<const uint8_t *>(d.words) + ((size_t)(f0 + t) * Cn + (size_t)b0 * G) * d.word_stride;
                    v[u] = __ldg(reinterpret_cast<const uint32_t *>(wrow + (size_t)j * d.word_stride));
                }
            }
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int k = k0 + u * kArbThreads;
                if (k < nt * row) words_s[k] = v[u];
            }
        }
        __syncthreads();
        if (owner) {
            for (int t = 0; t < nt; t++) {
                if (kG == 4 && have_prev && steady) {
                    // tight scan over the ticks whose four words repeat the last full pass's: one 16-byte load,
                    // one compare, one 8-byte store of the (unchanged) gains per tick
                    const uint2 gpk = make_uint2((uint32_t)legs[0].gain_q7 | ((uint32_t)legs[1].gain_q7 << 16),
                                                 (uint32_t)legs[2 % (kG > 0 ? kG : 1)].gain_q7 | ((uint32_t)legs[3 % (kG > 0 ? kG : 1)].gain_q7 << 16));
                    int t2 = t;
#pragma unroll 4
                    for (; t2 < nt; t2++) {
                        const uint4 w = *reinterpret_cast<const uint4 *>(words_s + t2 * row + threadIdx.x * 4);
                        if ((w.x ^ prevw[0]) | (w.y ^ prevw[1 % (kG > 0 ? kG : 1)]) | (w.z ^ prevw[2 % (kG > 0 ? kG : 1)]) |
                            (w.w ^ prevw[3 % (kG > 0 ? kG : 1)]))
                            break;
                        *reinterpret_cast<uint2 *>(gain_s + t2 * row + threadIdx.x * 4) = gpk;
                    }
                    if (counting) br.sqlStatusCount += t2 - t;
                    t = t2;
                    if (t >= nt) break;
                }
                const uint32_t *wt = words_s + t * row + threadIdx.x * G;
                auto word = [&](int g) { return wt[g]; };
                auto active = [&](int g) { return ((act_mask >> g) & 1u) != 0u; };
                uint16_t *gt = gain_s + t * row + threadIdx.x * G;
                // Steady-state skip.  checkEvents() is a deterministic function of (state, words): when a pass
                // left the state unchanged, every further pass over the SAME words leaves it unchanged too, so
                // the gains simply repeat (PTT / squelch states last for hundreds of ticks; the hold-off
                // counters settle within six).  SERVER mode has one more steady form: while a selection is in
                // force (sqlStatusOn) a pass only counts sqlStatusCount up (roip_ed137.cpp:6028) and nothing
                // reads the count again (:6029 needs !sqlStatusOn).  The full pass runs whenever the words
                // change or the last full pass still moved the state -- bit-exact by construction.
                bool same = have_prev;
                if (kG > 0) {
#pragma unroll
                    for (int g = 0; g < (kG > 0 ? kG : 1); g++) same = same && wt[g] == prevw[g];
                } else {
                    for (int g = 0; g < G && same; g++) same = wt[g] == prev_s[g];
                }
#ifdef IGD_X_ARB_NOSKIP
                same = false;
#endif
                if (same && steady) {
                    if (counting) br.sqlStatusCount++;
                } else {
                    // snapshot -> full pass -> did anything move?
                    uint64_t snap_fold = 0;
                    const int32_t c0 = br.sqlStatusCount, l0 = br.ptt_level;
                    const uint8_t o0 = br.sqlStatusOn;
                    if (kG > 0) {
#pragma unroll
                        for (int g = 0; g < (kG > 0 ? kG : 1); g++) snap[g] = arb_leg_bits(legs[g]);
                    } else {
                        for (int g = 0; g < G; g++) snap_s[g] = arb_leg_bits(legs[g]);
                    }
                    if (kG > 0) {
                        const igd_const_int<(kG > 0 ? kG : 1)> Gc;
                        if (d.mode == IGD_ARB_CLIENT_PTT) igd_arb_client_tick(br, legs, Gc, word, active);
                        else igd_arb_server_best_tick(br, legs, Gc, word, active);
                    } else {
                        if (d.mode == IGD_ARB_CLIENT_PTT) igd_arb_client_tick(br, legs, G, word, active);
                        else igd_arb_server_best_tick(br, legs, G, word, active);
                    }
                    if (kG > 0) {
#pragma unroll
                        for (int g = 0; g < (kG > 0 ? kG : 1); g++) {
                            snap_fold |= snap[g] ^ arb_leg_bits(legs[g]);
                            prevw[g] = wt[g];
                        }
                    } else {
                        for (int g = 0; g < G; g++) {
                            snap_fold |= snap_s[g] ^ arb_leg_bits(legs[g]);
                            prev_s[g] = wt[g];
                        }
                    }
                    const bool legs_same = snap_fold == 0 && br.ptt_level == l0 && br.sqlStatusOn == o0;
                    counting = legs_same && br.sqlStatusOn != 0 && br.sqlStatusCount == c0 + 1;
                    steady = legs_same && (br.sqlStatusCount == c0 || counting);
                    have_prev = true;
                }
                if (kG > 0) {
#pragma unroll
                    for (int g = 0; g < (kG > 0 ? kG : 1); g++) gt[g] = legs[g].gain_q7;
                } else {
                    for (int g = 0; g < G; g++) gt[g] = legs[g].gain_q7;
                }
            }
        }
        __syncthreads();
        if (wide) {
            for (int j = threadIdx.x; j < row; j += kArbThreads) {
                uint16_t *gcol = d.gain_q7 + (size_t)f0 * Cn + (size_t)b0 * G + j;
#pragma unroll 4
                for (int t = 0; t < nt; t++) {
                    uint16_t gv = gain_s[t * row + j];
                    if (!frame_s[t * row + j]) gv |= (uint16_t)IGD_GAIN_NO_AUDIO;   // no whole audio frame on this tick: silent
                    gcol[(size_t)t * Cn] = gv;
                }
            }
        } else
        for (int k0 = threadIdx.x; k0 < nt * row; k0 += kArbThreads * 8) {
            uint32_t fl[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {      // words are igd_rx_event records: the flags byte follows the word
                const int k = k0 + u * kArbThreads;
                fl[u] = IGD_RXE_FRAME;
                if (mark && k < nt * row) {
                    const int t = k / row, j = k - t * row;
                    const uint8_t *ev = reinterpret_cast<const uint8_t *>(d.words) + ((size_t)(f0 + t) * Cn + (size_t)b0 * G + j) * d.word_stride;
                    fl[u] = __ldg(ev + 4);
                }
            }
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int k = k0 + u * kArbThreads;
                if (k < nt * row) {
                    const int t = k / row, j = k - t * row;
                    uint16_t gv = gain_s[k];
                    if (!(fl[u] & IGD_RXE_FRAME)) gv |= (uint16_t)IGD_GAIN_NO_AUDIO;   // no whole audio frame on this tick: silent
                    d.gain_q7[(size_t)(f0 + t) * Cn + (size_t)b0 * G + j] = gv;
                }
            }
        }
    }
    __syncthreads();
    if (owner) d.bridges[b] = br;
    if (kG > 0) {
        if (owner) {
#pragma unroll
            for (int g = 0; g < (kG > 0 ? kG : 1); g++) d.legs[(size_t)b * G + g] = lr.v[g];
        }
    } else {
        for (int k = threadIdx.x; k < row; k += kArbThreads) d.legs[(size_t)b0 * G + k] = legs_s[k];
    }
}

// ============================================================ receive side of a wide, short call: one thread per bridge
// Tens of thousands of channels and a few ticks per call (65 536 x 100): enough independent walks to hide a
// thread's latency, so the thread-per-channel form stays -- but as ONE kernel: a thread walks the four legs of its
// bridge through transport_rtp_cb's state (igd_rx_step, header words straight out of the packets, as k_rx_track<3>)
// and hands the four latched words to checkEvents() (the steady-state skip of k_gate_arbitrate) in registers.  No
// event array between the two, one launch less, and the arbitration's own 100-tick latency chain (0.10 ms) rides on
// the header reads, which bound this kernel (every 20-byte header costs the DRAM line(s) it lies in: 0.94 GB).
constexpr int kRbAhead = 4;          // ticks whose header words are in flight per thread (4 legs x 4 words each)
__global__ void __launch_bounds__(64) k_rxarb_bridge(const igd_rxarb_args a)
{
    constexpr int G = 4;
    const int b = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (b >= a.B) return;
    const size_t Cn = (size_t)a.B * G, ch0 = (size_t)b * G;
    igd_rx_state s[G];
    arb_legs<G> lr;
#pragma unroll
    for (int g = 0; g < G; g++) { s[g] = a.rx_state[ch0 + g]; lr.v[g] = a.legs[ch0 + g]; }
    igd_arb_leg *legs = lr.v;
    igd_arb_bridge br = a.bridges[b];
    uint32_t act_mask = 0xFu;
    if (a.active) {
        act_mask = 0;
#pragma unroll
        for (int g = 0; g < G; g++) act_mask |= (a.active[ch0 + g] != 0 ? 1u : 0u) << g;
    }
    uint32_t prevw[G] = {0u, 0u, 0u, 0u};
    uint64_t snap[G];
    bool have_prev = false, steady = false, counting = false;
    uint4 raw[kRbAhead][G];              // {word 0, word 3, word 4, received size} of the next kRbAhead ticks
    auto fetch = [&](int f, uint4 (&r)[G]) {
        if (f < a.F) {
            const size_t i = (size_t)f * Cn + ch0;
            const uint32_t *pw = reinterpret_cast<const uint32_t *>(a.pkts + i * IGD_PKT_MAX);
#pragma unroll
            for (int g = 0; g < G; g++)
                r[g] = make_uint4(__ldg(pw + g * kPktWords), __ldg(pw + g * kPktWords + 3), __ldg(pw + g * kPktWords + 4),
                                  a.sizes ? __ldg(a.sizes + i + g) : (uint32_t)IGD_PKT_MAX);
        }
    };
#pragma unroll
    for (int u = 0; u < kRbAhead; u++) fetch(u, raw[u]);
    const int wd_ticks = a.wd_ticks;
    int wd_phase = wd_ticks > 0 ? (int)(a.frame0 % wd_ticks) : 0;
    long long now = a.now_ms0;
    for (int f0 = 0; f0 < a.F; f0 += kRbAhead) {
#pragma unroll
        for (int u = 0; u < kRbAhead; u++) {
            const int f = f0 + u;
            if (f >= a.F) break;
            const bool wd = wd_ticks > 0 && wd_phase == wd_ticks - 1;
            wd_phase = wd_phase + 1 == wd_ticks ? 0 : wd_phase + 1;
            uint32_t w[G], noaud = 0u;
#pragma unroll
            for (int g = 0; g < G; g++) {
                const uint4 r = raw[u][g];
                const uint32_t navail = min(r.w, (uint32_t)IGD_PKT_MAX) / 4;      // words transport_rtp_cb may look at
                const igd_ed137_fields fl = fields_of_header(navail > 0 ? r.x : 0u, navail > 3 ? r.y : 0u, navail > 4 ? r.z : 0u, r.w);
                const uint32_t ev = igd_rx_step(s[g], fl, r.w != 0u, wd, now, a.r2s_period_ms);
                w[g] = s[g].ed137_value;
                if (!(ev & IGD_RXE_FRAME)) noaud |= 1u << g;
                if (a.events) {
                    igd_rx_event e;
                    e.word = s[g].ed137_value; e.flags = (uint8_t)ev; e.r2sCount = s[g].r2sCount; e.reserved = 0;
                    *reinterpret_cast<uint2 *>(a.events + (size_t)f * Cn + ch0 + g) = *reinterpret_cast<const uint2 *>(&e);
                }
            }
            fetch(f + kRbAhead, raw[u]);                              // this slot's next tick goes in flight
            now += a.tick_ms;
            // checkEvents() with the steady-state skip (see k_gate_arbitrate)
            bool same = have_prev;
#pragma unroll
            for (int g = 0; g < G; g++) same = same && w[g] == prevw[g];
            if (same && steady) {
                if (counting) br.sqlStatusCount++;
            } else {
                uint64_t fold = 0;
                const int32_t c0 = br.sqlStatusCount, l0 = br.ptt_level;
                const uint8_t o0 = br.sqlStatusOn;
#pragma unroll
                for (int g = 0; g < G; g++) snap[g] = arb_leg_bits(legs[g]);
                auto word = [&](int g) { return w[g]; };
                auto active = [&](int g) { return ((act_mask >> g) & 1u) != 0u; };
                const igd_const_int<G> Gc;
                if (a.mode == IGD_ARB_CLIENT_PTT) igd_arb_client_tick(br, legs, Gc, word, active);
                else igd_arb_server_best_tick(br, legs, Gc, word, active);
#pragma unroll
                for (int g = 0; g < G; g++) {
                    fold |= snap[g] ^ arb_leg_bits(legs[g]);
                    prevw[g] = w[g];
                }
                const bool legs_same = fold == 0 && br.ptt_level == l0 && br.sqlStatusOn == o0;
                counting = legs_same && br.sqlStatusOn != 0 && br.sqlStatusCount == c0 + 1;
                steady = legs_same && (br.sqlStatusCount == c0 || counting);
                have_prev = true;
            }
            const uint32_t na = (uint32_t)IGD_GAIN_NO_AUDIO;       // a tick without a whole audio frame is silent (IGD_ARB_F_SILENCE)
            const uint32_t g01 = (uint32_t)legs[0].gain_q7 | ((uint32_t)legs[1].gain_q7 << 16) | ((noaud & 1u) ? na : 0u) | ((noaud & 2u) ? na << 16 : 0u);
            const uint32_t g23 = (uint32_t)legs[2].gain_q7 | ((uint32_t)legs[3].gain_q7 << 16) | ((noaud & 4u) ? na : 0u) | ((noaud & 8u) ? na << 16 : 0u);
            *reinterpret_cast<uint2 *>(a.gain_q7 + (size_t)f * Cn + ch0) = make_uint2(g01, g23);
        }
    }
#pragma unroll
    for (int g = 0; g < G; g++) { a.rx_state[ch0 + g] = s[g]; a.legs[ch0 + g] = lr.v[g]; }
    a.bridges[b] = br;
}

// Phase 1: one thread per channel walks its frames through the sender state
// machine (transport_send_rtp, TransportAdapter.cpp:635-874) and writes a plan
// record per packet.  The state is tiny and strictly sequential per channel.
__global__ void __launch_bounds__(128) k_ed137_plan(const igd_ed137_pack_desc d, igd_tx_plan_rec *__restrict__ plan,
                                                    int32_t *__restrict__ last_src)
{
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d.C) return;
    igd_ed137_state s = d.state[c];
    int32_t src = -1;
    const bool stuck = d.payload != nullptr && 12u + d.payload_len > 60u;   // gateway form: the payload does not exist yet
    igd_tx_plan last;                    // steady-state skip: result of the last full step
    last.word = 0; last.size = 0; last.pt123 = 0; last.marker = 0; last.copy_payload = 0;
    uint64_t last_ctl = 0;
    bool have_last = false, steady = false;
    constexpr int kAhead = 8;            // the walk is sequential, its inputs are not: fetch 8 frames ahead
    for (int f0 = 0; f0 < d.F; f0 += kAhead) {
        igd_ed137_ctl kk[kAhead];
        uint32_t a40[kAhead], a50[kAhead], a60[kAhead];
#pragma unroll
        for (int u = 0; u < kAhead; u++) {
            const int f = f0 + u;
            if (f < d.F) {
                const size_t i = (size_t)f * d.C + c;
                if (d.ctl) kk[u] = d.ctl[i];
                if (stuck) {
                    const uint8_t *pl = d.payload + i * IGD_FRAME;
                    a40[u] = pl[40 - 12]; a50[u] = pl[50 - 12]; a60[u] = pl[60 - 12];
                }
            }
        }
#pragma unroll
        for (int u = 0; u < kAhead; u++) {
            const int f = f0 + u;
            if (f >= d.F) break;
            const size_t i = (size_t)f * d.C + c;
            bool ctl_same = have_last;
            if (d.ctl) {                                                     // the setters, :135-213
                const igd_ed137_ctl k = kk[u];
                const uint64_t kbits = *reinterpret_cast<const uint64_t *>(&k);
                ctl_same = ctl_same && kbits == last_ctl;
                last_ctl = kbits;
                s.pttstatus = k.pttstatus; s.pttpriority = k.pttpriority; s.callRecorder = k.callRecorder;
                s.sqlstatus = k.sqlstatus; s.ed137_bssi = k.ed137_bssi; s.pttid = k.pttid;
            }
            // :675-679 -- on every call, also the ones the steady-state skip answers (the step itself repeats it)
            if (s.radiostatus && (s.calltype_flags & 1u) && s.callIn) { s.sqlstatus = 0; s.pttstatus = 0; }
            if (s.radiostatus && stuck) {                                    // stuck-audio detector :657-673
                if (a40[u] == a50[u] && a40[u] == a60[u] && a40[u] == 0xd5) s.rtpFalse += 1; else s.rtpFalse = 0;
            }
            const long long now = d.now_ms0 + (long long)f * d.tick_ms;
            // Steady-state skip.  transport_send_rtp is a deterministic function of (state, setter values, clock)
            // and the clock only enters through the keep-alive throttle (:685-706).  Once a call has left the
            // state as it found it (the 30-packet start burst and the 5-packet slave-enable latch are over),
            // every further call with the SAME setter values gives the same header; what is left per tick is
            // the throttle.  The full step runs whenever the setter values change, the last full step still
            // moved the state, or no sent header is cached for this situation -- bit-exact by construction.
            igd_tx_plan t;
            bool fast = false;
#ifdef IGD_X_PLAN_NOSKIP
            ctl_same = false;
#endif
            if (ctl_same && steady) {
                if (last.copy_payload) {                                     // gated audio: goes out on every tick
                    t = last; fast = true;
                } else {
                    const unsigned long long since = (unsigned long long)now - (unsigned long long)s.r2sSendtime;
                    const unsigned long long ka = (unsigned long long)(long long)s.keepAlivePeroid;
                    if (since < ka) {                                        // throttled (firstR2SPacket is over when steady)
                        t.word = 0; t.size = 0; t.pt123 = 0; t.marker = 0; t.copy_payload = 0; fast = true;
                    } else if (last.size != 0) {                             // keep-alive due: the cached header again
                        s.r2sSendtime = now;
                        t = last; fast = true;
                    }
                }
            }
            if (!fast) {
                igd_ed137_state before = s;
                t = igd_ed137_tx_step(s, d.payload_len, now);
                before.r2sSendtime = s.r2sSendtime;                          // the throttle clock is not part of "steady"
                const uint64_t *pa = reinterpret_cast<const uint64_t *>(&before), *pb = reinterpret_cast<const uint64_t *>(&s);
                steady = pa[0] == pb[0] && pa[1] == pb[1] && pa[2] == pb[2] && pa[3] == pb[3] && pa[4] == pb[4] &&
                         !s.firstR2SPacket;
                last = t;            // cached header = the one built by THIS step (a throttled step caches size 0, so the
                have_last = true;    // next keep-alive that is due takes the full step again, now in the settled state)
            }
            if (t.copy_payload) src = f;
            igd_tx_plan_rec r;
            r.word = t.word;
            r.size = (uint16_t)t.size;
            r.flags = (uint8_t)(t.pt123 | (t.marker << 1) | (t.copy_payload << 2));
            r.reserved = 0;
            r.src_frame = (d.flags & IGD_F_REF_QUIRKS) ? src : f;            // quirk Q2
            plan[i] = r;
        }
    }
    d.state[c] = s;
    last_src[c] = src;
}

// sendR2SStatus (TransportAdapter.cpp:422-633): thread per channel, one timer tick
__global__ void __launch_bounds__(128) k_ed137_keepalive(uint8_t *__restrict__ hdr20, igd_ed137_state *__restrict__ state,
                                                         size_t C, long long now, uint32_t *__restrict__ sizes)
{
    const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    igd_ed137_state s = state[c];
    uint32_t *h = reinterpret_cast<uint32_t *>(hdr20 + c * IGD_PKT_HDR);
    uint32_t w0 = h[0];
    const igd_tx_plan t = igd_ed137_r2s_step(s, now, (w0 >> 8) & 0x7Fu);
    if (t.copy_payload) {                                   // the header fields are stamped into the send buffer
        w0 |= 0x10u;                                                           // x = 1 (:495)
        w0 = (w0 & ~0x8000u) | (t.marker ? 0x8000u : 0u);                      // m (:485-493)
        if (t.pt123) w0 = (w0 & ~0x7F00u) | (123u << 8);
        h[0] = w0;
        h[3] = 0x01006701u;                                                    // 0x0167, 0x0001 big-endian
        h[4] = bswap32(t.word);
    }
    sizes[c] = t.size;
    state[c] = s;
}

// after the packets are assembled: remember the payload each adapter's send buffer ends up holding
__global__ void __launch_bounds__(256) k_ed137_stale_update(const igd_ed137_pack_desc d,
                                                            const int32_t *__restrict__ last_src)
{
    const uint32_t lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t c = warp; c < (size_t)d.C; c += nwarps) {
        const int32_t f = last_src[c];
        if (f < 0) continue;
        const uint32_t *src = reinterpret_cast<const uint32_t *>(d.payload + ((size_t)f * d.C + c) * IGD_FRAME);
        uint32_t *dst = reinterpret_cast<uint32_t *>(d.stale_payload + c * IGD_FRAME);
        for (uint32_t k = lane; k < IGD_FRAME / 4; k += 32) dst[k] = src[k];
    }
}

// Phase 2: one warp per packet assembles header + payload (4-byte words; the
// payload sits at byte 20 of a 180-byte packet, so 16-byte accesses do not apply)
__global__ void __launch_bounds__(256) k_ed137_assemble(const igd_ed137_pack_desc d,
                                                        const igd_tx_plan_rec *__restrict__ plan)
{
    const uint32_t lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const size_t npkts = (size_t)d.F * d.C;
    const bool sc = (d.flags & IGD_F_SIGNED_CHAR) != 0, quirks = (d.flags & IGD_F_REF_QUIRKS) != 0;
    const uint32_t nwords = d.payload_len / 4;
    for (size_t i = warp; i < npkts; i += nwarps) {
        const igd_tx_plan_rec r = plan[i];
        uint32_t *out = reinterpret_cast<uint32_t *>(d.pkts + i * d.out_stride);
        const uint32_t *hdr = reinterpret_cast<const uint32_t *>(d.rtp12 + i * 12);
        const size_t c = i % (size_t)d.C;
        if (lane == 0) d.sizes[i] = r.size;
        int bsum = 0;
        // the bytes of the slot past the packet are defined (zero): nobody has to clear the buffer first
        for (uint32_t k = r.size / 4 + lane; k < d.out_stride / 4; k += 32) out[k] = 0u;
        if (r.size == 0) {
            if (lane == 0) d.bytemean_out[i] = 0;
            continue;
        }
        if (lane < 5) {
            uint32_t v;
            if (lane < 3) {
                v = hdr[lane];
                if (lane == 0) {
                    v |= 0x10u;                                            // x = 1 (:725)
                    v = (v & ~0x8000u) | ((r.flags & 2u) ? 0x8000u : 0u);  // m (:715-723)
                    if (r.flags & 1u) v = (v & ~0x7F00u) | (123u << 8);    // pt = 123
                }
            } else if (lane == 3) {
                v = 0x01006701u;                                           // 0x0167, 0x0001 big-endian
            } else {
                v = bswap32(r.word);                                       // htonl (:800)
            }
            out[lane] = v;
        }
        const bool audio = !(r.flags & 1u);
        if (r.size > IGD_PKT_HDR) {
            const uint32_t *src = r.src_frame >= 0
                ? reinterpret_cast<const uint32_t *>(d.payload + ((size_t)r.src_frame * d.C + c) * IGD_FRAME)
                : (d.stale_payload ? reinterpret_cast<const uint32_t *>(d.stale_payload + c * IGD_FRAME) : nullptr);
            for (uint32_t k = lane; k < nwords; k += 32) out[5 + k] = src ? src[k] : 0u;
        }
        if (audio) {
            // setOutgoingRTP (roip_ed137.cpp:6500-6536).  Clean: mean of the payload
            // bytes.  Quirk Q3: mean of the first payload_len bytes of the ORIGINAL
            // packet (12 header bytes + payload[0 .. len-12)), TransportAdapter.cpp:654.
            const uint32_t *cur = reinterpret_cast<const uint32_t *>(d.payload + i * IGD_FRAME);
            if (!quirks) {
                for (uint32_t k = lane; k < nwords; k += 32) bsum = bytesum4(cur[k], sc, bsum);
            } else {
                for (uint32_t k = lane; k < nwords; k += 32) {
                    const uint32_t v = k < 3 ? hdr[k] : cur[k - 3];
                    bsum = bytesum4(v, sc, bsum);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) bsum += __shfl_xor_sync(0xffffffffu, bsum, o);
        }
        if (lane == 0) d.bytemean_out[i] = audio ? (uint8_t)igd_bytemean_from_sum(bsum, (int)d.payload_len) : 0;
    }
}

// The two tile kernels below (k_ed137_assemble_tile, k_fanout_tile) build 64 wire packets in a shared-memory
// image of 64 x 45 words and share its header rewrite and its write-out.
//
// Header rewrite of transport_send_rtp (TransportAdapter.cpp:715-725, 800): PJSIP's 12 bytes h0..h2 with x = 1, the
// plan's marker and PT 123, then the profile / length word and the ED-137 word -- the packet's first five words.
__device__ __forceinline__ void tile_header(uint32_t *o, const igd_tx_plan_rec &r, uint32_t h0, uint32_t h1, uint32_t h2)
{
    uint32_t v0 = h0 | 0x10u;                                              // x = 1 (:725)
    v0 = (v0 & ~0x8000u) | ((r.flags & 2u) ? 0x8000u : 0u);                // m (:715-723)
    if (r.flags & 1u) v0 = (v0 & ~0x7F00u) | (123u << 8);                  // pt = 123
    o[0] = v0; o[1] = h1; o[2] = h2; o[3] = 0x01006701u; o[4] = bswap32(r.word);   // 0x0167, 0x0001 big-endian; htonl (:800)
}

// Write-out of a finished image of np packets to dst (= packet 0 of the tile): ONE bulk async store (TMA) when the
// image holds every byte of the tile (*partial == 0: every packet is 180 bytes, or the image is zero past each packet's
// size), otherwise coalesced word stores of only the bytes each packet's size covers, the rest of its slot zero.
// Called by every thread of the CTA once the image and size_s are written.
__device__ __forceinline__ void tile_store(uint8_t *dst, const uint32_t *img, const uint32_t *size_s, uint32_t np,
                                           const uint32_t *partial)
{
    fence_proxy_async();             // the image is read by the async proxy below
    __syncthreads();
    const uint32_t tile_bytes = np * IGD_PKT_MAX;
    if (!*partial && (tile_bytes & 15u) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
        if (threadIdx.x == 0) {
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         ::"l"(dst), "r"(shared_addr(img)), "r"(tile_bytes) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");     // smem must outlive the read
        }
    } else {
        uint32_t *out = reinterpret_cast<uint32_t *>(dst);
        for (uint32_t w = threadIdx.x; w < np * kPktWords; w += blockDim.x) {
            const uint32_t p = w / kPktWords, k = w - p * kPktWords;
            out[w] = 4 * k < size_s[p] ? img[w] : 0u;              // past the packet the slot reads zero
        }
    }
}

// Tile form of the assembly for the wire shape (out_stride 180, 160-byte payloads): a CTA builds
// 64 packets in shared memory (headers by 64 threads, payload chunks by all threads with 16-byte
// loads) and writes the image out with coalesced word stores, only the bytes each packet's size
// covers -- same bytes, sizes and levels as k_ed137_assemble above.
__global__ void __launch_bounds__(256) k_ed137_assemble_tile(const igd_ed137_pack_desc d,
                                                             const igd_tx_plan_rec *__restrict__ plan)
{
    __shared__ __align__(128) uint32_t img[kPktTile * kPktWords];           // the 64 packets being built
    __shared__ __align__(128) uint32_t pay[kPktTile * (IGD_FRAME / 4)];      // this tick's payloads of the tile
    __shared__ uint64_t bar;
    __shared__ uint32_t size_s[kPktTile];
    __shared__ int32_t srcf_s[kPktTile];
    __shared__ uint32_t flag_s[kPktTile];
    __shared__ int bsum_s[kPktTile];
    __shared__ uint32_t chan_s[kPktTile];
    __shared__ int32_t frame_s[kPktTile];
    __shared__ uint32_t not_full;                                            // some packet of the tile is not 180 bytes
    const size_t npkts = (size_t)d.F * d.C;
    const size_t first = (size_t)blockIdx.x * kPktTile;
    const uint32_t np = (uint32_t)min((size_t)kPktTile, npkts - first);
    const bool sc = (d.flags & IGD_F_SIGNED_CHAR) != 0, quirks = (d.flags & IGD_F_REF_QUIRKS) != 0;
    const uint32_t bar_s = shared_addr(&bar);
    if (threadIdx.x == 0) {          // ONE bulk async copy (TMA) stages the tile's current payloads (np*160 contiguous bytes)
        not_full = 0u;
        mbar_init(bar_s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(bar_s, np * IGD_FRAME);
        bulk_g2s(shared_addr(pay), d.payload + first * IGD_FRAME, np * IGD_FRAME, bar_s);
    }
    if (threadIdx.x < np) {
        const uint32_t p = threadIdx.x;
        const size_t i = first + p;
        const igd_tx_plan_rec r = plan[i];
        const uint32_t *hdr = reinterpret_cast<const uint32_t *>(d.rtp12 + i * 12);
        const uint32_t h0 = hdr[0], h1 = hdr[1], h2 = hdr[2];
        tile_header(img + p * kPktWords, r, h0, h1, h2);
        size_s[p] = r.size;
        srcf_s[p] = r.src_frame;
        flag_s[p] = r.flags;
        frame_s[p] = (int32_t)(i / (size_t)d.C);
        chan_s[p] = (uint32_t)(i - (size_t)frame_s[p] * d.C);
        d.sizes[i] = r.size;
        // quirk Q3: the level sums the first 160 bytes of the ORIGINAL packet = these 12 header bytes ...
        int hs = 0;
        if (quirks) { hs = bytesum4(h0, sc, hs); hs = bytesum4(h1, sc, hs); hs = bytesum4(h2, sc, hs); }
        bsum_s[p] = hs;
    }
    __syncthreads();                 // barrier initialised, per-packet plan visible
    if (threadIdx.x < np && size_s[threadIdx.x] != IGD_PKT_MAX) not_full = 1u;
    mbar_wait(bar_s, 0);
    for (uint32_t j = threadIdx.x; j < np * kChunks; j += blockDim.x) {
        const uint32_t p = j / kChunks, ch = j - p * kChunks;
        const uint32_t size = size_s[p];
        if (size == 0) continue;
        const bool audio = !(flag_s[p] & 1u);
        const size_t c = chan_s[p];
        const int32_t f = frame_s[p], sf = srcf_s[p];
        const uint4 cur = *reinterpret_cast<const uint4 *>(pay + p * (IGD_FRAME / 4) + ch * 4);
        if (size > IGD_PKT_HDR) {
            uint4 v = cur;
            if (sf != f) {           // quirk Q2: the send buffer still holds an older frame's payload
                if (sf >= 0) v = __ldg(reinterpret_cast<const uint4 *>(d.payload + ((size_t)sf * d.C + c) * IGD_FRAME) + ch);
                else if (d.stale_payload) v = __ldg(reinterpret_cast<const uint4 *>(d.stale_payload + c * IGD_FRAME) + ch);
                else v = make_uint4(0u, 0u, 0u, 0u);
            }
            uint32_t *o = img + p * kPktWords + 5 + ch * 4;
            o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
        }
        if (audio) {        // setOutgoingRTP (roip_ed137.cpp:6500-6536): clean = the payload bytes;
            int bs = 0;     // Q3 = ... + payload[0 .. 148) (TransportAdapter.cpp:654)
            if (!quirks || ch < 9) {
                bs = bytesum4(cur.x, sc, bs); bs = bytesum4(cur.y, sc, bs); bs = bytesum4(cur.z, sc, bs); bs = bytesum4(cur.w, sc, bs);
            } else {
                bs = bytesum4(cur.x, sc, bs);                                  // bytes 144..147
            }
            atomicAdd(&bsum_s[p], bs);
        }
    }
    tile_store(d.pkts + first * IGD_PKT_MAX, img, size_s, np, &not_full);
    if (threadIdx.x < np) {
        const uint32_t p = threadIdx.x;
        const bool audio = size_s[p] != 0 && !(flag_s[p] & 1u);
        d.bytemean_out[first + p] = audio ? (uint8_t)igd_bytemean_from_sum(bsum_s[p], IGD_FRAME) : (uint8_t)0;
    }
}

// ============================================================ gateway fan-out
// igd_gateway_fanout's assembly: the same 64-packet tile as k_ed137_assemble_tile, its payloads encoded here from the
// bridges' PCM instead of read.  Packet i = f*B*G + b*G + g belongs to bridge-frame i / G, so a tile's 64 packets span
// at most ceil(63/G)+1 consecutive bridge-frames (G = 1: 64) whose PCM is one contiguous run: ONE bulk async copy
// stages it.  Every (bridge-frame, law) present among the tile's legs is encoded once (16 samples per thread, the
// packed compressor of igd_g711_encode_ch), its byte sum taken once for the level of every packet that carries it,
// and the 16 code bytes go into the payload of each of those packets that is sent whole (180 bytes).  The image is
// zero past each packet's size, so every tile of whole packets leaves with ONE bulk store, whatever its sizes (with
// word stores for the mixed tiles, which are most of them, the kernel ran at 37 % of the HBM peak).
constexpr int kFanBf = kPktTile;         // bridge-frames a tile can touch: ceil(63/G)+1 <= 64
__host__ __device__ constexpr uint32_t fanout_tile_bfs(int G) { return (uint32_t)((kPktTile - 2 + G) / G + 1); }
// 32 registers, no spills: eight CTAs per SM (19 KB of shared memory each at G = 4) keep more tiles' loads and stores
// in flight than the six that 40 registers allowed
__global__ void __launch_bounds__(256, 8) k_fanout_tile(const igd_ed137_pack_desc d, const int G,
                                                     const int16_t *__restrict__ pcm, const uint8_t *__restrict__ law,
                                                     const igd_tx_plan_rec *__restrict__ plan)
{
    __shared__ __align__(128) uint32_t img[kPktTile * kPktWords];             // the 64 packets being built
    extern __shared__ __align__(128) uint32_t pcm_s[];                       // the tile's bridge-frames (fanout_tile_bfs(G))
    __shared__ unsigned long long legs_s[2 * kFanBf];   // [bridge-frame][law]: bit p = packet p of the tile carries it
    __shared__ int bsum_s[2 * kFanBf];                  // [bridge-frame][law]: byte sum of the encoded frame
    __shared__ uint64_t bar;
    __shared__ uint32_t size_s[kPktTile];
    __shared__ uint32_t pair_s[kPktTile];               // packet p -> its [bridge-frame][law] entry; bit 31 = PT 123
    const size_t npkts = (size_t)d.F * d.C;
    const size_t first = (size_t)blockIdx.x * kPktTile;
    const uint32_t np = (uint32_t)min((size_t)kPktTile, npkts - first);
    const size_t bf0 = first / (uint32_t)G;
    const uint32_t nbf = (uint32_t)((first + np - 1) / (uint32_t)G - bf0) + 1;
    const bool sc = (d.flags & IGD_F_SIGNED_CHAR) != 0;
    const uint32_t bar_s = shared_addr(&bar);
    if (threadIdx.x == 0) {
        mbar_init(bar_s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(bar_s, nbf * IGD_FRAME * 2);
        bulk_g2s(shared_addr(pcm_s), pcm + bf0 * IGD_FRAME, nbf * IGD_FRAME * 2, bar_s);
    }
    for (uint32_t k = threadIdx.x; k < 2 * nbf; k += blockDim.x) { legs_s[k] = 0ull; bsum_s[k] = 0; }
    __syncthreads();                 // barrier initialised, leg masks cleared
    if (threadIdx.x < np) {
        const uint32_t p = threadIdx.x;
        const size_t i = first + p;
        const igd_tx_plan_rec r = plan[i];
        const uint32_t *hdr = reinterpret_cast<const uint32_t *>(d.rtp12 + i * 12);
        tile_header(img + p * kPktWords, r, hdr[0], hdr[1], hdr[2]);
        size_s[p] = r.size;
        d.sizes[i] = r.size;
        const size_t c = i % (size_t)d.C;                                     // leg b*G + g
        const uint32_t pr = 2u * (uint32_t)(i / (uint32_t)G - bf0) + (law[c] != 0 ? 1u : 0u);   // igd_enc_law_make: 0 = A-law, else u-law
        pair_s[p] = pr | ((r.flags & 1u) << 31);
        atomicOr(&legs_s[pr], 1ull << p);
    }
    __syncthreads();                 // leg masks and headers complete
    for (uint32_t w = threadIdx.x; w < np * kPktWords; w += blockDim.x) {     // zero past each packet (no payload there)
        const uint32_t p = w / kPktWords;
        if (4 * (w - p * kPktWords) >= size_s[p]) img[w] = 0u;
    }
    mbar_wait(bar_s, 0);             // the PCM has landed
    for (uint32_t j = threadIdx.x; j < 2 * nbf * kChunks; j += blockDim.x) {
        const uint32_t pr = j / kChunks, ch = j - pr * kChunks;
        const unsigned long long m = legs_s[pr];
        if (!m) continue;            // no leg of this bridge-frame in the tile uses this law
        const uint4 *src = reinterpret_cast<const uint4 *>(pcm_s + (pr >> 1) * (IGD_FRAME / 2) + ch * 8);
        const uint4 a = src[0], b = src[1];
        const uint32_t pk[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        const uint4 e = encode16_packed(pk, enc_pk_make((int)(pr & 1u)));
        int bs = 0;
        bs = bytesum4(e.x, sc, bs); bs = bytesum4(e.y, sc, bs); bs = bytesum4(e.z, sc, bs); bs = bytesum4(e.w, sc, bs);
        atomicAdd(&bsum_s[pr], bs);
        for (unsigned long long mm = m; mm; mm &= mm - 1) {
            const uint32_t p = (uint32_t)(__ffsll((long long)mm) - 1);
            if (size_s[p] != IGD_PKT_MAX) continue;
            uint32_t *o = img + p * kPktWords + 5 + ch * 4;
            o[0] = e.x; o[1] = e.y; o[2] = e.z; o[3] = e.w;
        }
    }
    const uint32_t whole = 0u;       // the image holds every byte of the tile
    tile_store(d.pkts + first * IGD_PKT_MAX, img, size_s, np, &whole);
    if (threadIdx.x < np && d.bytemean_out) {
        const uint32_t p = threadIdx.x, pr = pair_s[p];
        const bool audio = size_s[p] != 0 && !(pr >> 31);          // setOutgoingRTP (roip_ed137.cpp:6500-6536), clean
        d.bytemean_out[first + p] = audio ? (uint8_t)igd_bytemean_from_sum(bsum_s[pr & 0x7FFFFFFFu], IGD_FRAME) : (uint8_t)0;
    }
}

// ============================================================ gateway fan-out from packets
// igd_gateway_fanout_packets' assembly: k_fanout_tile's tile, with each payload mapped code by code out of the console
// call's received packet instead of encoded from PCM.  Bridge-frame bf's console packet is rx_pkts + bf*180, so a tile's
// bridge-frames are again one contiguous run.  bf0*180 is only 4-byte aligned, so ONE bulk async copy stages the
// 16-byte-aligned window that covers the run, and the run starts `lead` = 0, 1, 2 or 3 words into it: payload words in
// shared memory are 4-byte aligned and read as 32-bit words.  The window never leaves the array: when the array's size
// is not a multiple of 16, the last tile's copy stops at the last whole 16 bytes and threads load the <= 3 words after.
// Every output byte is enc_out(dec_in(code)): a 2 x 2 x 256 code table [in law][out law][code] from igd_g711_transcode1,
// built per CTA (one code per thread, four entries) while the staging copy and the plan loads are in flight.  A table
// in device memory would be context state that must exist before a graph capture, to save work that is hidden anyway.
// A bridge-frame whose console packet is not a whole G.711 audio frame (the IGD_RXE_FRAME rule: fields_of_header,
// then igd_fields_no_audio) sends digital silence: the out law's code for PCM 0.
__host__ __device__ constexpr uint32_t fanout_pkt_stage_bytes(int G)      // lead + the bridge-frames' packets, to 16 B
{
    return (12u + fanout_tile_bfs(G) * IGD_PKT_MAX + 15u) & ~15u;         // G = 1: 11 536, G = 4: 3072, G = 32: 560
}
__global__ void __launch_bounds__(256, 8) k_fanout_pkt_tile(const igd_ed137_pack_desc d, const int G,
                                                         const uint8_t *__restrict__ rx_pkts,
                                                         const uint32_t *__restrict__ rx_sizes,
                                                         const uint8_t *__restrict__ in_law, const uint8_t *__restrict__ law,
                                                         const igd_tx_plan_rec *__restrict__ plan)
{
    __shared__ __align__(128) uint32_t img[kPktTile * kPktWords];             // the 64 packets being built
    extern __shared__ __align__(128) uint32_t win_s[];                       // the staged window (fanout_pkt_stage_bytes(G))
    __shared__ unsigned long long legs_s[2 * kFanBf];   // [bridge-frame][law]: bit p = packet p of the tile carries it
    __shared__ int bsum_s[2 * kFanBf];                  // [bridge-frame][law]: byte sum of the mapped frame
    __shared__ __align__(4) uint8_t tab_s[2 * 2 * 256];  // [in law][out law][code] -> code
    __shared__ uint32_t rsz_s[kFanBf];                  // [bridge-frame]: received size of the console packet
    __shared__ uint32_t bfi_s[kFanBf];                  // [bridge-frame]: bit 0 = in law is u-law, bit 1 = no audio frame
    __shared__ uint64_t bar;
    __shared__ uint32_t size_s[kPktTile];
    __shared__ uint32_t pair_s[kPktTile];               // packet p -> its [bridge-frame][law] entry; bit 31 = PT 123
    const size_t npkts = (size_t)d.F * d.C;
    const size_t first = (size_t)blockIdx.x * kPktTile;
    const uint32_t np = (uint32_t)min((size_t)kPktTile, npkts - first);
    const size_t bf0 = first / (uint32_t)G;
    const uint32_t nbf = (uint32_t)((first + np - 1) / (uint32_t)G - bf0) + 1;
    const bool sc = (d.flags & IGD_F_SIGNED_CHAR) != 0;
    // the run [run0, run1) of console-packet bytes and the window [w0, w1) that stages it
    const size_t run0 = bf0 * IGD_PKT_MAX, run1 = run0 + (size_t)nbf * IGD_PKT_MAX;
    const size_t w0 = run0 & ~(size_t)15;
    const size_t w1 = min((run1 + 15) & ~(size_t)15, (npkts / (uint32_t)G * IGD_PKT_MAX) & ~(size_t)15);
    const uint32_t lead = (uint32_t)(run0 - w0) / 4;
    const uint32_t bar_s = shared_addr(&bar);
    if (threadIdx.x == 0) {
        mbar_init(bar_s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(bar_s, (uint32_t)(w1 - w0));
        bulk_g2s(shared_addr(win_s), rx_pkts + w0, (uint32_t)(w1 - w0), bar_s);
    }
    if (run1 > w1 && threadIdx.x < (uint32_t)(run1 - w1) / 4)      // the array's last words, past its last whole 16 bytes
        win_s[(w1 - w0) / 4 + threadIdx.x] = reinterpret_cast<const uint32_t *>(rx_pkts + w1)[threadIdx.x];
#pragma unroll
    for (int k = 0; k < 4; k++)                          // blockDim.x == 256: thread t maps code t for every law pair
        tab_s[k * 256 + threadIdx.x] = (uint8_t)igd_g711_transcode1(threadIdx.x, k >> 1, k & 1);
    for (uint32_t k = threadIdx.x; k < 2 * nbf; k += blockDim.x) { legs_s[k] = 0ull; bsum_s[k] = 0; }
    __syncthreads();                 // barrier initialised, leg masks cleared
    if (threadIdx.x < np) {
        const uint32_t p = threadIdx.x;
        const size_t i = first + p;
        const igd_tx_plan_rec r = plan[i];
        const uint32_t *hdr = reinterpret_cast<const uint32_t *>(d.rtp12 + i * 12);
        tile_header(img + p * kPktWords, r, hdr[0], hdr[1], hdr[2]);
        size_s[p] = r.size;
        d.sizes[i] = r.size;
        const size_t c = i % (size_t)d.C;                                     // leg b*G + g
        const uint32_t pr = 2u * (uint32_t)(i / (uint32_t)G - bf0) + (law[c] != 0 ? 1u : 0u);   // igd_enc_law_make: 0 = A-law, else u-law
        pair_s[p] = pr | ((r.flags & 1u) << 31);
        atomicOr(&legs_s[pr], 1ull << p);
        if (p < nbf) {               // nbf <= np: the console packet's size and its call's law
            const size_t bf = bf0 + p;
            rsz_s[p] = rx_sizes ? rx_sizes[bf] : (uint32_t)IGD_PKT_MAX;
            bfi_s[p] = in_law[bf % (size_t)((uint32_t)d.C / (uint32_t)G)] != 0 ? 1u : 0u;
        }
    }
    __syncthreads();                 // leg masks, headers and bridge-frame records complete
    for (uint32_t w = threadIdx.x; w < np * kPktWords; w += blockDim.x) {     // zero past each packet (no payload there)
        const uint32_t p = w / kPktWords;
        if (4 * (w - p * kPktWords) >= size_s[p]) img[w] = 0u;
    }
    mbar_wait(bar_s, 0);             // the console packets have landed
    if (threadIdx.x < nbf) {         // transport_rtp_cb's view of the console packet (the navail guard of k_rxarb_bridge)
        const uint32_t k = threadIdx.x, size = rsz_s[k];
        const uint32_t *hw = win_s + lead + k * kPktWords;
        const uint32_t navail = min(size, (uint32_t)IGD_PKT_MAX) / 4;
        const igd_ed137_fields fl = fields_of_header(navail > 0 ? hw[0] : 0u, navail > 3 ? hw[3] : 0u, navail > 4 ? hw[4] : 0u, size);
        const uint4 fw = *reinterpret_cast<const uint4 *>(&fl);
        if (igd_fields_no_audio(fw.y, fw.z, fw.w)) bfi_s[k] |= 2u;
    }
    __syncthreads();                 // no-audio flags complete
    // unit j = (pair, chunk ch): payload words ch, ch + 10, ch + 20, ch + 30, so that neighbouring lanes read and
    // write neighbouring words
    for (uint32_t j = threadIdx.x; j < 2 * nbf * kChunks; j += blockDim.x) {
        const uint32_t pr = j / kChunks, ch = j - pr * kChunks;
        const unsigned long long m = legs_s[pr];
        if (!m) continue;            // no leg of this bridge-frame in the tile uses this law
        const uint32_t info = bfi_s[pr >> 1], o = pr & 1u;
        uint32_t e[4];
        if (info & 2u) {             // silence: the table's entry for u-law 0xFF, which decodes to PCM 0
            const uint32_t s = tab_s[(2u + o) * 256u + 0xFFu] * 0x01010101u;
            e[0] = s; e[1] = s; e[2] = s; e[3] = s;
        } else {
            const uint8_t *tb = tab_s + ((info & 1u) * 2u + o) * 256u;
            const uint32_t *src = win_s + lead + (pr >> 1) * kPktWords + 5 + ch;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t w = src[q * kChunks];
                e[q] = __byte_perm(__byte_perm(tb[w & 0xFFu], tb[(w >> 8) & 0xFFu], 0x0040),
                                   __byte_perm(tb[(w >> 16) & 0xFFu], tb[w >> 24], 0x0040), 0x5410);
            }
        }
        int bs = 0;
        bs = bytesum4(e[0], sc, bs); bs = bytesum4(e[1], sc, bs); bs = bytesum4(e[2], sc, bs); bs = bytesum4(e[3], sc, bs);
        atomicAdd(&bsum_s[pr], bs);
        for (unsigned long long mm = m; mm; mm &= mm - 1) {
            const uint32_t p = (uint32_t)(__ffsll((long long)mm) - 1);
            if (size_s[p] != IGD_PKT_MAX) continue;
            uint32_t *o4 = img + p * kPktWords + 5 + ch;
            o4[0] = e[0]; o4[kChunks] = e[1]; o4[2 * kChunks] = e[2]; o4[3 * kChunks] = e[3];
        }
    }
    const uint32_t whole = 0u;       // the image holds every byte of the tile
    tile_store(d.pkts + first * IGD_PKT_MAX, img, size_s, np, &whole);
    if (threadIdx.x < np && d.bytemean_out) {
        const uint32_t p = threadIdx.x, pr = pair_s[p];
        const bool audio = size_s[p] != 0 && !(pr >> 31);          // setOutgoingRTP (roip_ed137.cpp:6500-6536), clean
        d.bytemean_out[first + p] = audio ? (uint8_t)igd_bytemean_from_sum(bsum_s[pr & 0x7FFFFFFFu], IGD_FRAME) : (uint8_t)0;
    }
}

// ============================================================ recorder sink
__global__ void k_wav_image(const uint8_t *__restrict__ payload, size_t n, int rate, int law, int ref_quirks,
                            uint8_t *__restrict__ out)
{
    const size_t body = ref_quirks ? 2 * n : n, total = 44 + body;
    if (blockIdx.x == 0 && threadIdx.x < 11) {
        const uint32_t channels = ref_quirks ? 2 : 1, bits = ref_quirks ? 16 : 8;
        const uint32_t fmt = ref_quirks ? 7u : (law == IGD_LAW_ALAW ? 6u : 7u);
        const uint32_t align = bits / 8 * channels;
        uint32_t h[11];
        h[0] = 0x46464952u;                      // "RIFF"
        h[1] = (uint32_t)(total - 8);
        h[2] = 0x45564157u;                      // "WAVE"
        h[3] = 0x20746d66u;                      // "fmt "
        h[4] = 16u;
        h[5] = fmt | (channels << 16);
        h[6] = (uint32_t)rate;
        h[7] = (uint32_t)rate * align;
        h[8] = align | (bits << 16);
        h[9] = 0x61746164u;                      // "data"
        h[10] = (uint32_t)body;
        reinterpret_cast<uint32_t *>(out)[threadIdx.x] = h[threadIdx.x];
    }
    uint8_t *dst = out + 44;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (size_t)gridDim.x * blockDim.x) {
        if (ref_quirks) reinterpret_cast<uint16_t *>(dst)[i] = payload[i];   // {b, 0x00}
        else dst[i] = payload[i];
    }
}

// Recorder sink for many calls at once: file image k = the WAV of channel chans[k], gathered from the
// frame-major batch layout codes [F][C][160] (a channel's frames are C*160 bytes apart), written to
// out + k*image_stride.  One warp moves one 160-byte frame (40 words in, 40 or 80 words out).
__global__ void __launch_bounds__(256) k_wav_images(const uint8_t *__restrict__ codes, size_t F, size_t C,
                                                    const uint32_t *__restrict__ chans, size_t nchan,
                                                    const uint8_t *__restrict__ law_ch, int rate, int ref_quirks,
                                                    uint8_t *__restrict__ out, size_t image_stride)
{
    const size_t n = F * IGD_FRAME;
    const size_t body = ref_quirks ? 2 * n : n, total = 44 + body;
    const uint32_t lane = threadIdx.x & 31;
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t u = warp; u < nchan * (F + 1); u += nwarps) {       // unit F of a channel = its header
        const size_t k = u / (F + 1), f = u - k * (F + 1);
        uint32_t ch = chans ? chans[k] : (uint32_t)k;
        if (ch >= C) ch = (uint32_t)(C - 1);             // device-side index list: never read outside the batch
        uint8_t *img = out + k * image_stride;
        if (f == F) {
            if (lane < 11) {
                const uint32_t law = law_ch ? law_ch[ch] : (uint32_t)IGD_LAW_ULAW;
                const uint32_t channels = ref_quirks ? 2 : 1, bits = ref_quirks ? 16 : 8;
                const uint32_t fmt = ref_quirks ? 7u : (law == IGD_LAW_ALAW ? 6u : 7u);
                const uint32_t align = bits / 8 * channels;
                const uint32_t h[11] = {0x46464952u, (uint32_t)(total - 8), 0x45564157u, 0x20746d66u, 16u,
                                        fmt | (channels << 16), (uint32_t)rate, (uint32_t)rate * align,
                                        align | (bits << 16), 0x61746164u, (uint32_t)body};
                reinterpret_cast<uint32_t *>(img)[lane] = h[lane];
            }
            continue;
        }
        const uint32_t *src = reinterpret_cast<const uint32_t *>(codes + (f * C + ch) * IGD_FRAME);
        uint32_t *dst = reinterpret_cast<uint32_t *>(img + 44 + (ref_quirks ? 2 : 1) * f * IGD_FRAME);
        for (uint32_t w = lane; w < IGD_FRAME / 4; w += 32) {
            const uint32_t v = __ldcs(src + w);
            if (ref_quirks) {                                            // every byte b -> {b, 0x00}
                dst[2 * w] = __byte_perm(v, 0u, 0x4140);
                dst[2 * w + 1] = __byte_perm(v, 0u, 0x4342);
            } else {
                dst[w] = v;
            }
        }
    }
}

}  // namespace

// ============================================================ launchers
cudaError_t igd_k_ed137_parse(const igd_launch_cfg &c, const uint8_t *pkts, const uint32_t *sizes,
                              size_t npkts, size_t stride, igd_ed137_fields *fields,
                              uint8_t *payload_out)
{
    if (!payload_out && npkts > 0) {
        k_ed137_fields<<<(unsigned)((npkts + 255) / 256), 256, 0, c.stream>>>(pkts, sizes, npkts, stride, fields);
        return cudaGetLastError();
    }
    const bool al16 = ((reinterpret_cast<uintptr_t>(pkts) | reinterpret_cast<uintptr_t>(payload_out)) & 15) == 0;
    if (stride == IGD_PKT_MAX && al16 && npkts > 0) {
        const size_t tiles = (npkts + kPktTile - 1) / kPktTile;
        k_ed137_parse_tile<<<(unsigned)tiles, 256, 0, c.stream>>>(pkts, sizes, npkts, fields, payload_out);
        return cudaGetLastError();
    }
    k_ed137_parse<<<grid_for(c, npkts * 32, 256, 8), 256, 0, c.stream>>>(pkts, sizes, npkts, stride, fields,
                                                                  payload_out);
    return cudaGetLastError();
}

cudaError_t igd_k_rx_track(const igd_launch_cfg &c, const igd_rx_track_desc &d, const uint8_t *pkts)
{
    const unsigned blocks = (unsigned)((d.C + 127) / 128);
    if (pkts) k_rx_track<3><<<blocks, 128, 0, c.stream>>>(d, pkts);
    else if (d.present) k_rx_track<1><<<blocks, 128, 0, c.stream>>>(d);
    else if (d.sizes) k_rx_track<2><<<blocks, 128, 0, c.stream>>>(d);
    else k_rx_track<0><<<blocks, 128, 0, c.stream>>>(d);
    return cudaGetLastError();
}

cudaError_t igd_k_rxarb_bridge(const igd_launch_cfg &c, const igd_rxarb_args &a)
{
    if (a.B <= 0 || a.F <= 0) return cudaSuccess;
    k_rxarb_bridge<<<(unsigned)((a.B + 63) / 64), 64, 0, c.stream>>>(a);
    return cudaGetLastError();
}

cudaError_t igd_k_gate_arbitrate(const igd_launch_cfg &c, const igd_arb_desc &d)
{
    // bridges per block: 64, or fewer so that the grid is ~4 blocks per SM (the walk over F is sequential)
    const int want_blocks = 4 * (c.sm_count > 0 ? c.sm_count : 148);
    int bpb = (d.B + want_blocks - 1) / want_blocks;
    bpb = bpb < 1 ? 1 : bpb > kArbMaxBpb ? kArbMaxBpb : bpb;
    const unsigned blocks = (unsigned)((d.B + bpb - 1) / bpb);
    const size_t stage = (size_t)kArbStageWords * 7;      // words (4 B) + gains (2 B) + frame flags (1 B)
    switch (d.G) {
    case 1: k_gate_arbitrate<1><<<blocks, kArbThreads, stage, c.stream>>>(d, bpb); break;
    case 2: k_gate_arbitrate<2><<<blocks, kArbThreads, stage, c.stream>>>(d, bpb); break;
    case 4: k_gate_arbitrate<4><<<blocks, kArbThreads, stage, c.stream>>>(d, bpb); break;
    default:   // runtime leg count: leg state + snapshots + last words in shared memory (<= 64 * 32 * 20 B = 40 KB, 64 KB in all)
        {
            const size_t smem = stage + (size_t)bpb * d.G * (sizeof(igd_arb_leg) + 8 + 4);
            cudaError_t e = cudaFuncSetAttribute(k_gate_arbitrate<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            k_gate_arbitrate<0><<<blocks, kArbThreads, smem, c.stream>>>(d, bpb);
        }
    }
    return cudaGetLastError();
}

cudaError_t igd_k_ed137_keepalive(const igd_launch_cfg &c, uint8_t *hdr20, igd_ed137_state *state, size_t C,
                                  long long now, uint32_t *sizes)
{
    k_ed137_keepalive<<<(unsigned)((C + 127) / 128), 128, 0, c.stream>>>(hdr20, state, C, now, sizes);
    return cudaGetLastError();
}

int igd_k_launches_ed137_pack() { return 3; }

cudaError_t igd_k_ed137_pack(const igd_launch_cfg &c, const igd_ed137_pack_desc &d,
                             igd_tx_plan_rec *plan, int32_t *last_src)
{
    cudaError_t e = igd_k_ed137_plan(c, d, plan, last_src);
    if (e != cudaSuccess) return e;
    const bool al16 = ((reinterpret_cast<uintptr_t>(d.payload) | reinterpret_cast<uintptr_t>(d.stale_payload)) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(d.pkts) & 3) == 0;
    if (d.out_stride == IGD_PKT_MAX && d.payload_len == IGD_FRAME && al16) {
        const size_t tiles = ((size_t)d.F * d.C + kPktTile - 1) / kPktTile;
        k_ed137_assemble_tile<<<(unsigned)tiles, 256, 0, c.stream>>>(d, plan);
    } else {
        k_ed137_assemble<<<grid_for(c, (size_t)d.F * d.C * 32, 256, 8), 256, 0, c.stream>>>(d, plan);
    }
    e = cudaGetLastError();
    if (e != cudaSuccess || !d.stale_payload) return e;
    k_ed137_stale_update<<<grid_for(c, (size_t)d.C * 32, 256, 8), 256, 0, c.stream>>>(d, last_src);
    return cudaGetLastError();
}

cudaError_t igd_k_gateway_fanout(const igd_launch_cfg &c, const igd_ed137_pack_desc &d, int G, const int16_t *pcm,
                                 const uint8_t *law, igd_tx_plan_rec *plan, int32_t *last_src)
{
    cudaError_t e = igd_k_ed137_plan(c, d, plan, last_src);
    if (e != cudaSuccess) return e;
    const size_t tiles = ((size_t)d.F * d.C + kPktTile - 1) / kPktTile;
    k_fanout_tile<<<(unsigned)tiles, 256, fanout_tile_bfs(G) * IGD_FRAME * 2, c.stream>>>(d, G, pcm, law, plan);
    return cudaGetLastError();
}

cudaError_t igd_k_gateway_fanout_packets(const igd_launch_cfg &c, const igd_ed137_pack_desc &d, int G,
                                         const uint8_t *rx_pkts, const uint32_t *rx_sizes, const uint8_t *in_law,
                                         const uint8_t *law, igd_tx_plan_rec *plan, int32_t *last_src)
{
    cudaError_t e = igd_k_ed137_plan(c, d, plan, last_src);
    if (e != cudaSuccess) return e;
    const size_t tiles = ((size_t)d.F * d.C + kPktTile - 1) / kPktTile;
    k_fanout_pkt_tile<<<(unsigned)tiles, 256, fanout_pkt_stage_bytes(G), c.stream>>>(d, G, rx_pkts, rx_sizes, in_law, law,
                                                                                    plan);
    return cudaGetLastError();
}

// the sender walk alone (gateway form: the fused kernel assembles the packets)
cudaError_t igd_k_ed137_plan(const igd_launch_cfg &c, const igd_ed137_pack_desc &d, igd_tx_plan_rec *plan, int32_t *last_src)
{
    // a call of several ticks: one warp per sender, tick axis across the lanes (k_plan_walk, igd_walks.cu)
    if (!(d.flags & IGD_F_WALK_SERIAL) && d.F >= IGD_WALK_MIN_TICKS) return igd_k_plan_walk(c, d, plan, last_src);
    k_ed137_plan<<<(d.C + 127) / 128, 128, 0, c.stream>>>(d, plan, last_src);
    return cudaGetLastError();
}

cudaError_t igd_k_wav_images(const igd_launch_cfg &c, const uint8_t *codes, size_t F, size_t C, const uint32_t *chans,
                             size_t nchan, const uint8_t *law_ch, int rate, int ref_quirks, uint8_t *out,
                             size_t image_stride)
{
    k_wav_images<<<grid_for(c, nchan * (F + 1) * 32, 256, 8), 256, 0, c.stream>>>(codes, F, C, chans, nchan, law_ch, rate,
                                                                             ref_quirks, out, image_stride);
    return cudaGetLastError();
}

cudaError_t igd_k_wav_image(const igd_launch_cfg &c, const uint8_t *payload, size_t n, int rate,
                            int law, int ref_quirks, uint8_t *out)
{
    k_wav_image<<<grid_for(c, n + 1, 256, 8), 256, 0, c.stream>>>(payload, n, rate, law, ref_quirks, out);
    return cudaGetLastError();
}
