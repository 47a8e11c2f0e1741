// igd_kernels.cuh -- launch interface between the C ABI (igd_capi.cu) and the
// sm_100a kernels (igd_fused.cu, igd_codec.cu, igd_packet.cu).  All pointers are device pointers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/igate_dsp.h"
#include "igd_math.cuh"      // igd_tx_plan_rec

struct igd_launch_cfg {
    int sm_count;
    cudaStream_t stream;
};


cudaError_t igd_k_g711_decode(const igd_launch_cfg &c, const uint8_t *codes, const uint8_t *law_ch,
                              int law, int16_t *pcm, size_t n, size_t nch);
cudaError_t igd_k_g711_encode(const igd_launch_cfg &c, const int16_t *pcm, const uint8_t *law_ch,
                              int law, uint8_t *codes, size_t n, size_t nch);
cudaError_t igd_k_frame_meter(const igd_launch_cfg &c, const int16_t *pcm, size_t nframes,
                              igd_meter_rec *out);
cudaError_t igd_k_bytemean(const igd_launch_cfg &c, const uint8_t *payloads, size_t n, size_t len,
                           size_t stride, unsigned flags, uint8_t *out);
cudaError_t igd_k_level_percent(const igd_launch_cfg &c, const int32_t *v, size_t n, int32_t *out);
cudaError_t igd_k_mix(const igd_launch_cfg &c, const int16_t *pcm, const uint16_t *gain,
                      size_t nframes, size_t nbridges, int legs, int16_t *mix);
cudaError_t igd_k_fused(const igd_launch_cfg &c, const igd_batch_desc &d);
cudaError_t igd_k_fused_packets(const igd_launch_cfg &c, const igd_packets_desc &d);
cudaError_t igd_k_fused_gateway(const igd_launch_cfg &c, const igd_packets_desc &d, const igd_tx_plan_rec *plan,
                                const uint8_t *tx_rtp12, uint8_t *tx_pkts, uint32_t *tx_sizes);
cudaError_t igd_k_ed137_plan(const igd_launch_cfg &c, const igd_ed137_pack_desc &d, igd_tx_plan_rec *plan, int32_t *last_src);
cudaError_t igd_k_event_summary(const igd_launch_cfg &c, const igd_meter_rec *meter,
                                const uint16_t *gain, size_t F, size_t C, igd_summary_rec *out,
                                igd_summary_db *db);
cudaError_t igd_k_ed137_parse(const igd_launch_cfg &c, const uint8_t *pkts, const uint32_t *sizes,
                              size_t npkts, size_t stride, igd_ed137_fields *fields,
                              uint8_t *payload_out);
cudaError_t igd_k_ed137_pack(const igd_launch_cfg &c, const igd_ed137_pack_desc &d,
                             igd_tx_plan_rec *plan, int32_t *last_src);
// igd_gateway_fanout: the sender walk over d.C = B*G legs (d.payload NULL), then k_fanout_tile encodes pcm [F][B][160]
// into every leg's packet (d.bytemean_out may be NULL); two launches
cudaError_t igd_k_gateway_fanout(const igd_launch_cfg &c, const igd_ed137_pack_desc &d, int G, const int16_t *pcm,
                                 const uint8_t *law, igd_tx_plan_rec *plan, int32_t *last_src);
// igd_gateway_fanout_packets: the same sender walk, then k_fanout_pkt_tile maps the console packets rx_pkts [F][B][180]
// (rx_sizes [F][B] or NULL = all 180, in_law [B]) into every leg's packet; two launches
cudaError_t igd_k_gateway_fanout_packets(const igd_launch_cfg &c, const igd_ed137_pack_desc &d, int G,
                                         const uint8_t *rx_pkts, const uint32_t *rx_sizes, const uint8_t *in_law,
                                         const uint8_t *law, igd_tx_plan_rec *plan, int32_t *last_src);
cudaError_t igd_k_ed137_keepalive(const igd_launch_cfg &c, uint8_t *hdr20, igd_ed137_state *state, size_t C,
                                  long long now, uint32_t *sizes);
// the walks with the tick axis across the lanes of a warp (igd_walks.cuh / igd_walks.cu)
#define IGD_WALK_MIN_TICKS 8       // below this many ticks per call the thread-per-channel kernels run
struct igd_rxarb_args;
cudaError_t igd_k_rxarb_walk(const igd_launch_cfg &c, const igd_rxarb_args &a);
// the same receive side with one thread per bridge (wide, short calls; igd_packet.cu)
cudaError_t igd_k_rxarb_bridge(const igd_launch_cfg &c, const igd_rxarb_args &a);
cudaError_t igd_k_plan_walk(const igd_launch_cfg &c, const igd_ed137_pack_desc &d, igd_tx_plan_rec *plan, int32_t *last_src);
// pkts != NULL: the walk reads the header words straight out of the packets [F][C][180] (d.fields unused)
cudaError_t igd_k_rx_track(const igd_launch_cfg &c, const igd_rx_track_desc &d, const uint8_t *pkts = nullptr);
cudaError_t igd_k_gate_arbitrate(const igd_launch_cfg &c, const igd_arb_desc &d);
cudaError_t igd_k_wav_images(const igd_launch_cfg &c, const uint8_t *codes, size_t F, size_t C, const uint32_t *chans,
                             size_t nchan, const uint8_t *law_ch, int rate, int ref_quirks, uint8_t *out,
                             size_t image_stride);
cudaError_t igd_k_wav_image(const igd_launch_cfg &c, const uint8_t *payload, size_t n, int rate,
                            int law, int ref_quirks, uint8_t *out);

// number of kernel launches each wrapper above performs (for gpu_launches)
int igd_k_launches_ed137_pack();
