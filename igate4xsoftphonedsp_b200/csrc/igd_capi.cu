// igd_capi.cu -- the extern "C" surface declared in include/igate_dsp.h.
//
// Host pointers (IGD_MEM_HOST) are staged through grow-only device scratch
// buffers owned by the context; device pointers (IGD_MEM_DEVICE) are used in
// place.  Every arithmetic entry point launches a CUDA kernel -- there is no
// CPU implementation behind this API.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "igd_kernels.cuh"
#include "igd_walks.cuh"      // igd_rxarb_args
#include "igd_math.cuh"

namespace {
constexpr int kSlots = 13;
}

struct igd_ctx {
    int device;
    cudaStream_t own_stream, stream;
    cudaStream_t copy_streams[2];
    cudaEvent_t ev[8];
    cudaStream_t walk_streams[2];       // igd_gateway_process: liveness walk / arbitration, pipelined against the fused kernel
    cudaEvent_t walk_ev[5 * 8];         // [chunk]: liveness walk done, [8 + chunk]: arbitration done, [16 + chunk]: sender walk done,
                                        // host form: [24 + chunk]: the chunk's inputs are on the device, [32 + chunk]: its outputs are ready
    cudaStream_t io_streams[2];         // igd_gateway_process, host form: chunk-wise H2D / D2H beside the kernels
    cudaDeviceProp prop;
    void *scratch[kSlots];
    size_t scratch_cap[kSlots];
    uint64_t launches;
    char err[256];
};

namespace {

int fail(igd_ctx *c, int code, const char *what, cudaError_t e = cudaSuccess)
{
    if (c) {
        if (e != cudaSuccess)
            snprintf(c->err, sizeof(c->err), "%s: %s", what, cudaGetErrorString(e));
        else
            snprintf(c->err, sizeof(c->err), "%s", what);
    }
    // a CUDA call failed in the middle of a call: nothing of this library may still be copying to or from the
    // caller's host buffers (or the shared scratch) when the error is returned -- drain whatever was queued on the
    // side streams (a sticky error makes this return at once; under stream capture it is refused, harmlessly)
    if (e != cudaSuccess) cudaDeviceSynchronize();
    return code;
}

#define IGD_CUDA(c, call)                                                 \
    do {                                                                  \
        cudaError_t e_ = (call);                                          \
        if (e_ != cudaSuccess) return fail((c), IGD_ECUDA, #call, e_);    \
    } while (0)

struct Bind {
    igd_ctx *c;
    cudaError_t err;
    explicit Bind(igd_ctx *ctx) : c(ctx), err(cudaSetDevice(ctx->device)) {}
};
// binds the calling thread to the context's device; a failure is an error of the call, not ignored
#define IGD_BIND(c)  \
    Bind b(c);       \
    if (b.err != cudaSuccess) return fail((c), IGD_ECUDA, "cudaSetDevice", b.err)

igd_launch_cfg cfg_of(igd_ctx *c)
{
    igd_launch_cfg k;
    k.sm_count = c->prop.multiProcessorCount;
    k.stream = c->stream;
    return k;
}

// grow-only device scratch
int scratch(igd_ctx *c, int slot, size_t bytes, void **out)
{
    if (bytes == 0) bytes = 16;
    if (c->scratch_cap[slot] < bytes) {
        if (c->scratch[slot]) {
            cudaStreamSynchronize(c->stream);
            cudaFree(c->scratch[slot]);
            c->scratch[slot] = nullptr;
            c->scratch_cap[slot] = 0;
        }
        size_t cap = bytes + bytes / 8;
        cap = (cap + 255) & ~(size_t)255;
        cudaError_t e = cudaMalloc(&c->scratch[slot], cap);
        if (e != cudaSuccess) return fail(c, IGD_ENOMEM, "cudaMalloc(scratch)", e);
        c->scratch_cap[slot] = cap;
    }
    *out = c->scratch[slot];
    return IGD_OK;
}

// resolves an input: device pointer as is, host pointer copied into `slot`
template <class T>
int in_arg(igd_ctx *c, int mem, int slot, const T *p, size_t count, const T **out)
{
    if (mem == IGD_MEM_DEVICE) { *out = p; return IGD_OK; }
    void *d = nullptr;
    int rc = scratch(c, slot, count * sizeof(T), &d);
    if (rc) return rc;
    if (count) IGD_CUDA(c, cudaMemcpyAsync(d, p, count * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    *out = static_cast<const T *>(d);
    return IGD_OK;
}
template <class T>
int out_arg(igd_ctx *c, int mem, int slot, T *p, size_t count, T **out)
{
    if (mem == IGD_MEM_DEVICE) { *out = p; return IGD_OK; }
    void *d = nullptr;
    int rc = scratch(c, slot, count * sizeof(T), &d);
    if (rc) return rc;
    *out = static_cast<T *>(d);
    return IGD_OK;
}
template <class T>
int out_done(igd_ctx *c, int mem, T *host, const T *dev, size_t count)
{
    if (mem == IGD_MEM_DEVICE || count == 0) return IGD_OK;
    IGD_CUDA(c, cudaMemcpyAsync(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    return IGD_OK;
}
int finish(igd_ctx *c, int mem)
{
    if (mem == IGD_MEM_HOST) IGD_CUDA(c, cudaStreamSynchronize(c->stream));
    return IGD_OK;
}
bool aligned(const void *p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

}  // namespace

extern "C" {

int igd_abi_version(void) { return IGD_ABI_VERSION; }

int igd_init(int device, igd_ctx **out)
{
    if (!out) return IGD_EINVAL;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return IGD_ENODEV;
    igd_ctx *c = new (std::nothrow) igd_ctx();
    if (!c) return IGD_ENOMEM;
    memset(c, 0, sizeof(*c));
    c->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&c->prop, device) != cudaSuccess) {
        delete c;
        return IGD_ENODEV;
    }
    if (c->prop.major < 10) {   // kernels are built for sm_100a only
        delete c;
        return IGD_ENODEV;
    }
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete c;
        return IGD_ECUDA;
    }
    c->stream = c->own_stream;
    bool ok = true;
    for (auto &s : c->copy_streams) ok = ok && cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess;
    for (auto &e : c->ev) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
    {
        // the walks are small, latency-bound grids: their blocks go ahead of the fused kernel's CTAs when both wait for an SM
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        for (auto &s : c->walk_streams) ok = ok && cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, hi) == cudaSuccess;
        for (auto &e : c->walk_ev) ok = ok && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) == cudaSuccess;
        for (auto &s : c->io_streams) ok = ok && cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess;
    }
    if (!ok) {          // never run with a null copy stream / event
        for (auto &e : c->ev) if (e) cudaEventDestroy(e);
        for (auto &e : c->walk_ev) if (e) cudaEventDestroy(e);
        for (auto &s : c->walk_streams) if (s) cudaStreamDestroy(s);
        for (auto &s : c->io_streams) if (s) cudaStreamDestroy(s);
        for (auto &s : c->copy_streams) if (s) cudaStreamDestroy(s);
        cudaStreamDestroy(c->own_stream);
        delete c;
        return IGD_ECUDA;
    }
    *out = c;
    return IGD_OK;
}

int igd_shutdown(igd_ctx *c)
{
    if (!c) return IGD_EINVAL;
    Bind b(c);
    cudaStreamSynchronize(c->stream);
    for (int i = 0; i < kSlots; i++)
        if (c->scratch[i]) cudaFree(c->scratch[i]);
    for (auto &e : c->ev) cudaEventDestroy(e);
    for (auto &e : c->walk_ev) cudaEventDestroy(e);
    for (auto &s : c->walk_streams) cudaStreamDestroy(s);
    for (auto &s : c->io_streams) cudaStreamDestroy(s);
    for (auto &s : c->copy_streams) cudaStreamDestroy(s);
    cudaStreamDestroy(c->own_stream);
    delete c;
    return IGD_OK;
}

int igd_set_stream(igd_ctx *c, void *s)
{
    if (!c) return IGD_EINVAL;
    c->stream = static_cast<cudaStream_t>(s);
    return IGD_OK;
}

int igd_use_own_stream(igd_ctx *c)
{
    if (!c) return IGD_EINVAL;
    c->stream = c->own_stream;
    return IGD_OK;
}

int igd_sync(igd_ctx *c)
{
    if (!c) return IGD_EINVAL;
    IGD_BIND(c);
    IGD_CUDA(c, cudaStreamSynchronize(c->stream));
    return IGD_OK;
}

const char *igd_last_error(igd_ctx *c) { return c ? c->err : "null context"; }

int igd_device_info(igd_ctx *c, igd_devinfo *o)
{
    if (!c || !o) return IGD_EINVAL;
    o->device = c->device;
    o->sm_count = c->prop.multiProcessorCount;
    o->cc_major = c->prop.major;
    o->cc_minor = c->prop.minor;
    o->total_mem = c->prop.totalGlobalMem;
    strncpy(o->name, c->prop.name, sizeof(o->name) - 1);
    o->name[sizeof(o->name) - 1] = 0;
    return IGD_OK;
}

uint64_t igd_launch_count(igd_ctx *c) { return c ? c->launches : 0; }

void *igd_host_alloc(size_t bytes)
{
    void *p = nullptr;
    return cudaMallocHost(&p, bytes ? bytes : 1) == cudaSuccess ? p : nullptr;
}
void igd_host_free(void *p) { if (p) cudaFreeHost(p); }

void *igd_dev_alloc(igd_ctx *c, size_t bytes)
{
    if (!c) return nullptr;
    Bind b(c);
    void *p = nullptr;
    return cudaMalloc(&p, bytes ? bytes : 1) == cudaSuccess ? p : nullptr;
}
void igd_dev_free(igd_ctx *c, void *p)
{
    if (!c || !p) return;
    Bind b(c);
    cudaFree(p);
}
int igd_copy_to_device(igd_ctx *c, void *dst, const void *src, size_t bytes)
{
    if (!c) return IGD_EINVAL;
    IGD_BIND(c);
    IGD_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    IGD_CUDA(c, cudaStreamSynchronize(c->stream));
    return IGD_OK;
}
int igd_copy_to_host(igd_ctx *c, void *dst, const void *src, size_t bytes)
{
    if (!c) return IGD_EINVAL;
    IGD_BIND(c);
    IGD_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    IGD_CUDA(c, cudaStreamSynchronize(c->stream));
    return IGD_OK;
}

// ---------------------------------------------------------------- G.711
static int g711_decode_impl(igd_ctx *c, const uint8_t *codes, const uint8_t *law_ch, int law,
                            int16_t *pcm, size_t n, size_t nch, int mem)
{
    if (!c || (n && (!codes || !pcm)) || (law != IGD_LAW_ALAW && law != IGD_LAW_ULAW))
        return fail(c, IGD_EINVAL, "igd_g711_decode: bad argument");
    if (n == 0) return IGD_OK;
    if (mem == IGD_MEM_DEVICE && (!aligned(codes, 16) || !aligned(pcm, 32)))
        return fail(c, IGD_EINVAL, "igd_g711_decode: device pointers must be 16/32-byte aligned");
    IGD_BIND(c);
    const uint8_t *dc; const uint8_t *dl = nullptr; int16_t *dp;
    int rc;
    if ((rc = in_arg(c, mem, 0, codes, n, &dc))) return rc;
    if (law_ch && (rc = in_arg(c, mem, 1, law_ch, nch, &dl))) return rc;
    if ((rc = out_arg(c, mem, 2, pcm, n, &dp))) return rc;
    IGD_CUDA(c, igd_k_g711_decode(cfg_of(c), dc, dl, law, dp, n, nch));
    c->launches++;
    if ((rc = out_done(c, mem, pcm, dp, n))) return rc;
    return finish(c, mem);
}

int igd_g711_decode(igd_ctx *c, const uint8_t *codes, int16_t *pcm, size_t n, int law, int mem)
{
    return g711_decode_impl(c, codes, nullptr, law, pcm, n, 1, mem);
}
int igd_g711_decode_ch(igd_ctx *c, const uint8_t *codes, const uint8_t *law, int16_t *pcm,
                       size_t nframes, size_t nch, int mem)
{
    if (!law || nch == 0) return fail(c, IGD_EINVAL, "igd_g711_decode_ch: bad argument");
    return g711_decode_impl(c, codes, law, 0, pcm, nframes * nch * IGD_FRAME, nch, mem);
}

static int g711_encode_impl(igd_ctx *c, const int16_t *pcm, const uint8_t *law_ch, int law,
                            uint8_t *codes, size_t n, size_t nch, int mem)
{
    if (!c || (n && (!codes || !pcm)) || (law != IGD_LAW_ALAW && law != IGD_LAW_ULAW))
        return fail(c, IGD_EINVAL, "igd_g711_encode: bad argument");
    if (n == 0) return IGD_OK;
    if (mem == IGD_MEM_DEVICE && (!aligned(codes, 16) || !aligned(pcm, 32)))
        return fail(c, IGD_EINVAL, "igd_g711_encode: device pointers must be 16/32-byte aligned");
    IGD_BIND(c);
    const int16_t *dp; const uint8_t *dl = nullptr; uint8_t *dc;
    int rc;
    if ((rc = in_arg(c, mem, 0, pcm, n, &dp))) return rc;
    if (law_ch && (rc = in_arg(c, mem, 1, law_ch, nch, &dl))) return rc;
    if ((rc = out_arg(c, mem, 2, codes, n, &dc))) return rc;
    IGD_CUDA(c, igd_k_g711_encode(cfg_of(c), dp, dl, law, dc, n, nch));
    c->launches++;
    if ((rc = out_done(c, mem, codes, dc, n))) return rc;
    return finish(c, mem);
}

int igd_g711_encode(igd_ctx *c, const int16_t *pcm, uint8_t *codes, size_t n, int law, int mem)
{
    return g711_encode_impl(c, pcm, nullptr, law, codes, n, 1, mem);
}
int igd_g711_encode_ch(igd_ctx *c, const int16_t *pcm, const uint8_t *law, uint8_t *codes,
                       size_t nframes, size_t nch, int mem)
{
    if (!law || nch == 0) return fail(c, IGD_EINVAL, "igd_g711_encode_ch: bad argument");
    return g711_encode_impl(c, pcm, law, 0, codes, nframes * nch * IGD_FRAME, nch, mem);
}

// ---------------------------------------------------------------- meters
int igd_frame_meter(igd_ctx *c, const int16_t *pcm, size_t nframes, igd_meter_rec *out, int mem)
{
    if (!c || (nframes && (!pcm || !out))) return fail(c, IGD_EINVAL, "igd_frame_meter: bad argument");
    if (nframes == 0) return IGD_OK;
    if (mem == IGD_MEM_DEVICE && (!aligned(pcm, 32) || !aligned(out, 16)))
        return fail(c, IGD_EINVAL, "igd_frame_meter: device pointers must be 32/16-byte aligned");
    IGD_BIND(c);
    const int16_t *dp; igd_meter_rec *dout;
    int rc;
    if ((rc = in_arg(c, mem, 0, pcm, nframes * IGD_FRAME, &dp))) return rc;
    if ((rc = out_arg(c, mem, 2, out, nframes, &dout))) return rc;
    IGD_CUDA(c, igd_k_frame_meter(cfg_of(c), dp, nframes, dout));
    c->launches++;
    if ((rc = out_done(c, mem, out, dout, nframes))) return rc;
    return finish(c, mem);
}

int igd_bytemean(igd_ctx *c, const uint8_t *payloads, size_t n, size_t len, size_t stride,
                 unsigned flags, uint8_t *out, int mem)
{
    if (!c || (n && (!payloads || !out)) || stride < len) return fail(c, IGD_EINVAL, "igd_bytemean: bad argument");
    if (n == 0) return IGD_OK;
    IGD_BIND(c);
    const uint8_t *dp; uint8_t *dout;
    int rc;
    if ((rc = in_arg(c, mem, 0, payloads, (n - 1) * stride + len, &dp))) return rc;
    if ((rc = out_arg(c, mem, 2, out, n, &dout))) return rc;
    IGD_CUDA(c, igd_k_bytemean(cfg_of(c), dp, n, len, stride, flags, dout));
    c->launches++;
    if ((rc = out_done(c, mem, out, dout, n))) return rc;
    return finish(c, mem);
}

int igd_level_percent(igd_ctx *c, const int32_t *v, size_t n, int32_t *out, int mem)
{
    if (!c || (n && (!v || !out))) return fail(c, IGD_EINVAL, "igd_level_percent: bad argument");
    if (n == 0) return IGD_OK;
    IGD_BIND(c);
    const int32_t *dv; int32_t *dout;
    int rc;
    if ((rc = in_arg(c, mem, 0, v, n, &dv))) return rc;
    if ((rc = out_arg(c, mem, 2, out, n, &dout))) return rc;
    IGD_CUDA(c, igd_k_level_percent(cfg_of(c), dv, n, dout));
    c->launches++;
    if ((rc = out_done(c, mem, out, dout, n))) return rc;
    return finish(c, mem);
}

// ---------------------------------------------------------------- gain / mix
int igd_gain_q7(float level)
{
    // pjsua_conf_adjust_rx_level(slot, level) as called at roip_ed137.cpp:5221
    return (int)((level - 1.0f) * 128) + 128;
}

int igd_mix(igd_ctx *c, const int16_t *pcm, const uint16_t *gain, size_t F, size_t B, int G,
            int16_t *mix, int mem)
{
    if (!c || G < 1 || G > IGD_MAX_LEGS || (F && B && (!pcm || !gain || !mix)))
        return fail(c, IGD_EINVAL, "igd_mix: bad argument");
    if (F == 0 || B == 0) return IGD_OK;
    if (mem == IGD_MEM_DEVICE && (!aligned(pcm, 16) || !aligned(mix, 16)))
        return fail(c, IGD_EINVAL, "igd_mix: device pointers must be 16-byte aligned");
    IGD_BIND(c);
    const int16_t *dp; const uint16_t *dg; int16_t *dm;
    int rc;
    if ((rc = in_arg(c, mem, 0, pcm, F * B * G * IGD_FRAME, &dp))) return rc;
    if ((rc = in_arg(c, mem, 1, gain, F * B * G, &dg))) return rc;
    if ((rc = out_arg(c, mem, 2, mix, F * B * IGD_FRAME, &dm))) return rc;
    IGD_CUDA(c, igd_k_mix(cfg_of(c), dp, dg, F, B, G, dm));
    c->launches++;
    if ((rc = out_done(c, mem, mix, dm, F * B * IGD_FRAME))) return rc;
    return finish(c, mem);
}

// ---------------------------------------------------------------- fused path
namespace {

// One description of both entry points: codes (160 B per leg-frame) or raw packets (180 B + a 16-byte
// field record per leg-frame) in; any subset of {mix, enc, meter, bmeter} out.
struct FusedJob {
    bool packets;
    size_t F, B, G;
    unsigned flags;
    const uint8_t *in;                 // codes or pkts
    const igd_ed137_fields *fields;    // packets only
    const uint8_t *law, *out_law;
    const uint16_t *gain;
    int16_t *mix;
    uint8_t *enc;
    igd_meter_rec *meter;
    igd_bridge_rec *bmeter;
};

cudaError_t launch_fused_job(igd_ctx *c, const FusedJob &j, size_t nf, const uint8_t *in, const igd_ed137_fields *fields,
                             const uint8_t *law, const uint16_t *gain, const uint8_t *out_law, int16_t *mix,
                             uint8_t *enc, igd_meter_rec *meter, igd_bridge_rec *bmeter)
{
    if (j.packets) {
        igd_packets_desc k;
        memset(&k, 0, sizeof k);
        k.struct_size = sizeof k; k.mem = IGD_MEM_DEVICE; k.F = (int32_t)nf; k.B = (int32_t)j.B; k.G = (int32_t)j.G;
        k.flags = j.flags; k.pkts = in; k.fields = fields; k.law = law; k.gain_q7 = gain; k.out_law = out_law;
        k.mix = mix; k.enc = enc; k.meter = meter; k.bmeter = bmeter;
        return igd_k_fused_packets(cfg_of(c), k);
    }
    igd_batch_desc k;
    memset(&k, 0, sizeof k);
    k.struct_size = sizeof k; k.mem = IGD_MEM_DEVICE; k.F = (int32_t)nf; k.B = (int32_t)j.B; k.G = (int32_t)j.G;
    k.flags = j.flags; k.codes = in; k.law = law; k.gain_q7 = gain; k.out_law = out_law;
    k.mix = mix; k.enc = enc; k.meter = meter; k.bmeter = bmeter;
    return igd_k_fused(cfg_of(c), k);
}

// Host buffers: staged through the GPU in frame chunks so that the H2D copy of chunk k+1, the kernel of
// chunk k and the D2H copy of chunk k-1 overlap (three streams, two buffers).  Only the outputs the caller
// asked for are copied back -- the int16 mix alone is 57 % of the full result set.
int fused_job_host(igd_ctx *c, const FusedJob &j)
{
    const size_t F = j.F, B = j.B, C = j.B * j.G;
    const size_t leg_bytes = j.packets ? (size_t)IGD_PKT_MAX : (size_t)IGD_FRAME;
    int rc;
    const uint8_t *dlaw, *dol;
    if ((rc = in_arg(c, IGD_MEM_HOST, 0, j.law, C, &dlaw))) return rc;
    if ((rc = in_arg(c, IGD_MEM_HOST, 1, j.out_law, B, &dol))) return rc;
    // chunk size: ~32 MiB of input per chunk, at least 1 frame
    // (measured on B200 / PCIe gen5: 4 / 8 / 16 / 32 / 64 MiB -> 3.2 / 4.0 / 4.6 / 4.8 / 4.8e10 channel-samples/s)
    size_t fc = (32u << 20) / (C * leg_bytes);
    if (fc < 1) fc = 1;
    if (fc > F) fc = F;
    const size_t nchunks = (F + fc - 1) / fc;
    const int nbuf = nchunks > 1 ? 2 : 1;
    void *din, *dgain, *dfields = nullptr, *dmix = nullptr, *denc = nullptr, *dmeter = nullptr, *dbm = nullptr;
    if ((rc = scratch(c, 2, nbuf * fc * C * leg_bytes, &din))) return rc;
    if ((rc = scratch(c, 3, nbuf * fc * C * sizeof(uint16_t), &dgain))) return rc;
    if (j.packets && (rc = scratch(c, 8, nbuf * fc * C * sizeof(igd_ed137_fields), &dfields))) return rc;
    if (j.mix && (rc = scratch(c, 4, nbuf * fc * B * IGD_FRAME * sizeof(int16_t), &dmix))) return rc;
    if (j.enc && (rc = scratch(c, 5, nbuf * fc * B * IGD_FRAME, &denc))) return rc;
    if (j.meter && (rc = scratch(c, 6, nbuf * fc * C * sizeof(igd_meter_rec), &dmeter))) return rc;
    if (j.bmeter && (rc = scratch(c, 7, nbuf * fc * B * sizeof(igd_bridge_rec), &dbm))) return rc;
    cudaStream_t sin = c->copy_streams[0], sout = c->copy_streams[1];
    // ev[0..1]: input of buffer i ready; ev[2..3]: kernel on buffer i done; ev[4..5]: output drained; ev[6]: fork.
    // The copy-in stream starts after the work already queued on the caller's stream: the device form of another call
    // may still be reading slots 2, 3 or 8 there (igd_gateway_process keeps its gains in slot 8, the fan-outs their
    // sender plan), and scratch() only synchronizes when a slot grows.
    IGD_CUDA(c, cudaEventRecord(c->ev[6], c->stream));
    IGD_CUDA(c, cudaStreamWaitEvent(sin, c->ev[6], 0));
    bool out_pending[2] = {false, false};
    auto chunk = [&](size_t ch) -> int {
        const int i = (int)(ch % nbuf);
        const size_t f0 = ch * fc, nf = (f0 + fc <= F) ? fc : F - f0;
        uint8_t *bi = static_cast<uint8_t *>(din) + (size_t)i * fc * C * leg_bytes;
        uint16_t *bg = static_cast<uint16_t *>(dgain) + (size_t)i * fc * C;
        igd_ed137_fields *bf = j.packets ? static_cast<igd_ed137_fields *>(dfields) + (size_t)i * fc * C : nullptr;
        int16_t *bm = j.mix ? static_cast<int16_t *>(dmix) + (size_t)i * fc * B * IGD_FRAME : nullptr;
        uint8_t *be = j.enc ? static_cast<uint8_t *>(denc) + (size_t)i * fc * B * IGD_FRAME : nullptr;
        igd_meter_rec *bmt = j.meter ? static_cast<igd_meter_rec *>(dmeter) + (size_t)i * fc * C : nullptr;
        igd_bridge_rec *bbr = j.bmeter ? static_cast<igd_bridge_rec *>(dbm) + (size_t)i * fc * B : nullptr;
        // the input buffer may only be overwritten once the kernel that read it is done
        if (ch >= (size_t)nbuf) IGD_CUDA(c, cudaStreamWaitEvent(sin, c->ev[2 + i], 0));
        IGD_CUDA(c, cudaMemcpyAsync(bi, j.in + f0 * C * leg_bytes, nf * C * leg_bytes, cudaMemcpyHostToDevice, sin));
        IGD_CUDA(c, cudaMemcpyAsync(bg, j.gain + f0 * C, nf * C * sizeof(uint16_t), cudaMemcpyHostToDevice, sin));
        if (j.packets)
            IGD_CUDA(c, cudaMemcpyAsync(bf, j.fields + f0 * C, nf * C * sizeof(igd_ed137_fields), cudaMemcpyHostToDevice, sin));
        IGD_CUDA(c, cudaEventRecord(c->ev[i], sin));
        IGD_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev[i], 0));
        // the output buffer may only be overwritten once its previous D2H is done
        if (out_pending[i]) IGD_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev[4 + i], 0));
        IGD_CUDA(c, launch_fused_job(c, j, nf, bi, bf, dlaw, bg, dol, bm, be, bmt, bbr));
        c->launches++;
        IGD_CUDA(c, cudaEventRecord(c->ev[2 + i], c->stream));
        IGD_CUDA(c, cudaStreamWaitEvent(sout, c->ev[2 + i], 0));
        if (j.mix)
            IGD_CUDA(c, cudaMemcpyAsync(j.mix + f0 * B * IGD_FRAME, bm, nf * B * IGD_FRAME * sizeof(int16_t), cudaMemcpyDeviceToHost, sout));
        if (j.enc)
            IGD_CUDA(c, cudaMemcpyAsync(j.enc + f0 * B * IGD_FRAME, be, nf * B * IGD_FRAME, cudaMemcpyDeviceToHost, sout));
        if (j.meter)
            IGD_CUDA(c, cudaMemcpyAsync(j.meter + f0 * C, bmt, nf * C * sizeof(igd_meter_rec), cudaMemcpyDeviceToHost, sout));
        if (j.bmeter)
            IGD_CUDA(c, cudaMemcpyAsync(j.bmeter + f0 * B, bbr, nf * B * sizeof(igd_bridge_rec), cudaMemcpyDeviceToHost, sout));
        IGD_CUDA(c, cudaEventRecord(c->ev[4 + i], sout));
        out_pending[i] = true;
        return IGD_OK;
    };
    rc = IGD_OK;
    for (size_t ch = 0; ch < nchunks && rc == IGD_OK; ch++) rc = chunk(ch);
    // also on an error: nothing may still be copying from / into the caller's buffers or the scratch when we return
    const cudaError_t e0 = cudaStreamSynchronize(sin), e1 = cudaStreamSynchronize(sout), e2 = cudaStreamSynchronize(c->stream);
    if (rc != IGD_OK) return rc;
    if (e0 != cudaSuccess) return fail(c, IGD_ECUDA, "cudaStreamSynchronize(copy in)", e0);
    if (e1 != cudaSuccess) return fail(c, IGD_ECUDA, "cudaStreamSynchronize(copy out)", e1);
    if (e2 != cudaSuccess) return fail(c, IGD_ECUDA, "cudaStreamSynchronize", e2);
    return IGD_OK;
}

}  // namespace

int igd_process_batch(igd_ctx *c, const igd_batch_desc *d)
{
    if (!c || !d || d->struct_size != sizeof(igd_batch_desc))
        return fail(c, IGD_EINVAL, "igd_process_batch: bad descriptor");
    if (d->F < 0 || d->B < 0 || d->G < 1 || d->G > IGD_MAX_LEGS)
        return fail(c, IGD_EINVAL, "igd_process_batch: bad shape");
    if (d->F == 0 || d->B == 0) return IGD_OK;
    if (!d->codes || !d->law || !d->gain_q7 || !d->out_law)
        return fail(c, IGD_EINVAL, "igd_process_batch: null input buffer");
    if (!d->mix && !d->enc && !d->meter && !d->bmeter)
        return fail(c, IGD_EINVAL, "igd_process_batch: no output requested (mix, enc, meter, bmeter are all NULL)");
    IGD_BIND(c);
    if (d->mem == IGD_MEM_DEVICE) {
        if (!aligned(d->codes, 16) || !aligned(d->mix, 32) || !aligned(d->enc, 16) || !aligned(d->meter, 16) ||
            !aligned(d->gain_q7, 2) || !aligned(d->bmeter, 4))
            return fail(c, IGD_EINVAL, "igd_process_batch: misaligned device pointer");
        IGD_CUDA(c, igd_k_fused(cfg_of(c), *d));
        c->launches++;
        return IGD_OK;
    }
    FusedJob j;
    j.packets = false; j.F = d->F; j.B = d->B; j.G = d->G; j.flags = d->flags;
    j.in = d->codes; j.fields = nullptr; j.law = d->law; j.out_law = d->out_law; j.gain = d->gain_q7;
    j.mix = d->mix; j.enc = d->enc; j.meter = d->meter; j.bmeter = d->bmeter;
    return fused_job_host(c, j);
}

// packets form for leg counts other than 4: the payloads are extracted into the context's scratch (k_ed137_parse
// writes codes = payload bytes, zero past payload_len), legs whose packet is not a whole audio frame get
// IGD_GAIN_NO_AUDIO, and the codes-form kernels (k_fused_w for G <= 4, k_fused_g up to 32 legs) run on that.
// Same results as the G = 4 packet kernel's rule; one extra pass over the packets.
__global__ void __launch_bounds__(256) k_mark_no_audio(const igd_ed137_fields *__restrict__ fields, const uint16_t *__restrict__ gain,
                                                       uint16_t *__restrict__ out, size_t n)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t *fw = reinterpret_cast<const uint32_t *>(fields + i);
    uint16_t g = gain[i];
    if (igd_fields_no_audio(__ldg(fw + 1), __ldg(fw + 2), __ldg(fw + 3))) g |= (uint16_t)IGD_GAIN_NO_AUDIO;
    out[i] = g;
}

static int process_packets_any_g(igd_ctx *c, const igd_packets_desc *d)
{
    const size_t F = d->F, B = d->B, G = d->G, C = B * G, n = F * C;
    const int mem = d->mem;
    int rc;
    const uint8_t *dpk, *dlaw, *dol; const igd_ed137_fields *dfl; const uint16_t *dg;
    if ((rc = in_arg(c, mem, 0, d->pkts, n * IGD_PKT_MAX, &dpk))) return rc;
    if ((rc = in_arg(c, mem, 1, d->fields, n, &dfl))) return rc;
    if ((rc = in_arg(c, mem, 2, d->law, C, &dlaw))) return rc;
    if ((rc = in_arg(c, mem, 3, d->gain_q7, n, &dg))) return rc;
    if ((rc = in_arg(c, mem, 4, d->out_law, B, &dol))) return rc;
    void *dcodes, *dgain2, *dfl2;
    if ((rc = scratch(c, 9, n * IGD_FRAME, &dcodes))) return rc;
    if ((rc = scratch(c, 10, n * sizeof(uint16_t), &dgain2))) return rc;
    if ((rc = scratch(c, 11, n * sizeof(igd_ed137_fields), &dfl2))) return rc;
    // the extraction copies bytes 20..179 of every slot; slots that do not hold a whole audio frame are flagged
    // IGD_GAIN_NO_AUDIO below (from the caller's field records), so what was copied for them is never interpreted
    igd_batch_desc k;
    memset(&k, 0, sizeof k);
    k.struct_size = sizeof k; k.mem = IGD_MEM_DEVICE; k.F = d->F; k.B = d->B; k.G = d->G; k.flags = d->flags;
    k.codes = static_cast<const uint8_t *>(dcodes); k.law = dlaw; k.gain_q7 = static_cast<const uint16_t *>(dgain2); k.out_law = dol;
    if ((rc = out_arg(c, mem, 5, d->mix, d->mix ? F * B * IGD_FRAME : 0, &k.mix))) return rc;
    if ((rc = out_arg(c, mem, 6, d->enc, d->enc ? F * B * IGD_FRAME : 0, &k.enc))) return rc;
    if ((rc = out_arg(c, mem, 7, d->meter, d->meter ? n : 0, &k.meter))) return rc;
    if ((rc = out_arg(c, mem, 8, d->bmeter, d->bmeter ? F * B : 0, &k.bmeter))) return rc;
    if (mem == IGD_MEM_HOST) { if (!d->mix) k.mix = nullptr; if (!d->enc) k.enc = nullptr; if (!d->meter) k.meter = nullptr; if (!d->bmeter) k.bmeter = nullptr; }
    IGD_CUDA(c, igd_k_ed137_parse(cfg_of(c), dpk, nullptr, n, IGD_PKT_MAX, static_cast<igd_ed137_fields *>(dfl2), static_cast<uint8_t *>(dcodes)));
    k_mark_no_audio<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(dfl, dg, static_cast<uint16_t *>(dgain2), n);
    IGD_CUDA(c, cudaGetLastError());
    IGD_CUDA(c, igd_k_fused(cfg_of(c), k));
    c->launches += 3;
    if (d->mix && (rc = out_done(c, mem, d->mix, k.mix, F * B * IGD_FRAME))) return rc;
    if (d->enc && (rc = out_done(c, mem, d->enc, k.enc, F * B * IGD_FRAME))) return rc;
    if (d->meter && (rc = out_done(c, mem, d->meter, k.meter, n))) return rc;
    if (d->bmeter && (rc = out_done(c, mem, d->bmeter, k.bmeter, F * B))) return rc;
    return finish(c, mem);
}

int igd_process_packets(igd_ctx *c, const igd_packets_desc *d)
{
    if (!c || !d || d->struct_size != sizeof(igd_packets_desc))
        return fail(c, IGD_EINVAL, "igd_process_packets: bad descriptor");
    if (d->F < 0 || d->B < 0 || d->G < 1 || d->G > IGD_MAX_LEGS) return fail(c, IGD_EINVAL, "igd_process_packets: bad shape");
    if (d->F == 0 || d->B == 0) return IGD_OK;
    if (!d->pkts || !d->fields || !d->law || !d->gain_q7 || !d->out_law)
        return fail(c, IGD_EINVAL, "igd_process_packets: null input buffer");
    if (!d->mix && !d->enc && !d->meter && !d->bmeter)
        return fail(c, IGD_EINVAL, "igd_process_packets: no output requested (mix, enc, meter, bmeter are all NULL)");
    IGD_BIND(c);
    if (d->mem == IGD_MEM_DEVICE &&
        (!aligned(d->pkts, 16) || !aligned(d->fields, 16) || !aligned(d->mix, 32) || !aligned(d->enc, 16) ||
         !aligned(d->meter, 16) || !aligned(d->gain_q7, d->G == 4 ? 8 : 2) || !aligned(d->law, d->G == 4 ? 4 : 1) || !aligned(d->bmeter, 4)))
        return fail(c, IGD_EINVAL, "igd_process_packets: misaligned device pointer");
    if (d->G != 4) return process_packets_any_g(c, d);
    if (d->mem == IGD_MEM_DEVICE) {
        IGD_CUDA(c, igd_k_fused_packets(cfg_of(c), *d));
        c->launches++;
        return IGD_OK;
    }
    FusedJob j;
    j.packets = true; j.F = d->F; j.B = d->B; j.G = d->G; j.flags = d->flags;
    j.in = d->pkts; j.fields = d->fields; j.law = d->law; j.out_law = d->out_law; j.gain = d->gain_q7;
    j.mix = d->mix; j.enc = d->enc; j.meter = d->meter; j.bmeter = d->bmeter;
    return fused_job_host(c, j);
}

// ---------------------------------------------------------------- summary
int igd_event_summary(igd_ctx *c, const igd_meter_rec *meter, const uint16_t *gain, size_t F, size_t C,
                      igd_summary_rec *out, igd_summary_db *db, int mem)
{
    if (!c || (C && (!out || (F && (!meter || !gain))))) return fail(c, IGD_EINVAL, "igd_event_summary: bad argument");
    if (C == 0) return IGD_OK;
    IGD_BIND(c);
    const igd_meter_rec *dm; const uint16_t *dg; igd_summary_rec *dout; igd_summary_db *ddb = nullptr;
    int rc;
    if ((rc = in_arg(c, mem, 0, meter, F * C, &dm))) return rc;
    if ((rc = in_arg(c, mem, 1, gain, F * C, &dg))) return rc;
    if ((rc = out_arg(c, mem, 2, out, C, &dout))) return rc;
    if (db && (rc = out_arg(c, mem, 3, db, C, &ddb))) return rc;
    IGD_CUDA(c, igd_k_event_summary(cfg_of(c), dm, dg, F, C, dout, ddb));
    c->launches++;
    if ((rc = out_done(c, mem, out, dout, C))) return rc;
    if (db && (rc = out_done(c, mem, db, ddb, C))) return rc;
    return finish(c, mem);
}

// ---------------------------------------------------------------- ED-137
unsigned igd_calltype_flags(const char *ct)
{
    // QString(calltype).contains(...) / == "Rx"  (TransportAdapter.cpp:675,801,821,826,830)
    unsigned f = 0;
    if (!ct) return 0;
    if (strstr(ct, "Idle")) f |= IGD_CT_IDLE;
    if (strstr(ct, "Rxonly") || strcmp(ct, "Rx") == 0) f |= IGD_CT_RXONLY;
    if (strstr(ct, "Tx") || strstr(ct, "TRx")) f |= IGD_CT_TXISH;
    return f;
}

void igd_ed137_state_init(igd_ed137_state *s, int radiocall, int callIn, const char *calltype,
                          int keepAlivePeroid, int64_t now_ms)
{
    // pjmedia_custom_tp_adapter_create, TransportAdapter.cpp:97-128
    memset(s, 0, sizeof(*s));
    s->radiostatus = radiocall != 0;
    s->callIn = callIn != 0;
    s->calltype_flags = (uint8_t)igd_calltype_flags(calltype);
    s->keepAlivePeroid = keepAlivePeroid;
    s->r2sSendtime = now_ms;
    s->firstR2SPacket = 1;
}

int igd_ed137_parse(igd_ctx *c, const uint8_t *pkts, const uint32_t *sizes, size_t npkts, size_t stride,
                    igd_ed137_fields *fields, uint8_t *payload_out, int mem)
{
    if (!c || (npkts && (!pkts || !fields)) || stride < IGD_PKT_HDR || (stride & 3))
        return fail(c, IGD_EINVAL, "igd_ed137_parse: bad argument (stride must be >= 20 and a multiple of 4)");
    if (npkts == 0) return IGD_OK;
    if (mem == IGD_MEM_DEVICE && (!aligned(pkts, 4) || !aligned(fields, 16) || (payload_out && !aligned(payload_out, 4))))
        return fail(c, IGD_EINVAL, "igd_ed137_parse: misaligned device pointer");
    IGD_BIND(c);
    const uint8_t *dp; const uint32_t *ds = nullptr; igd_ed137_fields *df; uint8_t *dpo = nullptr;
    int rc;
    if ((rc = in_arg(c, mem, 0, pkts, npkts * stride, &dp))) return rc;
    if (sizes && (rc = in_arg(c, mem, 1, sizes, npkts, &ds))) return rc;
    if ((rc = out_arg(c, mem, 2, fields, npkts, &df))) return rc;
    if (payload_out && (rc = out_arg(c, mem, 3, payload_out, npkts * IGD_FRAME, &dpo))) return rc;
    IGD_CUDA(c, igd_k_ed137_parse(cfg_of(c), dp, ds, npkts, stride, df, dpo));
    c->launches++;
    if ((rc = out_done(c, mem, fields, df, npkts))) return rc;
    if (payload_out && (rc = out_done(c, mem, payload_out, dpo, npkts * IGD_FRAME))) return rc;
    return finish(c, mem);
}

int igd_ed137_pack(igd_ctx *c, const igd_ed137_pack_desc *d)
{
    if (!c || !d || d->struct_size != sizeof(igd_ed137_pack_desc))
        return fail(c, IGD_EINVAL, "igd_ed137_pack: bad descriptor");
    if (d->F < 0 || d->C < 0 || d->payload_len == 0 || d->payload_len > IGD_FRAME || (d->payload_len & 3) ||
        d->out_stride < IGD_PKT_HDR + d->payload_len || (d->out_stride & 3))
        return fail(c, IGD_EINVAL, "igd_ed137_pack: bad shape (payload_len in 4..160 and out_stride must be multiples of 4)");
    if (d->F == 0 || d->C == 0) return IGD_OK;
    if (!d->rtp12 || !d->payload || !d->state || !d->pkts || !d->sizes || !d->bytemean_out)
        return fail(c, IGD_EINVAL, "igd_ed137_pack: null buffer");
    if (d->mem == IGD_MEM_DEVICE &&
        (!aligned(d->rtp12, 4) || !aligned(d->payload, 4) || !aligned(d->pkts, 4) || !aligned(d->sizes, 4) ||
         !aligned(d->state, 8) || (d->ctl && !aligned(d->ctl, 8)) || (d->stale_payload && !aligned(d->stale_payload, 4))))
        return fail(c, IGD_EINVAL, "igd_ed137_pack: misaligned device pointer (4 bytes; state / ctl 8)");
    IGD_BIND(c);
    const size_t n = (size_t)d->F * d->C;
    const int mem = d->mem;
    igd_ed137_pack_desc k = *d;
    int rc;
    const uint8_t *drtp, *dpay; const igd_ed137_ctl *dctl = nullptr;
    igd_ed137_state *dst; uint8_t *dpk; uint32_t *dsz; uint8_t *dbm; void *dplan;
    if ((rc = in_arg(c, mem, 0, d->rtp12, n * 12, &drtp))) return rc;
    if ((rc = in_arg(c, mem, 1, d->payload, n * IGD_FRAME, &dpay))) return rc;
    if (d->ctl && (rc = in_arg(c, mem, 2, d->ctl, n, &dctl))) return rc;
    {
        const igd_ed137_state *tmp = nullptr;
        if ((rc = in_arg(c, mem, 3, d->state, (size_t)d->C, &tmp))) return rc;
        dst = const_cast<igd_ed137_state *>(tmp);
    }
    if ((rc = out_arg(c, mem, 4, d->pkts, n * d->out_stride, &dpk))) return rc;
    if ((rc = out_arg(c, mem, 5, d->sizes, n, &dsz))) return rc;
    if ((rc = out_arg(c, mem, 6, d->bytemean_out, n, &dbm))) return rc;
    if ((rc = scratch(c, 8, n * sizeof(igd_tx_plan_rec), &dplan))) return rc;
    void *dlast;
    if ((rc = scratch(c, 9, (size_t)d->C * sizeof(int32_t), &dlast))) return rc;
    uint8_t *dstale = nullptr;
    if (d->stale_payload) {
        const uint8_t *tmp2 = nullptr;
        if ((rc = in_arg(c, mem, 10, static_cast<const uint8_t *>(d->stale_payload), (size_t)d->C * IGD_FRAME, &tmp2)))
            return rc;
        dstale = const_cast<uint8_t *>(tmp2);
    }
    k.rtp12 = drtp; k.payload = dpay; k.ctl = dctl; k.state = dst; k.pkts = dpk; k.sizes = dsz; k.bytemean_out = dbm;
    k.stale_payload = dstale;
    IGD_CUDA(c, igd_k_ed137_pack(cfg_of(c), k, static_cast<igd_tx_plan_rec *>(dplan), static_cast<int32_t *>(dlast)));
    c->launches += dstale ? 3 : 2;
    if (dstale && (rc = out_done(c, mem, d->stale_payload, dstale, (size_t)d->C * IGD_FRAME))) return rc;
    if ((rc = out_done(c, mem, d->pkts, dpk, n * d->out_stride))) return rc;
    if ((rc = out_done(c, mem, d->sizes, dsz, n))) return rc;
    if ((rc = out_done(c, mem, d->bytemean_out, dbm, n))) return rc;
    if ((rc = out_done(c, mem, d->state, dst, (size_t)d->C))) return rc;
    return finish(c, mem);
}

int igd_ed137_keepalive(igd_ctx *c, uint8_t *hdr20, igd_ed137_state *state, size_t C, int64_t now_ms,
                        uint32_t *sizes, int mem)
{
    if (!c || (C && (!hdr20 || !state || !sizes))) return fail(c, IGD_EINVAL, "igd_ed137_keepalive: bad argument");
    if (C == 0) return IGD_OK;
    if (mem == IGD_MEM_DEVICE && (!aligned(hdr20, 4) || !aligned(state, 8) || !aligned(sizes, 4)))
        return fail(c, IGD_EINVAL, "igd_ed137_keepalive: misaligned device pointer");
    IGD_BIND(c);
    int rc;
    const uint8_t *th = nullptr; const igd_ed137_state *ts = nullptr; uint32_t *dsz = nullptr;
    if ((rc = in_arg(c, mem, 0, hdr20, C * IGD_PKT_HDR, &th))) return rc;
    if ((rc = in_arg(c, mem, 1, state, C, &ts))) return rc;
    if ((rc = out_arg(c, mem, 2, sizes, C, &dsz))) return rc;
    uint8_t *dh = const_cast<uint8_t *>(th);
    igd_ed137_state *ds = const_cast<igd_ed137_state *>(ts);
    IGD_CUDA(c, igd_k_ed137_keepalive(cfg_of(c), dh, ds, C, (long long)now_ms, dsz));
    c->launches++;
    if ((rc = out_done(c, mem, hdr20, dh, C * IGD_PKT_HDR))) return rc;
    if ((rc = out_done(c, mem, state, ds, C))) return rc;
    if ((rc = out_done(c, mem, sizes, dsz, C))) return rc;
    return finish(c, mem);
}

// ---------------------------------------------------------------- RX liveness, gate arbitration
int igd_rx_track(igd_ctx *c, const igd_rx_track_desc *d)
{
    if (!c || !d || d->struct_size != sizeof(igd_rx_track_desc)) return fail(c, IGD_EINVAL, "igd_rx_track: bad descriptor");
    if (d->F < 0 || d->C < 0 || d->wd_ticks < 0 || d->frame0 < 0) return fail(c, IGD_EINVAL, "igd_rx_track: bad shape / frame0");
    if (d->F == 0 || d->C == 0) return IGD_OK;
    if (!d->fields || !d->state || !d->events) return fail(c, IGD_EINVAL, "igd_rx_track: null buffer");
    const int mem = d->mem;
    if (mem == IGD_MEM_DEVICE && (!aligned(d->fields, 16) || !aligned(d->state, 16) || !aligned(d->events, 8)))
        return fail(c, IGD_EINVAL, "igd_rx_track: misaligned device pointer");
    IGD_BIND(c);
    const size_t n = (size_t)d->F * d->C;
    igd_rx_track_desc k = *d;
    int rc;
    if ((rc = in_arg(c, mem, 0, d->fields, n, &k.fields))) return rc;
    if (d->present && (rc = in_arg(c, mem, 1, d->present, n, &k.present))) return rc;
    if (d->sizes && (rc = in_arg(c, mem, 4, d->sizes, n, &k.sizes))) return rc;
    {
        const igd_rx_state *tmp = nullptr;
        if ((rc = in_arg(c, mem, 2, d->state, (size_t)d->C, &tmp))) return rc;
        k.state = const_cast<igd_rx_state *>(tmp);
    }
    if ((rc = out_arg(c, mem, 3, d->events, n, &k.events))) return rc;
    IGD_CUDA(c, igd_k_rx_track(cfg_of(c), k));
    c->launches++;
    if ((rc = out_done(c, mem, d->state, k.state, (size_t)d->C))) return rc;
    if ((rc = out_done(c, mem, d->events, k.events, n))) return rc;
    return finish(c, mem);
}

int igd_gate_arbitrate(igd_ctx *c, const igd_arb_desc *d)
{
    if (!c || !d || d->struct_size != sizeof(igd_arb_desc)) return fail(c, IGD_EINVAL, "igd_gate_arbitrate: bad descriptor");
    if (d->F < 0 || d->B < 0 || d->G < 1 || d->G > IGD_MAX_LEGS || (d->word_stride != 4 && d->word_stride != 8) ||
        (d->mode != IGD_ARB_CLIENT_PTT && d->mode != IGD_ARB_SERVER_BEST))
        return fail(c, IGD_EINVAL, "igd_gate_arbitrate: bad shape / mode / word_stride");
    if (d->B == 0) return IGD_OK;
    if (!d->legs || !d->bridges || (d->F && (!d->words || !d->gain_q7)))
        return fail(c, IGD_EINVAL, "igd_gate_arbitrate: null buffer");
    const int mem = d->mem;
    if (mem == IGD_MEM_DEVICE && (!aligned(d->words, 4) || !aligned(d->legs, 8) || !aligned(d->bridges, 4)))
        return fail(c, IGD_EINVAL, "igd_gate_arbitrate: misaligned device pointer");
    IGD_BIND(c);
    const size_t Cn = (size_t)d->B * d->G, n = (size_t)d->F * Cn;
    igd_arb_desc k = *d;
    int rc;
    {
        const uint8_t *w = nullptr;
        if ((rc = in_arg(c, mem, 0, static_cast<const uint8_t *>(d->words), n * d->word_stride, &w))) return rc;
        k.words = w;
    }
    if (d->active && (rc = in_arg(c, mem, 1, d->active, Cn, &k.active))) return rc;
    {
        const igd_arb_leg *tl = nullptr; const igd_arb_bridge *tb = nullptr;
        if ((rc = in_arg(c, mem, 2, d->legs, Cn, &tl))) return rc;
        if ((rc = in_arg(c, mem, 3, d->bridges, (size_t)d->B, &tb))) return rc;
        k.legs = const_cast<igd_arb_leg *>(tl);
        k.bridges = const_cast<igd_arb_bridge *>(tb);
    }
    if ((rc = out_arg(c, mem, 4, d->gain_q7, n, &k.gain_q7))) return rc;
    IGD_CUDA(c, igd_k_gate_arbitrate(cfg_of(c), k));
    c->launches++;
    if ((rc = out_done(c, mem, d->legs, k.legs, Cn))) return rc;
    if ((rc = out_done(c, mem, d->bridges, k.bridges, (size_t)d->B))) return rc;
    if ((rc = out_done(c, mem, d->gain_q7, k.gain_q7, n))) return rc;
    return finish(c, mem);
}

// ---------------------------------------------------------------- gateway: packets in, packets out
int igd_gateway_process(igd_ctx *c, const igd_gateway_desc *d)
{
    if (!c || !d || d->struct_size != sizeof(igd_gateway_desc))
        return fail(c, IGD_EINVAL, "igd_gateway_process: bad descriptor");
    if (d->F < 0 || d->B < 0 || d->wd_ticks < 0 || d->frame0 < 0 ||
        (d->arb_mode != IGD_ARB_CLIENT_PTT && d->arb_mode != IGD_ARB_SERVER_BEST))
        return fail(c, IGD_EINVAL, "igd_gateway_process: bad shape / mode / frame0");
    if (d->G != 4) return fail(c, IGD_EINVAL, "igd_gateway_process: G must be 4");
    if (d->flags & ~(IGD_F_SIGNED_CHAR | IGD_F_KERNEL_W | IGD_F_WALK_SERIAL))
        return fail(c, IGD_EINVAL, "igd_gateway_process: flags (IGD_F_SIGNED_CHAR, IGD_F_KERNEL_W, IGD_F_WALK_SERIAL only)");
    if (d->F == 0 || d->B == 0) return IGD_OK;
    if (!d->rx_pkts || !d->law || !d->rx_state || !d->arb_legs || !d->arb_bridges || !d->out_law || !d->tx_rtp12 ||
        !d->tx_state || !d->tx_pkts || !d->tx_sizes)
        return fail(c, IGD_EINVAL, "igd_gateway_process: null buffer");
    const int mem = d->mem;
    if (mem == IGD_MEM_DEVICE &&
        (!aligned(d->rx_pkts, 16) || (d->rx_sizes && !aligned(d->rx_sizes, 4)) || !aligned(d->law, 4) ||
         !aligned(d->rx_state, 16) || !aligned(d->arb_legs, 8) || !aligned(d->arb_bridges, 4) || !aligned(d->tx_rtp12, 4) ||
         (d->tx_ctl && !aligned(d->tx_ctl, 8)) || !aligned(d->tx_state, 8) || !aligned(d->tx_pkts, 4) ||
         !aligned(d->tx_sizes, 4) || (d->rx_events && !aligned(d->rx_events, 8)) || (d->gain_q7 && !aligned(d->gain_q7, 8)) ||
         (d->meter && !aligned(d->meter, 16)) || (d->bmeter && !aligned(d->bmeter, 4)) || (d->mix && !aligned(d->mix, 32)) ||
         (d->enc && !aligned(d->enc, 16))))
        return fail(c, IGD_EINVAL, "igd_gateway_process: misaligned device pointer");
    IGD_BIND(c);
    const size_t F = d->F, B = d->B, Cn = B * 4, n = F * Cn, nb = F * B;
    int rc;
    // ---- inputs (host form: staged; slots 0..5 in, 6..11 scratch / out)
    const uint8_t *dpk, *dlaw, *dact = nullptr, *dol, *drtp; const uint32_t *dsz = nullptr; const igd_ed137_ctl *dctl = nullptr;
    // (host form: the four per-tick input arrays are only given room here; they come over chunk by chunk, beside the
    //  kernels of the chunk before -- see the pipeline below)
    const bool host = mem == IGD_MEM_HOST;
    if (!host) { dpk = d->rx_pkts; dsz = d->rx_sizes; }
    else {
        void *p0 = nullptr, *p1 = nullptr;
        if ((rc = scratch(c, 0, n * IGD_PKT_MAX, &p0))) return rc;
        if (d->rx_sizes && (rc = scratch(c, 1, n * sizeof(uint32_t), &p1))) return rc;
        dpk = static_cast<const uint8_t *>(p0); dsz = static_cast<const uint32_t *>(p1);
    }
    void *small = nullptr;       // law, active, out_law, states in one staged block (host form)
    igd_rx_state *drx; igd_arb_leg *dleg; igd_arb_bridge *dbr; igd_ed137_state *dtx;
    if (mem == IGD_MEM_DEVICE) {
        dlaw = d->law; dact = d->active; dol = d->out_law;
        drx = d->rx_state; dleg = d->arb_legs; dbr = d->arb_bridges; dtx = d->tx_state;
    } else {
        const size_t o_law = 0, o_act = o_law + ((Cn + 15) & ~(size_t)15), o_ol = o_act + ((Cn + 15) & ~(size_t)15),
                     o_rx = o_ol + ((B + 15) & ~(size_t)15), o_leg = o_rx + Cn * sizeof(igd_rx_state),
                     o_br = o_leg + Cn * sizeof(igd_arb_leg), o_tx = o_br + B * sizeof(igd_arb_bridge),
                     total = o_tx + B * sizeof(igd_ed137_state);
        if ((rc = scratch(c, 2, total, &small))) return rc;
        uint8_t *sb = static_cast<uint8_t *>(small);
        IGD_CUDA(c, cudaMemcpyAsync(sb + o_law, d->law, Cn, cudaMemcpyHostToDevice, c->stream));
        if (d->active) IGD_CUDA(c, cudaMemcpyAsync(sb + o_act, d->active, Cn, cudaMemcpyHostToDevice, c->stream));
        IGD_CUDA(c, cudaMemcpyAsync(sb + o_ol, d->out_law, B, cudaMemcpyHostToDevice, c->stream));
        IGD_CUDA(c, cudaMemcpyAsync(sb + o_rx, d->rx_state, Cn * sizeof(igd_rx_state), cudaMemcpyHostToDevice, c->stream));
        IGD_CUDA(c, cudaMemcpyAsync(sb + o_leg, d->arb_legs, Cn * sizeof(igd_arb_leg), cudaMemcpyHostToDevice, c->stream));
        IGD_CUDA(c, cudaMemcpyAsync(sb + o_br, d->arb_bridges, B * sizeof(igd_arb_bridge), cudaMemcpyHostToDevice, c->stream));
        IGD_CUDA(c, cudaMemcpyAsync(sb + o_tx, d->tx_state, B * sizeof(igd_ed137_state), cudaMemcpyHostToDevice, c->stream));
        dlaw = sb + o_law; dact = d->active ? sb + o_act : nullptr; dol = sb + o_ol;
        drx = reinterpret_cast<igd_rx_state *>(sb + o_rx); dleg = reinterpret_cast<igd_arb_leg *>(sb + o_leg);
        dbr = reinterpret_cast<igd_arb_bridge *>(sb + o_br); dtx = reinterpret_cast<igd_ed137_state *>(sb + o_tx);
    }
    if (!host) { drtp = d->tx_rtp12; dctl = d->tx_ctl; }
    else {
        void *p3 = nullptr, *p4 = nullptr;
        if ((rc = scratch(c, 3, nb * 12, &p3))) return rc;
        if (d->tx_ctl && (rc = scratch(c, 4, nb * sizeof(igd_ed137_ctl), &p4))) return rc;
        drtp = static_cast<const uint8_t *>(p3); dctl = static_cast<const igd_ed137_ctl *>(p4);
    }
    // ---- intermediates that never cross the API: field records, events, gains, sender plan
    void *dplan, *dlast, *dev_s = nullptr, *dgain_s = nullptr;
    if ((rc = scratch(c, 6, nb * sizeof(igd_tx_plan_rec) + B * sizeof(int32_t), &dplan))) return rc;
    dlast = static_cast<uint8_t *>(dplan) + nb * sizeof(igd_tx_plan_rec);
    // The receive side (liveness walk + gate arbitration) comes in three forms:
    //   lanes        one warp per bridge, tick axis across its lanes (igd_walks.cuh: k_rxarb_walk), sender k_plan_walk:
    //                calls of IGD_WALK_MIN_TICKS ticks and more below IGD_GW_LANE_MAX_CH channels;
    //   bridge_walk  one thread per bridge, both state machines in one kernel (k_rxarb_bridge): from 65 536 channels up,
    //                and every call of a few ticks (the real-time shape);
    //   otherwise    (IGD_F_WALK_SERIAL) header view / liveness walk / arbitration as separate thread-per-channel kernels,
    //                pipelined over chunks of ticks below 32 768 channels.
    // Measured (bench.py --chain; lanes / separate kernels / bridge_walk, ms per call): 4096 ch x 1640 ticks 0.61 / 1.26 /
    // 2.8, 16 384 x 400 0.61 / 0.96 / 1.5, 32 768 x 200 0.62 / 0.73 / 0.66, 65 536 x 100 0.668 / 0.663 / 0.575, 65 536 x 200
    // 1.31 / - / 1.14: from 65 536 channels up a thread per bridge has enough independent walks to be bound by the header
    // reads alone, below that the lanes' parallelism wins.
#ifndef IGD_GW_LANE_MAX_CH
#define IGD_GW_LANE_MAX_CH 65536
#endif
    const bool lanes = !(d->flags & IGD_F_WALK_SERIAL) && d->F >= IGD_WALK_MIN_TICKS && Cn < (size_t)IGD_GW_LANE_MAX_CH;
#ifndef IGD_GW_BRIDGE_MIN_CH
#define IGD_GW_BRIDGE_MIN_CH 32768
#endif
    const bool bridge_walk = !lanes && !(d->flags & IGD_F_WALK_SERIAL) &&
                             (Cn >= (size_t)IGD_GW_BRIDGE_MIN_CH || d->F < IGD_WALK_MIN_TICKS);      // ... and every call of a few ticks
    const bool one_kernel = lanes || bridge_walk;      // receive walk + arbitration in one launch, words handed over in registers
    igd_rx_event *dev = nullptr; uint16_t *dgain;
    if (mem == IGD_MEM_DEVICE && d->rx_events) dev = d->rx_events;
    else if (!one_kernel || d->rx_events) {      // no event array between the walk and the arbitration unless it is wanted
        if ((rc = scratch(c, 7, n * sizeof(igd_rx_event), &dev_s))) return rc;
        dev = static_cast<igd_rx_event *>(dev_s);
    }
    if (mem == IGD_MEM_DEVICE && d->gain_q7) dgain = d->gain_q7;
    else { if ((rc = scratch(c, 8, n * sizeof(uint16_t), &dgain_s))) return rc; dgain = static_cast<uint16_t *>(dgain_s); }
    // ---- outputs
    uint8_t *dtp; uint32_t *dts; igd_meter_rec *dmt = nullptr; igd_bridge_rec *dbm = nullptr; int16_t *dmix = nullptr; uint8_t *denc = nullptr;
    if ((rc = out_arg(c, mem, 9, d->tx_pkts, nb * IGD_PKT_MAX, &dtp))) return rc;
    if ((rc = out_arg(c, mem, 10, d->tx_sizes, nb, &dts))) return rc;
    if (mem == IGD_MEM_DEVICE) { dmt = d->meter; dbm = d->bmeter; dmix = d->mix; denc = d->enc; }
    else {
        // host form: the optional record / PCM outputs share slot 11
        const size_t o_mt = 0, o_bm = o_mt + (d->meter ? n * sizeof(igd_meter_rec) : 0), o_mx = (o_bm + (d->bmeter ? nb * sizeof(igd_bridge_rec) : 0) + 31) & ~(size_t)31,
                     o_en = o_mx + (d->mix ? nb * IGD_FRAME * sizeof(int16_t) : 0), total = o_en + (d->enc ? nb * IGD_FRAME : 0);
        void *ob = nullptr;
        if (total && (rc = scratch(c, 11, total, &ob))) return rc;
        uint8_t *o8 = static_cast<uint8_t *>(ob);
        if (d->meter) dmt = reinterpret_cast<igd_meter_rec *>(o8 + o_mt);
        if (d->bmeter) dbm = reinterpret_cast<igd_bridge_rec *>(o8 + o_bm);
        if (d->mix) dmix = reinterpret_cast<int16_t *>(o8 + o_mx);
        if (d->enc) denc = o8 + o_en;
    }
    const igd_launch_cfg k = cfg_of(c);
    // The sender walk does not depend on the receive side: it runs on a side stream, concurrently with the receive-side
    // walk(s).  Fork / join through events, so the whole call stays capturable in a CUDA graph.
    igd_launch_cfg kside = k;
    kside.stream = c->copy_streams[0];
    IGD_CUDA(c, cudaEventRecord(c->ev[6], c->stream));
    IGD_CUDA(c, cudaStreamWaitEvent(kside.stream, c->ev[6], 0));
    // With the separate thread-per-channel kernels (IGD_F_WALK_SERIAL) the call is a pipeline over chunks of ticks: liveness
    // walk (+ header pass) -> arbitration -> fused kernel, each stage on its own stream, chunk k of a stage waiting for
    // chunk k of the stage before it, and the sender walk of the same chunk beside them on the side stream (the fused
    // kernel needs its plan).  Those walks are latency-bound grids of a few thousand threads; back to back they cost twice
    // the fused kernel (4096 channels x 1640 ticks: 1.50 ms per call), pipelined 1.26-1.3 ms.  Every stage carries its
    // state from chunk to chunk in the caller's state arrays, exactly as from call to call, so the results do not depend
    // on the chunking.  The host form uses the same chunks to overlap its copies, whatever the walk.
#ifndef IGD_GW_CHUNKS
#define IGD_GW_CHUNKS 8
#endif
#ifndef IGD_GW_MIN_TICKS
#define IGD_GW_MIN_TICKS 16
#endif
    static_assert(IGD_GW_CHUNKS >= 1 && IGD_GW_CHUNKS <= 8, "walk_ev holds 8 chunks");
    // (from 32 768 channels up the walks are no longer idle time -- the liveness walk is a 6 TB/s header read -- and
    // chunking only adds launches: 0.67 ms unchunked, 0.68 / 0.77 / 0.78 ms with 2 / 4 / 6 chunks at 65 536 channels)
    int nchunk = Cn >= 32768 ? 1 : d->F / IGD_GW_MIN_TICKS;
    // the lane walks: a single launch of the receive-side walk, then the fused kernel (the persistent fused CTA leaves
    // no registers on its SM for a walk block, so chunks of the two do not overlap -- they only add launches)
#ifndef IGD_GW_LANE_CHUNKS
#define IGD_GW_LANE_CHUNKS 1
#endif
    if (lanes && nchunk > IGD_GW_LANE_CHUNKS) nchunk = IGD_GW_LANE_CHUNKS;
    // host form: the chunks are what the copies overlap with -- the call is bound by the packets coming in over PCIe,
    // so the chunk count follows the bytes (about 64 MiB of packets each), whatever the channel count
    if (host) nchunk = (int)((n * IGD_PKT_MAX + (48u << 20)) >> 26);
    if (nchunk > IGD_GW_CHUNKS) nchunk = IGD_GW_CHUNKS;
    if (nchunk > d->F) nchunk = d->F;
    if (nchunk < 1) nchunk = 1;
    const int chunk = (d->F + nchunk - 1) / nchunk;
    // (Leaving 12 / 20 / 32 / 48 SMs out of the fused kernel's grid for the walk blocks of the following chunks measured
    // 1.33 / 1.35 / 1.39 / 1.44 ms at the bench shape against 1.31 with the full grid: the stages stretch when they share
    // the machine -- a persistent one-CTA-per-SM kernel waits for whole SMs -- and the pipeline gains 13 %, not 2x.)
    igd_launch_cfg krx = k, karb = k;
    if (nchunk > 1) {
        krx.stream = c->walk_streams[0];
        karb.stream = c->walk_streams[1];
        IGD_CUDA(c, cudaStreamWaitEvent(krx.stream, c->ev[6], 0));       // fork: after the inputs are in place
        IGD_CUDA(c, cudaStreamWaitEvent(karb.stream, c->ev[6], 0));
    }
    void *dfields = nullptr;
    if (!one_kernel && Cn < 32768 && (rc = scratch(c, 5, n * sizeof(igd_ed137_fields), &dfields))) return rc;
#ifdef IGD_X_GW_TRACE      // measurement builds: when did each stage of each chunk start and end
    static cudaEvent_t tr[1 + 8 * 6];
    static bool tr_init = false;
    if (!tr_init) { for (auto &e : tr) cudaEventCreate(&e); tr_init = true; }
    cudaEventRecord(tr[0], c->stream);
#define IGD_TR(i, st) cudaEventRecord(tr[1 + ci * 6 + (i)], st)
#else
#define IGD_TR(i, st) ((void)0)
#endif
    for (int ci = 0, f0 = 0; f0 < d->F; ci++, f0 += chunk) {
        const int nf = d->F - f0 < chunk ? d->F - f0 : chunk;
        const size_t on = (size_t)f0 * Cn, onb = (size_t)f0 * B;       // channel-ticks / bridge-ticks before this chunk
        const size_t cn = (size_t)nf * Cn, cnb = (size_t)nf * B;        // ... and in it
        if (host) {      // this chunk's inputs, on the copy-in stream; every stage that reads them waits for the event
            cudaStream_t sin = c->io_streams[0];
            if (ci == 0) IGD_CUDA(c, cudaStreamWaitEvent(sin, c->ev[6], 0));
            IGD_CUDA(c, cudaMemcpyAsync(const_cast<uint8_t *>(dpk) + on * IGD_PKT_MAX, d->rx_pkts + on * IGD_PKT_MAX, cn * IGD_PKT_MAX, cudaMemcpyHostToDevice, sin));
            if (dsz) IGD_CUDA(c, cudaMemcpyAsync(const_cast<uint32_t *>(dsz) + on, d->rx_sizes + on, cn * sizeof(uint32_t), cudaMemcpyHostToDevice, sin));
            IGD_CUDA(c, cudaMemcpyAsync(const_cast<uint8_t *>(drtp) + onb * 12, d->tx_rtp12 + onb * 12, cnb * 12, cudaMemcpyHostToDevice, sin));
            if (dctl) IGD_CUDA(c, cudaMemcpyAsync(const_cast<igd_ed137_ctl *>(dctl) + onb, d->tx_ctl + onb, cnb * sizeof(igd_ed137_ctl), cudaMemcpyHostToDevice, sin));
            IGD_CUDA(c, cudaEventRecord(c->walk_ev[24 + ci], sin));
            IGD_CUDA(c, cudaStreamWaitEvent(krx.stream, c->walk_ev[24 + ci], 0));
            IGD_CUDA(c, cudaStreamWaitEvent(kside.stream, c->walk_ev[24 + ci], 0));
            if (krx.stream != c->stream) IGD_CUDA(c, cudaStreamWaitEvent(c->stream, c->walk_ev[24 + ci], 0));
        }
        // 1 + 2. transport_rtp_cb's view of every packet header and the liveness / latch / edge walk.  With tens of
        //        thousands of channels the walk reads the three header words it needs straight out of the packets (one
        //        kernel, no field array: enough walks in flight to hide the strided loads); with a few thousand channels
        //        and many ticks a fully parallel header pass first and the walk over its compact 16-byte records is
        //        faster (measured: 65 536 ch x 100 ticks 0.80 vs 0.83 ms per call; 4096 ch x 1640 ticks 1.64 vs 2.46 ms).
        if (one_kernel) {
            igd_rxarb_args ra;
            ra.F = nf; ra.B = d->B; ra.mode = d->arb_mode; ra.tick_ms = d->tick_ms; ra.r2s_period_ms = d->r2s_period_ms;
            ra.wd_ticks = d->wd_ticks; ra.frame0 = d->frame0 + f0; ra.now_ms0 = d->now_ms0 + (long long)f0 * d->tick_ms;
            ra.pkts = dpk + on * IGD_PKT_MAX; ra.sizes = dsz ? dsz + on : nullptr; ra.active = dact;
            ra.rx_state = drx; ra.legs = dleg; ra.bridges = dbr; ra.events = dev ? dev + on : nullptr; ra.gain_q7 = dgain + on;
            IGD_TR(0, krx.stream);
            IGD_CUDA(c, lanes ? igd_k_rxarb_walk(krx, ra) : igd_k_rxarb_bridge(krx, ra));
            IGD_TR(3, krx.stream);
            c->launches += 1;
            if (nchunk > 1) {
                IGD_CUDA(c, cudaEventRecord(c->walk_ev[8 + ci], krx.stream));
                IGD_CUDA(c, cudaStreamWaitEvent(c->stream, c->walk_ev[8 + ci], 0));
            }
        } else {
        igd_rx_track_desc rx;
        memset(&rx, 0, sizeof rx);
        rx.struct_size = sizeof rx; rx.mem = IGD_MEM_DEVICE; rx.F = nf; rx.C = (int32_t)Cn; rx.tick_ms = d->tick_ms;
        rx.r2s_period_ms = d->r2s_period_ms; rx.wd_ticks = d->wd_ticks; rx.frame0 = d->frame0 + f0;
        rx.now_ms0 = d->now_ms0 + (long long)f0 * d->tick_ms;
        rx.present = nullptr; rx.state = drx; rx.events = dev + on;
        rx.sizes = dsz ? dsz + on : nullptr;     // a leg without a packet on a tick has size 0: not a packet for the walk
        IGD_TR(0, krx.stream);
        if (Cn >= 32768) {
            rx.fields = nullptr;
            IGD_CUDA(c, igd_k_rx_track(krx, rx, dpk + on * IGD_PKT_MAX));
            c->launches += 1;
        } else {
            igd_ed137_fields *fl = static_cast<igd_ed137_fields *>(dfields) + on;
            IGD_CUDA(c, igd_k_ed137_parse(krx, dpk + on * IGD_PKT_MAX, dsz ? dsz + on : nullptr, (size_t)nf * Cn, IGD_PKT_MAX, fl, nullptr));
            rx.fields = fl;
            IGD_CUDA(c, igd_k_rx_track(krx, rx));
            c->launches += 2;
        }
        IGD_TR(1, krx.stream);
        if (nchunk > 1) {
            IGD_CUDA(c, cudaEventRecord(c->walk_ev[ci], krx.stream));
            IGD_CUDA(c, cudaStreamWaitEvent(karb.stream, c->walk_ev[ci], 0));
        }
        // 3. gate decisions; ticks without a whole audio frame carry IGD_GAIN_NO_AUDIO
        igd_arb_desc ar;
        memset(&ar, 0, sizeof ar);
        ar.struct_size = sizeof ar; ar.mem = IGD_MEM_DEVICE; ar.F = nf; ar.B = d->B; ar.G = 4; ar.mode = d->arb_mode;
        ar.word_stride = 8; ar.flags = IGD_ARB_F_SILENCE; ar.words = dev + on; ar.active = dact; ar.legs = dleg; ar.bridges = dbr;
        ar.gain_q7 = dgain + on;
        IGD_TR(2, karb.stream);
        IGD_CUDA(c, igd_k_gate_arbitrate(karb, ar));
        IGD_TR(3, karb.stream);
        if (nchunk > 1) {
            IGD_CUDA(c, cudaEventRecord(c->walk_ev[8 + ci], karb.stream));
            IGD_CUDA(c, cudaStreamWaitEvent(c->stream, c->walk_ev[8 + ci], 0));
        }
        }
        // 4. sender walk of the B outgoing calls over this chunk's ticks (independent of the receive side)
        igd_ed137_pack_desc pk;
        memset(&pk, 0, sizeof pk);
        pk.struct_size = sizeof pk; pk.mem = IGD_MEM_DEVICE; pk.F = nf; pk.C = d->B; pk.flags = d->flags & (IGD_F_SIGNED_CHAR | IGD_F_WALK_SERIAL);
        pk.payload_len = IGD_FRAME; pk.out_stride = IGD_PKT_MAX; pk.tick_ms = d->tick_ms; pk.now_ms0 = d->now_ms0 + (long long)f0 * d->tick_ms;
        pk.rtp12 = drtp + onb * 12; pk.payload = nullptr; pk.ctl = dctl ? dctl + onb : nullptr; pk.state = dtx;
        IGD_CUDA(c, igd_k_ed137_plan(kside, pk, static_cast<igd_tx_plan_rec *>(dplan) + onb, static_cast<int32_t *>(dlast)));
        IGD_CUDA(c, cudaEventRecord(c->walk_ev[16 + ci], kside.stream));
        IGD_CUDA(c, cudaStreamWaitEvent(c->stream, c->walk_ev[16 + ci], 0));            // join: this chunk's plan is there
        c->launches += 1;
        // 5. decode -> meter -> mix -> encode -> packets
        igd_packets_desc fp;
        memset(&fp, 0, sizeof fp);
        fp.struct_size = sizeof fp; fp.mem = IGD_MEM_DEVICE; fp.F = nf; fp.B = d->B; fp.G = 4; fp.flags = d->flags & (IGD_F_SIGNED_CHAR | IGD_F_KERNEL_W);
        fp.pkts = dpk + on * IGD_PKT_MAX; fp.fields = nullptr; fp.law = dlaw; fp.gain_q7 = dgain + on; fp.out_law = dol;
        fp.mix = dmix ? dmix + onb * IGD_FRAME : nullptr; fp.enc = denc ? denc + onb * IGD_FRAME : nullptr;
        fp.meter = dmt ? dmt + on : nullptr; fp.bmeter = dbm ? dbm + onb : nullptr;
        IGD_TR(4, c->stream);
        IGD_CUDA(c, igd_k_fused_gateway(k, fp, static_cast<igd_tx_plan_rec *>(dplan) + onb, drtp + onb * 12, dtp + onb * IGD_PKT_MAX, dts + onb));
        IGD_TR(5, c->stream);
        c->launches += 2;
        if (host) {      // this chunk's outputs, on the copy-out stream, beside the kernels of the next chunk
            cudaStream_t sout = c->io_streams[1];
            IGD_CUDA(c, cudaEventRecord(c->walk_ev[32 + ci], c->stream));
            IGD_CUDA(c, cudaStreamWaitEvent(sout, c->walk_ev[32 + ci], 0));
            IGD_CUDA(c, cudaMemcpyAsync(d->tx_pkts + onb * IGD_PKT_MAX, dtp + onb * IGD_PKT_MAX, cnb * IGD_PKT_MAX, cudaMemcpyDeviceToHost, sout));
            IGD_CUDA(c, cudaMemcpyAsync(d->tx_sizes + onb, dts + onb, cnb * sizeof(uint32_t), cudaMemcpyDeviceToHost, sout));
            if (d->rx_events) IGD_CUDA(c, cudaMemcpyAsync(d->rx_events + on, dev + on, cn * sizeof(igd_rx_event), cudaMemcpyDeviceToHost, sout));
            if (d->gain_q7) IGD_CUDA(c, cudaMemcpyAsync(d->gain_q7 + on, dgain + on, cn * sizeof(uint16_t), cudaMemcpyDeviceToHost, sout));
            if (d->meter) IGD_CUDA(c, cudaMemcpyAsync(d->meter + on, dmt + on, cn * sizeof(igd_meter_rec), cudaMemcpyDeviceToHost, sout));
            if (d->bmeter) IGD_CUDA(c, cudaMemcpyAsync(d->bmeter + onb, dbm + onb, cnb * sizeof(igd_bridge_rec), cudaMemcpyDeviceToHost, sout));
            if (d->mix) IGD_CUDA(c, cudaMemcpyAsync(d->mix + onb * IGD_FRAME, dmix + onb * IGD_FRAME, cnb * IGD_FRAME * sizeof(int16_t), cudaMemcpyDeviceToHost, sout));
            if (d->enc) IGD_CUDA(c, cudaMemcpyAsync(d->enc + onb * IGD_FRAME, denc + onb * IGD_FRAME, cnb * IGD_FRAME, cudaMemcpyDeviceToHost, sout));
        }
    }
#ifdef IGD_X_GW_TRACE
    cudaDeviceSynchronize();
    for (int ci = 0; ci < nchunk; ci++) {
        float t[6];
        for (int i = 0; i < 6; i++) cudaEventElapsedTime(&t[i], tr[0], tr[1 + ci * 6 + i]);
        fprintf(stderr, "chunk %d: rx %.0f-%.0f  arb %.0f-%.0f  fused %.0f-%.0f us\n", ci, 1e3 * t[0], 1e3 * t[1], 1e3 * t[2], 1e3 * t[3], 1e3 * t[4], 1e3 * t[5]);
    }
#endif
    if (mem == IGD_MEM_HOST) {
        // the per-tick outputs went out chunk by chunk; the state arrays follow, and the caller's stream waits for the
        // copy-out stream before the call returns
        IGD_CUDA(c, cudaEventRecord(c->ev[7], c->io_streams[1]));
        IGD_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev[7], 0));
        if ((rc = out_done(c, mem, d->rx_state, drx, Cn))) return rc;
        if ((rc = out_done(c, mem, d->arb_legs, dleg, Cn))) return rc;
        if ((rc = out_done(c, mem, d->arb_bridges, dbr, B))) return rc;
        if ((rc = out_done(c, mem, d->tx_state, dtx, B))) return rc;
    }
    return finish(c, mem);
}

// ---------------------------------------------------------------- gateway fan-out: one frame per bridge, a packet per leg
int igd_gateway_fanout(igd_ctx *c, const igd_fanout_desc *d)
{
    if (!c || !d || d->struct_size != sizeof(igd_fanout_desc))
        return fail(c, IGD_EINVAL, "igd_gateway_fanout: bad descriptor");
    if (d->F < 0 || d->B < 0 || d->G < 1 || d->G > IGD_MAX_LEGS || (d->flags & ~IGD_F_SIGNED_CHAR))
        return fail(c, IGD_EINVAL, "igd_gateway_fanout: bad shape (1 <= G <= 32) or flags (IGD_F_SIGNED_CHAR only)");
    if (d->F == 0 || d->B == 0) return IGD_OK;
    if ((int64_t)d->B * d->G > INT32_MAX) return fail(c, IGD_EINVAL, "igd_gateway_fanout: B*G exceeds 2^31 legs");
    if (!d->pcm || !d->law || !d->tx_rtp12 || !d->tx_state || !d->tx_pkts || !d->tx_sizes)
        return fail(c, IGD_EINVAL, "igd_gateway_fanout: null buffer");
    const int mem = d->mem;
    if (mem == IGD_MEM_DEVICE &&
        (!aligned(d->pcm, 16) || !aligned(d->tx_pkts, 16) || !aligned(d->tx_state, 8) || (d->tx_ctl && !aligned(d->tx_ctl, 8)) ||
         !aligned(d->tx_rtp12, 4) || !aligned(d->tx_sizes, 4)))
        return fail(c, IGD_EINVAL, "igd_gateway_fanout: misaligned device pointer (pcm / tx_pkts 16 bytes; tx_state / tx_ctl 8; "
                                   "tx_rtp12 / tx_sizes 4)");
    IGD_BIND(c);
    const size_t F = d->F, B = d->B, Cn = B * d->G, n = F * Cn;
    igd_ed137_pack_desc k;
    memset(&k, 0, sizeof k);
    k.struct_size = sizeof k; k.mem = IGD_MEM_DEVICE; k.F = d->F; k.C = (int32_t)Cn; k.flags = d->flags;
    k.payload_len = IGD_FRAME; k.out_stride = IGD_PKT_MAX; k.tick_ms = d->tick_ms; k.now_ms0 = d->now_ms0;
    k.payload = nullptr;             // the sender walk runs before the payloads exist (rtpFalse is not maintained)
    int rc;
    const int16_t *dpcm; const uint8_t *dlaw;
    if ((rc = in_arg(c, mem, 0, d->tx_rtp12, n * 12, &k.rtp12))) return rc;
    if ((rc = in_arg(c, mem, 1, d->pcm, F * B * IGD_FRAME, &dpcm))) return rc;
    if (d->tx_ctl && (rc = in_arg(c, mem, 2, d->tx_ctl, n, &k.ctl))) return rc;
    {
        const igd_ed137_state *tmp = nullptr;
        if ((rc = in_arg(c, mem, 3, d->tx_state, Cn, &tmp))) return rc;
        k.state = const_cast<igd_ed137_state *>(tmp);
    }
    if ((rc = out_arg(c, mem, 4, d->tx_pkts, n * IGD_PKT_MAX, &k.pkts))) return rc;
    if ((rc = out_arg(c, mem, 5, d->tx_sizes, n, &k.sizes))) return rc;
    if (d->tx_level && (rc = out_arg(c, mem, 6, d->tx_level, n, &k.bytemean_out))) return rc;
    if ((rc = in_arg(c, mem, 7, d->law, Cn, &dlaw))) return rc;
    void *dplan, *dlast;             // the slots igd_ed137_pack keeps its plan in
    if ((rc = scratch(c, 8, n * sizeof(igd_tx_plan_rec), &dplan))) return rc;
    if ((rc = scratch(c, 9, Cn * sizeof(int32_t), &dlast))) return rc;
    IGD_CUDA(c, igd_k_gateway_fanout(cfg_of(c), k, d->G, dpcm, dlaw, static_cast<igd_tx_plan_rec *>(dplan),
                                     static_cast<int32_t *>(dlast)));
    c->launches += 2;
    if ((rc = out_done(c, mem, d->tx_pkts, k.pkts, n * IGD_PKT_MAX))) return rc;
    if ((rc = out_done(c, mem, d->tx_sizes, k.sizes, n))) return rc;
    if (d->tx_level && (rc = out_done(c, mem, d->tx_level, k.bytemean_out, n))) return rc;
    if ((rc = out_done(c, mem, d->tx_state, k.state, Cn))) return rc;
    return finish(c, mem);
}

// ---------------------------------------------------------------- gateway fan-out from the console call's packets
int igd_gateway_fanout_packets(igd_ctx *c, const igd_fanout_pkt_desc *d)
{
    if (!c || !d || d->struct_size != sizeof(igd_fanout_pkt_desc))
        return fail(c, IGD_EINVAL, "igd_gateway_fanout_packets: bad descriptor");
    if (d->F < 0 || d->B < 0 || d->G < 1 || d->G > IGD_MAX_LEGS || (d->flags & ~IGD_F_SIGNED_CHAR))
        return fail(c, IGD_EINVAL, "igd_gateway_fanout_packets: bad shape (1 <= G <= 32) or flags (IGD_F_SIGNED_CHAR only)");
    if (d->F == 0 || d->B == 0) return IGD_OK;
    if ((int64_t)d->B * d->G > INT32_MAX) return fail(c, IGD_EINVAL, "igd_gateway_fanout_packets: B*G exceeds 2^31 legs");
    if (!d->rx_pkts || !d->in_law || !d->law || !d->tx_rtp12 || !d->tx_state || !d->tx_pkts || !d->tx_sizes)
        return fail(c, IGD_EINVAL, "igd_gateway_fanout_packets: null buffer");
    const int mem = d->mem;
    if (mem == IGD_MEM_DEVICE &&
        (!aligned(d->rx_pkts, 16) || !aligned(d->tx_pkts, 16) || !aligned(d->tx_state, 8) ||
         (d->tx_ctl && !aligned(d->tx_ctl, 8)) || !aligned(d->tx_rtp12, 4) || !aligned(d->tx_sizes, 4) ||
         (d->rx_sizes && !aligned(d->rx_sizes, 4))))
        return fail(c, IGD_EINVAL, "igd_gateway_fanout_packets: misaligned device pointer (rx_pkts / tx_pkts 16 bytes; "
                                   "tx_state / tx_ctl 8; tx_rtp12 / tx_sizes / rx_sizes 4)");
    IGD_BIND(c);
    const size_t F = d->F, B = d->B, Cn = B * d->G, n = F * Cn;
    igd_ed137_pack_desc k;
    memset(&k, 0, sizeof k);
    k.struct_size = sizeof k; k.mem = IGD_MEM_DEVICE; k.F = d->F; k.C = (int32_t)Cn; k.flags = d->flags;
    k.payload_len = IGD_FRAME; k.out_stride = IGD_PKT_MAX; k.tick_ms = d->tick_ms; k.now_ms0 = d->now_ms0;
    k.payload = nullptr;             // the sender walk runs before the payloads exist (rtpFalse is not maintained)
    int rc;
    const uint8_t *drx, *dinlaw, *dlaw;
    const uint32_t *drsz = nullptr;
    if ((rc = in_arg(c, mem, 0, d->tx_rtp12, n * 12, &k.rtp12))) return rc;
    if ((rc = in_arg(c, mem, 1, d->rx_pkts, F * B * IGD_PKT_MAX, &drx))) return rc;
    if (d->tx_ctl && (rc = in_arg(c, mem, 2, d->tx_ctl, n, &k.ctl))) return rc;
    {
        const igd_ed137_state *tmp = nullptr;
        if ((rc = in_arg(c, mem, 3, d->tx_state, Cn, &tmp))) return rc;
        k.state = const_cast<igd_ed137_state *>(tmp);
    }
    if ((rc = out_arg(c, mem, 4, d->tx_pkts, n * IGD_PKT_MAX, &k.pkts))) return rc;
    if ((rc = out_arg(c, mem, 5, d->tx_sizes, n, &k.sizes))) return rc;
    if (d->tx_level && (rc = out_arg(c, mem, 6, d->tx_level, n, &k.bytemean_out))) return rc;
    if ((rc = in_arg(c, mem, 7, d->law, Cn, &dlaw))) return rc;
    if (d->rx_sizes && (rc = in_arg(c, mem, 10, d->rx_sizes, F * B, &drsz))) return rc;
    if ((rc = in_arg(c, mem, 11, d->in_law, B, &dinlaw))) return rc;
    void *dplan, *dlast;             // the slots igd_ed137_pack keeps its plan in
    if ((rc = scratch(c, 8, n * sizeof(igd_tx_plan_rec), &dplan))) return rc;
    if ((rc = scratch(c, 9, Cn * sizeof(int32_t), &dlast))) return rc;
    IGD_CUDA(c, igd_k_gateway_fanout_packets(cfg_of(c), k, d->G, drx, drsz, dinlaw, dlaw,
                                             static_cast<igd_tx_plan_rec *>(dplan), static_cast<int32_t *>(dlast)));
    c->launches += 2;
    if ((rc = out_done(c, mem, d->tx_pkts, k.pkts, n * IGD_PKT_MAX))) return rc;
    if ((rc = out_done(c, mem, d->tx_sizes, k.sizes, n))) return rc;
    if (d->tx_level && (rc = out_done(c, mem, d->tx_level, k.bytemean_out, n))) return rc;
    if ((rc = out_done(c, mem, d->tx_state, k.state, Cn))) return rc;
    return finish(c, mem);
}

// ---------------------------------------------------------------- recorder
size_t igd_wav_size(size_t payload_bytes, int ref_quirks)
{
    return 44 + (ref_quirks ? 2 * payload_bytes : payload_bytes);
}

int igd_wav_image(igd_ctx *c, const uint8_t *payload, size_t n, int rate, int law, int ref_quirks,
                  uint8_t *out, size_t *out_len, int mem)
{
    if (!c || !out || (n && !payload)) return fail(c, IGD_EINVAL, "igd_wav_image: bad argument");
    if (mem == IGD_MEM_DEVICE && !aligned(out, 4)) return fail(c, IGD_EINVAL, "igd_wav_image: misaligned output");
    IGD_BIND(c);
    const size_t total = igd_wav_size(n, ref_quirks);
    const uint8_t *dp; uint8_t *dout;
    int rc;
    if ((rc = in_arg(c, mem, 0, payload, n, &dp))) return rc;
    if ((rc = out_arg(c, mem, 2, out, total, &dout))) return rc;
    IGD_CUDA(c, igd_k_wav_image(cfg_of(c), dp, n, rate, law, ref_quirks, dout));
    c->launches++;
    if ((rc = out_done(c, mem, out, dout, total))) return rc;
    if (out_len) *out_len = total;
    return finish(c, mem);
}

int igd_wav_images(igd_ctx *c, const uint8_t *codes, size_t F, size_t C, const uint32_t *chans, size_t nchan,
                   const uint8_t *law, int rate, int ref_quirks, uint8_t *out, size_t image_stride, int mem)
{
    const size_t need = igd_wav_size(F * IGD_FRAME, ref_quirks);
    if (!c || (nchan && (!out || (F && !codes))) || (image_stride & 3) || image_stride < need || (!chans && nchan > C))
        return fail(c, IGD_EINVAL, "igd_wav_images: bad argument (image_stride: multiple of 4, >= igd_wav_size)");
    if (nchan == 0) return IGD_OK;
    if (mem == IGD_MEM_DEVICE && (!aligned(codes, 4) || !aligned(out, 4)))
        return fail(c, IGD_EINVAL, "igd_wav_images: misaligned device pointer");
    if (chans && mem == IGD_MEM_HOST)
        for (size_t k = 0; k < nchan; k++)
            if (chans[k] >= C) return fail(c, IGD_EINVAL, "igd_wav_images: channel index out of range");
    IGD_BIND(c);
    const uint8_t *dc, *dl = nullptr; const uint32_t *dch = nullptr; uint8_t *dout;
    int rc;
    if ((rc = in_arg(c, mem, 0, codes, F * C * IGD_FRAME, &dc))) return rc;
    if (chans && (rc = in_arg(c, mem, 1, chans, nchan, &dch))) return rc;
    if (law && (rc = in_arg(c, mem, 3, law, C, &dl))) return rc;
    if ((rc = out_arg(c, mem, 2, out, nchan * image_stride, &dout))) return rc;
    if (mem == IGD_MEM_HOST && image_stride > need) IGD_CUDA(c, cudaMemsetAsync(dout, 0, nchan * image_stride, c->stream));
    IGD_CUDA(c, igd_k_wav_images(cfg_of(c), dc, F, C, dch, nchan, dl, rate, ref_quirks, dout, image_stride));
    c->launches++;
    if ((rc = out_done(c, mem, out, dout, nchan * image_stride))) return rc;
    return finish(c, mem);
}

}  // extern "C"
