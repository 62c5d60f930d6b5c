// cfb_api.cu -- C-ABI implementation (see include/cfhd_b200.h).
//
// Host side of the transform path: pyramid layout, quantisation schedule, CUDA
// context / staging management and the kernel launch sequences.  No transform
// arithmetic is ever done on the host: if no sm_100 device is usable every
// transform entry point fails with CFB_ERROR_NO_DEVICE.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <new>

#include "cfb_host.h"

#include <mutex>
#include <ctype.h>
#include <sched.h>
#include <stdio.h>

namespace cfb {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

cfb_error cuda_fail(cudaError_t e, const char *what)
{
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return CFB_ERROR_NO_DEVICE;
    if (e == cudaErrorMemoryAllocation) return CFB_ERROR_OUTOFMEMORY;
    return CFB_ERROR_CUDA;
}

// Codec/quantize.c:1395-1427: multiplier = 65536/d, midpoint = d/g (g in [2,9)), minus one when g == 2.
QuantParam make_quant_param(int divisor, int g, bool plain_midpoint)
{
    QuantParam q;
    if (divisor <= 1) { q.m = 65536; q.cpos = 0; q.cneg = 65535; q.pad = 0; return q; }
    int mid = 0;
    // plain_midpoint: the difference-filtered HL band of the field transform rounds with divisor / g and has no
    // "-1" adjustment (spatial.c:5356-5358), unlike QuantizeRow16sTo16s (quantize.c:1415-1427)
    if (g >= 2 && g < 9) { mid = divisor / g; if (g == 2 && mid && !plain_midpoint) mid--; }
    q.m = 65536 / divisor;
    q.cpos = mid * q.m;
    q.cneg = 65535 - mid * q.m;
    q.pad = 0;
    return q;
}

cudaError_t stream_wait(cfb_context *ctx)
{
    cudaError_t e = cudaEventRecord(ctx->done, ctx->stream);
    if (e != cudaSuccess) return e;
    return cudaEventSynchronize(ctx->done);
}

static inline int align16(int x) { return (x + 15) & ~15; }
static inline int64_t align64(int64_t x) { return (x + 63) & ~(int64_t)63; }
// bytes of one V210 row: whole groups of 6 pixels in 4 32-bit words
static inline int v210_row_bytes(int w) { return (w + 5) / 6 * 16; }

static int channels_of(int fmt) { return fmt == CFB_PIXEL_BYR4 ? 4 : 3; }

// Rows per warp.  Measured on B200 (tools/microbench.py, 16 x 4K frames): 8..16 rows per warp is the sweet
// spot -- enough warps (>= ~60 per SM over the launch) that wave quantisation and the tail vanish, while the
// one-pair halo each warp re-reads stays <= 6-12 % (and is served by L2).  Larger blocks only pay off when
// the launch is too small to fill the machine anyway.
static int pick_th(int strips, int oh, int planes, int sm_count)
{
    static const int cand[] = {16, 12, 8, 6, 4};
    if (const char *e = getenv("CFB_TH")) { int v = atoi(e); if (v >= 2) return v; }     // tuning knob (development)
    const long long want = (long long)sm_count * 48;
    for (int th : cand) {
        long long warps = (long long)strips * ((oh + th - 1) / th) * planes;
        if (warps >= want) return th;
    }
    return 4;
}

int pick_rows_per_warp(int strips, int rows, int planes, int sm_count) { return pick_th(strips, rows, planes, sm_count); }

}  // namespace cfb

using namespace cfb;

extern "C" {

int cfb_version(void) { return 100; }

const char *cfb_last_error_string(void) { return g_err; }

int cfb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// NUMA placement.  Host<->device copies run at full PCIe rate only from memory (and threads) on the GPU's own NUMA
// node; the reference pins its worker threads too (Codec/thread.c SetThreadAffinityMask / the SDK's thread
// "capabilities" masks).  Linux sysfs only: /sys/bus/pci/devices/<bdf>/numa_node, /sys/devices/system/node/nodeN/cpulist.
int cfb_device_numa_node(int device)
{
    char bdf[32] = {0};
    if (cudaDeviceGetPCIBusId(bdf, sizeof(bdf), device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char *c = bdf; *c; c++) *c = (char)tolower((unsigned char)*c);
    char path[128];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bdf);
    FILE *f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

cfb_error cfb_bind_thread_to_device(int device)
{
    const int node = cfb_device_numa_node(device);
    if (node < 0) return CFB_OK;                    // no NUMA information (single node, container without sysfs): leave as is
    char path[128];
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
    FILE *f = fopen(path, "r");
    if (!f) return CFB_OK;
    char list[4096] = {0};
    const size_t n = fread(list, 1, sizeof(list) - 1, f);
    fclose(f);
    list[n] = 0;
    cpu_set_t allowed, want;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof(allowed), &allowed) != 0) return CFB_OK;
    int count = 0;
    for (char *tok = strtok(list, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int a = 0, b = 0;
        const int k = sscanf(tok, "%d-%d", &a, &b);
        if (k == 1) b = a;
        if (k < 1) continue;
        for (int c = a; c <= b && c < CPU_SETSIZE; c++)
            if (CPU_ISSET(c, &allowed)) { CPU_SET(c, &want); count++; }
    }
    if (count == 0) return CFB_OK;                  // the node's CPUs are outside this process's mask: keep the mask
    if (sched_setaffinity(0, sizeof(want), &want) != 0) { set_error("sched_setaffinity failed"); return CFB_ERROR_INVALID_ARGUMENT; }
    return CFB_OK;
}

// ---------------------------------------------------------------------------
// Layout: Codec/wavelet.c:1208-1283 (AllocTransform), :427 (AllocWaveletStack), :302 (InitWaveletStack)
cfb_error cfb_layout_compute(const cfb_frame_desc *desc, cfb_layout *out)
{
    if (!desc || !out) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    const int W = desc->width, H = desc->height, fmt = desc->pixel_format;
    if (W <= 0 || H <= 0) { set_error("bad dimensions %dx%d", W, H); return CFB_ERROR_INVALID_ARGUMENT; }
    if (fmt < CFB_PIXEL_YUYV || fmt > CFB_PIXEL_DPX0) { set_error("bad pixel format %d", fmt); return CFB_ERROR_BADFORMAT; }
    memset(out, 0, sizeof(*out));
    int cw[CFB_MAX_CHANNELS], ch[CFB_MAX_CHANNELS];
    const int nc = channels_of(fmt);
    out->num_channels = nc;
    switch (fmt) {
    case CFB_PIXEL_YUYV: case CFB_PIXEL_UYVY: case CFB_PIXEL_YU64: case CFB_PIXEL_V210:
        out->precision = 10;
        cw[0] = W; cw[1] = cw[2] = W / 2; ch[0] = ch[1] = ch[2] = H;
        out->frame_pitch = (fmt == CFB_PIXEL_YU64) ? W * 4 : (fmt == CFB_PIXEL_V210) ? ((W + 47) / 48) * 128 : W * 2;
        if (W % 16) { set_error("4:2:2 width %d must be a multiple of 16 (the reference's own row unpackers need it, convert.c:4701)", W); return CFB_ERROR_UNSUPPORTED; }
        if (fmt == CFB_PIXEL_V210 && W % 48) { set_error("V210 width %d must be a multiple of 48 (whole 6-pixel groups and 16-pixel lanes; the reference's unpacker reads row padding otherwise)", W); return CFB_ERROR_UNSUPPORTED; }
        break;
    case CFB_PIXEL_RG48: case CFB_PIXEL_PLANAR16:
    case CFB_PIXEL_RG30: case CFB_PIXEL_AB10: case CFB_PIXEL_AR10: case CFB_PIXEL_R210: case CFB_PIXEL_DPX0:
        out->precision = 12;
        for (int c = 0; c < 3; c++) { cw[c] = W; ch[c] = H; }
        out->frame_pitch = (fmt == CFB_PIXEL_RG48) ? W * 6 : (fmt >= CFB_PIXEL_RG30 ? W * 4 : W * 2);
        if (W % 8) { set_error("4:4:4 width %d must be a multiple of 8", W); return CFB_ERROR_UNSUPPORTED; }
        break;
    case CFB_PIXEL_BYR4:
        out->precision = 12;
        for (int c = 0; c < 4; c++) { cw[c] = W / 2; ch[c] = H / 2; }
        out->frame_pitch = W * 2;
        if (W % 16 || H % 2) { set_error("Bayer width %d must be a multiple of 16", W); return CFB_ERROR_UNSUPPORTED; }
        break;
    }
    for (int c = 0; c < nc; c++)
        if (ch[c] % 8 || ch[c] < 48) { set_error("channel height %d must be a multiple of 8 and >= 48", ch[c]); return CFB_ERROR_UNSUPPORTED; }
    out->frame_bytes = (int64_t)out->frame_pitch * H * (fmt == CFB_PIXEL_PLANAR16 ? 3 : 1);

    // coded region: per channel LL3, then highpass of level 3, 2, 1
    int64_t off = 0;
    for (int c = 0; c < nc; c++) {
        for (int k = CFB_NUM_LEVELS - 1; k >= 0; k--) {
            const int w = cw[c] >> (k + 1), h = ch[c] >> (k + 1);
            const int pitch = align16(w * 2);
            const int64_t bsz = align64((int64_t)pitch * h);
            for (int b = (k == CFB_NUM_LEVELS - 1 ? 0 : 1); b < CFB_NUM_BANDS; b++) {
                cfb_band_layout &bl = out->band[c][k][b];
                bl.offset = off; bl.width = w; bl.height = h; bl.pitch = pitch;
                off += bsz;
            }
        }
    }
    out->coded_bytes = off;
    // scratch region: LL1, LL2
    for (int c = 0; c < nc; c++) {
        for (int k = 0; k < CFB_NUM_LEVELS - 1; k++) {
            const int w = cw[c] >> (k + 1), h = ch[c] >> (k + 1);
            const int pitch = align16(w * 2);
            cfb_band_layout &bl = out->band[c][k][0];
            bl.offset = off; bl.width = w; bl.height = h; bl.pitch = pitch;
            off += align64((int64_t)pitch * h);
        }
    }
    out->total_bytes = off;
    return CFB_OK;
}

// ---------------------------------------------------------------------------
// Quantisation schedule for a fixed quality, GOP 1, progressive, rate control idle:
// Codec/quantize.c:186-584 (QuantizationSetQuality), :2865-3356 (SetTransformQuantization, spatial
// case with vbrscale 256 => VSCALE(q,m,256) = 256 q), Codec/wavelet.c:7022 (SetTransformScale:
// band scales {4,2,2,1}, {16,8,8,4}, {64,32,32,16}), Codec/wavelet.c:1710 (SetTransformPrescale).
cfb_error cfb_quant_for_quality(const cfb_frame_desc *desc, int quality, cfb_quant *out)
{
    return cfb_quant_for_source(desc, quality, 0, out);
}

// Subband divisor tables of one frame BEFORE they are mapped onto a transform: quantize.c:186 QuantizationSetQuality
// (tables, precision scaling, !progressive rescaling).  ql / qc: luma / chroma, index = subband number.
static cfb_error quant_tables(const cfb_frame_desc *desc, int quality, int interlaced, int *ql_out, int *qc_out, int *g_out,
                              int *precision_out, int *nchan_out)
{
    if (!desc) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_layout lay;
    cfb_error err = cfb_layout_compute(desc, &lay);
    if (err) return err;
    static const int luma_tab[4][17] = {
        {4, 4, 5, 5, 4, 5, 5, 9, 8, 8, 8, 4, 4, 4, 4, 4, 4},            // default
        {4, 8, 8, 12, 8, 8, 12, 9, 12, 12, 16, 32, 32, 48, 32, 32, 48},   // low
        {4, 6, 6, 8, 6, 6, 8, 5, 8, 8, 12, 16, 16, 24, 16, 16, 24},       // medium
        {4, 4, 4, 6, 4, 4, 6, 5, 8, 8, 8, 8, 8, 12, 8, 8, 12}};           // high
    static const int chroma_tab[4][17] = {
        {4, 4, 5, 5, 4, 5, 5, 9, 8, 8, 8, 8, 8, 8, 8, 8, 8},
        {4, 8, 8, 12, 8, 8, 12, 9, 12, 12, 16, 32, 32, 48, 32, 32, 48},
        {4, 6, 6, 8, 6, 6, 8, 5, 8, 8, 12, 16, 16, 32, 16, 16, 32},
        {4, 6, 6, 8, 6, 6, 8, 5, 8, 8, 8, 8, 8, 16, 8, 8, 16}};
    const int precision = lay.precision;
    // ChromaFullRes = (format >= COLOR_FORMAT_BAYER) (encoder.c:1139): true for BYR4 (104) and RG48 (120)
    const bool chroma_full = (desc->pixel_format == CFB_PIXEL_BYR4 || desc->pixel_format == CFB_PIXEL_RG48 ||
                              desc->pixel_format == CFB_PIXEL_PLANAR16 || desc->pixel_format >= CFB_PIXEL_RG30);
    if (desc->pixel_format == CFB_PIXEL_BYR4) quality |= (3 << 25);     // encoder.c:2634: no extra quant on channels 1-3
    int factor = quality & 0xff;
    const int detail = (quality & 0x0e0000) >> 17;
    int rgb_quality = (quality & 0x06000000) >> 25;
    if (rgb_quality > 2) rgb_quality = 2;
    int g = detail + 2;
    if (g > 8) g = 0;
    if (quality & 0x1f00) factor = 5;
    const int new_quality = factor;
    int limiter = 0;                                    // FSratelimiter on the first frame
    if (new_quality == 5) limiter = 8; else if (new_quality == 6) limiter = 4;
    if (factor < 1 || factor > 10) factor = 0;
    if (factor > 3) factor = 3;
    int ql[17], qc[17];
    memcpy(ql, luma_tab[factor], sizeof(ql));
    memcpy(qc, chroma_full ? luma_tab[factor] : chroma_tab[factor], sizeof(qc));
    int lowfreq = 4;
    if (precision >= 10) {
        int scale = 4 * 16;
        if (limiter > 16) limiter = 16;
        if (new_quality == 4) { lowfreq = 3; scale = 3 * 16; }
        else if (new_quality >= 5 && new_quality <= 10) { lowfreq = 2; scale = 16 + limiter * 2; }
        if (new_quality >= 5 && scale >= 4) scale >>= 1;
        if (new_quality == 10 && scale >= 6) { scale *= 2; scale /= 3; }
        if (new_quality >= 4) for (int i = 1; i < 7; i++) ql[i] = qc[i] = lowfreq;
        for (int i = 8; i < 17; i++) {
            ql[i] = (ql[i] * scale) >> 4; if (ql[i] < 2) ql[i] = 2;
            qc[i] = (qc[i] * scale) >> 4; if (qc[i] < 2) qc[i] = 2;
        }
        ql[7] = qc[7] = 4;
    }
    if (precision == 12) {
        if (new_quality >= 4) for (int i = 1; i < 7; i++) ql[i] = qc[i] = lowfreq;
        for (int i = 4; i < 7; i++) { ql[i] *= 4; qc[i] *= 4; }
        static const int gains[4] = {8, 6, 4, 4};
        const int chromagain = gains[rgb_quality];
        for (int i = 11; i < 17; i++) { ql[i] *= 4; qc[i] *= chromagain; }
    }
    if (interlaced) {       // quantize.c:490-541 (!progressive): LH of the field transform * 3/2, HL * 2/3
        ql[11] = ql[11] * 3 / 2; ql[12] = ql[12] * 2 / 3; ql[14] = ql[14] * 3 / 2; ql[15] = ql[15] * 2 / 3;
        qc[11] = qc[11] * 3 / 2; qc[12] = qc[12] * 2 / 3; qc[14] = qc[14] * 3 / 2; qc[15] = qc[15] * 2 / 3;
    }
    memcpy(ql_out, ql, sizeof(ql)); memcpy(qc_out, qc, sizeof(qc));
    *g_out = g; *precision_out = precision; *nchan_out = lay.num_channels;
    return CFB_OK;
}

cfb_error cfb_quant_for_source(const cfb_frame_desc *desc, int quality, int interlaced, cfb_quant *out)
{
    if (!desc || !out) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    int ql[17], qc[17], g = 0, precision = 0, nchan = 0;
    cfb_error err = quant_tables(desc, quality, interlaced, ql, qc, &g, &precision, &nchan);
    if (err) return err;
    memset(out, 0, sizeof(*out));
    // GOP length 1 (quantize.c:552-567)
    for (int i = 0; i < 3; i++) { ql[7 + i] = ql[11 + i]; qc[7 + i] = qc[11 + i]; }

    static const int scale[3][4] = {{4, 2, 2, 1}, {16, 8, 8, 4}, {64, 32, 32, 16}};
    out->midpoint_prequant = g;
    out->prescale[0] = 0; out->prescale[1] = 2; out->prescale[2] = (precision == 12) ? 2 : 0;
    for (int c = 0; c < nchan; c++) {
        const int *q = (c > 0) ? qc : ql;
        int subband = 1;
        for (int k = 2; k >= 0; k--) {
            out->divisor[c][k][0] = 1;
            for (int b = 1; b < 4; b++) {
                int d = (k == 0) ? q[subband] : ((q[subband] * scale[k][b]) >> 2);
                if (g) { d *= g; d /= (g - 1) * 2; } else d /= 2;
                out->divisor[c][k][b] = d;
                subband++;
            }
        }
    }
    return CFB_OK;
}

// Two-frame GOP (TRANSFORM_TYPE_FIELDPLUS): quantize.c:3480-3640 maps the subbands onto the six wavelets as
// 1-3 -> wavelet 5, 4-6 -> wavelet 4, 7 -> LL of wavelet 3 (forced to 1 for >= 10 bit, encoder.c:8487), 8-10 -> wavelet 3,
// 11-13 -> wavelet 1, 14-16 -> wavelet 0, with the band scales of wavelet.c:7135-7180 (SetTransformScale, FIELDPLUS):
// wavelet 3 {16,8,8,4}, wavelet 4 {32,16,16,8}, wavelet 5 {128,64,64,32}; frame wavelets take the table value itself.
// No GOP-1 copy of subbands 11-13 into 7-9 (quantize.c:552).  Prescale {0,0,0,0,2,0} (wavelet.c:1710, 10 bit).
cfb_error cfb_gop2_quant_for_quality(const cfb_frame_desc *desc, int quality, int interlaced, cfb_gop2_quant *out)
{
    if (!desc || !out) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    int ql[17], qc[17], g = 0, precision = 0, nchan = 0;
    cfb_error err = quant_tables(desc, quality, interlaced, ql, qc, &g, &precision, &nchan);
    if (err) return err;
    if (precision != 10) { set_error("two-frame GOP: 10-bit 4:2:2 sources"); return CFB_ERROR_UNSUPPORTED; }
    memset(out, 0, sizeof(*out));
    out->midpoint_prequant = g;
    out->prescale[4] = 2;
    static const int wavelet_of[5] = {5, 4, 3, 1, 0};
    static const int first_subband[5] = {1, 4, 8, 11, 14};
    static const int scale[6][4] = {{4, 2, 2, 1}, {4, 2, 2, 1}, {8, 4, 0, 0}, {16, 8, 8, 4}, {32, 16, 16, 8}, {128, 64, 64, 32}};
    for (int c = 0; c < nchan; c++) {
        const int *q = (c > 0) ? qc : ql;
        for (int k = 0; k < CFB_GOP2_WAVELETS; k++) out->divisor[c][k][0] = 1;
        out->divisor[c][2][1] = 1;
        for (int i = 0; i < 5; i++) {
            const int k = wavelet_of[i];
            for (int b = 1; b < 4; b++) {
                const int v = q[first_subband[i] + b - 1];
                int d = (k <= 1) ? v : ((v * scale[k][b]) >> 2);
                if (g) { d *= g; d /= (g - 1) * 2; } else d /= 2;
                out->divisor[c][k][b] = d;
            }
        }
    }
    return CFB_OK;
}

// ---------------------------------------------------------------------------
cfb_error cfb_context_create(int device, cfb_context **out)
{
    if (!out) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s): the transform path has no CPU fallback",
                  e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return CFB_ERROR_NO_DEVICE;
    }
    if (device < 0 || device >= n) { set_error("device %d out of range [0,%d)", device, n); return CFB_ERROR_INVALID_ARGUMENT; }
    // three attributes, queried once per device: cudaGetDeviceProperties costs tens of milliseconds and serialises the
    // sixteen encoder threads of an SDK pool that all create their context at the same moment
    struct DevInfo { int major = -1, minor = 0, sms = 0; };
    static DevInfo info[64];
    static std::mutex info_mu;
    DevInfo di;
    {
        std::lock_guard<std::mutex> lk(info_mu);
        if (device < 64 && info[device].major >= 0) di = info[device];
        else {
            CFB_CUDA(cudaDeviceGetAttribute(&di.major, cudaDevAttrComputeCapabilityMajor, device));
            CFB_CUDA(cudaDeviceGetAttribute(&di.minor, cudaDevAttrComputeCapabilityMinor, device));
            CFB_CUDA(cudaDeviceGetAttribute(&di.sms, cudaDevAttrMultiProcessorCount, device));
            if (device < 64) info[device] = di;
        }
    }
    if (di.major != 10) {
        set_error("device %d is sm_%d%d; this library carries sm_100a code only", device, di.major, di.minor);
        return CFB_ERROR_NO_DEVICE;
    }
    CFB_CUDA(cudaSetDevice(device));
    cfb_context *ctx = new (std::nothrow) cfb_context();
    if (!ctx) return CFB_ERROR_OUTOFMEMORY;
    ctx->device = device;
    ctx->sm_count = di.sms;
    e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->done, cudaEventBlockingSync | cudaEventDisableTiming);
    if (e != cudaSuccess) { if (ctx->stream) cudaStreamDestroy(ctx->stream); delete ctx; return cuda_fail(e, "cudaStreamCreate"); }
    *out = ctx;
    return CFB_OK;
}

void cfb_context_destroy(cfb_context *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->done) cudaEventDestroy(ctx->done);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->d_range) cudaFree(ctx->d_range);
    if (ctx->h_range) cudaFreeHost(ctx->h_range);
    delete ctx;
}

cfb_error cfb_context_synchronize(cfb_context *ctx)
{
    if (!ctx) return CFB_ERROR_INVALID_ARGUMENT;
    CFB_CUDA(cudaSetDevice(ctx->device));
    CFB_CUDA(stream_wait(ctx));
    return CFB_OK;
}

void *cfb_context_stream(cfb_context *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

cfb_error cfb_context_stats(cfb_context *ctx, cfb_stats *out)
{
    if (!ctx || !out) return CFB_ERROR_INVALID_ARGUMENT;
    out->kernel_launches = ctx->kernel_launches.load();
    out->frames_forward = ctx->frames_forward.load();
    out->frames_inverse = ctx->frames_inverse.load();
    out->h2d_bytes = ctx->h2d_bytes.load();
    out->d2h_bytes = ctx->d2h_bytes.load();
    return CFB_OK;
}

// ---------------------------------------------------------------------------
cfb_error cfb_codec_create(cfb_context *ctx, const cfb_frame_desc *desc, int max_batch, cfb_codec **out)
{
    if (!ctx || !desc || !out) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    *out = nullptr;
    if (max_batch < 1 || max_batch > CFB_MAX_BATCH) { set_error("max_batch %d out of range", max_batch); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_layout lay;
    cfb_error err = cfb_layout_compute(desc, &lay);
    if (err) return err;
    CFB_CUDA(cudaSetDevice(ctx->device));
    cfb_codec *cd = new (std::nothrow) cfb_codec();
    if (!cd) return CFB_ERROR_OUTOFMEMORY;
    cd->ctx = ctx; cd->desc = *desc; cd->layout = lay; cd->max_batch = max_batch;
    // frame staging must also hold the PLANAR16 rendition (channel planes stacked at the frame's luma pitch)
    int64_t planar_rows = 0;
    for (int c = 0; c < lay.num_channels; c++) planar_rows += lay.band[c][0][0].height * 2;
    int64_t fbytes = lay.frame_bytes;
    if (planar_rows * desc->width * 2 > fbytes) fbytes = planar_rows * desc->width * 2;
    cd->frame_stride = (size_t)((fbytes + 255) & ~(int64_t)255);
    cd->pyramid_stride = (size_t)((lay.total_bytes + 255) & ~(int64_t)255);
    cudaError_t e = cudaMalloc((void **)&cd->d_frames, cd->frame_stride * max_batch);
    if (e == cudaSuccess) e = cudaMalloc((void **)&cd->d_pyramids, cd->pyramid_stride * max_batch);
    if (e != cudaSuccess) { cfb_codec_destroy(cd); return cuda_fail(e, "cudaMalloc(codec staging)"); }
    // deterministic contents for the pitch padding (the reference's entropy coder walks it, encoder.c:5811)
    e = cudaMemsetAsync(cd->d_pyramids, 0, cd->pyramid_stride * max_batch, ctx->stream);
    if (e != cudaSuccess) { cfb_codec_destroy(cd); return cuda_fail(e, "cudaMemsetAsync"); }
    *out = cd;
    return CFB_OK;
}

void cfb_codec_destroy(cfb_codec *cd)
{
    if (!cd) return;
    if (cd->ctx) cudaSetDevice(cd->ctx->device);
    if (cd->d_frames) cudaFree(cd->d_frames);
    if (cd->d_pyramids) cudaFree(cd->d_pyramids);
    if (cd->d_carry) cudaFree(cd->d_carry);
    if (cd->d_gop) cudaFree(cd->d_gop);
    if (cd->d_curve) cudaFree(cd->d_curve);
    if (cd->d_sparse) cudaFree(cd->d_sparse);
    if (cd->d_out64) cudaFree(cd->d_out64);
    if (cd->d_status) cudaFree(cd->d_status);
    if (cd->h_headers) cudaFreeHost(cd->h_headers);
    delete cd;
}

cfb_error cfb_codec_layout(const cfb_codec *cd, cfb_layout *out)
{
    if (!cd || !out) return CFB_ERROR_INVALID_ARGUMENT;
    *out = cd->layout;
    return CFB_OK;
}

cfb_error cfb_codec_set_bayer_phase(cfb_codec *cd, int bayer_format)
{
    if (!cd || bayer_format < 0 || bayer_format > 3) { set_error("bayer format %d out of range 0..3", bayer_format); return CFB_ERROR_INVALID_ARGUMENT; }
    cd->bayer_phase = bayer_format;
    return CFB_OK;
}

cfb_error cfb_codec_set_bayer_curve(cfb_codec *cd, const uint16_t *curve, int entries)
{
    if (!cd) { set_error("null codec"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (cd->desc.pixel_format != CFB_PIXEL_BYR4) { set_error("the encode curve applies to Bayer (BYR4) codecs"); return CFB_ERROR_BADFORMAT; }
    CFB_CUDA(cudaSetDevice(cd->ctx->device));
    if (!curve) {                                   // back to "curve already applied" (encode_curve_preset)
        if (cd->d_curve) { CFB_CUDA(stream_wait(cd->ctx)); cudaFree(cd->d_curve); cd->d_curve = nullptr; }
        return CFB_OK;
    }
    if (entries != (1 << 14)) { set_error("Bayer encode curve must have 1 << 14 entries (MAX_INPUT_PRECISION, frame.c:4843)"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (!cd->d_curve) CFB_CUDA(cudaMalloc((void **)&cd->d_curve, sizeof(uint16_t) << 14));
    CFB_CUDA(cudaMemcpyAsync(cd->d_curve, curve, sizeof(uint16_t) << 14, cudaMemcpyHostToDevice, cd->ctx->stream));
    CFB_CUDA(stream_wait(cd->ctx));                 // the caller's table may go away after this call
    return CFB_OK;
}

cfb_error cfb_codec_set_level_mask(cfb_codec *cd, int forward_mask, int inverse_mask)
{
    if (!cd) return CFB_ERROR_INVALID_ARGUMENT;
    cd->fwd_mask = forward_mask & 7; cd->inv_mask = inverse_mask & 7;
    return CFB_OK;
}

cfb_error cfb_codec_set_decode_resolution(cfb_codec *cd, int resolution)
{
    if (!cd) { set_error("null codec"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (resolution < CFB_RESOLUTION_FULL || resolution > CFB_RESOLUTION_QUARTER) {
        set_error("decode resolution %d not in {full=1, half=2, quarter=3}", resolution);
        return CFB_ERROR_INVALID_ARGUMENT;
    }
    cd->decode_res = resolution;
    return CFB_OK;
}

cfb_error cfb_codec_set_interlaced(cfb_codec *cd, int interlaced)
{
    if (!cd) { set_error("null codec"); return CFB_ERROR_INVALID_ARGUMENT; }
    const int fmt = cd->desc.pixel_format;
    if (interlaced && fmt != CFB_PIXEL_YUYV && fmt != CFB_PIXEL_UYVY && fmt != CFB_PIXEL_YU64 && fmt != CFB_PIXEL_V210) {
        set_error("the interlaced (field) transform is implemented for 4:2:2 sources (YUYV, UYVY, YU64, V210)");
        return CFB_ERROR_UNSUPPORTED;
    }
    if (interlaced && !cd->d_carry) {
        // per band row and strip carry-in of the difference-coded HL band, for up to kMaxBatch frames
        const cfb_band_layout &ll = cd->layout.band[0][0][0];
        cd->carry_strips = (ll.width + kInvStrip - 1) / kInvStrip;
        const size_t bytes = (size_t)kMaxBatch * 3 * ll.height * cd->carry_strips * sizeof(int);
        CFB_CUDA(cudaSetDevice(cd->ctx->device));
        cudaError_t e = cudaMalloc((void **)&cd->d_carry, bytes);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(field carries)");
    }
    cd->interlaced = (interlaced == CFB_INTERLACED_HL_INTEGRATED) ? 2 : (interlaced ? 1 : 0);
    return CFB_OK;
}

cfb_error cfb_codec_decoded_size(const cfb_codec *cd, int *width, int *height)
{
    if (!cd || !width || !height) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (cd->decode_res == CFB_RESOLUTION_FULL) { *width = cd->desc.width; *height = cd->desc.height; }
    else {      // the lowpass image of level (res - 1) of channel 0: decoder.c:26078 (half), :17000 (quarter)
        const cfb_band_layout &ll = cd->layout.band[0][cd->decode_res - 2][0];
        *width = ll.width; *height = ll.height;
    }
    return CFB_OK;
}

void *cfb_codec_device_frame(cfb_codec *cd, int slot)
{
    return (cd && slot >= 0 && slot < cd->max_batch) ? cd->d_frames + cd->frame_stride * slot : nullptr;
}
void *cfb_codec_device_pyramid(cfb_codec *cd, int slot)
{
    return (cd && slot >= 0 && slot < cd->max_batch) ? cd->d_pyramids + cd->pyramid_stride * slot : nullptr;
}

// ---------------------------------------------------------------------------
// forward
static void fill_level_geom(const cfb_codec *cd, const cfb_quant *q, int c, int k, PlaneGeom &g)
{
    const cfb_layout &L = cd->layout;
    const cfb_band_layout &ll = L.band[c][k][0];
    g.width = ll.width * 2; g.height = ll.height * 2;
    g.out_pitch = ll.pitch;
    for (int b = 0; b < 4; b++) {
        g.band_off[b] = L.band[c][k][b].offset;
        g.q[b] = make_quant_param(q->divisor[c][k][b], q->midpoint_prequant);
    }
    // only the unprescaled planar filter ever quantises LL (spatial.c:10480; compiled out at :12942, absent at :14726)
    g.quant_ll = 0;
    if (k > 0) { g.in_off = L.band[c][k - 1][0].offset; g.in_pitch = L.band[c][k - 1][0].pitch; }
    g.pad = 0;
}

cfb_error cfb_forward_device(cfb_codec *cd, int n, const void *const *d_frames, int frame_pitch,
                             const cfb_quant *quant, void *const *d_pyramids)
{
    if (!cd || !d_frames || !quant || !d_pyramids) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (n < 1 || n > kMaxBatch) { set_error("batch %d out of range [1,%d]", n, kMaxBatch); return CFB_ERROR_INVALID_ARGUMENT; }
    if (frame_pitch < cd->layout.frame_pitch || (frame_pitch & 15)) { set_error("frame pitch %d must be >= %d and 16-byte aligned", frame_pitch, cd->layout.frame_pitch); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_context *ctx = cd->ctx;
    const cfb_layout &L = cd->layout;
    const int fmt = cd->desc.pixel_format;
    CFB_CUDA(cudaSetDevice(ctx->device));
    for (int i = 0; i < n; i++)
        if (!d_frames[i] || !d_pyramids[i] || ((uintptr_t)d_frames[i] & 15) || ((uintptr_t)d_pyramids[i] & 15)) {
            set_error("frame/pyramid %d null or not 16-byte aligned", i);
            return CFB_ERROR_INVALID_ARGUMENT;
        }
    for (int lvl = 0; lvl < CFB_NUM_LEVELS; lvl++)
        if (quant->prescale[lvl] != 0 && quant->prescale[lvl] != 2) { set_error("prescale %d unsupported", quant->prescale[lvl]); return CFB_ERROR_UNSUPPORTED; }

    FwdParams p;
    memset(&p, 0, sizeof(p));
    p.nchan = L.num_channels; p.nframes = n;
    // ---- level 1 ----
    if (!(cd->fwd_mask & 1)) {
    } else if (fmt == CFB_PIXEL_YUYV || fmt == CFB_PIXEL_UYVY) {
        for (int c = 0; c < 3; c++) { fill_level_geom(cd, quant, c, 0, p.ch[c]); p.ch[c].in_off = 0; p.ch[c].in_pitch = frame_pitch; }
        for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_frames[i]; p.out_base[i] = (unsigned char *)d_pyramids[i]; }
        p.shift = L.precision - 8; p.uyvy = (fmt == CFB_PIXEL_UYVY);
        p.th = pick_th((p.ch[0].width + kStripIn - 1) / kStripIn, p.ch[0].height / 2, n, ctx->sm_count);
        if (cd->interlaced) {
            for (int c = 0; c < 3; c++)
                p.ch[c].q[2] = make_quant_param(quant->divisor[c][0][2], quant->midpoint_prequant, true);
            CFB_CUDA(launch_fwd_422_fields(p, ctx->stream));
        } else {
            CFB_CUDA(launch_fwd_422(p, ctx->stream));
        }
        ctx->kernel_launches++;
    } else if (fmt == CFB_PIXEL_YU64 || fmt == CFB_PIXEL_V210) {
        for (int c = 0; c < 3; c++) {
            fill_level_geom(cd, quant, c, 0, p.ch[c]); p.ch[c].in_off = 0; p.ch[c].in_pitch = frame_pitch;
            p.ch[c].quant_ll = quant->divisor[c][0][0] > 1;         // planar filter: LL quantised when its divisor > 1
        }
        for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_frames[i]; p.out_base[i] = (unsigned char *)d_pyramids[i]; }
        p.shift = 16 - L.precision;
        p.th = pick_th((p.ch[0].width + kStripIn - 1) / kStripIn, p.ch[0].height / 2, n, ctx->sm_count);
        if (cd->interlaced) {
            // planar field transform (filter.c:273): LH rounded with divisor / 2 (spatial.c:5856), HL as the packed path
            for (int c = 0; c < 3; c++) {
                if (quant->divisor[c][0][0] > 1) { set_error("interlaced 16-bit / 10-bit 4:2:2 sources: a quantised level-1 lowpass band is not supported"); return CFB_ERROR_UNSUPPORTED; }
                p.ch[c].q[1] = make_quant_param(quant->divisor[c][0][1], 2, true);
                p.ch[c].q[2] = make_quant_param(quant->divisor[c][0][2], quant->midpoint_prequant, true);
            }
            CFB_CUDA(launch_fwd_422_fields_src(p, fmt == CFB_PIXEL_V210 ? 1 : 0, ctx->stream));
        } else
        CFB_CUDA(fmt == CFB_PIXEL_V210 ? launch_fwd_v210(p, ctx->stream) : launch_fwd_yu64(p, ctx->stream));
        ctx->kernel_launches++;
    } else if (fmt == CFB_PIXEL_PLANAR16) {
        for (int c = 0; c < 3; c++) {
            fill_level_geom(cd, quant, c, 0, p.ch[c]);
            p.ch[c].in_pitch = frame_pitch; p.ch[c].in_off = (long long)c * frame_pitch * cd->desc.height;
            p.ch[c].quant_ll = quant->divisor[c][0][0] > 1;
        }
        for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_frames[i]; p.out_base[i] = (unsigned char *)d_pyramids[i]; }
        p.th = pick_th((p.ch[0].width + kStripIn - 1) / kStripIn, p.ch[0].height / 2, n * 3, ctx->sm_count);
        CFB_CUDA(launch_fwd_plane(p, quant->prescale[0], ctx->stream));
        ctx->kernel_launches++;
    } else if (fmt == CFB_PIXEL_RG48) {
        // channel order of the reference: plane 0 = G, 1 = R, 2 = B (Codec/frame.c:6155-6157); all three channels come out
        // of one pass over the 48-bit pixel groups (k_fwd_tma<SrcRG48>)
        for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_frames[i]; p.out_base[i] = (unsigned char *)d_pyramids[i]; }
        p.shift = 16 - L.precision;
        for (int c = 0; c < 3; c++) {
            fill_level_geom(cd, quant, c, 0, p.ch[c]);
            p.ch[c].in_off = 0; p.ch[c].in_pitch = frame_pitch;
            p.ch[c].quant_ll = quant->divisor[c][0][0] > 1;
        }
        p.th = pick_th((p.ch[0].width + kStripIn - 1) / kStripIn, p.ch[0].height / 2, n * 3, ctx->sm_count);
        if (getenv("CFB_FWDPLANE") && !strcmp(getenv("CFB_FWDPLANE"), "r1")) {
            static const int sel_of_channel[3] = {1, 0, 2};
            for (int c = 0; c < 3; c++) {
                FwdParams q = p;
                q.nchan = 1; q.ch[0] = p.ch[c];
                q.th = pick_th((q.ch[0].width + kStripIn - 1) / kStripIn, q.ch[0].height / 2, n, ctx->sm_count);
                CFB_CUDA(launch_fwd_rg48(q, sel_of_channel[c], ctx->stream));
                ctx->kernel_launches++;
            }
        } else {
            CFB_CUDA(launch_fwd_rg48_all(p, ctx->stream));
            ctx->kernel_launches += 4;
        }
    } else if (fmt >= CFB_PIXEL_RG30 && fmt <= CFB_PIXEL_DPX0) {
        // planes G, R, B; field position of each inside the (possibly byte-swapped) word: spatial.c:2118-2268
        static const int pos_rgb[5][3] = {{0, 10, 20}, {0, 10, 20}, {20, 10, 0}, {20, 10, 0}, {22, 12, 2}};   // R, G, B of RG30 AB10 AR10 R210 DPX0
        static const int chan_is[3] = {1, 0, 2};                                                              // channel 0 = G, 1 = R, 2 = B
        for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_frames[i]; p.out_base[i] = (unsigned char *)d_pyramids[i]; }
        for (int c = 0; c < 3; c++) {
            FwdParams q = p;
            q.nchan = 1;
            fill_level_geom(cd, quant, c, 0, q.ch[0]);
            q.ch[0].in_off = 0; q.ch[0].in_pitch = frame_pitch;
            q.ch[0].quant_ll = quant->divisor[c][0][0] > 1;
            q.shift = L.precision - 10;
            q.uyvy = (fmt == CFB_PIXEL_R210 || fmt == CFB_PIXEL_DPX0);
            q.pad = pos_rgb[fmt - CFB_PIXEL_RG30][chan_is[c]];
            q.th = pick_th((q.ch[0].width + kStripIn - 1) / kStripIn, q.ch[0].height / 2, n, ctx->sm_count);
            CFB_CUDA(launch_fwd_rgb30(q, ctx->stream));
            ctx->kernel_launches++;
        }
    } else if (fmt == CFB_PIXEL_BYR4) {
        for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_frames[i]; p.out_base[i] = (unsigned char *)d_pyramids[i]; }
        for (int c = 0; c < 4; c++) {
            fill_level_geom(cd, quant, c, 0, p.ch[c]);
            p.ch[c].in_off = 0; p.ch[c].in_pitch = frame_pitch;      // bytes per Bayer line
            p.ch[c].quant_ll = quant->divisor[c][0][0] > 1;
        }
        p.shift = 16 - L.precision; p.uyvy = cd->bayer_phase; p.lut = cd->d_curve;
        p.th = pick_th((p.ch[0].width + kStripIn - 1) / kStripIn * 4, p.ch[0].height / 2, n, ctx->sm_count);
        CFB_CUDA(launch_fwd_byr4(p, ctx->stream));
        ctx->kernel_launches++;
    } else {
        set_error("forward level 1 for pixel format %d not implemented yet", fmt);
        return CFB_ERROR_UNSUPPORTED;
    }
    // ---- levels 2, 3: input = LL of the previous level inside the pyramid ----
    for (int k = 1; k < CFB_NUM_LEVELS; k++) {
        if (!(cd->fwd_mask & (1 << k))) continue;
        for (int c = 0; c < L.num_channels; c++) {
            fill_level_geom(cd, quant, c, k, p.ch[c]);
            p.ch[c].quant_ll = (quant->prescale[k] == 0) && quant->divisor[c][k][0] > 1;
        }
        for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_pyramids[i]; p.out_base[i] = (unsigned char *)d_pyramids[i]; }
        int maxw = 0, maxoh = 0;
        for (int c = 0; c < L.num_channels; c++) { if (p.ch[c].width > maxw) maxw = p.ch[c].width; if (p.ch[c].height / 2 > maxoh) maxoh = p.ch[c].height / 2; }
        p.th = pick_th((maxw + kStripIn - 1) / kStripIn, maxoh, n * L.num_channels, ctx->sm_count);
        // the LL bands of every unsigned source format are non-negative (<= 4 * 4095): the prescaled level may use its
        // packed non-negative taps; caller-supplied planes (CFB_PIXEL_PLANAR16) carry no such promise
        p.pad = (fmt != CFB_PIXEL_PLANAR16) ? 1 : 0;
        CFB_CUDA(launch_fwd_plane(p, quant->prescale[k], ctx->stream));
        ctx->kernel_launches++;
    }
    ctx->frames_forward += n;
    return CFB_OK;
}

cfb_error cfb_forward_host(cfb_codec *cd, int n, const void *const *h_frames, int frame_pitch,
                           const cfb_quant *quant, void *const *h_coded)
{
    if (!cd || !h_frames || !quant || !h_coded) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_context *ctx = cd->ctx;
    cfb_error err = stage_fwd_upload(cd, n, h_frames, frame_pitch, ctx->stream);
    if (!err) err = stage_fwd_compute(cd, n, quant, false);
    if (!err) err = stage_fwd_download(cd, n, h_coded, false, 0, ctx->stream);
    if (err) return err;
    CFB_CUDA(stream_wait(ctx));
    return CFB_OK;
}

}  // extern "C"

namespace cfb {

cfb_error stage_fwd_upload(cfb_codec *cd, int n, const void *const *h_frames, int frame_pitch, cudaStream_t s)
{
    if (!cd || !h_frames) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (n < 1 || n > cd->max_batch) { set_error("batch %d exceeds codec max_batch %d", n, cd->max_batch); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_context *ctx = cd->ctx;
    const cfb_layout &L = cd->layout;
    if (frame_pitch < L.frame_pitch || (frame_pitch & 15)) { set_error("frame pitch %d must be >= %d and 16-byte aligned", frame_pitch, L.frame_pitch); return CFB_ERROR_INVALID_ARGUMENT; }
    CFB_CUDA(cudaSetDevice(ctx->device));
    const int rows = (int)(L.frame_bytes / L.frame_pitch);
    for (int i = 0; i < n; i++) {
        if (!h_frames[i]) { set_error("null host buffer %d", i); return CFB_ERROR_INVALID_ARGUMENT; }
        if (frame_pitch == L.frame_pitch)       // contiguous on both sides: one linear copy
            CFB_CUDA(cudaMemcpyAsync(cfb_codec_device_frame(cd, i), h_frames[i], (size_t)L.frame_pitch * rows, cudaMemcpyHostToDevice, s));
        else
            CFB_CUDA(cudaMemcpy2DAsync(cfb_codec_device_frame(cd, i), L.frame_pitch, h_frames[i], frame_pitch, L.frame_pitch, rows,
                                       cudaMemcpyHostToDevice, s));
        ctx->h2d_bytes += (uint64_t)L.frame_bytes;
    }
    return CFB_OK;
}

cfb_error stage_fwd_compute(cfb_codec *cd, int n, const cfb_quant *quant, bool sparse)
{
    if (!cd || !quant) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (n < 1 || n > cd->max_batch) { set_error("batch %d exceeds codec max_batch %d", n, cd->max_batch); return CFB_ERROR_INVALID_ARGUMENT; }
    const void *dfr[kMaxBatch];
    void *dpy[kMaxBatch];
    for (int i = 0; i < n; i++) { dfr[i] = cfb_codec_device_frame(cd, i); dpy[i] = cfb_codec_device_pyramid(cd, i); }
    cfb_error err = cfb_forward_device(cd, n, dfr, cd->layout.frame_pitch, quant, dpy);
    if (!err && sparse) err = sparse_compact_device(cd, n);
    return err;
}

}  // namespace cfb

extern "C" {

// ---------------------------------------------------------------------------
// inverse
static void fill_inv_geom(const cfb_codec *cd, const cfb_quant *q, int c, int k, InvGeom &g)
{
    const cfb_layout &L = cd->layout;
    const cfb_band_layout &ll = L.band[c][k][0];
    g.width = ll.width; g.height = ll.height; g.pitch = ll.pitch;
    for (int b = 0; b < 4; b++) {
        g.band_off[b] = L.band[c][k][b].offset;
        const int d = q->divisor[c][k][b];
        g.dq[b] = d > 1 ? d : 1;
    }
    g.dq[0] = 1;        // LL is carried unquantised through the pyramid (only LL3 is coded, raw)
    if (k > 0) { g.out_off = L.band[c][k - 1][0].offset; g.out_pitch = L.band[c][k - 1][0].pitch; }
}

cfb_error cfb_inverse_device(cfb_codec *cd, int n, void *const *d_pyramids, const cfb_quant *quant,
                             int out_format, void *const *d_frames, int frame_pitch)
{
    if (!cd || !d_pyramids || !quant || !d_frames) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (n < 1 || n > kMaxBatch) { set_error("batch %d out of range [1,%d]", n, kMaxBatch); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_context *ctx = cd->ctx;
    const cfb_layout &L = cd->layout;
    const int fmt = cd->desc.pixel_format;
    const bool is422 = (fmt == CFB_PIXEL_YUYV || fmt == CFB_PIXEL_UYVY || fmt == CFB_PIXEL_YU64 || fmt == CFB_PIXEL_V210);
    int out_w = 0, out_h = 0;
    cfb_codec_decoded_size(cd, &out_w, &out_h);
    const bool is444 = (fmt == CFB_PIXEL_RG48 || fmt == CFB_PIXEL_PLANAR16 || (fmt >= CFB_PIXEL_RG30 && fmt <= CFB_PIXEL_DPX0));
    if (out_format == CFB_PIXEL_YUYV || out_format == CFB_PIXEL_UYVY) {
        if (!is422) { set_error("8-bit 4:2:2 output needs a 4:2:2 codec"); return CFB_ERROR_BADFORMAT; }
        if (frame_pitch < out_w * 2 || (frame_pitch & 15)) { set_error("bad output pitch %d", frame_pitch); return CFB_ERROR_INVALID_ARGUMENT; }
    } else if (out_format == CFB_PIXEL_YU64 || out_format == CFB_PIXEL_RG48) {
        // 16-bit packed outputs of the final level (the reference's ...ToRow16u family): full resolution, progressive
        if (out_format == CFB_PIXEL_YU64 ? !is422 : !is444) { set_error("YU64 output needs a 4:2:2 codec, RG48 output a 4:4:4 codec"); return CFB_ERROR_BADFORMAT; }
        if (cd->decode_res != CFB_RESOLUTION_FULL || cd->interlaced) { set_error("16-bit packed output: full-resolution progressive decode only"); return CFB_ERROR_UNSUPPORTED; }
        const int bpp = (out_format == CFB_PIXEL_YU64) ? 4 : 6;
        if (frame_pitch < out_w * bpp || (frame_pitch & 15)) { set_error("bad output pitch %d", frame_pitch); return CFB_ERROR_INVALID_ARGUMENT; }
        for (int c = 0; c < L.num_channels; c++)
            if (L.band[c][0][0].width < 16) { set_error("16-bit packed output needs level-1 bands at least 16 coefficients wide"); return CFB_ERROR_UNSUPPORTED; }
    } else if (out_format == CFB_PIXEL_V210) {
        // 10-bit packed 4:2:2: the YU64 rows >> 6 (decoder.c:26292 -> convert.c:13526 ConvertPlanarYUVToV210).  The reference
        // renders V210 from a field transform only through its active-metadata path (decoder.c:26413), and reduced
        // resolutions through ConvertLowpass16s10bitToV210 (decoder.c:23054): neither is built here
        if (!is422) { set_error("V210 output needs a 4:2:2 codec"); return CFB_ERROR_BADFORMAT; }
        if (cd->decode_res != CFB_RESOLUTION_FULL || cd->interlaced) { set_error("V210 output: full-resolution progressive decode only"); return CFB_ERROR_UNSUPPORTED; }
        if (frame_pitch < v210_row_bytes(out_w) || (frame_pitch & 15)) { set_error("bad output pitch %d", frame_pitch); return CFB_ERROR_INVALID_ARGUMENT; }
    } else if (out_format >= CFB_PIXEL_RG30 && out_format <= CFB_PIXEL_DPX0) {
        // 10-bit packed RGB of an RGB 4:4:4 sample (decoder.c:26893 -> InvertHorizontalStrip16s.c:14812 ...RGB2RG30)
        if (!is444 || L.num_channels != 3 || L.precision != 12) { set_error("10-bit RGB output needs a three-channel 12-bit 4:4:4 codec"); return CFB_ERROR_BADFORMAT; }
        if (cd->decode_res != CFB_RESOLUTION_FULL || cd->interlaced) { set_error("10-bit RGB output: full-resolution progressive decode only"); return CFB_ERROR_UNSUPPORTED; }
        if (frame_pitch < out_w * 4 || (frame_pitch & 15)) { set_error("bad output pitch %d", frame_pitch); return CFB_ERROR_INVALID_ARGUMENT; }
        for (int c = 0; c < L.num_channels; c++)
            if (L.band[c][0][0].width < 16) { set_error("10-bit RGB output needs level-1 bands at least 16 coefficients wide"); return CFB_ERROR_UNSUPPORTED; }
    } else if (out_format == CFB_PIXEL_B64A) {
        // 16-bit A,R,G,B of an RGB 4:4:4 sample (decoder.c:26862 -> InvertHorizontalStrip16s.c:13298 ...RGB2B64A)
        if (!is444 || L.num_channels != 3 || L.precision != 12) { set_error("B64A output needs a three-channel 12-bit 4:4:4 codec"); return CFB_ERROR_BADFORMAT; }
        if (cd->decode_res != CFB_RESOLUTION_FULL || cd->interlaced) { set_error("B64A output: full-resolution progressive decode only"); return CFB_ERROR_UNSUPPORTED; }
        if (frame_pitch < out_w * 8 || (frame_pitch & 15)) { set_error("bad output pitch %d", frame_pitch); return CFB_ERROR_INVALID_ARGUMENT; }
        for (int c = 0; c < L.num_channels; c++)
            if (L.band[c][0][0].width < 16) { set_error("B64A output needs level-1 bands at least 16 coefficients wide"); return CFB_ERROR_UNSUPPORTED; }
    } else if (out_format == CFB_PIXEL_PLANAR16) {
        if (frame_pitch < out_w * 2 || (frame_pitch & 15)) { set_error("bad output pitch %d", frame_pitch); return CFB_ERROR_INVALID_ARGUMENT; }
    } else { set_error("output format %d not implemented", out_format); return CFB_ERROR_UNSUPPORTED; }
    for (int i = 0; i < n; i++)
        if (!d_frames[i] || !d_pyramids[i] || ((uintptr_t)d_frames[i] & 15) || ((uintptr_t)d_pyramids[i] & 15)) {
            set_error("frame/pyramid %d null or not 16-byte aligned", i);
            return CFB_ERROR_INVALID_ARGUMENT;
        }
    CFB_CUDA(cudaSetDevice(ctx->device));

    InvParams p;
    memset(&p, 0, sizeof(p));
    p.nchan = L.num_channels; p.nframes = n;
    // levels 3 -> 2 -> 1: output = LL of the level below, inside the pyramid
    for (int k = CFB_NUM_LEVELS - 1; k >= 1 && k >= cd->decode_res - 1; k--) {
        if (!(cd->inv_mask & (1 << k))) continue;
        int maxw = 0, maxh = 0;
        for (int c = 0; c < L.num_channels; c++) {
            fill_inv_geom(cd, quant, c, k, p.ch[c]);
            if (p.ch[c].width > maxw) maxw = p.ch[c].width;
            if (p.ch[c].height > maxh) maxh = p.ch[c].height;
        }
        for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_pyramids[i]; p.out_base[i] = (unsigned char *)d_pyramids[i]; }
        p.th = pick_th((maxw + kInvStrip - 1) / kInvStrip, maxh, n * L.num_channels, ctx->sm_count);
        CFB_CUDA(launch_inv_plane(p, quant->prescale[k], ctx->stream));
        ctx->kernel_launches++;
    }
    if (cd->decode_res != CFB_RESOLUTION_FULL) {
        // reduced resolution: the output is the lowpass image of level kk+1 (decoder.c:26078-26160 half,
        // decoder.c:11818 + :17000 quarter); the levels below are never inverted
        const int kk = cd->decode_res - 2;
        for (int c = 0; c < L.num_channels; c++) fill_inv_geom(cd, quant, c, kk, p.ch[c]);
        if (out_format == CFB_PIXEL_PLANAR16) {
            for (int i = 0; i < n; i++) {
                long long off = 0;
                for (int c = 0; c < L.num_channels; c++) {
                    const InvGeom &g = p.ch[c];
                    CFB_CUDA(cudaMemcpy2DAsync((unsigned char *)d_frames[i] + off, frame_pitch,
                                               (const unsigned char *)d_pyramids[i] + g.band_off[0], g.pitch,
                                               (size_t)g.width * 2, g.height, cudaMemcpyDeviceToDevice, ctx->stream));
                    off += (long long)frame_pitch * g.height;
                }
            }
        } else {
            for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_pyramids[i]; p.out_base[i] = (unsigned char *)d_frames[i]; }
            p.ch[0].out_pitch = frame_pitch;
            p.shift = 4;                                        // PRESCALE_LUMA10 / descale (frame.c:11742, temporal.c:11373)
            p.pad = (cd->decode_res == CFB_RESOLUTION_QUARTER); // unsigned shift + packus in the quarter path
            p.uyvy = (out_format == CFB_PIXEL_UYVY);
            CFB_CUDA(launch_lowpass_422(p, ctx->stream));
            ctx->kernel_launches++;
        }
        ctx->frames_inverse += n;
        return CFB_OK;
    }
    // level 1 -> pixels
    if (!(cd->inv_mask & 1)) { ctx->frames_inverse += n; return CFB_OK; }
    for (int c = 0; c < L.num_channels; c++) fill_inv_geom(cd, quant, c, 0, p.ch[c]);
    for (int i = 0; i < n; i++) { p.in_base[i] = (const unsigned char *)d_pyramids[i]; p.out_base[i] = (unsigned char *)d_frames[i]; }
    if (cd->interlaced) {
        FieldsAux aux;
        aux.carry = cd->d_carry; aux.nstrips = cd->carry_strips; aux.maxh = p.ch[0].height; aux.pad = (cd->interlaced == 2);
        long long off = 0;
        for (int c = 0; c < 3; c++) {
            p.ch[c].out_pitch = frame_pitch;
            p.ch[c].out_off = (out_format == CFB_PIXEL_PLANAR16) ? off : 0;
            off += (long long)frame_pitch * p.ch[c].height * 2;
        }
        p.shift = L.precision - 8; p.uyvy = (out_format == CFB_PIXEL_UYVY);
        p.th = pick_th((p.ch[0].width + kInvStrip - 1) / kInvStrip, p.ch[0].height, n, ctx->sm_count);
        CFB_CUDA(launch_inv_fields(p, aux, out_format == CFB_PIXEL_PLANAR16, ctx->stream));
        ctx->kernel_launches++;
    } else if (out_format == CFB_PIXEL_PLANAR16) {
        // planes stacked channel after channel, each channel at its own width, pitch = frame_pitch
        long long off = 0;
        int maxw = 0, maxh = 0;
        for (int c = 0; c < L.num_channels; c++) {
            p.ch[c].out_off = off; p.ch[c].out_pitch = frame_pitch;
            off += (long long)frame_pitch * p.ch[c].height * 2;
            if (p.ch[c].width > maxw) maxw = p.ch[c].width;
            if (p.ch[c].height > maxh) maxh = p.ch[c].height;
        }
        p.th = pick_th((maxw + kInvStrip - 1) / kInvStrip, maxh, n * L.num_channels, ctx->sm_count);
        CFB_CUDA(launch_inv_plane(p, quant->prescale[0], ctx->stream));
    } else {
        for (int c = 0; c < 3; c++) { p.ch[c].out_off = 0; p.ch[c].out_pitch = frame_pitch; }
        p.shift = L.precision - 8; p.uyvy = (out_format == CFB_PIXEL_UYVY);
        p.th = pick_th((p.ch[0].width + kInvStrip - 1) / kInvStrip, p.ch[0].height, n, ctx->sm_count);
        if (out_format >= CFB_PIXEL_RG30 && out_format <= CFB_PIXEL_DPX0) {
            // component positions and byte order as on the encode side (spatial.c:2118-2268 / InvertHorizontalStrip16s.c:15562-15613)
            static const int pos_rgb[5][3] = {{0, 10, 20}, {0, 10, 20}, {20, 10, 0}, {20, 10, 0}, {22, 12, 2}};   // R, G, B of RG30 AB10 AR10 R210 DPX0
            for (int c = 0; c < 3; c++) p.tail_col[c] = pos_rgb[out_format - CFB_PIXEL_RG30][c];
            p.uyvy = (out_format == CFB_PIXEL_R210 || out_format == CFB_PIXEL_DPX0);
            p.up_shift = 0; p.hi_simd = (1 << L.precision) - 1;
            CFB_CUDA(launch_inv_444_rg48(p, 2, ctx->stream));
        } else if (out_format == CFB_PIXEL_B64A) {
            // InvertHorizontalStrip16s.c:13319: the 8-column loop runs up to post_column = width - width % 8 and always leaves the
            // right border column to the scalar code, which saturates at 65535 instead of the 12-bit maximum
            p.up_shift = 16 - L.precision;
            p.hi_simd = ((1 << L.precision) - 1) << p.up_shift;
            for (int c = 0; c < 3; c++) {
                const int w = p.ch[c].width;
                p.tail_col[c] = (w % 8) ? w - w % 8 : w - 1;
            }
            CFB_CUDA(launch_inv_444_rg48(p, 1, ctx->stream));
        } else if (out_format == CFB_PIXEL_YU64 || out_format == CFB_PIXEL_RG48) {
            p.up_shift = 16 - L.precision;
            p.hi_simd = ((1 << L.precision) - 1) << p.up_shift;
            for (int c = 0; c < 3; c++) {
                // InvertHorizontalStrip16s.c:16589-16594: the 8-column loop ends at post_column = width - width % 8 - 16; one more
                // group of 7 columns is produced with the SIMD rule, everything right of it by the scalar code
                const int w = p.ch[c].width;
                p.tail_col[c] = (w - (w % 8) - 16) + 7;
            }
            if (out_format == CFB_PIXEL_RG48) CFB_CUDA(launch_inv_444_rg48(p, 0, ctx->stream));
            else CFB_CUDA(launch_inv_422(p, kInv422OutYU64, ctx->stream));
        } else if (out_format == CFB_PIXEL_V210) {
            CFB_CUDA(launch_inv_422(p, kInv422OutV210, ctx->stream));
        } else {
            CFB_CUDA(launch_inv_422(p, kInv422Out8, ctx->stream));
        }
    }
    ctx->kernel_launches++;
    ctx->frames_inverse += n;
    return CFB_OK;
}

cfb_error cfb_inverse_host(cfb_codec *cd, int n, const void *const *h_coded, const cfb_quant *quant,
                           int out_format, void *const *h_frames, int frame_pitch)
{
    if (!cd || !h_coded || !quant || !h_frames) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_context *ctx = cd->ctx;
    cfb_error err = stage_inv_upload(cd, n, h_coded, false, ctx->stream);
    if (!err) err = stage_inv_compute(cd, n, quant, out_format, false);
    if (!err) err = stage_inv_download(cd, n, h_frames, frame_pitch, out_format, ctx->stream);
    if (err) return err;
    CFB_CUDA(stream_wait(ctx));
    return CFB_OK;
}

}  // extern "C"

namespace cfb {

// geometry of what the inverse writes into the device frame staging / the caller's buffer at the current resolution
static cfb_error inv_output_geometry(const cfb_codec *cd, int out_format, int *rows, int *rowbytes, int *dpitch)
{
    const cfb_layout &L = cd->layout;
    int out_w = 0, out_h = 0;
    cfb_codec_decoded_size(cd, &out_w, &out_h);
    const int kk = cd->decode_res - 1;          // lowest level that is inverted (0 = all three)
    const bool rgb30 = (out_format >= CFB_PIXEL_RG30 && out_format <= CFB_PIXEL_DPX0);
    const int bpp = (out_format == CFB_PIXEL_YU64 || rgb30) ? 4 : (out_format == CFB_PIXEL_RG48) ? 6 : (out_format == CFB_PIXEL_B64A) ? 8 : 2;
    *rowbytes = (out_format == CFB_PIXEL_V210) ? v210_row_bytes(out_w) : out_w * bpp;
    *dpitch = (*rowbytes + 15) & ~15;
    // a 4:2:2 codec's staging holds at least the three planar16 planes (4 W bytes per row), more than V210's 8 W / 3 + 16
    if ((out_format == CFB_PIXEL_YU64 || out_format == CFB_PIXEL_RG48 || rgb30 || out_format == CFB_PIXEL_V210) &&
        (size_t)*dpitch * out_h > cd->frame_stride) {
        set_error("packed output does not fit the codec's frame staging"); return CFB_ERROR_UNSUPPORTED;
    }
    if (out_format == CFB_PIXEL_PLANAR16) {
        *rows = 0;
        for (int c = 0; c < L.num_channels; c++) *rows += kk ? L.band[c][kk - 1][0].height : L.band[c][0][0].height * 2;
        if ((size_t)*dpitch * *rows > cd->frame_stride) { set_error("planar16 output does not fit the codec's frame staging"); return CFB_ERROR_UNSUPPORTED; }
    } else {
        *rows = out_h;
    }
    return CFB_OK;
}

// device frame slot the inverse writes for `out_format` (B64A: its own, wider staging, allocated on first use)
static cfb_error inv_frame_slot(cfb_codec *cd, int out_format, int dpitch, int rows, int slot, unsigned char **out)
{
    if (out_format != CFB_PIXEL_B64A) { *out = (unsigned char *)cfb_codec_device_frame(cd, slot); return CFB_OK; }
    const size_t stride = ((size_t)dpitch * rows + 255) & ~(size_t)255;
    if (!cd->d_out64 || cd->out64_stride != stride) {
        CFB_CUDA(cudaSetDevice(cd->ctx->device));
        if (cd->d_out64) { CFB_CUDA(stream_wait(cd->ctx)); cudaFree(cd->d_out64); cd->d_out64 = nullptr; }
        CFB_CUDA(cudaMalloc((void **)&cd->d_out64, stride * cd->max_batch));
        cd->out64_stride = stride;
    }
    *out = cd->d_out64 + stride * slot;
    return CFB_OK;
}

cfb_error stage_inv_upload(cfb_codec *cd, int n, const void *const *h_in, bool sparse, cudaStream_t s)
{
    if (!cd || !h_in) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (n < 1 || n > cd->max_batch) { set_error("batch %d exceeds codec max_batch %d", n, cd->max_batch); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_context *ctx = cd->ctx;
    const cfb_layout &L = cd->layout;
    CFB_CUDA(cudaSetDevice(ctx->device));
    if (sparse) return sparse_upload(cd, n, h_in, s);
    const int kk = cd->decode_res - 1;
    for (int i = 0; i < n; i++) {
        if (!h_in[i]) { set_error("null host buffer %d", i); return CFB_ERROR_INVALID_ARGUMENT; }
        void *dpy = cfb_codec_device_pyramid(cd, i);
        if (kk == 0) {
            CFB_CUDA(cudaMemcpyAsync(dpy, h_in[i], (size_t)L.coded_bytes, cudaMemcpyHostToDevice, s));
            ctx->h2d_bytes += (uint64_t)L.coded_bytes;
        } else {
            // reduced resolution: each channel's bands are laid out LL3, level 3, level 2, level 1, so the levels a
            // half/quarter decode reads are one contiguous prefix per channel (the decoder skips the rest of the
            // sample the same way: decoder.c:1965-1984 decoded_subband_mask_half / _quarter)
            for (int c = 0; c < L.num_channels; c++) {
                const int64_t lo = L.band[c][CFB_NUM_LEVELS - 1][0].offset;
                const cfb_band_layout &last = L.band[c][kk][3];
                const int64_t hi = last.offset + (int64_t)last.pitch * last.height;
                CFB_CUDA(cudaMemcpyAsync((unsigned char *)dpy + lo, (const unsigned char *)h_in[i] + lo, (size_t)(hi - lo),
                                         cudaMemcpyHostToDevice, s));
                ctx->h2d_bytes += (uint64_t)(hi - lo);
            }
        }
    }
    return CFB_OK;
}

cfb_error stage_inv_compute(cfb_codec *cd, int n, const cfb_quant *quant, int out_format, bool sparse)
{
    if (!cd || !quant) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (n < 1 || n > cd->max_batch) { set_error("batch %d exceeds codec max_batch %d", n, cd->max_batch); return CFB_ERROR_INVALID_ARGUMENT; }
    int rows, rowbytes, dpitch;
    cfb_error err = inv_output_geometry(cd, out_format, &rows, &rowbytes, &dpitch);
    if (err) return err;
    if (sparse) { err = sparse_expand_device(cd, n); if (err) return err; }
    void *dpy[kMaxBatch], *dfr[kMaxBatch];
    for (int i = 0; i < n; i++) {
        dpy[i] = cfb_codec_device_pyramid(cd, i);
        unsigned char *slot = nullptr;
        err = inv_frame_slot(cd, out_format, dpitch, rows, i, &slot);
        if (err) return err;
        dfr[i] = slot;
    }
    return cfb_inverse_device(cd, n, dpy, quant, out_format, dfr, dpitch);
}

cfb_error stage_inv_download(cfb_codec *cd, int n, void *const *h_frames, int frame_pitch, int out_format, cudaStream_t s)
{
    if (!cd || !h_frames) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (n < 1 || n > cd->max_batch) { set_error("batch %d exceeds codec max_batch %d", n, cd->max_batch); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_context *ctx = cd->ctx;
    int rows, rowbytes, dpitch;
    cfb_error err = inv_output_geometry(cd, out_format, &rows, &rowbytes, &dpitch);
    if (err) return err;
    if (frame_pitch < rowbytes) { set_error("output pitch %d smaller than a row (%d bytes)", frame_pitch, rowbytes); return CFB_ERROR_INVALID_ARGUMENT; }
    CFB_CUDA(cudaSetDevice(ctx->device));
    for (int i = 0; i < n; i++) {
        if (!h_frames[i]) { set_error("null host buffer %d", i); return CFB_ERROR_INVALID_ARGUMENT; }
        unsigned char *slot = nullptr;
        err = inv_frame_slot(cd, out_format, dpitch, rows, i, &slot);
        if (err) return err;
        if (frame_pitch == rowbytes && dpitch == rowbytes)
            CFB_CUDA(cudaMemcpyAsync(h_frames[i], slot, (size_t)rowbytes * rows, cudaMemcpyDeviceToHost, s));
        else
            CFB_CUDA(cudaMemcpy2DAsync(h_frames[i], frame_pitch, slot, dpitch, rowbytes, rows, cudaMemcpyDeviceToHost, s));
        ctx->d2h_bytes += (uint64_t)rowbytes * rows;
    }
    return CFB_OK;
}

cfb_error stage_fwd_download(cfb_codec *cd, int n, void *const *h_out, bool sparse, unsigned guess, cudaStream_t s)
{
    if (!cd || !h_out) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (n < 1 || n > cd->max_batch) { set_error("batch %d exceeds codec max_batch %d", n, cd->max_batch); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_context *ctx = cd->ctx;
    CFB_CUDA(cudaSetDevice(ctx->device));
    if (sparse) return sparse_download(cd, n, h_out, guess, s);
    for (int i = 0; i < n; i++) {
        if (!h_out[i]) { set_error("null host buffer %d", i); return CFB_ERROR_INVALID_ARGUMENT; }
        CFB_CUDA(cudaMemcpyAsync(h_out[i], cfb_codec_device_pyramid(cd, i), (size_t)cd->layout.coded_bytes, cudaMemcpyDeviceToHost, s));
        ctx->d2h_bytes += (uint64_t)cd->layout.coded_bytes;
    }
    return CFB_OK;
}

}  // namespace cfb
