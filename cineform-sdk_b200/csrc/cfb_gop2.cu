// cfb_gop2.cu -- two-frame GOP (CFHD_ENCODING_FLAGS_YUV_2FRAME_GOP): the FIELDPLUS pyramid as one call.
//
// Replaces, for packed 8-bit 4:2:2 sources (progressive or interlaced level 1):
//   encoder: Codec/encoder.c:3121 / :2976 level 1 of frame A and frame B (wavelet[0], wavelet[1]),
//            Codec/encoder.c:8431 FinishFieldPlusTransformQuant:
//              wavelet[2] = temporal(LL of [0], LL of [1])      (temporal.c:498 FilterTemporal16s)
//              wavelet[3] = level(temporal high,  prescale[3])  (all four bands coded, LL divisor 1)
//              wavelet[4] = level(temporal low,   prescale[4])
//              wavelet[5] = level(LL of [4],      prescale[5])
//   decoder: Codec/decoder.c:13052-13170 ReconstructWaveletBand for index 5, 4, 3, 2 and the level-1 inverse of
//            both frames (decoder.c:11836 ReconstructSampleFrameToBuffer, frames 0 and 1).
// Everything runs on the kernels of the intra-frame path (k_fwd_422 / k_fwd_422_fields, k_fwd_plane, k_temporal_*,
// k_inv_plane, k_inv_422 / k_inv_fields); this file only owns the GOP buffer layout and the launch sequence.
#include "cfb_host.h"

namespace cfb {
int pick_rows_per_warp(int strips, int rows, int planes, int sm_count);     // cfb_api.cu
static inline int align16i(int x) { return (x + 15) & ~15; }
static inline int64_t align64l(int64_t x) { return (x + 63) & ~(int64_t)63; }
}
using namespace cfb;

extern "C" {

// Coded region, per channel: wavelet 5 (LL, LH, HL, HH), wavelet 4 (LH, HL, HH), wavelet 3 (LL, LH, HL, HH),
// wavelet 1 (LH, HL, HH), wavelet 0 (LH, HL, HH) -- the 17 subbands the entropy coder walks (quantize.c:3480).
// Scratch region (device only): LL of wavelets 0, 1 and 4 and the two temporal bands of wavelet 2.
cfb_error cfb_gop2_layout_compute(const cfb_frame_desc *desc, cfb_gop2_layout *out)
{
    if (!desc || !out) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (desc->pixel_format != CFB_PIXEL_YUYV && desc->pixel_format != CFB_PIXEL_UYVY) {
        set_error("two-frame GOP: packed 8-bit 4:2:2 sources (CFHD_ENCODING_FLAGS_YUV_2FRAME_GOP)");
        return CFB_ERROR_UNSUPPORTED;
    }
    cfb_layout intra;
    cfb_error e = cfb_layout_compute(desc, &intra);
    if (e) return e;
    memset(out, 0, sizeof(*out));
    out->num_channels = intra.num_channels;
    int64_t off = 0;
    auto place = [&](int c, int k, int b, int w, int h) {
        cfb_band_layout &bl = out->band[c][k][b];
        bl.width = w; bl.height = h; bl.pitch = align16i(2 * w); bl.offset = off;
        off = align64l(off + (int64_t)bl.pitch * h);
    };
    for (int pass = 0; pass < 2; pass++) {          // pass 0: coded bands, pass 1: scratch
        for (int c = 0; c < intra.num_channels; c++) {
            const int w1 = intra.band[c][0][0].width, h1 = intra.band[c][0][0].height;     // level-1 band size
            if ((w1 & 15) || (h1 & 3)) { set_error("two-frame GOP: level-1 bands must be a multiple of 16 wide"); return CFB_ERROR_UNSUPPORTED; }
            const int w2 = w1 / 2, h2 = h1 / 2, w3 = w1 / 4, h3 = h1 / 4;
            if (pass == 0) {
                for (int b = 0; b < 4; b++) place(c, 5, b, w3, h3);
                for (int b = 1; b < 4; b++) place(c, 4, b, w2, h2);
                for (int b = 0; b < 4; b++) place(c, 3, b, w2, h2);
                for (int b = 1; b < 4; b++) place(c, 1, b, w1, h1);
                for (int b = 1; b < 4; b++) place(c, 0, b, w1, h1);
            } else {
                place(c, 0, 0, w1, h1); place(c, 1, 0, w1, h1);
                place(c, 2, 0, w1, h1); place(c, 2, 1, w1, h1);
                place(c, 4, 0, w2, h2);
            }
        }
        if (pass == 0) out->coded_bytes = off;
    }
    out->total_bytes = off;
    return CFB_OK;
}

static cfb_error gop2_prepare(cfb_codec *cd, cfb_gop2_layout &G)
{
    if (!cd) { set_error("null codec"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (cd->max_batch < 2) { set_error("two-frame GOP needs a codec created with max_batch >= 2"); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_error e = cfb_gop2_layout_compute(&cd->desc, &G);
    if (e) return e;
    if (!cd->d_gop) {
        CFB_CUDA(cudaSetDevice(cd->ctx->device));
        CFB_CUDA(cudaMalloc((void **)&cd->d_gop, (size_t)G.total_bytes));
        CFB_CUDA(cudaMemsetAsync(cd->d_gop, 0, (size_t)G.total_bytes, cd->ctx->stream));   // deterministic pitch padding
    }
    return CFB_OK;
}

static void fwd_geom(const cfb_gop2_layout &G, const cfb_gop2_quant *q, int c, int k, PlaneGeom &g)
{
    const cfb_band_layout &ll = G.band[c][k][0];
    g.width = ll.width * 2; g.height = ll.height * 2; g.out_pitch = ll.pitch;
    for (int b = 0; b < 4; b++) {
        g.band_off[b] = G.band[c][k][b].offset;
        g.q[b] = make_quant_param(q->divisor[c][k][b], q->midpoint_prequant);
    }
    g.quant_ll = 0; g.pad = 0; g.in_off = 0; g.in_pitch = 0;
}

static void inv_geom(const cfb_gop2_layout &G, const cfb_gop2_quant *q, int c, int k, InvGeom &g)
{
    const cfb_band_layout &ll = G.band[c][k][0];
    g.width = ll.width; g.height = ll.height; g.pitch = ll.pitch;
    for (int b = 0; b < 4; b++) {
        g.band_off[b] = G.band[c][k][b].offset;
        const int d = q->divisor[c][k][b];
        g.dq[b] = d > 1 ? d : 1;
    }
    g.dq[0] = 1;
    g.out_off = 0; g.out_pitch = 0;
}

cfb_error cfb_gop2_forward_host(cfb_codec *cd, const void *frame_a, const void *frame_b, int frame_pitch,
                                const cfb_gop2_quant *q, void *h_coded)
{
    cfb_gop2_layout G;
    cfb_error e = gop2_prepare(cd, G);
    if (e) return e;
    if (!frame_a || !frame_b || !q || !h_coded) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    cfb_context *ctx = cd->ctx;
    const cfb_layout &L = cd->layout;
    if (frame_pitch < L.frame_pitch) { set_error("frame pitch %d too small", frame_pitch); return CFB_ERROR_INVALID_ARGUMENT; }
    CFB_CUDA(cudaSetDevice(ctx->device));
    const int rows = (int)(L.frame_bytes / L.frame_pitch);
    const void *src[2] = {frame_a, frame_b};
    const int nc = L.num_channels;
    for (int f = 0; f < 2; f++) {
        unsigned char *dfr = (unsigned char *)cfb_codec_device_frame(cd, f);
        CFB_CUDA(cudaMemcpy2DAsync(dfr, L.frame_pitch, src[f], frame_pitch, L.frame_pitch, rows, cudaMemcpyHostToDevice, ctx->stream));
        ctx->h2d_bytes += (uint64_t)L.frame_bytes;
        // level 1 of this frame straight into wavelet f of the GOP buffer (spatial or field transform)
        FwdParams p;
        memset(&p, 0, sizeof(p));
        p.nchan = nc; p.nframes = 1;
        for (int c = 0; c < nc; c++) {
            fwd_geom(G, q, c, f, p.ch[c]);
            p.ch[c].in_off = 0; p.ch[c].in_pitch = L.frame_pitch;
            if (cd->interlaced) p.ch[c].q[2] = make_quant_param(q->divisor[c][f][2], q->midpoint_prequant, true);
        }
        p.in_base[0] = dfr; p.out_base[0] = cd->d_gop;
        p.shift = L.precision - 8; p.uyvy = (cd->desc.pixel_format == CFB_PIXEL_UYVY);
        p.th = pick_rows_per_warp((p.ch[0].width + kStripIn - 1) / kStripIn, p.ch[0].height / 2, 1, ctx->sm_count);
        CFB_CUDA(cd->interlaced ? launch_fwd_422_fields(p, ctx->stream) : launch_fwd_422(p, ctx->stream));
        ctx->kernel_launches++;
    }
    // wavelet 2: temporal transform of the two level-1 lowpass images
    for (int c = 0; c < nc; c++) {
        const cfb_band_layout &a = G.band[c][0][0], &b = G.band[c][1][0], &lo = G.band[c][2][0], &hi = G.band[c][2][1];
        e = cfb_temporal_forward_device(ctx, cd->d_gop + a.offset, cd->d_gop + b.offset, a.pitch, cd->d_gop + lo.offset,
                                        cd->d_gop + hi.offset, lo.pitch, a.width, a.height);
        if (e) return e;
    }
    // wavelets 3 (from the temporal highpass), 4 (from the temporal lowpass), 5 (from LL of wavelet 4)
    static const int src_k[6] = {0, 0, 0, 2, 2, 4}, src_b[6] = {0, 0, 0, 1, 0, 0};
    for (int k = 3; k <= 5; k++) {
        FwdParams p;
        memset(&p, 0, sizeof(p));
        p.nchan = nc; p.nframes = 1;
        int maxw = 0, maxoh = 0;
        for (int c = 0; c < nc; c++) {
            fwd_geom(G, q, c, k, p.ch[c]);
            const cfb_band_layout &in = G.band[c][src_k[k]][src_b[k]];
            p.ch[c].in_off = in.offset; p.ch[c].in_pitch = in.pitch;
            p.ch[c].quant_ll = (q->prescale[k] == 0) && q->divisor[c][k][0] > 1;
            if (p.ch[c].width > maxw) maxw = p.ch[c].width;
            if (p.ch[c].height / 2 > maxoh) maxoh = p.ch[c].height / 2;
        }
        p.in_base[0] = cd->d_gop; p.out_base[0] = cd->d_gop;
        p.th = pick_rows_per_warp((maxw + kStripIn - 1) / kStripIn, maxoh, nc, ctx->sm_count);
        // wavelet 3 reads the temporal HIGHPASS: the only signed plane of the pyramid (+-4080 by range), audited
        if (k == 3) { e = audit_level_input(ctx, p, q->prescale[k]); if (e) return e; }
        CFB_CUDA(launch_fwd_plane(p, q->prescale[k], ctx->stream));
        ctx->kernel_launches++;
    }
    CFB_CUDA(cudaMemcpyAsync(h_coded, cd->d_gop, (size_t)G.coded_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->d2h_bytes += (uint64_t)G.coded_bytes;
    CFB_CUDA(stream_wait(ctx));
    int range_flags = 0;
    e = range_status(ctx, &range_flags);
    if (e) return e;
    if (range_flags) {
        set_error("temporal highpass outside the exact-arithmetic range (flags %d): the reference's saturating chains would differ", range_flags);
        return CFB_ERROR_RANGE;
    }
    ctx->frames_forward += 2;
    return CFB_OK;
}

cfb_error cfb_gop2_inverse_host(cfb_codec *cd, const void *h_coded, const cfb_gop2_quant *q, int out_format,
                                void *frame_a, void *frame_b, int frame_pitch)
{
    cfb_gop2_layout G;
    cfb_error e = gop2_prepare(cd, G);
    if (e) return e;
    if (!frame_a || !frame_b || !q || !h_coded) { set_error("null argument"); return CFB_ERROR_INVALID_ARGUMENT; }
    if (out_format != CFB_PIXEL_YUYV && out_format != CFB_PIXEL_UYVY) { set_error("two-frame GOP decodes to packed 8-bit 4:2:2"); return CFB_ERROR_UNSUPPORTED; }
    cfb_context *ctx = cd->ctx;
    const cfb_layout &L = cd->layout;
    const int nc = L.num_channels;
    CFB_CUDA(cudaSetDevice(ctx->device));
    CFB_CUDA(cudaMemcpyAsync(cd->d_gop, h_coded, (size_t)G.coded_bytes, cudaMemcpyHostToDevice, ctx->stream));
    ctx->h2d_bytes += (uint64_t)G.coded_bytes;
    // wavelet 5 -> LL of 4; wavelet 4 -> temporal low; wavelet 3 -> temporal high
    static const int dst_k[6] = {0, 0, 0, 2, 2, 4}, dst_b[6] = {0, 0, 0, 1, 0, 0};
    static const int order[3] = {5, 4, 3};
    for (int i = 0; i < 3; i++) {
        const int k = order[i];
        InvParams p;
        memset(&p, 0, sizeof(p));
        p.nchan = nc; p.nframes = 1;
        int maxw = 0, maxh = 0;
        for (int c = 0; c < nc; c++) {
            inv_geom(G, q, c, k, p.ch[c]);
            const cfb_band_layout &out = G.band[c][dst_k[k]][dst_b[k]];
            p.ch[c].out_off = out.offset; p.ch[c].out_pitch = out.pitch;
            if (p.ch[c].width > maxw) maxw = p.ch[c].width;
            if (p.ch[c].height > maxh) maxh = p.ch[c].height;
        }
        p.in_base[0] = cd->d_gop; p.out_base[0] = cd->d_gop;
        p.th = pick_rows_per_warp((maxw + kInvStrip - 1) / kInvStrip, maxh, nc, ctx->sm_count);
        CFB_CUDA(launch_inv_plane(p, q->prescale[k], ctx->stream));
        ctx->kernel_launches++;
    }
    for (int c = 0; c < nc; c++) {
        const cfb_band_layout &a = G.band[c][0][0], &b = G.band[c][1][0], &lo = G.band[c][2][0], &hi = G.band[c][2][1];
        e = cfb_temporal_inverse_device(ctx, cd->d_gop + lo.offset, cd->d_gop + hi.offset, lo.pitch, cd->d_gop + a.offset,
                                        cd->d_gop + b.offset, a.pitch, a.width, a.height, L.precision);
        if (e) return e;
    }
    // level 1 of both frames -> packed 8-bit frames
    void *dst[2] = {frame_a, frame_b};
    for (int f = 0; f < 2; f++) {
        InvParams p;
        memset(&p, 0, sizeof(p));
        p.nchan = nc; p.nframes = 1;
        for (int c = 0; c < nc; c++) { inv_geom(G, q, c, f, p.ch[c]); p.ch[c].out_off = 0; p.ch[c].out_pitch = L.frame_pitch; }
        unsigned char *dfr = (unsigned char *)cfb_codec_device_frame(cd, f);
        p.in_base[0] = cd->d_gop; p.out_base[0] = dfr;
        p.shift = L.precision - 8; p.uyvy = (out_format == CFB_PIXEL_UYVY);
        p.th = pick_rows_per_warp((p.ch[0].width + kInvStrip - 1) / kInvStrip, p.ch[0].height, 1, ctx->sm_count);
        if (cd->interlaced) {
            if (!cd->d_carry) { set_error("interlaced codec without carry buffer"); return CFB_ERROR_INVALID_ARGUMENT; }
            FieldsAux aux;
            aux.carry = cd->d_carry; aux.nstrips = cd->carry_strips; aux.maxh = p.ch[0].height; aux.pad = (cd->interlaced == 2);
            CFB_CUDA(launch_inv_fields(p, aux, false, ctx->stream));
        } else {
            CFB_CUDA(launch_inv_422(p, kInv422Out8, ctx->stream));
        }
        ctx->kernel_launches++;
        CFB_CUDA(cudaMemcpy2DAsync(dst[f], frame_pitch, dfr, L.frame_pitch, L.frame_pitch, (size_t)(L.frame_bytes / L.frame_pitch),
                                   cudaMemcpyDeviceToHost, ctx->stream));
        ctx->d2h_bytes += (uint64_t)L.frame_bytes;
    }
    CFB_CUDA(stream_wait(ctx));
    ctx->frames_inverse += 2;
    return CFB_OK;
}

}  // extern "C"
