// cfhd_gpu_shim.cpp -- drop-in integration of libcfhd_b200 under the UNMODIFIED reference SDK.
//
// Built by integration/Makefile into  integration/_build/libCFHDCodec.so  together with the reference sources
// compiled in place (never copied).  The library exports the reference's complete CFHD_* C ABI (the symbols
// come from the reference objects), so Example/TestCFHD.cpp links and runs unchanged, while the five transform
// call sites of SURVEY 8(b) are served by the CUDA path through ELF symbol interposition:
//
//   encoder   TransformForwardSpatialYUV   (Codec/wavelet.c:2823, called at Codec/encoder.c:3121)
//             TransformForwardSpatialRGB30 (Codec/wavelet.c:3597, called at :3171; RG30 / R210 / DPX0 / AR10 / AB10 sources)
//             ComputeGroupTransformQuant   (Codec/encoder.c:8366, called at :3254)
//             EncodeQuantLongRuns          (Codec/encoder.c:5386, called at :6497): the run-length / VLC stream of a band is
//                                          written straight from the SPARSE transfer format (cfb_sparse_vlc_band), so the
//                                          dense bands never cross PCIe and the host never scans them (SURVEY 8f rank 1)
//   decoder   ReconstructWaveletBand       (Codec/decoder.c:12984, called at :11756/:11765 and by the worker threads)
//             ReconstructSampleFrameToBuffer (Codec/decoder.c:13387, called at :11836)
//
// This file defines functions with those names; because the reference objects are compiled -fPIC with default
// visibility their calls bind to the first definition in load order, i.e. to these.  Whenever a frame is outside
// what the CUDA path covers (other pixel formats, interlaced, GOP 2, reduced resolutions, active metadata ...)
// the call is forwarded to the reference's own function (dlsym RTLD_NEXT) -- that is the reference running its
// own code, not a fallback of ours.  Entropy coding, bitstream syntax, metadata and threading stay the
// reference's host code, as the north star prescribes.
#ifndef _GNU_SOURCE
#define _GNU_SOURCE
#endif
#include <dlfcn.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <map>
#include <chrono>
#include <mutex>
#include <utility>
#include <vector>

extern "C" {
#include "config.h"
#include "encoder.h"
#include "decoder.h"
#include "wavelet.h"
#include "quantize.h"
#include "codec.h"
#include "image.h"
#include "vlc.h"
#include "bitstream.h"
}
#include "AVIExtendedHeader.h"     // CURVE_LOG_90
extern "C" void cfhd_shim_default_bayer_curve(uint16_t *table);       // bayer_curve.c (C on purpose, see there)
#include "cfhd_b200.h"
#include "CFHDEncoder.h"            // the public SDK entry points whose preparation calls pre-create the plans
#include <thread>

extern "C" int g_midpoint_prequant;     // Codec/quantize.c:183

namespace {

std::atomic<long> g_fwd_frames{0}, g_inv_frames{0}, g_fwd_ref{0}, g_inv_ref{0};
std::atomic<long> g_cuda_errors{0};
std::atomic<long> g_vlc_sparse_bands{0}, g_vlc_ref_bands{0};
std::atomic<long> g_plans_created{0}, g_plan_create_us{0}, g_gpu_us{0}, g_vlc_us{0};

struct StatsAtExit {
    ~StatsAtExit() {
        if (getenv("CFHD_B200_STATS"))
            fprintf(stderr, "cfhd_gpu_shim: forward frames on GPU %ld (reference CPU %ld), inverse frames on GPU %ld (reference CPU %ld), CUDA errors %ld, "
                            "bands coded from the sparse format %ld (dense, by the reference's coder %ld); plans created %ld in %.1f ms, "
                            "forward host calls %.1f ms, sparse VLC walk %.1f ms (summed over threads)\n",
                    g_fwd_frames.load(), g_fwd_ref.load(), g_inv_frames.load(), g_inv_ref.load(), g_cuda_errors.load(),
                    g_vlc_sparse_bands.load(), g_vlc_ref_bands.load(), g_plans_created.load(), g_plan_create_us.load() / 1e3,
                    g_gpu_us.load() / 1e3, g_vlc_us.load() / 1e3);
    }
} g_stats_at_exit;

template <class F> F next_symbol(const char *name)
{
    void *p = dlsym(RTLD_NEXT, name);
    if (!p) { fprintf(stderr, "cfhd_gpu_shim: reference symbol %s not found\n", name); abort(); }
    return (F)p;
}

bool gpu_enabled()
{
    static int state = -1;
    if (state < 0) {
        const char *e = getenv("CFHD_B200_DISABLE");
        state = (e && *e == '1') ? 0 : (cfb_device_count() > 0 ? 1 : 0);
        if (!state) fprintf(stderr, "cfhd_gpu_shim: CUDA path off (%s) -- the reference's own CPU transform runs\n",
                            (e && *e == '1') ? "CFHD_B200_DISABLE=1" : "no sm_100 device");
    }
    return state == 1;
}

// Plans = (context + stream, codec, pinned staging) for one geometry.  They live in a process-wide pool and are BORROWED by
// a thread for the duration of one frame (EncodeSample / one decode): TestCFHD -E creates a new encoder pool -- new threads
// -- for every row of its format table, and per-thread plans (the first version) re-created sixteen CUDA contexts and
// re-pinned 1.4 GB of host memory per row.  Two threads never share a plan at the same time, hence never a stream.
struct Plan {
    cfb_context *ctx = nullptr;
    cfb_codec *codec = nullptr;
    cfb_layout layout{};
    uint64_t key = 0;
    void *coded = nullptr;          // pinned staging for the dense coded region (allocated on first use)
    void *sparse = nullptr;         // pinned staging for the coded region in the sparse transfer format (allocated on first use)
    int curve_mode = -1;            // Bayer: encode curve the codec currently holds (-1 unknown, 0 none = curve applied, 1 = default log 90)
    void *frame = nullptr;          // pinned staging for a decoded frame at the ENCODED size (allocated on first use)
    size_t frame_cap = 0;           // bytes of `frame` (outputs differ in size: 8-bit 4:2:2 .. B64A)
    bool ensure_coded() { return coded || cfb_host_alloc((size_t)layout.coded_bytes, &coded) == CFB_OK; }
    bool ensure_frame(size_t bytes) {
        if (frame && frame_cap >= bytes) return true;
        if (frame) { cfb_host_free(frame); frame = nullptr; frame_cap = 0; }
        if (cfb_host_alloc(bytes, &frame) != CFB_OK) { frame = nullptr; return false; }
        frame_cap = bytes;
        return true;
    }
    bool ensure_sparse() { return sparse || cfb_host_alloc(cfb_sparse_max_bytes(&layout), &sparse) == CFB_OK; }
};

std::mutex g_plan_mu;
std::map<uint64_t, std::vector<Plan *>> g_free_plans;
std::map<uint64_t, bool> g_uncovered;                   // geometries cfb_layout_compute rejected
int g_next_device = 0;
thread_local std::vector<Plan *> t_held;                // plans this thread has borrowed for the frame in progress

void release_plans()
{
    if (t_held.empty()) return;
    std::lock_guard<std::mutex> lk(g_plan_mu);
    for (Plan *p : t_held) g_free_plans[p->key].push_back(p);
    t_held.clear();
}

// interlaced: CFB_PROGRESSIVE, CFB_INTERLACED (encoder: coded HL band) or CFB_INTERLACED_HL_INTEGRATED (decoder bands)
Plan *get_plan(int width, int height, int pixel_format, int interlaced = CFB_PROGRESSIVE)
{
    const uint64_t key = ((uint64_t)width << 40) | ((uint64_t)height << 16) | ((uint64_t)interlaced << 8) | (uint64_t)pixel_format;
    for (Plan *p : t_held) if (p->key == key) return p;
    int dev;
    {
        std::lock_guard<std::mutex> lk(g_plan_mu);
        if (g_uncovered.count(key)) return nullptr;
        std::vector<Plan *> &fl = g_free_plans[key];
        if (!fl.empty()) { Plan *p = fl.back(); fl.pop_back(); t_held.push_back(p); return p; }
        dev = g_next_device++ % cfb_device_count();     // frames sharded over the GPUs
    }
    const auto t0 = std::chrono::steady_clock::now();
    Plan *p = new Plan;
    p->key = key;
    cfb_frame_desc d = {width, height, pixel_format, 0};
    bool ok = cfb_layout_compute(&d, &p->layout) == CFB_OK;                 // else: geometry outside the CUDA path
    ok = ok && cfb_context_create(dev, &p->ctx) == CFB_OK;
    ok = ok && cfb_codec_create(p->ctx, &d, 1, &p->codec) == CFB_OK;
    ok = ok && (!interlaced || cfb_codec_set_interlaced(p->codec, interlaced) == CFB_OK);
    if (!ok) {
        if (p->codec) cfb_codec_destroy(p->codec);
        if (p->ctx) cfb_context_destroy(p->ctx);
        delete p;
        std::lock_guard<std::mutex> lk(g_plan_mu);
        g_uncovered[key] = true;
        return nullptr;
    }
    t_held.push_back(p);
    g_plans_created++;
    g_plan_create_us += std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    return p;
}

thread_local TRANSFORM *t_pyramid_done_for = nullptr;    // encoder: levels 2,3 already produced for this transform[0]
thread_local bool t_cuda_failed = false;                 // encoder: the CUDA pyramid of the current frame failed (no CPU fallback)
enum Took { NOT_COVERED, DONE, FAILED };

// Sparse hand-over of the current frame of this thread: the highpass bands were NOT copied to the encoder's band buffers;
// EncodeQuantLongRuns recognises a band by its buffer address and codes it from plan->sparse.  The token (encoder,
// frame_count) is taken in ComputeGroupTransformQuant and ends with the frame (encoder.c:3274 advances frame_count after
// the entropy coder has run), so a later frame that the reference transforms itself into the same buffers is never
// mistaken for this one.
struct SparseFrame {
    Plan *plan = nullptr;
    const void *band[CFB_MAX_CHANNELS][3][4] = {};
    const ENCODER *encoder = nullptr;
    uint32_t frame_count = 0;
    bool armed = false;             // bands recorded, token not taken yet
    bool valid = false;
};
thread_local SparseFrame t_sparse;

bool sparse_enabled()
{
    static int state = -1;
    if (state < 0) { const char *e = getenv("CFHD_B200_DENSE"); state = (e && *e == '1') ? 0 : 1; }
    return state == 1;
}

// The reference's code tables as the plain arrays the C ABI takes (built once per code set)
struct Book {
    std::vector<uint32_t> run_bits, run_count, value_bits;
    std::vector<uint8_t> run_size, value_size;
    cfb_vlc_codebook c{};
};
const cfb_vlc_codebook *codebook_for(ENCODER *encoder, int active_codebook)
{
    static std::mutex mu;
    static std::map<std::pair<const void *, const void *>, Book *> books;
    if (active_codebook < 0 || active_codebook >= CODEC_NUM_CODESETS) return nullptr;
    RLCBOOK *rb = encoder->codebook_runbook[active_codebook];
    VALBOOK *vb = encoder->valuebook[active_codebook];
    if (!rb || !vb) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    Book *&b = books[{rb, vb}];
    if (!b) {
        b = new Book;
        const RLC *rlc = (const RLC *)((const char *)rb + sizeof(RLCBOOK));         // vlc.h:105-131
        for (int i = 0; i < rb->length; i++) { b->run_bits.push_back(rlc[i].bits); b->run_size.push_back((uint8_t)rlc[i].size); b->run_count.push_back((uint32_t)rlc[i].count); }
        const VLE *tab = (const VLE *)((const char *)vb + sizeof(VALBOOK));         // vlc.h:67-73
        for (int i = 0; i < VALUE_TABLE_LENGTH; i++) { b->value_bits.push_back(tab[i].entry & VLE_CODEWORD_MASK); b->value_size.push_back((uint8_t)(tab[i].entry >> VLE_CODESIZE_SHIFT)); }
        b->c.run_length = rb->length; b->c.value_length = VALUE_TABLE_LENGTH;
        b->c.run_bits = b->run_bits.data(); b->c.run_size = b->run_size.data(); b->c.run_count = b->run_count.data();
        b->c.value_bits = b->value_bits.data(); b->c.value_size = b->value_size.data();
    }
    return &b->c;
}

// Sources the reference first converts to planes on the CPU (encoder.c:2518-2776: ConvertV210ToFrame16s,
// ConvertYU64ToFrame16s, ConvertRGB48ToFrame16s, ConvertBYR4ToFrame16s) and then transforms plane by plane
// (TransformForwardSpatial, encoder.c:3180-3193).  The CUDA kernels read the PACKED frame, so the converter hook only
// records where it is -- the conversion itself and the per-plane level-1 calls are skipped -- and
// ComputeGroupTransformQuant runs the whole pyramid in one pass.  The hooks only engage inside EncodeSample of an
// intra-frame, progressive, compressed encode whose geometry the plan covers (checked in the converter hook, while the
// reference's own path is still intact).
struct PendingSource {
    Plan *plan = nullptr;
    uint8_t *data = nullptr;
    int pitch = 0;
    int bayer_phase = -1;
    int curve_mode = 0;             // Bayer: 0 = the frame carries its curve, 1 = the encoder's default curve (log base 90)
    FRAME *frame = nullptr;
};
thread_local ENCODER *t_enc = nullptr;
thread_local TRANSFORM **t_transform = nullptr;
thread_local int t_num_transforms = 0;
thread_local PendingSource t_pending;

bool spatial3(TRANSFORM *t)
{
    return t && t->type == TRANSFORM_TYPE_SPATIAL && t->wavelet[0] && t->wavelet[1] && t->wavelet[2];
}

}  // namespace

extern "C" {
static Plan *covered_plan(const uint8_t *input, int input_pitch, int width, int height, TRANSFORM *transform[], int num_channels,
                          int precision, int interlaced, int cfb_format);
}

// converter hooks: true = the packed source was recorded for the GPU pass (the caller skips the CPU conversion)
static bool record_source(int cfb_format, uint8_t *data, int pitch, FRAME *frame, int width, int height, int precision, int bayer_phase,
                          int curve_mode = 0)
{
    t_pending = PendingSource();
    ENCODER *e = t_enc;
    static const bool debug = getenv("CFHD_B200_DEBUG") != nullptr;
    if (debug) fprintf(stderr, "cfhd_gpu_shim: record_source fmt %d enc %p gop %d progressive %d uncompressed %d num_spatial %d frame channels %d transforms %d %dx%d pitch %d\n",
                       cfb_format, (void *)e, e ? e->gop_length : -1, e ? (int)e->progressive : -1, e ? (int)e->uncompressed : -1, e ? e->num_spatial : -1,
                       frame ? frame->num_channels : -1, t_num_transforms, width, height, pitch);
    if (!e || !frame || e->gop_length != 1 || !e->progressive || e->uncompressed || e->num_spatial != 2) return false;     // num_spatial = wavelets above level 1 (encoder.c:8390: num_levels = num_spatial + 1)
    if (frame->num_channels != t_num_transforms) return false;
    // a source whose coded height was rounded up (encoder.c:2232; 1080-line Bayer -> 544-row planes) has no rows behind its
    // display height: the reference's converters replicate the last row into the planes, the packed frame does not hold them
    if (frame->display_height != frame->height) return false;
    Plan *plan = covered_plan(data, pitch, width, height, t_transform, t_num_transforms, precision, CFB_PROGRESSIVE, cfb_format);
    if (debug) fprintf(stderr, "cfhd_gpu_shim: record_source plan %p\n", (void *)plan);
    if (!plan) return false;
    t_pending.plan = plan; t_pending.data = data; t_pending.pitch = pitch; t_pending.bayer_phase = bayer_phase; t_pending.frame = frame;
    t_pending.curve_mode = curve_mode;
    return true;
}

extern "C" {

// ------------------------------------------------------------------------------------------------ encoder
// The whole 3-level pyramid of one packed 4:2:2 frame on the GPU (level 1 = spatial or field transform).
//   NOT_COVERED  geometry / options outside the CUDA path: the caller runs the reference's own function (the reference
//                running its own code for a format we do not claim -- counted in g_fwd_ref);
//   FAILED       the frame IS covered but a CUDA call failed: there is NO CPU fallback on the transform path -- the bands
//                are zero-filled, ComputeGroupTransformQuant reports CODEC_ERROR through encoder->error, the error is
//                printed, and CFHD_B200_ABORT_ON_ERROR=1 turns it into an abort().
// Is this source covered?  Returns the plan (context + codec of this thread for the geometry) or null.  width / height
// are what cfb_frame_desc wants (the Bayer mosaic's dimensions for BYR4), input_pitch bytes per row (per Bayer line).
static Plan *covered_plan(const uint8_t *input, int input_pitch, int width, int height, TRANSFORM *transform[], int num_channels,
                          int precision, int interlaced, int cfb_format)
{
    if (!gpu_enabled() || cfb_format < 0 || !transform || input_pitch <= 0 || (input_pitch & 15) || ((uintptr_t)input & 15)) return nullptr;
    if (num_channels < 3 || num_channels > CFB_MAX_CHANNELS) return nullptr;
    for (int c = 0; c < num_channels; c++) if (!spatial3(transform[c])) return nullptr;
    Plan *plan = get_plan(width, height, cfb_format, interlaced);
    if (!plan || plan->layout.num_channels != num_channels || precision != plan->layout.precision) return nullptr;
    if (input_pitch < plan->layout.frame_pitch) return nullptr;      // rows that overlap in memory (TestCFHD -E does that for R210): not a frame layout we read
    for (int c = 0; c < num_channels; c++)
        for (int k = 0; k < 3; k++) {
            IMAGE *w = transform[c]->wavelet[k];
            const cfb_band_layout &b = plan->layout.band[c][k][1];
            if (w->width != b.width || w->height != b.height || w->pitch != b.pitch) return nullptr;     // not the geometry the plan was built for
        }
    return plan;
}

static Took run_pyramid(Plan *plan, uint8_t *input, int input_pitch, TRANSFORM *transform[], int interlaced, int bayer_phase, int curve_mode = 0);

static Took forward_pyramid_on_gpu(uint8_t *input, int input_pitch, FRAME_INFO *frame, TRANSFORM *transform[], int frame_index,
                                   int num_channels, int precision, int limit_yuv, int conv_601_709, int interlaced, int cfb_format)
{
    t_pyramid_done_for = nullptr;
    t_cuda_failed = false;
    t_sparse.valid = t_sparse.armed = false;
    Plan *plan = nullptr;
    if (frame && frame_index == 0 && num_channels == 3 && !limit_yuv && !conv_601_709)
        plan = covered_plan(input, input_pitch, frame->width, frame->height, transform, num_channels, precision, interlaced, cfb_format);
    if (!plan) return NOT_COVERED;
    return run_pyramid(plan, input, input_pitch, transform, interlaced, -1);
}

// The encoder's default Bayer encode curve as the reference builds it inside ConvertBYR4ToFrame16s (frame.c:5208-5222:
// log base 90 over 1 << 14 input levels, 12-bit output), with the reference's own macro compiled as C (bayer_curve.c)
static const uint16_t *default_bayer_curve()
{
    static uint16_t table[1 << 14];
    static std::once_flag once;
    std::call_once(once, [] { cfhd_shim_default_bayer_curve(table); });
    return table;
}

static Took run_pyramid(Plan *plan, uint8_t *input, int input_pitch, TRANSFORM *transform[], int interlaced, int bayer_phase, int curve_mode)
{
    const int nc = plan->layout.num_channels;
    if (bayer_phase >= 0) {
        if (cfb_codec_set_bayer_phase(plan->codec, bayer_phase) != CFB_OK) return NOT_COVERED;
        if (plan->curve_mode != curve_mode) {       // the table is uploaded once per codec, not per frame
            if (cfb_codec_set_bayer_curve(plan->codec, curve_mode ? default_bayer_curve() : nullptr, curve_mode ? 1 << 14 : 0) != CFB_OK) return NOT_COVERED;
            plan->curve_mode = curve_mode;
        }
    }

    cfb_quant q;
    memset(&q, 0, sizeof(q));
    q.midpoint_prequant = g_midpoint_prequant;
    for (int k = 0; k < 3; k++) q.prescale[k] = transform[0]->prescale[k];
    for (int c = 0; c < nc; c++)
        for (int k = 0; k < 3; k++)
            for (int bnd = 0; bnd < 4; bnd++) q.divisor[c][k][bnd] = transform[c]->wavelet[k]->quant[bnd];
    const void *frames[1] = {input};
    // Progressive frames cross PCIe in the sparse format and are entropy coded from it (EncodeQuantLongRuns below); the
    // interlaced level-1 HL band is coded by EncodeQuantLongRunsPlusPeaks (encoder.c:6458), which wants it dense.
    const bool sparse = sparse_enabled() && interlaced == CFB_PROGRESSIVE && plan->ensure_sparse();
    if (!plan->ensure_coded()) return NOT_COVERED;
    bool failed;
    const auto tg0 = std::chrono::steady_clock::now();
    if (sparse) {
        void *out[1] = {plan->sparse};
        failed = cfb_forward_host_sparse(plan->codec, 1, frames, input_pitch, &q, out, nullptr) != CFB_OK;
    } else {
        void *coded[1] = {plan->coded};
        failed = cfb_forward_host(plan->codec, 1, frames, input_pitch, &q, coded) != CFB_OK;
    }
    g_gpu_us += std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - tg0).count();
    if (failed) {
        fprintf(stderr, "cfhd_gpu_shim: CUDA forward transform failed (%s); no CPU fallback on the transform path\n", cfb_last_error_string());
        g_cuda_errors++;
        if (getenv("CFHD_B200_ABORT_ON_ERROR")) abort();
        memset(plan->coded, 0, (size_t)plan->layout.coded_bytes);
        t_cuda_failed = true;
    }
    // hand the bands to the host entropy coder exactly where it expects them
    for (int c = 0; c < nc; c++)
        for (int k = 0; k < 3; k++) {
            IMAGE *w = transform[c]->wavelet[k];
            for (int bnd = (k == 2 ? 0 : 1); bnd < 4; bnd++) {
                const cfb_band_layout &b = plan->layout.band[c][k][bnd];
                if (!sparse || failed) memcpy(w->band[bnd], (const char *)plan->coded + b.offset, (size_t)b.pitch * b.height);
                else if (bnd == 0) {
                    // the lowpass band LL3 is coded by EncodeLowPassBand (encoder.c:4251) from the dense band: 1/64 of the frame
                    if (cfb_sparse_expand_band(&plan->layout, plan->sparse, c, k, 0, (int16_t *)w->band[0], w->pitch) != CFB_OK) {
                        fprintf(stderr, "cfhd_gpu_shim: damaged sparse buffer (%s)\n", cfb_last_error_string());
                        g_cuda_errors++; t_cuda_failed = true; failed = true;
                    }
                } else t_sparse.band[c][k][bnd] = w->band[bnd];
            }
            for (int bnd = 0; bnd < 4; bnd++) { w->pixel_type[bnd] = PIXEL_TYPE_16S; w->quantization[bnd] = w->quant[bnd]; }
        }
    if (sparse && !failed) { t_sparse.plan = plan; t_sparse.armed = true; }
    t_pyramid_done_for = transform[0];
    if (failed) return FAILED;
    g_fwd_frames++;
    return DONE;
}

static int cfb_format_of_422(const FRAME_INFO *frame)
{
    if (!frame) return -1;
    return frame->format == COLOR_FORMAT_YUYV ? CFB_PIXEL_YUYV : (frame->format == COLOR_FORMAT_UYVY ? CFB_PIXEL_UYVY : -1);
}

void TransformForwardSpatialYUV(uint8_t *input, int input_pitch, FRAME_INFO *frame, TRANSFORM *transform[], int frame_index,
                                int num_channels, PIXEL *buffer, size_t buffer_size, int chroma_offset, int IFrame,
                                int precision, int limit_yuv, int conv_601_709)
{
    typedef void (*fn_t)(uint8_t *, int, FRAME_INFO *, TRANSFORM *[], int, int, PIXEL *, size_t, int, int, int, int, int);
    static fn_t ref = next_symbol<fn_t>("TransformForwardSpatialYUV");
    if (forward_pyramid_on_gpu(input, input_pitch, frame, transform, frame_index, num_channels, precision, limit_yuv, conv_601_709, CFB_PROGRESSIVE, cfb_format_of_422(frame)) != NOT_COVERED) return;
    g_fwd_ref++;
    ref(input, input_pitch, frame, transform, frame_index, num_channels, buffer, buffer_size, chroma_offset, IFrame, precision, limit_yuv, conv_601_709);
}

// interlaced sources (CFHD_ENCODING_FLAGS_YUV_INTERLACED): Codec/encoder.c:2976 -> Codec/wavelet.c:6076
void TransformForwardFrameYUV(uint8_t *input, int input_pitch, FRAME_INFO *frame, TRANSFORM *transform[], int frame_index,
                              int num_channels, char *buffer, size_t buffer_size, int chroma_offset,
                              int precision, int limit_yuv, int conv_601_709)
{
    typedef void (*fn_t)(uint8_t *, int, FRAME_INFO *, TRANSFORM *[], int, int, char *, size_t, int, int, int, int);
    static fn_t ref = next_symbol<fn_t>("TransformForwardFrameYUV");
    if (forward_pyramid_on_gpu(input, input_pitch, frame, transform, frame_index, num_channels, precision, limit_yuv, conv_601_709, CFB_INTERLACED, cfb_format_of_422(frame)) != NOT_COVERED) return;
    g_fwd_ref++;
    ref(input, input_pitch, frame, transform, frame_index, num_channels, buffer, buffer_size, chroma_offset, precision, limit_yuv, conv_601_709);
}

// The codec-level entry of every encode (SampleEncoder.cpp:604 and the pool's worker threads call it): remembers which
// encoder and transforms the hooks below are working for.
bool EncodeSample(ENCODER *encoder, uint8_t *data, int width, int height, int pitch, int format, TRANSFORM *transform[], int num_transforms,
                  BITSTREAM *output, PIXEL *buffer, size_t buffer_size, int fixedquality, int fixedbitrate, uint8_t *pPreviewBuffer,
                  float framerate, custom_quant *custom)
{
    typedef bool (*fn_t)(ENCODER *, uint8_t *, int, int, int, int, TRANSFORM *[], int, BITSTREAM *, PIXEL *, size_t, int, int, uint8_t *, float, custom_quant *);
    static fn_t ref = next_symbol<fn_t>("EncodeSample");
    t_enc = encoder; t_transform = transform; t_num_transforms = num_transforms;
    t_pending = PendingSource();
    const bool r = ref(encoder, data, width, height, pitch, format, transform, num_transforms, output, buffer, buffer_size, fixedquality,
                       fixedbitrate, pPreviewBuffer, framerate, custom);
    t_enc = nullptr; t_transform = nullptr; t_num_transforms = 0;
    t_pending = PendingSource();
    t_sparse.valid = t_sparse.armed = false;
    release_plans();                // the frame is done: its plan goes back to the pool
    return r;
}

void ConvertV210ToFrame16s(uint8_t *data, int pitch, FRAME *frame, uint8_t *buffer)          // Codec/frame.c:1431, encoder.c:2532
{
    typedef void (*fn_t)(uint8_t *, int, FRAME *, uint8_t *);
    static fn_t ref = next_symbol<fn_t>("ConvertV210ToFrame16s");
    if (frame && record_source(CFB_PIXEL_V210, data, pitch, frame, frame->width, frame->height, 10, -1)) return;
    if (t_enc) g_fwd_ref++;         // this frame's planes and its transform stay with the reference's CPU code
    ref(data, pitch, frame, buffer);
}

void ConvertYU64ToFrame16s(uint8_t *data, int pitch, FRAME *frame, uint8_t *buffer)          // Codec/frame.c:1556, encoder.c:2547
{
    typedef void (*fn_t)(uint8_t *, int, FRAME *, uint8_t *);
    static fn_t ref = next_symbol<fn_t>("ConvertYU64ToFrame16s");
    if (frame && record_source(CFB_PIXEL_YU64, data, pitch, frame, frame->width, frame->height, 10, -1)) return;
    if (t_enc) g_fwd_ref++;
    ref(data, pitch, frame, buffer);
}

void ConvertRGB48ToFrame16s(uint8_t *data, int pitch, FRAME *frame, uint8_t *buffer, int precision, int origformat)   // frame.c:5968, encoder.c:2768
{
    typedef void (*fn_t)(uint8_t *, int, FRAME *, uint8_t *, int, int);
    static fn_t ref = next_symbol<fn_t>("ConvertRGB48ToFrame16s");
    // only the plain 16-bit RGB layout (the default branch, frame.c:6130-6164: planes G, R, B, samples >> 4)
    if (frame && origformat == COLOR_FORMAT_RG48 && precision == 12 &&
        record_source(CFB_PIXEL_RG48, data, pitch, frame, frame->width, frame->height, 12, -1)) return;
    if (t_enc) g_fwd_ref++;
    ref(data, pitch, frame, buffer, precision, origformat);
}

void ConvertBYR4ToFrame16s(int bayer_format, uint32_t encode_curve, uint32_t encode_curve_preset, uint8_t *data, int pitch,
                           FRAME *frame, int precision)                                       // Codec/frame.c:4993, encoder.c:2638
{
    typedef void (*fn_t)(int, uint32_t, uint32_t, uint8_t *, int, FRAME *, int);
    static fn_t ref = next_symbol<fn_t>("ConvertBYR4ToFrame16s");
    if (getenv("CFHD_B200_DEBUG")) fprintf(stderr, "cfhd_gpu_shim: ConvertBYR4ToFrame16s bayer %d curve %u preset %u pitch %d precision %d frame %dx%d\n",
                                           bayer_format, encode_curve, encode_curve_preset, pitch, precision, frame ? frame->width : -1, frame ? frame->height : -1);
    // frames that already carry their curve (metadata TAG_ENCODE_PRESET = 1: samples >> 4) and frames the encoder maps
    // through its default curve (no curve metadata: log base 90, the table built above); the other curve families
    // (frame.c:5224-5330) stay with the reference.  The SDK describes a Bayer frame by its PLANE dimensions and a pitch
    // of two Bayer lines (SampleEncoder.cpp:268-269, :494).
    const int curve_mode = encode_curve_preset == 1 ? 0 : ((encode_curve == 0 || encode_curve == CURVE_LOG_90) ? 1 : -1);
    if (frame && curve_mode >= 0 && precision == 12 && !(pitch & 31) &&
        record_source(CFB_PIXEL_BYR4, data, pitch / 2, frame, frame->width * 2, frame->height * 2, 12, bayer_format, curve_mode)) return;
    if (t_enc) g_fwd_ref++;
    ref(bayer_format, encode_curve, encode_curve_preset, data, pitch, frame, precision);
}

// level 1 of one plane (Codec/wavelet.c:2420, called per channel at encoder.c:3180-3193): nothing to do for the planes of
// a frame whose packed source is waiting for the GPU pass
IMAGE *TransformForwardSpatial(ALLOCATOR *allocator, IMAGE *image, int band, IMAGE *wavelet, int level, PIXEL *buffer, size_t size,
                               int prescale, int quantization[IMAGE_NUM_BANDS], int difference_LL)
{
    typedef IMAGE *(*fn_t)(ALLOCATOR *, IMAGE *, int, IMAGE *, int, PIXEL *, size_t, int, int *, int);
    static fn_t ref = next_symbol<fn_t>("TransformForwardSpatial");
    if (t_pending.plan && level == 1 && band == 0)
        for (int c = 0; c < t_pending.frame->num_channels; c++)
            if (t_pending.frame->channel[c] == image && t_transform && t_transform[c]->wavelet[0] == wavelet) return wavelet;
    return ref(allocator, image, band, wavelet, level, buffer, size, prescale, quantization, difference_LL);
}

// 10-bit packed RGB sources: Codec/encoder.c:3158-3176 -> Codec/wavelet.c:3597 (planes G, R, B; fields filtered after << 2)
void TransformForwardSpatialRGB30(uint8_t *input, int input_pitch, FRAME_INFO *frame, TRANSFORM *transform[], int frame_index,
                                  int num_channels, PIXEL *buffer, size_t buffer_size, int chroma_offset, int IFrame,
                                  int display_height, int precision, int format)
{
    typedef void (*fn_t)(uint8_t *, int, FRAME_INFO *, TRANSFORM *[], int, int, PIXEL *, size_t, int, int, int, int, int);
    static fn_t ref = next_symbol<fn_t>("TransformForwardSpatialRGB30");
    int fmt = -1;
    switch (format) {
    case COLOR_FORMAT_RG30: fmt = CFB_PIXEL_RG30; break;
    case COLOR_FORMAT_AB10: fmt = CFB_PIXEL_AB10; break;
    case COLOR_FORMAT_AR10: fmt = CFB_PIXEL_AR10; break;
    case COLOR_FORMAT_R210: fmt = CFB_PIXEL_R210; break;
    case COLOR_FORMAT_DPX0: fmt = CFB_PIXEL_DPX0; break;
    }
    // frames whose coded height is their display height (wavelet.c:3645-3648: the last row pair goes through the border
    // filters as everywhere else); a frame the encoder padded (display_height < height) is transformed by the reference
    // from stale filter rows (:4066-4073), which is not a transform we reproduce
    if (frame && display_height == frame->height &&
        forward_pyramid_on_gpu(input, input_pitch, frame, transform, frame_index, num_channels, precision, 0, 0, CFB_PROGRESSIVE, fmt) != NOT_COVERED) return;
    t_sparse.valid = t_sparse.armed = false;
    g_fwd_ref++;
    ref(input, input_pitch, frame, transform, frame_index, num_channels, buffer, buffer_size, chroma_offset, IFrame, display_height, precision, format);
}

// Run-length / VLC coding of one highpass band (Codec/encoder.c:5386).  Bands of the frame this thread has just
// transformed on the GPU are coded straight from the sparse transfer format; everything else is the reference's.
void EncodeQuantLongRuns(ENCODER *encoder, BITSTREAM *stream, PIXEL *image, int width, int height, int pitch, int divisor, int active_codebook)
{
    typedef void (*fn_t)(ENCODER *, BITSTREAM *, PIXEL *, int, int, int, int, int);
    static fn_t ref = next_symbol<fn_t>("EncodeQuantLongRuns");
    SparseFrame &sf = t_sparse;
    if (sf.valid && sf.encoder == encoder && sf.frame_count == (uint32_t)encoder->frame_count) {
        for (int c = 0; c < sf.plan->layout.num_channels; c++)
            for (int k = 0; k < 3; k++)
                for (int b = 1; b < 4; b++) {
                    if (sf.band[c][k][b] != (const void *)image) continue;
                    const cfb_band_layout &bl = sf.plan->layout.band[c][k][b];
                    const cfb_vlc_codebook *book = codebook_for(encoder, active_codebook);
                    if (!book || bl.width != width || bl.height != height || bl.pitch != pitch) break;
                    cfb_bitwriter bw;
                    bw.cur = stream->lpCurrentWord;
                    bw.end = stream->lpCurrentBuffer + stream->dwBlockLength;
                    bw.buffer = stream->wBuffer; bw.bits_free = stream->nBitsFree; bw.bytes = stream->nWordsUsed;
                    const auto tv0 = std::chrono::steady_clock::now();
                    const cfb_error ve = cfb_sparse_vlc_band(&sf.plan->layout, sf.plan->sparse, c, k, b, book, &bw);
                    g_vlc_us += std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - tv0).count();
                    if (ve != CFB_OK) {
                        fprintf(stderr, "cfhd_gpu_shim: coding band (%d, %d, %d) from the sparse format failed: %s\n", c, k, b, cfb_last_error_string());
                        if (getenv("CFHD_B200_ABORT_ON_ERROR")) abort();
                        encoder->error = CODEC_ERROR_UNEXPECTED;
                        stream->error = BITSTREAM_ERROR_OVERFLOW;
                        return;
                    }
                    stream->lpCurrentWord = bw.cur; stream->wBuffer = bw.buffer; stream->nBitsFree = bw.bits_free; stream->nWordsUsed = (int)bw.bytes;
                    g_vlc_sparse_bands++;
                    return;
                }
        // a band of this frame that we do not hold sparse must not exist: its buffer was never filled
        fprintf(stderr, "cfhd_gpu_shim: EncodeQuantLongRuns on an unknown band of a sparse frame\n");
        if (getenv("CFHD_B200_ABORT_ON_ERROR")) abort();
        encoder->error = CODEC_ERROR_UNEXPECTED;
        return;
    }
    g_vlc_ref_bands++;
    ref(encoder, stream, image, width, height, pitch, divisor, active_codebook);
}

void ComputeGroupTransformQuant(ENCODER *encoder, TRANSFORM *transform[], int num_transforms)
{
    typedef void (*fn_t)(ENCODER *, TRANSFORM *[], int);
    static fn_t ref = next_symbol<fn_t>("ComputeGroupTransformQuant");
    if (t_pending.plan && t_transform == transform) {
        // the frame's packed source has been waiting since the converter hook: the whole pyramid, all channels, one GPU pass
        PendingSource ps = t_pending;
        t_pending = PendingSource();
        t_pyramid_done_for = nullptr; t_cuda_failed = false; t_sparse.valid = t_sparse.armed = false;
        if (run_pyramid(ps.plan, ps.data, ps.pitch, transform, CFB_PROGRESSIVE, ps.bayer_phase, ps.curve_mode) == NOT_COVERED) {
            // cannot happen after covered_plan(); if it does the planes were never converted: report, do not guess
            fprintf(stderr, "cfhd_gpu_shim: recorded source no longer covered\n");
            g_cuda_errors++; t_cuda_failed = true; t_pyramid_done_for = transform[0];
        }
    }
    if (t_pyramid_done_for && t_pyramid_done_for == transform[0]) {
        // levels 2 and 3 came out of the same GPU pass as level 1: only the bookkeeping of encoder.c:8366-8420 / :8688-8790 remains
        t_pyramid_done_for = nullptr;
        if (t_cuda_failed) { encoder->error = CODEC_ERROR_UNEXPECTED; t_cuda_failed = false; }
        if (t_sparse.armed) { t_sparse.encoder = encoder; t_sparse.frame_count = (uint32_t)encoder->frame_count; t_sparse.valid = true; t_sparse.armed = false; }
        for (int c = 0; c < num_transforms; c++) {
            transform[c]->num_frames = encoder->gop_length;
            transform[c]->num_spatial = encoder->num_spatial;
            transform[c]->num_levels = encoder->num_spatial + 1;
            transform[c]->num_wavelets = encoder->num_spatial + 1;
        }
        return;
    }
    t_sparse.valid = t_sparse.armed = false;
    ref(encoder, transform, num_transforms);
}

// ------------------------------------------------------------------------------------------------ decoder
// The CFB_PIXEL_* output the decoder's DECODED_FORMAT_* maps to for this sample, -1 where the reference keeps the frame:
//   4:2:2 samples, precision 10: 8-bit YUYV / UYVY, progressive or interlaced (field transform at level 1); YU64 and V210
//     progressive only (decoder.c:26292 / :26351; the reference renders them from a field transform only through its
//     active-metadata path, decoder.c:26413);
//   RGB 4:4:4 samples, 3 channels, precision 12, progressive: RG48, B64A and the 10-bit words (decoder.c:26862-26907).
// Everything else stays with the reference: RGB 4:4:4 -> YU64 / V210 (a colour conversion, TransformInverseRGB444ToYU64
// at decoder.c:26874), 8-bit RGB, RG64, Bayer.
static int gpu_output_format(const DECODER *d)
{
    const CODEC_STATE *cs = &d->codec;
    if (cs->num_channels != 3) return -1;
    const int f = d->frame.format;
    if (cs->encoded_format == ENCODED_FORMAT_YUV_422 && cs->precision == 10) {
        if (f == DECODED_FORMAT_YUYV) return CFB_PIXEL_YUYV;
        if (f == DECODED_FORMAT_UYVY) return CFB_PIXEL_UYVY;
        if (!cs->progressive) return -1;
        if (f == DECODED_FORMAT_YU64) return CFB_PIXEL_YU64;
        if (f == DECODED_FORMAT_V210) return CFB_PIXEL_V210;
        return -1;
    }
    if (cs->encoded_format == ENCODED_FORMAT_RGB_444 && cs->precision == 12 && cs->progressive) {
        switch (f) {
        case DECODED_FORMAT_RG48: return CFB_PIXEL_RG48;
        case DECODED_FORMAT_B64A: return CFB_PIXEL_B64A;
        case DECODED_FORMAT_RG30: return CFB_PIXEL_RG30;
        case DECODED_FORMAT_AB10: return CFB_PIXEL_AB10;
        case DECODED_FORMAT_AR10: return CFB_PIXEL_AR10;
        case DECODED_FORMAT_R210: return CFB_PIXEL_R210;
        case DECODED_FORMAT_DPX0: return CFB_PIXEL_DPX0;
        default: return -1;
        }
    }
    return -1;
}

// bytes the inverse writes per row of `w` pixels in output format `fmt`
static size_t output_row_bytes(int fmt, int w)
{
    switch (fmt) {
    case CFB_PIXEL_YU64: case CFB_PIXEL_RG30: case CFB_PIXEL_AB10: case CFB_PIXEL_AR10: case CFB_PIXEL_R210: case CFB_PIXEL_DPX0:
        return (size_t)w * 4;
    case CFB_PIXEL_V210: return (size_t)(w + 5) / 6 * 16;
    case CFB_PIXEL_RG48: return (size_t)w * 6;
    case CFB_PIXEL_B64A: return (size_t)w * 8;
    default: return (size_t)w * 2;
    }
}

static bool decoder_on_gpu(DECODER *d)
{
    if (!gpu_enabled() || !d) return false;
    const int out = gpu_output_format(d);
    if (out < 0) return false;
    // V210 packs 6 pixels per group, so a display window narrower than the coded row (4:2:2 rows are coded in multiples of
    // 16 pixels) is not a prefix of it: decided here, before ReconstructWaveletBand skips the CPU levels
    if (out == CFB_PIXEL_V210 && d->frame.width % 16) return false;
    if (d->frame.resolution != DECODED_RESOLUTION_FULL) return false;
    if (d->use_active_metadata_decoder || d->channel_blend_type) return false;
    if (d->uncompressed_chunk && d->uncompressed_size && d->sample_uncompressed) return false;
    for (int c = 0; c < 3; c++) if (!d->transform[c] || d->transform[c]->type != TRANSFORM_TYPE_SPATIAL) return false;
    return true;
}

void ReconstructWaveletBand(DECODER *decoder, TRANSFORM *transform, int channel, IMAGE *wavelet, int index, int precision,
                            const SCRATCH *scratch, int allocations_only)
{
    typedef void (*fn_t)(DECODER *, TRANSFORM *, int, IMAGE *, int, int, const SCRATCH *, int);
    static fn_t ref = next_symbol<fn_t>("ReconstructWaveletBand");
    if (!decoder_on_gpu(decoder) || allocations_only || index <= 0 || index > 3) {
        ref(decoder, transform, channel, wavelet, index, precision, scratch, allocations_only);
        return;
    }
    // Keep the reference's bookkeeping (allocate the lower wavelet, band-valid flags: decoder.c:12998-13040) but skip the
    // CPU inverse of this level: the whole pyramid is inverted in one GPU pass in ReconstructSampleFrameToBuffer.
    ref(decoder, transform, channel, wavelet, index, precision, scratch, 1);
    if (!BANDS_ALL_VALID(wavelet)) { decoder->error = CODEC_ERROR_BAD_FRAME; return; }
    IMAGE *lowpass = transform->wavelet[index - 1];
    if (lowpass && (lowpass->band_valid_flags & BAND_VALID_MASK(0)) == 0) UpdateWaveletBandValidFlags(decoder, lowpass, 0);
}

void ReconstructSampleFrameToBuffer(DECODER *decoder, int frame, uint8_t *output, int pitch)
{
    typedef void (*fn_t)(DECODER *, int, uint8_t *, int);
    static fn_t ref = next_symbol<fn_t>("ReconstructSampleFrameToBuffer");
    Plan *plan = nullptr;
    if (decoder_on_gpu(decoder) && output && pitch > 0 && (pitch & 15) == 0 && ((uintptr_t)output & 15) == 0 &&
        (decoder->flags & DECODER_FLAGS_RENDER)) {
        WaitForTransformThread(decoder);        // all entropy / bookkeeping jobs of this sample have finished
        IMAGE *y1 = decoder->transform[0]->wavelet[0];
        // the plan's source format only names the sample's family: 4:2:2 (the 8-bit outputs keep their own, as before) or
        // RGB 4:4:4; the output format is chosen per call.  Interlaced samples: the entropy decoder has already
        // integrated the level-1 HL band (decoder.c:20822)
        const int out = gpu_output_format(decoder);
        const int family = (out == CFB_PIXEL_YUYV || out == CFB_PIXEL_UYVY) ? out
                         : (decoder->codec.encoded_format == ENCODED_FORMAT_YUV_422 ? CFB_PIXEL_YUYV : CFB_PIXEL_RG48);
        if (y1) plan = get_plan(y1->width * 2, y1->height * 2, family, decoder->codec.progressive ? CFB_PROGRESSIVE : CFB_INTERLACED_HL_INTEGRATED);
    }
    bool ok = plan != nullptr;
    for (int c = 0; c < 3 && ok; c++)
        for (int k = 0; k < 3 && ok; k++) {
            IMAGE *w = decoder->transform[c]->wavelet[k];
            const cfb_band_layout &b = plan->layout.band[c][k][1];
            ok = w && w->width == b.width && w->height == b.height && w->pitch == b.pitch;
        }
    if (!ok) { g_inv_ref++; release_plans(); ref(decoder, frame, output, pitch); return; }
    decoder->gop_frame_num = frame;
    // the FSM entropy decoder already multiplied by the quantiser (decoder.c:20551): divisors = 1 here
    cfb_quant q;
    memset(&q, 0, sizeof(q));
    q.midpoint_prequant = 2;
    for (int k = 0; k < 3; k++) q.prescale[k] = decoder->transform[0]->prescale[k];
    for (int c = 0; c < 3; c++) for (int k = 0; k < 3; k++) for (int b = 0; b < 4; b++) q.divisor[c][k][b] = 1;
    // Hand-over of the decoder's bands (the FSM entropy decoder wrote them dense, decoder.c:19534-19808).  Default: staged
    // copy + dense upload (33 MB per 4K frame; 8.8 ms per 4K decode on the B200 box).  CFHD_B200_DECODE_SPARSE=1: the host
    // reads the bands once, straight into the sparse transfer format, and ~1/8 of the bytes cross PCIe -- less PCIe and
    // host-memory traffic when many decoders share a link, but the single-threaded compaction makes one decode slower
    // (11.9 ms), so it is opt-in.
    static const bool decode_sparse = getenv("CFHD_B200_DECODE_SPARSE") && *getenv("CFHD_B200_DECODE_SPARSE") == '1';
    const bool sparse = decode_sparse && sparse_enabled() && plan->ensure_sparse();
    if (!sparse && !plan->ensure_coded()) { g_inv_ref++; release_plans(); ref(decoder, frame, output, pitch); return; }
    if (sparse) {
        const void *ptrs[CFB_MAX_CHANNELS * CFB_NUM_LEVELS * CFB_NUM_BANDS] = {};
        int32_t pitches[CFB_MAX_CHANNELS * CFB_NUM_LEVELS * CFB_NUM_BANDS] = {};
        for (int c = 0; c < 3; c++)
            for (int k = 0; k < 3; k++) {
                IMAGE *w = decoder->transform[c]->wavelet[k];
                for (int bnd = (k == 2 ? 0 : 1); bnd < 4; bnd++) {
                    ptrs[(c * CFB_NUM_LEVELS + k) * CFB_NUM_BANDS + bnd] = w->band[bnd];
                    pitches[(c * CFB_NUM_LEVELS + k) * CFB_NUM_BANDS + bnd] = w->pitch;
                }
            }
        if (cfb_sparse_compact_bands(&plan->layout, ptrs, pitches, plan->sparse, nullptr) != CFB_OK) { g_inv_ref++; release_plans(); ref(decoder, frame, output, pitch); return; }
    } else
    for (int c = 0; c < 3; c++)
        for (int k = 0; k < 3; k++) {
            IMAGE *w = decoder->transform[c]->wavelet[k];
            for (int bnd = (k == 2 ? 0 : 1); bnd < 4; bnd++) {
                const cfb_band_layout &b = plan->layout.band[c][k][bnd];
                memcpy((char *)plan->coded + b.offset, w->band[bnd], (size_t)b.pitch * b.height);
            }
        }
    const void *coded[1] = {sparse ? plan->sparse : plan->coded};
    const int fmt = gpu_output_format(decoder);
    // The pyramid has the ENCODED size (height rounded up to a multiple of 8, encoder.c:2232: 720x486 is coded as 488
    // rows) while the caller's buffer holds the DISPLAY size (decoder->frame): the reference writes info->height rows of
    // info->width pixels only.  When the two differ the frame is decoded into a staging buffer and the display window is
    // copied out, so nothing is ever written past the caller's last row.
    const int enc_w = plan->layout.band[0][0][0].width * 2, enc_h = plan->layout.band[0][0][0].height * 2;
    const int out_w = decoder->frame.width, out_h = decoder->frame.height;
    const size_t row_bytes = output_row_bytes(fmt, out_w);
    // V210 packs 6 pixels per group, and its last group depends on the row width: a narrower display window is not a
    // prefix of the coded row
    const bool window_ok = out_w == enc_w || fmt != CFB_PIXEL_V210;
    if (out_w <= 0 || out_h <= 0 || out_w > enc_w || out_h > enc_h || (size_t)pitch < row_bytes || !window_ok) {
        g_inv_ref++; release_plans(); ref(decoder, frame, output, pitch); return;
    }
    cfb_error err;
    if (out_w == enc_w && out_h == enc_h) {
        void *frames[1] = {output};
        err = sparse ? cfb_inverse_host_sparse(plan->codec, 1, coded, &q, fmt, frames, pitch) : cfb_inverse_host(plan->codec, 1, coded, &q, fmt, frames, pitch);
    } else {
        const int fpitch = (int)((output_row_bytes(fmt, enc_w) + 15) & ~(size_t)15);
        void *frames[1] = {plan->ensure_frame((size_t)fpitch * enc_h) ? plan->frame : nullptr};
        err = !frames[0] ? CFB_ERROR_OUTOFMEMORY : sparse ? cfb_inverse_host_sparse(plan->codec, 1, coded, &q, fmt, frames, fpitch)
                                                         : cfb_inverse_host(plan->codec, 1, coded, &q, fmt, frames, fpitch);
        if (err == CFB_OK)
            for (int r = 0; r < out_h; r++)
                memcpy(output + (size_t)r * pitch, (const char *)plan->frame + (size_t)r * fpitch, row_bytes);
    }
    if (err != CFB_OK) {
        fprintf(stderr, "cfhd_gpu_shim: CUDA inverse failed: %s\n", cfb_last_error_string());
        g_cuda_errors++;
        if (getenv("CFHD_B200_ABORT_ON_ERROR")) abort();
        decoder->error = CODEC_ERROR_BAD_FRAME;
    }
    g_inv_frames++;
    release_plans();
}

// ------------------------------------------------------------------------------------------------ preparation
// Plans (context, device staging, pinned buffers: tens of milliseconds each, more when sixteen threads create theirs at
// once) are created when the application PREPARES its encoder / encoder pool, as any allocation of that size would be,
// not inside its first EncodeSample calls.  Without this, Example/TestCFHD.cpp -E -- a new pool and 500 frames per row --
// spends most of a row creating plans.
static int cfb_format_of_pixel_format(CFHD_PixelFormat pf, CFHD_EncodedFormat ef)
{
    const bool yuv = (ef == CFHD_ENCODED_FORMAT_YUV_422), rgb = (ef == CFHD_ENCODED_FORMAT_RGB_444);
    switch (pf) {
    case CFHD_PIXEL_FORMAT_YUY2: return yuv ? CFB_PIXEL_YUYV : -1;
    case CFHD_PIXEL_FORMAT_2VUY: return yuv ? CFB_PIXEL_UYVY : -1;
    case CFHD_PIXEL_FORMAT_YU64: return yuv ? CFB_PIXEL_YU64 : -1;
    case CFHD_PIXEL_FORMAT_V210: return yuv ? CFB_PIXEL_V210 : -1;
    case CFHD_PIXEL_FORMAT_RG48: return rgb ? CFB_PIXEL_RG48 : -1;
    case CFHD_PIXEL_FORMAT_RG30: return rgb ? CFB_PIXEL_RG30 : -1;
    case CFHD_PIXEL_FORMAT_R210: return rgb ? CFB_PIXEL_R210 : -1;
    case CFHD_PIXEL_FORMAT_DPX0: return rgb ? CFB_PIXEL_DPX0 : -1;
    case CFHD_PIXEL_FORMAT_AB10: return rgb ? CFB_PIXEL_AB10 : -1;
    case CFHD_PIXEL_FORMAT_AR10: return rgb ? CFB_PIXEL_AR10 : -1;
    case CFHD_PIXEL_FORMAT_BYR4: return (ef == CFHD_ENCODED_FORMAT_BAYER) ? CFB_PIXEL_BYR4 : -1;
    default: return -1;
    }
}

static void prewarm_plans(int count, int width, int height, CFHD_PixelFormat pf, CFHD_EncodedFormat ef, CFHD_EncodingFlags flags)
{
    const int fmt = cfb_format_of_pixel_format(pf, ef);
    if (fmt < 0 || count < 1 || !gpu_enabled() || getenv("CFHD_B200_NO_PREWARM")) return;
    const int h8 = (height + 7) & ~7;                       // the coded height (encoder.c:2232)
    const int interlaced = ((flags & CFHD_ENCODING_FLAGS_YUV_INTERLACED) && (fmt == CFB_PIXEL_YUYV || fmt == CFB_PIXEL_UYVY)) ? CFB_INTERLACED : CFB_PROGRESSIVE;
    std::vector<std::thread> th;
    for (int i = 0; i < count && i < 64; i++)
        th.emplace_back([=] {
            Plan *p = get_plan(width, h8, fmt, interlaced);
            if (p) {
                // one transform of a grey frame: loads the kernels, allocates the codec's lazily created device buffers and pins
                // the host staging this plan will use
                const bool sparse = sparse_enabled() && interlaced == CFB_PROGRESSIVE && p->ensure_sparse();
                std::vector<uint8_t> frame((size_t)p->layout.frame_bytes + 64, 0x80);
                uint8_t *f = (uint8_t *)(((uintptr_t)frame.data() + 63) & ~(uintptr_t)63);
                cfb_quant q;
                cfb_frame_desc d = {width, h8, fmt, 0};
                if (p->ensure_coded() && cfb_quant_for_source(&d, 4, interlaced != CFB_PROGRESSIVE, &q) == CFB_OK) {
                    const void *frames[1] = {f};
                    void *out[1] = {sparse ? p->sparse : p->coded};
                    if (sparse) cfb_forward_host_sparse(p->codec, 1, frames, p->layout.frame_pitch, &q, out, nullptr);
                    else cfb_forward_host(p->codec, 1, frames, p->layout.frame_pitch, &q, out);
                }
            }
            release_plans();        // back to the pool, ready for whichever encoder thread asks first
        });
    for (auto &t : th) t.join();
}

static std::mutex g_pool_mu;
static std::map<void *, int> g_pool_threads;                // encoder pool -> its thread count

CFHD_Error CFHD_CreateEncoderPool(CFHD_EncoderPoolRef *encoderPoolRefOut, int encoderThreadCount, int jobQueueLength, CFHD_ALLOCATOR *allocator)
{
    typedef CFHD_Error (*fn_t)(CFHD_EncoderPoolRef *, int, int, CFHD_ALLOCATOR *);
    static fn_t ref = next_symbol<fn_t>("CFHD_CreateEncoderPool");
    const CFHD_Error e = ref(encoderPoolRefOut, encoderThreadCount, jobQueueLength, allocator);
    if (e == CFHD_ERROR_OKAY && encoderPoolRefOut && *encoderPoolRefOut) {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        g_pool_threads[(void *)*encoderPoolRefOut] = encoderThreadCount;
    }
    return e;
}

CFHD_Error CFHD_PrepareEncoderPool(CFHD_EncoderPoolRef encoderPoolRef, uint_least16_t frameWidth, uint_least16_t frameHeight,
                                   CFHD_PixelFormat pixelFormat, CFHD_EncodedFormat encodedFormat, CFHD_EncodingFlags encodingFlags,
                                   CFHD_EncodingQuality encodingQuality)
{
    typedef CFHD_Error (*fn_t)(CFHD_EncoderPoolRef, uint_least16_t, uint_least16_t, CFHD_PixelFormat, CFHD_EncodedFormat, CFHD_EncodingFlags, CFHD_EncodingQuality);
    static fn_t ref = next_symbol<fn_t>("CFHD_PrepareEncoderPool");
    const CFHD_Error e = ref(encoderPoolRef, frameWidth, frameHeight, pixelFormat, encodedFormat, encodingFlags, encodingQuality);
    if (e == CFHD_ERROR_OKAY) {
        int n = 0;
        { std::lock_guard<std::mutex> lk(g_pool_mu); auto it = g_pool_threads.find((void *)encoderPoolRef); if (it != g_pool_threads.end()) n = it->second; }
        prewarm_plans(n, frameWidth, frameHeight, pixelFormat, encodedFormat, encodingFlags);
    }
    return e;
}

CFHD_Error CFHD_PrepareToEncode(CFHD_EncoderRef encoderRef, int frameWidth, int frameHeight, CFHD_PixelFormat pixelFormat,
                                CFHD_EncodedFormat encodedFormat, CFHD_EncodingFlags encodingFlags, CFHD_EncodingQuality encodingQuality)
{
    typedef CFHD_Error (*fn_t)(CFHD_EncoderRef, int, int, CFHD_PixelFormat, CFHD_EncodedFormat, CFHD_EncodingFlags, CFHD_EncodingQuality);
    static fn_t ref = next_symbol<fn_t>("CFHD_PrepareToEncode");
    const CFHD_Error e = ref(encoderRef, frameWidth, frameHeight, pixelFormat, encodedFormat, encodingFlags, encodingQuality);
    if (e == CFHD_ERROR_OKAY) prewarm_plans(1, frameWidth, frameHeight, pixelFormat, encodedFormat, encodingFlags);
    return e;
}

}  // extern "C"
