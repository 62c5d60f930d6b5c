/* cfhd_b200.h -- C ABI of the B200-native CineForm transform path.
 *
 * Drop-in boundary for the one hot path of gopro/cineform-sdk that this library
 * replaces: the 3-level 2-6 wavelet pyramid + per-subband quantise/dequantise.
 * Plain C, plain pointers and sizes; no torch / C++ types cross this boundary.
 *
 * What each entry point replaces in the reference (paths relative to the
 * reference tree):
 *
 *   cfb_forward_*      Codec/encoder.c:3121  TransformForwardSpatialYUV (level 1, packed 4:2:2)
 *                      Codec/encoder.c:3193  TransformForwardSpatial    (level 1, planar channels)
 *                      Codec/encoder.c:3254  ComputeGroupTransformQuant (levels 2,3)
 *                      i.e. Codec/wavelet.c:2823/:2420 -> Codec/spatial.c:14726/:10026/:12942
 *                      + Codec/quantize.c:1395 QuantizeRow16sTo16s, for every channel of a frame.
 *   cfb_inverse_*      Codec/decoder.c:11756/:11765 ReconstructWaveletBand (levels 3->2, 2->1)
 *                      i.e. Codec/wavelet.c:5685 TransformInverseSpatialQuantLowpass ->
 *                      Codec/spatial.c:21877/:22414 + Codec/InvertHorizontalStrip16s.c:459/:1700,
 *                      and Codec/decoder.c:11836 ReconstructSampleFrameToBuffer (level 1 -> pixels),
 *                      with the dequantisation of Codec/decoder.c:20551 DeQuantFSM fused into the load.
 *   cfb_layout_*       Codec/wavelet.c:427 AllocWaveletStack / :302 InitWaveletStack / :1173 AllocTransform
 *                      (band pitch = ALIGN16(2*width), bands 64-byte aligned).
 *   cfb_quant_*        Codec/quantize.c:186 QuantizationSetQuality + :2865 SetTransformQuantization +
 *                      Codec/wavelet.c:1710 SetTransformPrescale (host-side table derivation).
 *   cfb_pool_*         EncoderSDK/EncoderPool.cpp:239 CEncoderPool::EncodeSample / EncoderQueue.h:311-352
 *                      (bounded, in-order frame queue) re-hosted on GPU streams, frames sharded over GPUs.
 *
 * There is NO CPU fallback: every transform call runs CUDA kernels on an sm_100a
 * device and fails with CFB_ERROR_NO_DEVICE / CFB_ERROR_CUDA otherwise.
 */
#ifndef CFHD_B200_H
#define CFHD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define CFB_API __declspec(dllexport)
#else
#define CFB_API __attribute__((visibility("default")))
#endif

/* Error codes: 0,1,2,10 carry the meaning of the same values in Common/CFHDError.h:25-84. */
typedef enum cfb_error {
    CFB_OK = 0,
    CFB_ERROR_INVALID_ARGUMENT = 1,
    CFB_ERROR_OUTOFMEMORY = 2,
    CFB_ERROR_BADFORMAT = 3,
    CFB_ERROR_UNEXPECTED = 10,
    CFB_ERROR_NOT_FINISHED = 13,
    CFB_ERROR_NO_DEVICE = 100,      /* no CUDA device / not sm_100 */
    CFB_ERROR_CUDA = 101,           /* a CUDA call failed; see cfb_last_error_string() */
    CFB_ERROR_UNSUPPORTED = 102,    /* geometry the kernels do not cover (see cfb_frame_desc) */
    CFB_ERROR_RANGE = 103           /* a signed plane outside the range in which exact and saturating arithmetic agree */
} cfb_error;

/* Input / output pixel layouts of level 1 (the reference's COLOR_FORMAT_* subset used by the
 * BASELINE configs; Codec/encoder.c:2336-2865). */
typedef enum cfb_pixel_format {
    CFB_PIXEL_YUYV = 0,     /* 8-bit packed 4:2:2  Y0 U Y1 V  (CFHD_PIXEL_FORMAT_YUY2)          */
    CFB_PIXEL_UYVY = 1,     /* 8-bit packed 4:2:2  U Y0 V Y1  (CFHD_PIXEL_FORMAT_2VUY)          */
    CFB_PIXEL_RG48 = 2,     /* 16-bit packed R,G,B -> 3 planes G,R,B at 12 bits (frame.c:5968)  */
    CFB_PIXEL_BYR4 = 3,     /* 16-bit Bayer -> 4 half-size planes at 12 bits   (frame.c:4993)  */
    CFB_PIXEL_PLANAR16 = 4, /* channels already unpacked to int16 planes (testing / chaining)   */
    CFB_PIXEL_YU64 = 5,     /* 16-bit packed 4:2:2  Y0 C1 Y1 C3 -> 10-bit planes, C1 -> channel 1, C3 -> channel 2
                             * (CFHD_PIXEL_FORMAT_YU64; frame.c:1556 ConvertYU64ToFrame16s); input only */
    CFB_PIXEL_V210 = 6,     /* 10-bit packed 4:2:2, components Cb Y Cr Y ... three per 32-bit word, rows padded to
                             * 128 bytes (CFHD_PIXEL_FORMAT_V210; encoder.c:2518 ConvertV210ToFrame16s: Cb -> channel 2,
                             * Cr -> channel 1).  As an OUTPUT (4:2:2 codecs, full resolution, progressive): see cfb_inverse_device */
    /* 10-bit packed RGB, one 32-bit word per pixel -> 3 planes G, R, B at 12 bits like RG48 (encoder.c:3158-3176
     * TransformForwardSpatialRGB30, field layouts spatial.c:2118-2268); input only */
    CFB_PIXEL_RG30 = 7,     /* R bits 0-9, G 10-19, B 20-29 (CFHD_PIXEL_FORMAT_RG30)                       */
    CFB_PIXEL_AB10 = 8,     /* same layout (A2B10G10R10)                                                   */
    CFB_PIXEL_AR10 = 9,     /* B bits 0-9, G 10-19, R 20-29 (A2R10G10B10)                                   */
    CFB_PIXEL_R210 = 10,    /* big-endian word: R 20-29, G 10-19, B 0-9 after the byte swap               */
    CFB_PIXEL_DPX0 = 11,    /* big-endian word: R 22-31, G 12-21, B 2-11 after the byte swap              */
    CFB_PIXEL_B64A = 12     /* OUTPUT only: 16-bit A,R,G,B words of an RGB 4:4:4 sample (DECODED_FORMAT_B64A at the codec level,
                             * Codec/decoder.c:26862 -> InvertHorizontalStrip16s.c:13298): alpha = 0xfff0, colours limited to
                             * 0xfff0 in the columns of the reference's SSE2 loop and to 65535 in its scalar tail / right
                             * border, native word order as the reference's decoder writes them */
} cfb_pixel_format;

enum { CFB_MAX_CHANNELS = 4, CFB_NUM_LEVELS = 3, CFB_NUM_BANDS = 4 };

/* Geometry of one frame. width/height are the FRAME dimensions in pixels.
 * Requirements (else CFB_ERROR_UNSUPPORTED): height % 8 == 0 (the reference rounds
 * up to 8, encoder.c:2236)
 * (4:2:2: width % 16 == 0, as the reference's row unpackers require; 4:4:4: width % 8 == 0; Bayer: width % 16 == 0;
 * channel heights % 8 == 0 and >= 48).  Band widths that are not a multiple of the kernels' lane granularity (e.g. 720 or
 * 1440 wide sources: chroma LL3 is 45 / 90 wide) are handled by small edge kernels. */
typedef struct cfb_frame_desc {
    int32_t width;
    int32_t height;
    int32_t pixel_format;       /* cfb_pixel_format */
    int32_t reserved;
} cfb_frame_desc;

/* One band of the pyramid inside a coefficient buffer. */
typedef struct cfb_band_layout {
    int64_t offset;     /* bytes from the start of the frame's coefficient buffer */
    int32_t width;      /* coefficients per row */
    int32_t height;     /* rows */
    int32_t pitch;      /* bytes per row = ALIGN16(2*width) (wavelet.c:439-442) */
    int32_t reserved;
} cfb_band_layout;

/* Per-frame coefficient buffer ("pyramid"). All int16, little endian.
 *   [0, coded_bytes)            what the entropy coder consumes / produces:
 *                               per channel: LL3, then LH,HL,HH of levels 3,2,1
 *   [coded_bytes, total_bytes)  device-side scratch: LL1, LL2 of every channel
 * band[c][k][b]: channel c, level k (0 = level 1 ... 2 = level 3), band b
 * (0 = LL, 1 = LH "lowhigh", 2 = HL "highlow", 3 = HH, numbering of Codec/image.h:237). */
typedef struct cfb_layout {
    int32_t num_channels;
    int32_t precision;          /* 10 (4:2:2 sources) or 12 (RGB / Bayer), encoder.c:2480 */
    int64_t coded_bytes;
    int64_t total_bytes;
    int64_t frame_bytes;        /* bytes of one packed input/output frame at the natural pitch */
    int32_t frame_pitch;        /* natural pitch of the packed frame in bytes */
    int32_t reserved;
    cfb_band_layout band[CFB_MAX_CHANNELS][CFB_NUM_LEVELS][CFB_NUM_BANDS];
} cfb_layout;

/* Quantisation schedule of one frame: divisors per channel/level/band (band 0 = LL, normally 1),
 * the level prescale shifts ({0,2,0} for 10-bit, {0,2,2} for 12-bit, wavelet.c:1710-1782) and the
 * quantiser midpoint rule (quantize.c:1415-1427: g = 2 + pre-emphasis bits). */
typedef struct cfb_quant {
    int32_t prescale[CFB_NUM_LEVELS];
    int32_t midpoint_prequant;
    int32_t divisor[CFB_MAX_CHANNELS][CFB_NUM_LEVELS][CFB_NUM_BANDS];
} cfb_quant;

typedef struct cfb_context cfb_context;     /* one CUDA device + stream pool      */
typedef struct cfb_codec cfb_codec;         /* plan for one frame geometry        */
typedef struct cfb_pool cfb_pool;           /* async, in-order, multi-GPU frame queue */

/* ---- library / device ---------------------------------------------------- */
CFB_API int cfb_version(void);
CFB_API const char *cfb_last_error_string(void);              /* thread-local */
CFB_API int cfb_device_count(void);                           /* 0 when no usable GPU */
/* NUMA placement (Linux): node of the GPU's PCIe root (-1 if unknown) and a helper that restricts the CALLING thread to
 * that node's CPUs, so that pinned buffers it allocates afterwards (cfb_host_alloc) and the copies it issues are local
 * to the GPU.  The pool binds its own worker threads.  The reference sets worker-thread affinity likewise
 * (Codec/thread.c:SetThreadAffinityMask). */
CFB_API int cfb_device_numa_node(int device);
CFB_API cfb_error cfb_bind_thread_to_device(int device);

CFB_API cfb_error cfb_context_create(int device, cfb_context **out);
CFB_API void cfb_context_destroy(cfb_context *ctx);
CFB_API cfb_error cfb_context_synchronize(cfb_context *ctx);
CFB_API void *cfb_context_stream(cfb_context *ctx);           /* the cudaStream_t kernels are launched on */

/* ---- geometry + quantisation tables (host only; usable without a GPU) ---- */
CFB_API cfb_error cfb_layout_compute(const cfb_frame_desc *desc, cfb_layout *out);
/* FILMSCAN-style fixed quality (CFHD_EncodingQuality low byte 1..6, Common/CFHDTypes.h:200-223). */
CFB_API cfb_error cfb_quant_for_quality(const cfb_frame_desc *desc, int quality, cfb_quant *out);
/* Same, for an interlaced source (parameters.progressive = 0): the level-1 LH divisor * 3/2 and HL * 2/3
 * (Codec/quantize.c:490-541). */
CFB_API cfb_error cfb_quant_for_source(const cfb_frame_desc *desc, int quality, int interlaced, cfb_quant *out);

/* ---- codec plan ---------------------------------------------------------- */
/* max_batch = frames processed per launch (1..CFB_MAX_BATCH). Allocates device staging for
 * max_batch packed frames and max_batch pyramids plus pinned host staging. */
enum { CFB_MAX_BATCH = 16 };
CFB_API cfb_error cfb_codec_create(cfb_context *ctx, const cfb_frame_desc *desc, int max_batch, cfb_codec **out);
CFB_API void cfb_codec_destroy(cfb_codec *codec);
CFB_API cfb_error cfb_codec_layout(const cfb_codec *codec, cfb_layout *out);
/* device staging owned by the codec: slot i in [0, max_batch) */
CFB_API void *cfb_codec_device_frame(cfb_codec *codec, int slot);
CFB_API void *cfb_codec_device_pyramid(cfb_codec *codec, int slot);

/* BYR4 only: Bayer phase of the source (TAG_BAYER_FORMAT): 0 RED_GRN, 1 GRN_RED, 2 GRN_BLU, 3 BLU_GRN
 * (Codec/DemoasicFrames.h:30-33). */
CFB_API cfb_error cfb_codec_set_bayer_phase(cfb_codec *codec, int bayer_format);
/* BYR4 only: the encode curve the reference builds per call (Codec/frame.c:5208-5330, default log base 90) as a table of
 * 1 << 14 12-bit values indexed by sample >> 2; the kernel applies it while loading.  NULL (default) = the frame already
 * carries its curve (CFHD_ENCODING_FLAGS_CURVE_APPLIED / encode_curve_preset): samples >> 4. */
CFB_API cfb_error cfb_codec_set_bayer_curve(cfb_codec *codec, const uint16_t *curve, int entries);

/* Interlaced sources (CFHD_ENCODING_FLAGS_YUV_INTERLACED, EncoderSDK/SampleEncoder.cpp:210 -> parameters.progressive = 0;
 * on decode the sample's progressive flag): level 1 of the following forward/inverse calls is the frame (field)
 * transform -- vertical Haar between the two fields + horizontal 2-6, HL band difference coded along each row --
 * instead of the spatial transform.  Replaces Codec/encoder.c:2976 TransformForwardFrameYUV (wavelet.c:6076; planar
 * form filter.c:273 FilterFrameQuant16s) and Codec/decoder.c:21493 TransformInverseFrameToYUV / :22027 ...ToRow16u
 * (temporal.c:3741 InvertInterlaced16s) including the HL row integration of decoder.c:20822-20836.
 * 4:2:2 codecs: packed 8-bit (YUYV, UYVY: the packed routine) and YU64 / V210 (the planar routine filter.c:273, whose LH
 * band is rounded with divisor / 2 in the columns of its SSE2 loop and without a midpoint in its scalar tail and last column,
 * spatial.c:5826-6266).  Reduced-resolution decodes of an interlaced sample (cfb_codec_set_decode_resolution)
 * return the lowpass image LL1 / LL2 exactly as the reference does: its half- and quarter-resolution paths
 * (Codec/decoder.c:26078 and :11818) run before / outside the progressive-vs-interlaced split of
 * ReconstructSampleFrameToBuffer, so the level-1 transform type does not enter. */
enum { CFB_PROGRESSIVE = 0, CFB_INTERLACED = 1,
       /* inverse only: the level-1 HL band arrives already integrated along its rows, i.e. exactly as the reference's
        * entropy decoder leaves it (decoder.c:20822-20836); the GPU then skips its own prefix sum */
       CFB_INTERLACED_HL_INTEGRATED = 2 };
CFB_API cfb_error cfb_codec_set_interlaced(cfb_codec *codec, int interlaced);

/* Decoded resolution of the following cfb_inverse_* calls: the decodedResolution argument of CFHD_PrepareToDecode
 * (DecoderSDK/CFHDDecoder.cpp; Common/CFHDTypes.h:453-456, same numbering).  HALF stops after level 2 -> 1 and
 * returns the lowpass image LL1 (Codec/decoder.c:26078-26160 -> CopyLowpass16sToBuffer :22883 ->
 * ConvertLowpass16s10bitToYUV frame.c:11742: sat_u8(ll >> 4)); QUARTER stops after level 3 -> 2 and returns LL2
 * (decoder.c:11818 -> ConvertQuarterFrameToBuffer :17000 -> CopyQuarterRowToBuffer temporal.c:11362:
 * packus((uint16)ll >> 4)).  CFB_PIXEL_PLANAR16 output returns the raw int16 lowpass planes instead.  The host
 * variants upload only the subbands the reduced decode reads (decoder.c:1965-1984 subband masks 0x7F / 0x0F). */
typedef enum cfb_resolution {
    CFB_RESOLUTION_FULL = 1,
    CFB_RESOLUTION_HALF = 2,
    CFB_RESOLUTION_QUARTER = 3
} cfb_resolution;
CFB_API cfb_error cfb_codec_set_decode_resolution(cfb_codec *codec, int resolution);
/* width/height (pixels) of the frames cfb_inverse_* writes at the current decode resolution */
CFB_API cfb_error cfb_codec_decoded_size(const cfb_codec *codec, int *width, int *height);

/* Profiling aid: restrict the following forward/inverse calls to a subset of pyramid levels
 * (bit k = level k+1; default 7 = all).  Used by bench.py to time one kernel in isolation. */
CFB_API cfb_error cfb_codec_set_level_mask(cfb_codec *codec, int forward_mask, int inverse_mask);

/* ---- forward: packed frames -> quantised pyramids ------------------------- */
/* Device-resident: frames and pyramids are DEVICE pointers (n of each); kernels only, asynchronous
 * on cfb_context_stream(). frame_pitch in bytes (16-byte aligned, positive). */
CFB_API cfb_error cfb_forward_device(cfb_codec *codec, int n, const void *const *d_frames, int frame_pitch,
                                     const cfb_quant *quant, void *const *d_pyramids);
/* Host buffers: copies each frame H2D, transforms, copies the coded region [0, coded_bytes)
 * of each pyramid D2H into h_coded[i]; returns when the data is in host memory. */
CFB_API cfb_error cfb_forward_host(cfb_codec *codec, int n, const void *const *h_frames, int frame_pitch,
                                   const cfb_quant *quant, void *const *h_coded);

/* ---- inverse: quantised pyramids -> packed frames -------------------------- */
/* The coded region holds QUANTISED values (as entropy-decoded with quant 1); dequantisation by
 * quant->divisor is fused into the kernels' loads. out_format: CFB_PIXEL_YUYV/UYVY (8-bit, see
 * DESIGN.md for the rounding rule), CFB_PIXEL_PLANAR16 (int16 planes at codec precision), and the 16-bit packed
 * outputs of the reference's final level, all bit-exact (no dither): CFB_PIXEL_YU64 from 4:2:2 codecs, CFB_PIXEL_RG48,
 * CFB_PIXEL_B64A and the 10-bit words CFB_PIXEL_RG30 / AB10 / AR10 / R210 / DPX0 (Codec/decoder.c:26893 ->
 * InvertHorizontalStrip16s.c:14812: the 12-bit sample limited to [0, 4095], >> 2) from RGB 4:4:4 codecs (full resolution,
 * progressive).  The reference's LOWPASS BAND DECODE adds a per-output-format constant to LL3 (decoder.c:12270-12316: 6 for
 * the 10-bit RGB outputs, 8 for 8-bit RGB, 0 for RG48 / B64A ...): that belongs to the host's band decode, the caller
 * passes the bands as its decoder holds them.
 * CFB_PIXEL_V210 from 4:2:2 codecs, full resolution and progressive only (else CFB_ERROR_UNSUPPORTED; a 4:4:4 codec gives
 * CFB_ERROR_BADFORMAT), bit-exact too: the reference renders it as YU64 rows (decoder.c:26292 ->
 * InvertHorizontalStrip16s.c:6490, the same ...ToRow16u rule as YU64) converted by convert.c:13526 ConvertPlanarYUVToV210
 * at precision 16, so every component is the YU64 sample >> 6 (both YU64 limits, 0xFFC0 and 65535, become 1023).  Words
 * Cb0 Y0 Cr0 | Y1 Cb2 Y2 | Cr2 Y3 Cb4 | Y4 Cr4 Y5 per 6 pixels, bits 0 / 10 / 20, Cb = channel 2, Cr = channel 1.  When
 * width % 6 != 0 the last group is completed as the reference's scalar tail does (convert.c:13888-13965: a component past
 * the right edge repeats the value its variable there last held), except the Cb field of word 2 when width % 6 == 4, which the
 * reference reads from outside the row (not reproducible); it is the row's last Cb here.  Exactly ceil(width / 6) * 16
 * bytes are written per row; frame_pitch must be at least that and a multiple of 16 (the SDK's own pitch rounds the row
 * to 128 bytes, SampleDecoder.cpp:367), the rest of the row is left untouched.  The LL3 constant of V210 is the YU64 one. */
CFB_API cfb_error cfb_inverse_device(cfb_codec *codec, int n, void *const *d_pyramids, const cfb_quant *quant,
                                     int out_format, void *const *d_frames, int frame_pitch);
CFB_API cfb_error cfb_inverse_host(cfb_codec *codec, int n, const void *const *h_coded, const cfb_quant *quant,
                                   int out_format, void *const *h_frames, int frame_pitch);



/* ---- two-frame GOP building block: temporal Haar between two int16 planes --------------------
 * In the reference's FIELDPLUS pyramid (CFHD_ENCODING_FLAGS_YUV_2FRAME_GOP; Codec/encoder.c:8431
 * FinishFieldPlusTransformQuant, Codec/decoder.c:13109) wavelet[2] is the temporal transform of the level-1 lowpass
 * images of frames A and B; the spatial levels above and below it are the same transforms as the intra-frame
 * pyramid.  forward replaces Codec/temporal.c:498 FilterTemporal16s (low = adds(f1, f2), high = subs(f2, f1));
 * inverse replaces Codec/temporal.c:9402 InvertTemporalQuant16s (f1 = subs(low, high) >> 1,
 * f2 = adds(low, high) >> 1 on dequantised coefficients; precision 8 adds the reference's half-tone bit).
 * Planes are int16, width a multiple of 16 (temporal.c:616), pitches in bytes, 16-byte aligned.
 * The _device forms take device pointers and run asynchronously on cfb_context_stream(). */
CFB_API cfb_error cfb_temporal_forward_device(cfb_context *ctx, const void *d_frame1, const void *d_frame2, int in_pitch,
                                              void *d_low, void *d_high, int out_pitch, int width, int height);
CFB_API cfb_error cfb_temporal_inverse_device(cfb_context *ctx, const void *d_low, const void *d_high, int in_pitch,
                                              void *d_frame1, void *d_frame2, int out_pitch, int width, int height,
                                              int precision);
CFB_API cfb_error cfb_temporal_forward_host(cfb_context *ctx, const void *frame1, const void *frame2, int in_pitch,
                                            void *low, void *high, int out_pitch, int width, int height);
CFB_API cfb_error cfb_temporal_inverse_host(cfb_context *ctx, const void *low, const void *high, int in_pitch,
                                            void *frame1, void *frame2, int out_pitch, int width, int height, int precision);

/* ---- single wavelet level on a free-standing int16 plane ----------------------------------------
 * forward = Codec/wavelet.c:2420 TransformForwardSpatial (spatial.c:10026 FilterSpatialQuant16s for prescale 0,
 * spatial.c:12942 FilterSpatialV210Quant16s for prescale 2); inverse = Codec/wavelet.c:5685
 * TransformInverseSpatialQuantLowpass (spatial.c:21877 / :22414, dequantisation fused).  With cfb_temporal_* these
 * compose the reference's other transform graphs, e.g. the two-frame-GOP FIELDPLUS pyramid (Codec/encoder.c:8431):
 *   wavelet[2] = temporal(LL1 of frame A, LL1 of frame B); wavelet[3] = level(temporal high);
 *   wavelet[4] = level(temporal low); wavelet[5] = level(LL of wavelet[4]).
 * width/height: the PLANE's dimensions (bands are width/2 x height/2); pitches in bytes, 16-byte aligned; bands[] in
 * the order LL, LH, HL, HH.  divisor[0] > 1 quantises LL in the forward direction only when prescale == 0, as the
 * reference does; the inverse carries LL undequantised. */
typedef struct cfb_level_desc {
    int32_t width, height;
    int32_t plane_pitch, band_pitch;
    int32_t prescale;               /* 0 or 2 (wavelet.c:1710 SetTransformPrescale) */
    int32_t midpoint_prequant;      /* quantiser midpoint rule, as cfb_quant */
    int32_t divisor[4];
} cfb_level_desc;
/* Value range.  The kernels compute in exact 32-bit arithmetic; the reference's SSE2 loops use saturating 16-bit chains
 * (spatial.c:290-413, :10290-10413).  The two agree whenever no chain input exceeds 8190 in magnitude (4 * 8190 + 4 is
 * the largest partial sum).  Every source format of the codec objects satisfies this by its declared precision
 * (DESIGN.md 4); a free-standing SIGNED plane (the temporal highpass of a two-frame GOP, +-4080 by range) need not.
 * The forward level therefore audits its input on the device -- |x| and both horizontal outputs of every pair against
 * the bound, one extra read of the plane -- and a violation is REPORTED, never silently computed differently from the
 * reference: the host forms return CFB_ERROR_RANGE, the asynchronous device form records it for
 * cfb_context_range_status (which waits for the stream, returns the flags and clears them; 0 = in range). */
CFB_API cfb_error cfb_context_range_status(cfb_context *ctx, int *flags);
CFB_API cfb_error cfb_level_forward_device(cfb_context *ctx, const cfb_level_desc *desc, const void *d_plane, void *const *d_bands);
CFB_API cfb_error cfb_level_inverse_device(cfb_context *ctx, const cfb_level_desc *desc, const void *const *d_bands, void *d_plane);
CFB_API cfb_error cfb_level_forward_host(cfb_context *ctx, const cfb_level_desc *desc, const void *plane, void *const *bands);
CFB_API cfb_error cfb_level_inverse_host(cfb_context *ctx, const cfb_level_desc *desc, const void *const *bands, void *plane);

/* ---- two-frame GOP as one call (CFHD_ENCODING_FLAGS_YUV_2FRAME_GOP; packed 8-bit 4:2:2) ------------
 * The FIELDPLUS pyramid of Codec/encoder.c:8431 FinishFieldPlusTransformQuant: wavelet 0 / 1 = level 1 of frame A / B
 * (spatial, or the field transform when the codec is interlaced), 2 = temporal (band 0 low, band 1 high),
 * 3 = level(temporal high), 4 = level(temporal low), 5 = level(LL of 4).  The coded region holds the 17 subbands the
 * entropy coder walks (quantize.c:3480): per channel wavelet 5 (LL, LH, HL, HH), 4 (LH, HL, HH), 3 (LL, LH, HL, HH),
 * 1 (LH, HL, HH), 0 (LH, HL, HH); LL of wavelets 0, 1, 4 and the temporal bands live in device scratch.
 * prescale[k] / divisor[c][k][b] are transform->prescale[k] and wavelet[k]->quant[b] of the reference
 * (cfb_gop2_quant_for_quality restates its schedule).  The codec must have been created with max_batch >= 2 and a width
 * that is a multiple of 64.  decoder side: Codec/decoder.c:13052-13170 + the level-1 inverse of both frames. */
enum { CFB_GOP2_WAVELETS = 6 };
typedef struct cfb_gop2_layout {
    int32_t num_channels;
    int32_t reserved;
    int64_t coded_bytes;
    int64_t total_bytes;
    cfb_band_layout band[CFB_MAX_CHANNELS][CFB_GOP2_WAVELETS][CFB_NUM_BANDS];
} cfb_gop2_layout;
typedef struct cfb_gop2_quant {
    int32_t midpoint_prequant;
    int32_t prescale[CFB_GOP2_WAVELETS];
    int32_t reserved;
    int32_t divisor[CFB_MAX_CHANNELS][CFB_GOP2_WAVELETS][CFB_NUM_BANDS];
} cfb_gop2_quant;
CFB_API cfb_error cfb_gop2_layout_compute(const cfb_frame_desc *desc, cfb_gop2_layout *out);
/* the reference's schedule for this transform type (quantize.c:3480-3640, wavelet.c:7135-7180), host only */
CFB_API cfb_error cfb_gop2_quant_for_quality(const cfb_frame_desc *desc, int quality, int interlaced, cfb_gop2_quant *out);
CFB_API cfb_error cfb_gop2_forward_host(cfb_codec *codec, const void *frame_a, const void *frame_b, int frame_pitch,
                                        const cfb_gop2_quant *quant, void *coded);
CFB_API cfb_error cfb_gop2_inverse_host(cfb_codec *codec, const void *coded, const cfb_gop2_quant *quant, int out_format,
                                        void *frame_a, void *frame_b, int frame_pitch);

/* ---- sparse transfer format of the coded region (lossless; SURVEY 8f rank 1) ---- */
/* Layout of a sparse buffer ('CFS2', cineform-sdk_b200/csrc/cfb_sparse_format.h):
 *   header 32 B {u32 'CFS2', u32 nwords, u32 total_bytes, u32 nblocks, 0...}; table nblocks x {u32 chunk offset, u32 groups,
 *   u32 values, u32 escapes}; one 16-byte aligned chunk per block of 8192 int16 words of the coded region [0, coded_bytes)
 *   (empty when the block is all zero): 32-byte bitmap of the block's non-empty 32-word groups, one 32-bit mask per
 *   non-empty group, one byte per non-zero word (-128 = escape), one int16 per escape.  Zero runs (incl. the pitch gap
 *   the reference's run-length coder walks, encoder.c:5653) are implicit in the bitmaps. */
CFB_API size_t cfb_sparse_max_bytes(const cfb_layout *layout);          /* worst case (no zero at all); every buffer handed to a
                                                                         * cfb_sparse_* / cfb_*_sparse call must be this large: readers bound a
                                                                         * damaged header's size field by it */
CFB_API size_t cfb_sparse_bytes(const void *sparse);                    /* actual size, from the header */
/* forward + GPU compaction; sparse_bytes[i] receives the size written to h_sparse[i] */
CFB_API cfb_error cfb_forward_host_sparse(cfb_codec *codec, int n, const void *const *h_frames, int frame_pitch,
                                          const cfb_quant *quant, void *const *h_sparse, size_t *sparse_bytes);
/* GPU expansion + inverse */
CFB_API cfb_error cfb_inverse_host_sparse(cfb_codec *codec, int n, const void *const *h_sparse, const cfb_quant *quant,
                                          int out_format, void *const *h_frames, int frame_pitch);
/* host-side format conversion (no transform arithmetic): sparse <-> dense coded region */
CFB_API cfb_error cfb_sparse_expand(const cfb_layout *layout, const void *sparse, void *dense_coded);
CFB_API cfb_error cfb_sparse_compact(const cfb_layout *layout, const void *dense_coded, void *sparse, size_t *bytes);
/* the same from one buffer per band, as an entropy decoder leaves them (Codec/decoder.c:19534-19808 writes
 * wavelet->band[b]): bands[(channel * CFB_NUM_LEVELS + level) * CFB_NUM_BANDS + band] with pitches[] bytes per row; bytes
 * between the band's width and its pitch are ignored; LL of levels 1, 2 may be null.  Host half of the decoder-side
 * hand-over: read the bands once, upload ~1/8 of them (cfb_inverse_host_sparse) */
CFB_API cfb_error cfb_sparse_compact_bands(const cfb_layout *layout, const void *const *bands, const int32_t *pitches,
                                           void *sparse, size_t *bytes);

/* ---- host run-length / VLC packing straight from the sparse format (SURVEY 8f rank 1, host side) ----
 * Replaces the walk of the reference's run-length coder over a DENSE band:
 *   Codec/encoder.c:5386-5700 EncodeQuantLongRuns (zero runs incl. the pitch gap :5653, greedy run-code split :5493-5545
 *   = Codec/vlc.c:366 PutZeroRun, value code with the +-(length/2 - 1) clamp :5553-5568 = vlc.c:188 PutVlcByte,
 *   32-bit big-endian bit buffer = bitstream.c:819 PutBits)
 * by a walk over the bitmap + values of the sparse format: zero runs are distances between set bits (the pitch gap is
 * part of the flat coded region and is zero), so the host never touches the 33 MB of dense int16 per 4K frame.  The
 * output is bit-for-bit what EncodeQuantLongRuns writes for the same band, incl. the state it leaves in the bit buffer.
 * The code tables belong to the host entropy coder (Codec/codebooks.c, out of scope): the caller passes them as plain
 * arrays (INTEGRATION.md shows how the shim fills them from encoder->codebook_runbook / encoder->valuebook). */
typedef struct cfb_vlc_codebook {
    int32_t run_length;             /* entries in run_* (RLCBOOK::length); entry i is used for runs >= i, i < length - 1 */
    int32_t value_length;           /* VALUE_TABLE_LENGTH: index v for 0 <= v < n/2, n + v for -n/2 < v < 0 */
    const uint32_t *run_bits;       /* code word, right justified */
    const uint8_t *run_size;        /* code size in bits (1..31) */
    const uint32_t *run_count;      /* zeros covered by the entry (>= 1) */
    const uint32_t *value_bits;
    const uint8_t *value_size;
} cfb_vlc_codebook;

typedef struct cfb_bitwriter {      /* the BITSTREAM fields the coder reads and leaves behind (Codec/bitstream.h) */
    uint8_t *cur;                   /* lpCurrentWord: the next 32-bit word is stored here, big-endian */
    uint8_t *end;                   /* first byte the writer may not touch */
    uint32_t buffer;                /* wBuffer: the low (32 - bits_free) bits are pending */
    int32_t bits_free;              /* nBitsFree: 32 = empty, 0 = a whole word pending */
    int64_t bytes;                  /* nWordsUsed */
} cfb_bitwriter;

/* band (channel, level 0..2 = wavelet level 1..3, band 0..3 = LL, LH, HL, HH) -> run-length / value codes appended to bw.
 * CFB_ERROR_INVALID_ARGUMENT for a band that is not in the coded region (LL of levels 1, 2), CFB_ERROR_BADFORMAT for a
 * damaged sparse buffer, CFB_ERROR_OUTOFMEMORY when bw->end would be passed (bw is then unusable). */
CFB_API cfb_error cfb_sparse_vlc_band(const cfb_layout *layout, const void *sparse, int channel, int level, int band,
                                      const cfb_vlc_codebook *book, cfb_bitwriter *bw);
/* number of non-zero coefficients of a band (what the walk above will emit as value codes) */
CFB_API cfb_error cfb_sparse_band_nonzeros(const cfb_layout *layout, const void *sparse, int channel, int level, int band,
                                           uint32_t *count);
/* one band of a sparse buffer -> dense int16 rows (pitch_bytes per row); the lowpass band LL3 is entropy coded by a
 * different routine that wants it dense (encoder.c:4251 EncodeLowPassBand) */
CFB_API cfb_error cfb_sparse_expand_band(const cfb_layout *layout, const void *sparse, int channel, int level, int band,
                                         int16_t *out, int pitch_bytes);
/* the same coder over a dense band (what the reference does); for A/B timing and for bands that never went sparse */
CFB_API cfb_error cfb_dense_vlc_band(const int16_t *band, int width, int height, int pitch_bytes,
                                     const cfb_vlc_codebook *book, cfb_bitwriter *bw);

/* ---- decoder side of the same row: entropy-decoded tokens -> sparse format (host) ----------------------------------
 * A decoder that produces (zero run, value) tokens -- which is what the reference's FSM decoder does internally before it
 * scatters them into a dense band (Codec/decoder.c:19534 DecodeBandFSM16sNoGap) -- can write the 'CFS2' buffer directly and
 * upload ~1/10 of the bytes (cfb_inverse_host_sparse).  The writer takes the bands in the order of the coded region
 * (per channel: LL3, then LH, HL, HH of levels 3, 2, 1); inside a band, runs count the pitch gap exactly as the
 * encoder's runs do (encoder.c:5653), so a token stream decoded from the reference's bit stream maps one to one. */
typedef struct cfb_sparse_writer cfb_sparse_writer;
CFB_API cfb_error cfb_sparse_writer_create(const cfb_layout *layout, cfb_sparse_writer **out);
CFB_API void cfb_sparse_writer_destroy(cfb_sparse_writer *w);
CFB_API cfb_error cfb_sparse_writer_begin(cfb_sparse_writer *w, void *sparse, size_t capacity);    /* capacity >= cfb_sparse_max_bytes */
CFB_API cfb_error cfb_sparse_writer_band(cfb_sparse_writer *w, int channel, int level, int band);  /* next band, coded order */
CFB_API cfb_error cfb_sparse_writer_run(cfb_sparse_writer *w, uint32_t zeros);
CFB_API cfb_error cfb_sparse_writer_value(cfb_sparse_writer *w, int value);
/* a band that arrives dense (the lowpass band LL3 is stored as plain 16-bit values, decoder.c DecodeLowPassBand) */
CFB_API cfb_error cfb_sparse_writer_dense_band(cfb_sparse_writer *w, int channel, int level, int band, const int16_t *rows, int pitch_bytes);
CFB_API cfb_error cfb_sparse_writer_end(cfb_sparse_writer *w, size_t *bytes);

/* A table-driven parser of the band bit stream for such a decoder.  The code set is the host entropy coder's (out of
 * scope): the caller lists every code word once -- kind 0 = coefficient with the (already decompanded, signed) value arg,
 * kind 1 = run of arg zeros, kind 2 = end of band.  Decoded coefficients are multiplied by `quant` and wrapped to int16,
 * as the reference's FSM tables are (decoder.c:20551 DeQuantFSM).  `consumed` receives the bytes read up to and including
 * the byte that holds the last bit of the end-of-band code. */
typedef struct cfb_vlc_decodebook {
    int32_t count;
    const uint32_t *bits;           /* code word, right justified */
    const uint8_t *size;            /* 1..31 bits */
    const uint8_t *kind;            /* 0 value, 1 zero run, 2 end of band */
    const int32_t *arg;
} cfb_vlc_decodebook;
typedef struct cfb_vlc_decoder cfb_vlc_decoder;
CFB_API cfb_error cfb_vlc_decoder_create(const cfb_vlc_decodebook *book, cfb_vlc_decoder **out);   /* fails if the set is not prefix free */
CFB_API void cfb_vlc_decoder_destroy(cfb_vlc_decoder *d);
CFB_API cfb_error cfb_vlc_decode_band(const cfb_vlc_decoder *d, cfb_sparse_writer *w, int channel, int level, int band,
                                      const uint8_t *stream, size_t stream_bytes, int quant, size_t *consumed);

/* ---- statistics record -------------------------------------------------------- */
typedef struct cfb_stats {
    uint64_t kernel_launches;   /* kernels launched by this library on this context */
    uint64_t frames_forward;
    uint64_t frames_inverse;
    uint64_t h2d_bytes;
    uint64_t d2h_bytes;
} cfb_stats;

/* ---- pinned host memory ------------------------------------------------------ */
/* Page-locked host buffers (cudaHostAlloc, portable) so that the pool's copies run asynchronously at
 * full PCIe rate.  Pageable buffers are accepted everywhere but serialise the copies. */
CFB_API cfb_error cfb_host_alloc(size_t bytes, void **out);
CFB_API void cfb_host_free(void *p);

/* ---- asynchronous, in-order, multi-GPU frame pool ---------------------------- */
/* GPU re-hosting of the reference's CEncoderPool (EncoderSDK/EncoderPool.cpp:239, EncoderQueue.h:311-352):
 *   - jobs are independent frames; job i goes to device devices[i % ndevices] (EncoderPool.cpp:284 round-robin);
 *   - every device runs `slots` worker slots (own stream + staging), each taking up to `batch` queued jobs per
 *     launch, so H2D copies, kernels and D2H copies of different slots overlap;
 *   - submit blocks while `queue_length` jobs are outstanding (AddEncoderJob, EncoderQueue.h:311);
 *   - results are delivered strictly in submission order (WaitForFinishedJob pops front(), EncoderQueue.h:331);
 *   - host buffers are BORROWED until the job is returned by cfb_pool_wait/cfb_pool_test (EncoderQueue.h:159).
 * A failed job is returned in order with its error; the pool keeps running. */
CFB_API cfb_error cfb_pool_create(const int *devices, int ndevices, const cfb_frame_desc *desc,
                                  int slots, int batch, int queue_length, cfb_pool **out);
/* progressive / interlaced mode (cfb_codec_set_interlaced) of every job submitted afterwards (call with the pool idle) */
CFB_API cfb_error cfb_pool_set_interlaced(cfb_pool *pool, int interlaced);
/* decode resolution of every inverse job submitted afterwards (call with the pool idle) */
CFB_API cfb_error cfb_pool_set_decode_resolution(cfb_pool *pool, int resolution);
CFB_API void cfb_pool_destroy(cfb_pool *pool);
/* forward: h_frame (frame_pitch bytes per row) -> h_coded (cfb_layout.coded_bytes) */
CFB_API cfb_error cfb_pool_submit_forward(cfb_pool *pool, uint32_t frame_number, const void *h_frame, int frame_pitch,
                                          const cfb_quant *quant, void *h_coded);
/* inverse: h_coded -> h_frame in out_format */
CFB_API cfb_error cfb_pool_submit_inverse(cfb_pool *pool, uint32_t frame_number, const void *h_coded,
                                          const cfb_quant *quant, int out_format, void *h_frame, int frame_pitch);
/* same, with the coded region in the sparse transfer format (h_sparse: cfb_sparse_max_bytes) */
CFB_API cfb_error cfb_pool_submit_forward_sparse(cfb_pool *pool, uint32_t frame_number, const void *h_frame, int frame_pitch,
                                                 const cfb_quant *quant, void *h_sparse);
CFB_API cfb_error cfb_pool_submit_inverse_sparse(cfb_pool *pool, uint32_t frame_number, const void *h_sparse,
                                                 const cfb_quant *quant, int out_format, void *h_frame, int frame_pitch);
/* oldest job: wait blocks until it has finished; test returns CFB_ERROR_NOT_FINISHED if it has not
 * (CFHD_ERROR_NOT_FINISHED = 13, EncoderPool.cpp:360).  *job_error receives the job's own result. */
CFB_API cfb_error cfb_pool_wait(cfb_pool *pool, uint32_t *frame_number, cfb_error *job_error);
CFB_API cfb_error cfb_pool_test(cfb_pool *pool, uint32_t *frame_number, cfb_error *job_error);
CFB_API cfb_error cfb_pool_stats(cfb_pool *pool, cfb_stats *out);     /* summed over all devices */

/* ---- statistics ------------------------------------------------------------ */

CFB_API cfb_error cfb_context_stats(cfb_context *ctx, cfb_stats *out);

#ifdef __cplusplus
}
#endif
#endif /* CFHD_B200_H */
