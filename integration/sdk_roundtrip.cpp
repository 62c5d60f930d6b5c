// sdk_roundtrip.cpp -- our driver over the reference's PUBLIC C API only (Common/CFHDEncoder.h, CFHDDecoder.h).
// It is what Example/TestCFHD.cpp does in -D (sync quality loop) and -E (encoder pool) modes, but with the frame
// size, frame count and pool shape on the command line (TestCFHD hard-codes 1920x1080, TestCFHD.cpp:70-71).
// Linked twice by integration/Makefile: against libCFHDCodec.so (CUDA transform interposed) and against the plain
// reference, so the same program times both and their outputs can be compared.
//
//   sdk_roundtrip <width> <height> <frames> [pool_threads [queue [interlaced [format [decode]]]]]
// format: yuy2 (default), 2vuy, yu64, v210, rg48, rg30, r210, dpx0, ab10, ar10, byr4 -- the source formats whose level-1
// kernels libcfhd_b200 has; V210 and BYR4 frames (which Example/qbist.cpp cannot draw) are packed here from its YU64 /
// RG48 frames.
// decode: without it only yuy2 samples are decoded (to YUY2, with a dither-insensitive digest).  "same" decodes every
// sample into its own source format; a format name (e.g. b64a for rg48 samples) decodes into that one.  The digest of the
// decoded frames then covers every byte of every decoded frame (none of these outputs is dithered).
// prints one JSON line: sync encode/decode ms, sample bytes, FNV-1a digests of the encoded samples (sync loop and pool;
// from byte 512 on: the sample header carries the wall-clock time of the encode as metadata, bytes 155-180 at 640x96),
// luma PSNR (yuy2 decodes), digest of the decoded frames, pool fps.
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <vector>

#include "CFHDDecoder.h"
#include "CFHDEncoder.h"
#include "qbist.h"

static double now_s() { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; }

static void *aligned(size_t n) { void *p = nullptr; if (posix_memalign(&p, 64, n)) return nullptr; memset(p, 0, n); return p; }

int main(int argc, char **argv)
{
    const int w = argc > 1 ? atoi(argv[1]) : 1920, h = argc > 2 ? atoi(argv[2]) : 1080, nframes = argc > 3 ? atoi(argv[3]) : 5;
    const int pool_threads = argc > 4 ? atoi(argv[4]) : 0, queue = argc > 5 ? atoi(argv[5]) : 24;
    const bool interlaced = argc > 6 && atoi(argv[6]) != 0;     // CFHD_ENCODING_FLAGS_YUV_INTERLACED: field transform at level 1
    const char *fname = argc > 7 ? argv[7] : "yuy2";
    struct Fmt { const char *name; CFHD_PixelFormat fmt, draw; CFHD_EncodedFormat enc; int bytes_num, bytes_den; };
    static const Fmt table[] = {
        {"yuy2", CFHD_PIXEL_FORMAT_YUY2, CFHD_PIXEL_FORMAT_YUY2, CFHD_ENCODED_FORMAT_YUV_422, 2, 1},
        {"2vuy", CFHD_PIXEL_FORMAT_2VUY, CFHD_PIXEL_FORMAT_2VUY, CFHD_ENCODED_FORMAT_YUV_422, 2, 1},
        {"yu64", CFHD_PIXEL_FORMAT_YU64, CFHD_PIXEL_FORMAT_YU64, CFHD_ENCODED_FORMAT_YUV_422, 4, 1},
        {"v210", CFHD_PIXEL_FORMAT_V210, CFHD_PIXEL_FORMAT_YU64, CFHD_ENCODED_FORMAT_YUV_422, 8, 3},
        {"rg48", CFHD_PIXEL_FORMAT_RG48, CFHD_PIXEL_FORMAT_RG48, CFHD_ENCODED_FORMAT_RGB_444, 6, 1},
        {"rg30", CFHD_PIXEL_FORMAT_RG30, CFHD_PIXEL_FORMAT_RG30, CFHD_ENCODED_FORMAT_RGB_444, 4, 1},
        {"r210", CFHD_PIXEL_FORMAT_R210, CFHD_PIXEL_FORMAT_R210, CFHD_ENCODED_FORMAT_RGB_444, 4, 1},
        {"dpx0", CFHD_PIXEL_FORMAT_DPX0, CFHD_PIXEL_FORMAT_DPX0, CFHD_ENCODED_FORMAT_RGB_444, 4, 1},
        {"ab10", CFHD_PIXEL_FORMAT_AB10, CFHD_PIXEL_FORMAT_AB10, CFHD_ENCODED_FORMAT_RGB_444, 4, 1},
        {"ar10", CFHD_PIXEL_FORMAT_AR10, CFHD_PIXEL_FORMAT_AR10, CFHD_ENCODED_FORMAT_RGB_444, 4, 1},
        {"byr4", CFHD_PIXEL_FORMAT_BYR4, CFHD_PIXEL_FORMAT_RG48, CFHD_ENCODED_FORMAT_BAYER, 2, 1},
        {"b64a", CFHD_PIXEL_FORMAT_B64A, CFHD_PIXEL_FORMAT_B64A, CFHD_ENCODED_FORMAT_RGB_444, 8, 1},     // decode only
    };
    const Fmt *F = nullptr, *D = nullptr;
    for (const Fmt &t : table) if (!strcmp(t.name, fname)) F = &t;
    if (!F || F->fmt == CFHD_PIXEL_FORMAT_B64A) { fprintf(stderr, "unknown source format %s\n", fname); return 1; }
    const char *dname = argc > 8 ? argv[8] : nullptr;
    if (dname) {
        for (const Fmt &t : table) if (!strcmp(t.name, strcmp(dname, "same") ? dname : fname)) D = &t;
        if (!D) { fprintf(stderr, "unknown decode format %s\n", dname); return 1; }
    }
    const bool is_yuy2 = F->fmt == CFHD_PIXEL_FORMAT_YUY2;
    const bool is_v210 = F->fmt == CFHD_PIXEL_FORMAT_V210, is_byr4 = F->fmt == CFHD_PIXEL_FORMAT_BYR4;
    CFHD_EncodingFlags eflags = interlaced ? CFHD_ENCODING_FLAGS_YUV_INTERLACED : CFHD_ENCODING_FLAGS_NONE;
    if (is_byr4) eflags = CFHD_ENCODING_FLAGS_CURVE_APPLIED;        // the mosaic already carries its curve
    const int pitch = is_v210 ? ((w + 47) / 48) * 128 : w * F->bytes_num / F->bytes_den;
    // the decoded frame: the source layout unless a decode format was named (V210: the SDK's 128-byte row rounding)
    const CFHD_PixelFormat dfmt = D ? D->fmt : F->fmt;
    const int dpitch = !D ? pitch : D->fmt == CFHD_PIXEL_FORMAT_V210 ? ((w + 47) / 48) * 128 : w * D->bytes_num / D->bytes_den;
    const bool decode = is_yuy2 || D;
    const CFHD_PixelFormat fmt = F->fmt;
    const CFHD_EncodedFormat encfmt = F->enc;
    std::vector<uint8_t *> frames;
    GetRand(50);                    // TestCFHD.cpp:1149 QBIST_SEED
    initBaseTransform();
    uint8_t *gen = (uint8_t *)aligned((size_t)w * h * 8);
    const int distinct = nframes < 4 ? nframes : 4;
    for (int i = 0; i < distinct; i++) {
        const int draw_pitch = (F->draw == CFHD_PIXEL_FORMAT_RG48) ? w * 6 : (F->draw == CFHD_PIXEL_FORMAT_YU64 ? w * 4 : pitch);
        RunQBist(w, h, draw_pitch, F->draw, 0, gen);
        uint8_t *f = (uint8_t *)aligned((size_t)pitch * h);
        if (is_v210) {              // 6 pixels = 12 components of 10 bits in four little-endian words, three per word
            for (int y = 0; y < h; y++) {
                const uint16_t *src = (const uint16_t *)(gen + (size_t)y * draw_pitch);     // Y0 C Y1 C ...
                uint32_t *dst = (uint32_t *)(f + (size_t)y * pitch);
                for (int x = 0; x + 6 <= w; x += 6) {
                    const uint16_t *q = src + 2 * x;
                    uint32_t c[12];
                    // component order of V210: Cb Y Cr Y ...; YU64 holds Y first, so swap inside each pair
                    for (int k = 0; k < 6; k++) { c[2 * k] = q[2 * k + 1] >> 6; c[2 * k + 1] = q[2 * k] >> 6; }
                    for (int k = 0; k < 4; k++) dst[x / 6 * 4 + k] = c[3 * k] | (c[3 * k + 1] << 10) | (c[3 * k + 2] << 20);
                }
            }
        } else if (is_byr4) {       // RGGB mosaic of the RG48 picture, 16 bits per sample
            for (int y = 0; y < h; y++) {
                const uint16_t *src = (const uint16_t *)(gen + (size_t)y * draw_pitch);
                uint16_t *dst = (uint16_t *)(f + (size_t)y * pitch);
                for (int x = 0; x < w; x++) dst[x] = src[3 * x + ((y & 1) ? ((x & 1) ? 2 : 1) : ((x & 1) ? 1 : 0))];
            }
        } else
            memcpy(f, gen, (size_t)pitch * h);
        if (interlaced && is_yuy2)  // make the two fields differ: shift the odd field by 8 pixels
            for (int y = 1; y < h; y += 2) memmove(f + (size_t)y * pitch + 16, gen + (size_t)y * pitch, (size_t)pitch - 16);
        frames.push_back(f);
    }
    CFHD_EncoderRef enc = nullptr;
    CFHD_DecoderRef dec = nullptr;
    CFHD_Error e = CFHD_OpenEncoder(&enc, nullptr);
    if (!e) e = CFHD_PrepareToEncode(enc, w, h, fmt, encfmt, eflags, CFHD_ENCODING_QUALITY_FILMSCAN1);
    if (e) { fprintf(stderr, "encoder setup failed: %d\n", (int)e); return 1; }
    e = CFHD_OpenDecoder(&dec, nullptr);
    if (e) { fprintf(stderr, "decoder open failed: %d\n", (int)e); return 1; }
    // 16 guard rows behind the decoded frame: a decoder that writes the ENCODED height (rounded up to a multiple of 8,
    // e.g. 488 rows for a 720x486 source) instead of the display height would trample them
    const size_t guard_bytes = (size_t)dpitch * 16;
    uint8_t *out = (uint8_t *)aligned((size_t)dpitch * h + guard_bytes);
    memset(out + (size_t)dpitch * h, 0xA5, guard_bytes);
    int decoded = 0;
    double enc_s = 0, dec_s = 0, mse_sum = 0;
    size_t bytes = 0;
    uint64_t hash = 1469598103934665603ull, sample_hash = 1469598103934665603ull, pool_hash = 1469598103934665603ull;
    bool prepared = false;
    for (int i = -1; i < nframes; i++) {          // i == -1: untimed warm-up (lazy allocations, CUDA context)
        uint8_t *f = frames[(i + distinct) % distinct];
        double t0 = now_s();
        e = CFHD_EncodeSample(enc, f, pitch);
        if (i >= 0) enc_s += now_s() - t0;
        if (e) { fprintf(stderr, "CFHD_EncodeSample failed: %d\n", (int)e); return 2; }
        void *sample = nullptr; size_t size = 0;
        CFHD_GetSampleData(enc, &sample, &size);
        if (i == 0 && getenv("CFHD_DUMP_SAMPLE")) {      // development aid: the first timed sample, for byte-level comparison of two builds
            FILE *fp = fopen(getenv("CFHD_DUMP_SAMPLE"), "wb");
            if (fp) { fwrite(sample, 1, size, fp); fclose(fp); }
        }
        if (i >= 0) {
            bytes += size;
            for (size_t k = 512; k < size; k++) { sample_hash ^= ((const uint8_t *)sample)[k]; sample_hash *= 1099511628211ull; }
        }
        if (!decode) continue;      // without a decode format the other sources are encode-only here
        if (!prepared) {
            int aw, ah; CFHD_PixelFormat af;
            e = CFHD_PrepareToDecode(dec, w, h, dfmt, CFHD_DECODED_RESOLUTION_FULL, CFHD_DECODING_FLAGS_NONE, sample, size, &aw, &ah, &af);
            if (e) { fprintf(stderr, "CFHD_PrepareToDecode failed: %d\n", (int)e); return 3; }
            if (D && af != dfmt) { fprintf(stderr, "CFHD_PrepareToDecode chose another output format\n"); return 3; }
            prepared = true;
        }
        t0 = now_s();
        e = CFHD_DecodeSample(dec, sample, size, out, dpitch);
        if (i >= 0) dec_s += now_s() - t0;
        if (e) { fprintf(stderr, "CFHD_DecodeSample failed: %d\n", (int)e); return 4; }
        if (i < 0) continue;
        decoded++;
        if (D) {                    // exact digest of the whole decoded frame
            for (size_t k = 0; k < (size_t)dpitch * h; k++) { hash ^= out[k]; hash *= 1099511628211ull; }
            continue;
        }
        double mse = 0;
        for (size_t k = 0; k < (size_t)pitch * h; k += 2) { const double d = (double)out[k] - (double)f[k]; mse += d * d; }
        mse_sum += mse / ((double)w * h);
        for (size_t k = 0; k < (size_t)pitch * h; k += 97) { hash ^= (uint64_t)(out[k] >> 1); hash *= 1099511628211ull; }     // dither-insensitive digest
    }
    bool guard_ok = true;
    for (size_t k = 0; k < guard_bytes; k++) guard_ok = guard_ok && out[(size_t)dpitch * h + k] == 0xA5;
    const double psnr = 10.0 * log10(255.0 * 255.0 / (mse_sum / nframes + 1e-12));

    // asynchronous encoder pool, exactly the TestCFHD -E call sequence (TestCFHD.cpp:783-1047)
    double pool_fps = 0;
    if (pool_threads > 0) {
        CFHD_EncoderPoolRef pool = nullptr;
        e = CFHD_CreateEncoderPool(&pool, pool_threads, queue, nullptr);
        if (!e) e = CFHD_PrepareEncoderPool(pool, w, h, fmt, encfmt, eflags, CFHD_ENCODING_QUALITY_FILMSCAN1);
        if (!e) e = CFHD_StartEncoderPool(pool);
        if (e) { fprintf(stderr, "encoder pool setup failed: %d\n", (int)e); return 5; }
        const int warm = 2 * pool_threads, total = warm + nframes * 16;
        int submitted = 0, received = 0;
        double t0 = now_s();
        while (received < total) {
            if (received == warm && submitted == warm) t0 = now_s();
            while (submitted < (received < warm ? warm : total) && submitted - received < queue) {
                e = CFHD_EncodeAsyncSample(pool, submitted, frames[submitted % distinct], pitch, nullptr);
                if (e) { fprintf(stderr, "CFHD_EncodeAsyncSample failed: %d\n", (int)e); return 6; }
                submitted++;
            }
            uint32_t frameNumber = 0; CFHD_SampleBufferRef sb = nullptr;
            e = CFHD_WaitForSample(pool, &frameNumber, &sb);
            if (e) { fprintf(stderr, "CFHD_WaitForSample failed: %d\n", (int)e); return 7; }
            if ((int)frameNumber != received) { fprintf(stderr, "out-of-order delivery %u != %d\n", frameNumber, received); return 8; }
            if (received < 8) {         // entropy-coded bytes of the first pool samples (all distinct source frames)
                void *data = nullptr; size_t size = 0;
                if (CFHD_GetEncodedSample(sb, &data, &size) == CFHD_ERROR_OKAY)
                    for (size_t k = 512; k < size; k++) { pool_hash ^= ((const uint8_t *)data)[k]; pool_hash *= 1099511628211ull; }
            }
            CFHD_ReleaseSampleBuffer(pool, sb);
            received++;
        }
        pool_fps = (total - warm) / (now_s() - t0);
        CFHD_StopEncoderPool(pool);
        CFHD_ReleaseEncoderPool(pool);
    }
    printf("{\"width\": %d, \"height\": %d, \"frames\": %d, \"enc_ms\": %.3f, \"dec_ms\": %.3f, \"sample_bytes\": %zu, "
           "\"sample_digest\": \"%016llx\", \"pool_sample_digest\": \"%016llx\", "
           "\"luma_psnr_db\": %.3f, \"decoded_digest\": \"%016llx\", \"pool_threads\": %d, \"pool_fps\": %.1f, \"interlaced\": %d, \"guard_ok\": %d, \"format\": \"%s\"",
           w, h, nframes, 1e3 * enc_s / nframes, 1e3 * dec_s / nframes, bytes / nframes, (unsigned long long)sample_hash, (unsigned long long)pool_hash,
           psnr, (unsigned long long)hash,
           pool_threads, pool_fps, interlaced ? 1 : 0, guard_ok ? 1 : 0, fname);
    if (D) printf(", \"decode_format\": \"%s\", \"decoded_frames\": %d", D->name, decoded);
    printf("}\n");
    CFHD_CloseEncoder(enc);
    CFHD_CloseDecoder(dec);
    return 0;
}
