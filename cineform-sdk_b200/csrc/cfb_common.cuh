// cfb_common.cuh -- shared device/host definitions for the sm_100a wavelet kernels.
//
// Arithmetic convention ("fast path"): every kernel computes the reference's 2-6
// lifting in exact 32-bit integer arithmetic.  The reference (SSE2) computes the
// same expressions with saturating 16-bit chains in its vector loops and int32 +
// clamp in its scalar tails; the two agree with exact arithmetic whenever no
// intermediate leaves int16, which holds for every coefficient produced from
// sources within their declared precision (10-bit 4:2:2, 12-bit RGB/Bayer) except
// the few positions handled explicitly (6-tap border filters are clamped exactly
// as the reference clamps them).  See DESIGN.md "Overflow semantics".
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cfb {

constexpr int kMaxBatch = 16;     // == CFB_MAX_BATCH
constexpr int kMaxChannels = 4;
constexpr int kStripIn = 256;     // input samples per warp-row (8 per lane)
constexpr int kStripOut = 128;    // output coefficients per warp-row per band

// q = (x*m + (x < 0 ? cneg : cpos)) >> 16  ==  sign(x) * (((|x| + mid) * m) >> 16)
// with m = 65536/divisor, cpos = mid*m, cneg = 65535 - mid*m   (Codec/quantize.c:1395-1516)
struct QuantParam {
    int m;
    int cpos;
    int cneg;
    int pad;
};

struct PlaneGeom {
    int width;          // input samples per row of this channel
    int height;         // input rows
    int in_pitch;       // bytes
    int out_pitch;      // bytes
    long long in_off;   // byte offset of the plane from the frame's input base
    long long band_off[4];  // byte offsets of LL,LH,HL,HH from the frame's output base
    QuantParam q[4];
    int quant_ll;       // != 0: LL is quantised with q[0] (plain variant with divisor > 1)
    int pad;
};

struct FwdParams {
    int nchan;
    int nframes;
    int th;             // output rows per warp
    int shift;          // 4:2:2 only: precision - 8
    int uyvy;           // 4:2:2 only: 1 = UYVY byte order
    int pad;
    PlaneGeom ch[kMaxChannels];
    const unsigned char *in_base[kMaxBatch];
    unsigned char *out_base[kMaxBatch];
    const unsigned short *lut;      // Bayer only: encode curve, 1 << 14 entries (frame.c:5208), null = samples >> shift
};

constexpr int kInvStrip = 120;    // band columns written per warp-row by the inverse kernels (30 lanes x 4)

// output of the final 4:2:2 inverse level (k_inv_422)
constexpr int kInv422Out8 = 0;    // packed 8-bit YUYV / UYVY
constexpr int kInv422OutYU64 = 1; // packed 16-bit Y0 C1 Y1 C3
constexpr int kInv422OutV210 = 2; // packed 10-bit V210, 6 pixels in 4 words

struct InvGeom {
    int width;          // band width (coefficients)
    int height;         // band rows
    int pitch;          // band pitch in bytes
    int out_pitch;      // bytes
    long long band_off[4];
    long long out_off;
    int dq[4];          // dequantisation factors (divisors); LL normally 1
};

struct InvParams {
    int nchan;
    int nframes;
    int th;             // band rows per warp
    int shift;          // 4:2:2 output: precision - 8
    int uyvy;
    int pad;
    InvGeom ch[kMaxChannels];
    const unsigned char *in_base[kMaxBatch];
    unsigned char *out_base[kMaxBatch];
    // 16-bit unsigned outputs (YU64, RG48): v = max(t >> 1, 0) << up_shift, limited to hi_simd in the columns the
    // reference's 8-column SSE2 loop produces and to 65535 from band column tail_col[c] on (scalar tail + right border:
    // InvertHorizontalStrip16s.c:16571 InvertHorizontalStrip16sToRow16u, `protection` clamp vs SATURATE_16U)
    int up_shift;       // 16 - precision
    int hi_simd;        // ((1 << precision) - 1) << up_shift
    int tail_col[kMaxChannels];
};

// interlaced (field) inverse: per (frame, channel, band row, strip) carry-in of the difference-coded HL band
struct FieldsAux {
    int *carry;         // [(frame * nchan + c) * maxh + row] * nstrips + strip
    int nstrips;        // strips of the luma band
    int maxh;           // band rows
    int pad;
};

// fire-and-forget prefetch into L2 (no destination register, no scoreboard): hides DRAM latency for rows that
// will be loaded a few iterations later
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }

__device__ __forceinline__ int clamp16(int v) { return max(-32768, min(32767, v)); }

__device__ __forceinline__ int quant1(int x, const QuantParam &q) {
    return x * q.m + (x < 0 ? q.cneg : q.cpos);     // result in the upper halfword
}

// pack the upper halfwords of two products / the lower halfwords of two values
__device__ __forceinline__ unsigned pack_hi(int a, int b) { return __byte_perm((unsigned)a, (unsigned)b, 0x7632); }
__device__ __forceinline__ unsigned pack_lo(int a, int b) { return __byte_perm((unsigned)a, (unsigned)b, 0x5410); }

__device__ __forceinline__ int lo16(unsigned w) { return (int)(short)(w & 0xffffu); }
__device__ __forceinline__ int hi16(unsigned w) { return ((int)w) >> 16; }

// dp4a with unsigned data bytes and signed coefficient bytes
__device__ __forceinline__ int dp4a_us(unsigned a, int b, int c) {
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

}  // namespace cfb
