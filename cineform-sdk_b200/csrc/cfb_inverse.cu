// cfb_inverse.cu -- inverse 2-6 wavelet level with fused dequantisation, sm_100a.
//
// Replaces (reference):
//   Codec/spatial.c:21877 InvertSpatialQuant16s + Codec/InvertHorizontalStrip16s.c:459   -> k_inv_plane<0>
//   Codec/spatial.c:22414 InvertSpatialQuantDescale16s + InvertHorizontalStrip16s.c:1700 -> k_inv_plane<2>
//   Codec/spatial.c:31341/:31511/:31975 InvertSpatial{Top,Middle,Bottom}Row16sToOutput +
//   Codec/InvertHorizontalStrip16s.c:3770/:5025 InvertHorizontalStrip16sToYUYV/ToUYVY   -> k_inv_422
//   Codec/decoder.c:20551 DeQuantFSM (coefficient * quant)                               -> fused into the loads
//
// Same structure as the forward kernels: no shared memory, one warp per strip, registers only.
// A lane owns 4 band columns; per band row it loads 8 bytes from each of the four bands, keeps a
// three-row window of the two vertically-lowpass bands (LL, LH) in registers, produces the even/odd
// intermediate rows, exchanges one value with each neighbour lane by shuffle for the horizontal
// stage and writes 8 output samples per row with one 128-bit store.  Lanes 0 and 31 of a warp are
// halo lanes (their columns belong to the neighbouring strips), so a strip covers 120 band columns.
#include "cfb_common.cuh"
#include "cfb_tma.cuh"

#include <cstdlib>
#include <cstring>
#include <type_traits>

namespace cfb {

constexpr unsigned kFullMask = 0xffffffffu;

// raw (still packed, still quantised) coefficients of NC columns of one band row
template <int NC> struct RawCols;
template <> struct RawCols<4> { uint2 w; };
template <> struct RawCols<2> { unsigned w; };

template <int NC>
__device__ __forceinline__ void load_raw(const unsigned char *in, long long band_off, unsigned off, bool active, RawCols<NC> &r);
template <>
__device__ __forceinline__ void load_raw<4>(const unsigned char *in, long long band_off, unsigned off, bool active, RawCols<4> &r) {
    r.w = active ? __ldg(reinterpret_cast<const uint2 *>(in + band_off + off)) : make_uint2(0, 0);
}
template <>
__device__ __forceinline__ void load_raw<2>(const unsigned char *in, long long band_off, unsigned off, bool active, RawCols<2> &r) {
    r.w = active ? __ldg(reinterpret_cast<const unsigned *>(in + band_off + off)) : 0u;
}

// dp2a with signed 16-bit halves (a) and unsigned byte coefficients (b): lo16(a)*b0 + hi16(a)*b1 (+ c)
__device__ __forceinline__ int dp2a_lo_su(unsigned a, unsigned b, int c) {
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// unpack + dequantise one packed pair.  SMALLDQ: divisor <= 255 -> one dp2a per coefficient.
template <bool SMALLDQ>
__device__ __forceinline__ void deq_pair(unsigned w, int dq, int &lo, int &hi) {
    if (SMALLDQ) {
        lo = dp2a_lo_su(w, (unsigned)dq, 0);
        hi = dp2a_lo_su(w, (unsigned)dq << 8, 0);
    } else {
        lo = lo16(w) * dq;
        hi = hi16(w) * dq;
    }
}
__device__ __forceinline__ void unpack_pair(unsigned w, int &lo, int &hi) { lo = lo16(w); hi = hi16(w); }

template <bool SMALLDQ, int NC>
struct Expand;
template <bool SMALLDQ>
struct Expand<SMALLDQ, 4> {
    static __device__ __forceinline__ void ll(const RawCols<4> &r, int *v) { unpack_pair(r.w.x, v[0], v[1]); unpack_pair(r.w.y, v[2], v[3]); }
    static __device__ __forceinline__ void hp(const RawCols<4> &r, int dq, int *v) {
        deq_pair<SMALLDQ>(r.w.x, dq, v[0], v[1]); deq_pair<SMALLDQ>(r.w.y, dq, v[2], v[3]);
    }
};
template <bool SMALLDQ>
struct Expand<SMALLDQ, 2> {
    static __device__ __forceinline__ void ll(const RawCols<2> &r, int *v) { unpack_pair(r.w, v[0], v[1]); }
    static __device__ __forceinline__ void hp(const RawCols<2> &r, int dq, int *v) { deq_pair<SMALLDQ>(r.w, dq, v[0], v[1]); }
};

// legacy helper used only on the border rows
template <int NC>
__device__ __forceinline__ void load_cols(const unsigned char *band, int pitch, int row, int colbyte, int dq, bool active, int *v)
{
    if (NC == 4) {
        uint2 w = active ? __ldg(reinterpret_cast<const uint2 *>(band + (long long)row * pitch + colbyte)) : make_uint2(0, 0);
        v[0] = lo16(w.x) * dq; v[1] = hi16(w.x) * dq; v[2] = lo16(w.y) * dq; v[3] = hi16(w.y) * dq;
    } else {
        unsigned w = active ? __ldg(reinterpret_cast<const unsigned *>(band + (long long)row * pitch + colbyte)) : 0u;
        v[0] = lo16(w) * dq; v[1] = hi16(w) * dq;
    }
}

// vertical inverse for NC columns: rows (p, c, n) of the low band and row c of the high band
template <int NC>
__device__ __forceinline__ void vinv_mid(const int *p, const int *c, const int *n, const int *h, int *e, int *o)
{
#pragma unroll
    for (int i = 0; i < NC; i++) {
        e[i] = (((p[i] - n[i] + 4) >> 3) + c[i] + h[i]) >> 1;
        o[i] = (((n[i] - p[i] + 4) >> 3) + c[i] - h[i]) >> 1;
    }
}
// top border: a0,a1,a2 = rows 0,1,2 ; bottom border: call with a0,a1,a2 = rows H-1,H-2,H-3 and bottom=true
template <int NC>
__device__ __forceinline__ void vinv_border(const int *a0, const int *a1, const int *a2, const int *h, bool bottom, int *e, int *o)
{
#pragma unroll
    for (int i = 0; i < NC; i++) {
        const int x = (11 * a0[i] - 4 * a1[i] + a2[i] + 4) >> 3;
        const int y = (5 * a0[i] + 4 * a1[i] - a2[i] + 4) >> 3;
        e[i] = ((bottom ? y : x) + h[i]) >> 1;
        o[i] = ((bottom ? x : y) - h[i]) >> 1;
    }
}

// horizontal inverse for NC columns -> 2*NC samples t (BEFORE the final >>1 / <<1):
//   t[2i] = ((l[i-1] - l[i+1] + 4) >> 3) + l[i] + h[i],  t[2i+1] = ((l[i+1] - l[i-1] + 4) >> 3) + l[i] - h[i]
template <int NC>
__device__ __forceinline__ void hinv(const int *l, const int *h, bool has_border, bool left_border, bool right_border, int *t)
{
    const int lp = __shfl_up_sync(kFullMask, l[NC - 1], 1);
    const int ln = __shfl_down_sync(kFullMask, l[0], 1);
#pragma unroll
    for (int i = 0; i < NC; i++) {
        const int a = (i == 0) ? lp : l[i - 1];
        const int b = (i == NC - 1) ? ln : l[i + 1];
        t[2 * i] = ((a - b + 4) >> 3) + l[i] + h[i];
        t[2 * i + 1] = ((b - a + 4) >> 3) + l[i] - h[i];
    }
    if (has_border) {
    if (left_border) {
        const int l2 = (NC > 2) ? l[2] : ln;
        t[0] = ((11 * l[0] - 4 * l[1] + l2 + 4) >> 3) + h[0];
        t[1] = ((5 * l[0] + 4 * l[1] - l2 + 4) >> 3) - h[0];
    }
    if (right_border) {
        const int k = NC - 1;
        const int l2 = (NC > 2) ? l[k - 2] : lp;
        t[2 * k] = ((5 * l[k] + 4 * l[k - 1] - l2 + 4) >> 3) + h[k];
        t[2 * k + 1] = ((11 * l[k] - 4 * l[k - 1] + l2 + 4) >> 3) - h[k];
    }
    }
}

__device__ __forceinline__ unsigned pack_sat16(int lo, int hi) {
    unsigned d;
    asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(d) : "r"(hi), "r"(lo));
    return d;
}

// ----------------------------------------------------------------------------
// Lane-distributed L2 prefetch.  A future band row of one strip touches <= 3 cache lines per luma band and <= 2 per
// chroma band; instead of every lane prefetching its own 8 bytes of each of the 12 bands (12 address computations
// per warp and row), each lane owns ONE (channel, band, 128-byte line) and the whole set costs one prefetch
// instruction per row.  LL/LH are fetched 4 rows ahead (the vertical window reads row r+1), HL/HH 3 rows ahead.
struct LanePrefetch {
    const unsigned char *base;      // in + band offset + line start (row 0)
    int pitch;
    int ahead;
    bool valid;
    __device__ __forceinline__ void issue(int r, int y1, int H) const {
        if (valid && r + 3 < y1) prefetch_l2(base + (long long)min(r + ahead, H - 1) * pitch);
    }
};

// chan_of_lane < 0: lane idle.  bytes_per_col = 2 for a full-width band, 1 for the half-width chroma bands of 4:2:2
// (their columns are addressed as luma_column / 2).
__device__ __forceinline__ LanePrefetch make_prefetch(const InvGeom &g, const unsigned char *in, int strip, int band, int line,
                                                      int bytes_per_col, bool on)
{
    LanePrefetch pf;
    const int col = ((max(strip * kInvStrip - 4, 0) * bytes_per_col) & ~127) + line * 128;
    pf.valid = on && col < g.pitch;
    pf.base = in + g.band_off[band] + col;
    pf.pitch = g.pitch;
    pf.ahead = (band < 2) ? 4 : 3;
    return pf;
}

// ----------------------------------------------------------------------------
// Per-channel inverse engine: a three-row window of LL and LH (already expanded to int32) plus a
// one-iteration-ahead prefetch of the raw band rows.
template <int NC>
struct InvChan {
    int lp[NC], lc[NC], hp[NC], hc[NC];                 // LL / LH rows r-1, r
    RawCols<NC> nll, nlh, nhl, nhh;                     // prefetched: LL,LH row r+1 ; HL,HH row r
};

template <int NC, bool SMALLDQ>
__device__ __forceinline__ void inv_prologue(InvChan<NC> &s, const InvGeom &g, const unsigned char *in, int y0, int H,
                                             unsigned colbyte, bool active)
{
    RawCols<NC> a, b;
    const unsigned rp = (unsigned)max(y0 - 1, 0) * g.pitch + colbyte, rc = (unsigned)y0 * g.pitch + colbyte;
    load_raw<NC>(in, g.band_off[0], rp, active, a); Expand<SMALLDQ, NC>::ll(a, s.lp);
    load_raw<NC>(in, g.band_off[1], rp, active, b); Expand<SMALLDQ, NC>::hp(b, g.dq[1], s.hp);
    load_raw<NC>(in, g.band_off[0], rc, active, a); Expand<SMALLDQ, NC>::ll(a, s.lc);
    load_raw<NC>(in, g.band_off[1], rc, active, b); Expand<SMALLDQ, NC>::hp(b, g.dq[1], s.hc);
    const unsigned rn = (unsigned)min(y0 + 1, H - 1) * g.pitch + colbyte;
    load_raw<NC>(in, g.band_off[0], rn, active, s.nll);
    load_raw<NC>(in, g.band_off[1], rn, active, s.nlh);
    load_raw<NC>(in, g.band_off[2], rc, active, s.nhl);
    load_raw<NC>(in, g.band_off[3], rc, active, s.nhh);
}

// One band row r -> the 2*NC "t" values (before the final shift) of output rows 2r (te) and 2r+1 (to).
template <int NC, bool SMALLDQ>
__device__ __forceinline__ void inv_step(InvChan<NC> &s, const InvGeom &g, const unsigned char *in, int r, int y1, int H,
                                         unsigned colbyte, bool active, bool has_border, bool left_border, bool right_border,
                                         int *te, int *to)
{
    int ln[NC], hn[NC], vhl[NC], vhh[NC];
    Expand<SMALLDQ, NC>::ll(s.nll, ln);
    Expand<SMALLDQ, NC>::hp(s.nlh, g.dq[1], hn);
    Expand<SMALLDQ, NC>::hp(s.nhl, g.dq[2], vhl);
    Expand<SMALLDQ, NC>::hp(s.nhh, g.dq[3], vhh);
    if (r + 1 < y1) {       // prefetch the next iteration's rows
        const unsigned rn = (unsigned)min(r + 2, H - 1) * g.pitch + colbyte, rc = (unsigned)(r + 1) * g.pitch + colbyte;
        load_raw<NC>(in, g.band_off[0], rn, active, s.nll);
        load_raw<NC>(in, g.band_off[1], rn, active, s.nlh);
        load_raw<NC>(in, g.band_off[2], rc, active, s.nhl);
        load_raw<NC>(in, g.band_off[3], rc, active, s.nhh);
    }
    int el[NC], ol[NC], eh[NC], oh[NC];
    vinv_mid<NC>(s.lp, s.lc, ln, vhl, el, ol);
    vinv_mid<NC>(s.hp, s.hc, hn, vhh, eh, oh);
    hinv<NC>(el, eh, has_border, left_border, right_border, te);
    hinv<NC>(ol, oh, has_border, left_border, right_border, to);
#pragma unroll
    for (int i = 0; i < NC; i++) { s.lp[i] = s.lc[i]; s.lc[i] = ln[i]; s.hp[i] = s.hc[i]; s.hc[i] = hn[i]; }
}

// Border band rows (r = 0 or r = H-1), computed from scratch by the border warps
// (spatial.c:21980-22060 top, :22320-22400 bottom).
template <int NC>
__device__ __forceinline__ void inv_border_row(const InvGeom &g, const unsigned char *in, bool bottom, int H, unsigned colbyte,
                                               bool active, bool has_border, bool left_border, bool right_border,
                                               int *te, int *to)
{
    const int r0 = bottom ? H - 1 : 0, r1 = bottom ? H - 2 : 1, r2 = bottom ? H - 3 : 2;
    int a0[NC], a1[NC], a2[NC], b0[NC], b1[NC], b2[NC], vhl[NC], vhh[NC];
    load_cols<NC>(in + g.band_off[0], g.pitch, r0, colbyte, 1, active, a0);
    load_cols<NC>(in + g.band_off[0], g.pitch, r1, colbyte, 1, active, a1);
    load_cols<NC>(in + g.band_off[0], g.pitch, r2, colbyte, 1, active, a2);
    load_cols<NC>(in + g.band_off[1], g.pitch, r0, colbyte, g.dq[1], active, b0);
    load_cols<NC>(in + g.band_off[1], g.pitch, r1, colbyte, g.dq[1], active, b1);
    load_cols<NC>(in + g.band_off[1], g.pitch, r2, colbyte, g.dq[1], active, b2);
    load_cols<NC>(in + g.band_off[2], g.pitch, r0, colbyte, g.dq[2], active, vhl);
    load_cols<NC>(in + g.band_off[3], g.pitch, r0, colbyte, g.dq[3], active, vhh);
    int el[NC], ol[NC], eh[NC], oh[NC];
    vinv_border<NC>(a0, a1, a2, vhl, bottom, el, ol);
    vinv_border<NC>(b0, b1, b2, vhh, bottom, eh, oh);
    hinv<NC>(el, eh, has_border, left_border, right_border, te);
    hinv<NC>(ol, oh, has_border, left_border, right_border, to);
}

// ----------------------------------------------------------------------------
// generic level: 4 bands -> int16 plane (2W x 2H)
template <int DESCALE, bool SMALLDQ>
__global__ void __launch_bounds__(128) k_inv_plane(const __grid_constant__ InvParams p)
{
    const int lane = threadIdx.x;
    const int f = blockIdx.z / p.nchan, c = blockIdx.z - f * p.nchan;
    const InvGeom &g = p.ch[c];
    const int strip = blockIdx.x;
    if (strip * kInvStrip >= g.width) return;
    const int H = g.height;

    const int col0 = strip * kInvStrip - 4 + lane * 4;          // first band column of this lane
    const bool active = (col0 >= 0) && (col0 < g.width);
    // a lane whose 4 columns are not all inside the band (width % 4 != 0) still loads (its first column is its left
    // neighbour's right tap) but does not write: those 1-3 columns, the right border among them, are k_inv_plane_edge's
    const bool writer = active && lane >= 1 && lane <= 30 && (col0 + 4 <= g.width);
    const bool left_border = (col0 == 0);
    const bool right_border = (col0 + 4 == g.width);
    const bool has_border = (strip == 0) || ((strip + 1) * kInvStrip + 4 >= g.width);
    const unsigned colbyte = (unsigned)(col0 * 2);
    const unsigned char *in = p.in_base[f];
    unsigned char *out = p.out_base[f] + g.out_off + (long long)col0 * 4;

    auto emit = [&](int r, const int *te, const int *to) {
        uint4 a, b;
        if (DESCALE) {
            a = make_uint4(pack_sat16(te[0] << 1, te[1] << 1), pack_sat16(te[2] << 1, te[3] << 1),
                           pack_sat16(te[4] << 1, te[5] << 1), pack_sat16(te[6] << 1, te[7] << 1));
            b = make_uint4(pack_sat16(to[0] << 1, to[1] << 1), pack_sat16(to[2] << 1, to[3] << 1),
                           pack_sat16(to[4] << 1, to[5] << 1), pack_sat16(to[6] << 1, to[7] << 1));
        } else {
            a = make_uint4(pack_sat16(te[0] >> 1, te[1] >> 1), pack_sat16(te[2] >> 1, te[3] >> 1),
                           pack_sat16(te[4] >> 1, te[5] >> 1), pack_sat16(te[6] >> 1, te[7] >> 1));
            b = make_uint4(pack_sat16(to[0] >> 1, to[1] >> 1), pack_sat16(to[2] >> 1, to[3] >> 1),
                           pack_sat16(to[4] >> 1, to[5] >> 1), pack_sat16(to[6] >> 1, to[7] >> 1));
        }
        unsigned char *o = out + (long long)(2 * r) * g.out_pitch;
        *reinterpret_cast<uint4 *>(o) = a;
        *reinterpret_cast<uint4 *>(o + g.out_pitch) = b;
    };

    if (blockIdx.y == gridDim.y - 1) {          // border warps: band rows 0 and H-1
        if (threadIdx.y > 1) return;
        const bool bottom = (threadIdx.y == 1);
        int te[8], to[8];
        inv_border_row<4>(g, in, bottom, H, colbyte, active, has_border, left_border, right_border, te, to);
        if (writer) emit(bottom ? H - 1 : 0, te, to);
        return;
    }
    const int y0 = max((int)(blockIdx.y * blockDim.y + threadIdx.y) * p.th, 1);
    const int y1 = min((int)(blockIdx.y * blockDim.y + threadIdx.y + 1) * p.th, H - 1);
    if (y0 >= y1) return;

    const LanePrefetch pf = make_prefetch(g, in, strip, lane / 3, lane % 3, 2, lane < 12);
    InvChan<4> st;
    inv_prologue<4, SMALLDQ>(st, g, in, y0, H, colbyte, active);
    for (int r = y0; r < y1; r++) {
        pf.issue(r, y1, H);
        int te[8], to[8];
        inv_step<4, SMALLDQ>(st, g, in, r, y1, H, colbyte, active, has_border, left_border, right_border, te, to);
        if (writer) emit(r, te, to);
    }
}

// ----------------------------------------------------------------------------
// Ragged widths: band columns [4 * (width / 4), width) of an inverse level, one thread per band coefficient position
// (-> a 2x2 block of output samples), written as the formulas read (spatial.c:21980-22400 vertical,
// InvertHorizontalStrip16s.c:459-896 / :1700-2166 horizontal).
template <int DESCALE>
__global__ void __launch_bounds__(128) k_inv_plane_edge(const __grid_constant__ InvParams p)
{
    const int f = blockIdx.z / p.nchan, c = blockIdx.z - f * p.nchan;
    const InvGeom &g = p.ch[c];
    const int W = g.width, H = g.height;
    const int col = (W >> 2) * 4 + blockIdx.y;
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= W || r >= H) return;
    const unsigned char *in = p.in_base[f];
    auto coef = [&](int b, int row, int cc) {
        return (int)*reinterpret_cast<const short *>(in + g.band_off[b] + (long long)row * g.pitch + 2 * cc) * (b ? g.dq[b] : 1);
    };
    // vertical inverse of (low band lb, high band hb) at band column cc -> even / odd intermediate rows
    auto vinv = [&](int lb, int hb, int cc, int &e, int &o) {
        const int hv = coef(hb, r, cc);
        if (r == 0 || r == H - 1) {
            const bool bottom = (r != 0);
            const int a0 = coef(lb, bottom ? H - 1 : 0, cc), a1 = coef(lb, bottom ? H - 2 : 1, cc), a2 = coef(lb, bottom ? H - 3 : 2, cc);
            const int x = (11 * a0 - 4 * a1 + a2 + 4) >> 3, y = (5 * a0 + 4 * a1 - a2 + 4) >> 3;
            e = ((bottom ? y : x) + hv) >> 1;
            o = ((bottom ? x : y) - hv) >> 1;
        } else {
            const int pv = coef(lb, r - 1, cc), cv = coef(lb, r, cc), nv = coef(lb, r + 1, cc);
            e = (((pv - nv + 4) >> 3) + cv + hv) >> 1;
            o = (((nv - pv + 4) >> 3) + cv - hv) >> 1;
        }
    };
    // columns col-2 .. col+1 of the vertically inverted lowpass (LL/HL) and column col of the highpass (LH/HH)
    int le[4], lo[4], he, ho;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int cc = min(max(col - 2 + k, 0), W - 1);
        vinv(0, 2, cc, le[k], lo[k]);
    }
    vinv(1, 3, col, he, ho);
    auto hpair = [&](const int *l, int hv, int &t0, int &t1) {      // l[0..3] = columns col-2 .. col+1
        if (col == W - 1) {
            t0 = ((5 * l[2] + 4 * l[1] - l[0] + 4) >> 3) + hv;
            t1 = ((11 * l[2] - 4 * l[1] + l[0] + 4) >> 3) - hv;
        } else {
            t0 = ((l[1] - l[3] + 4) >> 3) + l[2] + hv;
            t1 = ((l[3] - l[1] + 4) >> 3) + l[2] - hv;
        }
    };
    int e0, e1, o0, o1;
    hpair(le, he, e0, e1);
    hpair(lo, ho, o0, o1);
    unsigned char *out = p.out_base[f] + g.out_off + (long long)(2 * r) * g.out_pitch + (long long)col * 4;
    if (DESCALE) {
        *reinterpret_cast<unsigned *>(out) = pack_sat16(e0 << 1, e1 << 1);
        *reinterpret_cast<unsigned *>(out + g.out_pitch) = pack_sat16(o0 << 1, o1 << 1);
    } else {
        *reinterpret_cast<unsigned *>(out) = pack_sat16(e0 >> 1, e1 >> 1);
        *reinterpret_cast<unsigned *>(out + g.out_pitch) = pack_sat16(o0 >> 1, o1 >> 1);
    }
}

// ----------------------------------------------------------------------------
// final level of a 4:2:2 frame: 12 bands -> packed 8-bit YUYV / UYVY.
// 8-bit reduction: the reference computes v = max(t, 0) >> 1 (10-bit) and out = sat_u8((v + d) >> 2) with
// d = rand() & 1 per position (InvertHorizontalStrip16s.c:3807-3892) - not reproducible.  We use the
// deterministic ordered dither d = (x ^ y) & 1, i.e. out = sat_u8((t + 2d) >> 3), which stays inside the
// reference's envelope {(v) >> 2, (v + 1) >> 2} at every pixel.
__device__ __forceinline__ unsigned pack_u8x4(int a, int b, int c, int d) {
    // bytes (LSB first): a, b, c, d, each saturated to [0,255].
    // cvt.pack.sat.u8.s32.b32 r, x, y, z  ->  r = (z << 16) | (sat(x) << 8) | sat(y)
    unsigned t, r;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(d), "r"(c), "r"(0));
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(b), "r"(a), "r"(t));
    return r;
}

// 16-bit unsigned output sample of the final level: see InvParams::up_shift (the reference's ...ToRow16u rule)
__device__ __forceinline__ unsigned row16u(int t, int up_shift, int hi) {
    return (unsigned)min(max(t >> 1, 0) << up_shift, hi);
}

// One band row r of the final 4:2:2 level -> output rows 2r and 2r + 1 of the lane's 8 luma samples (+ 4 + 4 chroma).
// `out` already points at the lane's first sample of row 0.  t values arrive BEFORE the filter's final >> 1.
template <bool OUT16>
__device__ __forceinline__ void emit_422(const InvParams &p, unsigned char *out, int col0, int r, const int *ye, const int *yo,
                                         const int *ue, const int *uo, const int *ve, const int *vo)
{
    const InvGeom &gy = p.ch[0];
    const int sh = p.shift + 1;     // final >>1 of the filter merged with the >> (precision-8) reduction
    unsigned char *o = out + (long long)(2 * r) * gy.out_pitch;
    if (OUT16) {
        const int us = p.up_shift;
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
            const int *yy = rr ? yo : ye, *uu = rr ? uo : ue, *vv = rr ? vo : ve;
            unsigned w[8];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                // luma band column col0 + k -> samples 2k, 2k + 1; chroma band column col0 / 2 + (k >> 1) -> sample k
                const int hy = (col0 + k >= p.tail_col[0]) ? 65535 : p.hi_simd;
                const int hc1 = ((col0 >> 1) + (k >> 1) >= p.tail_col[1]) ? 65535 : p.hi_simd;
                const int hc2 = ((col0 >> 1) + (k >> 1) >= p.tail_col[2]) ? 65535 : p.hi_simd;
                // pixel pair k: words (Y0, C1) (Y1, C3); C1 = channel 1 (the v arrays), C3 = channel 2 (the u arrays)
                w[2 * k] = row16u(yy[2 * k], us, hy) | (row16u(vv[k], us, hc1) << 16);
                w[2 * k + 1] = row16u(yy[2 * k + 1], us, hy) | (row16u(uu[k], us, hc2) << 16);
            }
            unsigned char *q = o + (rr ? gy.out_pitch : 0);
            *reinterpret_cast<uint4 *>(q) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4 *>(q + 16) = make_uint4(w[4], w[5], w[6], w[7]);
        }
    } else {
#pragma unroll
    for (int rr = 0; rr < 2; rr++) {
        const int *yy = rr ? yo : ye, *uu = rr ? uo : ue, *vv = rr ? vo : ve;
        // ordered dither d = (x ^ y) & 1 on the sample's own column index, scaled to the merged shift;
        // band row r -> output rows 2r (even) and 2r+1 (odd)
        const int d0 = (rr ? 1 : 0) << (sh - 2), d1 = (rr ? 0 : 1) << (sh - 2);
        unsigned w[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int ya = (yy[2 * k] + d0) >> sh, yb = (yy[2 * k + 1] + d1) >> sh;
            const int cu = (uu[k] + ((k & 1) ? d1 : d0)) >> sh, cv = (vv[k] + ((k & 1) ? d1 : d0)) >> sh;
            w[k] = p.uyvy ? pack_u8x4(cu, ya, cv, yb) : pack_u8x4(ya, cu, yb, cv);
        }
        *reinterpret_cast<uint4 *>(o + (rr ? gy.out_pitch : 0)) = make_uint4(w[0], w[1], w[2], w[3]);
    }
    }
}

// V210 output: component word of three 10-bit values at bits 0, 10, 20
__device__ __forceinline__ unsigned v210_word(unsigned a, unsigned b, unsigned c) { return a | (b << 10) | (c << 20); }

// One band row r of the final 4:2:2 level -> V210 rows 2r and 2r + 1 (decoder.c:26292 -> InvertHorizontalStrip16s.c:6490
// InvertHorizontalYUVStrip16sToYUVOutput: the YU64 row rule, then convert.c:13526 ConvertPlanarYUVToV210 at precision 16).
// A component is row16u >> 6 = min(max(t >> 1, 0), 1023): both of the 16-bit rule's limits (0xFFC0, 65535) become 1023.
// Group of 6 pixels = 4 words: Cb0 Y0 Cr0 | Y1 Cb2 Y2 | Cr2 Y3 Cb4 | Y4 Cr4 Y5, Cb = channel 2 (the u arrays), Cr = channel 1.
// A lane owns 8 pixels, so three writer lanes (phase 0, 1, 2 = (lane - 1) % 3) own 24 pixels = 4 groups = 64 bytes and a
// strip (240 pixels) starts on a group boundary.  Phase 0 writes groups 0-1, phase 1 groups 2-3, phase 2 nothing; the part
// of a group that belongs to the next lane arrives by one shuffle-down of six partial words, so every lane of the warp
// must call this (`writer` gates the stores only).  `out` points at the lane's first byte of row 0 (its phase's groups).
// right_edge (the lane holds the last 8 pixels of the row, widths are multiples of 16): the row ends inside a group, and
// the reference's scalar tail (convert.c:13888-13965) fills the pixels past the edge with the component variables' last
// values.  Phase 0 at the edge: W % 6 == 2, group 1 holds pixels W-2, W-1.  Phase 1 at the edge: W % 6 == 4, group 2
// holds W-4 .. W-1, and no group 3 is written.  In that W % 6 == 4 group the reference's Cb field of word 2 reads one
// element past the Cb row of its scratch strip (the next scratch row's first luma sample, or stale scratch on the
// strip's last row); here it is defined as the last Cb of the row repeated.  Only ceil(W / 6) * 16 bytes per row are written.
__device__ __forceinline__ void emit_v210(const InvParams &p, unsigned char *out, int phase, bool writer, bool right_edge, int r,
                                          const int *ye, const int *yo, const int *ue, const int *uo, const int *ve, const int *vo)
{
    const InvGeom &gy = p.ch[0];
    unsigned char *o = out + (long long)(2 * r) * gy.out_pitch;
#pragma unroll
    for (int rr = 0; rr < 2; rr++) {
        const int *yy = rr ? yo : ye, *uu = rr ? uo : ue, *vv = rr ? vo : ve;
        unsigned y[8], cb[4], cr[4];
#pragma unroll
        for (int i = 0; i < 8; i++) y[i] = row16u(yy[i], 0, 1023);
#pragma unroll
        for (int k = 0; k < 4; k++) { cb[k] = row16u(uu[k], 0, 1023); cr[k] = row16u(vv[k], 0, 1023); }
        // what the previous lane needs from this one: phase 1 -> phase 0 (the rest of its group 1: pixels 0-3 here),
        // phase 2 -> phase 1 (the rest of its group 2: pixels 0-1, and its whole group 3: pixels 2-7)
        const bool p1 = (phase == 1);
        unsigned s[6];
        s[0] = p1 ? (cb[0] << 10) | (y[0] << 20) : cb[0] << 20;
        s[1] = p1 ? v210_word(cr[0], y[1], cb[1]) : v210_word(y[0], cr[0], y[1]);
        s[2] = p1 ? v210_word(y[2], cr[1], y[3]) : v210_word(cb[1], y[2], cr[1]);
        s[3] = v210_word(y[3], cb[2], y[4]);
        s[4] = v210_word(cr[2], y[5], cb[3]);
        s[5] = v210_word(y[6], cr[3], y[7]);
        unsigned n[6];
#pragma unroll
        for (int i = 0; i < 6; i++) n[i] = __shfl_down_sync(kFullMask, s[i], 1);
        unsigned char *q = o + (rr ? gy.out_pitch : 0);
        if (!writer) continue;
        if (phase == 0) {
            *reinterpret_cast<uint4 *>(q) = make_uint4(v210_word(cb[0], y[0], cr[0]), v210_word(y[1], cb[1], y[2]),
                                                       v210_word(cr[1], y[3], cb[2]), v210_word(y[4], cr[2], y[5]));
            *reinterpret_cast<uint4 *>(q + 16) =
                right_edge ? make_uint4(v210_word(cb[3], y[6], cr[3]), v210_word(y[7], cb[3], y[6]), v210_word(cr[3], y[7], cb[3]),
                                        v210_word(y[7], cr[3], y[6]))
                           : make_uint4(v210_word(cb[3], y[6], cr[3]), y[7] | n[0], n[1], n[2]);
        } else if (phase == 1) {
            *reinterpret_cast<uint4 *>(q) =
                make_uint4(v210_word(cb[2], y[4], cr[2]), v210_word(y[5], cb[3], y[6]),
                           cr[3] | (y[7] << 10) | (right_edge ? cb[3] << 20 : n[0]), right_edge ? v210_word(y[7], cr[3], y[6]) : n[1]);
            if (!right_edge) *reinterpret_cast<uint4 *>(q + 16) = make_uint4(n[2], n[3], n[4], n[5]);
        }
    }
}

// OUT = kInv422Out8: packed 8-bit YUYV / UYVY.  kInv422OutYU64: packed 16-bit Y0 C1 Y1 C3 (C1 = channel 1, C3 = channel 2,
// as the YU64 encoder input assigns them), the reference's 16-bit row output (decoder.c:26351-26366 ->
// TransformInverseSpatialUniversalThreadedToRow16u -> InvertHorizontalStrip16s.c:17462 / :16571) -- no dither, bit-exact.
// kInv422OutV210: packed 10-bit V210 (emit_v210), bit-exact too.
template <bool SMALLDQ, int OUT, int MINB>
__global__ void __launch_bounds__(128, MINB) k_inv_422(const __grid_constant__ InvParams p)
{
    constexpr bool OUT16 = (OUT == kInv422OutYU64);
    const int lane = threadIdx.x;
    const int f = blockIdx.z;
    const InvGeom &gy = p.ch[0];
    const InvGeom &gv = p.ch[1];
    const InvGeom &gu = p.ch[2];
    const int strip = blockIdx.x;
    if (strip * kInvStrip >= gy.width) return;
    const int H = gy.height;

    const int col0 = strip * kInvStrip - 4 + lane * 4;      // luma band column
    const bool active = (col0 >= 0) && (col0 < gy.width);
    const bool writer = active && lane >= 1 && lane <= 30;
    const bool left_border = (col0 == 0);
    const bool right_border = (col0 + 4 == gy.width);
    const bool has_border = (strip == 0) || ((strip + 1) * kInvStrip + 4 >= gy.width);
    const unsigned ycol = (unsigned)(col0 * 2), ccol = (unsigned)col0;      // byte offsets (chroma: 2 columns of 2 bytes)
    const unsigned char *in = p.in_base[f];
    // V210: lanes of phase (lane - 1) % 3 = (col0 % 12) / 4 write at 64 bytes per 12 band columns + 32 per phase
    const int phase = (lane + 2) % 3;
    unsigned char *out = p.out_base[f] + gy.out_off +
                         (OUT == kInv422OutV210 ? (long long)(col0 / 12) * 64 + 32 * phase
                                                : (long long)col0 * (OUT16 ? 8 : 4));     // 2 (4) bytes per luma sample, 2 samples per column

    // every lane calls this (the V210 emitter shuffles); the 8- and 16-bit emitters run on the writer lanes only
    auto emit = [&](int r, const int *ye, const int *yo, const int *ue, const int *uo, const int *ve, const int *vo) {
        if constexpr (OUT == kInv422OutV210) emit_v210(p, out, phase, writer, right_border, r, ye, yo, ue, uo, ve, vo);
        else if (writer) emit_422<OUT16>(p, out, col0, r, ye, yo, ue, uo, ve, vo);
    };

    if (blockIdx.y == gridDim.y - 1) {          // border warps: band rows 0 and H-1
        if (threadIdx.y > 1) return;
        const bool bottom = (threadIdx.y == 1);
        int ye[8], yo[8], ue[4], uo[4], ve[4], vo[4];
        inv_border_row<4>(gy, in, bottom, H, ycol, active, has_border, left_border, right_border, ye, yo);
        inv_border_row<2>(gu, in, bottom, H, ccol, active, has_border, left_border, right_border, ue, uo);
        inv_border_row<2>(gv, in, bottom, H, ccol, active, has_border, left_border, right_border, ve, vo);
        emit(bottom ? H - 1 : 0, ye, yo, ue, uo, ve, vo);
        return;
    }
    const int y0 = max((int)(blockIdx.y * blockDim.y + threadIdx.y) * p.th, 1);
    const int y1 = min((int)(blockIdx.y * blockDim.y + threadIdx.y + 1) * p.th, H - 1);
    if (y0 >= y1) return;

    // lanes 0-11: luma (band = lane / 3, line = lane % 3); lanes 12-27: chroma (channel 1 + i / 8, band (i % 8) / 2, line i % 2)
    const int pi = lane - 12;
    const LanePrefetch pf = (lane < 12) ? make_prefetch(gy, in, strip, lane / 3, lane % 3, 2, true)
                                        : make_prefetch((pi & 8) ? gu : gv, in, strip, (pi & 7) >> 1, pi & 1, 1, lane < 28);
    InvChan<4> sy;
    InvChan<2> su, sv;
    inv_prologue<4, SMALLDQ>(sy, gy, in, y0, H, ycol, active);
    inv_prologue<2, SMALLDQ>(su, gu, in, y0, H, ccol, active);
    inv_prologue<2, SMALLDQ>(sv, gv, in, y0, H, ccol, active);
    for (int r = y0; r < y1; r++) {
        pf.issue(r, y1, H);
        int ye[8], yo[8], ue[4], uo[4], ve[4], vo[4];
        inv_step<4, SMALLDQ>(sy, gy, in, r, y1, H, ycol, active, has_border, left_border, right_border, ye, yo);
        inv_step<2, SMALLDQ>(su, gu, in, r, y1, H, ccol, active, has_border, left_border, right_border, ue, uo);
        inv_step<2, SMALLDQ>(sv, gv, in, r, y1, H, ccol, active, has_border, left_border, right_border, ve, vo);
        emit(r, ye, yo, ue, uo, ve, vo);
    }
}

#include "cfb_inverse_tma.inl"

// ----------------------------------------------------------------------------
// final level of a 4:4:4 frame (channels G, R, B): 12 bands -> packed 16-bit R,G,B (RG48).
// Reference: Codec/decoder.c:26886 -> wavelet.c:4947 TransformInverseRGB444ToRGB48: InvertSpatial{Top,Middle,Bottom}Row16sToYUV16
// per channel (horizontal stage InvertHorizontalStrip16s.c:16571 ...ToRow16u: max(t >> 1, 0) << (16 - precision), limited
// as InvParams::hi_simd / tail_col describe), then ConvertPlanarRGB16uToPackedRGB48 (plane 1 -> R, 0 -> G, 2 -> B).
// One warp reconstructs all three channels of its strip, so every lane owns 8 whole pixels = 48 contiguous bytes.
// B64A = true: 16-bit A,R,G,B words instead (64 contiguous bytes per lane), decoder.c:26862 ->
// InvertHorizontalStrip16s.c:13298 InvertHorizontalStrip16sRGB2B64A: alpha is the constant 0xfff << 4 (:13385 a_epi16); colour
// samples are limited to the 12-bit maximum where its SSE2 loop runs (:13387 limiterRGB) and to 65535 in its scalar tail and
// right border column (InvParams::tail_col, here the same for the three channels); native (little-endian) words as the
// reference's decoder leaves them.
// OUT = 2: one 32-bit word per pixel with 10-bit components (RG30 / AB10 / AR10 / R210 / DPX0; decoder.c:26893 ->
// InvertHorizontalStrip16s.c:14812 InvertHorizontalStrip16sRGB2RG30): the 12-bit sample limited to [0, 4095] in every column
// (:14892 limiterRGB; the scalar code clamps alike), >> 2 (:15552), components at bit positions tail_col[0..2] = R, G, B,
// the word byte-swapped when p.uyvy is set (R210, DPX0; :15577-15613).  32 contiguous bytes per lane.
template <bool SMALLDQ, int OUT>
__global__ void __launch_bounds__(128) k_inv_444_rg48(const __grid_constant__ InvParams p)
{
    const int lane = threadIdx.x;
    const int f = blockIdx.z;
    const InvGeom &gg = p.ch[0];
    const InvGeom &gr = p.ch[1];
    const InvGeom &gb = p.ch[2];
    const int strip = blockIdx.x;
    if (strip * kInvStrip >= gg.width) return;
    const int H = gg.height;
    const int col0 = strip * kInvStrip - 4 + lane * 4;
    const bool active = (col0 >= 0) && (col0 < gg.width);
    const bool writer = active && lane >= 1 && lane <= 30;
    const bool left_border = (col0 == 0);
    const bool right_border = (col0 + 4 == gg.width);
    const bool has_border = (strip == 0) || ((strip + 1) * kInvStrip + 4 >= gg.width);
    const unsigned cb = (unsigned)(col0 * 2);
    const unsigned char *in = p.in_base[f];
    constexpr bool B64A = (OUT == 1);
    unsigned char *out = p.out_base[f] + gg.out_off + (long long)col0 * (OUT == 2 ? 8 : B64A ? 16 : 12);      // 2 pixels per band column, 6 (8, 4) bytes per pixel
    const int us = p.up_shift;

    auto emit = [&](int r, const int *ge, const int *go, const int *re, const int *ro, const int *be, const int *bo) {
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
            const int *G = rr ? go : ge, *R = rr ? ro : re, *B = rr ? bo : be;
            if constexpr (OUT == 2) {
                unsigned char *q = out + (long long)(2 * r + rr) * gg.out_pitch;
                unsigned w[8];
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const unsigned word = ((row16u(R[i], 0, 4095) >> 2) << p.tail_col[0]) | ((row16u(G[i], 0, 4095) >> 2) << p.tail_col[1]) |
                                          ((row16u(B[i], 0, 4095) >> 2) << p.tail_col[2]);
                    w[i] = p.uyvy ? __byte_perm(word, 0, 0x0123) : word;
                }
                *reinterpret_cast<uint4 *>(q) = make_uint4(w[0], w[1], w[2], w[3]);
                *reinterpret_cast<uint4 *>(q + 16) = make_uint4(w[4], w[5], w[6], w[7]);
            } else if constexpr (B64A) {
                unsigned char *q = out + (long long)(2 * r + rr) * gg.out_pitch;
                const unsigned alpha = (unsigned)p.hi_simd;
#pragma unroll
                for (int i = 0; i < 8; i += 2) {        // pixels i and i + 1 belong to band column col0 + i / 2
                    const int hi = (col0 + (i >> 1) >= p.tail_col[0]) ? 65535 : p.hi_simd;
                    uint4 w;
                    w.x = alpha | (row16u(R[i], us, hi) << 16);
                    w.y = row16u(G[i], us, hi) | (row16u(B[i], us, hi) << 16);
                    w.z = alpha | (row16u(R[i + 1], us, hi) << 16);
                    w.w = row16u(G[i + 1], us, hi) | (row16u(B[i + 1], us, hi) << 16);
                    *reinterpret_cast<uint4 *>(q + 8 * i) = w;
                }
            } else {
                unsigned short v[24];
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const int bc = col0 + (i >> 1);
                    v[3 * i + 0] = (unsigned short)row16u(R[i], us, bc >= p.tail_col[1] ? 65535 : p.hi_simd);
                    v[3 * i + 1] = (unsigned short)row16u(G[i], us, bc >= p.tail_col[0] ? 65535 : p.hi_simd);
                    v[3 * i + 2] = (unsigned short)row16u(B[i], us, bc >= p.tail_col[2] ? 65535 : p.hi_simd);
                }
                unsigned w[12];
#pragma unroll
                for (int i = 0; i < 12; i++) w[i] = (unsigned)v[2 * i] | ((unsigned)v[2 * i + 1] << 16);
                unsigned char *q = out + (long long)(2 * r + rr) * gg.out_pitch;
                *reinterpret_cast<uint4 *>(q) = make_uint4(w[0], w[1], w[2], w[3]);
                *reinterpret_cast<uint4 *>(q + 16) = make_uint4(w[4], w[5], w[6], w[7]);
                *reinterpret_cast<uint4 *>(q + 32) = make_uint4(w[8], w[9], w[10], w[11]);
            }
        }
    };

    if (blockIdx.y == gridDim.y - 1) {          // border warps: band rows 0 and H-1
        if (threadIdx.y > 1) return;
        const bool bottom = (threadIdx.y == 1);
        int ge[8], go[8], re[8], ro[8], be[8], bo[8];
        inv_border_row<4>(gg, in, bottom, H, cb, active, has_border, left_border, right_border, ge, go);
        inv_border_row<4>(gr, in, bottom, H, cb, active, has_border, left_border, right_border, re, ro);
        inv_border_row<4>(gb, in, bottom, H, cb, active, has_border, left_border, right_border, be, bo);
        if (writer) emit(bottom ? H - 1 : 0, ge, go, re, ro, be, bo);
        return;
    }
    const int y0 = max((int)(blockIdx.y * blockDim.y + threadIdx.y) * p.th, 1);
    const int y1 = min((int)(blockIdx.y * blockDim.y + threadIdx.y + 1) * p.th, H - 1);
    if (y0 >= y1) return;
    InvChan<4> sg, sr, sb;
    inv_prologue<4, SMALLDQ>(sg, gg, in, y0, H, cb, active);
    inv_prologue<4, SMALLDQ>(sr, gr, in, y0, H, cb, active);
    inv_prologue<4, SMALLDQ>(sb, gb, in, y0, H, cb, active);
    for (int r = y0; r < y1; r++) {
        int ge[8], go[8], re[8], ro[8], be[8], bo[8];
        inv_step<4, SMALLDQ>(sg, gg, in, r, y1, H, cb, active, has_border, left_border, right_border, ge, go);
        inv_step<4, SMALLDQ>(sr, gr, in, r, y1, H, cb, active, has_border, left_border, right_border, re, ro);
        inv_step<4, SMALLDQ>(sb, gb, in, r, y1, H, cb, active, has_border, left_border, right_border, be, bo);
        if (writer) emit(r, ge, go, re, ro, be, bo);
    }
}

// ----------------------------------------------------------------------------
// Interlaced sources: inverse of the frame (field) transform at level 1
//   Codec/decoder.c:21493 TransformInverseFrameToYUV / :22027 TransformInverseFrameToRow16u:
//   t_low = hinv(LL, LH), t_high = hinv(HL, HH) (InvertHorizontalRow16s8sTo16sBuffered), then
//   even row = (t_low - t_high) >> 1, odd row = (t_low + t_high) >> 1 (Codec/temporal.c:3741 InvertInterlaced16s).
// The coded HL band is difference coded along each row; the reference integrates it on the host after the FSM
// decode (decoder.c:20822-20836 `line[x] += line[x-1]`, int16 wrap).  Here k_fields_carry computes, per band row
// and strip, the sum of all coefficients left of the strip, and the inverse kernel finishes the prefix sum with a
// warp scan, so the coded buffer keeps the exact format the forward path wrote.
template <int NC>
__device__ __forceinline__ int row_segment_sum(const unsigned char *row, int c0, int c1, int lane)
{
    const int col = c0 + NC * lane;
    int v = 0;
    if (col < c1) {
        if (NC == 4) { const uint2 w = __ldg(reinterpret_cast<const uint2 *>(row + col * 2)); v = lo16(w.x) + hi16(w.x) + lo16(w.y) + hi16(w.y); }
        else { const unsigned w = __ldg(reinterpret_cast<const unsigned *>(row + col * 2)); v = lo16(w) + hi16(w); }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(kFullMask, v, d);
    return v;
}

__global__ void __launch_bounds__(128) k_fields_carry(const __grid_constant__ InvParams p, const FieldsAux a)
{
    const int lane = threadIdx.x;
    const int row = blockIdx.x * blockDim.y + threadIdx.y;
    const int c = blockIdx.y, f = blockIdx.z;
    const InvGeom &g = p.ch[c];
    if (row >= g.height) return;
    const unsigned char *hl = p.in_base[f] + g.band_off[2] + (long long)row * g.pitch;
    int *out = a.carry + ((long long)(f * p.nchan + c) * a.maxh + row) * a.nstrips;
    const int W = (c == 0) ? kInvStrip : kInvStrip / 2, halo = (c == 0) ? 4 : 2;
    int total = 0;
    for (int s = 0; s < a.nstrips; s++) {
        const int c0 = max(s * W - halo, 0), c1 = min((s + 1) * W - halo, g.width);
        if (lane == 0) out[s] = total;
        if (c0 >= g.width) continue;
        total += (c == 0) ? row_segment_sum<4>(hl, c0, c1, lane) : row_segment_sum<2>(hl, c0, c1, lane);
    }
}

// inclusive prefix of the lane's NC raw HL values across the warp (lane order = column order) + carry-in
template <int NC>
__device__ __forceinline__ void integrate_row(int *h, int carry)
{
#pragma unroll
    for (int i = 1; i < NC; i++) h[i] += h[i - 1];
    int t = h[NC - 1];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int u = __shfl_up_sync(kFullMask, t, d);
        if ((int)threadIdx.x >= d) t += u;
    }
    const int excl = t - h[NC - 1] + carry;
#pragma unroll
    for (int i = 0; i < NC; i++) h[i] += excl;
}

template <int NC>
__device__ __forceinline__ void fields_channel(const InvGeom &g, const unsigned char *in, int r, unsigned colbyte, bool active,
                                               int carry, bool integrate, bool has_border, bool left_border, bool right_border,
                                               int *even, int *odd)
{
    RawCols<NC> a, b, c, d;
    const unsigned off = (unsigned)r * g.pitch + colbyte;
    load_raw<NC>(in, g.band_off[0], off, active, a);
    load_raw<NC>(in, g.band_off[1], off, active, b);
    load_raw<NC>(in, g.band_off[2], off, active, c);
    load_raw<NC>(in, g.band_off[3], off, active, d);
    int ll[NC], lh[NC], hl[NC], hh[NC];
    Expand<false, NC>::ll(a, ll);
    Expand<false, NC>::hp(b, g.dq[1], lh);
    Expand<false, NC>::ll(c, hl);               // raw: integrate first, dequantise after (ring arithmetic, same result)
    Expand<false, NC>::hp(d, g.dq[3], hh);
    if (integrate) integrate_row<NC>(hl, carry);     // warp-uniform: off when the host already integrated the band
#pragma unroll
    for (int i = 0; i < NC; i++) hl[i] = (int)(short)(hl[i] * g.dq[2]);     // int16 wrap as `line[x] += line[x-1]` on PIXEL
    int tl[2 * NC], th[2 * NC];
    hinv<NC>(ll, lh, has_border, left_border, right_border, tl);
    hinv<NC>(hl, hh, has_border, left_border, right_border, th);
#pragma unroll
    for (int i = 0; i < 2 * NC; i++) {
        const int lo = tl[i] >> 1, hi = th[i] >> 1;
        even[i] = (lo - hi) >> 1;
        odd[i] = (lo + hi) >> 1;
    }
}

template <bool PLANAR>
__global__ void __launch_bounds__(128) k_inv_fields(const __grid_constant__ InvParams p, const FieldsAux a)
{
    const int lane = threadIdx.x;
    const int f = blockIdx.z;
    const InvGeom &gy = p.ch[0];
    const InvGeom &gv = p.ch[1];
    const InvGeom &gu = p.ch[2];
    const int strip = blockIdx.x;
    if (strip * kInvStrip >= gy.width) return;
    const int H = gy.height;
    const int col0 = strip * kInvStrip - 4 + lane * 4;      // luma band column
    const bool active = (col0 >= 0) && (col0 < gy.width);
    const bool writer = active && lane >= 1 && lane <= 30;
    const bool left_border = (col0 == 0);
    const bool right_border = (col0 + 4 == gy.width);
    const bool has_border = (strip == 0) || ((strip + 1) * kInvStrip + 4 >= gy.width);
    const unsigned ycol = (unsigned)(col0 * 2), ccol = (unsigned)col0;
    const unsigned char *in = p.in_base[f];
    unsigned char *out = p.out_base[f];
    const int y0 = (blockIdx.y * blockDim.y + threadIdx.y) * p.th;
    const int y1 = min(y0 + p.th, H);
    const int sh = p.shift;         // precision - 8
    const int *cy = a.carry + ((long long)(f * 3 + 0) * a.maxh) * a.nstrips + strip;
    const int *cv = a.carry + ((long long)(f * 3 + 1) * a.maxh) * a.nstrips + strip;
    const int *cu = a.carry + ((long long)(f * 3 + 2) * a.maxh) * a.nstrips + strip;
    for (int r = y0; r < y1; r++) {
        int ye[8], yo[8], ue[4], uo[4], ve[4], vo[4];
        const bool integ = (a.pad == 0);
        fields_channel<4>(gy, in, r, ycol, active, integ ? __ldg(cy + (long long)r * a.nstrips) : 0, integ, has_border, left_border, right_border, ye, yo);
        fields_channel<2>(gu, in, r, ccol, active, integ ? __ldg(cu + (long long)r * a.nstrips) : 0, integ, has_border, left_border, right_border, ue, uo);
        fields_channel<2>(gv, in, r, ccol, active, integ ? __ldg(cv + (long long)r * a.nstrips) : 0, integ, has_border, left_border, right_border, ve, vo);
        if (!writer) continue;
        if (PLANAR) {
#pragma unroll
            for (int rr = 0; rr < 2; rr++) {
                const int *yy = rr ? yo : ye, *uu = rr ? uo : ue, *vv = rr ? vo : ve;
                const long long row = 2 * r + rr;
                *reinterpret_cast<uint4 *>(out + gy.out_off + row * gy.out_pitch + (long long)col0 * 4) =
                    make_uint4(pack_sat16(yy[0], yy[1]), pack_sat16(yy[2], yy[3]), pack_sat16(yy[4], yy[5]), pack_sat16(yy[6], yy[7]));
                *reinterpret_cast<uint2 *>(out + gu.out_off + row * gu.out_pitch + (long long)col0 * 2) =
                    make_uint2(pack_sat16(uu[0], uu[1]), pack_sat16(uu[2], uu[3]));
                *reinterpret_cast<uint2 *>(out + gv.out_off + row * gv.out_pitch + (long long)col0 * 2) =
                    make_uint2(pack_sat16(vv[0], vv[1]), pack_sat16(vv[2], vv[3]));
            }
        } else {
            // 8-bit reduction with the same ordered dither as k_inv_422: out = sat_u8((v + d) >> (precision - 8)),
            // d = (x ^ y) & 1 scaled to the shift, inside the reference's {v >> 2, (v + 1) >> 2} envelope
            unsigned char *o = out + gy.out_off + (long long)(2 * r) * gy.out_pitch + (long long)col0 * 4;
#pragma unroll
            for (int rr = 0; rr < 2; rr++) {
                const int *yy = rr ? yo : ye, *uu = rr ? uo : ue, *vv = rr ? vo : ve;
                const int d0 = (rr ? 1 : 0) << (sh - 2), d1 = (rr ? 0 : 1) << (sh - 2);
                unsigned w[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int ya = (yy[2 * k] + d0) >> sh, yb = (yy[2 * k + 1] + d1) >> sh;
                    const int cu8 = (uu[k] + ((k & 1) ? d1 : d0)) >> sh, cv8 = (vv[k] + ((k & 1) ? d1 : d0)) >> sh;
                    w[k] = p.uyvy ? pack_u8x4(cu8, ya, cv8, yb) : pack_u8x4(ya, cu8, yb, cv8);
                }
                *reinterpret_cast<uint4 *>(o + (rr ? gy.out_pitch : 0)) = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
    }
}

// ----------------------------------------------------------------------------
// Reduced-resolution decode: pack the lowpass images of the three 4:2:2 channels to 8-bit YUYV/UYVY.
//   half    (LL1): Codec/frame.c:11742 ConvertLowpass16s10bitToYUV   out = sat_u8(ll >> 4)        (signed shift)
//   quarter (LL2): Codec/temporal.c:11362 CopyQuarterRowToBuffer     out = packus((uint16)ll >> 4) (unsigned shift)
// Byte order Y0 U Y1 V with U = channel 2, V = channel 1 (the reference's "u"/"v" names are swapped, the bytes are
// these).  One thread = 8 luma + 4 + 4 chroma coefficients = 16 output bytes; purely streaming.
__global__ void __launch_bounds__(256) k_lowpass_422(const __grid_constant__ InvParams p)
{
    const int frame = blockIdx.z;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int x8 = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
    const InvGeom &gy = p.ch[0], &gv = p.ch[1], &gu = p.ch[2];
    if (y >= gy.height || x8 >= gy.width) return;
    const unsigned char *in = p.in_base[frame];
    const uint4 yr = *reinterpret_cast<const uint4 *>(in + gy.band_off[0] + (long long)y * gy.pitch + x8 * 2);
    const uint2 ur = *reinterpret_cast<const uint2 *>(in + gu.band_off[0] + (long long)y * gu.pitch + x8);
    const uint2 vr = *reinterpret_cast<const uint2 *>(in + gv.band_off[0] + (long long)y * gv.pitch + x8);
    const unsigned yw[4] = {yr.x, yr.y, yr.z, yr.w}, uw[2] = {ur.x, ur.y}, vw[2] = {vr.x, vr.y};
    const int sh = p.shift;
    const bool uns = p.pad != 0;
    auto lo = [&](unsigned w) { return uns ? (int)(w & 0xffffu) >> sh : lo16(w) >> sh; };
    auto hi = [&](unsigned w) { return uns ? (int)(w >> 16) >> sh : hi16(w) >> sh; };
    unsigned o[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int ya = lo(yw[k]), yb = hi(yw[k]);
        const int cu = (k & 1) ? hi(uw[k >> 1]) : lo(uw[k >> 1]);
        const int cv = (k & 1) ? hi(vw[k >> 1]) : lo(vw[k >> 1]);
        o[k] = p.uyvy ? pack_u8x4(cu, ya, cv, yb) : pack_u8x4(ya, cu, yb, cv);
    }
    unsigned char *out = p.out_base[frame] + (long long)y * gy.out_pitch + x8 * 2;
    const int rem = gy.width - x8;          // widths are even; a ragged tail stores whole 4-byte pairs
    if (rem >= 8) *reinterpret_cast<uint4 *>(out) = make_uint4(o[0], o[1], o[2], o[3]);
    else for (int k = 0; k < rem / 2; k++) reinterpret_cast<unsigned *>(out)[k] = o[k];
}

// ----------------------------------------------------------------------------
static inline int ceil_div_i(int a, int b) { return (a + b - 1) / b; }

cudaError_t launch_inv_plane(const InvParams &p, int descale, cudaStream_t stream)
{
    int maxw = 0, maxh = 0;
    for (int c = 0; c < p.nchan; c++) { maxw = max(maxw, p.ch[c].width); maxh = max(maxh, p.ch[c].height); }
    dim3 block(32, 4);
    dim3 grid(ceil_div_i(maxw, kInvStrip), ceil_div_i(ceil_div_i(maxh, p.th), (int)block.y) + 1, p.nframes * p.nchan);
    bool small = true;
    for (int c = 0; c < p.nchan; c++) for (int b = 1; b < 4; b++) small = small && (p.ch[c].dq[b] >= 0 && p.ch[c].dq[b] <= 255);
    if (descale) { if (small) k_inv_plane<2, true><<<grid, block, 0, stream>>>(p); else k_inv_plane<2, false><<<grid, block, 0, stream>>>(p); }
    else { if (small) k_inv_plane<0, true><<<grid, block, 0, stream>>>(p); else k_inv_plane<0, false><<<grid, block, 0, stream>>>(p); }
    bool ragged = false;
    for (int c = 0; c < p.nchan; c++) ragged = ragged || (p.ch[c].width & 3);
    if (ragged) {       // the 1-3 band columns right of the last full lane (they include the right border)
        dim3 eblock(128), egrid(ceil_div_i(maxh, 128), 3, p.nframes * p.nchan);
        if (descale) k_inv_plane_edge<2><<<egrid, eblock, 0, stream>>>(p); else k_inv_plane_edge<0><<<egrid, eblock, 0, stream>>>(p);
    }
    return cudaGetLastError();
}

// CFB_INV422 selects the variant of the final 4:2:2 level (A/B evidence in profiles/r02_ab_inv422.txt):
//   r1 (default)  global loads straight into registers, 4 CTAs per SM; r1b5: the same capped at 102 registers (5 CTAs per SM)
//   tma<R><NS>    TMA ring with R band rows per stage and NS stages per warp -- measured SLOWER than r1 (183 vs 171 us per
//                 16 4K frames at best): twelve bands per row mean six copy instructions per stage, each wrapped in an
//                 elect / uniform-register sequence, i.e. as many issue slots as the loads they replace, and the rings
//                 cost occupancy
static int inv422_variant()
{
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("CFB_INV422");
        v = 0;
        if (e && !strcmp(e, "r1b5")) v = 5;
        else if (e && !strncmp(e, "tma", 3) && strlen(e) == 5) v = atoi(e + 3);
    }
    return v;
}

template <bool SMALLDQ, bool OUT16, int R, int NS>
static cudaError_t launch_inv_422_tma_t(const InvParams &p, const InvTmaMaps &tm, dim3 grid, dim3 block, cudaStream_t stream)
{
    constexpr int smem = 4 * NS * InvStage<R>::kBytes + 4 * NS * 8;
    constexpr int minb = (smem <= 56 * 1024) ? 4 : (smem <= 75 * 1024 ? 3 : (smem <= 113 * 1024 ? 2 : 1));
    static_assert(smem <= 227 * 1024, "ring does not fit the shared memory of an SM");
    auto kern = k_inv_422_tma<SMALLDQ, OUT16, R, NS, minb>;
    static bool attr_set = false;       // per instantiation
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        attr_set = true;
    }
    kern<<<grid, block, smem, stream>>>(p, tm);
    return cudaGetLastError();
}

template <bool SMALLDQ, bool OUT16>
static cudaError_t launch_inv_422_tma(const InvParams &p, const InvTmaMaps &tm, dim3 grid, dim3 block, int variant, cudaStream_t stream)
{
    switch (variant) {
    case 16: return launch_inv_422_tma_t<SMALLDQ, OUT16, 1, 6>(p, tm, grid, block, stream);
    case 18: return launch_inv_422_tma_t<SMALLDQ, OUT16, 1, 8>(p, tm, grid, block, stream);
    case 23: return launch_inv_422_tma_t<SMALLDQ, OUT16, 2, 3>(p, tm, grid, block, stream);
    case 44: return launch_inv_422_tma_t<SMALLDQ, OUT16, 4, 4>(p, tm, grid, block, stream);
    case 43: return launch_inv_422_tma_t<SMALLDQ, OUT16, 4, 3>(p, tm, grid, block, stream);
    case 42: return launch_inv_422_tma_t<SMALLDQ, OUT16, 4, 2>(p, tm, grid, block, stream);
    case 22: return launch_inv_422_tma_t<SMALLDQ, OUT16, 2, 2>(p, tm, grid, block, stream);
    default: return launch_inv_422_tma_t<SMALLDQ, OUT16, 2, 4>(p, tm, grid, block, stream);
    }
}

cudaError_t launch_inv_422(const InvParams &p, int out, cudaStream_t stream)
{
    dim3 block(32, 4);
    dim3 grid(ceil_div_i(p.ch[0].width, kInvStrip), ceil_div_i(ceil_div_i(p.ch[0].height, p.th), (int)block.y) + 1, p.nframes);
    bool small = true;
    for (int c = 0; c < 3; c++) for (int b = 1; b < 4; b++) small = small && (p.ch[c].dq[b] >= 0 && p.ch[c].dq[b] <= 255);
    if (out == kInv422OutV210) {        // register kernel only: the TMA variant lost its A/B (profiles/r02_ab_inv422.txt)
        if (small) k_inv_422<true, kInv422OutV210, 4><<<grid, block, 0, stream>>>(p);
        else k_inv_422<false, kInv422OutV210, 4><<<grid, block, 0, stream>>>(p);
        return cudaGetLastError();
    }
    const bool out16 = (out == kInv422OutYU64);
    // The TMA path needs 16-byte aligned band starts and pitches (cfb_layout_compute guarantees both for pyramids it laid
    // out), whole 32-bit elements per band row, and LH / HL / HH of a channel equally spaced
    const int variant = inv422_variant();
    bool tma_ok = variant >= 10;
    for (int c = 0; c < 3 && tma_ok; c++) {
        const InvGeom &g = p.ch[c];
        const long long d1 = g.band_off[2] - g.band_off[1], d2 = g.band_off[3] - g.band_off[2];
        tma_ok = !(g.width & 1) && !(g.pitch & 15) && d1 == d2 && d1 > 0 && !(d1 & 15) && !(g.band_off[0] & 15) && !(g.band_off[1] & 15);
    }
    for (int i = 0; i < p.nframes && tma_ok; i++) tma_ok = !((uintptr_t)p.in_base[i] & 15);
    if (tma_ok) {
        InvTmaMaps tm;
        for (int i = 0; i < p.nframes; i++)
            for (int c = 0; c < 3; c++) {
                const InvGeom &g = p.ch[c];
                const uint32_t box = (c == 0) ? kInvBoxY : kInvBoxC;
                const int R = variant / 10;
                cudaError_t e = tmap_encode_2d(&tm.m[i][2 * c], p.in_base[i] + g.band_off[0], (uint64_t)g.width * 2, (uint64_t)g.height,
                                               (uint64_t)g.pitch, box, R);
                if (e == cudaSuccess)
                    e = tmap_encode_3d(&tm.m[i][2 * c + 1], p.in_base[i] + g.band_off[1], (uint64_t)g.width * 2, (uint64_t)g.height,
                                       (uint64_t)g.pitch, 3, (uint64_t)(g.band_off[2] - g.band_off[1]), box, R, 3);
                if (e != cudaSuccess) return e;
            }
        if (out16) return small ? launch_inv_422_tma<true, true>(p, tm, grid, block, variant, stream) : launch_inv_422_tma<false, true>(p, tm, grid, block, variant, stream);
        return small ? launch_inv_422_tma<true, false>(p, tm, grid, block, variant, stream) : launch_inv_422_tma<false, false>(p, tm, grid, block, variant, stream);
    }
    constexpr int O8 = kInv422Out8, O16 = kInv422OutYU64;
    if (out16) { if (small) k_inv_422<true, O16, 3><<<grid, block, 0, stream>>>(p); else k_inv_422<false, O16, 3><<<grid, block, 0, stream>>>(p); }
    else if (variant == 5) { if (small) k_inv_422<true, O8, 5><<<grid, block, 0, stream>>>(p); else k_inv_422<false, O8, 5><<<grid, block, 0, stream>>>(p); }
    else { if (small) k_inv_422<true, O8, 4><<<grid, block, 0, stream>>>(p); else k_inv_422<false, O8, 4><<<grid, block, 0, stream>>>(p); }
    return cudaGetLastError();
}

// out: 0 RG48, 1 B64A, 2 10-bit packed RGB
cudaError_t launch_inv_444_rg48(const InvParams &p, int out, cudaStream_t stream)
{
    dim3 block(32, 4);
    dim3 grid(ceil_div_i(p.ch[0].width, kInvStrip), ceil_div_i(ceil_div_i(p.ch[0].height, p.th), (int)block.y) + 1, p.nframes);
    bool small = true;
    for (int c = 0; c < 3; c++) for (int b = 1; b < 4; b++) small = small && (p.ch[c].dq[b] >= 0 && p.ch[c].dq[b] <= 255);
    if (out == 2) { if (small) k_inv_444_rg48<true, 2><<<grid, block, 0, stream>>>(p); else k_inv_444_rg48<false, 2><<<grid, block, 0, stream>>>(p); }
    else if (out == 1) { if (small) k_inv_444_rg48<true, 1><<<grid, block, 0, stream>>>(p); else k_inv_444_rg48<false, 1><<<grid, block, 0, stream>>>(p); }
    else { if (small) k_inv_444_rg48<true, 0><<<grid, block, 0, stream>>>(p); else k_inv_444_rg48<false, 0><<<grid, block, 0, stream>>>(p); }
    return cudaGetLastError();
}

cudaError_t launch_inv_fields(const InvParams &p, const FieldsAux &a, bool planar, cudaStream_t stream)
{
    dim3 block(32, 4);
    dim3 cgrid(ceil_div_i(p.ch[0].height, (int)block.y), 3, p.nframes);
    if (a.pad == 0) k_fields_carry<<<cgrid, block, 0, stream>>>(p, a);     // pad != 0: HL arrives integrated (decoder.c:20822)
    dim3 grid(ceil_div_i(p.ch[0].width, kInvStrip), ceil_div_i(ceil_div_i(p.ch[0].height, p.th), (int)block.y), p.nframes);
    if (planar) k_inv_fields<true><<<grid, block, 0, stream>>>(p, a);
    else k_inv_fields<false><<<grid, block, 0, stream>>>(p, a);
    return cudaGetLastError();
}

cudaError_t launch_lowpass_422(const InvParams &p, cudaStream_t stream)
{
    dim3 block(32, 8);
    dim3 grid(ceil_div_i(ceil_div_i(p.ch[0].width, 8), 32), ceil_div_i(p.ch[0].height, 8), p.nframes);
    k_lowpass_422<<<grid, block, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace cfb
