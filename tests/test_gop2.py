"""Two-frame GOP (FIELDPLUS pyramid, Codec/encoder.c:8431): the reference's gop_length = 2 encode leaves six wavelets
per channel; they are reproduced (a) on CPU by composing the oracle's level / temporal functions and (b) on the GPU by
composing the C-ABI building blocks device-resident (cfb_forward_device for level 1 of both frames,
cfb_temporal_forward_device, cfb_level_forward_device), then inverted the same way."""
import glob
import importlib
import os

import ctypes as C
import numpy as np
import pytest

import oracle_lib as ol
import parity_util as pu
from ref_golden import Golden

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gop2_*.npz")))
needs_ref = pytest.mark.skipif(not ol.ref_available(), reason="oracle/_ref not built (reference absent)")


def _load(path):
    z = np.load(path)
    bands = {tuple(int(v) for v in k.split("_")[1:]): z[k] for k in z.files if k.startswith("g_")}
    return z["frame_a"], z["frame_b"], z["quant"].tolist(), z["prescale"].tolist(), int(z["quality"]), bands


def _oracle_blocks():
    orc, lib = ol.oracle(), ol.load_oracle()
    vp = C.c_void_p

    def temporal(a, b):
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        lo, hi = np.zeros_like(a), np.zeros_like(a)
        h, w = a.shape
        lib.orc_temporal_fwd(vp(a.ctypes.data), vp(b.ctypes.data), w * 2, w, h, vp(lo.ctypes.data), vp(hi.ctypes.data), w * 2)
        return lo, hi

    return (lambda f, c, q: orc.fwd_level_422(f, c, 0, q, 10, 2), temporal,
            lambda p, pre, q: orc.fwd_level(p, 1 if pre == 2 else 0, q, 2))


def _compare(got, want):
    for key in sorted(want):
        assert np.array_equal(got[key], want[key]), f"(channel, wavelet, band) {key}"


def test_golden_present():
    assert GOLDEN


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_oracle_gop2_reproduces_golden(path):
    fa, fb, quant, prescale, _, bands = _load(path)
    assert prescale[0][4] == 2 and prescale[0][3] == 0          # FIELDPLUS schedule (wavelet.c:1710)
    _compare(pu.gop2_pyramid(*_oracle_blocks(), fa, fb, quant, prescale), bands)


@needs_ref
@pytest.mark.parametrize("size,quality", [((256, 64), 3), ((704, 96), 5), ((1920, 1080), 4)])
def test_oracle_gop2_matches_reference_encoder(size, quality):
    w, h = size
    ref_lib = ol.load_ref()
    fa, fb = pu.qbist_yuy2(ref_lib, w, h, 1), pu.qbist_yuy2(ref_lib, w, h, 3)
    bands, quant, prescale = pu.ref_encode_gop2(ref_lib, fa, fb, w, h, quality)
    got = pu.gop2_pyramid(*_oracle_blocks(), fa, fb, quant, prescale)
    _compare(got, {k: v for k, v in bands.items() if k in got})


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("shape,prescale,div", [((48, 24), 0, [1, 6, 6, 3]), ((64, 128), 2, [1, 12, 12, 6]), ((96, 960), 0, [4, 48, 48, 24]),
                                                 ((540, 960), 2, [1, 24, 24, 12]), ((1080, 1920), 0, [1, 48, 48, 24])])
def test_cuda_single_level_vs_oracle(shape, prescale, div):
    """cfb_level_forward/inverse_host on free-standing planes, incl. a quantised LL (divisor[0] = 4)."""
    pkg = importlib.import_module("cineform-sdk_b200")
    h, w = shape
    rng = np.random.default_rng(h + w)
    plane = rng.integers(0, 4096, (h, w)).astype(np.int16)
    orc = ol.oracle()
    want = orc.fwd_level(plane, 1 if prescale == 2 else 0, div, 2)
    with pkg.Context(0) as ctx:
        got = ctx.level_forward(plane, prescale, div)
        for g, w_ in zip(got, want):
            assert np.array_equal(g, w_)
        if div[0] == 1:
            deq = [want[0]] + [pu.dequantize(want[b], div[b]) for b in (1, 2, 3)]
            back = ctx.level_inverse(want, prescale, div)
            assert np.array_equal(back, orc.inv_level(*deq, 2 if prescale == 2 else 0))


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_cuda_gop2_device_resident(path):
    """Whole FIELDPLUS pyramid on the device through public entry points only, checked against the reference's bands;
    then the inverse composition back to the two frames' level-1 lowpass images."""
    import torch
    pkg = importlib.import_module("cineform-sdk_b200")
    fa, fb, quant, prescale, quality, bands = _load(path)
    h, w2 = fa.shape
    w = w2 // 2
    desc = pkg.FrameDesc(w, h, pkg.PIXEL_YUYV)
    with pkg.Context(0) as ctx, pkg.Codec(ctx, desc, 2) as codec:
        stream = torch.cuda.ExternalStream(ctx.stream)
        lay = codec.layout
        q = pkg.make_quant([[quant[c][0], [1, 1, 1, 1], [1, 1, 1, 1]] for c in range(3)], (0, 0, 0))
        with torch.cuda.stream(stream):
            d_frames = [torch.from_numpy(f).cuda() for f in (fa, fb)]
            d_pyr = [torch.zeros(lay.total_bytes, dtype=torch.uint8, device="cuda") for _ in range(2)]
        codec.set_level_mask(1, 7)                      # level 1 only: bands of wavelet 0 / 1 + LL1 in the scratch region
        codec.forward_device([t.data_ptr() for t in d_frames], lay.frame_pitch, q, [t.data_ptr() for t in d_pyr])
        got = {}
        ctx.synchronize()
        host = [t.cpu().numpy() for t in d_pyr]
        for k in (0, 1):
            for c in range(3):
                for b in (1, 2, 3):
                    got[(c, k, b)] = codec.band_view(host[k], c, 0, b).copy()

        def dev_plane(hh, ww):
            with torch.cuda.stream(stream):
                return torch.zeros((hh, (ww * 2 + 15) // 16 * 8), dtype=torch.int16, device="cuda")

        def fetch(t, hh, ww):
            ctx.synchronize()
            return t.cpu().numpy()[:hh, :ww].copy()

        for c in range(3):
            ll = lay.band[c][0][0]
            lw, lh, lp = ll.width, ll.height, ll.pitch
            a_ptr, b_ptr = d_pyr[0].data_ptr() + ll.offset, d_pyr[1].data_ptr() + ll.offset
            low, high = dev_plane(lh, lw), dev_plane(lh, lw)
            tp = low.stride(0) * 2
            ctx.temporal_forward_device(a_ptr, b_ptr, lp, low.data_ptr(), high.data_ptr(), tp, lw, lh)
            got[(c, 2, 0)], got[(c, 2, 1)] = fetch(low, lh, lw), fetch(high, lh, lw)

            def level(src, sw, sh, k):
                bands_d = [dev_plane(sh // 2, sw // 2) for _ in range(4)]
                ctx.level_forward_device(sw, sh, src.stride(0) * 2, bands_d[0].stride(0) * 2, prescale[c][k], quant[c][k], 2,
                                         src.data_ptr(), [t.data_ptr() for t in bands_d])
                return bands_d

            w3 = level(high, lw, lh, 3)
            w4 = level(low, lw, lh, 4)
            w5 = level(w4[0], lw // 2, lh // 2, 5)
            for b in range(4):
                got[(c, 3, b)] = fetch(w3[b], lh // 2, lw // 2)
                got[(c, 5, b)] = fetch(w5[b], lh // 4, lw // 4)
            for b in (1, 2, 3):
                got[(c, 4, b)] = fetch(w4[b], lh // 2, lw // 2)

            # inverse composition: wavelet 5 -> LL of wavelet 4 -> temporal low; wavelet 3 -> temporal high;
            # temporal inverse -> the two frames' LL1 (decoder.c:13109-13170).  Checked against the oracle.
            orc = ol.oracle()
            ll4 = dev_plane(lh // 2, lw // 2)
            ctx.level_inverse_device(lw // 2, lh // 2, ll4.stride(0) * 2, w5[0].stride(0) * 2, prescale[c][5], quant[c][5],
                                     [t.data_ptr() for t in w5], ll4.data_ptr())
            tl, th = dev_plane(lh, lw), dev_plane(lh, lw)
            ctx.level_inverse_device(lw, lh, tl.stride(0) * 2, ll4.stride(0) * 2, prescale[c][4], quant[c][4],
                                     [ll4.data_ptr()] + [t.data_ptr() for t in w4[1:]], tl.data_ptr())
            ctx.level_inverse_device(lw, lh, th.stride(0) * 2, w3[0].stride(0) * 2, prescale[c][3], quant[c][3],
                                     [t.data_ptr() for t in w3], th.data_ptr())
            ra, rb = dev_plane(lh, lw), dev_plane(lh, lw)
            ctx.temporal_inverse_device(tl.data_ptr(), th.data_ptr(), tl.stride(0) * 2, ra.data_ptr(), rb.data_ptr(), ra.stride(0) * 2, lw, lh)

            def orc_inv(bands4, k):
                deq = [bands4[0]] + [pu.dequantize(bands4[b], quant[c][k][b]) for b in (1, 2, 3)]
                return orc.inv_level(*deq, 2 if prescale[c][k] == 2 else 0)

            o_ll4 = orc_inv([got[(c, 5, b)] for b in range(4)], 5)
            o_tl = orc_inv([o_ll4] + [got[(c, 4, b)] for b in (1, 2, 3)], 4)
            o_th = orc_inv([got[(c, 3, b)] for b in range(4)], 3)
            lib = ol.load_oracle()
            oa, ob = np.zeros_like(o_tl), np.zeros_like(o_tl)
            vp = C.c_void_p
            lib.orc_temporal_inv(vp(o_tl.ctypes.data), vp(o_th.ctypes.data), lw * 2, lw, lh, 10, vp(oa.ctypes.data), vp(ob.ctypes.data), lw * 2)
            assert np.array_equal(fetch(ra, lh, lw), oa) and np.array_equal(fetch(rb, lh, lw), ob)
        _compare(got, bands)


def test_gop2_layout_host_only():
    """cfb_gop2_layout_compute needs no GPU: 17 coded subbands per channel, 64-byte aligned, scratch after the coded region."""
    pkg = importlib.import_module("cineform-sdk_b200")
    with_desc = pkg.FrameDesc(1920, 1080, pkg.PIXEL_YUYV)
    g = pkg.Gop2Layout()
    assert pkg.lib().cfb_gop2_layout_compute(C.byref(with_desc), C.byref(g)) == 0
    coded = [(c, k, b) for c in range(3) for k, bs in ((5, range(4)), (4, range(1, 4)), (3, range(4)), (1, range(1, 4)), (0, range(1, 4))) for b in bs]
    assert len(coded) == 3 * 17
    for (c, k, b) in coded:
        bl = g.band[c][k][b]
        assert bl.offset % 64 == 0 and bl.pitch % 16 == 0 and bl.offset + bl.pitch * bl.height <= g.coded_bytes
    for c in range(3):
        for (k, b) in ((0, 0), (1, 0), (2, 0), (2, 1), (4, 0)):
            assert g.band[c][k][b].offset >= g.coded_bytes
    assert g.band[0][5][0].width == 1920 // 8 and g.band[1][3][0].width == 1920 // 8
    bad = pkg.FrameDesc(720, 480, pkg.PIXEL_YUYV)          # chroma level-1 band 180 wide: not a multiple of 16
    assert pkg.lib().cfb_gop2_layout_compute(C.byref(bad), C.byref(g)) != 0


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_cuda_gop2_single_call(path):
    """cfb_gop2_forward_host / cfb_gop2_inverse_host: every coded band equals the reference's two-frame encode; the
    decoded frames lie inside the dither envelope of the oracle's inverse composition."""
    pkg = importlib.import_module("cineform-sdk_b200")
    fa, fb, quant, prescale, quality, bands = _load(path)
    h, w2 = fa.shape
    desc = pkg.FrameDesc(w2 // 2, h, pkg.PIXEL_YUYV)
    gq = pkg.make_gop2_quant(quant, prescale[0][:6])
    orc, lib = ol.oracle(), ol.load_oracle()
    with pkg.Context(0) as ctx, pkg.Codec(ctx, desc, 2) as codec:
        g = codec.gop2_layout()
        coded = codec.gop2_forward_host(fa, fb, gq)
        for (c, k, b), want in sorted(bands.items()):
            if k == 2:
                continue                                    # temporal bands are device scratch, not coded
            got = codec.gop2_band_view(g, coded, c, k, b)
            assert np.array_equal(got, want), f"(channel, wavelet, band) {(c, k, b)}"
        out_a, out_b = codec.gop2_inverse_host(coded, gq, pkg.PIXEL_YUYV, fa.shape)

    def inv(bands4, c, k):
        deq = [bands4[0]] + [pu.dequantize(bands4[b], quant[c][k][b]) for b in (1, 2, 3)]
        return orc.inv_level(*deq, 2 if prescale[c][k] == 2 else 0)

    planes_a, planes_b = [], []
    vp = C.c_void_p
    for c in range(3):
        ll4 = inv([bands[(c, 5, b)] for b in range(4)], c, 5)
        tl = inv([ll4] + [bands[(c, 4, b)] for b in (1, 2, 3)], c, 4)
        th = inv([bands[(c, 3, b)] for b in range(4)], c, 3)
        la, lb = np.zeros_like(tl), np.zeros_like(tl)
        hh, ww = tl.shape
        lib.orc_temporal_inv(vp(tl.ctypes.data), vp(th.ctypes.data), ww * 2, ww, hh, 10, vp(la.ctypes.data), vp(lb.ctypes.data), ww * 2)
        planes_a.append(inv([la] + [bands[(c, 0, b)] for b in (1, 2, 3)], c, 0))
        planes_b.append(inv([lb] + [bands[(c, 1, b)] for b in (1, 2, 3)], c, 1))
    for out, planes, src in ((out_a, planes_a, fa), (out_b, planes_b, fb)):
        a, b = pu.yuyv_envelope(planes)
        assert ((out == a) | (out == b)).all()
        assert pu.psnr(out[:, 0::2], src[:, 0::2]) > 45.0


@pytest.mark.parametrize("quality", [1, 2, 3, 4, 5, 6, 4 | (1 << 17)])
@pytest.mark.parametrize("interlaced", [False, True])
def test_gop2_quant_schedule_matches_reference(request, quality, interlaced):
    """cfb_gop2_quant_for_quality == the divisors / prescale the reference's encoder really used (quantize.c:3480;
    stored in tests/golden/ref_digests.json)."""
    pkg = importlib.import_module("cineform-sdk_b200")
    w, h = 256, 64
    coded = lambda k, d: d[1:] if k in (0, 1, 4) else d            # LL of wavelets 0, 1, 4 is never coded

    def want():
        ref_lib = ol.load_ref()
        fa, fb = pu.qbist_yuy2(ref_lib, w, h, 1), pu.qbist_yuy2(ref_lib, w, h, 2)
        ref_lib.ref_set_interlaced(1 if interlaced else 0)
        try:
            _, quant, prescale = pu.ref_encode_gop2(ref_lib, fa, fb, w, h, quality)
        finally:
            ref_lib.ref_set_interlaced(0)
        return [prescale[0][:6]] + [[coded(k, quant[c][k][:2 if k == 2 else 4]) for k in range(6)] for c in range(3)]
    q = pkg.gop2_quant_for_quality(pkg.FrameDesc(w, h, pkg.PIXEL_YUYV), quality, interlaced)
    got = [[int(v) for v in q.prescale]] + [[coded(k, [int(q.divisor[c][k][b]) for b in range(2 if k == 2 else 4)])
                                             for k in range(6)] for c in range(3)]
    Golden(request).check_values(got, want, "prescale, divisors per channel and wavelet")


@needs_ref
@pytest.mark.parametrize("size,quality", [((256, 64), 4), ((704, 96), 3)])
def test_oracle_gop2_interlaced_matches_reference_encoder(size, quality):
    """Interlaced two-frame GOP: level 1 of both frames is the field transform, everything above is unchanged."""
    w, h = size
    ref_lib, orc = ol.load_ref(), ol.oracle()
    fa, fb = pu.qbist_yuy2(ref_lib, w, h, 1).copy(), pu.qbist_yuy2(ref_lib, w, h, 3).copy()
    for f in (fa, fb):
        f[1::2] = np.roll(f[1::2], 8, axis=1)
    ref_lib.ref_set_interlaced(1)
    try:
        bands, quant, prescale = pu.ref_encode_gop2(ref_lib, fa, fb, w, h, quality)
    finally:
        ref_lib.ref_set_interlaced(0)
    _, temporal, level = _oracle_blocks()
    got = pu.gop2_pyramid(lambda f, c, q: orc.fwd_fields_422(f, c, 0, q, 10, 2), temporal, level, fa, fb, quant, prescale)
    _compare(got, {k: v for k, v in bands.items() if k in got})


@pytest.mark.gpu
@pytest.mark.parametrize("interlaced", [False, True])
@pytest.mark.parametrize("size", [(256, 64), (704, 96), (1920, 1080)])
def test_cuda_gop2_vs_oracle(size, interlaced):
    """cfb_gop2_* with the restated schedule, progressive and interlaced level 1, against the oracle composition."""
    pkg = importlib.import_module("cineform-sdk_b200")
    w, h = size
    rng = np.random.default_rng(w + h + int(interlaced))
    fa = pu.synthetic_yuyv(rng, w, h, "natural")
    fb = np.roll(fa, 2, axis=0).copy()
    fb[:, 0::2] = np.clip(fb[:, 0::2].astype(np.int32) + rng.integers(-3, 4, (h, w)), 16, 235).astype(np.uint8)
    if interlaced:
        for f in (fa, fb):
            f[1::2] = np.roll(f[1::2], 8, axis=1)
    desc = pkg.FrameDesc(w, h, pkg.PIXEL_YUYV)
    gq = pkg.gop2_quant_for_quality(desc, 4, interlaced)
    quant = [[[int(gq.divisor[c][k][b]) for b in range(4)] for k in range(6)] for c in range(3)]
    prescale = [[int(v) for v in gq.prescale] + [0, 0]] * 3
    orc = ol.oracle()
    _, temporal, level = _oracle_blocks()
    level1 = (lambda f, c, q: orc.fwd_fields_422(f, c, 0, q, 10, 2)) if interlaced else (lambda f, c, q: orc.fwd_level_422(f, c, 0, q, 10, 2))
    want = pu.gop2_pyramid(level1, temporal, level, fa, fb, quant, prescale)
    with pkg.Context(0) as ctx, pkg.Codec(ctx, desc, 2) as codec:
        if interlaced:
            codec.set_interlaced(True)
        g = codec.gop2_layout()
        coded = codec.gop2_forward_host(fa, fb, gq)
        for (c, k, b), wv in sorted(want.items()):
            if k == 2:
                continue
            assert np.array_equal(codec.gop2_band_view(g, coded, c, k, b), wv), f"(channel, wavelet, band) {(c, k, b)}"
        out_a, out_b = codec.gop2_inverse_host(coded, gq, pkg.PIXEL_YUYV, fa.shape)
    assert pu.psnr(out_a[:, 0::2], fa[:, 0::2]) > 40.0 and pu.psnr(out_b[:, 0::2], fb[:, 0::2]) > 40.0
