"""V210 output of the final 4:2:2 inverse level: the reference renders YU64 rows and packs each component >> 6
(Codec/decoder.c:26292 -> InvertHorizontalStrip16s.c:6490 -> convert.c:13526 ConvertPlanarYUVToV210 at precision 16).  No
dither, so the chain is bit-exact: the oracle rule (v210_oracle.pack_v210_output, incl. the scalar tail's partial last
group) is pinned to the reference's real decoder on the CPU, and the CUDA path is compared with both on the GPU.  The one
field the reference fills from outside the row (v210_oracle.v210_output_tail_cb_word) is left out of the comparisons with
the reference; against the oracle every written byte is compared."""
import importlib

import numpy as np
import pytest

import oracle_lib as ol
import parity_util as pu
import v210_oracle as vo

needs_ref = pytest.mark.skipif(not ol.ref_available(), reason="oracle/_ref not built (reference absent)")
DECODED_FORMAT_V210, DECODED_FORMAT_YU64 = 10, 12
GUARD = 0xA5C3E10F
GUARD_ROWS = 16


@pytest.fixture(scope="module")
def pkg():
    return importlib.import_module("cineform-sdk_b200")


def sdk_v210_pitch(w):
    """The SDK's V210 frame pitch, rows rounded up to 128 bytes (DecoderSDK/SampleDecoder.cpp:367 V210FramePitch)."""
    return (w + 47) // 48 * 128


def v210_words(w):
    return (w + 5) // 6 * 4


def tail_field_mask(w, h):
    """uint32 mask of the bits that are compared with the reference (all but the Cb field it reads from outside the row)."""
    m = np.full((h, v210_words(w)), 0xFFFFFFFF, np.uint32)
    k = vo.v210_output_tail_cb_word(w)
    if k is not None:
        m[:, k] = 0x000FFFFF
    return m


def _sample_422(ref_lib, w, h, kind):
    rng = np.random.default_rng(w + len(kind))
    frame = pu.qbist_yuy2(ref_lib, w, h, 2) if kind == "qbist" else pu.synthetic_yuyv(rng, w, h, kind)
    _, div, prescale, sample = pu.ref_encode_frame(ref_lib, frame, w, h, pu.COLOR_FORMAT_YUYV, 0, 3, 4)
    return sample, prescale[0]


def guarded_frame(w, h):
    """(h + GUARD_ROWS) x SDK pitch words filled with the guard; the caller decodes into the first h rows."""
    return np.full((h + GUARD_ROWS, sdk_v210_pitch(w) // 4), GUARD, np.uint32)


def check_guarded(buf, want, what=""):
    h, nw = want.shape
    got = buf[:h, :nw]
    assert np.array_equal(got, want), (what, np.argwhere(got != want)[:5].tolist())
    assert (buf[:h, nw:] == GUARD).all(), f"{what}: row padding written"
    assert (buf[h:] == GUARD).all(), f"{what}: rows after the frame written"


# ------------------------------------------------------------------------------------------------ CPU: oracle vs reference
def test_pack_v210_output_tail_rule():
    """The partial last group, spelled out for one row (widths % 6 == 2 and 4) and a full one."""
    y = np.arange(10, 10 + 16, dtype=np.int16)[None, :]
    cr = np.arange(100, 108, dtype=np.int16)[None, :]
    cb = np.arange(200, 208, dtype=np.int16)[None, :]
    word = lambda a, b, c: a | (b << 10) | (c << 20)
    out = vo.pack_v210_output([y, cr, cb])[0]
    assert out.size == 12 and vo.v210_output_tail_cb_word(16) == 10
    assert out[8:].tolist() == [word(206, 22, 106), word(23, 207, 24), word(107, 25, 207), word(25, 107, 24)]
    out = vo.pack_v210_output([y[:, :14], cr[:, :7], cb[:, :7]])[0]
    assert out.size == 12 and vo.v210_output_tail_cb_word(14) is None
    assert out[8:].tolist() == [word(206, 22, 106), word(23, 206, 22), word(106, 23, 206), word(23, 106, 22)]
    out = vo.pack_v210_output([y[:, :12], cr[:, :6], cb[:, :6]])[0]
    assert out.size == 8 and out[4:].tolist() == [word(203, 16, 103), word(17, 204, 18), word(104, 19, 205), word(20, 105, 21)]


@needs_ref
@pytest.mark.parametrize("size", [(640, 96), (208, 48), (704, 96), (720, 480), (4096, 48)])
@pytest.mark.parametrize("kind", ["qbist", "extreme"])
def test_oracle_v210_matches_reference_decoder(size, kind):
    w, h = size
    ref_lib, orc = ol.load_ref(), ol.oracle()
    sample, prescale = _sample_422(ref_lib, w, h, kind)
    pitch = sdk_v210_pitch(w)
    out, bands = pu.ref_decode_sample_raw(ref_lib, sample, w, h, DECODED_FORMAT_V210, 3, pitch)
    yu64, bands64 = pu.ref_decode_sample_raw(ref_lib, sample, w, h, DECODED_FORMAT_YU64, 3, w * 4)
    # the lowpass decode adds the same LL3 constant for V210 as for YU64 (decoder.c:12272-12275)
    for key in bands64:
        assert np.array_equal(bands[key], bands64[key]), key
    nw = v210_words(w)
    got = out[:, :nw * 4].copy().view(np.uint32)
    want = vo.pack_v210_output(pu.inverse_pyramid(orc, bands, pu.UNIT_DIVISORS, tuple(prescale)))
    assert want.shape == got.shape
    mask = tail_field_mask(w, h)
    assert np.array_equal(got & mask, want & mask), np.argwhere((got & mask) != (want & mask))[:5].tolist()
    # nothing behind the last group: the probe's zeroed buffer stays zero
    assert not out[:, nw * 4:].any()
    # the full groups are the YU64 frame >> 6
    ng = w // 6
    y16 = yu64.view(np.uint16).reshape(h, 2 * w)
    y, c1, c3 = (y16[:, 0::2] >> 6).astype(np.uint32), (y16[:, 1::4] >> 6).astype(np.uint32), (y16[:, 3::4] >> 6).astype(np.uint32)
    comp = np.zeros((h, 12 * ng), np.uint32)
    comp[:, 0::4], comp[:, 1::4], comp[:, 2::4], comp[:, 3::4] = c3[:, :3 * ng], y[:, 0:6 * ng:2], c1[:, :3 * ng], y[:, 1:6 * ng:2]
    assert np.array_equal(got[:, :4 * ng], comp[:, 0::3] | (comp[:, 1::3] << 10) | (comp[:, 2::3] << 20))
    if kind == "extreme":
        assert ((got & 1023) == 1023).any() and ((got & 1023) == 0).any()


def test_v210_pitch_helper(pkg):
    assert [pkg.v210_pitch(w) for w in (640, 704, 720, 1920, 3840)] == [1712, 1888, 1920, 5120, 10240]


# ------------------------------------------------------------------------------------------------ GPU
def _oracle_case(pkg, w, h, kind):
    rng = np.random.default_rng(w + h)
    frame = pu.synthetic_yuyv(rng, w, h, kind)
    desc = pkg.FrameDesc(w, h, pkg.PIXEL_YUYV)
    quant = pkg.quant_for_quality(desc, 4)
    orc = ol.oracle()
    coded_bands = pu.oracle_forward_422(orc, frame, quant, 0)
    want = vo.pack_v210_output(pu.inverse_pyramid(orc, coded_bands, quant.table(3), tuple(quant.prescale)))
    return desc, quant, coded_bands, want


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(256, 64), (640, 96), (704, 96), (720, 480), (1280, 720), (1920, 1080), (3840, 2160)])
@pytest.mark.parametrize("kind", ["natural", "extreme"])
def test_gpu_v210_output_vs_oracle(pkg, size, kind):
    """inverse_host (batch of 2), inverse_device and inverse_host_sparse into SDK-pitched frames with guarded padding."""
    import torch
    w, h = size
    desc, quant, coded_bands, want = _oracle_case(pkg, w, h, kind)
    pitch = sdk_v210_pitch(w)
    with pkg.Context(0) as ctx, pkg.Codec(ctx, desc, 2) as codec:
        coded = codec.pack_coded(coded_bands)
        bufs = [guarded_frame(w, h) for _ in range(2)]
        codec.inverse_host([coded, coded], quant, pkg.PIXEL_V210, [b[:h] for b in bufs])
        for i, b in enumerate(bufs):
            check_guarded(b, want, f"inverse_host[{i}]")

        d_pyr = torch.zeros(codec.layout.total_bytes, dtype=torch.uint8, device="cuda")     # + LL1 / LL2 scratch
        d_pyr[:coded.size] = torch.from_numpy(coded).cuda()
        d_frame = torch.from_numpy(guarded_frame(w, h).view(np.int32)).cuda()
        torch.cuda.synchronize()
        codec.inverse_device([d_pyr.data_ptr()], quant, pkg.PIXEL_V210, [d_frame.data_ptr()], pitch)
        ctx.synchronize()
        check_guarded(d_frame.cpu().numpy().view(np.uint32), want, "inverse_device")

        sparse = pkg.sparse_compact(codec.layout, coded)
        buf = guarded_frame(w, h)
        codec.inverse_host_sparse([sparse], quant, pkg.PIXEL_V210, [buf[:h]])
        check_guarded(buf, want, "inverse_host_sparse")


@pytest.mark.gpu
def test_gpu_v210_output_pool_4k(pkg):
    w, h = 3840, 2160
    desc, quant, coded_bands, want = _oracle_case(pkg, w, h, "natural")
    with pkg.Pool([0], desc, slots=2, batch=2, queue_length=8) as pool:
        coded = pkg.pack_coded(pool.layout, coded_bands)
        bufs = [guarded_frame(w, h) for _ in range(3)]
        for i, b in enumerate(bufs):
            pool.submit_inverse(i, coded, quant, pkg.PIXEL_V210, b[:h])
        assert [pool.wait() for _ in bufs] == [0, 1, 2]
    for i, b in enumerate(bufs):
        check_guarded(b, want, f"pool[{i}]")


@needs_ref
@pytest.mark.gpu
@pytest.mark.parametrize("size", [(640, 96), (1920, 1080)])
def test_gpu_v210_vs_reference_decoder(pkg, size):
    """The reference encodes and decodes a Qbist frame; our inverse, fed the bands its decoder held, reproduces its V210
    frame byte for byte (but for the field it reads from outside the row) and writes nothing past the last group."""
    w, h = size
    ref_lib = ol.load_ref()
    sample, prescale = _sample_422(ref_lib, w, h, "qbist")
    ref_out, bands = pu.ref_decode_sample_raw(ref_lib, sample, w, h, DECODED_FORMAT_V210, 3, sdk_v210_pitch(w))
    bands = {k: v for k, v in bands.items() if not (k[2] == "LL" and k[1] != 3)}
    desc = pkg.FrameDesc(w, h, pkg.PIXEL_YUYV)
    unit = pkg.make_quant(pu.UNIT_DIVISORS, prescale)
    with pkg.Context(0) as ctx, pkg.Codec(ctx, desc, 1) as codec:
        buf = guarded_frame(w, h)
        codec.inverse_host([codec.pack_coded(bands)], unit, pkg.PIXEL_V210, [buf[:h]])
    nw = v210_words(w)
    want = ref_out[:, :nw * 4].copy().view(np.uint32)
    mask = tail_field_mask(w, h)
    assert np.array_equal(buf[:h, :nw] & mask, want & mask)
    assert (buf[:h, nw:] == GUARD).all() and (buf[h:] == GUARD).all()


@pytest.mark.gpu
def test_gpu_v210_round_trip_flat(pkg):
    """A V210 source encoded and decoded to V210 at 1536x864: a flat frame comes back exactly, a textured one closely."""
    w, h = 1536, 864
    desc = pkg.FrameDesc(w, h, pkg.PIXEL_V210)
    quant = pkg.quant_for_quality(desc, 4)
    flat = pu.pack_v210(np.full((h, w), 601, np.uint32), np.full((h, w // 2), 419, np.uint32), np.full((h, w // 2), 583, np.uint32))
    rng = np.random.default_rng(864)
    textured, _ = pu.v210_from_yuyv(pu.synthetic_yuyv(rng, w, h, "natural"), rng)
    assert flat.shape[1] * 4 == sdk_v210_pitch(w) == pkg.v210_pitch(w)
    with pkg.Context(0) as ctx, pkg.Codec(ctx, desc, 1) as codec:
        for src, exact in ((flat, True), (textured, False)):
            coded = codec.forward_host([src], quant)[0]
            buf = guarded_frame(w, h)
            codec.inverse_host([coded], quant, pkg.PIXEL_V210, [buf[:h]])
            assert (buf[h:] == GUARD).all()
            got = buf[:h]
            if exact:
                assert np.array_equal(got, src)
            else:
                comps = lambda a: np.stack([(a >> s) & 1023 for s in (0, 10, 20)]).astype(np.float64)
                mse = np.mean((comps(got) - comps(src)) ** 2)
                assert 10 * np.log10(1023.0 ** 2 / mse) > 40.0


@pytest.mark.gpu
def test_gpu_v210_output_errors(pkg):
    w, h = 640, 96
    rng = np.random.default_rng(1)
    with pkg.Context(0) as ctx:
        desc444 = pkg.FrameDesc(w, h, pkg.PIXEL_RG48)
        with pkg.Codec(ctx, desc444, 1) as codec:
            coded = codec.forward_host([pu.synthetic_rg48(rng, w, h)], pkg.quant_for_quality(desc444, 4))[0]
            with pytest.raises(pkg.CfbError) as ei:
                codec.inverse_host([coded], pkg.quant_for_quality(desc444, 4), pkg.PIXEL_V210, [guarded_frame(w, h)[:h]])
            assert ei.value.code == 3       # BADFORMAT
        desc = pkg.FrameDesc(w, h, pkg.PIXEL_YUYV)
        frame = pu.synthetic_yuyv(rng, w, h)
        with pkg.Codec(ctx, desc, 1) as codec:
            quant = pkg.quant_for_quality(desc, 4)
            coded = codec.forward_host([frame], quant)[0]
            with pytest.raises(pkg.CfbError) as ei:        # pitch one group short
                codec.inverse_host([coded], quant, pkg.PIXEL_V210, [np.zeros((h, pkg.v210_pitch(w) // 4 - 4), np.uint32)])
            assert ei.value.code == 1       # INVALID_ARGUMENT
            d_coded = codec.device_pyramid(0)
            with pytest.raises(pkg.CfbError) as ei:        # not a multiple of 16
                codec.inverse_device([d_coded], quant, pkg.PIXEL_V210, [codec.device_frame(0)], pkg.v210_pitch(w) + 8)
            assert ei.value.code == 1
            codec.set_decode_resolution(pkg.RESOLUTION_HALF)
            with pytest.raises(pkg.CfbError) as ei:
                codec.inverse_host([coded], quant, pkg.PIXEL_V210, [guarded_frame(w, h)[:h]])
            assert ei.value.code == 102     # UNSUPPORTED
            codec.set_decode_resolution(pkg.RESOLUTION_FULL)
        iquant = pkg.quant_for_quality(desc, 4, interlaced=True)
        with pkg.Codec(ctx, desc, 1) as codec:
            codec.set_interlaced(True)
            coded = codec.forward_host([frame], iquant)[0]
            with pytest.raises(pkg.CfbError) as ei:
                codec.inverse_host([coded], iquant, pkg.PIXEL_V210, [guarded_frame(w, h)[:h]])
            assert ei.value.code == 102
