"""CPU-side gates: (1) the oracle composed into a 3-level pyramid reproduces what the reference's real
EncodeSample leaves in transform[c]->wavelet[k]->band[b] for Qbist frames (the known-answer this repo
pins parity on, SURVEY 8c); (2) the product library's host-side tables (layout, quantisation schedule)
match the reference; (3) the C-ABI library loads and exports every declared symbol."""
import importlib
import os
import re

import numpy as np
import pytest

import oracle_lib as ol
import parity_util as pu
from ref_golden import Golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_ref = pytest.mark.skipif(not ol.ref_available(), reason="oracle/_ref not built (reference absent)")


@pytest.fixture(scope="module")
def pkg():
    return importlib.import_module("cineform-sdk_b200")


@needs_ref
@pytest.mark.parametrize("size,frame_no", [((256, 64), 1), ((512, 128), 3), ((1920, 1080), 1),
                                           ((720, 480), 1), ((1440, 1080), 2), ((208, 48), 1), ((400, 56), 1)])     # ragged band widths
def test_oracle_pyramid_matches_reference_encoder(size, frame_no):
    w, h = size
    ref_lib = ol.load_ref()
    frame = pu.qbist_yuy2(ref_lib, w, h, frame_no)
    bands_ref, div, prescale, sample = pu.ref_encode_frame(ref_lib, frame, w, h, pu.COLOR_FORMAT_YUYV, 0, 3, 4)
    assert prescale[0] == [0, 2, 0]
    assert div[0] == [[1, 24, 24, 36], [1, 6, 6, 3], [1, 24, 24, 12]]          # BASELINE.md, FS1 luma
    assert div[1] == [[1, 24, 24, 48], [1, 6, 6, 3], [1, 24, 24, 12]]
    pyr = pu.forward_pyramid_422(ol.oracle(), frame, div, tuple(prescale[0]), fmt=0)
    for key, want in bands_ref.items():
        assert np.array_equal(pyr[key], want), f"band {key}"


@needs_ref
def test_known_answer_sample_size():
    """TestCFHD -D, 1920x1080 YUY2 FS1 frame 1 encodes to ~592 268 bytes (BASELINE.md 2; metadata varies by ~100 B)."""
    ref_lib = ol.load_ref()
    frame = pu.qbist_yuy2(ref_lib, 1920, 1080, 1)
    _, _, _, sample = pu.ref_encode_frame(ref_lib, frame, 1920, 1080, pu.COLOR_FORMAT_YUYV, 0, 3, 4)
    assert abs(sample.size - 592268) < 2048


@pytest.mark.parametrize("quality", [1, 2, 3, 4, 5, 6, 4 | (1 << 17), 4 | (3 << 17)])
def test_quant_schedule_matches_reference(pkg, request, quality):
    """Divisors and prescale of the reference's EncodeSample (a Qbist frame; stored in tests/golden/ref_digests.json)."""
    w, h = 256, 64

    def want():
        ref_lib = ol.load_ref()
        frame = pu.qbist_yuy2(ref_lib, w, h, 1)
        _, div, prescale, _ = pu.ref_encode_frame(ref_lib, frame, w, h, pu.COLOR_FORMAT_YUYV, 0, 3, quality)
        return [div, prescale[0]]
    q = pkg.quant_for_quality(pkg.FrameDesc(w, h, pkg.PIXEL_YUYV), quality)
    Golden(request).check_values([q.table(3), list(q.prescale)], want, "divisors, prescale")


@pytest.mark.parametrize("quality", [1, 2, 3, 4, 5, 6, 4 | (1 << 17)])
def test_interlaced_quant_schedule_matches_reference(pkg, request, quality):
    """parameters.progressive = 0 (CFHD_ENCODING_FLAGS_YUV_INTERLACED): quantize.c:490-541 rescales level 1."""
    w, h = 256, 64

    def want():
        ref_lib = ol.load_ref()
        frame = pu.qbist_yuy2(ref_lib, w, h, 1)
        ref_lib.ref_set_interlaced(1)
        try:
            _, div, prescale, _ = pu.ref_encode_frame(ref_lib, frame, w, h, pu.COLOR_FORMAT_YUYV, 0, 3, quality)
        finally:
            ref_lib.ref_set_interlaced(0)
        return [div, prescale[0]]
    q = pkg.quant_for_quality(pkg.FrameDesc(w, h, pkg.PIXEL_YUYV), quality, interlaced=True)
    Golden(request).check_values([q.table(3), list(q.prescale)], want, "divisors, prescale")


@needs_ref
@pytest.mark.parametrize("size,quality,kind", [((640, 368), 4, "qbist"), ((256, 64), 3, "natural"), ((1920, 1080), 4, "qbist"),
                                               ((320, 56), 1, "natural"), ((704, 96), 5, "random"), ((192, 48), 6, "random")])
def test_oracle_field_transform_matches_reference_codec(size, quality, kind):
    """Interlaced source through the reference's real encoder and decoder: the oracle's field transform reproduces
    every band EncodeSample left behind (natural content; for full-range noise the entropy coder rewrites band values
    in place, so the check goes through the sample instead: what the reference's DECODER recovered from the bitstream
    must equal the oracle's bands, dequantised and with HL integrated), and the oracle's inverse of the decoder's
    bands lies inside the dither envelope of the frame the decoder produced."""
    w, h = size
    ref_lib, orc = ol.load_ref(), ol.oracle()
    rng = np.random.default_rng(w * 7 + h)
    if kind == "qbist":
        frame = pu.qbist_yuy2(ref_lib, w, h).copy()
        frame[1::2] = np.roll(frame[1::2], 12, axis=1)
    else:
        frame = pu.synthetic_yuyv(rng, w, h, kind)
    ref_lib.ref_set_interlaced(1)
    try:
        bands_ref, div, prescale, sample = pu.ref_encode_frame(ref_lib, frame, w, h, pu.COLOR_FORMAT_YUYV, 0, 3, quality)
    finally:
        ref_lib.ref_set_interlaced(0)
    pyr = pu.forward_pyramid_422(orc, frame, div, tuple(prescale[0]), fmt=0, interlaced=True)
    if kind != "random":
        for key, want in bands_ref.items():
            if not (key[2] == "LL" and key[1] != 3):
                assert np.array_equal(pyr[key], want), f"band {key}"
    _, db = pu.ref_decode_sample_bands(ref_lib, sample, w, h)        # Codec-level decode: the decoder's own bands
    for c in range(3):
        hl = np.cumsum(pyr[(c, 1, "HL")].astype(np.int64), axis=1) * div[c][0][2]
        assert np.array_equal(db[(c, 1, "HL")], hl.astype(np.int16)), f"channel {c}: decoder HL != integrated oracle HL"
    coded = {k: v.copy() for k, v in db.items() if not (k[2] == "LL" and k[1] != 3)}
    for c in range(3):
        hl = coded[(c, 1, "HL")].astype(np.int32)
        hl[:, 1:] -= hl[:, :-1].copy()
        coded[(c, 1, "HL")] = hl.astype(np.int16)
    planes = pu.inverse_pyramid(orc, coded, pu.UNIT_DIVISORS, tuple(prescale[0]), interlaced=True)
    a, b = pu.yuyv_envelope(planes)
    # The picture comes from the public API (CFHD_DecodeSample).  The reference's threaded decoder occasionally returns
    # an interlaced frame whose last chroma rows are not finished yet (its output conversion can overtake a transform
    # worker; roughly 1 decode in 8 at 1080p on this host) -- the reference's race, not the transform's: decode again.
    import ctypes as C
    for attempt in range(5):
        dec = np.zeros_like(frame)
        rc = ref_lib.ref_decode_sample(sample.ctypes.data_as(C.c_void_p), C.c_int64(sample.size), w, h,
                                       ol.CFHD_PIXEL_FORMAT_YUY2, dec.ctypes.data_as(C.c_void_p), w * 2)
        assert rc == 0
        bad = np.argwhere(~((dec == a) | (dec == b)))
        if len(bad) == 0:
            break
    # (a second, rarer artefact of the reference: the first 8 chroma bytes of a row come out as stale memory; tolerate a
    # handful of bytes -- a transform error would put thousands outside)
    assert len(bad) <= 64, (f"{len(bad)} bytes outside the dither envelope in 5 decodes, first at {bad[0].tolist()}: decoded "
                            f"{dec[tuple(bad[0])]}, envelope {a[tuple(bad[0])]}..{b[tuple(bad[0])]}")


def test_layout_rules(pkg):
    lay = pkg.layout_for(pkg.FrameDesc(3840, 2160, pkg.PIXEL_YUYV))
    assert lay.num_channels == 3 and lay.precision == 10
    y1 = lay.band[0][0][1]
    assert (y1.width, y1.height, y1.pitch) == (1920, 1080, 3840)
    c3 = lay.band[1][2][0]
    assert (c3.width, c3.height, c3.pitch) == (240, 270, 480)
    # coded region = exactly one int16 per plane pixel for these (pitch == 2*width) sizes, 64-byte aligned bands
    assert lay.coded_bytes >= 2 * 3840 * 2160 * 2 and lay.coded_bytes < 2 * 3840 * 2160 * 2 + 64 * 30
    offs = []
    for c in range(3):
        for k in range(3):
            for b in range(4):
                bl = lay.band[c][k][b]
                assert bl.offset % 64 == 0 and bl.pitch % 16 == 0 and bl.pitch >= 2 * bl.width
                offs.append((bl.offset, bl.offset + bl.pitch * bl.height))
    offs.sort()
    for (a0, a1), (b0, b1) in zip(offs, offs[1:]):
        assert a1 <= b0, "bands overlap"
    assert offs[-1][1] <= lay.total_bytes
    with pytest.raises(pkg.CfbError):
        pkg.layout_for(pkg.FrameDesc(100, 64, pkg.PIXEL_YUYV))


def test_abi_exports_every_declared_symbol(pkg):
    hdr = open(os.path.join(ROOT, "include", "cfhd_b200.h")).read()
    names = set(re.findall(r"CFB_API\s+[\w\s\*]+?\b(cfb_\w+)\s*\(", hdr))
    assert len(names) >= 15
    lib = pkg.lib()
    for n in sorted(names):
        assert hasattr(lib, n), f"{n} declared in include/cfhd_b200.h but not exported"
    assert lib.cfb_version() >= 100


def test_no_cpu_fallback_without_device(pkg):
    """On a box without a GPU the transform entry points must fail loudly (never compute on the host)."""
    if pkg.device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(pkg.CfbError) as ei:
        pkg.Context(0)
    assert ei.value.code == 100


def test_product_does_not_depend_on_the_checker():
    """oracle/ and tests/ are test infrastructure: the shipped library must not link against them and neither the package
    nor bench.py's product arm may import them (bench.py may, inside its CPU-baseline / --impl reference leg only)."""
    import subprocess
    lib = os.path.join(ROOT, "cineform-sdk_b200", "libcfhd_b200.so")
    needed = subprocess.run(["readelf", "-d", lib], capture_output=True, text=True).stdout
    assert "oracle" not in needed and "cfhd_ref" not in needed and "CFHDCodec" not in needed
    pkg_src = open(os.path.join(ROOT, "cineform-sdk_b200", "__init__.py")).read()
    assert "oracle" not in pkg_src and "parity_util" not in pkg_src
    for name in sorted(os.listdir(os.path.join(ROOT, "cineform-sdk_b200", "csrc"))):
        if not name.endswith((".cu", ".cuh", ".h")):
            continue
        src = open(os.path.join(ROOT, "cineform-sdk_b200", "csrc", name)).read()
        assert "oracle/" not in src and "cfhd_oracle" not in src, name
    bench_src = open(os.path.join(ROOT, "bench.py")).read()
    # the only function of bench.py that imports the checker is the CPU baseline / reference-arm timer
    importing = [seg.split("(")[0] for seg in bench_src.split("\ndef ")[1:] if "import oracle_lib" in seg or "import parity_util" in seg]
    assert importing == ["cpu_reference_run"], importing
