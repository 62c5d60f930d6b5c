"""Pin the oracle (oracle/cfhd_oracle.c) against the unmodified reference built in
place (oracle/_ref/libcfhd_ref.so): every restated function must agree bit for bit,
both on natural-range data and on adversarial data that drives intermediates out
of int16 (where the reference's SSE2 / scalar column split becomes visible).
Without oracle/_ref the reference's results come from tests/golden/ref_digests.json."""
import numpy as np
import pytest

import oracle_lib as ol
from ref_golden import Golden


@pytest.fixture(scope="module")
def impls():
    return ol.oracle(), (ol.ref() if ol.ref_available() else None)


def _rows(rng, width, kind):
    if kind == "natural10":
        return rng.integers(0, 1021, width).astype(np.int16)
    if kind == "natural12":
        return rng.integers(0, 4096, width).astype(np.int16)
    if kind == "full":
        return rng.integers(-32768, 32768, width).astype(np.int16)
    if kind == "checker":
        x = np.empty(width, np.int16)
        x[0::2], x[1::2] = 32767, -32768
        return x
    if kind == "checker2":
        x = np.empty(width, np.int16)
        x[0::4], x[1::4], x[2::4], x[3::4] = 32767, 32767, -32768, -32768
        return x
    raise ValueError(kind)


@pytest.mark.parametrize("width", [18, 32, 34, 48, 50, 64, 100, 240, 480, 482, 960, 1920])
@pytest.mark.parametrize("prescale", [0, 2])
@pytest.mark.parametrize("kind", ["natural10", "natural12", "full", "checker", "checker2"])
def test_fwd_row(impls, request, width, prescale, kind):
    orc, ref = impls
    rng = np.random.default_rng(width * 7 + prescale)
    x = _rows(rng, width, kind)
    Golden(request).check(orc.fwd_row(x, prescale), lambda: ref.fwd_row(x, prescale))


@pytest.mark.parametrize("divisor", [1, 2, 3, 6, 12, 24, 36, 48, 96, 144, 192, 288, 1000])
@pytest.mark.parametrize("midpoint", [2, 3, 5, 9])
def test_quantize_row(impls, request, divisor, midpoint):
    orc, ref = impls
    rng = np.random.default_rng(divisor)
    g = Golden(request)
    for n in (8, 13, 64, 251):
        x = rng.integers(-32768, 32768, n).astype(np.int16)
        x[:4] = [-32768, 32767, 0, -1]
        g.check([orc.quantize_row(x, divisor, midpoint)], lambda: [ref.quantize_row(x, divisor, midpoint)], f"n {n}")


def _plane(rng, h, w, kind):
    if kind == "natural12":
        return rng.integers(0, 4096, (h, w)).astype(np.int16)
    if kind == "natural14":
        return rng.integers(0, 16381, (h, w)).astype(np.int16)
    if kind == "full":
        return rng.integers(-32768, 32768, (h, w)).astype(np.int16)
    if kind == "checker":
        p = np.zeros((h, w), np.int16)
        yy, xx = np.mgrid[0:h, 0:w]
        p[:] = np.where(((yy // 2) + (xx // 2)) % 2 == 0, 4095, 0)
        return p
    if kind == "checker_full":
        yy, xx = np.mgrid[0:h, 0:w]
        return np.where((yy + xx) % 2 == 0, 32767, -32768).astype(np.int16)
    raise ValueError(kind)


@pytest.mark.parametrize("shape", [(16, 32), (18, 36), (32, 64), (24, 100), (64, 240), (40, 482)])
@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("kind", ["natural12", "natural14", "full", "checker", "checker_full"])
def test_fwd_level(impls, request, shape, variant, kind):
    orc, ref = impls
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    plane = _plane(rng, shape[0], shape[1], kind)
    g = Golden(request)
    for quant in ([1, 24, 24, 36], [1, 6, 6, 3], [4, 96, 96, 144]):
        g.check(orc.fwd_level(plane, variant, quant), lambda: ref.fwd_level(plane, variant, quant), f"bands, quant {quant}")


# the reference asserts unless the packed row is a multiple of 32 bytes per chroma pass (convert.c:5168),
# i.e. frame width % 16 == 0
@pytest.mark.parametrize("shape", [(16, 64), (32, 128), (24, 208), (64, 480)])
@pytest.mark.parametrize("fmt", [0, 1])
def test_fwd_level_422(impls, request, shape, fmt):
    orc, ref = impls
    g = Golden(request)
    h, w = shape
    rng = np.random.default_rng(h * w)
    for kind in ("random", "extreme"):
        if kind == "random":
            frame = rng.integers(0, 256, (h, w * 2)).astype(np.uint8)
        else:
            frame = np.where(rng.integers(0, 2, (h, w * 2)) == 0, 0, 255).astype(np.uint8)
        for channel, quant in ((0, [1, 24, 24, 36]), (1, [1, 24, 24, 48]), (2, [1, 24, 24, 48])):
            g.check(orc.fwd_level_422(frame, channel, fmt, quant), lambda: ref.fwd_level_422(frame, channel, fmt, quant),
                    f"{kind} ch {channel} bands")


@pytest.mark.parametrize("shape", [(8, 16), (9, 17), (16, 24), (12, 40), (30, 120), (17, 241)])
@pytest.mark.parametrize("descale", [0, 2])
@pytest.mark.parametrize("kind", ["natural", "large", "full"])
def test_inv_level(impls, request, shape, descale, kind):
    orc, ref = impls
    h, w = shape
    rng = np.random.default_rng(h * 977 + w)
    if kind == "natural":
        ll = rng.integers(0, 16381, (h, w)).astype(np.int16)
        hi = [rng.integers(-600, 601, (h, w)).astype(np.int16) for _ in range(3)]
    elif kind == "large":
        ll = rng.integers(-20000, 20001, (h, w)).astype(np.int16)
        hi = [rng.integers(-20000, 20001, (h, w)).astype(np.int16) for _ in range(3)]
    else:
        ll = rng.integers(-32768, 32768, (h, w)).astype(np.int16)
        hi = [rng.integers(-32768, 32768, (h, w)).astype(np.int16) for _ in range(3)]
    Golden(request).check([orc.inv_level(ll, hi[0], hi[1], hi[2], descale)],
                          lambda: [ref.inv_level(ll, hi[0], hi[1], hi[2], descale)], "inverse level, mismatches as (row, col)")
