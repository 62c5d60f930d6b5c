"""Two-frame GOP building block: temporal Haar between two int16 planes (Codec/temporal.c:498 FilterTemporal16s,
:9402 InvertTemporalQuant16s).  CPU: oracle vs the reference functions themselves (oracle/_ref, or their results stored
in tests/golden/ref_digests.json).  GPU: CUDA vs oracle."""
import ctypes as C
import importlib

import numpy as np
import pytest

import oracle_lib as ol
from ref_golden import Golden

SHAPES = [(16, 4), (48, 6), (80, 5), (96, 7), (1920, 8), (960, 540)]


def _planes(rng, w, h, kind):
    lim = 32768 if kind == "full" else 4096
    return (rng.integers(-lim, lim, (h, w)).astype(np.int16), rng.integers(-lim, lim, (h, w)).astype(np.int16))


def _run(lib, prefix, a, b):
    h, w = a.shape
    vp = C.c_void_p
    out = []
    lo, hi = np.zeros_like(a), np.zeros_like(a)
    getattr(lib, prefix + "temporal_fwd")(vp(a.ctypes.data), vp(b.ctypes.data), w * 2, w, h, vp(lo.ctypes.data), vp(hi.ctypes.data), w * 2)
    out += [lo, hi]
    for precision in (8, 10):
        x, y = np.zeros_like(a), np.zeros_like(a)
        getattr(lib, prefix + "temporal_inv")(vp(a.ctypes.data), vp(b.ctypes.data), w * 2, w, h, precision,
                                              vp(x.ctypes.data), vp(y.ctypes.data), w * 2)
        out += [x, y]
    return out


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("kind", ["small", "full"])
def test_oracle_temporal_matches_reference(request, shape, kind):
    """Saturating SSE2 body, int scalar tail (width % 40) and the precision-8 half-tone quirk, full int16 range."""
    w, h = shape
    a, b = _planes(np.random.default_rng(w + h), w, h, kind)
    Golden(request).check(_run(ol.load_oracle(), "orc_", a, b), lambda: _run(ol.load_ref(), "ref_", a, b))


def test_oracle_temporal_roundtrip():
    """In-range data: inverse(forward(a, b)) == (a, b) exactly (low +- high is even)."""
    a, b = _planes(np.random.default_rng(3), 96, 9, "small")
    lib = ol.load_oracle()
    vp = C.c_void_p
    lo, hi, x, y = (np.zeros_like(a) for _ in range(4))
    lib.orc_temporal_fwd(vp(a.ctypes.data), vp(b.ctypes.data), 192, 96, 9, vp(lo.ctypes.data), vp(hi.ctypes.data), 192)
    lib.orc_temporal_inv(vp(lo.ctypes.data), vp(hi.ctypes.data), 192, 96, 9, 10, vp(x.ctypes.data), vp(y.ctypes.data), 192)
    assert np.array_equal(x, a) and np.array_equal(y, b)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES + [(3840 // 2, 2160 // 2)])
@pytest.mark.parametrize("kind", ["small", "full"])
def test_cuda_temporal_matches_oracle(shape, kind):
    pkg = importlib.import_module("cineform-sdk_b200")
    w, h = shape
    a, b = _planes(np.random.default_rng(w * 3 + h), w, h, kind)
    want = _run(ol.load_oracle(), "orc_", a, b)
    with pkg.Context(0) as ctx:
        got = list(ctx.temporal_forward(a, b))
        for precision in (8, 10):
            got += list(ctx.temporal_inverse(a, b, precision))
    for g, w_ in zip(got, want):
        assert np.array_equal(g, w_)


@pytest.mark.gpu
def test_cuda_temporal_rejects_bad_width():
    pkg = importlib.import_module("cineform-sdk_b200")
    with pkg.Context(0) as ctx:
        with pytest.raises(pkg.CfbError):
            ctx.temporal_forward(np.zeros((4, 24), np.int16), np.zeros((4, 24), np.int16))
