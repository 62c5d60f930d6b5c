"""cineform-sdk_b200 -- host-side mirror (ctypes) of the C ABI in include/cfhd_b200.h.

The product is the native library ``libcfhd_b200.so`` (CUDA kernels for sm_100a +
C-ABI); this module only marshals numpy buffers into it for tests and bench.py.
There is no Python or CPU implementation of the transform here: if the native
library is missing or no B200 is present, calls fail loudly.

Import with ``importlib.import_module("cineform-sdk_b200")`` (the directory name
follows the reference repo's name and is not a Python identifier).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcfhd_b200.so")

PIXEL_YUYV, PIXEL_UYVY, PIXEL_RG48, PIXEL_BYR4, PIXEL_PLANAR16, PIXEL_YU64, PIXEL_V210 = 0, 1, 2, 3, 4, 5, 6
PIXEL_RG30, PIXEL_AB10, PIXEL_AR10, PIXEL_R210, PIXEL_DPX0 = 7, 8, 9, 10, 11
PIXEL_B64A = 12     # output only: 16-bit A,R,G,B from an RGB 4:4:4 codec
RESOLUTION_FULL, RESOLUTION_HALF, RESOLUTION_QUARTER = 1, 2, 3
MAX_CHANNELS, NUM_LEVELS, NUM_BANDS, MAX_BATCH = 4, 3, 4, 16
BAND_NAMES = ("LL", "LH", "HL", "HH")

OK = 0
ERROR_NAMES = {0: "OK", 1: "INVALID_ARGUMENT", 2: "OUTOFMEMORY", 3: "BADFORMAT", 10: "UNEXPECTED", 13: "NOT_FINISHED",
               100: "NO_DEVICE", 101: "CUDA", 102: "UNSUPPORTED", 103: "RANGE"}


class CfbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"cfb error {code} ({ERROR_NAMES.get(code, '?')}): {msg}")
        self.code = code


class FrameDesc(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("pixel_format", C.c_int32), ("reserved", C.c_int32)]

    def __init__(self, width=0, height=0, pixel_format=0):
        super().__init__(width, height, pixel_format, 0)


class BandLayout(C.Structure):
    _fields_ = [("offset", C.c_int64), ("width", C.c_int32), ("height", C.c_int32), ("pitch", C.c_int32),
                ("reserved", C.c_int32)]


class Layout(C.Structure):
    _fields_ = [("num_channels", C.c_int32), ("precision", C.c_int32), ("coded_bytes", C.c_int64),
                ("total_bytes", C.c_int64), ("frame_bytes", C.c_int64), ("frame_pitch", C.c_int32),
                ("reserved", C.c_int32), ("band", BandLayout * NUM_BANDS * NUM_LEVELS * MAX_CHANNELS)]


class Quant(C.Structure):
    _fields_ = [("prescale", C.c_int32 * NUM_LEVELS), ("midpoint_prequant", C.c_int32),
                ("divisor", C.c_int32 * NUM_BANDS * NUM_LEVELS * MAX_CHANNELS)]

    def table(self, nchan=3):
        return [[[self.divisor[c][k][b] for b in range(4)] for k in range(3)] for c in range(nchan)]


GOP2_WAVELETS = 6


class Gop2Layout(C.Structure):
    _fields_ = [("num_channels", C.c_int32), ("reserved", C.c_int32), ("coded_bytes", C.c_int64), ("total_bytes", C.c_int64),
                ("band", BandLayout * NUM_BANDS * GOP2_WAVELETS * MAX_CHANNELS)]


class Gop2Quant(C.Structure):
    _fields_ = [("midpoint_prequant", C.c_int32), ("prescale", C.c_int32 * GOP2_WAVELETS), ("reserved", C.c_int32),
                ("divisor", C.c_int32 * NUM_BANDS * GOP2_WAVELETS * MAX_CHANNELS)]


class LevelDesc(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("plane_pitch", C.c_int32), ("band_pitch", C.c_int32),
                ("prescale", C.c_int32), ("midpoint_prequant", C.c_int32), ("divisor", C.c_int32 * 4)]


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("frames_forward", C.c_uint64), ("frames_inverse", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]


_lib = None


def lib():
    """Load the native library (built in-tree by __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python __graft_entry__.py` (nvcc, sm_100a) first; "
                          "there is no Python/CPU fallback for the transform path")
    L = C.CDLL(LIB_PATH)
    vp, i = C.c_void_p, C.c_int
    L.cfb_version.restype = i
    L.cfb_last_error_string.restype = C.c_char_p
    L.cfb_device_count.restype = i
    L.cfb_device_numa_node.argtypes = [i]
    L.cfb_bind_thread_to_device.argtypes = [i]
    L.cfb_context_create.argtypes = [i, C.POINTER(vp)]
    L.cfb_context_destroy.argtypes = [vp]
    L.cfb_context_destroy.restype = None
    L.cfb_context_synchronize.argtypes = [vp]
    L.cfb_context_stream.argtypes = [vp]
    L.cfb_context_stream.restype = vp
    L.cfb_context_stats.argtypes = [vp, C.POINTER(Stats)]
    L.cfb_layout_compute.argtypes = [C.POINTER(FrameDesc), C.POINTER(Layout)]
    L.cfb_quant_for_quality.argtypes = [C.POINTER(FrameDesc), i, C.POINTER(Quant)]
    L.cfb_codec_create.argtypes = [vp, C.POINTER(FrameDesc), i, C.POINTER(vp)]
    L.cfb_codec_destroy.argtypes = [vp]
    L.cfb_codec_destroy.restype = None
    L.cfb_codec_layout.argtypes = [vp, C.POINTER(Layout)]
    L.cfb_codec_device_frame.argtypes = [vp, i]
    L.cfb_codec_device_frame.restype = vp
    L.cfb_codec_device_pyramid.argtypes = [vp, i]
    L.cfb_codec_device_pyramid.restype = vp
    L.cfb_codec_set_level_mask.argtypes = [vp, i, i]
    L.cfb_codec_set_bayer_phase.argtypes = [vp, i]
    L.cfb_codec_set_bayer_curve.argtypes = [vp, vp, i]
    L.cfb_codec_set_decode_resolution.argtypes = [vp, i]
    L.cfb_codec_set_interlaced.argtypes = [vp, i]
    L.cfb_gop2_layout_compute.argtypes = [C.POINTER(FrameDesc), C.POINTER(Gop2Layout)]
    L.cfb_gop2_quant_for_quality.argtypes = [C.POINTER(FrameDesc), i, i, C.POINTER(Gop2Quant)]
    L.cfb_gop2_forward_host.argtypes = [vp, vp, vp, i, C.POINTER(Gop2Quant), vp]
    L.cfb_gop2_inverse_host.argtypes = [vp, vp, C.POINTER(Gop2Quant), i, vp, vp, i]
    L.cfb_context_range_status.argtypes = [vp, C.POINTER(C.c_int)]
    L.cfb_level_forward_device.argtypes = [vp, C.POINTER(LevelDesc), vp, C.POINTER(vp)]
    L.cfb_level_inverse_device.argtypes = [vp, C.POINTER(LevelDesc), C.POINTER(vp), vp]
    L.cfb_level_forward_host.argtypes = [vp, C.POINTER(LevelDesc), vp, C.POINTER(vp)]
    L.cfb_level_inverse_host.argtypes = [vp, C.POINTER(LevelDesc), C.POINTER(vp), vp]
    L.cfb_temporal_forward_device.argtypes = [vp, vp, vp, i, vp, vp, i, i, i]
    L.cfb_temporal_inverse_device.argtypes = [vp, vp, vp, i, vp, vp, i, i, i, i]
    L.cfb_temporal_forward_host.argtypes = [vp, vp, vp, i, vp, vp, i, i, i]
    L.cfb_temporal_inverse_host.argtypes = [vp, vp, vp, i, vp, vp, i, i, i, i]
    L.cfb_quant_for_source.argtypes = [C.POINTER(FrameDesc), i, i, C.POINTER(Quant)]
    L.cfb_codec_decoded_size.argtypes = [vp, C.POINTER(i), C.POINTER(i)]
    L.cfb_pool_set_decode_resolution.argtypes = [vp, i]
    L.cfb_pool_set_interlaced.argtypes = [vp, i]
    L.cfb_forward_device.argtypes = [vp, i, C.POINTER(vp), i, C.POINTER(Quant), C.POINTER(vp)]
    L.cfb_forward_host.argtypes = [vp, i, C.POINTER(vp), i, C.POINTER(Quant), C.POINTER(vp)]
    L.cfb_inverse_device.argtypes = [vp, i, C.POINTER(vp), C.POINTER(Quant), i, C.POINTER(vp), i]
    L.cfb_inverse_host.argtypes = [vp, i, C.POINTER(vp), C.POINTER(Quant), i, C.POINTER(vp), i]
    L.cfb_sparse_max_bytes.argtypes = [C.POINTER(Layout)]
    L.cfb_sparse_max_bytes.restype = C.c_size_t
    L.cfb_sparse_bytes.argtypes = [vp]
    L.cfb_sparse_bytes.restype = C.c_size_t
    L.cfb_forward_host_sparse.argtypes = [vp, i, C.POINTER(vp), i, C.POINTER(Quant), C.POINTER(vp), C.POINTER(C.c_size_t)]
    L.cfb_inverse_host_sparse.argtypes = [vp, i, C.POINTER(vp), C.POINTER(Quant), i, C.POINTER(vp), i]
    L.cfb_sparse_expand.argtypes = [C.POINTER(Layout), vp, vp]
    L.cfb_sparse_compact.argtypes = [C.POINTER(Layout), vp, vp, C.POINTER(C.c_size_t)]
    L.cfb_sparse_compact_bands.argtypes = [C.POINTER(Layout), C.POINTER(vp), C.POINTER(C.c_int32), vp, C.POINTER(C.c_size_t)]
    L.cfb_sparse_writer_create.argtypes = [C.POINTER(Layout), C.POINTER(vp)]
    L.cfb_sparse_writer_destroy.argtypes = [vp]
    L.cfb_sparse_writer_destroy.restype = None
    L.cfb_sparse_writer_begin.argtypes = [vp, vp, C.c_size_t]
    L.cfb_sparse_writer_band.argtypes = [vp, i, i, i]
    L.cfb_sparse_writer_run.argtypes = [vp, C.c_uint32]
    L.cfb_sparse_writer_value.argtypes = [vp, i]
    L.cfb_sparse_writer_dense_band.argtypes = [vp, i, i, i, vp, i]
    L.cfb_sparse_writer_end.argtypes = [vp, C.POINTER(C.c_size_t)]
    L.cfb_vlc_decoder_create.argtypes = [C.POINTER(VlcDecodebook), C.POINTER(vp)]
    L.cfb_vlc_decoder_destroy.argtypes = [vp]
    L.cfb_vlc_decoder_destroy.restype = None
    L.cfb_vlc_decode_band.argtypes = [vp, vp, i, i, i, vp, C.c_size_t, i, C.POINTER(C.c_size_t)]
    L.cfb_sparse_vlc_band.argtypes = [C.POINTER(Layout), vp, i, i, i, C.POINTER(VlcCodebook), C.POINTER(BitWriter)]
    L.cfb_dense_vlc_band.argtypes = [vp, i, i, i, C.POINTER(VlcCodebook), C.POINTER(BitWriter)]
    L.cfb_sparse_band_nonzeros.argtypes = [C.POINTER(Layout), vp, i, i, i, C.POINTER(C.c_uint32)]
    L.cfb_sparse_expand_band.argtypes = [C.POINTER(Layout), vp, i, i, i, vp, i]
    L.cfb_pool_submit_forward_sparse.argtypes = [vp, C.c_uint32, vp, i, C.POINTER(Quant), vp]
    L.cfb_pool_submit_inverse_sparse.argtypes = [vp, C.c_uint32, vp, C.POINTER(Quant), i, vp, i]
    L.cfb_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.cfb_host_free.argtypes = [vp]
    L.cfb_host_free.restype = None
    L.cfb_pool_create.argtypes = [C.POINTER(C.c_int), i, C.POINTER(FrameDesc), i, i, i, C.POINTER(vp)]
    L.cfb_pool_destroy.argtypes = [vp]
    L.cfb_pool_destroy.restype = None
    L.cfb_pool_submit_forward.argtypes = [vp, C.c_uint32, vp, i, C.POINTER(Quant), vp]
    L.cfb_pool_submit_inverse.argtypes = [vp, C.c_uint32, vp, C.POINTER(Quant), i, vp, i]
    L.cfb_pool_wait.argtypes = [vp, C.POINTER(C.c_uint32), C.POINTER(i)]
    L.cfb_pool_test.argtypes = [vp, C.POINTER(C.c_uint32), C.POINTER(i)]
    L.cfb_pool_stats.argtypes = [vp, C.POINTER(Stats)]
    _lib = L
    return L


def _check(code):
    if code != OK:
        raise CfbError(code, lib().cfb_last_error_string().decode("utf-8", "replace"))


def device_count():
    return lib().cfb_device_count()


def layout_for(desc):
    out = Layout()
    _check(lib().cfb_layout_compute(C.byref(desc), C.byref(out)))
    return out


def v210_pitch(width):
    """Smallest pitch of a V210 output frame: whole 6-pixel groups of 16 bytes (the inverse writes exactly this much per
    row).  The SDK's own V210 frames round the row up to 128 bytes, which the inverse accepts as well."""
    return (width + 5) // 6 * 16


def device_numa_node(device):
    return int(lib().cfb_device_numa_node(device))


def bind_thread_to_device(device):
    """Restrict the calling thread to the CPUs of the GPU's NUMA node (pinned allocations that follow are local)."""
    _check(lib().cfb_bind_thread_to_device(device))


def quant_for_quality(desc, quality, interlaced=False):
    out = Quant()
    _check(lib().cfb_quant_for_source(C.byref(desc), quality, int(bool(interlaced)), C.byref(out)))
    return out


def sparse_max_bytes(layout):
    return int(lib().cfb_sparse_max_bytes(C.byref(layout)))


def sparse_bytes(buf):
    return int(lib().cfb_sparse_bytes(buf.ctypes.data))


def sparse_expand(layout, sparse):
    """Host-side format conversion: sparse buffer -> dense coded region (uint8 array)."""
    out = np.empty(layout.coded_bytes, np.uint8)
    _check(lib().cfb_sparse_expand(C.byref(layout), sparse.ctypes.data, out.ctypes.data))
    return out


def sparse_compact(layout, dense):
    out = np.zeros(sparse_max_bytes(layout), np.uint8)
    n = C.c_size_t()
    _check(lib().cfb_sparse_compact(C.byref(layout), dense.ctypes.data, out.ctypes.data, C.byref(n)))
    return out[:n.value]


def sparse_compact_bands(layout, bands):
    """{(c, level 1..3, band name): 2-D int16 array (any row stride)} -> sparse buffer, as cfb_sparse_compact_bands."""
    n = MAX_CHANNELS * NUM_LEVELS * NUM_BANDS
    ptrs, pitches = (C.c_void_p * n)(), (C.c_int32 * n)()
    for (c, lvl, name), arr in bands.items():
        idx = (c * NUM_LEVELS + (lvl - 1)) * NUM_BANDS + BAND_NAMES.index(name)
        ptrs[idx], pitches[idx] = arr.ctypes.data, arr.strides[0]
    out = np.zeros(sparse_max_bytes(layout), np.uint8)
    nbytes = C.c_size_t()
    _check(lib().cfb_sparse_compact_bands(C.byref(layout), ptrs, pitches, out.ctypes.data, C.byref(nbytes)))
    return out[:nbytes.value]


class VlcCodebook(C.Structure):
    """cfb_vlc_codebook: the host entropy coder's run-length and value tables as plain arrays."""
    _fields_ = [("run_length", C.c_int32), ("value_length", C.c_int32), ("run_bits", C.c_void_p), ("run_size", C.c_void_p),
                ("run_count", C.c_void_p), ("value_bits", C.c_void_p), ("value_size", C.c_void_p)]

    @classmethod
    def from_arrays(cls, run_bits, run_size, run_count, value_bits, value_size):
        self = cls()
        self._keep = [np.ascontiguousarray(run_bits, np.uint32), np.ascontiguousarray(run_size, np.uint8),
                      np.ascontiguousarray(run_count, np.uint32), np.ascontiguousarray(value_bits, np.uint32),
                      np.ascontiguousarray(value_size, np.uint8)]
        self.run_length, self.value_length = len(self._keep[0]), len(self._keep[3])
        self.run_bits, self.run_size, self.run_count, self.value_bits, self.value_size = [a.ctypes.data for a in self._keep]
        return self


class VlcDecodebook(C.Structure):
    """cfb_vlc_decodebook: every code word of the band stream once -- kind 0 value, 1 zero run, 2 end of band."""
    _fields_ = [("count", C.c_int32), ("bits", C.c_void_p), ("size", C.c_void_p), ("kind", C.c_void_p), ("arg", C.c_void_p)]

    @classmethod
    def from_arrays(cls, bits, size, kind, arg):
        self = cls()
        self._keep = [np.ascontiguousarray(bits, np.uint32), np.ascontiguousarray(size, np.uint8),
                      np.ascontiguousarray(kind, np.uint8), np.ascontiguousarray(arg, np.int32)]
        self.count = len(self._keep[0])
        self.bits, self.size, self.kind, self.arg = [a.ctypes.data for a in self._keep]
        return self


class VlcDecoder:
    """Compiled code set (cfb_vlc_decoder) + a sparse writer: band bit streams -> one 'CFS2' buffer."""

    def __init__(self, layout, book):
        self.layout, self.book = layout, book
        self.d, self.w = C.c_void_p(), C.c_void_p()
        _check(lib().cfb_vlc_decoder_create(C.byref(book), C.byref(self.d)))
        _check(lib().cfb_sparse_writer_create(C.byref(layout), C.byref(self.w)))
        self.out = None

    def begin(self, out=None):
        """out: a caller-owned buffer of sparse_max_bytes(layout) to write into (a frame loop reuses one)."""
        self.out = np.zeros(sparse_max_bytes(self.layout), np.uint8) if out is None else out
        _check(lib().cfb_sparse_writer_begin(self.w, self.out.ctypes.data, self.out.size))

    def dense_band(self, c, k, b, rows):
        rows = np.ascontiguousarray(rows, np.int16)
        _check(lib().cfb_sparse_writer_dense_band(self.w, c, k, b, rows.ctypes.data, rows.strides[0]))

    def band(self, c, k, b, stream, quant):
        stream = np.ascontiguousarray(stream, np.uint8)
        used = C.c_size_t()
        _check(lib().cfb_vlc_decode_band(self.d, self.w, c, k, b, stream.ctypes.data, stream.size, quant, C.byref(used)))
        return int(used.value)

    def end(self):
        n = C.c_size_t()
        _check(lib().cfb_sparse_writer_end(self.w, C.byref(n)))
        return self.out[:n.value]

    def close(self):
        if self.d:
            lib().cfb_vlc_decoder_destroy(self.d); self.d = C.c_void_p()
        if self.w:
            lib().cfb_sparse_writer_destroy(self.w); self.w = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BitWriter(C.Structure):
    """cfb_bitwriter: the BITSTREAM fields the reference's coder reads and leaves behind."""
    _fields_ = [("cur", C.c_void_p), ("end", C.c_void_p), ("buffer", C.c_uint32), ("bits_free", C.c_int32), ("bytes", C.c_int64)]


def _bitwriter(buf, lead_bits):
    bw = BitWriter()
    bw.cur, bw.end = buf.ctypes.data, buf.ctypes.data + buf.size
    bw.buffer, bw.bits_free, bw.bytes = (1 << lead_bits) - 1, 32 - lead_bits, 0
    return bw


def sparse_vlc_band(layout, sparse, channel, level, band, book, capacity, lead_bits=0):
    """Run-length / VLC codes of one band straight from a sparse buffer -> (whole words written, pending buffer, bits free)."""
    out = np.zeros(capacity, np.uint8)
    bw = _bitwriter(out, lead_bits)
    _check(lib().cfb_sparse_vlc_band(C.byref(layout), sparse.ctypes.data, channel, level, band, C.byref(book), C.byref(bw)))
    return out[:bw.bytes].copy(), int(bw.buffer), int(bw.bits_free)


def dense_vlc_band(band, pitch_bytes, width, book, capacity, lead_bits=0):
    out = np.zeros(capacity, np.uint8)
    bw = _bitwriter(out, lead_bits)
    band = np.ascontiguousarray(band)
    _check(lib().cfb_dense_vlc_band(band.ctypes.data, width, band.shape[0], pitch_bytes, C.byref(book), C.byref(bw)))
    return out[:bw.bytes].copy(), int(bw.buffer), int(bw.bits_free)


def sparse_band_nonzeros(layout, sparse, channel, level, band):
    n = C.c_uint32()
    _check(lib().cfb_sparse_band_nonzeros(C.byref(layout), sparse.ctypes.data, channel, level, band, C.byref(n)))
    return int(n.value)


def sparse_expand_band(layout, sparse, channel, level, band):
    bl = layout.band[channel][level][band]
    out = np.zeros((bl.height, bl.width), np.int16)
    _check(lib().cfb_sparse_expand_band(C.byref(layout), sparse.ctypes.data, channel, level, band, out.ctypes.data, bl.width * 2))
    return out


def gop2_quant_for_quality(desc, quality, interlaced=False):
    out = Gop2Quant()
    _check(lib().cfb_gop2_quant_for_quality(C.byref(desc), quality, int(bool(interlaced)), C.byref(out)))
    return out


def make_gop2_quant(divisors, prescale, midpoint_prequant=2):
    """divisors[c][wavelet 0..5][b], prescale[wavelet] (transform->prescale of the reference)."""
    q = Gop2Quant()
    q.midpoint_prequant = midpoint_prequant
    for k in range(GOP2_WAVELETS):
        q.prescale[k] = int(prescale[k])
    for c, per_c in enumerate(divisors):
        for k, per_k in enumerate(per_c):
            for b, d in enumerate(per_k):
                q.divisor[c][k][b] = int(d)
    return q


def make_quant(divisors, prescale, midpoint_prequant=2):
    """divisors[c][k][b] (k = 0 is level 1)."""
    q = Quant()
    for k in range(NUM_LEVELS):
        q.prescale[k] = prescale[k]
    q.midpoint_prequant = midpoint_prequant
    for c, per_c in enumerate(divisors):
        for k, per_k in enumerate(per_c):
            for b, d in enumerate(per_k):
                q.divisor[c][k][b] = d
    return q


def _ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))()
    for n, p in enumerate(ptrs):
        arr[n] = p
    return arr


class Context:
    def __init__(self, device=0):
        self.h = C.c_void_p()
        _check(lib().cfb_context_create(device, C.byref(self.h)))

    def close(self):
        if self.h:
            lib().cfb_context_destroy(self.h)
            self.h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def synchronize(self):
        _check(lib().cfb_context_synchronize(self.h))

    @property
    def stream(self):
        return lib().cfb_context_stream(self.h)

    # -- single wavelet level on a free-standing int16 plane (host arrays) --
    @staticmethod
    def _level_desc(w, h, plane_pitch, band_pitch, prescale, divisor, midpoint):
        d = LevelDesc(w, h, plane_pitch, band_pitch, prescale, midpoint)
        for b in range(4):
            d.divisor[b] = int(divisor[b])
        return d

    def level_forward(self, plane, prescale, divisor, midpoint=2):
        plane = np.ascontiguousarray(plane, np.int16)
        h, w = plane.shape
        bands = [np.zeros((h // 2, w // 2), np.int16) for _ in range(4)]
        d = self._level_desc(w, h, plane.strides[0], bands[0].strides[0], prescale, divisor, midpoint)
        _check(lib().cfb_level_forward_host(self.h, C.byref(d), plane.ctypes.data, _ptr_array([b.ctypes.data for b in bands])))
        return bands

    def level_inverse(self, bands, prescale, divisor):
        bands = [np.ascontiguousarray(b, np.int16) for b in bands]
        h2, w2 = bands[0].shape
        plane = np.zeros((2 * h2, 2 * w2), np.int16)
        d = self._level_desc(2 * w2, 2 * h2, plane.strides[0], bands[0].strides[0], prescale, divisor, 2)
        _check(lib().cfb_level_inverse_host(self.h, C.byref(d), _ptr_array([b.ctypes.data for b in bands]), plane.ctypes.data))
        return plane

    def range_status(self):
        """Flags of the range audit since the last call (waits for the stream); 0 = every audited plane was in range."""
        f = C.c_int()
        _check(lib().cfb_context_range_status(self.h, C.byref(f)))
        return int(f.value)

    def level_forward_device(self, w, h, plane_pitch, band_pitch, prescale, divisor, midpoint, d_plane, d_bands):
        d = self._level_desc(w, h, plane_pitch, band_pitch, prescale, divisor, midpoint)
        _check(lib().cfb_level_forward_device(self.h, C.byref(d), d_plane, _ptr_array(d_bands)))

    def level_inverse_device(self, w, h, plane_pitch, band_pitch, prescale, divisor, d_bands, d_plane):
        d = self._level_desc(w, h, plane_pitch, band_pitch, prescale, divisor, 2)
        _check(lib().cfb_level_inverse_device(self.h, C.byref(d), _ptr_array(d_bands), d_plane))

    def temporal_forward_device(self, d_a, d_b, in_pitch, d_low, d_high, out_pitch, w, h):
        _check(lib().cfb_temporal_forward_device(self.h, d_a, d_b, in_pitch, d_low, d_high, out_pitch, w, h))

    def temporal_inverse_device(self, d_low, d_high, in_pitch, d_a, d_b, out_pitch, w, h, precision=10):
        _check(lib().cfb_temporal_inverse_device(self.h, d_low, d_high, in_pitch, d_a, d_b, out_pitch, w, h, precision))

    # -- two-frame GOP building block (temporal Haar on int16 planes, host arrays) --
    def temporal_forward(self, frame1, frame2):
        a, b = np.ascontiguousarray(frame1, np.int16), np.ascontiguousarray(frame2, np.int16)
        h, w = a.shape
        low, high = np.zeros_like(a), np.zeros_like(a)
        _check(lib().cfb_temporal_forward_host(self.h, a.ctypes.data, b.ctypes.data, a.strides[0], low.ctypes.data,
                                               high.ctypes.data, low.strides[0], w, h))
        return low, high

    def temporal_inverse(self, low, high, precision=10):
        lo, hi = np.ascontiguousarray(low, np.int16), np.ascontiguousarray(high, np.int16)
        h, w = lo.shape
        a, b = np.zeros_like(lo), np.zeros_like(lo)
        _check(lib().cfb_temporal_inverse_host(self.h, lo.ctypes.data, hi.ctypes.data, lo.strides[0], a.ctypes.data,
                                               b.ctypes.data, a.strides[0], w, h, precision))
        return a, b

    def stats(self):
        s = Stats()
        _check(lib().cfb_context_stats(self.h, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in Stats._fields_}


class Codec:
    def __init__(self, ctx, desc, max_batch=1):
        self.ctx, self.desc, self.max_batch = ctx, desc, max_batch
        self.h = C.c_void_p()
        _check(lib().cfb_codec_create(ctx.h, C.byref(desc), max_batch, C.byref(self.h)))
        self.layout = Layout()
        _check(lib().cfb_codec_layout(self.h, C.byref(self.layout)))

    def close(self):
        if self.h:
            lib().cfb_codec_destroy(self.h)
            self.h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def device_frame(self, slot):
        return lib().cfb_codec_device_frame(self.h, slot)

    def device_pyramid(self, slot):
        return lib().cfb_codec_device_pyramid(self.h, slot)

    def set_bayer_phase(self, bayer_format):
        _check(lib().cfb_codec_set_bayer_phase(self.h, bayer_format))

    def set_bayer_curve(self, curve):
        """curve: uint16 array of 1 << 14 entries (the reference's per-call encode curve), or None = already applied."""
        if curve is None:
            _check(lib().cfb_codec_set_bayer_curve(self.h, None, 0))
        else:
            c = np.ascontiguousarray(curve, np.uint16)
            _check(lib().cfb_codec_set_bayer_curve(self.h, c.ctypes.data, c.size))

    def set_level_mask(self, forward_mask=7, inverse_mask=7):
        _check(lib().cfb_codec_set_level_mask(self.h, forward_mask, inverse_mask))

    # -- two-frame GOP (FIELDPLUS pyramid) as one call --
    def gop2_layout(self):
        g = Gop2Layout()
        _check(lib().cfb_gop2_layout_compute(C.byref(self.desc), C.byref(g)))
        return g

    def gop2_forward_host(self, frame_a, frame_b, gquant):
        g = self.gop2_layout()
        a, b = np.ascontiguousarray(frame_a), np.ascontiguousarray(frame_b)
        coded = np.zeros(g.coded_bytes, np.uint8)
        _check(lib().cfb_gop2_forward_host(self.h, a.ctypes.data, b.ctypes.data, a.strides[0], C.byref(gquant), coded.ctypes.data))
        return coded

    def gop2_inverse_host(self, coded, gquant, out_format, shape):
        a, b = np.zeros(shape, np.uint8), np.zeros(shape, np.uint8)
        _check(lib().cfb_gop2_inverse_host(self.h, coded.ctypes.data, C.byref(gquant), out_format, a.ctypes.data, b.ctypes.data, a.strides[0]))
        return a, b

    @staticmethod
    def gop2_band_view(glayout, buf, c, k, b):
        bl = glayout.band[c][k][b]
        flat = buf[bl.offset: bl.offset + bl.pitch * bl.height].view(np.int16)
        return flat.reshape(bl.height, bl.pitch // 2)[:, :bl.width]

    def set_interlaced(self, interlaced=True):
        """Level 1 = field transform (CFHD_ENCODING_FLAGS_YUV_INTERLACED)."""
        _check(lib().cfb_codec_set_interlaced(self.h, int(bool(interlaced))))

    def set_decode_resolution(self, resolution):
        """RESOLUTION_FULL / _HALF / _QUARTER (CFHD_PrepareToDecode's decodedResolution)."""
        _check(lib().cfb_codec_set_decode_resolution(self.h, resolution))

    def decoded_size(self):
        w, h = C.c_int(0), C.c_int(0)
        _check(lib().cfb_codec_decoded_size(self.h, C.byref(w), C.byref(h)))
        return w.value, h.value

    # -- forward -----------------------------------------------------------
    def forward_device(self, d_frames, frame_pitch, quant, d_pyramids):
        n = len(d_frames)
        _check(lib().cfb_forward_device(self.h, n, _ptr_array(d_frames), frame_pitch, C.byref(quant),
                                        _ptr_array(d_pyramids)))

    def forward_host(self, frames, quant, out=None):
        """frames: list of 2-D uint8/uint16 arrays (rows x pitch-bytes/itemsize). Returns coded buffers (uint8)."""
        n = len(frames)
        frames = [np.ascontiguousarray(f) for f in frames]
        pitch = frames[0].strides[0]
        if out is None:
            out = [np.empty(self.layout.coded_bytes, np.uint8) for _ in range(n)]
        _check(lib().cfb_forward_host(self.h, n, _ptr_array([f.ctypes.data for f in frames]), pitch, C.byref(quant),
                                      _ptr_array([o.ctypes.data for o in out])))
        return out

    def forward_host_sparse(self, frames, quant, out=None):
        n = len(frames)
        frames = [np.ascontiguousarray(f) for f in frames]
        if out is None:
            out = [np.zeros(sparse_max_bytes(self.layout), np.uint8) for _ in range(n)]
        sizes = (C.c_size_t * n)()
        _check(lib().cfb_forward_host_sparse(self.h, n, _ptr_array([f.ctypes.data for f in frames]), frames[0].strides[0],
                                             C.byref(quant), _ptr_array([o.ctypes.data for o in out]), sizes))
        return out, [int(s) for s in sizes]

    def inverse_host_sparse(self, sparse, quant, out_format, out_frames):
        n = len(sparse)
        _check(lib().cfb_inverse_host_sparse(self.h, n, _ptr_array([s.ctypes.data for s in sparse]), C.byref(quant),
                                             out_format, _ptr_array([o.ctypes.data for o in out_frames]),
                                             out_frames[0].strides[0]))
        return out_frames

    # -- inverse -----------------------------------------------------------
    def inverse_device(self, d_pyramids, quant, out_format, d_frames, frame_pitch):
        n = len(d_pyramids)
        _check(lib().cfb_inverse_device(self.h, n, _ptr_array(d_pyramids), C.byref(quant), out_format,
                                        _ptr_array(d_frames), frame_pitch))

    def inverse_host(self, coded, quant, out_format, out_frames):
        n = len(coded)
        pitch = out_frames[0].strides[0]
        _check(lib().cfb_inverse_host(self.h, n, _ptr_array([c.ctypes.data for c in coded]), C.byref(quant),
                                      out_format, _ptr_array([o.ctypes.data for o in out_frames]), pitch))
        return out_frames

    # -- helpers -----------------------------------------------------------
    def band_view(self, buf, c, k, b):
        """View of band (channel c, level index k, band b) inside a coefficient buffer (uint8 array)."""
        bl = self.layout.band[c][k][b]
        flat = buf[bl.offset: bl.offset + bl.pitch * bl.height].view(np.int16)
        return flat.reshape(bl.height, bl.pitch // 2)[:, :bl.width]

    def unpack_coded(self, buf):
        """dict {(c, level(1..3), band_name): array} of every band in the coded region."""
        out = {}
        for c in range(self.layout.num_channels):
            for k in range(NUM_LEVELS):
                for b in range(NUM_BANDS):
                    if b == 0 and k != NUM_LEVELS - 1:
                        continue
                    out[(c, k + 1, BAND_NAMES[b])] = self.band_view(buf, c, k, b).copy()
        return out

    def pack_coded(self, bands):
        buf = np.zeros(self.layout.coded_bytes, np.uint8)
        for (c, lvl, name), arr in bands.items():
            self.band_view(buf, c, lvl - 1, BAND_NAMES.index(name))[:] = arr
        return buf


def band_view(layout, buf, c, k, b):
    """View of band (channel c, level index k, band b) inside a coefficient buffer (uint8 array); host only."""
    bl = layout.band[c][k][b]
    flat = buf[bl.offset: bl.offset + bl.pitch * bl.height].view(np.int16)
    return flat.reshape(bl.height, bl.pitch // 2)[:, :bl.width]


def pack_coded(layout, bands):
    """{(c, level 1..3, band name): array} -> dense coded region as cfb_layout describes it; host only."""
    buf = np.zeros(layout.coded_bytes, np.uint8)
    for (c, lvl, name), arr in bands.items():
        if name == "LL" and lvl != NUM_LEVELS:
            continue
        band_view(layout, buf, c, lvl - 1, BAND_NAMES.index(name))[:] = arr
    return buf


def pinned_empty(shape, dtype=np.uint8):
    """numpy array backed by page-locked host memory from cfb_host_alloc (freed when the array dies)."""
    shape = (shape,) if isinstance(shape, int) else tuple(shape)
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = C.c_void_p()
    _check(lib().cfb_host_alloc(nbytes, C.byref(ptr)))
    buf = (C.c_ubyte * nbytes).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)

    class _Owner:
        def __init__(self, p):
            self.p = p

        def __del__(self):
            try:
                lib().cfb_host_free(self.p)
            except Exception:
                pass

    _PINNED[id(buf)] = (_Owner(ptr), buf)
    return arr


_PINNED = {}


class Pool:
    """Asynchronous, in-order, multi-GPU frame pool (cfb_pool_*)."""

    def __init__(self, devices, desc, slots=3, batch=4, queue_length=24):
        self.h = C.c_void_p()
        devs = (C.c_int * len(devices))(*devices)
        _check(lib().cfb_pool_create(devs, len(devices), C.byref(desc), slots, batch, queue_length, C.byref(self.h)))
        self.layout = layout_for(desc)

    def close(self):
        if self.h:
            lib().cfb_pool_destroy(self.h)
            self.h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_decode_resolution(self, resolution):
        _check(lib().cfb_pool_set_decode_resolution(self.h, resolution))

    def set_interlaced(self, interlaced=1):
        _check(lib().cfb_pool_set_interlaced(self.h, int(interlaced)))

    def submit_forward(self, frame_number, frame, quant, coded):
        _check(lib().cfb_pool_submit_forward(self.h, frame_number, frame.ctypes.data, frame.strides[0], C.byref(quant),
                                             coded.ctypes.data))

    def submit_inverse(self, frame_number, coded, quant, out_format, frame):
        _check(lib().cfb_pool_submit_inverse(self.h, frame_number, coded.ctypes.data, C.byref(quant), out_format,
                                             frame.ctypes.data, frame.strides[0]))

    def submit_forward_sparse(self, frame_number, frame, quant, sparse):
        _check(lib().cfb_pool_submit_forward_sparse(self.h, frame_number, frame.ctypes.data, frame.strides[0],
                                                    C.byref(quant), sparse.ctypes.data))

    def submit_inverse_sparse(self, frame_number, sparse, quant, out_format, frame):
        _check(lib().cfb_pool_submit_inverse_sparse(self.h, frame_number, sparse.ctypes.data, C.byref(quant), out_format,
                                                    frame.ctypes.data, frame.strides[0]))

    def wait(self):
        n, e = C.c_uint32(), C.c_int()
        _check(lib().cfb_pool_wait(self.h, C.byref(n), C.byref(e)))
        if e.value != OK:
            raise CfbError(e.value, f"job {n.value} failed")
        return n.value

    def test(self):
        """Returns the frame number of the oldest job if it has finished, else None."""
        n, e = C.c_uint32(), C.c_int()
        code = lib().cfb_pool_test(self.h, C.byref(n), C.byref(e))
        if code == 13:
            return None
        _check(code)
        if e.value != OK:
            raise CfbError(e.value, f"job {n.value} failed")
        return n.value

    def stats(self):
        s = Stats()
        _check(lib().cfb_pool_stats(self.h, C.byref(s)))
        return {k: int(getattr(s, k)) for k, _ in Stats._fields_}
