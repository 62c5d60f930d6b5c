"""BASELINE.json configs[0]: "WaveletDemo 1920x1080 PGM 3-level forward+inverse on CPU (bit-exact gate, no GPU)".

The reference's toy int32 model (Example/WaveletDemo/wavelets.c:83, utils.c) compiled in place by oracle/Makefile
(oracle/_ref/WaveletDemo) must reproduce the known answers the reference itself publishes:
  * the transcript of README.md:101-111 (per-level min/max, quantised min/max, energy, PSNR), character for character;
  * the three images it writes (BASELINE.md: md5 of -wavelet / -decoded / -x10-diff, produced by running
    `WaveletDemo testpatt.pgm` inside the data directory: the PGM header carries the output path as a comment, so
    the file hashes are only reproducible with that invocation; the pixel payloads are hashed separately).
It is its own gate (SURVEY 8, note on config 1): the demo shares the 2-6 taps and the +4 >> 3 rounding with the SDK but
not its prescale / quantiser rules, so it does not stand in for rows a3-a8."""
import hashlib
import lzma
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEMO = os.path.join(ROOT, "oracle", "_ref", "WaveletDemo")
# the reference's data/testpatt.pgm, byte for byte (the output hashes depend on every byte of it)
PATTERN = os.path.join(ROOT, "tests", "golden", "testpatt.pgm.xz")

needs_demo = pytest.mark.skipif(not os.path.exists(DEMO),
                                reason="oracle/_ref/WaveletDemo not built (oracle/Makefile compiles it from the reference sources)")

# README.md:101-111 of the reference
TRANSCRIPT = """source image size = 1920,1080
source size = 2073656 bytes
High pass (960,540) min,max =  -8385,  8119, minq,maxq = -111, 106, overflow 0.000%, energy = 4131033
High pass (480,270) min,max = -13619, 14005, minq,maxq = -160, 162, overflow 0.000%, energy = 3095823
High pass (240,135) min,max = -18358, 17590, minq,maxq = -186, 195, overflow 0.000%, energy = 1130216
Low Pass (240,135) min = 53, max = 32711

PSNR = 54.386
"""
FILE_MD5 = {            # BASELINE.md (config-1 known answer)
    "testpatt-wavelet.pgm": "2cda01173a13c0106f19cf6946ab6023",
    "testpatt-decoded.pgm": "5eddb9c0160d2f9f56bd3ed40dba752a",
    "testpatt-x10-diff.pgm": "301b7ca472551e97f2b9716f7186db61",
}
PAYLOAD_MD5 = {         # the 1920 x 1080 bytes behind the header (independent of the path in the header comment)
    "testpatt-wavelet.pgm": "7bee31170614ce5426f85b1ed835cecd",
    "testpatt-decoded.pgm": "80ecaabe99881b198cbc379a02e2d567",
    "testpatt-x10-diff.pgm": "60eebe4a77f146518186ce67f505d4dd",
}


def _payload(path):
    data = open(path, "rb").read()
    magic, comment, dims, maxval, pixels = data.split(b"\n", 4)
    assert magic == b"P5" and comment.startswith(b"#") and dims == b"1920 1080" and maxval == b"255"
    return pixels


@needs_demo
def test_waveletdemo_known_answers(tmp_path):
    (tmp_path / "testpatt.pgm").write_bytes(lzma.decompress(open(PATTERN, "rb").read()))
    p = subprocess.run([DEMO, "testpatt.pgm"], cwd=tmp_path, capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr
    assert p.stdout.replace("\r\n", "\n").strip() == TRANSCRIPT.strip()
    for name, want in FILE_MD5.items():
        assert hashlib.md5(open(tmp_path / name, "rb").read()).hexdigest() == want, name
        assert hashlib.md5(_payload(tmp_path / name)).hexdigest() == PAYLOAD_MD5[name], name
    # the printed PSNR is the PSNR of the decoded image it wrote, against the 8-bit source
    src = np.frombuffer(open(tmp_path / "testpatt.pgm", "rb").read()[-1920 * 1080:], np.uint8)
    dec = np.frombuffer(_payload(tmp_path / "testpatt-decoded.pgm"), np.uint8)
    assert src.size == dec.size == 1920 * 1080
    # (the demo measures at its 12-bit working depth with rand() noise added, README "PSNR = 54.386"; the 8-bit files
    # must at least agree to within the 8-bit rounding of that figure)
    mse = np.mean((src.astype(np.float64) - dec.astype(np.float64)) ** 2)
    assert 10 * np.log10(255.0 ** 2 / max(mse, 1e-12)) > 48.0
