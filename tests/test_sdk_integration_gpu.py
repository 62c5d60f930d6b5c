"""The reference SDK with the CUDA transform interposed (integration/): programs that use only the public CFHD_* API
-- our sdk_roundtrip driver and the reference's own Example/TestCFHD.cpp, both compiled unchanged against
integration/_build/libCFHDCodec.so -- must behave as with the plain reference: identical entropy-coded sample sizes
(same coefficients), same PSNR (up to the reference's rand() dither), in-order pool delivery."""
import json
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "integration", "_build")
have = all(os.path.exists(os.path.join(BUILD, f)) for f in ("sdk_roundtrip", "sdk_roundtrip_ref", "TestCFHD", "libCFHDCodec.so"))
needs_build = pytest.mark.skipif(not have, reason="integration/_build not built: the shim and the programs it serves compile "
                                                  "against the reference's headers and objects, so build() makes them only "
                                                  "where the reference sources are present")


def shim_stats(stderr):
    """Counters the shim prints at exit (CFHD_B200_STATS=1)."""
    line = stderr.split("cfhd_gpu_shim: forward frames on GPU")[-1]
    num = lambda after: int("".join(ch for ch in line.split(after)[1].split()[0] if ch.isdigit()))
    return {"fwd_gpu": int(line.split()[0]), "fwd_ref": num("(reference CPU"), "inv_gpu": num("inverse frames on GPU"),
            "cuda_errors": num("CUDA errors"), "sparse_bands": num("bands coded from the sparse format"),
            "dense_bands": num("(dense, by the reference's coder")}


def run(exe, *args, env=None):
    e = dict(os.environ, CFHD_B200_STATS="1")
    e.update(env or {})
    p = subprocess.run([os.path.join(BUILD, exe), *map(str, args)], capture_output=True, text=True, timeout=600, env=e, cwd=BUILD)
    assert p.returncode == 0, p.stderr[-2000:]
    return p


@needs_build
@pytest.mark.parametrize("size", [(1920, 1080), (3840, 2160), (1440, 1080)])
def test_public_api_roundtrip_matches_reference(size):
    w, h = size
    gpu = run("sdk_roundtrip", w, h, 4, 4)
    ref = run("sdk_roundtrip_ref", w, h, 4, 4)
    g, r = json.loads(gpu.stdout.strip().splitlines()[-1]), json.loads(ref.stdout.strip().splitlines()[-1])
    assert "forward frames on GPU" in gpu.stderr
    stats = gpu.stderr.split("cfhd_gpu_shim: forward frames on GPU")[-1]
    fwd_gpu = int(stats.split()[0])
    inv_gpu = int(stats.split("inverse frames on GPU")[1].split()[0])
    assert fwd_gpu >= 4 + 64 and inv_gpu >= 4          # sync loop + pool frames went through the CUDA path
    assert g["sample_bytes"] == r["sample_bytes"]       # identical coefficients -> identical entropy-coded size
    # ... and identical BYTES: the samples were entropy coded straight from the sparse transfer format
    # (cfb_sparse_vlc_band in place of EncodeQuantLongRuns), in the sync loop and by the pool's worker threads
    assert g["sample_digest"] == r["sample_digest"] and g["pool_sample_digest"] == r["pool_sample_digest"]
    st = shim_stats(gpu.stderr)
    assert st["fwd_ref"] == 0 and st["cuda_errors"] == 0                # no frame of a covered format took the CPU transform
    assert st["sparse_bands"] == 27 * st["fwd_gpu"] and st["dense_bands"] == 0      # 9 highpass bands x 3 channels, every frame
    # the dense hand-over (33 MB per 4K frame over PCIe + the reference's own coder) must give the same bytes
    dense = run("sdk_roundtrip", w, h, 2, 0, env={"CFHD_B200_DENSE": "1"})
    sparse2 = run("sdk_roundtrip", w, h, 2, 0)
    d, s2 = json.loads(dense.stdout.strip().splitlines()[-1]), json.loads(sparse2.stdout.strip().splitlines()[-1])
    assert d["sample_digest"] == s2["sample_digest"]
    assert shim_stats(dense.stderr)["sparse_bands"] == 0
    assert abs(g["luma_psnr_db"] - r["luma_psnr_db"]) < 0.1
    assert g["pool_fps"] > 0


@needs_build
def test_samples_are_byte_identical_up_to_the_timestamp(tmp_path):
    """The first sample of either arm, byte by byte: the only bytes allowed to differ are ASCII digits in the sample
    header (the wall-clock time the encoder stores as metadata); everything behind it -- every band header, the lowpass
    bands and the run-length / VLC streams written from the sparse format -- is identical."""
    import numpy as np
    files = {}
    for arm, exe, env in (("sparse", "sdk_roundtrip", {}), ("dense", "sdk_roundtrip", {"CFHD_B200_DENSE": "1"}), ("ref", "sdk_roundtrip_ref", {})):
        path = str(tmp_path / f"{arm}.bin")
        run(exe, 1920, 1080, 1, 0, env=dict(env, CFHD_DUMP_SAMPLE=path))
        files[arm] = np.fromfile(path, np.uint8)
    ref = files["ref"]
    for arm in ("sparse", "dense"):
        got = files[arm]
        assert got.size == ref.size
        diff = np.nonzero(got != ref)[0]
        assert diff.size <= 8 and (diff < 512).all(), f"{arm}: {diff[:10].tolist()}"
        assert all(48 <= int(got[o]) <= 57 and 48 <= int(ref[o]) <= 57 for o in diff)


@needs_build
def test_public_api_roundtrip_height_not_multiple_of_8():
    """720x486 (NTSC) is coded as 488 rows (encoder.c:2232) but the caller's buffer holds 486: the interposed decoder
    must write the display window only (guard rows behind the frame stay untouched), with the reference's sample size."""
    gpu = run("sdk_roundtrip", 720, 486, 3, 2)
    ref = run("sdk_roundtrip_ref", 720, 486, 3, 2)
    g, r = json.loads(gpu.stdout.strip().splitlines()[-1]), json.loads(ref.stdout.strip().splitlines()[-1])
    assert g["guard_ok"] == 1 and r["guard_ok"] == 1
    stats = gpu.stderr.split("cfhd_gpu_shim: forward frames on GPU")[-1]
    assert int(stats.split("inverse frames on GPU")[1].split()[0]) >= 3      # the decode did run on the GPU
    assert g["sample_bytes"] == r["sample_bytes"] and g["sample_digest"] == r["sample_digest"]
    assert abs(g["luma_psnr_db"] - r["luma_psnr_db"]) < 0.1


@needs_build
def test_testcfhd_runs_unchanged():
    """Example/TestCFHD.cpp -E (encoder pool speed test over its format table) against libCFHDCodec.so."""
    p = run("TestCFHD", "-E")
    assert "fps" in p.stdout
    assert "forward frames on GPU" in p.stderr
    fwd_gpu = int(p.stderr.split("cfhd_gpu_shim: forward frames on GPU")[-1].split()[0])
    assert fwd_gpu >= 500                               # at least the YUY2 row of the table ran on the GPU
    assert shim_stats(p.stderr)["cuda_errors"] == 0


@needs_build
@pytest.mark.parametrize("size", [(1920, 1080), (720, 480)])
def test_public_api_interlaced_roundtrip_matches_reference(size):
    """CFHD_ENCODING_FLAGS_YUV_INTERLACED through the unmodified SDK: the field transform (forward incl. the
    difference-coded HL band, inverse on the decoder's already-integrated band) runs on the GPU and the entropy coder
    produces byte-for-byte the same sample size as with the reference's CPU transform.  720x480: ragged band widths."""
    w, h = size
    gpu = run("sdk_roundtrip", w, h, 3, 2, 24, 1)
    ref = run("sdk_roundtrip_ref", w, h, 3, 2, 24, 1)
    g, r = json.loads(gpu.stdout.strip().splitlines()[-1]), json.loads(ref.stdout.strip().splitlines()[-1])
    assert g["interlaced"] == 1
    stats = gpu.stderr.split("cfhd_gpu_shim: forward frames on GPU")[-1]
    fwd_gpu = int(stats.split()[0])
    inv_gpu = int(stats.split("inverse frames on GPU")[1].split()[0])
    assert fwd_gpu >= 3 + 32 and inv_gpu >= 3
    assert g["sample_bytes"] == r["sample_bytes"] and g["sample_digest"] == r["sample_digest"]
    # >= : the reference's own threaded decode of interlaced frames occasionally returns unfinished chroma rows (see
    # tests/test_pyramid_cpu.py), which can only lower ITS luma-independent score; ours must not be worse
    assert g["luma_psnr_db"] > r["luma_psnr_db"] - 0.1 and g["luma_psnr_db"] > 45.0


@needs_build
@pytest.mark.parametrize("fmt", ["2vuy", "yu64", "v210", "rg48", "rg30", "r210", "dpx0", "ab10", "ar10", "byr4"])
def test_public_api_encode_of_every_wired_source_format(fmt):
    """Every source format whose level-1 kernel exists is served by the GPU under the unmodified SDK: the packed frame is
    read by the kernels directly (the reference's CPU conversion to planes and its per-plane level-1 calls are skipped),
    the samples -- sync loop and encoder pool -- are byte-identical to the reference's, and no frame of these formats
    takes the CPU transform."""
    # V210 rows are whole 48-pixel groups; Bayer planes (half size) need a height that is a multiple of 8 as well, else the
    # encoder pads the planes and the frame stays with the reference's converter
    w, h = {"v210": (1536, 864), "byr4": (2048, 1152)}.get(fmt, (1920, 1080))
    gpu = run("sdk_roundtrip", w, h, 3, 2, 24, 0, fmt)
    ref = run("sdk_roundtrip_ref", w, h, 3, 2, 24, 0, fmt)
    g, r = json.loads(gpu.stdout.strip().splitlines()[-1]), json.loads(ref.stdout.strip().splitlines()[-1])
    assert g["format"] == fmt
    assert g["sample_bytes"] == r["sample_bytes"]
    assert g["sample_digest"] == r["sample_digest"] and g["pool_sample_digest"] == r["pool_sample_digest"]
    st = shim_stats(gpu.stderr)
    assert st["fwd_gpu"] >= 4 + 32 and st["fwd_ref"] == 0 and st["cuda_errors"] == 0
    assert st["sparse_bands"] > 0 and st["dense_bands"] == 0
