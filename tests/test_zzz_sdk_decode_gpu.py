"""The decode side of the interposed SDK (integration/): CFHD_DecodeSample into the 16-bit and 10-bit outputs -- YU64 and V210
from 4:2:2 samples, RG48, B64A and the five 10-bit RGB words from RGB 4:4:4 samples -- runs the CUDA inverse and returns
the plain reference's bytes exactly (none of these outputs is dithered), for the dense and the sparse band hand-over."""
import json
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "integration", "_build")
have = all(os.path.exists(os.path.join(BUILD, f)) for f in ("sdk_roundtrip", "sdk_roundtrip_ref", "libCFHDCodec.so"))
needs_build = pytest.mark.skipif(not have, reason="integration/_build not built: the shim and the programs it serves compile "
                                                  "against the reference's headers and objects, so build() makes them only "
                                                  "where the reference sources are present")
FRAMES = 2
# (source format, decode format): every non-YUY2 output the shim decodes on the GPU, plus B64A from an RG48 sample
CASES = [("yu64", "same"), ("v210", "same"), ("rg48", "same"), ("rg48", "b64a"), ("rg30", "same"), ("r210", "same"),
         ("dpx0", "same"), ("ab10", "same"), ("ar10", "same")]


def inverse_stats(stderr):
    """Decode counters the shim prints at exit (CFHD_B200_STATS=1)."""
    line = stderr.split("cfhd_gpu_shim: forward frames on GPU")[-1]
    num = lambda after: int("".join(ch for ch in line.split(after)[1].split()[0] if ch.isdigit()))
    inv = line.split("inverse frames on GPU")[1]        # " <n> (reference CPU <m>), CUDA errors <k>, ..."
    return {"inv_gpu": num("inverse frames on GPU"), "inv_ref": int(inv.split("(reference CPU")[1].split(")")[0]),
            "cuda_errors": num("CUDA errors")}


def run(exe, *args, env=None):
    e = dict(os.environ, CFHD_B200_STATS="1")
    e.update(env or {})
    p = subprocess.run([os.path.join(BUILD, exe), *map(str, args)], capture_output=True, text=True, timeout=600, env=e, cwd=BUILD)
    assert p.returncode == 0, p.stderr[-2000:]
    return p, json.loads(p.stdout.strip().splitlines()[-1])


@needs_build
@pytest.mark.parametrize("size", [(1920, 1080), (1280, 720), (720, 486)])
@pytest.mark.parametrize("src,dst", CASES)
def test_sdk_decode_outputs_match_reference(size, src, dst):
    w, h = size
    if (w, h) == (720, 486) and (src, dst) not in (("yu64", "same"), ("v210", "same"), ("rg48", "same")):
        pytest.skip("display window smaller than the coded frame: covered by yu64, v210 and rg48")
    args = (w, h, FRAMES, 0, 24, 0, src, dst)
    _, ref = run("sdk_roundtrip_ref", *args)
    assert ref["decoded_frames"] == FRAMES and ref["guard_ok"] == 1
    for env in ({}, {"CFHD_B200_DECODE_SPARSE": "1"}):
        p, got = run("sdk_roundtrip", *args, env=env)
        st = inverse_stats(p.stderr)
        assert got["decoded_frames"] == FRAMES and got["guard_ok"] == 1, env
        assert got["decoded_digest"] == ref["decoded_digest"], env
        assert st["inv_gpu"] >= FRAMES and st["inv_ref"] == 0 and st["cuda_errors"] == 0, (env, st)
