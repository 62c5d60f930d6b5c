"""Oracle of the V210 decode output (test infrastructure): the reference decoder's V210 frame from reconstructed planes."""
import numpy as np

import parity_util as pu


def v210_output_tail_cb_word(width):
    """Index of the word (within a row, None if none) whose bits 20-29 the reference's decoder fills from outside the row:
    for width % 6 == 4 the scalar tail of Codec/convert.c:13526 ConvertPlanarYUVToV210 reads u_row_ptr[width / 2], one past
    the Cb row of its scratch strip (the next scratch row's first luma sample, or stale scratch on a strip's last row).
    pack_v210_output defines that field as the row's last Cb; parity with the reference excludes it."""
    return (width // 6) * 4 + 2 if width % 6 == 4 else None


def pack_v210_output(planes, precision=10):
    """[Y, ch1, ch2] int16 planes -> the reference decoder's V210 frame for DECODED_FORMAT_V210 (height x 4*ceil(width/6)
    uint32): Codec/decoder.c:26292 -> InvertHorizontalStrip16s.c:6490 renders YU64 rows (parity_util.row16u) and
    convert.c:13526 ConvertPlanarYUVToV210 at precision 16 takes each >> 6.  Words Cb0 Y0 Cr0 | Y1 Cb2 Y2 | Cr2 Y3 Cb4 |
    Y4 Cr4 Y5 at bits 0 / 10 / 20, Cb = channel 2, Cr = channel 1.  A partial last group is completed as the scalar tail
    (:13888-13965) does: a component past the right edge repeats what its variable last held -- width % 6 == 2: luma
    y0 y1 y0 y1 y1 y0 with the one chroma pair thrice; width % 6 == 4: luma y0 y1 y2 y3 y3 y2, chroma pairs 0 1 1 (see
    v210_output_tail_cb_word for the one field the reference takes from outside the row)."""
    y, cr, cb = [pu.row16u(p, precision).astype(np.uint32) >> (16 - precision) for p in planes]
    h, w = y.shape
    rem = w % 6
    if rem == 2:
        y = np.concatenate([y, y[:, [-2, -1, -1, -2]]], axis=1)
        cb, cr = (np.concatenate([c, c[:, [-1, -1]]], axis=1) for c in (cb, cr))
    elif rem == 4:
        y = np.concatenate([y, y[:, [-1, -2]]], axis=1)
        cb, cr = (np.concatenate([c, c[:, [-1]]], axis=1) for c in (cb, cr))
    comp = np.zeros((h, 2 * y.shape[1]), np.uint32)
    comp[:, 0::4], comp[:, 1::4], comp[:, 2::4], comp[:, 3::4] = cb, y[:, 0::2], cr, y[:, 1::2]
    return (comp[:, 0::3] | (comp[:, 1::3] << 10) | (comp[:, 2::3] << 20)).astype(np.uint32)
