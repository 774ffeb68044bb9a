"""Numpy reference of the compressed 2:4 weight format (include/vlmc.h, "Compressed 2:4 weights"): the rules K24 / K25
(vlm-compression_b200/csrc/sparse24.cu) are tested against.  Bit patterns in, bit patterns out: fp16 and bf16 alike."""
import numpy as np


def sparse24_compress(Wbits):
    """Wbits: uint16 bit patterns [R, C] of an fp16 / bf16 weight, C % 16 == 0 -> (values uint16 [R, C/2],
    meta uint16 [R, C/16]).  Kept = bits of |w| non-zero (NaN kept, +-0 pruned); groups with fewer than two kept
    elements are padded with their lowest-index pruned positions, stored as +0.  More than two kept: ValueError."""
    W = np.asarray(Wbits, np.uint16)
    R, C = W.shape
    assert C % 16 == 0
    g = W.reshape(R, C // 4, 4)
    kept = (g & 0x7FFF) != 0
    if (kept.sum(-1) > 2).any():
        raise ValueError("not 2:4 sparse")
    key = (~kept).astype(np.int64) * 4 + np.arange(4)                    # kept first, then pruned, each by column
    sel = np.sort(np.argsort(key, axis=-1, kind="stable")[..., :2], axis=-1)
    values = np.take_along_axis(np.where(kept, g, 0).astype(np.uint16), sel, -1).reshape(R, C // 2)
    nib = (sel[..., 0] | (sel[..., 1] << 2)).astype(np.uint16).reshape(R, C // 16, 4)
    meta = nib[..., 0] | (nib[..., 1] << 4) | (nib[..., 2] << 8) | (nib[..., 3] << 12)
    return values.astype(np.uint16), meta.astype(np.uint16)


def sparse24_decompress(values, meta):
    """(values uint16 [R, C/2], meta uint16 [R, C/16]) -> dense uint16 bit patterns [R, C], +0 at pruned positions."""
    values, meta = np.asarray(values, np.uint16), np.asarray(meta, np.uint16)
    R, H = values.shape
    C = 2 * H
    nib = ((meta[..., None].astype(np.int64) >> (4 * np.arange(4))) & 15).reshape(R, C // 4)
    out = np.zeros((R, C // 4, 4), np.uint16)
    v = values.reshape(R, C // 4, 2)
    np.put_along_axis(out, (nib & 3)[..., None], v[..., 0:1], -1)
    np.put_along_axis(out, (nib >> 2)[..., None], v[..., 1:2], -1)
    return out.reshape(R, C)
