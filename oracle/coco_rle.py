"""TEST INFRASTRUCTURE: COCO run-length encoding restated in numpy from pycocotools' maskApi.c (rleEncode, rleToString,
rleFrString, rleDecode), the reference for the device encoder (psalm_b200.coco / csrc/rle.cu).  pycocotools itself is
third-party and optional; tests/test_coco_rle_cpu.py compares this module with it when it can be imported.

Conventions of maskApi.c: a mask [H, W] is traversed in column-major (Fortran) order; the counts alternate 0-runs and
1-runs and start with a 0-run (length 0 when pixel (0, 0) is set); counts are uint32."""
import numpy as np


def rle_encode(mask):
    """maskApi.c rleEncode of one binary mask [H, W] (non-zero = foreground) -> uint32 counts."""
    m = np.asarray(mask)
    if m.ndim != 2:
        raise ValueError("rle_encode: expected a 2-D mask, got shape %s" % (m.shape,))
    a = (m != 0).ravel(order="F")
    prev = np.concatenate([[False], a[:-1]])
    starts = np.flatnonzero(a != prev)                   # every pixel that differs from its predecessor (an implicit 0)
    bounds = np.concatenate([[0], starts, [a.size]]).astype(np.int64)
    return np.diff(bounds).astype(np.uint32)


def rle_to_string(counts):
    """maskApi.c rleToString: delta against counts[i-2] for i > 2, 5-bit groups least significant first, 0x20 = more
    groups follow, + 48."""
    c = [int(v) for v in counts]
    out = bytearray()
    for i, v in enumerate(c):
        x = v - c[i - 2] if i > 2 else v
        more = True
        while more:
            ch = x & 0x1F
            x >>= 5                                          # arithmetic shift (Python ints)
            more = (x != -1) if (ch & 0x10) else (x != 0)
            if more:
                ch |= 0x20
            out.append(ch + 48)
    return bytes(out)


def rle_fr_string(s):
    """maskApi.c rleFrString: compressed counts string -> uint32 counts."""
    if isinstance(s, str):
        s = s.encode()
    cnts, p = [], 0
    while p < len(s):
        x, k, more = 0, 0, True
        while more:
            ch = s[p] - 48
            x |= (ch & 0x1F) << (5 * k)
            more = bool(ch & 0x20)
            p += 1
            k += 1
            if not more and (ch & 0x10):
                x |= -1 << (5 * k)
        if len(cnts) > 2:
            x += cnts[-2]
        cnts.append(x & 0xFFFFFFFF)
    return np.array(cnts, dtype=np.uint32)


def rle_decode(counts, h, w):
    """maskApi.c rleDecode: counts -> uint8 mask [h, w]."""
    counts = np.asarray(counts, dtype=np.int64)
    vals = np.arange(counts.size) % 2
    flat = np.repeat(vals, counts).astype(np.uint8)
    if flat.size != h * w:
        raise ValueError("rle_decode: counts sum to %d, not %d pixels" % (flat.size, h * w))
    return flat.reshape(w, h).T.copy()


def encode(mask):
    """pycocotools.mask.encode of one mask [H, W]: {"size": [H, W], "counts": bytes}."""
    m = np.asarray(mask)
    return {"size": [int(m.shape[0]), int(m.shape[1])], "counts": rle_to_string(rle_encode(m))}


def decode(rle):
    """pycocotools.mask.decode of one RLE dict -> uint8 mask [H, W]."""
    h, w = rle["size"]
    return rle_decode(rle_fr_string(rle["counts"]), h, w)
