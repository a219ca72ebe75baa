"""numpy port of the dropout keep masks of csrc/dropout.cuh, bit for bit.

Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11) with
key = seed (low word, high word) and counter = (row, col / 8, layer, step).  One call gives four 32-bit words =
eight 16-bit lanes, one per feature of the 8-column chunk: feature 8c + 2j takes the low half of word j, 8c + 2j + 1
its high half.  A unit is kept iff its lane >= thr = round(p * 65536); kept units are scaled by
s = 1 / (1 - thr / 65536) in fp32.
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
_LO = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10: counters and keys are uint32 arrays (broadcast); returns four uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint32) for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0 = np.asarray(k0, dtype=np.uint32).copy()
    k1 = np.asarray(k1, dtype=np.uint32).copy()
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = _M0 * c[0].astype(np.uint64)
            p1 = _M1 * c[2].astype(np.uint64)
            n0 = (p1 >> np.uint64(32)).astype(np.uint32) ^ c[1] ^ k0
            n2 = (p0 >> np.uint64(32)).astype(np.uint32) ^ c[3] ^ k1
            c = [n0, (p1 & _LO).astype(np.uint32), n2, (p0 & _LO).astype(np.uint32)]
            k0 = k0 + _W0
            k1 = k1 + _W1
    return c


def threshold(p):
    """thr = round(p * 65536) of the fp32 probability, as the kernels compute it."""
    return int(round(float(np.float32(p)) * 65536.0))


def scale(p):
    """s = 1 / (1 - thr / 65536), rounded to fp32."""
    return np.float32(1.0) / (np.float32(1.0) - np.float32(threshold(p)) / np.float32(65536.0))


def keep_mask(n, width, p, seed, step, layer, row0=0):
    """(n, width) bool keep mask of one hidden layer."""
    seed = int(seed) % (1 << 64)
    chunks = (width + 7) // 8
    rows = (np.arange(n, dtype=np.int64) + int(row0)).astype(np.uint64) & _LO
    r = rows.astype(np.uint32)[:, None]
    c = np.arange(chunks, dtype=np.uint32)[None, :]
    w = philox4x32_10(r, c, np.uint32(layer & 0xFFFFFFFF), np.uint32(step & 0xFFFFFFFF),
                      np.uint32(seed & 0xFFFFFFFF), np.uint32(seed >> 32))
    lanes = np.empty((n, chunks, 8), dtype=np.uint32)
    for j in range(4):
        lanes[:, :, 2 * j] = w[j] & np.uint32(0xFFFF)
        lanes[:, :, 2 * j + 1] = w[j] >> np.uint32(16)
    return (lanes >= np.uint32(threshold(p))).reshape(n, chunks * 8)[:, :width]
