"""ITU-T G.711 restated in numpy (the g711.c tables that audioop and the library use): the tests' reference codec."""
import numpy as np


def mulaw_decode(codes):
    """uint8 mu-law codes -> int16 linear values (audioop.ulaw2lin(b, 2))."""
    u = (~np.asarray(codes, dtype=np.uint8)).astype(np.int32)
    t = (((u & 0x0F) << 3) + 0x84) << ((u & 0x70) >> 4)
    return np.where(u & 0x80, 0x84 - t, t - 0x84).astype(np.int16)


def alaw_decode(codes):
    """uint8 A-law codes -> int16 linear values (audioop.alaw2lin(b, 2))."""
    a = np.asarray(codes, dtype=np.uint8).astype(np.int32) ^ 0x55
    seg = (a & 0x70) >> 4
    t = ((a & 0x0F) << 4) + np.where(seg > 0, 0x108, 8)
    t = np.where(seg > 1, t << np.maximum(seg - 1, 0), t)
    return np.where(a & 0x80, t, -t).astype(np.int16)


def _segment(v, first_end):
    """g711.c search(): the first segment whose end (first_end·2^s + 2^s − 1) is >= v, or 8."""
    ends = (first_end + 1) * (1 << np.arange(8)) - 1
    return np.searchsorted(ends, v, side="left")


def mulaw_encode(x):
    """int16 values -> uint8 mu-law codes (audioop.lin2ulaw(x, 2): g711.c's 14-bit encoder on x >> 2)."""
    v = np.asarray(x, dtype=np.int16).astype(np.int32) >> 2
    mask = np.where(v < 0, 0x7F, 0xFF)
    v = np.minimum(np.abs(v), 8159) + (0x84 >> 2)
    seg = _segment(v, 0x3F)
    code = np.where(seg >= 8, 0x7F, (seg << 4) | ((v >> (np.minimum(seg, 7) + 1)) & 0x0F))
    return (code ^ mask).astype(np.uint8)


def alaw_encode(x):
    """int16 values -> uint8 A-law codes (audioop.lin2alaw(x, 2): g711.c's 13-bit encoder on x >> 3)."""
    v = np.asarray(x, dtype=np.int16).astype(np.int32) >> 3
    mask = np.where(v < 0, 0x55, 0xD5)
    v = np.where(v < 0, -v - 1, v)
    seg = _segment(v, 0x1F)
    q = np.where(seg < 2, v >> 1, v >> np.minimum(seg, 7)) & 0x0F
    code = np.where(seg >= 8, 0x7F, (seg << 4) | q)
    return (code ^ mask).astype(np.uint8)


DECODE = {"mulaw": mulaw_decode, "alaw": alaw_decode}
ENCODE = {"mulaw": mulaw_encode, "alaw": alaw_encode}
