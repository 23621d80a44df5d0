"""G.711 mu-law / A-law input (VBX_MULAW8 / VBX_ALAW8), the CPU side: the numpy codec the GPU tests compare against is
checked against Python's audioop (the g711.c tables) on every code and every int16 value, and the dtype values of the header,
the Python binding and the Rust shim agree."""
import os
import re
import warnings

import numpy as np
import pytest

from g711_codec import alaw_decode, alaw_encode, mulaw_decode, mulaw_encode
from gpu_util import ROOT, vb

with warnings.catch_warnings():
    warnings.simplefilter("ignore", DeprecationWarning)
    try:
        import audioop  # removed in Python 3.13
    except ImportError:
        audioop = None

needs_audioop = pytest.mark.skipif(audioop is None, reason="audioop is not part of this Python (>= 3.13)")
CODES = np.arange(256, dtype=np.uint8)
PCM = np.arange(-32768, 32768, dtype=np.int16)


@needs_audioop
def test_decode_matches_audioop_on_every_code():
    assert np.array_equal(mulaw_decode(CODES), np.frombuffer(audioop.ulaw2lin(CODES.tobytes(), 2), dtype=np.int16))
    assert np.array_equal(alaw_decode(CODES), np.frombuffer(audioop.alaw2lin(CODES.tobytes(), 2), dtype=np.int16))


@needs_audioop
def test_encode_matches_audioop_on_every_int16():
    assert np.array_equal(mulaw_encode(PCM), np.frombuffer(audioop.lin2ulaw(PCM.tobytes(), 2), dtype=np.uint8))
    assert np.array_equal(alaw_encode(PCM), np.frombuffer(audioop.lin2alaw(PCM.tobytes(), 2), dtype=np.uint8))


def test_codec_ranges_and_round_trip():
    assert mulaw_decode(CODES).min() == -32124 and mulaw_decode(CODES).max() == 32124
    assert alaw_decode(CODES).min() == -32256 and alaw_decode(CODES).max() == 32256
    # every code's value encodes back to a code of the same value (mu-law has two codes for 0)
    assert np.array_equal(mulaw_decode(mulaw_encode(mulaw_decode(CODES))), mulaw_decode(CODES))
    assert np.array_equal(alaw_encode(alaw_decode(CODES)), CODES)


def test_dtype_constants_agree():
    hdr = open(os.path.join(ROOT, "include", "voxbox_b200.h")).read()
    m = re.search(r"typedef enum vbx_dtype \{([^}]*)\}", hdr)
    enum = {k: int(v) for k, v in re.findall(r"(VBX_\w+)\s*=\s*(\d+)", m.group(1))}
    assert enum == {"VBX_F32": 0, "VBX_F64": 1, "VBX_I16": 2, "VBX_MULAW8": 3, "VBX_ALAW8": 4}
    assert (vb.F32, vb.F64, vb.I16, vb.MULAW8, vb.ALAW8) == (0, 1, 2, 3, 4)
    rs = open(os.path.join(ROOT, "rust", "vox_box_b200", "src", "lib.rs")).read()
    consts = {k: int(v) for k, v in re.findall(r"pub const (VBX_(?:F32|F64|I16|MULAW8|ALAW8)): i32 = (\d+);", rs)}
    assert consts == enum


def test_uint8_host_samples_need_a_law():
    codes = np.zeros(16, dtype=np.uint8)
    with pytest.raises(ValueError):
        vb._sample_dtype(codes)
    with pytest.raises(ValueError):
        vb._host_audio(codes)
    with pytest.raises(ValueError):  # a law for samples that are not bytes
        vb._sample_dtype(np.zeros(16, dtype=np.int16), vb.MULAW8)
    assert vb._sample_dtype(codes, vb.MULAW8) == vb.MULAW8 and vb._host_audio(codes, vb.ALAW8)[1] == vb.ALAW8
    assert vb._sample_dtype(np.zeros(4, dtype=np.int16)) == vb.I16 and vb._sample_dtype(np.zeros(4, dtype=np.float32)) == vb.F32
