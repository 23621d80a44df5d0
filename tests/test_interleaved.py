"""Interleaved (multi-channel) views on the host side: the `channels=` view of the Python `_host` helpers and the numpy
statement of the planar-equivalent rule of include/voxbox_b200.h.  No device is needed."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vox_box.rs_b200", "python"))
import voxbox_b200 as vb  # noqa: E402
from interleave_util import frame_samples, planar_equivalent, planar_len  # noqa: E402


def test_frames_struct_sample_step_aliases_reserved():
    assert C.sizeof(vb.Frames) == 56
    fr = vb.Context.frames(0, 10, 400, 320, sample_step=2)
    assert fr.sample_step == 2 and fr.reserved == 2
    fr.reserved = 0
    assert fr.sample_step == 0
    assert vb.Frames.sample_step.offset == 52
    assert vb.Context.frames(0, 10, 400, 160).sample_step == 0


def test_header_declares_the_union():
    src = open(vb.HEADER_PATH).read()
    body = src[src.index("typedef struct vbx_frames {"):src.index("} vbx_frames;")]
    assert re.search(r"union\s*\{\s*int32_t reserved;.*int32_t sample_step;.*\};", body, re.S), body
    assert "multiple of 64 samples" in src


@pytest.mark.parametrize("args", [(0, 160, 0, 0), (98, 160, 0, 0), (98, 160, 98, 8000), (5, 80, 5, 200)])
def test_channel_view_of_one_channel_is_unchanged(args):
    n_frames, stride, J, seg = args
    assert vb.channel_view(n_frames, stride, J, seg) == (n_frames, stride, J, seg, 0)
    assert vb.channel_view(n_frames, stride, J, seg, channels=1) == (n_frames, stride, J, seg, 0)
    fr, F = vb.Context._host_view(1234, n_frames, 400, stride, vb.WINDOW_HANN_SYMMETRIC, vb.I16, J, seg)
    assert (F, fr.n_frames, fr.frame_stride, fr.frames_per_segment, fr.segment_stride, fr.sample_step) == (
        n_frames, n_frames, stride, J, seg, 0)
    assert (fr.base, fr.frame_len, fr.dtype, fr.window) == (1234, 400, vb.I16, vb.WINDOW_HANN_SYMMETRIC)


@pytest.mark.parametrize("C_", [2, 3, 6])
def test_channel_view_is_one_segment_per_channel(C_):
    F, fst, J, seg, step = vb.channel_view(98, 160, channels=C_)
    assert (F, fst, J, seg, step) == (98 * C_, 160 * C_, 98, 1, C_)
    fr, n = vb.Context._host_view(0, 98, 400, 160, vb.WINDOW_NONE, vb.MULAW8, channels=C_)
    assert n == 98 * C_ and fr.sample_step == C_ and fr.frames_per_segment == 98 and fr.segment_stride == 1


def test_channel_view_rejects_what_it_cannot_express():
    with pytest.raises(ValueError):
        vb.channel_view(10, 160, 10, 4000, channels=2)  # a batch of stereo files needs a third level
    with pytest.raises(ValueError):
        vb.channel_view(10, 160, channels=0)


@pytest.mark.parametrize("C_", [2, 3])
def test_channel_view_frames_are_the_channels_frames(C_):
    """Frame j of segment u of the helper's view is frame j of channel u of the deinterleaved recording."""
    rng = np.random.default_rng(C_)
    ns, N, hop = 3000, 200, 80
    x = rng.integers(-32768, 32767, size=(ns, C_), dtype=np.int16)  # WAV layout: [time][channel]
    J = (ns - N) // hop + 1
    F, fst, Jv, seg, step = vb.channel_view(J, hop, channels=C_)
    inter = x.reshape(-1)
    for f in (0, 1, J - 1, J, F - 1):
        u, j = divmod(f, J)
        got = frame_samples(inter, f, N, fst, Jv, seg, step)
        assert np.array_equal(got, x[j * hop:j * hop + N, u]), f


def test_planar_equivalent_hand_built_stereo():
    # L = 0, 1, 2, ...; R = 100, 101, ...; 2 frames of 3 samples, hop 2 (frame_stride 4 in interleaved samples)
    L = np.arange(10, dtype=np.int16)
    R = L + 100
    buf = np.stack([L, R], axis=1).reshape(-1)
    P, view = planar_equivalent(buf, n_frames=4, frame_len=3, frame_stride=4, frames_per_segment=2, segment_stride=1,
                                sample_step=2)
    S = ((2 - 1) * 4) // 2 + 3
    assert S == 5 == planar_len(4, 3, 4, 2, 2)
    assert P.shape == (2, 64) and P.dtype == np.int16
    assert np.array_equal(P[0, :5], L[:5]) and np.array_equal(P[1, :5], R[:5])
    assert not P[:, 5:].any()
    assert view == dict(n_frames=4, frame_len=3, frame_stride=2, frames_per_segment=2, segment_stride=64)
    # frame f of the planar view holds exactly frame f of the interleaved view
    flat = P.reshape(-1)
    for f in range(4):
        assert np.array_equal(frame_samples(buf, f, 3, 4, 2, 1, 2), frame_samples(flat, f, 3, 2, 2, 64, 0))


def test_planar_equivalent_rounds_rows_to_64_samples():
    for S_want, Sp in ((1, 64), (64, 64), (65, 128), (200, 256)):
        buf = np.arange(4 * S_want, dtype=np.float32)
        P, view = planar_equivalent(buf, n_frames=4, frame_len=S_want, frame_stride=4, frames_per_segment=1, segment_stride=1,
                                    sample_step=4)
        assert P.shape == (4, Sp) and view["segment_stride"] == Sp
        assert np.array_equal(P[3, :S_want], buf[3::4][:S_want])


def test_planar_equivalent_single_segment_and_contiguous():
    buf = (np.arange(600, dtype=np.uint8) * 7) % 251
    # one channel of three, single-segment view starting at channel 1 (base offset by the channel)
    P, view = planar_equivalent(buf[1:], n_frames=3, frame_len=50, frame_stride=60, sample_step=3)
    assert P.shape == (1, 128) and view["segment_stride"] == 0 and view["frame_stride"] == 20
    assert np.array_equal(P[0, :90], buf[1::3][:90])
    # step 0 and 1 are the contiguous view: the planar equivalent is the samples themselves
    for step in (0, 1):
        P, view = planar_equivalent(buf, n_frames=2, frame_len=100, frame_stride=50, frames_per_segment=1, segment_stride=300,
                                    sample_step=step)
        assert np.array_equal(P[0, :100], buf[:100]) and np.array_equal(P[1, :100], buf[300:400])


def test_planar_equivalent_segments_apart():
    """Channel 1 of a batch of equally long stereo files: segments do not share memory."""
    rng = np.random.default_rng(7)
    files = rng.standard_normal((3, 500, 2)).astype(np.float32)
    buf = files.reshape(-1)
    N, hop = 100, 40
    J = (500 - N) // hop + 1
    P, view = planar_equivalent(buf[1:], n_frames=3 * J, frame_len=N, frame_stride=hop * 2, frames_per_segment=J,
                                segment_stride=1000, sample_step=2)
    S = (J - 1) * hop + N
    for u in range(3):
        assert np.array_equal(P[u, :S], files[u, :S, 1])
