"""numpy statement of the planar equivalent of an interleaved vbx_frames view (include/voxbox_b200.h, sample_step): the
array every interleaved call must match bit for bit, built exactly as the header defines it."""
import numpy as np

ROW_ALIGN = 64  # samples: the planar rows S' = S rounded up to a multiple of this


def planar_len(n_frames, frame_len, frame_stride, frames_per_segment, sample_step):
    """S: the channel samples one segment spans."""
    J = frames_per_segment or n_frames
    s = max(sample_step, 1)
    return ((J - 1) * frame_stride) // s + frame_len


def planar_equivalent(buf, n_frames, frame_len, frame_stride, frames_per_segment=0, segment_stride=0, sample_step=0):
    """(P, view) for an interleaved view over the 1-D sample array `buf`: P [U][S'] of buf's dtype with P[u][k] =
    buf[u*segment_stride + k*s] for k < S and zeros after, and view = the keyword arguments of the planar view
    (frame_stride / s, segment stride S', step 0)."""
    buf = np.asarray(buf).reshape(-1)
    s = max(sample_step, 1)
    assert frame_stride % s == 0
    J = frames_per_segment or n_frames
    U = n_frames // J if J else 0
    S = planar_len(n_frames, frame_len, frame_stride, frames_per_segment, sample_step)
    Sp = -(-S // ROW_ALIGN) * ROW_ALIGN
    P = np.zeros((U, Sp), dtype=buf.dtype)
    seg = segment_stride if frames_per_segment else 0
    for u in range(U):
        P[u, :S] = buf[u * seg + np.arange(S) * s]
    view = dict(n_frames=n_frames, frame_len=frame_len, frame_stride=frame_stride // s, frames_per_segment=frames_per_segment,
                segment_stride=Sp if frames_per_segment else 0)
    return P, view


def frame_samples(buf, f, frame_len, frame_stride, frames_per_segment=0, segment_stride=0, sample_step=0):
    """Sample i of frame f of a view, straight from the header's indexing rule: base[u*seg + j*frame_stride + i*s]."""
    buf = np.asarray(buf).reshape(-1)
    s = max(sample_step, 1)
    J = frames_per_segment
    u, j = (f // J, f % J) if J else (0, f)
    return buf[u * (segment_stride if J else 0) + j * frame_stride + np.arange(frame_len) * s]
