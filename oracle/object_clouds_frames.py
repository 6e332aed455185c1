"""CPU restatement (numpy, test-only) of gp_backproject_frames (DESIGN.md section 4.13): stage A over F frames of one
size.  Objects are numbered frame-major, and the result is oracle.object_clouds.backproject_instances of every frame,
with its own intrinsics, concatenated in frame order after the device's clamp of the frame offsets (frame_ranges).
Stage B is oracle.object_clouds.sample_points unchanged."""
import numpy as np

from oracle.object_clouds import backproject_instances


def frame_ranges(frame_offsets, B):
    """The object ranges gp_backproject_frames uses for frame offsets [F+1] as given: frame f holds objects
    r[f] .. r[f+1]-1.  r[0] = 0 and r[F] = B whatever the array holds; in between, offsets[f] is raised to the largest
    of offsets[1..f] and clamped into [0, B].  Well-formed offsets (0 = o_0 <= ... <= o_F = B) are unchanged."""
    o = np.asarray(frame_offsets, dtype=np.int64)
    F = len(o) - 1
    r = np.empty(F + 1, dtype=np.int64)
    r[0], r[F] = 0, B
    r[1:F] = np.clip(np.maximum.accumulate(o[1:F]), 0, B)
    return r


def backproject_frames(depth, labels, intrinsics, frame_offsets, B):
    """depth float32 [F,H,W], labels int32 [F,H,W], intrinsics [F][4] (fx, fy, cx, cy), frame_offsets [F+1] ->
    (xyz float32 [total, 3], offsets int32 [B+1]): backproject_instances of every frame with its own intrinsics and
    its n_f = r[f+1] - r[f] objects (frame_ranges), concatenated in frame order; frame f's label l is object r[f] + l - 1.
    Zero or non-finite intrinsics give non-finite points, as on the device."""
    r = frame_ranges(frame_offsets, B)
    xs, offsets = [], [0]
    with np.errstate(divide="ignore"):   # fx or fy == 0: IEEE inf / nan points, no warning
        for f in range(len(r) - 1):
            xyz, off = backproject_instances(depth[f], labels[f], *np.asarray(intrinsics[f]), int(r[f + 1] - r[f]))
            xs.append(xyz)
            base = offsets[-1]
            offsets.extend(base + int(o) for o in off[1:])
    return np.concatenate(xs).astype(np.float32), np.asarray(offsets, dtype=np.int32)
