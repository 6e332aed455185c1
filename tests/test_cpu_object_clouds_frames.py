"""CPU: per-object point clouds from a batch of frames (genpose2_b200.clouds.backproject_frames /
object_clouds_frames).  The oracle's frames restatement against its per-frame restatement concatenated (empty frames,
labels above a frame's count, the device's clamp of malformed frame offsets), every Python validation error before any
device work, the C ABI's refusals and its workspace formula."""
import ctypes

import numpy as np
import pytest
import torch

from genpose2_b200 import _lib, clouds, synthetic
from oracle import object_clouds as oc
from oracle import object_clouds_frames as ocf


def per_frame(depth, labels, intr, counts):
    xs, offsets = [], [0]
    for f, n in enumerate(counts):
        xyz, off = oc.backproject_instances(depth[f], labels[f], *intr[f], n)
        xs.append(xyz)
        offsets += [offsets[-1] + int(o) for o in off[1:]]
    return np.concatenate(xs), np.asarray(offsets, np.int32)


def offsets_of(counts):
    return np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)


@pytest.mark.parametrize("counts", [[3], [2, 0, 4], [0, 0, 5, 0], [1] * 7, [0, 6]])
def test_oracle_frames_is_the_per_frame_concatenation(counts):
    depth, labels, intr = synthetic.make_instance_frames(24, 40, counts, seed=len(counts), bad_depth=0.05,
                                                         stray_labels=0.05)
    B = sum(counts)
    # a label of the next frame's range (above this frame's count) is background
    labels[0, :2, :3] = counts[0] + 1
    xyz, off = ocf.backproject_frames(depth, labels, intr, offsets_of(counts), B)
    want_xyz, want_off = per_frame(depth, labels, intr, counts)
    assert np.array_equal(off, want_off) and off[-1] == len(xyz)
    assert np.array_equal(xyz.view(np.int32), want_xyz.view(np.int32))
    for f, n in enumerate(counts):   # frame f's label l is object base_f + l - 1
        base = sum(counts[:f])
        for l in range(1, n + 1):
            z = depth[f][labels[f] == l]
            k = int(((z > 0) & np.isfinite(z)).sum())
            assert off[base + l] - off[base + l - 1] == k


def test_oracle_frame_ranges_clamp_rule():
    B = 6
    # well-formed offsets are unchanged
    assert ocf.frame_ranges([0, 2, 2, 6], B).tolist() == [0, 2, 2, 6]
    # the ends are 0 and B whatever the array holds
    assert ocf.frame_ranges([4, 1, 3], B).tolist() == [0, 1, 6]
    assert ocf.frame_ranges([-3, 2, 99], B).tolist() == [0, 2, 6]
    assert ocf.frame_ranges([7, 7], B).tolist() == [0, 6]
    # in between: raised to the running maximum, clamped into [0, B]
    assert ocf.frame_ranges([0, 5, 3, 4, 6], B).tolist() == [0, 5, 5, 5, 6]
    assert ocf.frame_ranges([0, -2, 9, 1, 6], B).tolist() == [0, 0, 6, 6, 6]
    # the frames restatement of non-monotone offsets is the per-frame one with the clamped counts
    counts = [2, 1, 3]
    depth, labels, intr = synthetic.make_instance_frames(16, 32, counts, seed=9)
    bad = [5, 3, 1, 0]
    r = ocf.frame_ranges(bad, 6)
    xyz, off = ocf.backproject_frames(depth, labels, intr, bad, 6)
    want_xyz, want_off = per_frame(depth, labels, intr, np.diff(r).tolist())
    assert r.tolist() == [0, 3, 3, 6]
    assert np.array_equal(off, want_off) and np.array_equal(xyz.view(np.int32), want_xyz.view(np.int32))


def test_oracle_zero_intrinsics_give_non_finite_points():
    depth = np.ones((1, 2, 3), np.float32)
    labels = np.ones((1, 2, 3), np.int32)
    xyz, off = ocf.backproject_frames(depth, labels, [[0.0, float("nan"), 1.0, 1.0]], [0, 1], 1)
    assert off.tolist() == [0, 6] and not np.isfinite(xyz[:, :2]).any() and (xyz[:, 2] == 1).all()


def test_synthetic_frames_helper():
    depth, labels, intr = synthetic.make_instance_frames(48, 64, [2, 0, 3], seed=4)
    assert depth.shape == labels.shape == (3, 48, 64) and depth.dtype == np.float32 and labels.dtype == np.int32
    assert intr.shape == (3, 4) and len(np.unique(intr[:, 0])) == 3
    d1, l1 = synthetic.make_instance_frame(48, 64, 3, seed=6)
    assert np.array_equal(depth[2], d1) and np.array_equal(labels[2], l1)


class _Cuda(torch.Tensor):
    """A tensor that reports is_cuda: it stands in for a device tensor, so the checks after the device check run
    where no GPU exists (a check that let it through would fail in the library call, not in validation)."""
    is_cuda = True


def cu(t):
    return t.as_subclass(_Cuda)


def test_validation_before_device_work(monkeypatch):
    def no_device_work(*a, **k):
        raise AssertionError("validation let a bad argument reach the library")
    monkeypatch.setattr(_lib, "call", no_device_work)
    monkeypatch.setattr(clouds, "_backproject_frames", no_device_work)
    monkeypatch.setattr(clouds, "_sample", no_device_work)
    monkeypatch.setattr(clouds, "_upload", no_device_work)
    F, H, W = 3, 4, 5
    depth, labels = cu(torch.ones(F, H, W)), cu(torch.ones(F, H, W, dtype=torch.int32))
    intr = [(500.0, 500.0, 2.0, 2.0)] * F
    counts = [1, 0, 2]
    keys = cu(torch.arange(3))
    bp, ocf = clouds.backproject_frames, clouds.object_clouds_frames
    with pytest.raises(RuntimeError, match="no CPU path"):
        bp(torch.ones(F, H, W), labels, intr, counts)
    with pytest.raises(RuntimeError, match="no CPU path"):
        ocf(depth, labels, intr, counts, torch.arange(3))
    with pytest.raises(TypeError, match="float32"):
        bp(cu(torch.ones(F, H, W, dtype=torch.float64)), labels, intr, counts)
    with pytest.raises(TypeError, match="int32"):
        bp(depth, cu(torch.ones(F, H, W, dtype=torch.int64)), intr, counts)
    with pytest.raises(ValueError, match="3-D"):
        bp(cu(torch.ones(H, W)), cu(torch.ones(H, W, dtype=torch.int32)), intr, counts)
    with pytest.raises(ValueError, match="same shape"):
        bp(depth, cu(torch.ones(F, H, W + 1, dtype=torch.int32)), intr, counts)
    with pytest.raises(RuntimeError, match="contiguous"):
        bp(cu(torch.ones(F, W, H).transpose(1, 2)), labels, intr, counts)
    with pytest.raises(ValueError, match="at least one"):
        bp(cu(torch.ones(0, H, W)), cu(torch.ones(0, H, W, dtype=torch.int32)), [], [])
    big = torch.empty(5, 1 << 14, 1 << 14, device="meta")   # 2^30 + 2^28 pixels, no memory
    with pytest.raises(NotImplementedError, match="2\\^30"):
        bp(cu(big), cu(big.int()), [intr[0]] * 5, [1] * 5)
    many = torch.ones(clouds.MAX_FRAMES + 1, 1, 1)
    with pytest.raises(NotImplementedError, match=str(clouds.MAX_FRAMES)):
        bp(cu(many), cu(many.int()), [intr[0]] * (clouds.MAX_FRAMES + 1), [1] * (clouds.MAX_FRAMES + 1))
    # host intrinsics
    for f in range(F):
        for bad in ((0.0, 500.0, 2.0, 2.0), (500.0, 0.0, 2.0, 2.0), (float("nan"), 500.0, 2.0, 2.0),
                    (500.0, 500.0, float("inf"), 2.0), (1e300, 500.0, 2.0, 2.0), (1e-300, 500.0, 2.0, 2.0)):
            with pytest.raises(ValueError, match=f"intrinsics.*frame {f}"):
                bp(depth, labels, intr[:f] + [bad] + intr[f + 1:], counts)
    with pytest.raises(ValueError, match="\\[3, 4\\]"):
        bp(depth, labels, intr[:2], counts)
    with pytest.raises(ValueError, match="\\[3, 4\\]"):
        bp(depth, labels, intr[0], counts)
    with pytest.raises(TypeError, match="intrinsics"):
        bp(depth, labels, "fx", counts)
    # CUDA intrinsics
    with pytest.raises(TypeError, match="float32"):
        bp(depth, labels, cu(torch.ones(F, 4, dtype=torch.float64)), counts)
    with pytest.raises(ValueError, match="\\[3, 4\\]"):
        bp(depth, labels, cu(torch.ones(F, 3)), counts)
    with pytest.raises(ValueError, match="2-D"):
        bp(depth, labels, cu(torch.ones(F * 4)), counts)
    with pytest.raises(RuntimeError, match="contiguous"):
        bp(depth, labels, cu(torch.ones(4, F).t()), counts)
    # host counts
    with pytest.raises(ValueError, match="one count per frame"):
        bp(depth, labels, intr, [1, 2])
    with pytest.raises(ValueError, match=">= 0"):
        bp(depth, labels, intr, [2, -1, 2])
    with pytest.raises(TypeError, match="ints"):
        bp(depth, labels, intr, [1, 1.0, 1])
    with pytest.raises(TypeError, match="ints"):
        bp(depth, labels, intr, [1, True, 1])
    with pytest.raises(TypeError, match="sequence"):
        bp(depth, labels, intr, 3)
    with pytest.raises(ValueError, match="at least one object"):
        bp(depth, labels, intr, [0, 0, 0])
    with pytest.raises(NotImplementedError, match=str(clouds.MAX_OBJECTS)):
        bp(depth, labels, intr, [clouds.MAX_OBJECTS, 0, 1])
    with pytest.raises(ValueError, match="sums to 3 objects, expected 4"):
        bp(depth, labels, intr, counts, num_objects=4)
    with pytest.raises(ValueError, match="sums to 3 objects, expected 2"):
        ocf(depth, labels, intr, counts, cu(torch.arange(2)))
    # CUDA frame offsets
    offs = cu(torch.tensor([0, 1, 1, 3], dtype=torch.int32))
    with pytest.raises(TypeError, match="number of objects"):
        bp(depth, labels, intr, offs)
    with pytest.raises(TypeError, match="int32"):
        bp(depth, labels, intr, cu(torch.tensor([0, 1, 1, 3])), num_objects=3)
    with pytest.raises(ValueError, match="\\[4\\]"):
        bp(depth, labels, intr, cu(torch.tensor([0, 1, 3], dtype=torch.int32)), num_objects=3)
    with pytest.raises(NotImplementedError, match=str(clouds.MAX_OBJECTS)):
        bp(depth, labels, intr, offs, num_objects=clouds.MAX_OBJECTS + 1)
    with pytest.raises(ValueError, match="at least one object"):
        bp(depth, labels, intr, offs, num_objects=0)
    with pytest.raises(TypeError, match="num_objects"):
        bp(depth, labels, intr, offs, num_objects=3.0)
    # keys and points
    with pytest.raises(TypeError, match="int64"):
        ocf(depth, labels, intr, counts, cu(torch.arange(3, dtype=torch.int32)))
    with pytest.raises(TypeError, match="1-D"):
        ocf(depth, labels, intr, counts, [1, 2, 3])
    with pytest.raises(ValueError, match="num_points"):
        ocf(depth, labels, intr, counts, keys, num_points=0)
    with pytest.raises(TypeError, match="num_points"):
        ocf(depth, labels, intr, offs, keys, num_points=1024.0)


def test_c_abi_refuses_bad_arguments():
    """Status returns before any device access (the dummy pointers are never read)."""
    lib = _lib.load()
    p = ctypes.c_void_p(256)
    cap, fcap = clouds.MAX_OBJECTS, clouds.MAX_FRAMES
    wsq = lib.gp_backproject_frames_workspace_bytes
    for F, H, W, B in ((1, 480, 640, 8), (30, 720, 1280, 1024), (8, 480, 640, 1), (fcap, 32, 32, 5), (3, 1, 1, 2)):
        T = -(-H * W // 1024)
        assert wsq(F, H, W, B) == (B * T + B + F + 1) * 4, (F, H, W, B)
    # one frame: the single-frame workspace plus the F + 1 clamped offsets
    assert wsq(1, 480, 640, 8) == lib.gp_backproject_instances_workspace_bytes(480, 640, 8) + 2 * 4
    for args in ((0, 480, 640, 8), (fcap + 1, 32, 32, 8), (2, 0, 640, 8), (2, 480, -1, 8), (2, 480, 640, 0),
                 (2, 480, 640, cap + 1), (2, 1 << 15, (1 << 14) + 1, 8), (1, 1 << 15, (1 << 15) + 1, 8)):
        assert wsq(*args) == 0, args
    assert wsq(2, 1 << 15, 1 << 14, 8) > 0 and wsq(8, 1 << 12, 1 << 15, 8) > 0   # 2^30 pixels in all: the largest
    ws = wsq(4, 480, 640, 8)

    def bp(depth=p, labels=p, F=4, H=480, W=640, intr=p, foff=p, B=8, xyz=p, off=p, wsp=p, wsb=ws):
        return lib.gp_backproject_frames(depth, labels, F, H, W, intr, foff, B, xyz, off, wsp, wsb, None)

    for kw in ({"depth": None}, {"labels": None}, {"intr": None}, {"foff": None}, {"xyz": None}, {"off": None},
               {"wsp": None}):
        assert bp(**kw) == -1 and "null" in _lib.last_error(), kw
    for kw in ({"F": 0}, {"H": 0}, {"W": -3}, {"B": 0}):
        assert bp(**kw) == -1 and "bad sizes" in _lib.last_error(), kw
    assert bp(F=2, H=1 << 15, W=(1 << 14) + 1) == -1 and "too large" in _lib.last_error()
    assert bp(B=cap + 1) == -2 and str(cap) in _lib.last_error()
    assert bp(F=fcap + 1, H=1, W=1) == -2 and str(fcap) in _lib.last_error()
    assert bp(wsb=ws - 1) == -3 and "workspace" in _lib.last_error()


def test_new_entries_match_the_header():
    import os
    import re
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                               "genpose_b200.h")).read()
    assert re.search(r"GP_MAX_FRAMES = (\d+)", header).group(1) == str(clouds.MAX_FRAMES)
    lib = _lib.load()
    for name in ("gp_backproject_frames_workspace_bytes", "gp_backproject_frames"):
        assert f" {name}(" in header and name in _lib.SIGNATURES and hasattr(lib, name), name
    assert lib.gp_version() == 1
