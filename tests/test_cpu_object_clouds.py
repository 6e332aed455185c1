"""CPU: per-object point clouds from a depth frame (genpose2_b200.clouds).  The oracle's keyed permutation is a
bijection, the tiling / remainder / K == N rules and the back-projection on small hand-checked cases, every Python
validation error before any device work, and the C ABI's refusals (status returns, never an exit)."""
import ctypes

import numpy as np
import pytest
import torch

from genpose2_b200 import _lib, clouds
from oracle import object_clouds as oc
from oracle import object_noise as on


@pytest.mark.parametrize("key", [0, -1, 123456789012345])
def test_oracle_permutation_is_a_bijection_for_every_small_K(key):
    for K in range(1, 4098):
        p = oc.permutation(key, K, np.arange(K))
        assert np.array_equal(np.sort(p), np.arange(K)), K


@pytest.mark.parametrize("K", [(1 << 20) - 1, 1 << 20, (1 << 20) + 1])
def test_oracle_permutation_is_a_bijection_for_large_K(K):
    p = oc.permutation(7, K, np.arange(K))
    assert np.array_equal(np.sort(p), np.arange(K))
    assert not np.array_equal(p, np.arange(K))


def test_feistel_width_and_one_round_by_hand():
    assert [oc.feistel_bits(K) for K in (1, 2, 3, 4, 5, 16, 17, 64, 65, 300000)] == [2, 2, 2, 2, 4, 4, 6, 6, 8, 20]
    # K = 16: k = 4, halves of 2 bits, no cycle walking; the four rounds written out from Philox calls
    key, K = -5, 16
    kw = on.key_words(key)

    def F(R, r):
        return int(on.philox4x32_10(np.array([R, r, 1, 0], dtype=np.uint32), kw)[0]) & 3

    want = []
    for x in range(K):
        L, R = x >> 2, x & 3
        for r in range(4):
            L, R = R, L ^ F(R, r)
        want.append((L << 2) | R)
    assert oc.permutation(key, K, np.arange(K)).tolist() == want
    # a different key is a different permutation; the stream is not gp_object_noise's (counter word 2 = 1)
    assert oc.permutation(key + 1, 1000, np.arange(1000)).tolist() != oc.permutation(key, 1000, np.arange(1000)).tolist()


def test_sampling_rules_on_small_cases():
    key = 11
    pi = lambda K, n: oc.permutation(key, K, np.arange(n)).tolist()
    assert oc.sample_indices(key, 4, 4).tolist() == [0, 1, 2, 3]                  # K == N: unchanged
    assert oc.sample_indices(key, 1, 5).tolist() == [0] * 5                        # N % K == 0: tiles only
    assert oc.sample_indices(key, 3, 6).tolist() == [0, 1, 2, 0, 1, 2]
    got = oc.sample_indices(key, 3, 8).tolist()                                    # 2 tiles + 2 keyed points
    assert got[:6] == [0, 1, 2, 0, 1, 2] and got[6:] == pi(3, 2) and len(set(got[6:])) == 2
    got = oc.sample_indices(key, 2, 5).tolist()
    assert got == [0, 1, 0, 1, pi(2, 1)[0]]
    got = oc.sample_indices(key, 7, 3).tolist()                                    # K > N: permutation(K)[:N]
    assert got == pi(7, 3) and len(set(got)) == 3
    # ragged clouds: point ids in x, K = 0 gives zeros, offsets clamped into [0, rows]
    xyz = np.stack([np.arange(6), np.zeros(6), np.ones(6)], 1).astype(np.float32)
    pts, centre, counts = oc.sample_points(xyz, [0, 3, 3, 5, 99], [key, 1, key, 2], 4)
    assert counts.tolist() == [3, 0, 2, 1]
    assert pts[0, :3, 0].tolist() == [0, 1, 2] and pts[0, 3, 0] == pi(3, 1)[0]
    assert not pts[1].any() and not centre[1].any()
    assert pts[2, :, 0].tolist() == [3, 4, 3, 4]
    assert pts[3, :, 0].tolist() == [5] * 4 and centre[3].tolist() == [5, 0, 1]
    assert centre[2, 0] == np.float32(3.5)


def test_backprojection_on_a_hand_checked_frame():
    nan, inf = float("nan"), float("inf")
    depth = np.array([[1.0, 2.0, 0.0, 4.0],
                      [-1.0, nan, inf, 0.5]], dtype=np.float32)
    labels = np.array([[1, 2, 1, 3],
                       [1, 1, 2, 2]], dtype=np.int32)
    fx, fy, cx, cy = 2.0, 4.0, 1.0, 0.5
    xyz, off = oc.backproject_instances(depth, labels, fx, fy, cx, cy, B=2)   # label 3 is background for B = 2
    assert off.tolist() == [0, 1, 3]
    assert xyz.tolist() == [[(0 - 1) * 1.0 / 2, (0 - 0.5) * 1.0 / 4, 1.0],
                            [(1 - 1) * 2.0 / 2, (0 - 0.5) * 2.0 / 4, 2.0],
                            [(3 - 1) * 0.5 / 2, (1 - 0.5) * 0.5 / 4, 0.5]]
    xyz, off = oc.backproject_instances(depth, labels, fx, fy, cx, cy, B=3)
    assert off.tolist() == [0, 1, 3, 4] and xyz[3].tolist() == [(3 - 1) * 4.0 / 2, (0 - 0.5) * 4.0 / 4, 4.0]


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
    monkeypatch.setattr(clouds, "_backproject", no_device_work)
    monkeypatch.setattr(clouds, "_sample", no_device_work)
    H, W = 4, 5
    depth, labels = cu(torch.ones(H, W)), cu(torch.ones(H, W, dtype=torch.int32))
    intr = (500.0, 500.0, 2.0, 2.0)
    keys = cu(torch.arange(3))
    bp, oc_ = clouds.backproject_instances, clouds.object_clouds
    with pytest.raises(RuntimeError, match="no CPU path"):
        bp(torch.ones(H, W), labels, intr, 3)
    with pytest.raises(RuntimeError, match="no CPU path"):
        oc_(depth, labels, intr, torch.arange(3))
    with pytest.raises(TypeError, match="float32"):
        bp(cu(torch.ones(H, W, dtype=torch.float64)), labels, intr, 3)
    with pytest.raises(TypeError, match="int32"):
        bp(depth, cu(torch.ones(H, W, dtype=torch.int64)), intr, 3)
    with pytest.raises(ValueError, match="2-D"):
        bp(cu(torch.ones(1, H, W)), labels, intr, 3)
    with pytest.raises(ValueError, match="same shape"):
        bp(depth, cu(torch.ones(H, W + 1, dtype=torch.int32)), intr, 3)
    with pytest.raises(RuntimeError, match="contiguous"):
        bp(cu(torch.ones(W, H).t()), labels, intr, 3)
    for bad in ((0.0, 500.0, 2.0, 2.0), (500.0, 0.0, 2.0, 2.0), (float("nan"), 500.0, 2.0, 2.0),
                (500.0, 500.0, float("inf"), 2.0), (1e300, 500.0, 2.0, 2.0), (1e-300, 500.0, 2.0, 2.0)):
        with pytest.raises(ValueError, match="intrinsics"):
            bp(depth, labels, bad, 3)
    with pytest.raises(ValueError, match="four"):
        bp(depth, labels, (500.0, 500.0, 2.0), 3)
    with pytest.raises(TypeError, match="intrinsics"):
        bp(depth, labels, "fx", 3)
    with pytest.raises(TypeError, match="host"):
        bp(depth, labels, cu(torch.tensor(intr)), 3)
    with pytest.raises(ValueError, match="num_objects"):
        bp(depth, labels, intr, 0)
    with pytest.raises(TypeError, match="num_objects"):
        bp(depth, labels, intr, 2.0)
    with pytest.raises(NotImplementedError, match=str(clouds.MAX_OBJECTS)):
        bp(depth, labels, intr, clouds.MAX_OBJECTS + 1)
    with pytest.raises(NotImplementedError, match=str(clouds.MAX_OBJECTS)):
        oc_(depth, labels, intr, cu(torch.arange(clouds.MAX_OBJECTS + 1)))
    with pytest.raises(TypeError, match="int64"):
        oc_(depth, labels, intr, cu(torch.arange(3, dtype=torch.int32)))
    with pytest.raises(TypeError, match="1-D"):
        oc_(depth, labels, intr, [1, 2, 3])
    with pytest.raises(ValueError, match="num_points"):
        oc_(depth, labels, intr, keys, num_points=0)
    # stage B
    xyz, off = cu(torch.zeros(10, 3)), cu(torch.tensor([0, 4, 6, 10], dtype=torch.int32))
    sp = clouds.sample_points
    with pytest.raises(RuntimeError, match="no CPU path"):
        sp(torch.zeros(10, 3), off, keys=keys)
    with pytest.raises(RuntimeError, match="no CPU path"):
        sp(xyz, off, keys=torch.arange(3))
    with pytest.raises(ValueError, match=r"\[rows, 3\]"):
        sp(cu(torch.zeros(10, 4)), off, keys=keys)
    with pytest.raises(TypeError, match="int32"):
        sp(xyz, cu(torch.tensor([0, 4, 6, 10])), keys=keys)
    with pytest.raises(ValueError, match="B \\+ 1"):
        sp(xyz, cu(torch.tensor([0], dtype=torch.int32)), keys=cu(torch.arange(0)))
    with pytest.raises(ValueError, match="shape"):
        sp(xyz, off, keys=cu(torch.arange(4)))
    with pytest.raises(TypeError, match="int64"):
        sp(xyz, off, keys=cu(torch.arange(3).float()))
    with pytest.raises(TypeError, match="None"):
        sp(xyz, off, keys=None)
    with pytest.raises(ValueError, match="num_points"):
        sp(xyz, off, -1, keys=keys)
    with pytest.raises(TypeError, match="num_points"):
        sp(xyz, off, 1024.0, keys=keys)


def test_c_abi_refuses_bad_arguments():
    """Status returns before any device access (the dummy pointers are never read)."""
    lib = _lib.load()
    p = ctypes.c_void_p(256)
    cap = 1024
    ws = lib.gp_backproject_instances_workspace_bytes(480, 640, 8)
    assert ws >= 8 * 4 * 300
    assert lib.gp_backproject_instances_workspace_bytes(480, 640, cap) > 0
    assert lib.gp_backproject_instances_workspace_bytes(480, 640, cap + 1) == 0
    assert lib.gp_backproject_instances_workspace_bytes(0, 640, 8) == 0
    assert lib.gp_backproject_instances_workspace_bytes(480, 640, 0) == 0
    assert lib.gp_backproject_instances_workspace_bytes(1 << 16, 1 << 16, 8) == 0
    assert lib.gp_backproject_instances_workspace_bytes(1 << 15, 1 << 15, 8) > 0        # 2^30 pixels: the largest frame
    assert lib.gp_backproject_instances_workspace_bytes(1 << 15, (1 << 15) + 1, 8) == 0

    def bp(depth=p, labels=p, H=480, W=640, fx=500.0, fy=500.0, cx=320.0, cy=240.0, B=8, xyz=p, off=p, wsp=p,
           wsb=ws):
        return lib.gp_backproject_instances(depth, labels, H, W, fx, fy, cx, cy, B, xyz, off, wsp, wsb, None)

    for kw in ({"depth": None}, {"labels": None}, {"xyz": None}, {"off": None}, {"wsp": None}):
        assert bp(**kw) == -1 and "null" in _lib.last_error(), kw
    assert bp(H=0) == -1 and "bad sizes" in _lib.last_error()
    assert bp(W=-3) == -1 and "bad sizes" in _lib.last_error()
    assert bp(B=0) == -1 and "bad sizes" in _lib.last_error()
    assert bp(H=1 << 16, W=1 << 16) == -1 and "too large" in _lib.last_error()
    assert bp(H=1 << 15, W=(1 << 15) + 1) == -1 and "too large" in _lib.last_error()
    assert bp(B=cap + 1) == -2 and str(cap) in _lib.last_error()
    assert bp(fx=0.0) == -1 and "intrinsics" in _lib.last_error()
    assert bp(fy=float("nan")) == -1 and "intrinsics" in _lib.last_error()
    assert bp(cx=float("inf")) == -1 and "intrinsics" in _lib.last_error()
    assert bp(wsb=ws - 1) == -3 and "workspace" in _lib.last_error()

    def sp(xyz=p, rows=100, off=p, keys=p, B=4, N=1024, pts=p, ctr=p, cnt=p):
        return lib.gp_sample_points(xyz, rows, off, keys, B, N, pts, ctr, cnt, None)

    for kw in ({"xyz": None}, {"off": None}, {"keys": None}, {"pts": None}, {"ctr": None}, {"cnt": None}):
        assert sp(**kw) == -1 and "null" in _lib.last_error(), kw
    assert sp(B=0) == -1 and "bad sizes" in _lib.last_error()
    assert sp(N=0) == -1 and "bad sizes" in _lib.last_error()
    assert sp(rows=-1) == -1 and "bad sizes" in _lib.last_error()


def test_new_entries_match_the_header():
    import os
    import re
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                               "genpose_b200.h")).read()
    assert re.search(r"GP_MAX_FRAME_OBJECTS = (\d+)", header).group(1) == str(clouds.MAX_OBJECTS)
    assert 1 << int(re.search(r"GP_MAX_FRAME_PIXELS = 1 << (\d+)", header).group(1)) == clouds.MAX_PIXELS
    lib = _lib.load()
    for name in ("gp_backproject_instances_workspace_bytes", "gp_backproject_instances", "gp_sample_points"):
        assert f" {name}(" in header and name in _lib.SIGNATURES and hasattr(lib, name), name
    assert lib.gp_version() == 1
