"""CPU: the C-ABI library loads and exports every symbol include/genpose_b200.h declares (no
compute without a GPU), the host mirror has the reference's state-dict layout and config keys,
unsupported configurations raise instead of falling back, and the multi-GPU sharding logic works
over gloo with world_size 2."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from genpose2_b200 import _lib
    header = open(os.path.join(ROOT, "include", "genpose_b200.h")).read()
    declared = set(re.findall(r"GP_API [^;(]*?\b(gp_[a-z0-9_]+)\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    lib2 = _lib.load()
    assert lib2.gp_version() == 1
    assert lib2.gp_trunk_packed_bytes() > 4 * (768 * 1024 + 256 * 768)
    assert lib2.gp_scorenet_ode_workspace_bytes(3200) >= 9 * 3200 * 9 * 8


def test_ctypes_signatures_have_the_declared_arity():
    """ABI drift guard: every prototype in the header has as many parameters as its ctypes signature."""
    from genpose2_b200 import _lib
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "genpose_b200.h")).read(), flags=re.S)
    protos = re.findall(r"GP_API [^;(]*?\b(gp_[a-z0-9_]+)\(([^;]*?)\);", header, flags=re.S)
    assert len(protos) == len(_lib.SIGNATURES)
    for name, params in protos:
        params = params.strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert n == len(_lib.SIGNATURES[name][1]), (name, n, len(_lib.SIGNATURES[name][1]))


def test_bad_arguments_return_status_not_exit():
    from genpose2_b200 import _lib
    lib = _lib.load()
    rc = lib.gp_fps(None, 1, 16, 4, None, None, None)
    assert rc == -1 and b"null" in lib.gp_last_error()
    rc = lib.gp_aggregate(ctypes.c_void_p(8), ctypes.c_void_p(8), 1, 100, 20, 1, 0.05, 3, ctypes.c_void_p(8), None, None, None)
    assert rc == -1 and b"R=100" in lib.gp_last_error()


def test_cpu_tensors_are_rejected_no_fallback():
    from genpose2_b200 import pointnet2_utils as pu
    with pytest.raises(RuntimeError, match="no CPU path"):
        pu.furthest_point_sample(torch.randn(1, 8, 3), 2)
    with pytest.raises(RuntimeError, match="no CPU path"):
        pu.ball_query(0.1, 4, torch.randn(1, 8, 3), torch.randn(1, 2, 3))


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    from genpose2_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU / PyTorch fallback"):
        _lib.load()


def test_state_dict_layout_matches_reference_layout():
    """the synthetic state dicts were loaded with strict load_state_dict into the REFERENCE modules
    by tests/golden/make_golden.py; here the same dicts must load strictly into the mirror."""
    from genpose2_b200 import synthetic
    from genpose2_b200.config import get_config
    from genpose2_b200.posenet import GFObjectPose
    from genpose2_b200.scalenet import ScaleNet
    from genpose2_b200.sde import init_sde
    cfg = get_config()
    cfg.device = "cpu"
    for agent_type in ("score", "energy"):
        cfg.agent_type = agent_type
        net = GFObjectPose(cfg, *init_sde("ve"))
        sd = synthetic.random_gfobjectpose_state_dict(1)
        assert set(net.state_dict().keys()) == set(sd.keys())
        net.load_state_dict(sd, strict=True)
        assert sum(p.numel() for p in net.parameters()) == 3776937  # SURVEY.md 8(c) probe
    sn = ScaleNet(1024, 0, 180)
    sn.load_state_dict(synthetic.random_scalenet_state_dict(2), strict=True)
    assert sum(p.numel() for p in sn.parameters()) == 440835


def test_config_keys_and_unsupported_modes_raise():
    from genpose2_b200.config import get_config
    from genpose2_b200.posenet import GFObjectPose
    from genpose2_b200.sde import init_sde
    cfg = get_config()
    for key, val in dict(pose_mode="rot_matrix", sde_mode="ve", regression_head="Rx_Ry_and_T", pts_encoder="pointnet2",
                         energy_mode="IP", s_theta_mode="score", norm_energy="identical", scale_embedding=180,
                         num_points=1024, eval_repeat_num=50, retain_ratio=0.4, clustering=1, clustering_eps=0.05,
                         clustering_minpts=0.1667, seed=0, T0=1.0).items():
        assert getattr(cfg, key) == val, key
    assert get_config(["--T0", "0.55", "--sampler_mode", "ode"]).T0 == 0.55
    with pytest.raises(NotImplementedError):
        init_sde("vp")
    cfg.device = "cpu"
    for key, bad in (("dino", "pointwise"), ("pts_encoder", "pointnet"), ("regression_head", "RT"), ("pose_mode", "quat_wxyz")):
        c = get_config()
        c.device = "cpu"
        setattr(c, key, bad)
        with pytest.raises(NotImplementedError):
            GFObjectPose(c, *init_sde("ve"))
    c = get_config()
    c.device = "cpu"
    c.agent_type = "energy"
    c.energy_mode = "L2"
    with pytest.raises(NotImplementedError):
        GFObjectPose(c, *init_sde("ve"))


def test_sde_matches_oracle():
    from genpose2_b200 import sde
    from oracle import pose_oracle as po
    prior, marg, sde_fn, eps, T = sde.init_sde("ve")
    assert eps == 1e-5 and T == 1.0
    t = torch.tensor([[0.3], [0.9]])
    assert torch.equal(marg(None, t)[1], po.ve_marginal_std(t))
    assert torch.equal(sde_fn(t)[1], po.ve_sde(t)[1])
    torch.manual_seed(3)
    a = prior((4, 9), T=0.55)
    torch.manual_seed(3)
    assert torch.equal(a, po.ve_prior((4, 9), T=0.55))


def test_shard_range_partitions_contiguously():
    from genpose2_b200.pipeline import shard_range
    for n in (0, 1, 7, 64, 8192, 8191):
        for w in (1, 2, 3, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["GP_ROOT"])
from genpose2_b200.pipeline import gather_results, shard_range
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["GP_PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world = dist.get_rank(), dist.get_world_size()
B = 7  # ragged: 4 + 3
lo, hi = shard_range(B, rank, world)
g = torch.Generator().manual_seed(0)
pose_full = torch.randn(B, 4, 4, generator=g); length_full = torch.randn(B, 3, generator=g)
pose, length = gather_results(pose_full[lo:hi].clone(), length_full[lo:hi].clone())
assert torch.equal(pose, pose_full) and torch.equal(length, length_full), (rank, pose.shape)
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_gather_results_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", GP_PORT=str(port), GP_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0, out.decode()


def test_oracle_pointnet2_matches_bruteforce_numpy():
    """the C restatement itself: FPS against a direct numpy transcription for a power-of-two N
    without ties (where the tree tie-break cannot matter), ball query against a brute-force scan."""
    import numpy as np
    from oracle import pointnet2_oracle as pn
    rng = np.random.default_rng(0)
    xyz = rng.normal(size=(2, 256, 3)).astype(np.float32)
    idx = pn.furthest_point_sample(xyz, 40)
    for b in range(2):
        d = np.full(256, 1e10, np.float32)
        cur = 0
        for j in range(1, 40):
            diff = xyz[b] - xyz[b, cur]
            dist = (diff[:, 1] * diff[:, 1]).astype(np.float32)
            dist = (diff[:, 0].astype(np.float64) * diff[:, 0] + dist).astype(np.float32)  # one fma
            dist = (diff[:, 2].astype(np.float64) * diff[:, 2] + dist).astype(np.float32)
            d = np.minimum(d, dist)
            cur = int(np.argmax(d))
            assert idx[b, j] == cur
    new_xyz = np.take_along_axis(xyz, idx[..., None].astype(np.int64), 1)
    bq = pn.ball_query(0.9, 6, xyz, new_xyz)
    for b in range(2):
        for i in range(40):
            diff = new_xyz[b, i] - xyz[b]
            d2 = (diff ** 2).sum(1)
            hits = np.nonzero(d2 < np.float32(0.9) ** 2 * 0.999)[0]
            got = bq[b, i]
            n = min(len(hits), 6)
            assert set(got[:n]) <= set(np.nonzero(d2 < np.float32(0.9) ** 2 * 1.001)[0])
            assert (got[n:] == got[0]).all() or len(hits) >= 6
    assert pn.fps_block_size(1000) == 512 and pn.fps_block_size(1024) == 1024 and pn.fps_block_size(5000) == 1024


def test_stage_files_are_plain_pickles_in_the_reference_layout(tmp_path):
    """SURVEY 8 f4: what evaluation_single.py:120,157,219,254 dump and :127,164-167,226-228 load"""
    import pickle
    from genpose2_b200 import stage_io
    g = torch.Generator().manual_seed(0)
    poses = [torch.randn(3, 50, 9, generator=g, dtype=torch.float64), torch.randn(2, 50, 9, generator=g, dtype=torch.float64)]
    feats = [torch.randn(3, 1024, generator=g), torch.randn(2, 1024, generator=g)]
    energy = [torch.randn(3, 50, 2, generator=g), torch.randn(2, 50, 2, generator=g)]
    agg = [torch.eye(4).repeat(3, 1, 1), torch.eye(4).repeat(2, 1, 1)]
    length = [torch.rand(3, 3, generator=g), torch.rand(2, 3, generator=g)]
    p = stage_io.stage_paths(str(tmp_path / "run"), "score.pth", "energy.pth", "scale.pth")
    p = {k: str(tmp_path / v) for k, v in p.items()}
    stage_io.save_score_stage(p["score"], poses, feats)
    stage_io.save_energy_stage(p["energy"], energy)
    stage_io.save_aggregate_stage(p["aggregate"], agg)
    stage_io.save_scale_stage(p["scale"], agg, length)
    # read them back exactly as the reference does
    all_pred_pose, all_score_feature = pickle.load(open(p["score"], "rb"))
    assert len(all_pred_pose) == 2 and all_pred_pose[0].dtype == torch.float64 and tuple(all_pred_pose[1].shape) == (2, 50, 9)
    assert set(all_score_feature[0]) == {"pts_feat", "rgb_feat"} and all_score_feature[0]["rgb_feat"] is None
    assert torch.equal(all_score_feature[1]["pts_feat"], feats[1])
    all_pred_energy = pickle.load(open(p["energy"], "rb"))
    assert torch.equal(all_pred_energy[0], energy[0])
    assert torch.equal(pickle.load(open(p["aggregate"], "rb"))[1], agg[1])
    a2, l2 = pickle.load(open(p["scale"], "rb"))
    assert torch.equal(a2[0], agg[0]) and torch.equal(l2[1], length[1])
    # the runner's fallback box size (evaluation_single.py:232-250) against its own formulation
    pcl = torch.randn(3, 64, 3, generator=g)
    pose = torch.eye(4).repeat(3, 1, 1)
    q, _ = torch.linalg.qr(torch.randn(3, 3, 3, generator=g))
    pose[:, :3, :3] = q
    pose[:, :3, 3] = torch.randn(3, 3, generator=g)
    rot_t = torch.repeat_interleave(pose[:, :3, :3].transpose(1, 2), 64, dim=0)
    want = 2 * torch.bmm(rot_t, (pcl - pose[:, :3, 3].unsqueeze(1)).reshape(-1, 3, 1)).reshape(-1, 64, 3).abs().max(dim=1)[0]
    assert torch.allclose(stage_io.bbox_length_from_points(pcl, pose), want, atol=1e-6)


def test_load_ckpt_reads_a_checkpoint_written_by_the_reference(tmp_path):
    """SURVEY 8 row f4: PoseNet.load_ckpt (posenet_agent.py:171-203) on a file produced by the REFERENCE's own
    PoseNet.save_ckpt (posenet_agent.py:141-169: torch.save of {clock, model_state_dict, optimizer_state_dict,
    scheduler_state_dict} after the EMA copy) -- for the score, energy and scale agents."""
    from oracle import ref_shim
    if not ref_shim.available():
        pytest.skip("reference modules not available (neither /root/reference nor oracle/_ref/refpkg)")
    import copy
    from genpose2_b200 import synthetic
    from genpose2_b200.config import get_config
    from genpose2_b200.posenet_agent import PoseNet
    ns = ref_shim.load()
    for kind, sd in (("score", synthetic.random_gfobjectpose_state_dict(100)),
                     ("energy", synthetic.random_gfobjectpose_state_dict(200)),
                     ("scale", synthetic.random_scalenet_state_dict(300))):
        rcfg = copy.copy(ns.cfg)
        rcfg.device, rcfg.agent_type = "cpu", kind
        ref_agent = ns.posenet_agent.PoseNet(rcfg)
        ref_agent.net.load_state_dict(sd)
        # save_ckpt stores the EMA shadow (initialised from the construction-time weights): refresh it like a
        # training step would have, so that the file holds the weights loaded above
        ref_agent.ema = type(ref_agent.ema)(ref_agent.net.parameters(), decay=rcfg.ema_rate)
        ref_agent.model_dir = str(tmp_path)
        ref_agent.save_ckpt(name=f"ckpt_{kind}")
        path = tmp_path / f"ckpt_{kind}.pth"
        assert path.exists()
        cfg = get_config()
        cfg.device, cfg.agent_type = "cpu", kind
        agent = PoseNet(cfg)
        agent.load_ckpt(model_dir=str(path), model_path=True, load_model_only=True)
        got = agent.net.state_dict()
        want = ref_agent.net.state_dict()
        assert set(got.keys()) == set(want.keys())
        for k in want:
            assert torch.equal(got[k].cpu(), want[k].cpu()), k
            if k in sd:
                assert torch.equal(got[k].cpu(), sd[k]), k


def test_aggregation_limits_raise_instead_of_misbehaving():
    """ADVICE r1: the aggregation kernel's caps (64 hypotheses, 32 retained with clustering) and DBSCAN's
    min_samples >= 1 are enforced loudly on the Python side, before any device work."""
    from genpose2_b200.aggregation import aggregate_pose, sort_poses_by_energy
    poses = torch.zeros(2, 80, 9, dtype=torch.float64)
    energy = torch.zeros(2, 80, 2)
    with pytest.raises(NotImplementedError):
        sort_poses_by_energy(poses, energy)
    with pytest.raises(NotImplementedError):
        aggregate_pose(poses[:, :64], energy[:, :64], eval_repeat_num=64, retain_ratio=0.75)   # 48 retained, clustering on
    with pytest.raises(ValueError):
        aggregate_pose(poses[:, :50], energy[:, :50], eval_repeat_num=50, retain_ratio=0.1)    # int(0.1667 * 5) = 0


def test_trajectory_buffer_is_bounded_by_a_byte_budget():
    """return_trajectory=True records accepted steps into [slots, N, 9] f64: 512 slots for small batches, capped by
    TRAJ_BYTES_BUDGET for large ones (15 GB at 8192 x 50 rows in round 1), never below 64 slots"""
    from genpose2_b200 import samplers
    assert samplers._traj_slots(50) == samplers.MAX_TRAJ
    n = 8192 * 50
    slots = samplers._traj_slots(n)
    assert 64 <= slots < samplers.MAX_TRAJ and slots * n * 72 <= samplers.TRAJ_BYTES_BUDGET + 64 * n * 72
    assert samplers._traj_slots(10 ** 9) == 64


def test_bench_rejects_zero_timed_steps():
    """bench.py refuses, before any work, a run with no timed step"""
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert run.returncode == 2 and "--steps" in run.stderr, run.stderr


def test_bench_reference_arm_runs_every_step_and_dumps_the_last(tmp_path):
    """bench.py --impl reference times exactly --steps steps, and --dump-outputs writes what the last one returned:
    the CPU path on the bench's first cloud with the prior noise drawn after torch.manual_seed(1)"""
    import json
    import numpy as np
    from genpose2_b200 import synthetic
    from oracle import pose_oracle as po
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--ref_objects", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True)
    assert run.returncode == 0, run.stderr[-3000:]
    line = json.loads([s for s in run.stdout.splitlines() if s.startswith("{")][-1])
    assert line["steps"] == line["steps_timed"] == 2
    pose, length = np.load(tmp_path / "aggregated_pose.npy"), np.load(tmp_path / "length.npy")
    assert pose.dtype == length.dtype == np.float32 and pose.shape == (1, 4, 4) and length.shape == (1, 3)
    if line["cpu_baseline"]["kind"] != "port":
        return   # the reference's own modules computed it: compared with the port by tests/test_gpu_reference.py
    pts, center = synthetic.make_point_clouds(1, 1024, seed=0)
    threads = torch.get_num_threads()
    torch.set_num_threads(os.cpu_count() or 1)   # the bench's setting: torch-CPU sums in a thread-count-dependent order
    try:
        torch.manual_seed(1)
        noise = po.ve_prior((50, 9), T=0.55)
        want = po.full_pipeline(synthetic.random_gfobjectpose_state_dict(100), synthetic.random_gfobjectpose_state_dict(200),
                                synthetic.random_scalenet_state_dict(300), pts, center, noise, repeat_num=50, T0=0.55,
                                integrator="scipy")
    finally:
        torch.set_num_threads(threads)
    np.testing.assert_array_equal(pose, want["aggregated_pose"].float().numpy())
    np.testing.assert_array_equal(length, want["length"].float().numpy())
