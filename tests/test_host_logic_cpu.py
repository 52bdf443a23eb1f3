"""CPU: host-side logic — BN folding / weight packing, hypothesis grid, sharding arithmetic, the world_size-2 gather
and the whole sharded register over gloo (host-side engine double), the replica pool's scheduling."""
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from foundationpose_b200 import hypotheses, packing, synth
from foundationpose_b200.engine import pack_network
from foundationpose_b200.parallel import gather_rows, shard_bounds, shard_counts
from foundationpose_b200.weights import random_state_dict


def test_fold_bn_equals_conv_then_bn():
    torch.manual_seed(0)
    conv = nn.Conv2d(8, 16, 3, padding=1)
    bn = nn.BatchNorm2d(16).eval()
    bn.running_mean.normal_(0, 0.2)
    bn.running_var.uniform_(0.5, 1.5)
    bn.weight.data.uniform_(0.5, 1.5)
    bn.bias.data.normal_(0, 0.2)
    x = torch.randn(2, 8, 10, 10)
    w, b = packing.fold_bn(conv.weight, conv.bias, dict(weight=bn.weight, bias=bn.bias, running_mean=bn.running_mean,
                                                          running_var=bn.running_var, eps=bn.eps))
    with torch.no_grad():
        ref = bn(conv(x))
        got = torch.nn.functional.conv2d(x, w, b, padding=1)
    assert (ref - got).abs().max() < 1e-5


def test_pack_layouts():
    w = torch.arange(2 * 3 * 3 * 3, dtype=torch.float32).reshape(2, 3, 3, 3)
    p = packing.pack_conv3(w)
    assert p.shape == (2, 27) and p.dtype == torch.float16
    # K order (r, s, c)
    assert float(p[1, (1 * 3 + 2) * 3 + 1]) == float(w[1, 1, 1, 2])
    w7 = torch.randn(4, 6, 7, 7)
    p7 = packing.pack_conv7(w7).float()  # [r][s][e][co][c], tap = 2s + e
    assert p7.shape == (7, 4, 2, 4, 8)
    taps = p7.reshape(7, 8, 4, 8)
    assert torch.allclose(taps[:, :7, :, :6], w7.permute(2, 3, 0, 1).half().float())
    assert taps[:, 7].abs().max() == 0 and taps[..., 6:].abs().max() == 0
    x = torch.rand(2, 6, 160, 160)
    xp = packing.pad_image_c8(x)
    assert xp.shape == (2, 166, 2, 84, 8)
    canvas = packing.unpad_image_c8(xp)
    assert torch.equal(canvas[:, 3:163, 3:163, :6], x.permute(0, 2, 3, 1).half())
    assert canvas[:, :3].abs().max() == 0 and canvas[..., 6:].abs().max() == 0
    # even columns first, then odd columns: padded column 3 (image column 0) is odd, pair 1
    assert torch.equal(xp[:, 3, 1, 1, :6], x[:, :, 0, 0].half())


def test_pack_network_names_and_shapes():
    r = pack_network(random_state_dict("refine", 0), "refine")
    assert r["enc.0.w"].shape == (7, 4, 2, 64, 8) and r["enc.14.w"].shape == (512, 4608) and r["heads.in_w"].shape == (3072, 512)
    assert r["pe"].shape == (400, 512) and r["head1.fin_w"].shape == (3, 512)
    s = pack_network(random_state_dict("score", 0), "score")
    assert s["cross.in_w"].dtype == np.float32 and s["att.in_w"].dtype == np.float16 and s["lin.w"].shape == (512,)
    # use_BN = False checkpoints fold to the plain conv
    sd = random_state_dict("refine", 0, use_bn=False)
    r2 = pack_network(sd, "refine")
    assert np.allclose(r2["enc.1.b"], sd["encodeA.1.net.0.bias"].numpy())


def test_rotation_grid_is_252_rigid_poses():
    g = hypotheses.make_rotation_grid()
    assert g.shape == (252, 4, 4)
    R = g[:, :3, :3]
    assert np.allclose(R @ R.transpose(0, 2, 1), np.eye(3)[None], atol=1e-5)
    assert np.allclose(np.linalg.det(R), 1, atol=1e-5)
    # a 2-fold symmetry about z halves the in-plane set
    sym = np.stack([np.eye(4), np.diag([-1.0, -1.0, 1.0, 1.0])])
    assert len(hypotheses.make_rotation_grid(symmetry_tfs=sym)) < 252


def test_guess_translation_edge_cases():
    K = synth.DEFAULT_K
    depth = np.full((480, 640), 0.7, dtype=np.float32)
    mask = np.zeros((480, 640), dtype=bool)
    assert np.array_equal(hypotheses.guess_translation(depth, mask, K), np.zeros(3))
    mask[100:200, 300:400] = True
    t = hypotheses.guess_translation(depth, mask, K)
    assert abs(t[2] - 0.7) < 1e-6 and abs(t[0] - (349.5 - 320) / 615 * 0.7) < 1e-6
    depth[:] = 0
    assert np.array_equal(hypotheses.guess_translation(depth, mask, K), np.zeros(3))


def test_shard_bounds():
    assert shard_counts(252, 8) == [32, 32, 32, 32, 31, 31, 31, 31]
    assert shard_counts(252, 1) == [252]
    assert shard_counts(3, 8) == [1, 1, 1, 0, 0, 0, 0, 0]
    cover = []
    for r in range(4):
        lo, hi = shard_bounds(253, 4, r)
        cover += list(range(lo, hi))
    assert cover == list(range(253))


def _gather_worker(rank, world, n_total, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    full = torch.arange(n_total * 5, dtype=torch.float32).reshape(n_total, 5)
    lo, hi = shard_bounds(n_total, world, rank)
    out = gather_rows(full[lo:hi].clone(), n_total)
    q.put((rank, torch.equal(out, full)))
    dist.destroy_process_group()


def test_gather_rows_world2_gloo():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    for n_total in (252, 7):
        q = ctx.Queue()
        port = 29400 + n_total % 50
        procs = [ctx.Process(target=_gather_worker, args=(r, 2, n_total, port, q)) for r in range(2)]
        for p in procs:
            p.start()
        res = [q.get(timeout=120) for _ in procs]
        for p in procs:
            p.join(timeout=60)
        assert all(ok for _, ok in res), res


class _HostEngine:
    """Test double for engine.Engine: same three entry points ShardedRegister drives, computed on the host with a
    per-hypothesis refine / featurise step and a tail that couples ALL hypotheses (like att_cross,
    score_network.py:84-88) — so a wrong shard order, a dropped row or a rank-dependent tail shows up in the result."""
    tensor_device = "cpu"

    def refine(self, poses, iterations):
        out = poses.clone()
        for _ in range(iterations):
            out[:, :3, 3] += 0.01 * torch.tanh(out[:, :3, :3].sum(-1))
        return out, None, None

    def score_features(self, poses):
        g = torch.Generator().manual_seed(0)
        W = torch.randn(16, 512, generator=g)
        # row by row: the same vector-matrix product whatever the shard height (bit-exact comparison below)
        return torch.stack([torch.sin(r @ W) for r in poses.reshape(-1, 16)]) if len(poses) else poses.new_zeros(0, 512)

    def score_tail(self, feats):
        att = torch.softmax(feats @ feats.T / 512 ** 0.5, dim=-1)
        scores = (att @ feats).sum(-1) + 100.0
        return scores, scores.argmax().reshape(1).to(torch.int32)


def _sharded_worker(rank, world, n_total, port, q):
    import torch.distributed as dist

    from foundationpose_b200.parallel import ShardedRegister

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(1)
    poses = torch.eye(4).repeat(n_total, 1, 1) + 0.1 * torch.randn(n_total, 4, 4)
    sr = ShardedRegister(_HostEngine())
    outs = [sr.run(poses, 3) for _ in range(2)]  # twice: the second call reuses the cached gather workspaces
    q.put((rank, [tuple(t.clone().numpy() for t in o) for o in outs]))
    dist.destroy_process_group()


def test_sharded_register_world2_gloo_matches_single_process():
    """SURVEY 8e: shard -> refine + featurise locally -> ONE gather -> identical tail on every rank.  Both ranks must
    return the single-process result bit for bit, for even, ragged and empty shards."""
    import torch.multiprocessing as mp

    from foundationpose_b200.parallel import ShardedRegister

    ctx = mp.get_context("spawn")
    for n_total in (8, 7, 1):
        torch.manual_seed(1)
        poses = torch.eye(4).repeat(n_total, 1, 1) + 0.1 * torch.randn(n_total, 4, 4)
        ref = [t.numpy() for t in ShardedRegister(_HostEngine()).run(poses, 3)]
        q = ctx.Queue()
        port = 29470 + n_total
        procs = [ctx.Process(target=_sharded_worker, args=(r, 2, n_total, port, q)) for r in range(2)]
        for p in procs:
            p.start()
        res = dict(q.get(timeout=120) for _ in procs)
        for p in procs:
            p.join(timeout=60)
        assert sorted(res) == [0, 1]
        for rank, outs in res.items():
            for o in outs:
                for got, want in zip(o, ref):
                    assert np.array_equal(got, want), (n_total, rank)


class _HostEstimator:
    """Test double for FoundationPose inside replicas.ReplicaPool: records what it is asked and answers with a pose
    that encodes (frame tag, object tag); slow on one replica so that the dynamic scheduling is exercised."""
    log = []

    def __init__(self, device, model_pts, model_normals, mesh, symmetry_tfs):
        self.device, self.obj = device, mesh
        _HostEstimator.log.append(("build", device, mesh))

    def reset_object(self, model_pts, model_normals, symmetry_tfs=None, mesh=None):
        self.obj = mesh
        _HostEstimator.log.append(("reset", self.device, mesh))

    def register(self, K, rgb, depth, ob_mask, iteration):
        import time

        if rgb == "bad":
            raise RuntimeError("frame could not be processed")
        time.sleep(0.02 if self.device == 0 else 0.002)
        pose = np.eye(4)
        pose[0, 3], pose[1, 3], pose[2, 3] = rgb, self.obj, iteration
        _HostEstimator.log.append(("register", self.device, rgb))
        return pose


def test_replica_pool_scheduling_order_and_errors():
    """SURVEY 8f N3 host logic: one estimator per replica, frames handed out dynamically, results in input order, every
    replica re-targeted by reset_object, a failing frame surfaces as the caller's exception (run_ycb_video.py:116-121 is
    the sequential loop this replaces)."""
    from foundationpose_b200.replicas import ReplicaPool

    _HostEstimator.log = []
    pool = ReplicaPool([0, 1, 2], make_estimator=_HostEstimator)
    try:
        for obj in (11, 12):
            pool.reset_object(None, None, mesh=obj)
            frames = [(None, i, None, None) for i in range(40)]
            poses = pool.register_many(frames, iteration=5)
            assert [int(p[0, 3]) for p in poses] == list(range(40))  # input order
            assert all(int(p[1, 3]) == obj and int(p[2, 3]) == 5 for p in poses)  # every replica saw the reset
        builds = [e for e in _HostEstimator.log if e[0] == "build"]
        resets = [e for e in _HostEstimator.log if e[0] == "reset"]
        assert sorted(d for _, d, _ in builds) == [0, 1, 2] and sorted(d for _, d, _ in resets) == [0, 1, 2]
        per_dev = {d: sum(1 for e in _HostEstimator.log if e[0] == "register" and e[1] == d) for d in (0, 1, 2)}
        assert sum(per_dev.values()) == 80 and sum(1 for v in per_dev.values() if v) >= 2
        assert per_dev[0] < max(per_dev[1], per_dev[2])  # dynamic scheduling: the slow replica did not take an equal share
        assert pool.register_many([]) == []
        with pytest.raises(RuntimeError, match="could not be processed"):
            pool.register_many([(None, 0, None, None), (None, "bad", None, None), (None, 2, None, None)])
        # the pool survives a failed frame
        assert int(pool.register_many([(None, 7, None, None)])[0][0, 3]) == 7
    finally:
        pool.close()
    assert not any(w.is_alive() for w in pool.workers)


def test_meshprep_diameter_and_voxel_downsample():
    """reset_object helpers (estimater.py:43-64, Utils.py:559-574) without open3d: exact diameter, voxel means."""
    from foundationpose_b200 import meshprep, synth

    rng = np.random.default_rng(0)
    for k in range(4):
        p = rng.normal(size=(400, 3)) * rng.uniform(0.1, 3.0, 3)
        brute = float(np.sqrt(((p[None] - p[:, None]) ** 2).sum(-1).max()))
        assert abs(meshprep.mesh_diameter(p) - brute) < 1e-12
    assert meshprep.mesh_diameter(np.zeros((1, 3))) == 0.0
    m = synth.make_mesh(3)
    assert abs(meshprep.mesh_diameter(m.vertices) - 2 * synth.RADII.max()) < 1e-9
    # voxel grid: every output point is the mean of the inputs of one voxel (origin = min bound - voxel / 2)
    vox = 0.02
    q, n = meshprep.voxel_down_sample(m.vertices, vox, normals=m.vertex_normals)
    assert q.shape == n.shape and 1 < len(q) < len(m.vertices)
    origin = m.vertices.min(axis=0) - vox / 2
    idx_in = np.floor((m.vertices - origin) / vox).astype(np.int64)
    idx_out = np.floor((q - origin) / vox).astype(np.int64)
    assert len(np.unique(idx_in, axis=0)) == len(q) == len(np.unique(idx_out, axis=0))
    k0 = idx_out[0]
    sel = (idx_in == k0).all(1)
    np.testing.assert_allclose(q[0], m.vertices[sel].mean(0), atol=1e-12)
    np.testing.assert_allclose(n[0], m.vertex_normals[sel].mean(0), atol=1e-12)
    single, _ = meshprep.voxel_down_sample(m.vertices, 10.0)
    np.testing.assert_allclose(single, m.vertices.mean(0)[None], atol=1e-12)


def test_reference_config_defaults(tmp_path):
    """weights/<run>/config.yml is read the way the reference predictors read it (predict_pose_refine.py:107-131,
    predict_score.py:131-143): missing keys get the reference's backward-compatibility defaults, per predictor."""
    from foundationpose_b200 import weights

    p = tmp_path / "config.yml"
    p.write_text("crop_ratio: 1.1\nuse_BN: true\nc_in: 6\nnormalize_xyz: true\nzfar: .inf\nrot_normalizer: 0.3\n")
    c = weights.load_reference_config(str(p), "score")
    assert c["crop_ratio"] == 1.1 and c["use_BN"] is True and c["zfar"] == float("inf") and c["rot_normalizer"] == 0.3
    c = weights.load_reference_config(str(tmp_path / "missing.yml"), "refine")
    assert c["crop_ratio"] == 1.2 and c["use_BN"] is False and c["c_in"] == 4 and c["zfar"] == 3 and c["trans_rep"] == "tracknet"
    p.write_text("crop_ratio: null\nzfar: 'Inf'\n")
    c = weights.load_reference_config(str(p), "refine")
    assert c["crop_ratio"] == 1.2 and c["zfar"] == float("inf")


def test_reference_config_defaults_match_the_reference_statements(tmp_path):
    """The same, against what the reference's own `if '<key>' not in self.cfg` statements produce
    (tests/golden/predictor_defaults.json, extracted from the two constructors by tools/make_golden_config.py): every key
    the reference sets has the reference's value, for both predictors and five partial configs."""
    import json

    import yaml

    from foundationpose_b200 import weights

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cases = json.load(open(os.path.join(root, "tests", "golden", "predictor_defaults.json")))
    assert len(cases) == 10
    for name, case in cases.items():
        kind = name.split(".")[0]
        p = tmp_path / (name + ".yml")
        p.write_text(yaml.safe_dump(case["in"]))
        got = weights.load_reference_config(str(p), kind)
        for k, want in case["out"].items():
            have = got[k]
            if isinstance(have, float) and np.isinf(have):
                have = "inf"
            if isinstance(want, str) and want.lower() == "inf":
                want = "inf"  # the reference's scorer keeps a textual 'inf'; every consumer treats it as infinity
            assert have == want, (name, k, have, want)


def test_unsupported_config_raises():
    """A cfg value the engine cannot honour is an error, not silently ignored (ADVICE r1)."""
    import pytest

    from foundationpose_b200 import estimater, weights

    sd = {}
    with pytest.raises(ValueError):
        estimater._load_cfg_and_weights("x", "refine", sd, {"no_such_key": 1})
    with pytest.raises(NotImplementedError):
        estimater._load_cfg_and_weights("x", "refine", sd, {"rot_rep": "6d"})
    with pytest.raises(NotImplementedError):
        estimater._load_cfg_and_weights("x", "score", sd, {"input_resize": [128, 128]})
    cfg, _ = estimater._load_cfg_and_weights("x", "score", sd, {"crop_ratio": 1.1})
    assert cfg["crop_ratio"] == 1.1 and cfg["rot_rep"] == weights.DEFAULT_CFG["rot_rep"]


def test_replica_pool_surfaces_a_missing_device():
    """A replica whose GPU does not exist fails every call with the reason instead of leaving the caller waiting."""
    from foundationpose_b200.replicas import ReplicaPool

    pool = ReplicaPool([4096])
    try:
        with pytest.raises(RuntimeError):
            pool.reset_object(None, None)
        with pytest.raises(RuntimeError):
            pool.register_many([(None, 0, None, None)])
    finally:
        pool.close()
    assert not any(w.is_alive() for w in pool.workers)
