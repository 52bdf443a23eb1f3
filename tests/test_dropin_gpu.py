"""GPU: the drop-in module tree (foundationpose_b200/dropin) against what the reference's own drivers (run_demo.py,
run_linemod.py, run_ycb_video.py), UNMODIFIED, wrote on top of it over synthetic scenes in the reference's data layouts.
Those poses are stored in tests/golden/drivers_golden.npz (tools/make_golden_drivers.py); each test writes the same
synthetic scene, makes the driver's calls through the drop-in names, and must reproduce them."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN = os.path.join(ROOT, "foundationpose_b200", "dropin")


def _golden(prefix):
    """{(video, frame id string, ob_id): pose} that the reference's driver wrote to its result file."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "drivers_golden.npz"))
    return {(int(v), f"{f:06d}", int(o)): p for (v, f, o), p in zip(g[prefix + ".keys"], g[prefix + ".poses"])}


def _env():
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([DROPIN, ROOT, env.get("PYTHONPATH", "")])
    return env


@pytest.mark.parametrize("debug", [0, 2])
def test_run_demo_unmodified(tmp_path, debug):
    """run_demo.py's sequence (register on the first frame, track_one on the others, the box / axis overlay written per
    frame at debug >= 2) in a fresh process through the drop-in names: the poses the driver wrote."""
    from foundationpose_b200 import synth

    scene = str(tmp_path / "demo_data" / "synth0")
    mesh, gt = synth.write_demo_scene(scene, n_frames=4, subdivisions=3)
    dbg = str(tmp_path / "debug")
    code = f"""
from estimater import *
from datareader import *
set_seed(0)
mesh = trimesh.load({scene!r} + '/mesh/textured_simple.obj')
to_origin, extents = trimesh.bounds.oriented_bounds(mesh)
bbox = np.stack([-extents / 2, extents / 2], axis=0).reshape(2, 3)
scorer = ScorePredictor()
refiner = PoseRefinePredictor()
est = FoundationPose(model_pts=mesh.vertices, model_normals=mesh.vertex_normals, mesh=mesh, scorer=scorer, refiner=refiner,
                     debug_dir={dbg!r}, debug={debug}, glctx=dr.RasterizeCudaContext())
reader = YcbineoatReader(video_dir={scene!r}, shorter_side=None, zfar=np.inf)
os.makedirs({dbg!r} + '/ob_in_cam', exist_ok=True)
os.makedirs({dbg!r} + '/track_vis', exist_ok=True)
for i in range(len(reader.color_files)):
    color, depth = reader.get_color(i), reader.get_depth(i)
    if i == 0:
        pose = est.register(K=reader.K, rgb=color, depth=depth, ob_mask=reader.get_mask(0).astype(bool), iteration=5)
    else:
        pose = est.track_one(rgb=color, depth=depth, K=reader.K, iteration=2)
    np.savetxt(f'{dbg}/ob_in_cam/{{reader.id_strs[i]}}.txt', pose.reshape(4, 4))
    if {debug} >= 2:
        center_pose = pose @ np.linalg.inv(to_origin)
        vis = draw_posed_3d_box(reader.K, img=color, ob_in_cam=center_pose, bbox=bbox)
        vis = draw_xyz_axis(color, ob_in_cam=center_pose, scale=0.1, K=reader.K, thickness=3, transparency=0, is_input_rgb=True)
        imageio.imwrite(f'{dbg}/track_vis/{{reader.id_strs[i]}}.png', vis)
"""
    out = subprocess.run([sys.executable, "-c", code], env=_env(), capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert out.returncode == 0, (out.stdout + out.stderr)[-4000:]
    want = np.load(os.path.join(ROOT, "tests", "golden", "drivers_golden.npz"))[f"demo.debug{debug}.poses"]
    poses = []
    for i in range(4):
        f = os.path.join(dbg, "ob_in_cam", f"{i:06d}.txt")
        assert os.path.exists(f), f"{f} missing\n" + (out.stdout + out.stderr)[-2000:]
        p = np.loadtxt(f).reshape(4, 4)
        assert np.isfinite(p).all() and abs(np.linalg.det(p[:3, :3]) - 1) < 1e-3
        np.testing.assert_allclose(p, want[i], atol=1e-5, err_msg=f"frame {i}")
        poses.append(p)
    # random-init weights: no accuracy claim, but the seeded stand-in moves a pose by millimetres per pass, so the
    # tracked object stays near where the first frame's mask put it
    assert all(0.4 < p[2, 3] < 0.8 for p in poses), [p[:3, 3] for p in poses]
    if debug >= 2:
        assert os.path.exists(os.path.join(dbg, "track_vis", "000003.png"))


def test_run_linemod_unmodified(tmp_path):
    """SURVEY.md §8f N3: the reference's LINEMOD driver (run_linemod.py: 13 objects, `reset_object` per object, one
    `register` per frame, results to linemod_res.yml) over a synthetic dataset in its directory layout.  Every pose it
    wrote must be the pose the native API returns for the same reader inputs."""
    from foundationpose_b200 import synth

    root = str(tmp_path / "LINEMOD")
    gts = synth.write_bop_dataset(root, "lm", n_frames=1)
    res = _golden("linemod.frames1")
    assert sorted({v for v, _, _ in res}) == [1, 2, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14, 15]
    assert sorted(res) == sorted(gts)
    sys.path[:0] = [DROPIN, ROOT]
    try:
        import datareader
        from foundationpose_b200.estimater import FoundationPose

        trimesh = datareader.trimesh  # the real package or the stand-in, whichever `Utils` resolved

        box = trimesh.primitives.Box(extents=np.ones(3), transform=np.eye(4)).to_mesh()
        est = FoundationPose(model_pts=box.vertices.copy(), model_normals=box.vertex_normals.copy(), mesh=box, debug_dir=str(tmp_path / "dbg2"))
        for (scene, frame, ob), gt in sorted(gts.items()):
            r = datareader.LinemodReader(f"{root}/lm_test_all/test/{ob:06d}", split=None)
            mesh = r.get_gt_mesh(ob)
            # the driver's sequence (run_linemod.py:100-112): one estimator, `reset_object` per object.  Like the
            # reference's, `reset_object` keeps the rotation grid built at construction (estimater.py:40-41 vs :43-85):
            # the per-object symmetries do not thin the 252 start poses on this route
            est.reset_object(model_pts=mesh.vertices.copy(), model_normals=mesh.vertex_normals.copy(), symmetry_tfs=r.symmetry_tfs[ob], mesh=mesh)
            i = r.id_strs.index(frame)
            p = est.register(K=r.K, rgb=r.get_color(i), depth=r.get_depth(i), ob_mask=r.get_mask(i, ob) > 0, ob_id=ob)
            assert p.shape == (4, 4) and np.isfinite(p).all() and abs(np.linalg.det(p[:3, :3]) - 1) < 1e-3
            assert np.linalg.norm(p[:3, 3] - gt[:3, 3]) < 0.08, (scene, p[:3, 3], gt[:3, 3])  # stand-in weights: stays near the mask
            np.testing.assert_allclose(res[(scene, frame, ob)], p, atol=1e-5)
            assert len(est.rot_grid) == 252
        # constructed WITH the symmetry (obj 6: half turn about z in models_info.json) the grid is clustered under it
        r = datareader.LinemodReader(f"{root}/lm_test_all/test/000006", split=None)
        mesh = r.get_gt_mesh(6)
        sym = FoundationPose(model_pts=mesh.vertices.copy(), model_normals=mesh.vertex_normals.copy(), symmetry_tfs=r.symmetry_tfs[6], mesh=mesh,
                             debug_dir=str(tmp_path / "dbg3"))
        assert len(sym.rot_grid) < 252
    finally:
        del sys.path[:2]


def test_run_ycb_video_unmodified(tmp_path, monkeypatch):
    """The YCB-Video driver (run_ycb_video.py: 21 objects x the scenes that contain them, key frames only,
    zfar = 1.5) over a synthetic dataset of three one-object scenes: the native API returns the poses it wrote."""
    from foundationpose_b200 import synth

    root = str(tmp_path / "YCB_Video")
    gts = synth.write_bop_dataset(root, "ycbv", n_frames=2, scene_objects={48: 1, 49: 6, 50: 13})
    res = _golden("ycbv")
    assert sorted({v for v, _, _ in res}) == [48, 49, 50]
    assert sorted(res) == sorted(gts) and len(res) == 6
    monkeypatch.setenv("YCB_VIDEO_DIR", root)  # as the driver sets it from --ycbv_dir
    sys.path[:0] = [DROPIN, ROOT]
    try:
        import datareader
        from foundationpose_b200.estimater import FoundationPose

        trimesh = datareader.trimesh
        video_dirs = sorted(os.path.join(root, "test", d) for d in os.listdir(os.path.join(root, "test")))
        reader_tmp = datareader.YcbVideoReader(video_dirs[0])
        box = trimesh.primitives.Box(extents=np.ones(3), transform=np.eye(4)).to_mesh()
        est =FoundationPose(model_pts=box.vertices.copy(), model_normals=box.vertex_normals.copy(), mesh=box, debug_dir=str(tmp_path / "dbg2"))
        n = 0
        for ob in reader_tmp.ob_ids:
            mesh = reader_tmp.get_gt_mesh(ob)
            est.reset_object(model_pts=mesh.vertices.copy(), model_normals=mesh.vertex_normals.copy(), symmetry_tfs=reader_tmp.symmetry_tfs[ob], mesh=mesh)
            for video_dir in video_dirs:
                r = datareader.YcbVideoReader(video_dir, zfar=1.5)
                if ob not in r.get_instance_ids_in_image(0):
                    continue
                for i in range(len(r.color_files)):
                    if not r.is_keyframe(i) or ob not in r.get_instance_ids_in_image(i):
                        continue
                    p = est.register(K=r.K, rgb=r.get_color(i), depth=r.get_depth(i), ob_mask=r.get_mask(i, ob, type="mask_visib") > 0,
                                     ob_id=ob, iteration=5)
                    key = (r.get_video_id(), r.id_strs[i], ob)
                    assert p.shape == (4, 4) and np.isfinite(p).all() and abs(np.linalg.det(p[:3, :3]) - 1) < 1e-3
                    assert np.linalg.norm(p[:3, 3] - gts[key][:3, 3]) < 0.08
                    np.testing.assert_allclose(res[key], p, atol=1e-5, err_msg=str(key))
                    n += 1
        assert n == 6
    finally:
        del sys.path[:2]


def test_linemod_over_replicas_matches_the_sequential_driver(tmp_path):
    """examples/run_linemod_replicas.py (frames of an object spread over the GPUs by ReplicaPool) writes the same
    linemod_res.yml as the reference's sequential driver loop wrote through one estimator."""
    import torch
    import yaml

    from foundationpose_b200 import synth

    root = str(tmp_path / "LINEMOD")
    synth.write_bop_dataset(root, "lm", n_frames=2)
    dbg = str(tmp_path / "debug_pool")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "run_linemod_replicas.py"), "--linemod_dir", root, "--debug_dir", dbg,
                          "--gpus", str(min(2, torch.cuda.device_count()))], env=_env(), capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert out.returncode == 0, (out.stdout + out.stderr)[-4000:]
    with open(os.path.join(dbg, "linemod_res.yml")) as fh:
        a = yaml.safe_load(fh)
    b = _golden("linemod.frames2")
    assert sorted((vid, frame, ob) for vid in a for frame in a[vid] for ob in a[vid][frame]) == sorted(b)
    for (vid, frame, ob), want in b.items():
        np.testing.assert_allclose(np.array(a[vid][frame][ob]), want, atol=1e-5)
