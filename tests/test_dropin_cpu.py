"""CPU: the drop-in module tree (foundationpose_b200/dropin) resolves every name the reference's UNMODIFIED
run_demo.py uses, the trimesh / imageio stand-ins round-trip the demo-scene files, and the reader parses them."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN = os.path.join(ROOT, "foundationpose_b200", "dropin")


def _env():
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([DROPIN, ROOT, env.get("PYTHONPATH", "")])
    return env


def _driver_names(script):
    """Import statements, unqualified names and first-level attributes of one of the reference's drivers, read from the
    driver with `ast` by tools/make_golden_drivers.py --names."""
    with open(os.path.join(ROOT, "tests", "golden", "driver_names.json")) as fh:
        d = json.load(fh)[script]
    return d["imports"], d["names"], [tuple(a) for a in d["attrs"]]


def test_every_name_run_demo_uses_resolves():
    """Static check against the reference's own driver: all unqualified names and first-level attributes
    (`trimesh.load`, `dr.RasterizeCudaContext`, `np.stack`, ...) exist after its two star-imports."""
    _, need, mod_attrs = _driver_names("run_demo.py")
    assert {"trimesh", "dr", "np", "cv2", "imageio", "logging", "set_seed", "YcbineoatReader", "FoundationPose"} <= set(need)
    code = ("from estimater import *\nfrom datareader import *\nimport argparse\n"
            f"missing = [n for n in {need!r} if n not in globals()]\n"
            f"missing += [f'{{m}}.{{a}}' for (m, a) in {mod_attrs!r} if m in globals() and not hasattr(globals()[m], a)]\n"
            "missing += [] if hasattr(trimesh.bounds, 'oriented_bounds') else ['trimesh.bounds.oriented_bounds']\n"
            "print('MISSING', missing)\n")
    out = subprocess.run([sys.executable, "-c", code], env=_env(), capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "MISSING []" in out.stdout, out.stdout[-2000:]


def test_demo_scene_round_trip(tmp_path):
    code = f"""
import numpy as np
from estimater import *
from datareader import *
from foundationpose_b200 import synth
mesh0, gt = synth.write_demo_scene({str(tmp_path)!r}, n_frames=2, subdivisions=2)
mesh = trimesh.load({str(tmp_path)!r} + '/mesh/textured_simple.obj')
assert np.abs(mesh.vertices[mesh.faces] - mesh0.vertices[mesh0.faces]).max() < 1e-6
assert np.abs(mesh.visual.uv[mesh.faces] - mesh0.visual.uv[mesh0.faces]).max() < 1e-6
assert np.abs(mesh.vertex_normals[mesh.faces] - mesh0.vertex_normals[mesh0.faces]).max() < 1e-6
img = np.asarray(mesh.visual.material.image.convert('RGB'))
assert (img == mesh0.visual.image).all()
mt, mt0 = make_mesh_tensors(mesh), make_mesh_tensors(mesh0)
assert (mt['tex'] == mt0['tex']).all() and mt['uv'].shape == (len(mesh.vertices), 2)
to_origin, extents = trimesh.bounds.oriented_bounds(mesh)
assert np.allclose(sorted(extents), sorted(2 * synth.RADII), rtol=0.03), extents
assert np.allclose(to_origin[:3, :3] @ to_origin[:3, :3].T, np.eye(3), atol=1e-9)
reader = YcbineoatReader(video_dir={str(tmp_path)!r}, shorter_side=None, zfar=np.inf)
assert len(reader.color_files) == 2 and reader.id_strs == ['000000', '000001'] and reader.K.shape == (3, 3)
color, depth, mask = reader.get_color(0), reader.get_depth(0), reader.get_mask(0).astype(bool)
rgb0, depth0, mask0 = synth.make_scene(mesh0.visual.image, gt[0], seed=1)
assert color.dtype == np.uint8 and (color == rgb0).all()
assert np.abs(depth - depth0).max() <= 0.00051 and (mask == mask0).all()
assert np.allclose(reader.get_gt_pose(1), gt[1])
vis = draw_posed_3d_box(reader.K, img=color.copy(), ob_in_cam=gt[0], bbox=np.stack([-extents / 2, extents / 2]))
vis = draw_xyz_axis(vis, ob_in_cam=gt[0], scale=0.1, K=reader.K, thickness=3, transparency=0, is_input_rgb=True)
assert vis.shape == color.shape and (vis != color).any()
xyz = depth2xyzmap(depth, reader.K)
assert xyz.shape == (480, 640, 3) and abs(xyz[240, 320, 2] - depth[240, 320]) < 1e-6
print('OK')
"""
    out = subprocess.run([sys.executable, "-c", code], env=_env(), capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "OK" in out.stdout, (out.stdout + out.stderr)[-3000:]


@pytest.mark.parametrize("script", ["run_linemod.py", "run_ycb_video.py"])
def test_every_name_the_dataset_drivers_use_resolves(script):
    """Same static check for the reference's dataset drivers (SURVEY.md §8f N3): replay the script's own import
    statements on top of the drop-in tree, then every unqualified name / first-level attribute must exist."""
    imports, need, mod_attrs = _driver_names(script)
    assert {"wp", "NestDict", "make_yaml_dumpable", "dr", "trimesh", "FoundationPose", "set_seed", "argparse"} <= set(need)
    code = ("\n".join(imports) + "\n"
            f"missing = [n for n in {need!r} if n not in globals()]\n"
            f"missing += [f'{{m}}.{{a}}' for (m, a) in {mod_attrs!r} if m in globals() and not hasattr(globals()[m], a)]\n"
            "print('MISSING', missing)\n")
    out = subprocess.run([sys.executable, "-c", code], env=_env(), capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "MISSING []" in out.stdout, out.stdout[-2000:]


def test_bop_readers_parse_the_synthetic_datasets(tmp_path):
    """LinemodReader / YcbVideoReader (datareader.py:155-531) on trees written by synth.write_bop_dataset: ids, K,
    colour / depth / mask, ground-truth poses, PLY models in millimetres, symmetry tables, key frames."""
    code = f"""
import os
import numpy as np
from foundationpose_b200 import synth
root = {str(tmp_path)!r}
gt_lm = synth.write_bop_dataset(root + '/LINEMOD', 'lm', n_frames=2)
gt_y = synth.write_bop_dataset(root + '/YCB_Video', 'ycbv', n_frames=2)
os.environ['YCB_VIDEO_DIR'] = root + '/YCB_Video'
from datareader import *
r = LinemodReader(root + '/LINEMOD/lm_test_all/test/000006', split=None)
assert r.ob_ids == [1, 2, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14, 15] and r.get_video_id() == 6 and len(r.color_files) == 2
assert r.id_strs == ['000000', '000001'] and np.allclose(r.K, synth.DEFAULT_K) and np.allclose(r.get_K(1), synth.DEFAULT_K)
assert list(r.get_instance_ids_in_image(0)) == [6]
c, d, m = r.get_color(0), r.get_depth(0), r.get_mask(0, 6)
assert c.shape == (480, 640, 3) and c.dtype == np.uint8 and d.shape == (480, 640) and m.dtype == bool and 2000 < m.sum() < 60000
assert abs(np.median(d[m]) - gt_lm[(6, '000000', 6)][2, 3]) < 0.08 and d[~m].min() > 1.0
assert r.get_mask(0, 5) is None or True
assert np.allclose(r.get_gt_pose(0, 6), gt_lm[(6, '000000', 6)], atol=1e-9)
assert np.allclose(r.get_gt_pose(1, 6, mask=m), gt_lm[(6, '000001', 6)], atol=1e-9)
assert r.get_gt_poses(0, 6).shape == (1, 4, 4) and r.get_gt_poses(0, 5).shape == (0, 4, 4)
mesh = r.get_gt_mesh(6)
ref = synth.make_mesh(2)
assert np.abs(mesh.vertices - ref.vertices).max() < 1e-6 and (mesh.faces == ref.faces).all()
assert mesh.visual.vertex_colors.shape == (len(ref.vertices), 4)
assert abs(r.get_model_diameter(6) - synth.mesh_diameter(ref.vertices)) < 1e-6
assert r.symmetry_tfs[6].shape == (2, 4, 4) and r.symmetry_tfs[5].shape == (1, 4, 4)
xyz = r.get_xyz_map(0)
assert xyz.shape == (480, 640, 3) and abs(xyz[240, 320, 2] - d[240, 320]) < 1e-6
y = YcbVideoReader(root + '/YCB_Video/test/000049', zfar=1.5)
assert y.ob_ids == list(range(1, 22)) and len(y.ob_id_to_names) == 21 and y.get_video_id() == 49
assert list(y.get_instance_ids_in_image(0)) == [6] and y.is_keyframe(0) and y.is_keyframe(1)
assert y.get_depth(0).max() <= 1.5
assert np.abs(y.get_gt_mesh(13).vertices - ref.vertices).max() < 1e-6
assert 'symmetries_continuous' in y.geometry_symmetry_info_table[13] and len(y.geometry_symmetry_info_table[2]['symmetries_discrete']) == 8
assert isinstance(get_bop_reader(root + '/YCB_Video/test/000048'), YcbVideoReader)
print('OK')
"""
    out = subprocess.run([sys.executable, "-c", code], env=_env(), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK" in out.stdout, (out.stdout + out.stderr)[-3000:]


def test_remaining_bop_readers(tmp_path):
    """TUD-L / T-LESS style readers (datareader.py:533-613): dispatch by path, model directory three levels up, uniform
    grey for the texture-less CAD models."""
    code = f"""
import json, os, shutil
import numpy as np
from foundationpose_b200 import synth
d = {str(tmp_path)!r}
synth.write_bop_dataset(d + '/LM', 'lm')
def info(path, n):
    json.dump({{str(i): {{"diameter": 100.0}} for i in range(1, n + 1)}}, open(path, 'w'))
os.makedirs(d + '/tudl/tudl_test_bop19/test')
shutil.copytree(d + '/LM/lm_test_all/test/000001', d + '/tudl/tudl_test_bop19/test/000001')
shutil.copytree(d + '/LM/lm_models/models', d + '/tudl/tudl_models/models')
info(d + '/tudl/tudl_models/models/models_info.json', 3)
os.makedirs(d + '/tless/split/test_primesense')
shutil.copytree(d + '/LM/lm_test_all/test/000002', d + '/tless/split/test_primesense/000002')
shutil.copytree(d + '/LM/lm_models/models', d + '/tless/models_cad')
info(d + '/tless/models_cad/models_info.json', 30)
from datareader import *
r = get_bop_reader(d + '/tudl/tudl_test_bop19/test/000001')
assert type(r).__name__ == 'TudlReader' and r.ob_ids == [1, 2, 3] and r.dataset_name == 'tudl'
assert r.get_gt_mesh(1).vertices.shape[1] == 3 and r.symmetry_tfs[2].shape == (1, 4, 4) and abs(r.get_model_diameter(1) - 0.1) < 1e-12
t = get_bop_reader(d + '/tless/split/test_primesense/000002')
assert type(t).__name__ == 'TlessReader' and len(t.ob_ids) == 30
m = t.get_gt_mesh(2)
assert (np.asarray(m.visual.vertex_colors)[:, :3] == 200).all() and np.abs(m.vertices).max() < 0.2
assert IcbinReader.__name__ == 'IcbinReader' and issubclass(HomebrewedReader, BopBaseReader) and issubclass(ItoddReader, BopBaseReader)
print('OK')
"""
    out = subprocess.run([sys.executable, "-c", code], env=_env(), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK" in out.stdout, (out.stdout + out.stderr)[-3000:]


def test_bop_reader_multi_instance_and_missing_files(tmp_path):
    """datareader.py:266-350 edge cases: two instances of one object in a frame (the `mask` argument picks the
    annotation by visible-mask IoU), a second object's mask index, a missing mask file (None), frames without
    scene_gt.json (ids from the mask file names)."""
    code = f"""
import json, os
import cv2
import numpy as np
from foundationpose_b200 import synth
d = {str(tmp_path)!r}
synth.write_bop_dataset(d + '/LM', 'lm')
scene = d + '/LM/lm_test_all/test/000001'
gt = json.load(open(scene + '/scene_gt.json'))
a = dict(gt['0'][0]); b = dict(a); c = dict(a)
b['cam_t_m2c'] = [100.0, 0.0, 700.0]           # second instance of object 1
c['obj_id'] = 5; c['cam_t_m2c'] = [-100.0, 50.0, 650.0]
gt['0'] = [a, c, b]
json.dump(gt, open(scene + '/scene_gt.json', 'w'))
m0 = cv2.imread(scene + '/mask_visib/000000_000000.png', -1)
m1 = np.zeros_like(m0); m1[100:200, 400:500] = 255   # object 5
m2 = np.zeros_like(m0); m2[300:400, 100:200] = 255   # second instance of object 1
cv2.imwrite(scene + '/mask_visib/000000_000001.png', m1)
cv2.imwrite(scene + '/mask_visib/000000_000002.png', m2)
from datareader import *
r = LinemodReader(scene, split=None)
assert list(r.get_instance_ids_in_image(0)) == [1, 5, 1]
assert r.get_gt_poses(0, 1).shape == (2, 4, 4) and r.get_gt_poses(0, 5).shape == (1, 4, 4)
assert np.allclose(r.get_gt_pose(0, 1)[:3, 3], np.array(a['cam_t_m2c']) / 1e3)          # first annotation without a mask
assert np.allclose(r.get_gt_pose(0, 1, mask=m2 > 0)[:3, 3], [0.1, 0.0, 0.7])            # IoU picks the second instance
assert np.allclose(r.get_gt_pose(0, 1, mask=m0 > 0)[:3, 3], np.array(a['cam_t_m2c']) / 1e3)
assert (r.get_mask(0, 5) == (m1 > 0)).all() and (r.get_mask(0, 1) == (m0 > 0)).all()
assert r.get_mask(0, 5, type='mask') is None                                              # no such file: None, not an exception
assert np.allclose(r.get_gt_pose(0, 9), np.eye(4))                                        # object not in the frame
os.remove(scene + '/scene_gt.json')
r2 = LinemodReader(scene, split=None)
assert r2.scene_gt is None and list(r2.get_instance_ids_in_image(0)) == [0, 1, 2]         # annotation slots from the mask files
print('OK')
"""
    out = subprocess.run([sys.executable, "-c", code], env=_env(), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "OK" in out.stdout, (out.stdout + out.stderr)[-3000:]

