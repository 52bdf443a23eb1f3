"""Golden vectors for tests/test_dropin_cpu.py and tests/test_dropin_gpu.py, produced by the reference's own drivers
(run_demo.py, run_linemod.py, run_ycb_video.py), UNMODIFIED:

  * `--names` (CPU): what each driver needs from its star-imports — its import statements, every unqualified name it
    reads and every first-level attribute of those names (`trimesh.load`, `dr.RasterizeCudaContext`, ...), found with
    `ast` -> tests/golden/driver_names.json;
  * default (GPU): the poses each driver writes when it runs on top of foundationpose_b200/dropin over the synthetic
    scenes the tests write (same generator calls, same arguments) -> tests/golden/drivers_golden.npz.

    FPOSE_REFERENCE=<FoundationPose checkout> python tools/make_golden_drivers.py --names
    python tools/make_golden_drivers.py [--out F]      # needs a GPU and the drivers: $FPOSE_REFERENCE, or the copies
                                                       # __graft_entry__.build() stages into oracle/_ref/
"""
import argparse
import ast
import builtins
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DROPIN = os.path.join(ROOT, "foundationpose_b200", "dropin")
REF = os.environ.get("FPOSE_REFERENCE", "")
DATASET_DRIVERS = ("run_linemod.py", "run_ycb_video.py")


def driver(name):
    for cand in ([os.path.join(REF, name)] if REF else []) + [os.path.join(ROOT, "oracle", "_ref", name)]:
        if os.path.exists(cand):
            return cand
    raise FileNotFoundError(f"{name}: neither $FPOSE_REFERENCE nor oracle/_ref/ holds it")


def names(path, dataset_driver):
    """(import statements, unqualified names read, first-level attributes of those names) of one driver."""
    tree = ast.parse(open(path).read())
    imports = [ast.unparse(n) for n in tree.body if isinstance(n, (ast.Import, ast.ImportFrom))]
    assigned, used, attrs = set(), set(), set()
    for node in ast.walk(tree):
        if isinstance(node, ast.Name):
            (assigned if isinstance(node.ctx, ast.Store) else used).add(node.id)
        elif isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name):
            attrs.add((node.value.id, node.attr))
        elif dataset_driver and isinstance(node, (ast.FunctionDef, ast.arg)):
            assigned.add(node.name if isinstance(node, ast.FunctionDef) else node.arg)
    need = sorted(n for n in used - assigned - set(dir(builtins)) if n != "__file__")
    skip = ("opt", "parser", "o3d", "reader", "reader_tmp", "est") if dataset_driver else ("args", "parser", "o3d")
    mod_attrs = sorted([m, a] for (m, a) in attrs if m in need and m not in skip)
    return {"imports": imports, "names": need, "attrs": mod_attrs}


def write_names():
    out = {"run_demo.py": names(driver("run_demo.py"), False)}
    for name in DATASET_DRIVERS:
        out[name] = names(driver(name), True)
    dst = os.path.join(ROOT, "tests", "golden", "driver_names.json")
    with open(dst, "w") as fh:
        json.dump(out, fh, indent=1)
        fh.write("\n")
    print(f"wrote {dst}")


def _run(cmd, cwd, site=None):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join(([site] if site else []) + [DROPIN, ROOT, env.get("PYTHONPATH", "")])
    env["QT_QPA_PLATFORM"] = "offscreen"
    out = subprocess.run([sys.executable] + cmd, env=env, capture_output=True, text=True, timeout=900, cwd=cwd)
    assert out.returncode == 0, (out.stdout + out.stderr)[-4000:]


def _flatten(res_yml):
    """{video: {frame: {ob: pose}}} -> (keys (n, 3) int64 rows (video, frame, ob), poses (n, 4, 4)), rows sorted."""
    import yaml

    with open(res_yml) as fh:
        res = yaml.safe_load(fh)
    rows = sorted((int(v), int(f), int(o)) for v in res for f in res[v] for o in res[v][f])
    poses = [np.array(res[v][f"{f:06d}"][o], dtype=np.float64) for v, f, o in rows]
    return np.array(rows, dtype=np.int64).reshape(-1, 3), np.stack(poses)


def write_runs(dst):
    from foundationpose_b200 import synth

    out = {}
    with tempfile.TemporaryDirectory(prefix="fpose_drivers_") as tmp:
        # run_demo.py: the scene of tests/test_dropin_gpu.py::test_run_demo_unmodified, --debug 0 and 2
        for debug in (0, 2):
            work = os.path.join(tmp, f"demo{debug}")
            scene = os.path.join(work, "demo_data", "synth0")
            synth.write_demo_scene(scene, n_frames=4, subdivisions=3)
            dbg = os.path.join(work, "debug")
            site = None
            if debug >= 1:  # headless OpenCV: imshow / waitKey become no-ops for this process only
                site = os.path.join(work, "site")
                os.makedirs(site)
                with open(os.path.join(site, "sitecustomize.py"), "w") as fh:
                    fh.write("import cv2\ncv2.imshow = lambda *a, **k: None\ncv2.waitKey = lambda *a, **k: -1\n")
            _run([driver("run_demo.py"), "--mesh_file", scene + "/mesh/textured_simple.obj", "--test_scene_dir", scene,
                  "--est_refine_iter", "5", "--track_refine_iter", "2", "--debug", str(debug), "--debug_dir", dbg], work, site)
            out[f"demo.debug{debug}.poses"] = np.stack([np.loadtxt(os.path.join(dbg, "ob_in_cam", f"{i:06d}.txt")).reshape(4, 4)
                                                        for i in range(4)])
        # run_linemod.py over the 1-frame (test_run_linemod_unmodified) and 2-frame (the replica test) datasets
        for n_frames in (1, 2):
            work = os.path.join(tmp, f"lm{n_frames}")
            root = os.path.join(work, "LINEMOD")
            synth.write_bop_dataset(root, "lm", n_frames=n_frames)
            dbg = os.path.join(work, "debug")
            _run([driver("run_linemod.py"), "--linemod_dir", root, "--debug_dir", dbg], work)
            out[f"linemod.frames{n_frames}.keys"], out[f"linemod.frames{n_frames}.poses"] = _flatten(os.path.join(dbg, "linemod_res.yml"))
        # run_ycb_video.py over three one-object scenes
        work = os.path.join(tmp, "ycbv")
        root = os.path.join(work, "YCB_Video")
        synth.write_bop_dataset(root, "ycbv", n_frames=2, scene_objects={48: 1, 49: 6, 50: 13})
        dbg = os.path.join(work, "debug")
        _run([driver("run_ycb_video.py"), "--ycbv_dir", root, "--debug_dir", dbg], work)
        out["ycbv.keys"], out["ycbv.poses"] = _flatten(os.path.join(dbg, "ycbv_res.yml"))
    os.makedirs(os.path.dirname(os.path.abspath(dst)), exist_ok=True)
    np.savez_compressed(dst, **out)
    print(f"wrote {dst}: " + ", ".join(f"{k} {v.shape}" for k, v in out.items()))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--names", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "drivers_golden.npz"))
    a = ap.parse_args()
    write_names() if a.names else write_runs(a.out)
