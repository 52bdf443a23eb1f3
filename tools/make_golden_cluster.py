"""Golden vectors for the start-pose grid, produced by the reference's own code:

  * `cluster_poses` + `Utils::rotationGeodesicDistance` — the reference's C++ (mycpp/src/app/pybind_api.cpp:24-68,
    mycpp/src/Utils.cpp:21-26) compiled by oracle/build_ref.py from the function texts where they lie (Eigen replaced by
    oracle/eigen_shim.h; the reference's own CMake recipe needs Eigen + Boost, which are not in the image);
  * `FoundationPose.make_rotation_grid` (estimater.py:106-124) and `sample_views_icosphere` (Utils.py:483-507) — method /
    function sources extracted with `ast` and executed, calling that compiled `cluster_poses` as `mycpp.cluster_poses`.
    Two third-party pieces are substituted: `trimesh.creation.icosphere` (trimesh is absent; this repository's icosphere
    is used — its VERTEX ORDER is therefore not pinned, SURVEY.md §8c) and `transformations.euler_matrix` (scipy).

    python tools/make_golden_cluster.py     # needs the reference tree (FPOSE_REFERENCE); writes
                                            # tests/golden/cluster_golden.npz and cluster_random_golden.npz

tests/test_cluster_golden_cpu.py holds foundationpose_b200.hypotheses (cluster_poses, sample_views_icosphere,
make_rotation_grid) to these vectors.
"""
import logging
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
REF = os.environ.get("FPOSE_REFERENCE", "/root/reference")


def euler_matrix(ai, aj, ak, axes="sxyz"):
    from scipy.spatial.transform import Rotation

    M = np.eye(4)
    M[:3, :3] = Rotation.from_euler("xyz", [ai, aj, ak]).as_matrix()
    return M


def symmetry_sets():
    return {"identity": np.eye(4)[None],
            "half_z": np.stack([np.eye(4), np.diag([-1.0, -1.0, 1.0, 1.0])]),
            "cont_z": np.stack([euler_matrix(0, 0, a) for a in np.arange(0, 360, 5) / 180 * np.pi]),
            "box": np.stack([euler_matrix(rx, ry, rz) for rz in (0, np.pi) for rx in (0, np.pi) for ry in (0, np.pi)])}


def main():
    from make_golden_flow import _TorchProxy
    from make_golden_geometry import extract

    from foundationpose_b200 import synth
    from oracle import build_ref

    build_ref.build()
    cluster = build_ref.load()
    icosphere = lambda subdivisions=3, radius=1.0: types.SimpleNamespace(vertices=synth.icosphere(subdivisions)[0] * radius)
    ns = {"np": np, "torch": _TorchProxy("torch"), "logging": logging, "euler_matrix": euler_matrix,
          "trimesh": types.SimpleNamespace(creation=types.SimpleNamespace(icosphere=icosphere)),
          "mycpp": types.SimpleNamespace(cluster_poses=lambda a, d, poses, syms: list(cluster(a, d, poses, syms)))}
    exec(extract(os.path.join(REF, "Utils.py"), "sample_views_icosphere"), ns)
    exec(extract(os.path.join(REF, "estimater.py"), "make_rotation_grid", cls="FoundationPose"), ns)
    torch.Tensor.cuda = lambda self, *a, **k: self
    out = {"views_40": ns["sample_views_icosphere"](n_views=40), "views_sub2": ns["sample_views_icosphere"](n_views=1, subdivisions=2, radius=0.5)}
    for name, syms in symmetry_sets().items():
        est = types.SimpleNamespace(symmetry_tfs=torch.as_tensor(syms, dtype=torch.float32))
        ns["make_rotation_grid"](est, min_n_views=40, inplane_step=60)
        out[f"rot_grid.{name}"] = est.rot_grid.numpy()
        print(name, "->", tuple(est.rot_grid.shape))
    est = types.SimpleNamespace(symmetry_tfs=torch.eye(4)[None])
    ns["make_rotation_grid"](est, min_n_views=10, inplane_step=90)
    out["rot_grid.identity_10_90"] = est.rot_grid.numpy()
    # cluster_poses alone: other thresholds, and translations that matter
    grid = out["rot_grid.identity"]
    rng = np.random.default_rng(0)
    moved = grid.copy()
    moved[:, :3, 3] = rng.normal(0, 0.01, (len(grid), 3))
    out["moved_poses"] = moved
    for name, syms in symmetry_sets().items():
        for ang in (10, 61):
            out[f"cluster.{name}.{ang}"] = cluster(ang, 99999, grid, syms)
    out["cluster.moved.half_z"] = cluster(30, 0.01, moved, symmetry_sets()["half_z"])
    # random pose sets with translations spread over the distance threshold, one angle threshold per set; what the
    # reference keeps is stored as indices into the set (it returns a subset of its input poses, unchanged)
    from scipy.spatial.transform import Rotation

    rng = np.random.default_rng(3)
    rand = {}
    for trial in range(4):
        n = 150
        poses = np.tile(np.eye(4, dtype=np.float32), (n, 1, 1))
        poses[:, :3, :3] = Rotation.random(n, random_state=trial).as_matrix()
        poses[:, :3, 3] = rng.normal(0, 0.02, (n, 3))
        rand[f"poses.{trial}"] = poses
        for name, syms in symmetry_sets().items():
            kept = cluster(25 + 5 * trial, 0.03, poses, syms)
            idx = [int(np.flatnonzero((poses == k).all(axis=(1, 2)))[0]) for k in kept]
            assert np.array_equal(poses[idx], kept)
            rand[f"kept.{trial}.{name}"] = np.array(idx, dtype=np.int16)
    dst = os.path.join(ROOT, "tests", "golden", "cluster_random_golden.npz")
    np.savez_compressed(dst, **rand)
    print(f"wrote {dst}: {len(rand)} entries, {os.path.getsize(dst) / 1024:.0f} KiB")
    dst = os.path.join(ROOT, "tests", "golden", "cluster_golden.npz")
    np.savez_compressed(dst, **out)
    print(f"wrote {dst}: {len(out)} entries, {os.path.getsize(dst) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
