"""CPU: the start-pose grid (foundationpose_b200/hypotheses.py: sample_views_icosphere, make_rotation_grid, cluster_poses)
against golden vectors produced by the reference's own code (tools/make_golden_cluster.py): the C++ `cluster_poses` +
`rotationGeodesicDistance` compiled from the reference tree (oracle/build_ref.py, Eigen replaced by oracle/eigen_shim.h),
called from the reference's unmodified `FoundationPose.make_rotation_grid` (estimater.py:106-124) and
`sample_views_icosphere` (Utils.py:483-507).  Unpinned by construction: trimesh's icosphere vertex ORDER (trimesh is absent;
both sides use this repository's icosphere)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def golden():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_golden_cluster as gen  # symmetry_sets() only

    return gen, dict(np.load(os.path.join(ROOT, "tests", "golden", "cluster_golden.npz")))


def test_views_and_rotation_grid_match_the_reference_methods(golden):
    from foundationpose_b200 import hypotheses as hy

    gen, g = golden
    assert np.abs(hy.sample_views_icosphere(40) - g["views_40"]).max() < 1e-12
    assert np.abs(hy.sample_views_icosphere(1, subdivisions=2, radius=0.5) - g["views_sub2"]).max() < 1e-12
    for name, syms in gen.symmetry_sets().items():
        got = hy.make_rotation_grid(40, 60, syms)
        want = g[f"rot_grid.{name}"]
        assert got.shape == want.shape, (name, got.shape, want.shape)      # 252 / 126 / 20 / 63 start poses
        assert np.abs(got - want).max() < 1e-6, name
    assert np.abs(hy.make_rotation_grid(10, 90, None) - g["rot_grid.identity_10_90"]).max() < 1e-6


def test_cluster_poses_matches_the_reference_cpp(golden):
    from foundationpose_b200 import hypotheses as hy

    gen, g = golden
    grid = g["rot_grid.identity"]
    for name, syms in gen.symmetry_sets().items():
        for ang in (10, 61):
            assert np.array_equal(hy.cluster_poses(ang, 99999, grid, syms), g[f"cluster.{name}.{ang}"]), (name, ang)
    assert np.array_equal(hy.cluster_poses(30, 0.01, g["moved_poses"], gen.symmetry_sets()["half_z"]), g["cluster.moved.half_z"])


def test_cluster_poses_against_the_compiled_reference_function(golden):
    """The same, on random pose sets: what the compiled reference function (oracle/_ref/libcluster_ref.so, built by
    oracle/build_ref.py) kept of each set, stored as indices into it by tools/make_golden_cluster.py."""
    from foundationpose_b200 import hypotheses as hy

    gen, _ = golden
    g = np.load(os.path.join(ROOT, "tests", "golden", "cluster_random_golden.npz"))
    for trial in range(4):
        poses = g[f"poses.{trial}"]
        for name, syms in gen.symmetry_sets().items():
            a = hy.cluster_poses(25 + 5 * trial, 0.03, poses, syms)
            b = poses[g[f"kept.{trial}.{name}"]]
            assert a.shape == b.shape and np.array_equal(a, b), (trial, name, a.shape, b.shape)
