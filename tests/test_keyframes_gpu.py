"""SLAM keyframe overlap score on the GPU (must3r_b200/engine/keyframes.py) against the UNMODIFIED reference's own
functions (must3r/slam/model.py:62-91 get_overlap_score, must3r/slam/nns.py searchers on scipy KD-trees), whose outputs
on the same seeded frames are stored in tests/golden/keyframes.npz (tests/golden/make_golden.py keyframes)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from helpers import KEYFRAME_CAM, KEYFRAME_DB, KEYFRAME_METHODS, KEYFRAME_QUERIES, keyframe_frame, load_golden  # noqa: E402
from must3r_b200.engine import keyframes as kf  # noqa: E402

pytestmark = pytest.mark.gpu


def test_nn_min_dist_matches_brute_force_and_kdtree():
    from scipy.spatial import KDTree
    g = torch.Generator().manual_seed(0)
    db, q = torch.randn(5000, 3, generator=g), torch.randn(777, 3, generator=g) * 1.5
    d = kf.nn_min_dist(q.cuda(), db.cuda()).cpu()
    want, _ = KDTree(db.numpy()).query(q.numpy(), k=1)
    assert np.allclose(d.numpy(), want, rtol=1e-5, atol=1e-6)
    assert torch.isinf(kf.nn_min_dist(q.cuda(), torch.zeros(0, 3).cuda())).all()


@pytest.mark.parametrize("method", KEYFRAME_METHODS)
@pytest.mark.parametrize("mode", ["nn", "nn-norm"])
def test_overlap_score_matches_reference(method, mode):
    g = load_golden("keyframes.npz")
    tree = kf.get_searcher(method)
    cam = torch.tensor(KEYFRAME_CAM)
    for seed, shift in KEYFRAME_DB:                      # three keyframes in the database
        fr = keyframe_frame(seed, shift=shift)
        sel = fr["pts3d"][0, 0, ::2, ::2][fr["conf"][0, 0, ::2, ::2] > 1.5]
        tree.add_pts(sel.cuda(), cam_center=cam.cuda())
    for seed, shift in KEYFRAME_QUERIES:                 # an overlapping and a far-away frame
        fr = keyframe_frame(seed, shift=shift)
        want = float(g[f"{method}.{mode}.{seed}.score"])
        got = kf.get_overlap_score({k: v.cuda() for k, v in fr.items()}, tree, cam.cuda(), mode=mode, kf_x_subsamp=2,
                                   min_conf_keyframe=1.5, percentile=70)
        assert abs(got - want) <= 2e-5 * max(1.0, abs(want)), (method, mode, got, want)
        assert kf.choose_keyframe_from_overlap(got, 0.1, mode) == bool(g[f"{method}.{mode}.{seed}.choice"])
    empty = kf.get_searcher(method)                      # nothing stored yet: every distance is "infinite"
    fr = keyframe_frame(60)
    want = float(g[f"{method}.empty.score"])
    got = kf.get_overlap_score({k: v.cuda() for k, v in fr.items()}, empty, cam.cuda(), mode="nn", kf_x_subsamp=2)
    assert got == pytest.approx(want, rel=1e-6) or (got > 1e30 and want > 1e30)


def test_conf_modes_and_quadrants():
    g = load_golden("keyframes.npz")
    fr = keyframe_frame(70)
    for mode in ("meanconf", "medianconf"):
        assert float(kf.get_overlap_score({k: v.cuda() for k, v in fr.items()}, None, None, mode=mode)) == pytest.approx(
            float(g[f"{mode}.score"]), rel=1e-6)
    rays = torch.randn(4000, 3, generator=torch.Generator().manual_seed(3))
    for div in (2, 4):
        want = g[f"quadrant{div}"]
        got = kf.get_quadrant_id(rays.cuda(), div).cpu().numpy()
        assert (got != want).mean() < 1e-3                # bin edges: fp32 vs fp64 trig may differ on a handful of rays
