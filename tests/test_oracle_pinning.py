"""Pin the CPU oracle before trusting it (no GPU needed):
  * against the reference's OWN CPU code compiled unmodified into oracle/_ref (Chamfer fwd/bwd bit-exact, EMD); its results on these
    inputs are stored in tests/golden/reference_cpu.npz (tests/golden/make_ref_golden.py),
  * against the known-answer vectors printed in the reference's self-tests
    (registration/src/soft_projection.py:161-222, classification/soft_projection.py:90-119),
  * against tests/golden/*.npz, produced by importing the reference Python classes (tests/golden/make_golden.py).
"""
import os

import numpy as np
import pytest

from oracle import golden


def _rng(seed):
    return np.random.default_rng(seed)


@pytest.fixture(scope="module")
def ref_cpu(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_cpu.npz"))


@pytest.mark.parametrize("b,n,m", [(1, 1, 1), (2, 64, 1024), (3, 37, 129), (2, 513, 511), (1, 1024, 64), (4, 5, 3)])
def test_chamfer_oracle_bitexact_vs_reference_cpu(oracle, ref_cpu, b, n, m):
    r = _rng(b * 1000 + n + m)
    a = r.standard_normal((b, n, 3)).astype(np.float32)
    c = r.standard_normal((b, m, 3)).astype(np.float32)
    # duplicated points => exact ties; lowest index must win in both
    if n > 4:
        a[:, 3] = a[:, 1]
    if m > 4:
        c[:, 4] = c[:, 0]
    d1, i1, d2, i2 = oracle.nn_distance(a, c, contract=False)
    key = "chamfer_%d_%d_%d" % (b, n, m)
    assert golden.digest(i1, i2) == ref_cpu[key + "_idx"]
    assert golden.digest(d1, d2) == ref_cpu[key + "_dist"]
    g1 = r.standard_normal((b, n)).astype(np.float32)
    g2 = r.standard_normal((b, m)).astype(np.float32)
    gx1, gx2 = oracle.nn_distance_grad(a, c, g1, i1, g2, i2)
    assert golden.digest(gx1, gx2) == ref_cpu[key + "_grad"]


def test_chamfer_oracle_vs_reference_autograd_fixture(oracle, golden_dir):
    z = np.load(os.path.join(golden_dir, "chamfer_reg.npz"))
    d1, i1, d2, i2 = oracle.nn_distance(z["xyz1"], z["xyz2"], contract=False)
    assert np.array_equal(d1, z["dist1"]) and np.array_equal(d2, z["dist2"])
    gx1, gx2 = oracle.nn_distance_grad(z["xyz1"], z["xyz2"], z["w1"], i1, z["w2"], i2)
    assert np.array_equal(gx1, z["grad_xyz1"]) and np.array_equal(gx2, z["grad_xyz2"])


def test_chamfer_contracted_arithmetic_is_close(oracle):
    """contract=True restates the reference CUDA kernels' FMA order; it may only differ from the CPU order in the last ulp."""
    r = _rng(7)
    a = r.standard_normal((2, 64, 3)).astype(np.float32)
    c = r.standard_normal((2, 1024, 3)).astype(np.float32)
    d1, i1, d2, i2 = oracle.nn_distance(a, c, contract=False)
    e1, j1, e2, j2 = oracle.nn_distance(a, c, contract=True)
    np.testing.assert_allclose(d1, e1, rtol=3e-7, atol=0)
    np.testing.assert_allclose(d2, e2, rtol=3e-7, atol=0)
    assert (i1 != j1).mean() < 0.01 and (i2 != j2).mean() < 0.01


# ---- known-answer vectors of the reference self-tests ------------------------------------------------------
_A = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [5, 4, 4], [4, 5, 4], [4, 4, 5], [8, 7, 7], [7, 8, 7], [7, 7, 8]], np.float32)
_Bc = np.array([[0, 0, 0], [1, 0, 0], [2, 0, 0], [5, 5, 5], [7, 7, 8], [7, 7, 8.5]], np.float32)


def test_reg_selftest_known_answers(oracle):
    """registration/src/soft_projection.py:158-284: k=3; propagate at T=1 -> expected_features_nn_3 (:210-222);
    project with roles swapped at T=0.1 -> expected_nn_cloud (:187-196).  3-decimal golden values."""
    feats = np.arange(1, 31, dtype=np.float32).reshape(6, 5)
    exp_feat = np.array([[6.0, 7.0, 8.0, 9.0, 10.0], [2.459, 3.459, 4.459, 5.459, 6.459], [2.459, 3.459, 4.459, 5.459, 6.459],
                         [16.0, 17.0, 18.0, 19.0, 20.0], [16.0, 17.0, 18.0, 19.0, 20.0], [16.0, 17.0, 18.0, 19.0, 20.0],
                         [22.113, 23.113, 24.113, 25.113, 26.113], [22.113, 23.113, 24.113, 25.113, 26.113],
                         [23.189, 24.189, 25.189, 26.189, 27.189]], np.float32)
    exp_cloud = np.array([[0.333, 0.333, 0.333], [1, 0, 0], [1, 0, 0], [4.333, 4.333, 4.333], [7, 7, 8], [7, 7, 8]], np.float32)
    pts, qry = _Bc[None], _A[None]  # point_cloud = 6 pts, query = 9 pts
    for tie_mode in (0, 1):
        _, idx = oracle.knn_point(3, pts, qry, tie_mode=tie_mode)
        sigma = max(1.0 ** 2, 1e-4)
        _, _, _, prop = oracle.soft_project(pts, qry, idx, sigma, feats=feats[None])
        assert np.abs(prop[0] - exp_feat).max() < 6e-4
        _, idx2 = oracle.knn_point(3, qry, pts, tie_mode=tie_mode)  # roles swapped
        sigma = max(np.float32(0.1) ** 2, 1e-4)
        proj, _, _ = oracle.soft_project(qry, pts, idx2, float(sigma))
        assert np.abs(proj[0] - exp_cloud).max() < 6e-4


def test_cls_selftest_known_answers(oracle):
    """classification/soft_projection.py:86-161: batch of 2 (cloud, 3*cloud), k=3, T=0.01, sigma=T^2 (no clamp):
    soft -> expected_cloud_soft (:106-115), hard -> expected_cloud_hard (:117-119)."""
    exp_soft = np.array([[0.333, 0.333, 0.333], [1, 0, 0], [1, 0, 0], [4.333, 4.333, 4.333], [7, 7, 8], [7, 7, 8]], np.float32)
    exp_hard = np.array([[1, 0, 0], [1, 0, 0], [1, 0, 0], [5, 4, 4], [7, 7, 8], [7, 7, 8]], np.float32)
    pts = np.stack([_A, _A * 3]); qry = np.stack([_Bc, _Bc * 3])
    sigma = float(np.float32(0.01) ** 2)
    _, idx = oracle.knn_point(3, pts, qry, tie_mode=0)
    soft, w, d = oracle.soft_project(pts, qry, idx, sigma)
    hard, wh, _ = oracle.soft_project(pts, qry, idx, sigma, hard=True)
    assert np.abs(soft[0] - exp_soft).max() < 1.1e-3 and np.abs(soft[1] - 3 * exp_soft).max() < 3.1e-3
    assert np.abs(hard[0] - exp_hard).max() < 1e-6 and np.abs(hard[1] - 3 * exp_hard).max() < 1e-6
    assert w.shape == (2, 6, 3) and d.shape == (2, 6, 3)
    np.testing.assert_allclose(w.sum(-1), 1.0, rtol=1e-6)


def test_softproj_oracle_vs_reference_fixture(oracle, golden_dir):
    z = np.load(os.path.join(golden_dir, "softproj_reg.npz"))
    pc = z["point_cloud"].transpose(0, 2, 1); qc = z["query_cloud"].transpose(0, 2, 1)
    feats = z["feats"].transpose(0, 2, 1)
    k = int(z["k"]); sigma = float(max(np.float32(z["temperature"]) ** 2, np.float32(z["min_sigma"])))
    for tie_mode in (0, 1):
        _, idx = oracle.knn_point(k, pc, qc, tie_mode=tie_mode)
        proj, w, d, prop = oracle.soft_project(pc, qc, idx, sigma, feats=feats)
        np.testing.assert_allclose(proj, z["proj"].transpose(0, 2, 1), rtol=2e-6, atol=2e-6)
        np.testing.assert_allclose(prop, z["prop"].transpose(0, 2, 1), rtol=2e-6, atol=2e-6)
        np.testing.assert_allclose(proj, z["only_proj"].transpose(0, 2, 1), rtol=2e-6, atol=2e-6)


def test_knn_tie_modes_agree_without_ties_and_group_point(oracle):
    r = _rng(11)
    pts = r.standard_normal((2, 300, 3)).astype(np.float32)
    qry = r.standard_normal((2, 40, 3)).astype(np.float32)
    v0, i0 = oracle.knn_point(16, pts, qry, tie_mode=0)
    v1, i1 = oracle.knn_point(16, pts, qry, tie_mode=1)
    assert np.array_equal(i0, i1) and np.array_equal(v0, v1)
    assert np.all(np.diff(v0, axis=-1) >= 0)
    # brute force check of the values
    d = ((pts[:, None] - qry[:, :, None]) ** 2).sum(-1)
    np.testing.assert_allclose(np.sort(d, axis=-1)[..., :16], v0, rtol=1e-6)
    g = oracle.group_point(pts, i0)
    assert np.array_equal(g, np.take_along_axis(pts[:, None].repeat(40, 1), i0[..., None].repeat(3, -1), axis=2))
    go = r.standard_normal(g.shape).astype(np.float32)
    gp = oracle.group_point_grad(pts.shape, i0, go)
    ref = np.zeros_like(pts)
    for b in range(2):
        np.add.at(ref[b], i0[b].reshape(-1), go[b].reshape(-1, 3))
    np.testing.assert_allclose(gp, ref, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("n,m", [(64, 64), (96, 32), (40, 120)])
def test_emd_oracle_vs_reference_cpu(oracle, ref_cpu, n, m):
    """approxmatch.cpp:17-125 (double accumulators, (n,m) layout, 10 levels) vs the GPU-semantics restatement
    (float accumulators, (m,n) layout).  Its own self-check flags |diff| > 1e-2 (approxmatch.cpp:222).  The reference's match is
    stored as a seeded sample of its entries and its row-wise arg-max; its cost is of its own match, its gradient of the oracle's."""
    r = _rng(n * 7 + m)
    a = r.random((2, n, 3)).astype(np.float32)
    c = r.random((2, m, 3)).astype(np.float32)
    mt = oracle.approx_match(a, c)  # (b, m, n)
    key = "emd_%d_%d" % (n, m)
    ours, rmt = golden.pair(ref_cpu, key + "_match", mt.transpose(0, 2, 1))  # reference layout (b, n, m)
    assert np.abs(ours - rmt).max() < 5e-3  # float vs double accumulators + 1e-9 placement; the reference flags > 1e-2
    assert np.array_equal(mt.argmax(axis=2), ref_cpu[key + "_argmax"])
    cost = oracle.match_cost(a, c, mt)
    np.testing.assert_allclose(cost, ref_cpu[key + "_cost"], rtol=1e-4)
    g1, g2 = oracle.match_cost_grad(a, c, mt)
    np.testing.assert_allclose(*golden.pair(ref_cpu, key + "_grad2", g2), rtol=1e-4, atol=1e-5)
    # mass conservation property of the matching: every point of the smaller side is fully assigned
    tot = mt.sum(axis=1) if n <= m else mt.sum(axis=2)
    np.testing.assert_allclose(tot, max(n, m) // min(n, m), rtol=2e-3)


def test_nn_matching_oracle_vs_reference_fixture(oracle, golden_dir):
    z = np.load(os.path.join(golden_dir, "samplenet_reg_b2.npz"))
    e = np.load(os.path.join(golden_dir, "samplenet_reg_b2_eval.npz"))
    out = oracle.nn_matching(z["x"], e["nn_idx"], 64, complete_fps=True)
    assert np.array_equal(out, e["match"])
    # and the NN indices themselves: oracle Chamfer idx1 of (simp_eval -> x)
    _, i1, _, _ = oracle.nn_distance(e["simp_eval"], z["x"], contract=False)
    assert np.array_equal(i1, e["nn_idx"])


def test_simplification_loss_oracle_vs_reference_fixture(oracle, golden_dir):
    z = np.load(os.path.join(golden_dir, "samplenet_reg_b2.npz"))
    loss = oracle.simplification_loss(z["x"], z["simp"], 64, 1, 0)
    np.testing.assert_allclose(loss, z["loss_simplification"], rtol=2e-6)
