"""GPU parity against the REFERENCE'S OWN CUDA KERNELS: the reference's .cu files compiled unmodified for sm_100 into
oracle/_ref/libsamplenet_ref_cuda.so (oracle/Makefile, oracle/ref_cuda_shim.cu) and run on a B200 on the inputs generated here; their
results are stored in tests/golden/reference_cuda.npz (tests/golden/make_ref_golden.py: digests where the comparison is bit-exact,
arrays or seeded samples of them where it has a tolerance) -- north_star: "outputs match the reference's own TF/CUDA ops on identical
inputs (kNN indices and match assignments bit-exact, distances/losses within a stated fp32 tolerance)".
"""
import os

import numpy as np
import pytest
import torch

from oracle import golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    import samplenet_b200

    samplenet_b200._lib.lib()
    return samplenet_b200


@pytest.fixture(scope="module")
def ref_cuda(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_cuda.npz"))


def _clouds(seed, b, n, m, noise=0.02):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(b, n, 3, generator=g) - 0.5
    if m <= n:
        q = x[:, torch.randperm(n, generator=g)[:m]] + noise * torch.randn(b, m, 3, generator=g)
    else:
        q = torch.rand(b, m, 3, generator=g) - 0.5
    return x.cuda().contiguous(), q.cuda().contiguous()


@pytest.mark.parametrize("b,n,m", [(32, 64, 1024), (4, 37, 129), (2, 513, 511), (32, 1024, 1024), (50, 2048, 2048), (3, 5, 2000)])
def test_chamfer_forward_equals_reference_kernels(sb, ref_cuda, b, n, m):
    """registration ChamferDistanceKernel and TF NmDistanceKernel (same algorithm, two files): indices AND squared distances bit-identical
    to this library's kernel in its default (FMA-contracted, what nvcc gives the reference) arithmetic."""
    x, q = _clouds(b + n + m, b, m, n)          # xyz1 = q (b, n, 3), xyz2 = x (b, m, 3)
    d1, i1, d2, i2 = sb.ops.nn_distance_forward(q, x)
    for fn in ("chamfer_forward", "nn_distance"):
        key = "%s_%d_%d_%d" % (fn, b, n, m)
        assert golden.digest(i1, i2) == ref_cuda[key + "_idx"]
        assert golden.digest(d1, d2) == ref_cuda[key + "_dist"]


def test_chamfer_backward_vs_reference_kernels(sb, ref_cuda):
    x, q = _clouds(3, 8, 1024, 64)
    d1, i1, d2, i2 = sb.ops.nn_distance_forward(q, x)
    g = torch.Generator().manual_seed(5)
    g1 = torch.rand(d1.shape, generator=g).cuda(); g2 = torch.rand(d2.shape, generator=g).cuda()
    gx1, gx2 = sb.ops.nn_distance_backward(q, x, g1, i1, g2, i2)
    # the reference's float atomics: order-dependent rounding
    np.testing.assert_allclose(*golden.pair(ref_cuda, "chamfer_backward_grad1", gx1), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(*golden.pair(ref_cuda, "chamfer_backward_grad2", gx2), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("b,n,m,k", [(32, 1024, 64, 8), (32, 1024, 32, 7), (4, 2048, 64, 16), (3, 200, 17, 3), (2, 1024, 1024, 7)])
def test_knn_equals_reference_selection_sort(sb, ref_cuda, b, n, m, k):
    """tf_grouping.knn_point = TF distance matrix + the reference's selection-sort kernel (tf_grouping_g.cu:83-123): neighbour indices
    bit-exact (tie-free inputs), squared distances bit-exact in this library's unfused arithmetic mode (three roundings, the order TF's
    elementwise graph evaluates)."""
    x, q = _clouds(b * 7 + k, b, n, m)
    o = sb.ops.knn_soft_project_forward(x, q, k, "bnc", want=("idx", "val"), unfused=True)
    key = "knn_%d_%d_%d_%d" % (b, n, m, k)
    assert golden.digest(o["idx"]) == ref_cuda[key + "_idx"]
    assert golden.digest(o["val"]) == ref_cuda[key + "_val"]
    # group_point on those indices
    assert golden.digest(sb.tf_ops.group_point(x, o["idx"])) == ref_cuda[key + "_group"]


@pytest.mark.parametrize("n,m", [(64, 64), (96, 32), (300, 300), (2048, 2048)])
def test_emd_vs_reference_kernels(sb, ref_cuda, oracle, n, m):
    """approxmatch / matchcost / matchcostgrad of tf_approxmatch_g.cu (float, __expf, 512-thread tree reductions) on identical inputs.
    The reference GPU kernel is itself only an approximation of its CPU twin (its self-test flags |diff| > 1e-2, approxmatch.cpp:222);
    this library's fast kernel and its exact mode are both compared (on a seeded sample of the reference match's entries), and cost /
    gradients on IDENTICAL match: the oracle's, which both sides can reproduce."""
    b = 2 if n < 2048 else 1
    g = torch.Generator().manual_seed(n + m)
    a = torch.rand(b, n, 3, generator=g).cuda(); c = torch.rand(b, m, 3, generator=g).cuda()
    key = "emd_%d_%d" % (n, m)
    fast = sb.tf_ops.approx_match(a, c)
    ours, rm = golden.pair(ref_cuda, key + "_match", fast)
    assert np.abs(ours - rm).max() < 5e-3
    if n <= 300:
        exact = sb.tf_ops.approx_match(a, c, exact=True)
        ours, rm = golden.pair(ref_cuda, key + "_match", exact)
        assert np.abs(ours - rm).max() < 5e-3
        # assignments: each one among the columns within that tolerance of the row maximum of the reference's match
        am = exact.argmax(dim=2).cpu().numpy()
        assert bool((ref_cuda[key + "_near"] == am[..., None]).any(axis=2).all())
    om = torch.from_numpy(oracle.approx_match(a.cpu().numpy(), c.cpu().numpy())).cuda()
    oc = sb.ops.match_cost_forward(a, c, om)
    np.testing.assert_allclose(oc.cpu().numpy(), ref_cuda[key + "_cost"], rtol=2e-5)
    og1, og2 = sb.ops.match_cost_grad(a, c, om)
    np.testing.assert_allclose(*golden.pair(ref_cuda, key + "_grad1", og1), rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(*golden.pair(ref_cuda, key + "_grad2", og2), rtol=2e-4, atol=2e-5)
