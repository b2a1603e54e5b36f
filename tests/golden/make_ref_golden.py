"""Results of the reference's own compiled code on the seeded inputs of the tests that compare against it.

oracle/Makefile compiles the reference's CPU code into oracle/_ref/libsamplenet_ref.so and its CUDA kernels into
oracle/_ref/libsamplenet_ref_cuda.so, where the reference sources are available.  This script runs those libraries on exactly the
inputs that tests/test_oracle_pinning.py, tests/test_gpu_parity.py and tests/test_vs_reference_cuda.py generate, and stores what
those tests compare with (oracle/golden.py: digests for bit-exact comparisons, arrays or seeded samples for tolerance ones):

    python tests/golden/make_ref_golden.py cpu  [OUT]   -> tests/golden/reference_cpu.npz    (no GPU needed)
    python tests/golden/make_ref_golden.py cuda [OUT]   -> tests/golden/reference_cuda.npz   (needs a GPU; the stored file was written on an
                                                                                          NVIDIA B200 by the kernels as built for sm_100)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import golden  # noqa: E402
from oracle import oracle as orc  # noqa: E402

# test_chamfer_oracle_bitexact_vs_reference_cpu (first six, with backward) and test_chamfer_forward_bitexact (all eight)
CPU_CHAMFER = [(1, 1, 1), (2, 64, 1024), (3, 37, 129), (2, 513, 511), (1, 1024, 64), (4, 5, 3), (2, 33, 4099), (1, 6000, 70)]
CPU_CHAMFER_BWD = CPU_CHAMFER[:6]
CPU_EMD = [(64, 64), (96, 32), (40, 120)]                                   # test_emd_oracle_vs_reference_cpu
CPU_EMD_ARGMAX = [(64, 64), (96, 32), (40, 120), (77, 77), (300, 300)]      # test_emd_exact_mode_bitexact_vs_oracle (n <= 300)

CUDA_CHAMFER = [(32, 64, 1024), (4, 37, 129), (2, 513, 511), (32, 1024, 1024), (50, 2048, 2048), (3, 5, 2000)]
CUDA_KNN = [(32, 1024, 64, 8), (32, 1024, 32, 7), (4, 2048, 64, 16), (3, 200, 17, 3), (2, 1024, 1024, 7)]
CUDA_EMD = [(64, 64), (96, 32), (300, 300), (2048, 2048)]
EMD_NEAR = 5e-3     # test_emd_vs_reference_kernels: an assignment may be any column this close to the row maximum


def chamfer_inputs(b, n, m):
    r = np.random.default_rng(b * 1000 + n + m)
    a = r.standard_normal((b, n, 3)).astype(np.float32)
    c = r.standard_normal((b, m, 3)).astype(np.float32)
    if n > 4:
        a[:, 3] = a[:, 1]
    if m > 4:
        c[:, 4] = c[:, 0]
    return r, a, c


def make_cpu():
    z = {}
    for b, n, m in CPU_CHAMFER:
        r, a, c = chamfer_inputs(b, n, m)
        d1, i1, d2, i2 = orc.ref_chamfer_forward(a, c)
        key = "chamfer_%d_%d_%d" % (b, n, m)
        z[key + "_idx"] = golden.digest(i1, i2)
        z[key + "_dist"] = golden.digest(d1, d2)
        if (b, n, m) in CPU_CHAMFER_BWD:
            g1 = r.standard_normal((b, n)).astype(np.float32)
            g2 = r.standard_normal((b, m)).astype(np.float32)
            z[key + "_grad"] = golden.digest(*orc.ref_chamfer_backward(a, c, g1, i1, g2, i2))
    for n, m in CPU_EMD:
        r = np.random.default_rng(n * 7 + m)
        a = r.random((2, n, 3)).astype(np.float32)
        c = r.random((2, m, 3)).astype(np.float32)
        key = "emd_%d_%d" % (n, m)
        rmt = orc.ref_approxmatch_cpu(a, c)                              # (b, n, m)
        golden.put(z, key + "_match", rmt)
        z[key + "_argmax"] = rmt.transpose(0, 2, 1).argmax(axis=2).astype(np.int32)
        z[key + "_cost"] = orc.ref_matchcost_cpu(a, c, rmt)
        mt = orc.approx_match(a, c)                                      # the oracle's match, (b, m, n)
        golden.put(z, key + "_grad2", orc.ref_matchcostgrad_cpu(a, c, np.ascontiguousarray(mt.transpose(0, 2, 1))))
    for n, m in CPU_EMD_ARGMAX:
        r = np.random.default_rng(n * 13 + m)
        a = r.random((3, n, 3)).astype(np.float32)
        c = r.random((3, m, 3)).astype(np.float32)
        z["emd_exact_%d_%d_argmax" % (n, m)] = orc.ref_approxmatch_cpu(a, c).transpose(0, 2, 1).argmax(axis=2).astype(np.int32)
    return z


def clouds(seed, b, n, m, noise=0.02):
    import torch

    g = torch.Generator().manual_seed(seed)
    x = torch.rand(b, n, 3, generator=g) - 0.5
    if m <= n:
        q = x[:, torch.randperm(n, generator=g)[:m]] + noise * torch.randn(b, m, 3, generator=g)
    else:
        q = torch.rand(b, m, 3, generator=g) - 0.5
    return x.cuda().contiguous(), q.cuda().contiguous()


def make_cuda():
    import torch

    from oracle import ref_cuda as refcu

    def n_(t):
        return t.detach().cpu().numpy()

    z = {}
    for b, n, m in CUDA_CHAMFER:
        x, q = clouds(b + n + m, b, m, n)
        for fn in (refcu.chamfer_forward, refcu.nn_distance):
            d1, i1, d2, i2 = fn(q, x)
            key = "%s_%d_%d_%d" % (fn.__name__, b, n, m)
            z[key + "_idx"] = golden.digest(i1, i2)
            z[key + "_dist"] = golden.digest(d1, d2)
    x, q = clouds(3, 8, 1024, 64)
    d1, i1, d2, i2 = refcu.chamfer_forward(q, x)
    g = torch.Generator().manual_seed(5)
    g1 = torch.rand(d1.shape, generator=g).cuda(); g2 = torch.rand(d2.shape, generator=g).cuda()
    rx1, rx2 = refcu.chamfer_backward(q, x, g1, i1, g2, i2)
    golden.put(z, "chamfer_backward_grad1", n_(rx1))
    golden.put(z, "chamfer_backward_grad2", n_(rx2))
    for b, n, m, k in CUDA_KNN:
        x, q = clouds(b * 7 + k, b, n, m)
        val, idx = refcu.knn_point(k, x, q)
        key = "knn_%d_%d_%d_%d" % (b, n, m, k)
        z[key + "_idx"] = golden.digest(idx)
        z[key + "_val"] = golden.digest(val)
        z[key + "_group"] = golden.digest(refcu.group_point(x, idx))
    for n, m in CUDA_EMD:
        b = 2 if n < 2048 else 1
        g = torch.Generator().manual_seed(n + m)
        a = torch.rand(b, n, 3, generator=g).cuda(); c = torch.rand(b, m, 3, generator=g).cuda()
        key = "emd_%d_%d" % (n, m)
        rm = n_(refcu.approx_match(a, c))                                # (b, m, n)
        golden.put(z, key + "_match", rm)
        if n <= 300:   # per row, every column within EMD_NEAR of the row maximum (-1 pads): the assignments the test accepts
            near = rm.max(axis=2, keepdims=True) - rm < EMD_NEAR
            cols = np.full(rm.shape[:2] + (int(near.sum(axis=2).max()),), -1, np.int32)
            for i in range(b):
                for j in range(m):
                    js = np.nonzero(near[i, j])[0]
                    cols[i, j, :len(js)] = js
            z[key + "_near"] = cols
        om = torch.from_numpy(orc.approx_match(n_(a), n_(c))).cuda()    # the oracle's match: an input both sides can reproduce
        z[key + "_cost"] = n_(refcu.match_cost(a, c, om))
        rg1, rg2 = refcu.match_cost_grad(a, c, om)
        golden.put(z, key + "_grad1", n_(rg1))
        golden.put(z, key + "_grad2", n_(rg2))
    torch.cuda.synchronize()
    return z


if __name__ == "__main__":
    what = sys.argv[1]
    out = sys.argv[2] if len(sys.argv) > 2 else os.path.join(HERE, "reference_%s.npz" % what)
    z = make_cpu() if what == "cpu" else make_cuda()
    np.savez_compressed(out, **z)
    print(out, os.path.getsize(out), "bytes,", len(z), "entries")
