"""torch-facing wrappers of the C-ABI kernels: argument checks, output allocation, autograd Functions.

Every function launches on torch's CURRENT CUDA stream and never synchronises, so whole steps can be captured into
CUDA graphs.  CPU tensors are rejected: there is no fallback path.
"""
import ctypes
import os
import threading

import torch

from . import _lib
from ._lib import BCN, BNC, DIST_FMA, DIST_UNFUSED, Layer, LayerGrad, check, lib

_LAYOUTS = {"bnc": BNC, "bcn": BCN}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _req(t, name, dtype=torch.float32):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise RuntimeError("samplenet_b200: %s is on %s; the ops are CUDA-only (no CPU fallback)" % (name, t.device))
    if t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    return t.contiguous()


def _layout(s):
    try:
        return _LAYOUTS[s]
    except KeyError:
        raise ValueError("layout must be 'bnc' or 'bcn', got %r" % (s,))


# ----------------------------------------------------------------------------------------------------- Chamfer
def nn_distance_forward(xyz1, xyz2, unfused=False):
    """dist1 (B,n), idx1 (B,n) int32, dist2 (B,m), idx2 (B,m) int32 for BNC clouds xyz1 (B,n,3), xyz2 (B,m,3)."""
    xyz1, xyz2 = _req(xyz1, "xyz1"), _req(xyz2, "xyz2")
    if xyz1.dim() != 3 or xyz2.dim() != 3 or xyz1.shape[2] != 3 or xyz2.shape[2] != 3:
        raise ValueError("nn_distance expects (batch, points, 3) tensors, got %s and %s" % (tuple(xyz1.shape), tuple(xyz2.shape)))
    if xyz1.shape[0] != xyz2.shape[0]:
        raise ValueError("nn_distance: batch sizes differ (%d vs %d)" % (xyz1.shape[0], xyz2.shape[0]))
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    with torch.cuda.device(xyz1.device):
        dist1 = torch.empty(b, n, device=xyz1.device, dtype=torch.float32)
        dist2 = torch.empty(b, m, device=xyz1.device, dtype=torch.float32)
        idx1 = torch.empty(b, n, device=xyz1.device, dtype=torch.int32)
        idx2 = torch.empty(b, m, device=xyz1.device, dtype=torch.int32)
        check(lib().snb200_nn_distance_forward(b, n, _p(xyz1), m, _p(xyz2), _p(dist1), _p(idx1), _p(dist2), _p(idx2),
                                               DIST_UNFUSED if unfused else DIST_FMA, _stream()), "nn_distance_forward")
    return dist1, idx1, dist2, idx2


def nn_distance_backward(xyz1, xyz2, g1, idx1, g2, idx2):
    xyz1, xyz2, g1, g2 = _req(xyz1, "xyz1"), _req(xyz2, "xyz2"), _req(g1, "grad_dist1"), _req(g2, "grad_dist2")
    idx1, idx2 = _req(idx1, "idx1", torch.int32), _req(idx2, "idx2", torch.int32)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    with torch.cuda.device(xyz1.device):
        gx1 = torch.empty_like(xyz1)
        gx2 = torch.empty_like(xyz2)
        check(lib().snb200_nn_distance_backward(b, n, _p(xyz1), m, _p(xyz2), _p(g1), _p(idx1), _p(g2), _p(idx2), _p(gx1), _p(gx2),
                                                _stream()), "nn_distance_backward")
    return gx1, gx2


class NNDistanceFunction(torch.autograd.Function):
    """Mirrors ChamferDistanceFunction (registration/src/chamfer_distance/chamfer_distance.py:14-61) and the TF op pair
    NnDistance / NnDistanceGrad (classification/structural_losses/tf_nndistance.py:12-47): returns all four outputs;
    the index outputs are non-differentiable."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, unfused=False):
        dist1, idx1, dist2, idx2 = nn_distance_forward(xyz1, xyz2, unfused)
        ctx.save_for_backward(xyz1.contiguous(), xyz2.contiguous(), idx1, idx2)
        ctx.mark_non_differentiable(idx1, idx2)
        return dist1, idx1, dist2, idx2

    @staticmethod
    def backward(ctx, g1, gi1, g2, gi2):
        xyz1, xyz2, idx1, idx2 = ctx.saved_tensors
        if g1 is None:
            g1 = torch.zeros(idx1.shape, device=xyz1.device, dtype=torch.float32)
        if g2 is None:
            g2 = torch.zeros(idx2.shape, device=xyz1.device, dtype=torch.float32)
        gx1, gx2 = nn_distance_backward(xyz1, xyz2, g1, idx1, g2, idx2)
        return gx1, gx2, None


def simplification_loss_forward(samp, ref, weight21, unfused=False):
    """Fused Chamfer + reductions.  Returns (out4, dist1, idx1, dist2, idx2); out4 = [mean c12, mean max c12, mean c21, loss]."""
    samp, ref = _req(samp, "samp_pc"), _req(ref, "ref_pc")
    if samp.dim() != 3 or ref.dim() != 3 or samp.shape[2] != 3 or ref.shape[2] != 3 or samp.shape[0] != ref.shape[0]:
        raise ValueError("simplification loss expects (B,M,3) and (B,N,3) tensors")
    b, n, _ = samp.shape
    m = ref.shape[1]
    dev = samp.device
    with torch.cuda.device(dev):
        dist1 = torch.empty(b, n, device=dev); dist2 = torch.empty(b, m, device=dev)
        idx1 = torch.empty(b, n, device=dev, dtype=torch.int32); idx2 = torch.empty(b, m, device=dev, dtype=torch.int32)
        out4 = torch.empty(4, device=dev)
        check(lib().snb200_simplification_loss_forward(b, n, _p(samp), m, _p(ref), float(weight21), _p(dist1), _p(idx1), _p(dist2), _p(idx2),
                                                       _p(out4), None, 0, DIST_UNFUSED if unfused else DIST_FMA, _stream()),
              "simplification_loss_forward")
    return out4, dist1, idx1, dist2, idx2


class SimplificationLossFunction(torch.autograd.Function):
    """loss = mean(c12) + mean_b(max c12) + w * mean(c21), c12/c21 = Chamfer(samp, ref)
    (registration/src/samplenet.py:171-181).  Backward routes through the deterministic Chamfer backward kernel."""

    @staticmethod
    def forward(ctx, samp, ref, weight21):
        out4, dist1, idx1, dist2, idx2 = simplification_loss_forward(samp, ref, weight21)
        ctx.save_for_backward(samp.contiguous(), ref.contiguous(), dist1, idx1, idx2)
        ctx.w = float(weight21)
        return out4[3].clone()

    @staticmethod
    def backward(ctx, g):
        samp, ref, dist1, idx1, idx2 = ctx.saved_tensors
        b, n = dist1.shape
        m = idx2.shape[1]
        # d loss / d dist1[b,j] = 1/(b n) + [j == argmax_j dist1[b]] / b ;  d loss / d dist2 = w / (b m)
        g1 = torch.full((b, n), 1.0 / (b * n), device=samp.device)
        am = dist1.argmax(dim=1, keepdim=True)
        g1.scatter_add_(1, am, torch.full((b, 1), 1.0 / b, device=samp.device))
        g2 = torch.full((b, m), ctx.w / (b * m), device=samp.device)
        g1 = g1 * g
        g2 = g2 * g
        gs, gr = nn_distance_backward(samp, ref, g1, idx1, g2, idx2)
        return gs, gr, None


# ----------------------------------------------------------------------------------------------------- kNN / projection
def knn_soft_project_forward(points, query, k, layout, sigma=None, hard=False, feats=None, want=("proj",), unfused=False,
                             sigma_mode=0, sigma_floor=0.0):
    """One fused launch.  `want` is a subset of {"proj","prop","idx","val","weights","dist"}; returns a dict of tensors.
    sigma_mode / sigma_floor: how the `sigma` scalar is interpreted (see SNB200_SIGMA_* in the header)."""
    lay = _layout(layout)
    points, query = _req(points, "point_cloud"), _req(query, "query_cloud")
    if points.dim() != 3 or query.dim() != 3 or points.shape[0] != query.shape[0]:
        raise ValueError("soft projection expects 3-D clouds with equal batch sizes")
    cdim = 2 if lay == BNC else 1
    if points.shape[cdim] != 3 or query.shape[cdim] != 3:
        raise ValueError("soft projection: channel dimension must be 3 for layout %r, got %s / %s" % (layout, tuple(points.shape), tuple(query.shape)))
    b = points.shape[0]
    n = points.shape[1] if lay == BNC else points.shape[2]
    m = query.shape[1] if lay == BNC else query.shape[2]
    k = int(k)
    dev = points.device
    f = 0
    if feats is not None:
        feats = _req(feats, "point_features")
        f = feats.shape[2] if lay == BNC else feats.shape[1]
        nf = feats.shape[1] if lay == BNC else feats.shape[2]
        if nf != n or feats.shape[0] != b:
            raise ValueError("point_features must cover the same points as point_cloud")
    if sigma is not None:
        sigma = _req(sigma.reshape(1), "sigma")
    out = {}
    with torch.cuda.device(dev):
        if "proj" in want:
            out["proj"] = torch.empty_like(query)
        if "prop" in want:
            out["prop"] = torch.empty((b, m, f) if lay == BNC else (b, f, m), device=dev)
        if "idx" in want:
            out["idx"] = torch.empty(b, m, k, device=dev, dtype=torch.int32)
        if "val" in want:
            out["val"] = torch.empty(b, m, k, device=dev)
        if "weights" in want:
            out["weights"] = torch.empty(b, m, k, device=dev)
        if "dist" in want:
            out["dist"] = torch.empty(b, m, k, device=dev)
        check(lib().snb200_knn_soft_project_forward(
            b, n, m, k, lay, _p(points), _p(query), _p(sigma), int(sigma_mode), float(sigma_floor), int(bool(hard)), _p(feats), f,
            _p(out.get("proj")), _p(out.get("prop")),
            _p(out.get("idx")), _p(out.get("val")), _p(out.get("weights")), _p(out.get("dist")), DIST_UNFUSED if unfused else DIST_FMA,
            _stream()), "knn_soft_project_forward")
    return out


def soft_project_backward(points, query, sigma, feats, idx, weights, grad_proj, grad_prop, layout, need_points, need_query, need_feats,
                          need_sigma, sigma_mode=0, sigma_floor=0.0):
    lay = _layout(layout)
    b = points.shape[0]
    n = points.shape[1] if lay == BNC else points.shape[2]
    m = query.shape[1] if lay == BNC else query.shape[2]
    k = idx.shape[2]
    f = 0 if feats is None else (feats.shape[2] if lay == BNC else feats.shape[1])
    dev = points.device
    with torch.cuda.device(dev):
        gp = torch.empty_like(points) if need_points else None
        gq = torch.empty_like(query) if need_query else None
        gf = torch.empty_like(feats) if (need_feats and feats is not None) else None
        gs = torch.empty(1, device=dev) if need_sigma else None
        wsb = lib().snb200_soft_project_backward_workspace_bytes(b, n, m, k, f)
        ws = torch.empty(max(int(wsb), 4), device=dev, dtype=torch.uint8)
        gproj = None if grad_proj is None else _req(grad_proj, "grad_proj")
        gprop = None if grad_prop is None else _req(grad_prop, "grad_prop")
        check(lib().snb200_soft_project_backward(
            b, n, m, k, lay, _p(points), _p(query), _p(sigma), int(sigma_mode), float(sigma_floor), _p(feats), f, _p(idx), _p(weights),
            _p(gproj), _p(gprop), _p(gp), _p(gq),
            _p(gf), _p(gs), _p(ws), int(wsb), _stream()), "soft_project_backward")
    return gp, gq, gf, gs


class SoftProjectFunction(torch.autograd.Function):
    """(points, query, t[, feats]) -> (proj, prop, weights, dist, idx); differentiable in points, query, t, feats.

    `t` is either sigma itself (sigma_mode 0) or the temperature parameter, in which case the kernel evaluates the
    sub-project's clamp (sigma_mode 1: max(T^2, floor) registration; 2: T^2 classification; 3: max(T, floor)^2 reconstruction)
    and the chain rule d sigma / d T is applied here in backward."""

    @staticmethod
    def forward(ctx, points, query, t, feats, k, layout, hard, want_proj, want_prop, sigma_mode=0, sigma_floor=0.0):
        want = ["idx", "weights", "dist"]
        if want_proj:
            want.append("proj")
        if want_prop:
            want.append("prop")
        points = points.contiguous(); query = query.contiguous()
        sig = t.detach().reshape(1).contiguous()
        o = knn_soft_project_forward(points, query, k, layout, sig, hard, feats, want, sigma_mode=sigma_mode, sigma_floor=sigma_floor)
        ctx.layout = layout
        ctx.hard = hard
        ctx.has_feats = feats is not None
        ctx.sigma_mode, ctx.sigma_floor = int(sigma_mode), float(sigma_floor)
        ctx.save_for_backward(points, query, sig, feats.contiguous() if feats is not None else None, o["idx"], o["weights"])
        proj = o.get("proj"); prop = o.get("prop")
        # weights / dist are returned for inspection (the TF SoftProjection returns them too); only the projection and the propagated features
        # carry gradients, as in every reference caller -- marked so autograd does not pretend otherwise
        ctx.mark_non_differentiable(o["idx"], o["weights"], o["dist"])
        ctx.sigma_shape = t.shape
        dev = points.device
        if proj is None:
            proj = torch.empty(0, device=dev)
        if prop is None:
            prop = torch.empty(0, device=dev)
        return proj, prop, o["weights"], o["dist"], o["idx"]

    @staticmethod
    def backward(ctx, g_proj, g_prop, g_w, g_d, g_i):
        points, query, sig, feats, idx, weights = ctx.saved_tensors
        if ctx.hard:
            raise NotImplementedError("hard projection is not differentiable (registration/src/soft_projection.py:144-145)")
        if g_proj is not None and g_proj.numel() == 0:
            g_proj = None
        if g_prop is not None and g_prop.numel() == 0:
            g_prop = None
        if g_proj is None and g_prop is None:
            return (None,) * 11
        need = ctx.needs_input_grad
        gp, gq, gf, gs = soft_project_backward(points, query, sig, feats, idx, weights, g_proj, g_prop, ctx.layout, need[0], need[1],
                                               need[3] and ctx.has_feats, need[2], ctx.sigma_mode, ctx.sigma_floor)
        if gs is not None:   # d sigma / d T for the temperature modes
            tt, fl = sig, ctx.sigma_floor
            if ctx.sigma_mode == 1:
                gs = gs * torch.where(tt * tt > fl, 2.0 * tt, torch.zeros_like(tt))
            elif ctx.sigma_mode == 2:
                gs = gs * 2.0 * tt
            elif ctx.sigma_mode == 3:
                gs = gs * torch.where(tt > fl, 2.0 * tt, torch.zeros_like(tt))
            gs = gs.reshape(ctx.sigma_shape)
        return gp, gq, gs, gf, None, None, None, None, None, None, None


_TICKETS = {}


def _ticket(dev):
    """One zero-initialised device counter per (GPU, stream) for the last-CTA reductions (fused tail, progressive loss); the kernels leave
    it zero.  Launches that share a word are stream-ordered by construction; concurrent launches on different streams get different
    words.  (A kernel that traps leaves the context unusable anyway.)  The C ABI takes the word as an argument."""
    key = (dev.type, dev.index, torch.cuda.current_stream(dev).cuda_stream)   # launches on different streams never share a word
    t = _TICKETS.get(key)
    if t is None:
        t = torch.zeros(1, device=dev, dtype=torch.int32)
        _TICKETS[key] = t
    return t


def project_and_loss_forward(ref, samp, k, t, sigma_mode, sigma_floor, weight21, unfused=False):
    """One launch: proj, (idx, weights, dist) for the projection backward, Chamfer dist/idx both ways, out4 loss terms."""
    ref, samp = _req(ref, "ref_pc"), _req(samp, "samp_pc")
    b, n, _ = ref.shape
    m = samp.shape[1]
    dev = ref.device
    tt = _req(t.detach().reshape(1), "temperature")
    with torch.cuda.device(dev):
        proj = torch.empty_like(samp)
        idx = torch.empty(b, m, k, device=dev, dtype=torch.int32)
        w = torch.empty(b, m, k, device=dev); d = torch.empty(b, m, k, device=dev)
        dist1 = torch.empty(b, m, device=dev); idx1 = torch.empty(b, m, device=dev, dtype=torch.int32)
        dist2 = torch.empty(b, n, device=dev); idx2 = torch.empty(b, n, device=dev, dtype=torch.int32)
        out4 = torch.empty(4, device=dev)
        wsb = int(lib().snb200_project_and_loss_workspace_bytes(b, m, n))
        ws = torch.empty(max(wsb, 4), device=dev, dtype=torch.uint8)
        check(lib().snb200_project_and_loss_forward(b, n, m, int(k), _p(ref), _p(samp), _p(tt), int(sigma_mode), float(sigma_floor), _p(proj), _p(idx),
                                                    _p(w), _p(d), _p(dist1), _p(idx1), _p(dist2), _p(idx2), float(weight21), _p(out4), _p(ws), wsb,
                                                    _p(_ticket(dev)), DIST_UNFUSED if unfused else DIST_FMA, _stream()), "project_and_loss_forward")
    return proj, idx, w, d, dist1, idx1, dist2, idx2, out4


class ProjectAndLossFunction(torch.autograd.Function):
    """(ref, samp, temperature) -> (proj, loss_w1, terms): the projection of `samp` onto `ref` together with the simplification
    loss of (samp, ref) evaluated for weight 1 (`loss_w1`) and its three terms (`terms` = [mean c12, mean max c12, mean c21]).
    Backward = soft-projection backward + Chamfer backward (both deterministic kernels)."""

    @staticmethod
    def forward(ctx, ref, samp, t, k, sigma_mode, sigma_floor):
        ref = ref.contiguous(); samp = samp.contiguous()
        proj, idx, w, d, dist1, idx1, dist2, idx2, out4 = project_and_loss_forward(ref, samp, k, t, sigma_mode, sigma_floor, 1.0)
        ctx.save_for_backward(ref, samp, t.detach().reshape(1).contiguous(), idx, w, dist1, idx1, idx2)
        ctx.sigma_mode, ctx.sigma_floor, ctx.t_shape = int(sigma_mode), float(sigma_floor), t.shape
        return proj, out4[3], out4[:3]

    @staticmethod
    def backward(ctx, g_proj, g_unit, g_terms):
        ref, samp, tt, idx, w, dist1, idx1, idx2 = ctx.saved_tensors
        need = ctx.needs_input_grad
        b, m = dist1.shape
        n = idx2.shape[1]
        dev = ref.device
        g_ref = g_samp = g_t = None
        if g_proj is not None:
            gp, gq, _, gs = soft_project_backward(ref, samp, tt, None, idx, w, g_proj.contiguous(), None, "bnc", need[0], need[1], False, need[2],
                                                  ctx.sigma_mode, ctx.sigma_floor)
            g_ref, g_samp = gp, gq
            if gs is not None:
                fl = ctx.sigma_floor
                if ctx.sigma_mode == 1:
                    gs = gs * torch.where(tt * tt > fl, 2.0 * tt, torch.zeros_like(tt))
                elif ctx.sigma_mode == 2:
                    gs = gs * 2.0 * tt
                elif ctx.sigma_mode == 3:
                    gs = gs * torch.where(tt > fl, 2.0 * tt, torch.zeros_like(tt))
                g_t = gs.reshape(ctx.t_shape)
        if g_unit is not None or g_terms is not None:
            zero = torch.zeros((), device=dev)
            gu = g_unit if g_unit is not None else zero
            gt = g_terms if g_terms is not None else torch.zeros(3, device=dev)
            a0, a1, a2 = gu + gt[0], gu + gt[1], gu + gt[2]
            g1 = (a0 / (b * m)).expand(b, m).clone()
            g1.scatter_add_(1, dist1.argmax(dim=1, keepdim=True), (a1 / b).expand(b, 1).contiguous())
            g2 = (a2 / (b * n)).expand(b, n).contiguous()
            gs_c, gr_c = nn_distance_backward(samp, ref, g1, idx1, g2, idx2)
            g_samp = gs_c if g_samp is None else g_samp + gs_c
            if need[0]:
                g_ref = gr_c if g_ref is None else g_ref + gr_c
        return (g_ref if need[0] else None), g_samp, g_t, None, None, None


# ----------------------------------------------------------------------------------------------------- progressive loss
def progressive_loss_forward(ref, samp, sizes, weights, unfused=False):
    """One launch: dist1/idx1 (B,M), dist2/idx2 (B,P,N) for the P prefixes `sizes` of the ordered samples, terms (3P+1,)."""
    ref, samp = _req(ref, "ref_pc"), _req(samp, "samp_pc")
    b, n, _ = ref.shape
    m = samp.shape[1]
    npf = len(sizes)
    dev = ref.device
    csz = (ctypes.c_int * npf)(*[int(v) for v in sizes])
    cw = (ctypes.c_float * npf)(*[float(v) for v in weights])
    with torch.cuda.device(dev):
        dist1 = torch.empty(b, m, device=dev); idx1 = torch.empty(b, m, device=dev, dtype=torch.int32)
        dist2 = torch.empty(b, npf, n, device=dev); idx2 = torch.empty(b, npf, n, device=dev, dtype=torch.int32)
        terms = torch.empty(3 * npf + 1, device=dev)
        wsb = int(lib().snb200_progressive_loss_workspace_bytes(b, n, m, npf))
        ws = torch.empty(max(wsb, 4), device=dev, dtype=torch.uint8)
        check(lib().snb200_progressive_loss_forward(b, n, m, _p(ref), _p(samp), npf, csz, cw, _p(dist1), _p(idx1), _p(dist2), _p(idx2), _p(terms), _p(ws), wsb,
                                                    _p(_ticket(dev)), DIST_UNFUSED if unfused else DIST_FMA, _stream()), "progressive_loss_forward")
    return dist1, idx1, dist2, idx2, terms


class ProgressiveLossFunction(torch.autograd.Function):
    """sum over prefixes s of [mean(c12[:s]) + mean_b(max c12[:s]) + w_s mean(c21^(s))]  (train_samplenet_progressive.py:196-220) in one
    forward launch; backward = one deterministic Chamfer-backward launch over the concatenated prefix index sets."""

    @staticmethod
    def forward(ctx, samp, ref, sizes, weights):
        samp = samp.contiguous(); ref = ref.contiguous()
        dist1, idx1, dist2, idx2, terms = progressive_loss_forward(ref, samp, sizes, weights)
        ctx.save_for_backward(samp, ref, dist1, idx1, idx2)
        ctx.sizes, ctx.weights = [int(v) for v in sizes], [float(v) for v in weights]
        return terms[3 * len(sizes)].clone(), terms[:3 * len(sizes)].view(len(sizes), 3)

    @staticmethod
    def backward(ctx, g, g_terms):
        samp, ref, dist1, idx1, idx2 = ctx.saved_tensors
        b, m = dist1.shape
        npf, n = idx2.shape[1], idx2.shape[2]
        dev = samp.device
        sizes = torch.tensor(ctx.sizes, device=dev)
        w = torch.tensor(ctx.weights, device=dev)
        gt = g_terms if g_terms is not None else torch.zeros(npf, 3, device=dev)
        gg = g if g is not None else torch.zeros((), device=dev)
        a0 = gg + gt[:, 0]; a1 = gg + gt[:, 1]; a2 = gg * w + gt[:, 2]           # d total / d term, per prefix
        # mean(c12[:s]) : every j < s gets 1/(b s);  as a function of j: sum over prefixes with s > j
        j = torch.arange(m, device=dev)
        cover = (sizes[None, :] > j[:, None]).to(dist1.dtype)                     # (m, P)
        g1 = (cover * (a0 / (b * sizes.to(dist1.dtype)))[None, :]).sum(1)[None, :].expand(b, m).clone()
        # mean_b max(c12[:s]) : the running arg-max at position s-1
        am = torch.cummax(dist1, dim=1).indices[:, sizes - 1]                     # (b, P)
        g1.scatter_add_(1, am, (a1 / b)[None, :].expand(b, npf).contiguous())
        g2 = (a2 / (b * n))[None, :, None].expand(b, npf, n).reshape(b, npf * n).contiguous()
        ref_rep = ref[:, None].expand(b, npf, n, 3).reshape(b, npf * n, 3).contiguous()
        gs, gr = nn_distance_backward(samp, ref_rep, g1.contiguous(), idx1, g2, idx2.reshape(b, npf * n).contiguous())
        return gs, gr.view(b, npf, n, 3).sum(1), None, None


def group_point(points, idx, layout="bnc"):
    lay = _layout(layout)
    points, idx = _req(points, "points"), _req(idx, "idx", torch.int32)
    b = points.shape[0]
    if lay == BNC:
        n, c = points.shape[1], points.shape[2]
    else:
        c, n = points.shape[1], points.shape[2]
    _, m, ns = idx.shape
    with torch.cuda.device(points.device):
        out = torch.empty((b, m, ns, c) if lay == BNC else (b, c, m, ns), device=points.device)
        check(lib().snb200_group_point(b, n, c, m, ns, lay, _p(points), _p(idx), _p(out), _stream()), "group_point")
    return out


def group_point_grad(points_shape, idx, grad_out, layout="bnc"):
    lay = _layout(layout)
    idx, grad_out = _req(idx, "idx", torch.int32), _req(grad_out, "grad_out")
    b = points_shape[0]
    if lay == BNC:
        n, c = points_shape[1], points_shape[2]
    else:
        c, n = points_shape[1], points_shape[2]
    _, m, ns = idx.shape
    with torch.cuda.device(idx.device):
        gp = torch.empty(tuple(points_shape), device=idx.device)
        check(lib().snb200_group_point_grad(b, n, c, m, ns, lay, _p(grad_out), _p(idx), _p(gp), _stream()), "group_point_grad")
    return gp


class GroupPointFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, idx, layout):
        ctx.save_for_backward(idx)
        ctx.shape = tuple(points.shape)
        ctx.layout = layout
        return group_point(points, idx, layout)

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        return group_point_grad(ctx.shape, idx, g, ctx.layout), None, None


# ----------------------------------------------------------------------------------------------------- generator
def make_layers(specs):
    """specs: list of dicts(weight, bias, bn=(weight,bias,running_mean,running_var,eps,momentum[,num_batches_tracked]) or None, relu=bool)."""
    arr = (Layer * len(specs))()
    keep = []
    for i, s in enumerate(specs):
        w = _req(s["weight"].reshape(s["weight"].shape[0], -1), "weight")
        bias = _req(s["bias"], "bias") if s.get("bias") is not None else torch.zeros(w.shape[0], device=w.device)
        keep += [w, bias]
        arr[i].c_out, arr[i].c_in = w.shape[0], w.shape[1]
        arr[i].weight, arr[i].bias = w.data_ptr(), bias.data_ptr()
        bn = s.get("bn")
        if bn is not None:
            gw, gb, rm, rv, eps, mom = bn[:6]
            nbt = bn[6] if len(bn) > 6 else None
            gw, gb = _req(gw, "bn.weight"), _req(gb, "bn.bias")
            keep += [gw, gb]
            arr[i].bn_weight, arr[i].bn_bias = gw.data_ptr(), gb.data_ptr()
            arr[i].bn_running_mean = None if rm is None else rm.data_ptr()
            arr[i].bn_running_var = None if rv is None else rv.data_ptr()
            arr[i].bn_eps, arr[i].bn_momentum = float(eps), float(0.1 if mom is None else mom)
            if nbt is not None:
                if nbt.dtype != torch.int64 or not nbt.is_cuda:
                    raise TypeError("num_batches_tracked must be an int64 CUDA tensor")
                arr[i].bn_num_batches_tracked = nbt.data_ptr()
            else:
                arr[i].bn_num_batches_tracked = None
        else:
            arr[i].bn_weight = arr[i].bn_bias = arr[i].bn_running_mean = arr[i].bn_running_var = arr[i].bn_num_batches_tracked = None
            arr[i].bn_eps, arr[i].bn_momentum = 0.0, 0.0
        arr[i].relu = int(bool(s.get("relu", False)))
    return arr, keep


class PrimedWorkspaces:
    """Generator workspaces that persist across calls (one per size), zero-initialised once.  With one of these active
    (`with primed_workspaces(pw): ...`) `generator_forward` passes SNB200_GEN_WORKSPACE_PRIMED: the persistent kernel cleans its own
    scratch, so no memset is issued in front of it.  The owner promises the calls that share a buffer are stream-ordered
    (GraphedStep / GraphedTrainStep own one each); plain calls outside such a context allocate and memset per call as before."""

    def __init__(self):
        self.bufs = {}

    def get(self, dev, nbytes):
        key = (dev.index, int(nbytes))
        t = self.bufs.get(key)
        if t is None:
            t = torch.zeros(max(int(nbytes), 256), device=dev, dtype=torch.uint8)
            self.bufs[key] = t
        return t

    def get_named(self, dev, name, shapes):
        """Persistent float buffers (e.g. the activations kept for the backward pass), one list per (device, name, shapes)."""
        key = (dev.index, name, tuple(tuple(s) for s in shapes))
        t = self.bufs.get(key)
        if t is None:
            t = [torch.empty(*s, device=dev) for s in shapes]
            self.bufs[key] = t
        return t


_ACTIVE_PW = threading.local()


class primed_workspaces:
    def __init__(self, pw):
        self.pw = pw

    def __enter__(self):
        self.prev = getattr(_ACTIVE_PW, "pw", None)
        _ACTIVE_PW.pw = self.pw
        return self.pw

    def __exit__(self, *exc):
        _ACTIVE_PW.pw = self.prev
        return False


def generator_forward(x, layout, conv_specs, fc_specs, training, out_transpose_inner=0, exact_fp32=False, _profile_flags=0, per_layer_kernels=False, separate_head=False):
    """x (B,N,3)/(B,3,N) -> (out (B, c_out_last), feat (B, c_conv_last)): conv stack + max-pool + FC head in ONE C-ABI call.
    Default: conv layers on the tensor cores (tcgen05, 3xTF32) + cluster-fused FC head; exact_fp32=True: CUDA-core conv stack."""
    lay = _layout(layout)
    x = _req(x, "x")
    cdim = 2 if lay == BNC else 1
    if x.dim() != 3 or x.shape[cdim] != 3:
        raise RuntimeError("shape of x must be of [Batch x 3 x NumInPoints]")
    b = x.shape[0]
    n = x.shape[1] if lay == BNC else x.shape[2]
    dev = x.device
    conv, keep1 = make_layers(conv_specs)
    fc, keep2 = make_layers(fc_specs)
    with torch.cuda.device(dev):
        wsb = int(lib().snb200_generator_workspace_bytes(b, n, len(conv_specs), conv, len(fc_specs), fc))
        pw = getattr(_ACTIVE_PW, "pw", None)
        primed = 0
        if pw is not None and not _profile_flags:
            ws = pw.get(dev, wsb)
            primed = _lib.GEN_WORKSPACE_PRIMED
        else:
            ws = torch.empty(max(wsb, 4), device=dev, dtype=torch.uint8)
        feat = torch.empty(b, conv[len(conv_specs) - 1].c_out, device=dev)
        out = torch.empty(b, fc[len(fc_specs) - 1].c_out, device=dev)
        check(lib().snb200_generator_forward(b, n, lay, _p(x), len(conv_specs), conv, len(fc_specs), fc, int(bool(training)), _p(out),
                                             int(out_transpose_inner), _p(feat), (_lib.GEN_EXACT_FP32 if exact_fp32 else 0) | (8 if per_layer_kernels else 0) | (16 if separate_head else 0) | int(_profile_flags) | primed, _p(ws), wsb,
                                             _stream()), "generator_forward")
    del keep1, keep2
    return out, feat


def generator_backward_supported(x, layout, conv_specs, fc_specs):
    """True when the CUDA backward (csrc/generator_bwd.cu) covers this shape: the persistent conv-stack envelope, 2 <= B <= 64,
    BatchNorm + ReLU on every conv layer."""
    lay = _layout(layout)
    b = x.shape[0]
    n = x.shape[1] if lay == BNC else x.shape[2]
    conv, keep1 = make_layers(conv_specs)
    fc, keep2 = make_layers(fc_specs)
    return bool(lib().snb200_generator_backward_supported(b, n, len(conv_specs), conv, len(fc_specs), fc))


def generator_train_forward(x, layout, conv_specs, fc_specs, out_transpose_inner=0):
    """Training-mode forward that keeps what the CUDA backward needs.  Returns (out, feat, saved) with saved = (zsave list, workspace)."""
    lay = _layout(layout)
    x = _req(x, "x")
    b = x.shape[0]
    n = x.shape[1] if lay == BNC else x.shape[2]
    dev = x.device
    conv, keep1 = make_layers(conv_specs)
    fc, keep2 = make_layers(fc_specs)
    with torch.cuda.device(dev):
        wsb = int(lib().snb200_generator_workspace_bytes(b, n, len(conv_specs), conv, len(fc_specs), fc))
        pw = getattr(_ACTIVE_PW, "pw", None)
        primed = 0
        if pw is not None:
            ws = pw.get(dev, wsb)
            primed = _lib.GEN_WORKSPACE_PRIMED
            zs = pw.get_named(dev, "zsave", [(b * n, conv[l].c_out) for l in range(len(conv_specs))])
        else:
            ws = torch.empty(max(wsb, 4), device=dev, dtype=torch.uint8)
            zs = [torch.empty(b * n, conv[l].c_out, device=dev) for l in range(len(conv_specs))]
        zp = (ctypes.c_void_p * len(zs))(*[z.data_ptr() for z in zs])
        feat = torch.empty(b, conv[len(conv_specs) - 1].c_out, device=dev)
        out = torch.empty(b, fc[len(fc_specs) - 1].c_out, device=dev)
        check(lib().snb200_generator_train_forward(b, n, lay, _p(x), len(conv_specs), conv, len(fc_specs), fc, _p(out), int(out_transpose_inner), _p(feat),
                                                   zp, primed, _p(ws), wsb, _stream()), "generator_train_forward")
    del keep1, keep2
    return out, feat, (zs, ws)


def generator_backward(x, layout, conv_specs, fc_specs, saved, grad_out, out_transpose_inner=0, dest=None):
    """Gradients of every generator parameter (hand-written CUDA; csrc/generator_bwd.cu).  Returns a list, in layer order (conv then fc), of
    dicts {weight, bias, bn_weight, bn_bias} (bn_* None for layers without BatchNorm).  dest: optional list of such dicts of preallocated
    contiguous tensors the kernels write into (e.g. the parameters' .grad views of a flat bucket) instead of fresh tensors."""
    lay = _layout(layout)
    x = _req(x, "x"); grad_out = _req(grad_out, "grad_out")
    b = x.shape[0]
    n = x.shape[1] if lay == BNC else x.shape[2]
    dev = x.device
    zs, fwd_ws = saved
    conv, keep1 = make_layers(conv_specs)
    fc, keep2 = make_layers(fc_specs)
    grads = []

    def grad_structs(specs):
        arr = (LayerGrad * len(specs))()
        for i, s in enumerate(specs):
            w = s["weight"]
            if dest is not None:
                g = dest[len(grads)]
            else:
                g = {"weight": torch.empty_like(w), "bias": torch.empty(w.shape[0], device=dev) if s.get("bias") is not None else None,
                     "bn_weight": None, "bn_bias": None}
                if s.get("bn") is not None:
                    g["bn_weight"] = torch.empty(w.shape[0], device=dev); g["bn_bias"] = torch.empty(w.shape[0], device=dev)
            arr[i].weight, arr[i].bias = _p(g["weight"]), _p(g["bias"])
            arr[i].bn_weight, arr[i].bn_bias = _p(g["bn_weight"]), _p(g["bn_bias"])
            grads.append(g)
        return arr

    with torch.cuda.device(dev):
        gconv = grad_structs(conv_specs)
        gfc = grad_structs(fc_specs)
        wsb = int(lib().snb200_generator_backward_workspace_bytes(b, n, len(conv_specs), conv, len(fc_specs), fc))
        ws = torch.empty(max(wsb, 4), device=dev, dtype=torch.uint8)
        zp = (ctypes.c_void_p * len(zs))(*[z.data_ptr() for z in zs])
        check(lib().snb200_generator_backward(b, n, lay, _p(x), len(conv_specs), conv, len(fc_specs), fc, zp, _p(fwd_ws), _p(grad_out), int(out_transpose_inner),
                                              gconv, gfc, _p(ws), wsb, _stream()), "generator_backward")
    global _LAST_BWD_WS
    _LAST_BWD_WS = ws          # (bring-up: tools/diag_bwd_layers.py inspects the intermediate gradients)
    del keep1, keep2
    return grads


_LAST_BWD_WS = None


def generator_forward_unfused(x, layout, conv_specs, fc_specs, training, out_transpose_inner=0):
    """Same result through the two stand-alone entry points snb200_encoder_forward + snb200_fc_head_forward
    (exact-fp32 CUDA-core kernels, one launch per layer)."""
    lay = _layout(layout)
    x = _req(x, "x")
    b = x.shape[0]
    n = x.shape[1] if lay == BNC else x.shape[2]
    dev = x.device
    conv, keep1 = make_layers(conv_specs)
    fc, keep2 = make_layers(fc_specs)
    with torch.cuda.device(dev):
        ws1b = int(lib().snb200_encoder_workspace_bytes(b, n, len(conv_specs), conv))
        ws2b = int(lib().snb200_fc_head_workspace_bytes(b, len(fc_specs), fc))
        ws1 = torch.empty(max(ws1b, 4), device=dev, dtype=torch.uint8)
        ws2 = torch.empty(max(ws2b, 4), device=dev, dtype=torch.uint8)
        feat = torch.empty(b, conv[len(conv_specs) - 1].c_out, device=dev)
        out = torch.empty(b, fc[len(fc_specs) - 1].c_out, device=dev)
        check(lib().snb200_encoder_forward(b, n, lay, _p(x), len(conv_specs), conv, int(bool(training)), _p(feat), _p(ws1), ws1b, _stream()),
              "encoder_forward")
        check(lib().snb200_fc_head_forward(b, _p(feat), len(fc_specs), fc, int(bool(training)), _p(out), int(out_transpose_inner), _p(ws2), ws2b, _stream()),
              "fc_head_forward")
    del keep1, keep2
    return out, feat


# ----------------------------------------------------------------------------------------------------- EMD
def approx_match(xyz1, xyz2, exact=None):
    """exact=True (or SNB200_EMD_EXACT_EXP=1 in the environment): the parity kernel -- exact exponential, index-order float sums, the
    reference's level order; bit-identical to the CPU oracle.  Default: the fast kernel (ex2.approx, blocked sums)."""
    if exact is None:
        exact = os.environ.get("SNB200_EMD_EXACT_EXP", "0") == "1"
    xyz1, xyz2 = _req(xyz1, "xyz1"), _req(xyz2, "xyz2")
    if xyz1.dim() != 3 or xyz2.dim() != 3 or xyz1.shape[2] != 3 or xyz2.shape[2] != 3 or xyz1.shape[0] != xyz2.shape[0]:
        raise ValueError("ApproxMatch expects (batch_size,num_points,3) xyz1 and xyz2 with equal batch sizes")
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    dev = xyz1.device
    with torch.cuda.device(dev):
        match = torch.empty(b, m, n, device=dev)
        wsb = int(lib().snb200_approxmatch_workspace_bytes(b, n, m))
        ws = torch.empty(max(wsb, 4), device=dev, dtype=torch.uint8)
        check(lib().snb200_approxmatch_mode(b, n, m, _p(xyz1), _p(xyz2), _p(match), _lib.EMD_EXACT if exact else 0, _p(ws), wsb, _stream()), "approxmatch")
    return match


def match_cost_forward(xyz1, xyz2, match):
    xyz1, xyz2, match = _req(xyz1, "xyz1"), _req(xyz2, "xyz2"), _req(match, "match")
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    if tuple(match.shape) != (b, m, n):
        raise ValueError("MatchCost expects (batch_size,#query,#dataset) match shape, got %s" % (tuple(match.shape),))
    dev = xyz1.device
    with torch.cuda.device(dev):
        cost = torch.empty(b, device=dev)
        wsb = int(lib().snb200_matchcost_workspace_bytes(b))
        ws = torch.empty(max(wsb, 4), device=dev, dtype=torch.uint8)
        check(lib().snb200_matchcost(b, n, m, _p(xyz1), _p(xyz2), _p(match), _p(cost), _p(ws), wsb, _stream()), "matchcost")
    return cost


def match_cost_grad(xyz1, xyz2, match):
    xyz1, xyz2, match = _req(xyz1, "xyz1"), _req(xyz2, "xyz2"), _req(match, "match")
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    with torch.cuda.device(xyz1.device):
        g1 = torch.empty_like(xyz1); g2 = torch.empty_like(xyz2)
        check(lib().snb200_matchcostgrad(b, n, m, _p(xyz1), _p(xyz2), _p(match), _p(g1), _p(g2), _stream()), "matchcostgrad")
    return g1, g2


class MatchCostFunction(torch.autograd.Function):
    """tf_approxmatch.py:35-64: cost (B,), gradients to xyz1 and xyz2 only, scaled by grad_cost[b]."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, match):
        ctx.save_for_backward(xyz1.contiguous(), xyz2.contiguous(), match.contiguous())
        return match_cost_forward(xyz1, xyz2, match)

    @staticmethod
    def backward(ctx, g):
        xyz1, xyz2, match = ctx.saved_tensors
        g1, g2 = match_cost_grad(xyz1, xyz2, match)
        return g1 * g.view(-1, 1, 1), g2 * g.view(-1, 1, 1), None


# ----------------------------------------------------------------------------------------------------- inference matching
def nn_matching(full_pc, nn_idx, k, complete_fps=True, return_idx=False):
    """GPU twin of sputils.nn_matching: full_pc (B,N,3), nn_idx (B,T) int32 -> (B,k,3)."""
    full_pc, nn_idx = _req(full_pc, "full_pc"), _req(nn_idx, "idx", torch.int32)
    b, n, _ = full_pc.shape
    t = nn_idx.shape[1]
    with torch.cuda.device(full_pc.device):
        out = torch.empty(b, k, 3, device=full_pc.device)
        oi = torch.empty(b, k, device=full_pc.device, dtype=torch.int32) if return_idx else None
        check(lib().snb200_nn_matching(b, n, t, int(k), _p(full_pc), _p(nn_idx), int(bool(complete_fps)), _p(out), _p(oi), _stream()),
              "nn_matching")
    return (out, oi) if return_idx else out


# ----------------------------------------------------------------------------------------------------- bring-up hook
def debug_tc_gemm(A, W, bias, desc_hi=0, k_adv16=0, swizzle=0):
    """D = A @ W.T + bias through the tcgen05 layer kernel (3xTF32).  A (rows, c_in), W (c_out, c_in), bias (c_out)."""
    A, W, bias = _req(A, "A"), _req(W, "W"), _req(bias, "bias")
    rows, c_in = A.shape
    c_out = W.shape[0]
    with torch.cuda.device(A.device):
        D = torch.empty(rows, c_out, device=A.device)
        check(lib().snb200_debug_tc_gemm(rows, c_in, c_out, _p(A), _p(W), _p(bias), _p(D), int(desc_hi), int(k_adv16), int(swizzle), _stream()),
              "debug_tc_gemm")
    return D
