"""Layer-by-layer check of the CUDA generator backward: dy_{l-1} (gradient wrt the BN output of layer l-1, ReLU mask applied) and its
BatchNorm sums after each conv kernel, against float64 autograd intermediates of the same stack (routing forced to the CUDA arg-max)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import samplenet_b200 as sb
b, n, m, layout = [int(v) if v.isdigit() else v for v in (sys.argv[1:5] if len(sys.argv) >= 5 else ["64", "512", "64", "bnc"])]
torch.manual_seed(b + n)
net = sb.SampleNet(m, 128, group_size=8, input_shape=layout, output_shape=layout).cuda().train()
with torch.no_grad():
    for p in net.parameters():
        if p.dim() == 1:
            p.add_(0.1 * torch.randn_like(p))
x = torch.rand(b, n, 3, device="cuda") - 0.5
conv_specs, fc_specs = net._layer_specs()
rw = torch.randn(b, 3 * m, device="cuda")
names = [k for k, _ in net._generator_named_parameters()]
params = [p for _, p in net._generator_named_parameters()]
with torch.no_grad():
    out, feat, saved = sb.ops.generator_train_forward(x, layout, conv_specs, fc_specs, m)
zs = saved[0]
sgn = torch.where(net.bn5.weight >= 0, 1.0, -1.0)
route = (zs[4].view(b, n, -1) * sgn).argmax(dim=1)
# float64 graph with retained intermediates
ps64 = {nm: p.detach().double().requires_grad_(True) for nm, p in zip(names, params)}
h = x.double().reshape(-1, 3)
ys = []
zfc = []
layers = net._convs() + net._fcs()
for i, (lin, bn) in enumerate(layers):
    if i == 5:
        h = torch.gather(h.view(b, n, -1), 1, route[:, None, :]).squeeze(1)
    h = torch.nn.functional.linear(h, ps64["l%d.w" % i].reshape(ps64["l%d.w" % i].shape[0], -1), ps64["l%d.b" % i])
    if i >= 5:
        h.retain_grad(); zfc.append(h)
    if bn is not None:
        h = torch.nn.functional.batch_norm(h, None, None, ps64["l%d.g" % i], ps64["l%d.beta" % i], True, 0.0, bn.eps)
        if i < 5:
            h.retain_grad(); ys.append(h)       # y_i = BN output (pre-ReLU): its grad is dy_i
        h = torch.relu(h)
    if i == 4:
        a5 = h; a5.retain_grad()
hh = h.view(b, -1, m).permute(0, 2, 1).reshape(b, -1)
(hh * rw.double()).sum().backward()
print("forward out max diff", (out.double() - hh.detach()).abs().max().item())
for i in range(5):
    zref = None
P = b * n
maxc = 128
dyb = (P * maxc * 4 + 255) // 256 * 256
for stop in (4, 3, 2, 1):
    os.environ["SNB200_BWD_STOP"] = str(stop)
    sb.ops.generator_backward(x, layout, conv_specs, fc_specs, saved, rw, m)
    torch.cuda.synchronize()
    ws = sb.ops._LAST_BWD_WS
    lm1 = stop - 1
    c = ys[lm1].shape[1]
    off = ((lm1) & 1) * dyb
    dy = ws[off:off + P * c * 4].view(torch.float32).view(P, c).double()
    ref = ys[lm1].grad
    err = (dy - ref).abs().max().item()
    print("after conv layer %d kernel: dy_%d max err %.3e (scale %.3e); col-sum err %.3e (scale %.3e); sum(dy*zhat) n/a" %
          (stop, lm1, err, ref.abs().max().item(), (dy.sum(0) - ref.sum(0)).abs().max().item(), ref.sum(0).abs().max().item()))
    bad = (dy - ref).abs().max(dim=1)[0]
    top = torch.topk(bad, 5)
    print("   worst rows", top.indices.tolist(), ["%.2e" % v for v in top.values.tolist()])
del os.environ["SNB200_BWD_STOP"]
s12b = sum(((2 * c * 8 + 255) // 256) * 256 for c in (64, 64, 64, 128, 128))
o = 2 * dyb + s12b
pstar = ws[o:o + b * 128 * 4].view(torch.int32).view(b, 128); o += (b * 128 * 4 + 255) // 256 * 256
gval = ws[o:o + b * 128 * 4].view(torch.float32).view(b, 128)
o += (b * 128 * 4 + 255) // 256 * 256
for li, cw in enumerate((256, 256, 256, 3 * m)):
    dz = ws[o:o + b * cw * 4].view(torch.float32).view(b, cw).double(); o += (b * cw * 4 + 255) // 256 * 256
    ref = zfc[li].grad
    if li == 3:
        ref = ref      # fc4 output layout: our grad_out is in the permuted layout; dz stored per channel cw (unpermuted)
    e = (dz - ref).abs().max(dim=1)[0]
    print("fc%d dz max err %.3e (scale %.3e) worst rows %s" % (li + 1, e.max().item(), ref.abs().max().item(), torch.topk(e, 3).indices.tolist()))
print("pstar == route:", bool(((pstar.long() - torch.arange(b, device="cuda")[:, None] * n) == route).all()))
ga5 = a5.grad.view(b, n, 128)                      # grad wrt relu(y5): nonzero only at the routed points
gref = torch.gather(ga5, 1, route[:, None, :]).squeeze(1) * (torch.gather(ys[4].detach().view(b, n, 128), 1, route[:, None, :]).squeeze(1) > 0)
eg = (gval.double() - gref).abs().max(dim=1)[0]
print("gval max err per cloud (top 5):", torch.topk(eg, 5).indices.tolist(), ["%.2e" % v for v in torch.topk(eg, 5).values.tolist()], "scale %.2e" % gref.abs().max().item())
