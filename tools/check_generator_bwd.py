"""Bring-up check of the CUDA generator backward: gradients of every parameter vs the torch recompute path (autograd through stock ops,
TF32 off) on several shapes, and the time of backward alone and of a whole training step (CUDA events, warm)."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import samplenet_b200 as sb

torch.manual_seed(0)
ok = True
for (b, n, m, layout) in [(32, 1024, 64, "bnc"), (4, 1024, 64, "bnc"), (7, 1000, 32, "bnc"), (16, 333, 64, "bcn"), (32, 1024, 64, "bcn")]:
    net = sb.SampleNet(m, 128, group_size=8, input_shape=layout, output_shape=layout).cuda().train()
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    x = torch.rand(b, n, 3, device="cuda") - 0.5
    if layout == "bcn":
        x = x.permute(0, 2, 1).contiguous()
    rw = torch.randn(b, m, 3, device="cuda") if layout == "bnc" else torch.randn(b, 3, m, device="cuda")
    res = {}
    for mode in ("cuda", "torch"):
        net.generator_backward = mode
        net.zero_grad()
        simp, proj = net(x)
        ((simp * rw).sum() + 0.3 * (proj * rw).sum()).backward()
        res[mode] = {k: p.grad.detach().clone() for k, p in net.named_parameters() if p.grad is not None}
    worst = 0.0
    bad = []
    for k in res["torch"]:
        a, r = res["cuda"][k].double(), res["torch"][k].double()
        scale = r.abs().max().item() + 1e-12
        err = (a - r).abs().max().item()
        # biases in front of a training-mode BatchNorm: the true gradient is 0, both sides hold rounding noise
        tol = 5e-4 * scale + 2e-5
        if ("conv" in k or k in ("fc1.bias", "fc2.bias", "fc3.bias")) and k.endswith("bias"):
            tol = 1e-3
        if err > tol:
            bad.append((k, err, scale))
        worst = max(worst, err / scale if scale > 1e-3 else 0.0)
    good = not bad
    ok = ok and good
    print("b=%d n=%d m=%d %s: worst rel err %.2e  %s %s" % (b, n, m, layout, worst, "ok" if good else "MISMATCH", bad[:6]), flush=True)
print("ALL OK" if ok else "FAILED")

net = sb.SampleNet(64, 128, group_size=8, input_shape="bnc", output_shape="bnc").cuda().train()
x = torch.rand(32, 1024, 3, device="cuda") - 0.5
for mode in ("cuda", "torch"):
    net.generator_backward = mode
    def step():
        net.zero_grad(set_to_none=False) if any(p.grad is not None for p in net.parameters()) else None
        simp, proj = net(x)
        loss = 0.01 * net.get_simplification_loss(x, simp, 64) + 0.01 * net.get_projection_loss() + proj.sum() * 0.0
        loss.backward()
    for _ in range(5):
        step()
    torch.cuda.synchronize()
    a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20):
        step()
    bb.record(); bb.synchronize()
    print("eager training step (fwd + losses + bwd), generator_backward=%s: %.1f us" % (mode, a.elapsed_time(bb) * 1e3 / 20))
try:
    net.generator_backward = "cuda"
    gs = sb.GraphedTrainStep(net, 32, 1024)
    for _ in range(5):
        gs(x)
    torch.cuda.synchronize()
    a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(50):
        gs(x)
    bb.record(); bb.synchronize()
    print("GraphedTrainStep (fwd + bwd + Adam, one graph): %.1f us/step, %d library-side launches counted" % (a.elapsed_time(bb) * 1e3 / 50, gs.launches_per_step))
except Exception as e:
    print("GraphedTrainStep failed:", repr(e)[:300])
