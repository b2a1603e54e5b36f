"""Which side is closer to the truth?  Gradients of every generator parameter from (a) the CUDA backward, (b) the torch fp32 recompute,
against (c) a float64 evaluation of the same layer stack (torch autograd in double)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import samplenet_b200 as sb
torch.manual_seed(0)
for (b, n, m, layout) in [(64, 512, 64, "bnc"), (48, 512, 64, "bnc"), (64, 256, 64, "bnc")]:
    net = sb.SampleNet(m, 128, group_size=8, input_shape=layout, output_shape=layout).cuda().train()
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    x = torch.rand(b, n, 3, device="cuda") - 0.5
    if layout == "bcn":
        x = x.permute(0, 2, 1).contiguous()
    rw = torch.randn(b, 3 * m, device="cuda")
    names = [k for k, _ in net._generator_named_parameters()]
    params = [p for _, p in net._generator_named_parameters()]
    out_inner = m if layout == "bnc" else 0
    res = {}
    for mode in ("cuda", "cuda2", "torch"):
        net.generator_backward = "torch" if mode == "torch" else "cuda"
        net.zero_grad()
        y = net._generate(x, layout, out_inner)
        (y * rw).sum().backward()
        res[mode] = [p.grad.detach().clone().double() for p in params]
    # float64 truth
    ps64 = {nm: p.detach().double().requires_grad_(True) for nm, p in zip(names, params)}
    y64 = net._torch_generator(x.double(), layout, True, ps64)
    if out_inner:
        y64 = y64.view(b, -1, out_inner).permute(0, 2, 1).reshape(b, -1)
    g64 = torch.autograd.grad(y64, list(ps64.values()), rw.double())
    print("config", b, n, m, layout)
    pnames = [k for k, _ in net.named_parameters()]
    for i, nm in enumerate(names):
        t = g64[i]
        sc = t.abs().max().item() + 1e-30
        ec = (res["cuda"][i].reshape(t.shape) - t).abs().max().item()
        ec2 = (res["cuda2"][i].reshape(t.shape) - res["cuda"][i].reshape(t.shape)).abs().max().item()
        et = (res["torch"][i].reshape(t.shape) - t).abs().max().item()
        flag = "  <<<" if ec > 3 * et + 1e-6 * sc else ""
        print("  %-10s scale %.3e  |cuda-f64| %.3e  |torch32-f64| %.3e  |cuda run2 - run1| %.1e%s" % (nm, sc, ec, et, ec2, flag))
