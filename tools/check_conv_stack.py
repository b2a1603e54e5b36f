"""Bring-up check of the persistent conv-stack kernel: fused generator vs the per-layer tcgen05 kernels and the exact-fp32 CUDA-core
path on several shapes (train + eval), then the clock64 timeline of the headline shape."""
import os, sys, ctypes
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import samplenet_b200 as sb

torch.manual_seed(0)
ok = True
QUICK = os.environ.get("SNB200_CS_DEBUG", "0") != "0" or os.environ.get("CS_QUICK", "0") != "0"
for (b, n, m, train) in ([] if QUICK else [(32, 1024, 64, True), (2, 1024, 64, True), (7, 1000, 64, True), (37, 1024, 64, True), (3, 77, 32, True), (70, 500, 64, True),
                         (32, 1024, 64, False), (5, 333, 32, False), (32, 1024, 32, True), (2, 2048, 64, True), (64, 512, 64, False),
                         # more than one 256-point slice per SM: the multi-slice instantiation (2, 3 and 4 slices per CTA, ragged last slices)
                         (64, 1024, 64, True), (128, 1024, 64, True), (50, 2048, 64, True), (200, 777, 32, True), (128, 1024, 64, False), (41, 1999, 64, True)]):
    net = sb.SampleNet(m, 128, group_size=8, input_shape="bnc", output_shape="bnc").cuda()
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    net.train(train)
    if not train:
        for bn in [net.bn1, net.bn2, net.bn3, net.bn4, net.bn5, net.bn_fc1, net.bn_fc2, net.bn_fc3]:
            bn.running_mean.normal_(0, 0.1); bn.running_var.uniform_(0.5, 1.5)
    x = (torch.rand(b, n, 3, device="cuda") - 0.5)
    conv, fc = net._layer_specs()
    with torch.no_grad():
        o1, f1 = sb.ops.generator_forward(x, "bnc", conv, fc, train, m)
        o2, f2 = sb.ops.generator_forward(x, "bnc", conv, fc, train, m, per_layer_kernels=True)
        o3, f3 = sb.ops.generator_forward(x, "bnc", conv, fc, train, m, exact_fp32=True)
        xb = x.permute(0, 2, 1).contiguous()
        o4, f4 = sb.ops.generator_forward(xb, "bcn", conv, fc, train, 0)
    torch.cuda.synchronize()
    e12f, e13f = (f1 - f2).abs().max().item(), (f1 - f3).abs().max().item()
    e12, e13 = (o1 - o2).abs().max().item(), (o1 - o3).abs().max().item()
    e14f = (f1 - f4).abs().max().item()
    otol = 2e-2 if b <= 4 else 2e-3    # (BatchNorm over <= 4 rows in the FC head amplifies rounding: judged on the pooled feature)
    good = e12f < 2e-4 and e13f < 2e-4 and e12 < otol and e13 < otol and e14f < 2e-4 and torch.isfinite(o1).all().item()
    ok = ok and good
    print("b=%d n=%d m=%d train=%d  feat: vs per-layer %.2e vs fp32 %.2e bcn %.2e | out: vs per-layer %.2e vs fp32 %.2e  %s" %
          (b, n, m, train, e12f, e13f, e14f, e12, e13, "ok" if good else "MISMATCH"), flush=True)
print("ALL OK" if ok else "FAILED")

net = sb.SampleNet(64, 128, group_size=8, input_shape="bnc", output_shape="bnc").cuda().train()
x = torch.rand(int(os.environ.get("CS_TL_B", "32")), 1024, 3, device="cuda") - 0.5   # (CS_TL_B=28: 128 CTAs, none partially filled)
conv, fc = net._layer_specs()
with torch.no_grad():
    for _ in range(5):
        sb.ops.generator_forward(x, "bnc", conv, fc, True, 64)
    torch.cuda.synchronize()
    buf = (ctypes.c_longlong * 64)()
    sb._lib.lib().snb200_debug_conv_stack_timestamps(ctypes.addressof(buf))
    ts = list(buf); t0 = ts[0]
    names = {0: "start", 1: "setup done", 2: "moments + barrier done"}
    for l in range(4):
        for i, nm in enumerate(["layer start", "scale/shift", "operand stored/issued", "acc ready", "D loaded + stats", "atomics/pool out", "grid barrier done", "(ring slot free: operand write starts; last layer: barrier arrive issued)"]):
            names[3 + l * 8 + i] = "L%d %s" % (l + 2, nm)
    names[35] = "conv stack left (CTA barrier)"; names[36] = "head: start"; names[37] = "head: pooled"
    for l in range(4):
        for i, nm in enumerate(["start", "input staged", "partials done", "combined", "BN scale/shift", "stored"]):
            names[39 + l * 6 + i] = "FC%d %s" % (l + 1, nm)
    prev = t0
    for i in sorted(names):
        print("%-28s %8d cycles  (+%d)" % (names[i], ts[i] - t0, ts[i] - prev)); prev = ts[i]
    # timing
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        sb.ops.generator_forward(x, "bnc", conv, fc, True, 64)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            for _ in range(20):
                sb.ops.generator_forward(x, "bnc", conv, fc, True, 64)
    g.replay(); torch.cuda.synchronize()
    a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20):
        g.replay()
    bb.record(); bb.synchronize()
    print("generator (conv stack): %.2f us per launch (in-graph, warm)" % (a.elapsed_time(bb) * 1e3 / 400))
