#!/usr/bin/env python
"""bench.py -- the headline benchmark: point-clouds/sec, SampleNet forward (train mode: generator -> soft projection)
+ Chamfer simplification loss at B=32 per GPU, N=1024 -> 64, k=8 (BASELINE.json metric; registration flavour).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Prints ONE JSON line from rank 0 (see the repo task contract).  Key points:
  * a step = one pass of the hot path over one batch of synthetic clouds, through the public API
    (samplenet_b200.GraphedStep: net(x) + net.get_simplification_loss captured into one CUDA graph);
  * `value`: inputs resident in HBM (a rotating pool of batches larger than the 126 MB L2, so every step reads cold inputs);
  * `e2e`: the same step fed from PINNED HOST memory, host->device copy and device->host read of the loss inside the
    timed region, synchronised every step (the reference trainer calls loss.item() every step, main.py:354);
  * multi-GPU: batch-sharded replicas (weak scaling, 32 clouds per GPU), no data-path collective in forward + loss;
    timing = max over ranks of CUDA-event time;
  * `roofline`: the dominant kernel timed live with CUDA events; `cpu_baseline`: the same step on the host cores
    (torch CPU layer stack + C oracle kNN/projection + the reference's own CPU Chamfer from oracle/_ref);
  * `--impl reference`: that CPU path as the measured arm (all host threads);
  * `--dump-outputs DIR`: after the timed steps, rank 0 writes what the last step of the `value` leg returned (simp, proj, loss) as
    DIR/<name>.npy in float32.  Inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

if "reference" in sys.argv[1:]:
    # CPU arm: the step alternates between torch's OpenMP pool (layer stack) and a cloud-parallel worker pool (kNN / Chamfer); idle OpenMP
    # threads must sleep, not spin, or they steal the cores from the workers (2x on 8 cores).  torchrun pins OMP_NUM_THREADS=1: undo that.
    os.environ["OMP_WAIT_POLICY"] = "PASSIVE"
    os.environ["KMP_BLOCKTIME"] = "0"
    os.environ["GOMP_SPINCOUNT"] = "0"
    os.environ.pop("OMP_NUM_THREADS", None)
    os.environ.pop("MKL_NUM_THREADS", None)

import numpy as np  # noqa: E402
import torch  # noqa: E402

B, N, M, K_NN = 32, 1024, 64, 8
B_SAT = 2048
B_SAT_GEN = 128
BOTTLENECK = 128
L2_BYTES = 126 * 1024 * 1024
METRIC = "point-clouds/sec SampleNet fwd+Chamfer (B=32, N=1024->64)"
WORKLOAD = "registration SampleNet fwd(train)+soft-proj+simplification loss, B=32/GPU, N=1024->64, k=8, fp32"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]),
                    bf16_tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def synth_batch(seed, b=B, n=N):
    """rand-0.5, then OnUnitCube.method2 per cloud (registration/src/pctransforms.py:162-166)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(b, n, 3, generator=g) - 0.5
    s = (x.max(dim=1)[0] - x.min(dim=1)[0]).max(dim=1)[0].view(-1, 1, 1)
    v = x / s
    return (v - v.mean(dim=1, keepdim=True)).contiguous()


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [t.strip() for t in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------- CPU arm
def _numa_cores():
    """The logical CPUs of ONE NUMA node that this process may run on (the largest such group): a 32x3x1024 layer stack spread over
    two sockets with 128 OpenMP threads is ~50x slower than the same code on 8-16 cores of one node (round-1 BENCH: 11.8 clouds/s)."""
    import glob

    aff = set(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else set(range(os.cpu_count() or 1))
    best = sorted(aff)
    groups = []
    for path in sorted(glob.glob("/sys/devices/system/node/node*/cpulist")):
        try:
            cpus = set()
            for part in open(path).read().strip().split(","):
                if "-" in part:
                    a, b = part.split("-")
                    cpus.update(range(int(a), int(b) + 1))
                elif part:
                    cpus.add(int(part))
            g = sorted(cpus & aff)
            if g:
                groups.append(g)
        except Exception:
            pass
    if groups:
        best = max(groups, key=len)
    return best


def cpu_reference_arm(steps, warmup):
    """The reference's CPU path for the step, tuned once: pinned to one NUMA node; torch intra-op threads for the layer stack and the
    number of cloud-parallel workers for kNN / projection / Chamfer are each chosen by a short sweep in the warm-up (the two phases
    are sequential, so the sweep is separable); then `steps` full B=32 steps are timed with the best pair."""
    from oracle import oracle as orc
    from oracle.torch_reference import ReferenceGenerator, cpu_generator, cpu_pairwise

    orc._lib()
    cores = _numa_cores()
    if hasattr(os, "sched_setaffinity"):
        try:
            os.sched_setaffinity(0, cores)      # before the OpenMP / worker pools exist: their threads inherit it
        except OSError:
            pass
    ncore = len(cores)
    torch.manual_seed(0)
    gen = ReferenceGenerator(M, BOTTLENECK).train()
    xs = [synth_batch(100 + i) for i in range(4)]

    def best_of(fn, reps=3):
        fn()
        t = []
        for _ in range(reps):
            t0 = time.perf_counter(); fn(); t.append(time.perf_counter() - t0)
        return min(t)

    cand_t = sorted({t for t in (1, 2, 4, 8, 16, 24, 32, 48, 64) if t <= ncore} | {min(ncore, 64)})
    sweep_t = {}
    for t in cand_t:
        torch.set_num_threads(t)
        sweep_t[t] = best_of(lambda: cpu_generator(gen, xs[0]))
    threads = min(sweep_t, key=sweep_t.get)
    torch.set_num_threads(threads)
    simp0 = cpu_generator(gen, xs[0])
    cand_w = sorted({w for w in (1, 2, 4, 8, 16, 32) if w <= min(ncore, B)} | {min(ncore, B)})
    sweep_w = {w: best_of(lambda: cpu_pairwise(xs[0], simp0, K_NN, 1.0, workers=w)) for w in cand_w}
    workers = min(sweep_w, key=sweep_w.get)

    def step(x):
        simp = cpu_generator(gen, x)
        return cpu_pairwise(x, simp, K_NN, 1.0, workers=workers)

    for i in range(max(warmup, 1)):
        step(xs[i % 4])
    t0 = time.perf_counter()
    for i in range(steps):
        step(xs[i % 4])
    dt = time.perf_counter() - t0
    info = {"numa_node_cpus": ncore, "host_cpus": os.cpu_count(), "torch_threads": threads, "pairwise_workers": workers,
            "sweep_generator_ms": {str(k): round(v * 1e3, 2) for k, v in sweep_t.items()},
            "sweep_pairwise_ms": {str(k): round(v * 1e3, 2) for k, v in sweep_w.items()}}
    return B * steps / dt, dt / steps * 1e3, max(threads, workers), ("port+reference" if orc.have_ref() else "port"), info


CPU_SAMPLE = ("%d full steps of B=32 pinned to one NUMA node: torch CPU layer stack (restated module, %d intra-op threads) + C-oracle kNN/soft-proj "
              "(port) + the reference's own CPU Chamfer compiled from its sources (oracle/_ref), cloud-parallel on %d worker threads; thread "
              "counts picked by a sweep in the warm-up")


def cpu_arm_subprocess(steps, warmup):
    """Run the CPU arm in a fresh interpreter (clean OpenMP pool and affinity, no CUDA context) and return its parsed JSON line."""
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    env["CUDA_VISIBLE_DEVICES"] = ""
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", str(warmup)],
                       env=env, capture_output=True, text=True, timeout=900)
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("CPU arm produced no JSON line: %s" % r.stderr[-400:])


def run_reference(args, rank, world):
    if rank != 0:
        return
    val, ms, cores, kind, info = cpu_reference_arm(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "clouds/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": B, "note": "CPU arm: rank 0 only, one replica, every step a full B=32 batch"},
        "cpu_baseline": {"value": val, "unit": "clouds/s", "cores": cores, "kind": kind,
                         "sample": CPU_SAMPLE % (args.steps, info["torch_threads"], info["pairwise_workers"]), "tuning": info},
        "e2e": {"value": val, "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------- GPU arm
def graph_time_us(fn, reps=20, replays=20):
    """Warm in-graph time of one stage: R back-to-back launches captured in one CUDA graph, CUDA events on the replay stream."""
    if os.environ.get("SNB200_NO_GRAPH") == "1":   # profiler runs: plain launches (numbers then include host launch gaps)
        fn(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record(); b.synchronize()
        return a.elapsed_time(b) * 1e3 / reps
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn(); fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(replays):
        g.replay()
    b.record(); b.synchronize()
    return a.elapsed_time(b) * 1e3 / (reps * replays)


def time_kernels(sb, net, x):
    """Per-stage device time, measured live: each stage alone, launched through the C-ABI wrappers, R launches per graph."""
    conv_specs, fc_specs = net._layer_specs()
    out = {}
    with torch.no_grad():
        sigma = net.project.sigma().detach().reshape(1).contiguous()
        simp = net(x)[0].detach()
        out["generator_us"] = graph_time_us(lambda: sb.ops.generator_forward(x, "bnc", conv_specs, fc_specs, True, M))
        out["conv_stack_us"] = graph_time_us(lambda: sb.ops.generator_forward(x, "bnc", conv_specs, fc_specs, True, M, _profile_flags=2))
        out["fc_head_us"] = graph_time_us(lambda: sb.ops.generator_forward(x, "bnc", conv_specs, fc_specs, True, M, _profile_flags=4))
        out["generator_per_layer_kernels_us"] = graph_time_us(lambda: sb.ops.generator_forward(x, "bnc", conv_specs, fc_specs, True, M, per_layer_kernels=True), reps=10)
        out["generator_exact_fp32_us"] = graph_time_us(lambda: sb.ops.generator_forward(x, "bnc", conv_specs, fc_specs, True, M, exact_fp32=True), reps=5)
        out["knn_softproj_us"] = graph_time_us(lambda: sb.ops.knn_soft_project_forward(x, simp, K_NN, "bnc", sigma, want=("proj", "idx", "weights", "dist")))
        out["chamfer_us"] = graph_time_us(lambda: sb.ops.nn_distance_forward(simp, x))
        out["chamfer_plus_reduce_us"] = graph_time_us(lambda: sb.ops.simplification_loss_forward(simp, x, 1.0))
        out["tail_fused_us"] = graph_time_us(lambda: sb.ops.project_and_loss_forward(x, simp, K_NN, net.project._temperature, 1, 1e-2, 1.0))
        # the same pairwise kernels with the machine filled (B_SAT clouds per launch): what they do when launch latency is amortised
        g = torch.Generator(device="cpu").manual_seed(7)
        xs = (torch.rand(B_SAT, N, 3, generator=g) - 0.5).to(x.device)
        ss = (xs[:, torch.randperm(N, generator=g)[:M]] + 0.02 * torch.randn(B_SAT, M, 3, generator=g).to(x.device)).contiguous()
        out["sat_knn_softproj_us"] = graph_time_us(lambda: sb.ops.knn_soft_project_forward(xs, ss, K_NN, "bnc", sigma, want=("proj", "idx", "weights", "dist")), reps=5)
        out["sat_chamfer_us"] = graph_time_us(lambda: sb.ops.nn_distance_forward(ss, xs), reps=5)
        out["sat_tail_fused_us"] = graph_time_us(lambda: sb.ops.project_and_loss_forward(xs, ss, K_NN, net.project._temperature, 1, 1e-2, 1.0), reps=5)
        # the generator with the machine full: B_SAT_GEN clouds = 7 tiles of 128 points per SM, beyond the persistent kernel's envelope,
        # so the per-layer tcgen05 kernels run (activations through L2/HBM) -- the tensor-pipe counterpart of the saturated pairwise line
        try:
            xg = xs[:B_SAT_GEN].contiguous()
            out["sat_generator_us"] = graph_time_us(lambda: sb.ops.generator_forward(xg, "bnc", conv_specs, fc_specs, True, M), reps=3, replays=10)
        except Exception as exc:   # a reporting extra must never take the bench line down
            out["sat_generator_error"] = str(exc)[:200]
    return out


def run_ours(args, rank, world, local_rank):
    import samplenet_b200 as sb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    sb._lib.lib()
    pk = peaks()
    torch.manual_seed(0)
    net = sb.SampleNet(M, BOTTLENECK, group_size=K_NN, initial_temperature=1.0, input_shape="bnc", output_shape="bnc").to(dev).train()

    # rotating input pool larger than L2, on device (value leg) and in pinned host memory (e2e leg)
    nbytes = B * N * 3 * 4
    pool_n = (int(1.2 * L2_BYTES) + nbytes - 1) // nbytes
    host_pool = torch.empty(pool_n, B, N, 3).pin_memory()
    base = [synth_batch(1000 * rank + i) for i in range(8)]
    for i in range(pool_n):
        host_pool[i].copy_(base[i % 8].roll(i // 8, dims=1))
    dev_pool = host_pool.to(dev)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed_region(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- value leg: inputs already resident in HBM.  The rotating pool (> L2) forces a device-to-device copy of the batch into a capture
    #      buffer; PipelinedHostStep.run_async puts that copy on the copy stream, into the idle one of two graph instances, so it overlaps the
    #      other instance's kernels (same double buffering as the e2e leg, without the host read-back).  The single-graph variant (copy and
    #      replay on one stream) is timed as well and reported as `value_single_graph`.
    step = sb.GraphedStep(net, B, N)
    vpipe = sb.PipelinedHostStep(net, B, N)
    for i in range(args.warmup):
        step(dev_pool[i % pool_n])
        vpipe.run_async(dev_pool[i % pool_n])
    ms_single = timed_region(lambda i: step(dev_pool[(args.warmup + i) % pool_n]), args.steps)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    last = {}

    def value_step(i):
        last["slot"] = vpipe.run_async(dev_pool[(args.warmup + i) % pool_n])

    ms_val = timed_region(value_step, args.steps)
    if args.dump_outputs and rank == 0:   # the slot's static buffers are rewritten only by its own replays, none of which follow
        outputs = {name: getattr(last["slot"], name).detach().float().cpu().numpy() for name in ("simp", "proj", "loss")}
    # ---- e2e leg: pinned host batch -> device, step, loss -> host, every step, through the public streaming API
    #      (PipelinedHostStep: two steps in flight, H2D on a copy stream; every step's loss is read on the host).  The timed region
    #      starts and ends with an EMPTY pipeline: exactly K steps are submitted, launched and finished inside it.
    pipe = sb.PipelinedHostStep(net, B, N)

    def e2e_run(first, count):
        losses = 0.0
        for j in range(count):
            if j >= 2:
                losses += pipe.finish()                                   # loss of step j-2 on the host
            pipe.submit(host_pool[(first + j) % pool_n])                  # batch j crosses PCIe while earlier steps compute
            pipe.launch()                                                 # queue step j behind them
        for _ in range(min(2, count)):
            losses += pipe.finish()
        return losses

    e2e_run(0, max(args.warmup, 3))
    ms_e2e = timed_region(lambda i: e2e_run(args.warmup, args.steps) if i == 0 else None, 1)
    clocks = sampler.stop() if sampler else None

    if rank != 0:
        return
    value = world * B * args.steps / (ms_val * 1e-3)
    e2e = world * B * args.steps / (ms_e2e * 1e-3)

    # ---- roofline of the dominant kernel, timed live (alone, warm, in-graph: R launches per CUDA graph, CUDA events)
    kt = time_kernels(sb, net, dev_pool[0])
    widths = [3, 64, 64, 64, 128, BOTTLENECK]
    conv_flops = sum(2.0 * B * N * widths[i] * widths[i + 1] for i in range(5))
    fcw = [BOTTLENECK, 256, 256, 256, 3 * M]
    head_flops = sum(2.0 * B * fcw[i] * fcw[i + 1] for i in range(4))
    gen_flops = conv_flops + head_flops
    # the dominant kernel of the step is the WHOLE fused launch (conv layers + pool + FC head); its duration is measured live above
    ach_tf = gen_flops / (kt["generator_us"] * 1e-6) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")     # dram bytes of one launch, from the committed ncu --set full capture
    if os.path.exists(tpath):
        try:
            traffic = float(json.load(open(tpath))["conv_stack_kernel"]["dram_bytes_per_launch"])
        except Exception:
            traffic = None
    roofline = {
        "kernel": "conv_stack_kernel (the whole generator in one persistent cooperative launch: conv layers 2-5 as TRANSPOSED GEMMs on tcgen05.mma "
                  "kind::tf32 (3xTF32): weights = A operand in tensor memory, activations = B operand in swizzled shared memory, one channel per thread, "
                  "224 points per CTA on all 148 SMs; max-pool; FC head; BatchNorm batch statistics exchanged as self-counting fixed-point words, one grid barrier left)",
        "bound": "tensor", "achieved": ach_tf, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach_tf / pk["bf16_tflops"],
        "peak_source": pk["source"] + " cuBLAS bf16 burst. `achieved` counts the ALGORITHMIC fp32 flops (2*M*N*K over the 5 conv + 4 FC layers = %.2f GFLOP "
                       "per launch); the kernel issues 3 TF32 MMAs per product (error compensation to fp32 accuracy) and TF32 runs at half the "
                       "bf16 rate, so the ceiling for this number is peak/6; the launch is a dependent chain (one grid-wide BatchNorm statistics exchange per conv layer -- self-counting fixed-point words, one grid barrier left -- and "
                       "4 dependent FC layers on 32 rows): latency-bound, see profiles/ for the tensor-pipe share" % (gen_flops / 1e9),
        "frac_of_3xtf32_ceiling": ach_tf / (pk["bf16_tflops"] / 6.0), "traffic": traffic, "us_per_launch": kt["generator_us"],
        "algorithmic_flops_per_launch": gen_flops,
        "conv_phase_only": {"us": kt["conv_stack_us"], "achieved_tflops": conv_flops / (kt["conv_stack_us"] * 1e-6) / 1e12},
    }
    if "sat_generator_us" in kt:   # same layer stack, B_SAT_GEN clouds per call: the same persistent launch, every CTA walking several 256-point slices per layer
        sat_flops = gen_flops / B * B_SAT_GEN
        sat_tf = sat_flops / (kt["sat_generator_us"] * 1e-6) / 1e12
        roofline["saturated_B"] = {"clouds_per_call": B_SAT_GEN, "us": kt["sat_generator_us"], "clouds_per_s": B_SAT_GEN / (kt["sat_generator_us"] * 1e-6),
                                   "achieved_tflops": sat_tf, "frac": sat_tf / pk["bf16_tflops"], "frac_of_3xtf32_ceiling": sat_tf / (pk["bf16_tflops"] / 6.0),
                                   "path": "conv_stack_kernel<multi-slice>: one cooperative launch, raw layer outputs parked in L2 between layers"}
    pair_bytes_sp = B * (12 * N + 12 * M + 12 * M)
    pair_bytes_cd = B * (12 * (N + M) + 8 * (N + M))
    roofline_pairwise = {
        "knn_softproj": {"bound": "hbm", "achieved": pair_bytes_sp / (kt["knn_softproj_us"] * 1e-6) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                         "frac": pair_bytes_sp / (kt["knn_softproj_us"] * 1e-6) / 1e9 / pk["hbm_gbs"], "us": kt["knn_softproj_us"],
                         "algorithmic_bytes": pair_bytes_sp},
        "chamfer": {"bound": "hbm", "achieved": pair_bytes_cd / (kt["chamfer_us"] * 1e-6) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": pair_bytes_cd / (kt["chamfer_us"] * 1e-6) / 1e9 / pk["hbm_gbs"], "us": kt["chamfer_us"],
                    "algorithmic_bytes": pair_bytes_cd},
        "note": "0.4-0.7 MB per launch: these launches are latency-bound at B=32 (SURVEY.md section 7); fractions reported as required",
    }
    sat_bytes = B_SAT * (12 * N + 12 * M + 12 * M + 8 * (N + M))          # fused single pass, SURVEY.md section 8(d): 22 528 B/cloud
    sat_pairs = 3.0 * B_SAT * N * M                                       # kNN + both Chamfer directions
    roofline_pairwise["saturated_B"] = {
        "clouds_per_launch": B_SAT,
        "tail_fused": {"us": kt["sat_tail_fused_us"], "clouds_per_s": B_SAT / (kt["sat_tail_fused_us"] * 1e-6),
                       "hbm_gbs_algorithmic": sat_bytes / (kt["sat_tail_fused_us"] * 1e-6) / 1e9,
                       "hbm_frac": sat_bytes / (kt["sat_tail_fused_us"] * 1e-6) / 1e9 / pk["hbm_gbs"],
                       "pair_gflops": 8.0 * sat_pairs / (kt["sat_tail_fused_us"] * 1e-6) / 1e9},
        "knn_softproj": {"us": kt["sat_knn_softproj_us"], "hbm_gbs_algorithmic": pair_bytes_sp / B * B_SAT / (kt["sat_knn_softproj_us"] * 1e-6) / 1e9},
        "chamfer": {"us": kt["sat_chamfer_us"], "hbm_gbs_algorithmic": pair_bytes_cd / B * B_SAT / (kt["sat_chamfer_us"] * 1e-6) / 1e9},
        "note": "arithmetic intensity of the pair work is 3*N*M*8 flop / 22.5 KB = 70 flop/B per cloud before top-k bookkeeping: with the machine "
                "full these kernels are FP32-issue bound, not HBM bound (SURVEY.md section 8(d) caveat)",
    }
    # ---- the reference's GPU path on this box (row G0), N=1 only: stock torch layer stack + the reference's Chamfer kernels for sm_100
    gpu_ref = None
    if world == 1:
        try:
            from oracle import ref_cuda
            from oracle.torch_reference import time_gpu_reference

            if ref_cuda.available():
                gpu_ref = time_gpu_reference(dev_pool, M, BOTTLENECK, K_NN, steps=100, warmup=10)
                gpu_ref["clouds_per_s"] = B / (gpu_ref["step_us"] * 1e-6)
                gpu_ref["ours_over_reference_gpu"] = gpu_ref["step_us"] / (ms_val / args.steps * 1e3)
            else:
                gpu_ref = {"unavailable": "oracle/_ref/libsamplenet_ref_cuda.so not built"}
        except Exception as exc:
            gpu_ref = {"error": str(exc)[:300]}
    # ---- CPU baseline beside it (N=1 only; bounded: a few full B=32 steps, in a fresh interpreter pinned to one NUMA node)
    cpu_base = None
    if world == 1:
        try:
            cl = cpu_arm_subprocess(10, 3)
            cpu_base = cl["cpu_baseline"]
            cpu_base["ms_per_step"] = cl["ms_per_step"]
        except Exception as exc:
            cpu_base = {"error": str(exc)[:300]}
    line = {
        "metric": METRIC, "value": value, "unit": "clouds/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_val / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "global_batch": B * world, "parallelism": "batch-sharded replicas x%d (no collective in fwd+loss)" % world,
                   "l2": "rotating pool of %d distinct input batches (%.0f MB > 126 MB L2); weights (1 MB) stay resident as in training" % (pool_n, pool_n * nbytes / 1e6),
                   "api": "samplenet_b200.PipelinedHostStep (SampleNet.forward + get_simplification_loss in one CUDA graph per slot; value: run_async with device-resident batches, e2e: submit/launch/finish from pinned host memory)"},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "clouds/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
                "sync": "every step's loss is read on the host; two steps in flight, H2D on a copy stream, the 4-byte loss D2H on a third stream behind each graph (samplenet_b200.PipelinedHostStep); the timed region starts and ends with an empty pipeline"},
        "gpu_launches": int(step.launches_per_step) * args.steps,
        "launches_per_step": int(step.launches_per_step),
        "value_single_graph": {"value": world * B * args.steps / (ms_single * 1e-3), "ms_per_step": ms_single / args.steps,
                               "note": "same step with the device-to-device copy of the rotating input and the graph replay on ONE stream"},
        "roofline": roofline,
        "roofline_pairwise": roofline_pairwise,
        "kernel_us": kt,
        "cpu_baseline": cpu_base,
        "gpu_reference": gpu_ref,
    }
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (value leg, rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
