"""CPU-only checks (no GPU needed): the C-ABI library builds, loads and exports every symbol include/*.h declares;
the host-side mirror of the reference interface behaves like the reference (constructor errors, warnings, state-dict
keys, parser flags); the product refuses CPU tensors instead of falling back."""
import os
import re
import subprocess
import warnings

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sb():
    import __graft_entry__ as ge

    ge.build()
    import samplenet_b200

    return samplenet_b200


def test_library_exports_every_declared_symbol(sb):
    hdr = open(os.path.join(ROOT, "include", "samplenet_b200.h")).read() + open(os.path.join(ROOT, "include", "samplenet_b200_debug.h")).read()
    assert "snb200_debug" not in open(os.path.join(ROOT, "include", "samplenet_b200.h")).read()   # bring-up hooks live in their own header
    declared = sorted(set(re.findall(r"\b(snb200_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 20
    lib = sb._lib.lib()
    for name in declared:
        assert hasattr(lib, name), "libsamplenet_b200.so does not export %s" % name
    assert sorted(sb._lib.exported_symbols()) == declared  # the ctypes table covers exactly the header
    out = subprocess.run(["nm", "-D", "--defined-only", sb._lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (\w+)", out))
    assert set(declared) <= exported
    # nothing but the C ABI leaks out of the library
    assert all(s.startswith("snb200_") for s in exported), sorted(exported)[:10]
    assert lib.snb200_version() == 100


def test_library_is_sm100a_with_tma_bulk_copies(sb):
    sass = subprocess.run(["cuobjdump", "-sass", sb._lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    assert "UBLKCP" in sass  # cp.async.bulk (TMA) staging of the point tiles
    assert "UTCHMMA" in sass and "LDTM" in sass  # tcgen05.mma kind::tf32 with the accumulators read back from tensor memory
    assert "ACQBULK" in sass and "PREEXIT" in sass  # griddepcontrol.wait / launch_dependents (programmatic dependent launch)


def test_primed_workspace_context_is_scoped_and_nestable(sb):
    """Host logic of the self-cleaning-workspace opt-in (no launch): the provider is thread-local, scoped, and restored on exit."""
    ops = sb.ops
    assert getattr(ops._ACTIVE_PW, "pw", None) is None
    a, b = ops.PrimedWorkspaces(), ops.PrimedWorkspaces()
    with ops.primed_workspaces(a) as got:
        assert got is a and ops._ACTIVE_PW.pw is a
        with ops.primed_workspaces(b):
            assert ops._ACTIVE_PW.pw is b
        assert ops._ACTIVE_PW.pw is a
        with pytest.raises(RuntimeError):
            with ops.primed_workspaces(b):
                raise RuntimeError("boom")
        assert ops._ACTIVE_PW.pw is a
    assert ops._ACTIVE_PW.pw is None
    import threading
    seen = []
    with ops.primed_workspaces(a):
        t = threading.Thread(target=lambda: seen.append(getattr(ops._ACTIVE_PW, "pw", None)))
        t.start(); t.join()
    assert seen == [None]
    assert sb._lib.GEN_WORKSPACE_PRIMED == 32
    hdr = open(os.path.join(ROOT, "include", "samplenet_b200.h")).read()
    assert re.search(r"#define\s+SNB200_GEN_WORKSPACE_PRIMED\s+32", hdr)


def test_generator_rejects_undefined_flag_bits(sb):
    """A generator flag bit the header does not define is an error, checked before any other argument (no launch), so a caller that
    still sets the retired bit 64 is told so instead of silently getting a different kernel."""
    lib = sb._lib.lib()
    rc = lib.snb200_generator_forward(2, 16, 0, None, 5, None, 4, None, 1, None, 0, None, 64, None, 0, None)
    assert rc == -1
    assert "flags" in lib.snb200_last_error().decode()
    rc = lib.snb200_generator_train_forward(2, 16, 0, None, 5, None, 4, None, None, 0, None, None, 64, None, 0, None)
    assert rc == -1
    assert "flags" in lib.snb200_last_error().decode()


def test_samplenet_constructor_contract(sb):
    with pytest.raises(ValueError):
        sb.SampleNet(64, 128, 8, input_shape="nbc")
    with pytest.raises(ValueError):
        sb.SampleNet(64, 128, 8, output_shape="xyz")
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        sb.SampleNet(64, 128, 8, input_shape="bnc", output_shape="bcn")
        assert any("input_shape is different to output_shape" in str(x.message) for x in w)
    net = sb.SampleNet(64, 128, 8)
    assert net.name == "samplenet" and net.project._group_size == 8
    keys = set(net.state_dict().keys())
    want = {"project._temperature"}
    for i in range(1, 6):
        want |= {"conv%d.weight" % i, "conv%d.bias" % i} | {"bn%d.%s" % (i, s) for s in ("weight", "bias", "running_mean", "running_var", "num_batches_tracked")}
    for i in range(1, 5):
        want |= {"fc%d.weight" % i, "fc%d.bias" % i}
    for i in range(1, 4):
        want |= {"bn_fc%d.%s" % (i, s) for s in ("weight", "bias", "running_mean", "running_var", "num_batches_tracked")}
    assert keys == want
    assert net.conv5.weight.shape == (128, 128, 1) and net.fc4.weight.shape == (192, 256)
    assert float(net.project.sigma()) == 1.0 and float(sb.SoftProjection(4, 0.05, min_sigma=1e-2).sigma()) == pytest.approx(1e-2)
    n_params = sum(p.numel() for p in net.parameters())
    assert n_params == 33408 + 213952 + 2432 + 1  # SURVEY.md section 5


def test_default_init_matches_torch_seed_order(sb):
    """Same parameter registration order as the reference => same default init under the same seed."""
    torch.manual_seed(0)
    a = sb.SampleNet(64, 128, 8)
    torch.manual_seed(0)
    conv1 = torch.nn.Conv1d(3, 64, 1)
    assert torch.equal(a.conv1.weight, conv1.weight)


def test_parser_flags(sb):
    p = sb.sputils.get_parser()
    a = p.parse_args([])
    assert (a.num_in_points, a.num_out_points, a.bottleneck_size, a.projection_group_size) == (1024, 64, 128, 8)
    assert (a.alpha, a.lmbda, a.gamma, a.delta, a.skip_projection) == (0.01, 0.01, 1, 0, False)
    b = p.parse_args(["-in", "2048", "-out", "32", "-gs", "7", "--skip-projection", "--alpha", "30"])
    assert (b.num_in_points, b.num_out_points, b.projection_group_size, b.skip_projection, b.alpha) == (2048, 32, 7, True, 30.0)


def test_no_cpu_fallback(sb):
    with pytest.raises(RuntimeError, match="CUDA-only"):
        sb.ChamferDistance()(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3))
    net = sb.SampleNet(8, 16, 2, input_shape="bnc", output_shape="bnc")
    with pytest.raises(RuntimeError, match="CUDA-only"):
        net(torch.zeros(2, 16, 3))
    with pytest.raises(RuntimeError, match="CUDA-only"):
        sb.tf_ops.approx_match(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3))
    # the product never imports the oracle
    import sys
    assert not any(m.startswith("oracle") for m in sys.modules if "samplenet_b200" in (getattr(sys.modules[m], "__file__", "") or ""))
    for root, _, files in os.walk(os.path.join(ROOT, "samplenet_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(root, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "liboracle" not in src, f


def test_eval_and_skip_projection_losses_are_zero_without_gpu(sb):
    net = sb.SampleNet(8, 16, 2, skip_projection=True)
    x = torch.zeros(2, 3, 16)
    assert float(net.get_simplification_loss(x, x, 8)) == 0.0
    assert float(net.get_projection_loss()) == 0.0
    net2 = sb.SampleNet(8, 16, 2).eval()
    assert float(net2.get_simplification_loss(x, x, 8)) == 0.0 and float(net2.get_projection_loss()) == 0.0
