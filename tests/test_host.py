"""CPU tests of the host side: the C-ABI library loads and exports exactly what
include/ganet_b200.h declares, the drop-in import surface resolves, the product
path refuses to run without a GPU (no silent fallback), and the pure-Python
pieces (losses, normalisation) match the reference's arithmetic."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def native_so():
    from ganet_b200 import build
    return build.build()


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "ganet_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ganet_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(native_so):
    handle = ctypes.CDLL(native_so)
    names = _declared_symbols()
    assert len(names) >= 13
    for n in names:
        assert hasattr(handle, n), "libganet_b200.so does not export " + n
    from ganet_b200 import _lib
    assert sorted(_lib.EXPORTED_SYMBOLS) == names      # the Python binding covers the whole header
    handle.ganet_abi_version.restype = ctypes.c_int
    assert handle.ganet_abi_version() == 2
    handle.ganet_error_string.restype = ctypes.c_char_p
    assert b"workspace" in handle.ganet_error_string(-3)


def test_library_contains_only_sm100a_code(native_so):
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-lelf", native_so], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_argument_validation_without_gpu(native_so):
    """Argument errors are reported before any CUDA call, so this runs on CPU."""
    from ganet_b200 import _lib
    L = _lib.lib()
    i64 = ctypes.c_int64
    sz = ctypes.c_size_t
    assert L.ganet_sga_forward(None, None, None, None, None, None, None, None, None, sz(0),
                               i64(1), i64(1), i64(1), i64(1), i64(1), None) == -1
    dummy = ctypes.c_void_p(16)
    assert L.ganet_sga_forward(dummy, dummy, dummy, dummy, dummy, dummy, dummy, None, dummy, sz(1 << 20),
                               i64(1), i64(1), i64(1000), i64(1), i64(1), None) == -2   # D > 768
    assert L.ganet_sga_forward(dummy, dummy, dummy, dummy, dummy, dummy, dummy, None, dummy, sz(16),
                               i64(1), i64(1), i64(8), i64(4), i64(4), None) == -3     # workspace too small
    assert L.ganet_sga_forward(dummy, dummy, dummy, dummy, dummy, dummy, dummy, dummy, dummy, sz(1 << 20),
                               i64(1), i64(1), i64(300), i64(1), i64(1), None) == -2   # kept aggregates need D <= 288
    dims = (i64(2), i64(3), i64(4), i64(5), i64(6))
    S, HW = 4 * 5 * 6, 5 * 6
    fmin, fbest = L.ganet_sga_forward_workspace_min(*dims), L.ganet_sga_forward_workspace_best(*dims)
    bmin, bbest = L.ganet_sga_backward_workspace_min(*dims), L.ganet_sga_backward_workspace_best(*dims)
    assert 9 * S + 40 * HW <= fmin <= 9 * S + 40 * HW + 6 * 256      # xT, outT (f32) + maskT (u8) + 2 guidance
    assert 17 * S + 40 * HW <= bmin <= 17 * S + 40 * HW + 7 * 256    # a, xT, goT, giT + maskT + g, gg
    assert fmin < fbest <= 6 * fmin and bmin < bbest <= 6 * bmin
    d2 = ctypes.c_void_p(32)
    assert L.ganet_lga_forward(dummy, dummy, d2, i64(1), i64(1), i64(1), i64(1), 9, None) == -2
    assert L.ganet_lga_forward(dummy, dummy, dummy, i64(1), i64(1), i64(1), i64(1), 2, None) == -1   # y aliases x


def test_product_path_refuses_cpu_tensors(native_so):
    """No CPU fallback: CPU tensors raise instead of silently computing elsewhere."""
    from ganet_b200 import _lib, modules
    x = torch.zeros(1, 1, 2, 3, 4)
    g = torch.zeros(1, 1, 5, 3, 4)
    with pytest.raises(_lib.GanetNativeError):
        modules.SGA()(x, g, g, g, g)
    with pytest.raises(_lib.GanetNativeError):
        modules.LGA2(2)(torch.zeros(1, 3, 4, 5), torch.zeros(1, 75, 4, 5))
    with pytest.raises(_lib.GanetNativeError):
        modules.DisparityRegression(2)(torch.zeros(1, 3, 4, 5))
    with pytest.raises(_lib.GanetNativeError):
        modules.GetCostVolume(2)(torch.zeros(1, 3, 4, 5), torch.zeros(1, 3, 4, 5))


def test_product_package_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "ganet_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text, \
                    "%s mentions the oracle" % f
    for dirpath, _, files in os.walk(os.path.join(ROOT, "libs")):
        for f in files:
            if f.endswith(".py"):
                assert "oracle" not in open(os.path.join(dirpath, f)).read()


def test_reference_import_surface():
    """Every name the reference's consumers import resolves (models/GANet_deep.py:4-8,
    train.py:5), with the reference's constructor signatures."""
    from libs.GANet.modules.GANet import (SGA, LGA, LGA2, LGA3, LGA3D, LGA3D2, LGA3D3,  # noqa: F401
                                          DisparityRegression, GetCostVolume, MyLoss, MyLoss2,
                                          MyNormalize)
    from libs.GANet.functions.GANet import (SgaFunction, Lga2Function, Lga3Function,  # noqa: F401
                                            LgaFunction, Lga3dFunction, Lga3d2Function,
                                            Lga3d3Function, MyLoss2Function, MyLossFunction, GANet)
    from libs.sync_bn.modules.sync_bn import BatchNorm2d, BatchNorm3d
    assert GetCostVolume(64).maxdisp == 65 and DisparityRegression(192).maxdisp == 193
    assert LGA2(radius=2).radius == 2 and LGA3(2).radius == 2 and LGA(2).radius == 2
    assert len(list(SGA().parameters())) == 0 and len(SGA().state_dict()) == 0
    assert sorted(BatchNorm3d(4).state_dict()) == ["bias", "num_batches_tracked", "running_mean",
                                                   "running_var", "weight"]
    assert isinstance(BatchNorm2d(4), torch.nn.BatchNorm2d)
    for name in ("sga_cuda_forward", "sga_cuda_backward", "lga_cuda_forward", "lga_cuda_backward",
                 "lga3d_cuda_forward", "lga3d_cuda_backward"):
        assert callable(getattr(GANet, name))         # GANet_cuda.cpp:67-75
    from libs.GANet.build.lib import GANet as G2      # the compiled pybind11 module when it has been built
    for name in ("sga_cuda_forward", "sga_cuda_backward", "lga_cuda_forward", "lga_cuda_backward",
                 "lga3d_cuda_forward", "lga3d_cuda_backward"):
        assert callable(getattr(G2, name))


def test_reference_models_construct_unchanged():
    """models/GANet_deep.py and GANet11.py (as copied by oracle/build_ref.py into baseline/_ref/models)
    import and build on the new modules; the parameter counts are the reference's (SURVEY.md Appendix C.4)."""
    from baseline import refmodels
    if not refmodels.available():
        pytest.skip("baseline/_ref/models not built (no reference tree at build time)")
    deep, g11 = refmodels.build("GANet_deep", 192), refmodels.build("GANet11", 192)
    assert sum(p.numel() for p in deep.parameters()) == 6580112
    assert sum(p.numel() for p in g11.parameters()) == 4483728
    assert len(deep.state_dict()) == 479 and len(g11.state_dict()) == 364
    import ganet_b200.modules as M
    assert isinstance(deep.cost_agg.sga1.SGA, M.SGA)
    assert isinstance(deep.cv, M.GetCostVolume)


def _ref_myloss2(input1, input2, thresh=1, alpha=2):
    """MyLoss2Function restated with the reference's in-place masked updates
    (functions/GANet.py:266-289) as the checker for the functional port."""
    diff = input1 - input2
    temp = torch.abs(diff)
    temp[temp < thresh] = temp[temp < thresh] ** 2 / thresh
    tag = (temp <= thresh + alpha) & (temp >= thresh)
    temp[tag] = temp[tag] * 2 - (temp[tag] - thresh) ** 2 / (2.0 * alpha) - thresh
    temp[temp > thresh + alpha] += (alpha / 2.0)
    loss = torch.mean(temp)
    scale = torch.abs(diff)
    scale[scale > thresh + alpha] = 1
    tag = (scale <= thresh + alpha) & (scale >= thresh)
    scale[tag] = 2 - (scale[tag] - thresh) / alpha
    tag = scale < thresh
    scale[tag] = 2 * scale[tag] / thresh
    d = diff.clone()
    d[d > 0] = 1.0
    d[d < 0] = -1.0
    return loss, d * scale / scale.numel()


def test_myloss2_matches_reference_arithmetic():
    from ganet_b200.modules import MyLoss2
    torch.manual_seed(0)
    a = (torch.randn(4, 9, 11) * 3).requires_grad_()
    b = torch.randn(4, 9, 11)
    loss = MyLoss2(1, 2)(a, b)
    loss.backward()
    ref_loss, ref_grad = _ref_myloss2(a.detach(), b)
    assert torch.allclose(loss, ref_loss, rtol=1e-6)
    assert torch.allclose(a.grad, ref_grad, rtol=1e-6, atol=1e-9)


def test_myloss_and_mynormalize():
    from ganet_b200.modules import MyLoss, MyNormalize
    torch.manual_seed(1)
    a = (torch.randn(3, 50) * 4).requires_grad_()
    b = torch.randn(3, 50)
    loss = MyLoss()(a, b)
    assert torch.allclose(loss, (a - b).abs().mean())
    loss.backward()
    diff = (a - b).detach()
    s = diff.abs()
    s = torch.where(s > 5, torch.ones_like(s), s)
    s = torch.where((s <= 5) & (s >= 1), 2 - (s - 3).abs() / 2, s)
    assert torch.allclose(a.grad, torch.sign(diff) * s)
    x = torch.randn(2, 5, 3)
    x[0, :, 0] = 0
    y = MyNormalize(1)(x)
    n = x.abs().sum(1, keepdim=True)
    assert torch.allclose(y[:, :, 1:], (x / (n + 1e-6))[:, :, 1:])
    assert torch.all(y[0, :, 0] == 0)


def test_bench_shard_plan_and_roofline_arithmetic():
    import bench
    assert bench.shard_samples(8, 1, 0) == list(range(8))
    assert bench.shard_samples(8, 8, 3) == [3]
    assert bench.shard_samples(8, 4, 3) == [6, 7]
    got = sorted(s for r in range(2) for s in bench.shard_samples(8, 2, r))
    assert got == list(range(8))
    # SURVEY.md 8d: SGA fwd+bwd = 22 + 240/D bytes per voxel, LGA2 = 20 + 900/D
    assert abs(bench.sga_bytes_per_voxel(192) - 23.25) < 1e-9
    assert abs(bench.lga2_bytes_per_voxel(192) - 24.6875) < 1e-9


def test_bench_samples_per_call():
    import bench
    assert bench.samples_per_call(2, 8, lambda c: True) == 2
    assert bench.samples_per_call(2, 1, lambda c: True) == 1          # 8 ranks: one sample each
    assert bench.samples_per_call(4, 8, lambda c: c <= 1) == 1        # no room: shrink, never loop forever
    assert bench.samples_per_call(4, 8, lambda c: c <= 2) == 2
    assert bench.samples_per_call(2, 0, lambda c: False) == 1         # a rank without samples
    assert bench.samples_per_call(3, 8, lambda c: False) == 1


def test_bench_output_dump(tmp_path, monkeypatch):
    """--dump-outputs: one float32 file per output of the timed path, filled call by call at the caller's batch
    offset; an output larger than its share of DUMP_ELEMENTS is kept at the same seeded positions in every sample,
    chosen when the dump is set up (before the timed window)."""
    import bench
    monkeypatch.setattr(bench, "DUMP_ELEMENTS", 200)
    B, C, D, H, W = 3, 2, 4, 3, 5
    gen = torch.Generator().manual_seed(0)

    def outputs(n):
        out = torch.randn(n, C, D, H, W, generator=gen)
        return (out, (out > 0).to(torch.uint8), -out, [torch.randn(n, C, 5, H, W, generator=gen) for _ in range(4)],
                torch.randn(n, D, H, W, generator=gen), torch.randn(n, D, H, W, generator=gen),
                torch.randn(n, 75, H, W, generator=gen))

    first, second = outputs(2), outputs(1)
    dump = bench.OutputDump(torch, "cpu", B, C, D, H, W)
    dump.keep(0, first)
    dump.keep(2, second)
    dump.write(str(tmp_path))
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(n + ".npy" for n in bench.DUMP_NAMES)
    pos = bench.dump_positions(C * D * H * W, B)
    assert pos is not None and np.array_equal(pos, bench.dump_positions(C * D * H * W, B))
    out = np.load(tmp_path / "sga_out.npy")
    assert out.dtype == np.float32 and out.shape == (B, len(pos))
    assert np.array_equal(out[:2], first[0].reshape(2, -1)[:, pos].numpy())
    assert np.array_equal(out[2], second[0].reshape(-1)[pos].numpy())
    assert np.array_equal(np.load(tmp_path / "sga_mask.npy"), (out > 0).astype(np.float32))
    y = np.load(tmp_path / "lga2_out.npy")                      # small enough to keep whole
    assert y.shape == (B, D, H, W) and np.array_equal(y, torch.cat([first[4], second[4]]).numpy())


def test_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver launches next to ours) prints exactly
    one JSON line with the contract keys; rank != 0 prints nothing and exits 0."""
    import json
    import subprocess
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
           "--warmup", "0", "--batch", "1", "--channels", "2", "--depth", "8", "--height", "8", "--width", "16"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-1000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in d["config"]
    r2 = subprocess.run(cmd, capture_output=True, text=True, timeout=60, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r2.returncode == 0 and r2.stdout.strip() == ""


def test_reference_arm_is_pinned_fixed_and_flagged():
    """VERDICT r1 #5: the CPU arm times a FIXED sample (two full (n,c) slices), with one bound OpenMP thread
    per physical core, reports the median step and says that ms_per_step is an extrapolation."""
    import json
    import subprocess
    import bench
    assert bench._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert 1 <= bench.physical_cores() <= (os.cpu_count() or 1)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3",
           "--warmup", "1", "--depth", "8", "--height", "8", "--width", "16"]
    env = {k: v for k, v in os.environ.items() if not k.startswith("OMP_")}
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stderr[-1000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["ms_per_step_extrapolated"] is True and d["measured_s_per_step"] > 0
    assert d["value_min_max"][0] <= d["value"] <= d["value_min_max"][1]          # the median step
    cb = d["cpu_baseline"]
    assert cb["omp"] == {"OMP_NUM_THREADS": str(bench.physical_cores()), "OMP_PLACES": "cores",
                         "OMP_PROC_BIND": "close"}
    assert "1x2x8x8x16" in cb["sample"] and "1x8x8x16" in cb["sample"]            # fixed shapes, 2 slices
    # an explicit user setting wins
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=dict(env, OMP_NUM_THREADS="2"))
    assert json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]["threads"] == 2


def test_sync_bn_shim_signature_and_conversion():
    """libs/sync_bn shim: the reference's constructor arguments (modules/sync_bn.py:64-66) are accepted,
    state_dict keys are the reference's, and the classes convert to nn.SyncBatchNorm for DDP."""
    from libs.sync_bn.modules.sync_bn import BatchNorm1d, BatchNorm2d, BatchNorm3d
    m = BatchNorm2d(4, eps=1e-5, momentum=0.1, sync=False, activation="leaky_relu", slope=0.1, inplace=True)
    x = torch.randn(2, 4, 3, 3)
    y = m(x)
    ref = torch.nn.functional.leaky_relu(torch.nn.functional.batch_norm(x, None, None, m.weight, m.bias, True, 0.1, 1e-5), 0.1)
    assert torch.allclose(y, ref, atol=1e-6)
    assert torch.equal(BatchNorm3d(2)(torch.ones(1, 2, 2, 2, 2)), torch.nn.BatchNorm3d(2)(torch.ones(1, 2, 2, 2, 2)))
    with pytest.raises(ValueError):
        BatchNorm1d(3, activation="swish")
    net = torch.nn.Sequential(torch.nn.Conv2d(3, 4, 1), BatchNorm2d(4), torch.nn.Conv3d(1, 2, 1), BatchNorm3d(2))
    conv = torch.nn.SyncBatchNorm.convert_sync_batchnorm(net)
    assert sum(isinstance(k, torch.nn.SyncBatchNorm) for k in conv.modules()) == 2
    assert sorted(conv[1].state_dict()) == ["bias", "num_batches_tracked", "running_mean", "running_var", "weight"]


def test_model_harness_loads_the_copied_reference_models():
    """baseline/refmodels.py loads models/*.py as copied by oracle/build_ref.py into baseline/_ref/models and
    wires them to THIS repository's operators; baseline/refops.py finds every hot-path module instance."""
    from baseline import refmodels
    if not refmodels.available():
        pytest.skip("baseline/_ref/models not built (no reference tree at build time)")
    import ganet_b200.modules as M
    deep = refmodels.build("GANet_deep", 192, seed=1)
    assert sum(p.numel() for p in deep.parameters()) == 6580112
    kinds = [type(m).__name__ for m in deep.modules() if isinstance(m, (M.SGA, M.LGA2, M.GetCostVolume, M.DisparityRegression))]
    assert kinds.count("SGA") == 7 and kinds.count("GetCostVolume") == 1
    assert kinds.count("LGA2") == 1 and kinds.count("DisparityRegression") == 3
    g11 = refmodels.build("GANet11", 192, seed=1)
    assert sum(isinstance(m, M.SGA) for m in g11.modules()) == 4
    from baseline.ddp_check import loss_fn
    import torch.nn.functional as F
    t = torch.zeros(1, 4, 4)
    assert float(loss_fn(F, (t + 1, t + 1, t + 1), t)) == pytest.approx(0.2 * 0.5 + 0.6 * 0.5 + 0.5)
    assert float(loss_fn(F, (t + 1, t + 1), t)) == pytest.approx(0.4 * 0.5 + 1.2 * 0.5)


def test_aggregate_volumes_and_workspace_are_consistent(native_so):
    """The kept-aggregates buffer is 4 volumes where the horizontal scans run in the standard layout (needs the
    driver's tensor-map encoder, so 5 on a CPU-only box), and then no scratch beyond two aggregates is asked."""
    from ganet_b200 import _lib
    L = _lib.lib()
    i64 = ctypes.c_int64
    dims = (i64(1), i64(2), i64(24), i64(16), i64(48))
    S = 24 * 16 * 48
    v = L.ganet_sga_aggregate_volumes(*dims)
    assert v in (4, 5)
    if v == 4:
        assert L.ganet_sga_forward_workspace_min(*dims) <= 2 * 4 * S + 512
        assert L.ganet_sga_backward_workspace_min(*dims) <= 4 * S + 256
    assert L.ganet_sga_aggregate_volumes(i64(1), i64(2), i64(24), i64(16), i64(50)) == 5      # W % 16 != 0
    assert L.ganet_sga_aggregate_volumes(i64(1), i64(2), i64(288), i64(16), i64(48)) == 5     # D > 256


def test_model_patchers_find_the_reference_blocks():
    """ganet_b200.fused patches the reference's SGABlock / DispAgg instances by class name (models/*.py stay
    untouched) and undoes it; counts are the models' (GANet_deep.py:305-315: 7 SGABlocks, one DispAgg)."""
    from baseline import refmodels
    if not refmodels.available():
        pytest.skip("baseline/_ref/models not built")
    from ganet_b200 import fused
    deep = refmodels.build("GANet_deep", 192, seed=1)
    assert fused.fuse_sga_blocks(deep) == 7 and fused.fuse_disp_heads(deep) == 1
    blk = deep.cost_agg.sga1
    assert "forward" in blk.__dict__ and blk.forward.__func__ is fused._fused_sga_block_forward
    assert fused.unfuse_sga_blocks(deep) == 7 and fused.unfuse_disp_heads(deep) == 1
    assert "forward" not in blk.__dict__ and type(blk).forward is not fused._fused_sga_block_forward
    assert fused.fuse_sga_blocks(refmodels.build("GANet11", 192, seed=1)) == 4
