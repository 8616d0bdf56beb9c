"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI,
against
  (1) the UNMODIFIED reference CUDA extension, through its results on the same seeded
      inputs (tests/golden/ref_cuda_*, written by tests/golden/make_golden.py --cuda):
      SGA forward values, direction mask and depth arg-max BIT-EXACT (SHA-256 digests);
      gradients and LGA within the north_star tolerance of 1e-4 relative fp32 (values at
      fixed sample positions and each tensor's largest magnitude);
  (2) the CPU oracle (oracle/ganet_oracle.c, fused rounding): same criteria;
  (3) the committed golden vectors (tests/golden/, generated from the reference's
      kernel bodies on the host; unfused rounding, hence tolerance not bit-exactness).
"""
import os

import numpy as np
import pytest
import torch

from oracle import api as oracle
from oracle import ref_gpu
from util import (GOLD, assert_close, assert_close_to_golden, case_id, digest, golden_json, golden_values,
                  lga_inputs, sga_inputs)

pytestmark = pytest.mark.gpu
RTOL = 1e-4          # north_star: 1e-4 relative fp32

needs_ref = pytest.mark.skipif(not ref_gpu.available(),
                               reason="oracle/_ref/GANet*.so (reference CUDA extension) not built")


@pytest.fixture(scope="module")
def ref_digests():
    return golden_json("ref_cuda_digests.json")


@pytest.fixture(scope="module")
def ref_values():
    return golden_values("ref_cuda_values.npz")


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def npy(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def ops():
    from ganet_b200 import ops as o
    return o


# shapes: tiny edge cases (D=1, H=1, W=1, odd/even D, D not a multiple of the lane
# chunking), config 1 of BASELINE.json, and the model's 1/6-resolution D=33
SGA_SHAPES = [(2, 3, 7, 5, 6), (1, 2, 1, 4, 3), (1, 1, 2, 1, 5), (1, 2, 3, 6, 1), (1, 1, 1, 1, 1),
              (1, 2, 9, 8, 10), (1, 1, 33, 9, 13), (1, 2, 65, 6, 11), (1, 1, 192, 5, 9),
              (1, 1, 288, 3, 5), (1, 1, 100, 4, 35), (1, 8, 48, 48, 96),
              # H and W multiples of 16: the TMA-staged kernels run in both layouts; partial
              # 32-column strips (48, 80), depth not filling the last warp (65, 33), one stage
              (1, 2, 24, 16, 48), (2, 2, 65, 32, 80), (1, 1, 192, 16, 32), (1, 2, 33, 16, 16),
              (1, 1, 256, 16, 16),
              # D > 288: the generic line kernels (sga_forward_lines / sga_backward_lines) carry the
              # whole call -- MODE_FIRST / MODE_COMBINE and the vertical line-kernel backward
              (1, 1, 300, 4, 6), (1, 2, 513, 3, 5)]


@pytest.mark.parametrize("shape", SGA_SHAPES)
def test_sga_forward_bit_exact_vs_reference_cuda(ops, ref_digests, shape):
    x, g, _ = sga_inputs(shape, seed=1 + sum(shape))
    xt, gt = cu(x), [cu(a) for a in g]
    out, mask = ops.sga_forward(xt, *gt)
    key = "sga_forward/%s/" % case_id(shape)
    assert digest(out) == ref_digests[key + "out"], "SGA forward values differ from the reference CUDA kernels"
    assert digest(mask, np.uint8) == ref_digests[key + "mask"], "direction mask differs"
    assert digest(ops.sga_direction(xt, gt[3], 3)) == ref_digests[key + "left"], "left aggregate differs"


DIRECTION_SHAPE = (1, 2, 12, 20, 24)


@pytest.mark.parametrize("direction", [0, 1, 2, 3])
def test_each_direction_bit_exact_vs_reference_cuda(ops, ref_digests, direction):
    """Isolate one scan kernel of the reference: x in [1, 1.1) with positive weights
    keeps every aggregate in [1, 1.1); scaling the guidance of `direction` by 1.2
    lifts that aggregate above 1.2 everywhere, so it wins the max at every voxel and
    `out` IS that direction's aggregate (make_golden.py asserts that the reference's
    mask is `direction` everywhere)."""
    x, g, _ = sga_inputs(DIRECTION_SHAPE, seed=40 + direction, positive=True)
    g[direction] = (g[direction] * 1.2).astype(np.float32)
    xt, gt = cu(x), [cu(a) for a in g]
    key = "sga_direction/%d/" % direction
    mine = ops.sga_direction(xt, gt[direction], direction)
    assert digest(mine) == ref_digests[key + "out"]
    out, mask = ops.sga_forward(xt, *gt)
    assert bool((mask == direction).all()), "construction failed: direction does not dominate"
    assert digest(out) == ref_digests[key + "out"] and digest(mask, np.uint8) == ref_digests[key + "mask"]


@pytest.mark.parametrize("shape", SGA_SHAPES)
def test_sga_forward_bit_exact_vs_oracle(ops, shape):
    x, g, _ = sga_inputs(shape, seed=2 + sum(shape))
    out, mask = ops.sga_forward(cu(x), *[cu(a) for a in g])
    oo, om, od = oracle.sga_forward(x, *g, fused=True, want_dirs=True)
    assert np.array_equal(npy(out), oo)
    assert np.array_equal(npy(mask), om)
    for d in range(4):
        assert np.array_equal(npy(ops.sga_direction(cu(x), cu(g[d]), d)), od[d])


@pytest.mark.parametrize("shape", SGA_SHAPES)
def test_sga_backward_vs_reference_cuda(ops, ref_digests, ref_values, shape):
    x, g, go = sga_inputs(shape, seed=3 + sum(shape))
    xt, gt, got = cu(x), [cu(a) for a in g], cu(go)
    out, mask = ops.sga_forward(xt, *gt)
    gi, gg, idx = ops.sga_backward(xt, *gt, mask, got, want_max_idx=True)
    key = "sga_backward/%s/" % case_id(shape)
    assert digest(idx, np.int32) == ref_digests[key + "idx"], "max_idx (depth arg-max) differs"
    assert_close_to_golden(gi, ref_values, key + "gi", RTOL, what="gradInput")
    for d in range(4):
        assert_close_to_golden(gg[d], ref_values, key + "gg%d" % d, RTOL, what="guidance grad %d" % d)


@pytest.mark.parametrize("shape", SGA_SHAPES)
def test_sga_backward_vs_oracle(ops, shape):
    """Every element of every gradient against the CPU oracle (pinned to the reference's kernel bodies by
    test_oracle.py), including the D > 288 shapes that exercise the generic line-kernel backward."""
    x, g, go = sga_inputs(shape, seed=4 + sum(shape))
    xt, gt = cu(x), [cu(a) for a in g]
    out, mask = ops.sga_forward(xt, *gt)
    gi, gg, idx = ops.sga_backward(xt, *gt, mask, cu(go), want_max_idx=True)
    ogi, ogg, oidx = oracle.sga_backward(x, *g, npy(mask), go, fused=True)
    assert np.array_equal(npy(idx), oidx)
    assert_close(npy(gi), ogi, RTOL, "gradInput")
    for d in range(4):
        assert_close(npy(gg[d]), ogg[d], RTOL, "guidance grad %d" % d)


def test_sga_backward_workspace_chunking_is_invisible(ops):
    """Slices are independent: a one-slice workspace and a full one give the same bits."""
    shape = (2, 3, 10, 7, 9)
    x, g, go = sga_inputs(shape, seed=9)
    xt, gt, got = cu(x), [cu(a) for a in g], cu(go)
    out, mask = ops.sga_forward(xt, *gt)
    a = ops.sga_backward(xt, *gt, mask, got, workspace_bytes=1)          # -> minimum: one slice
    b = ops.sga_backward(xt, *gt, mask, got, workspace_bytes=1 << 30)
    assert torch.equal(a[0], b[0])
    assert all(torch.equal(p, q) for p, q in zip(a[1], b[1]))
    o1, m1 = ops.sga_forward(xt, *gt, workspace_bytes=1)
    assert torch.equal(o1, out) and torch.equal(m1, mask)


@pytest.mark.parametrize("shape", [(2, 3, 10, 7, 9), (1, 2, 24, 32, 48), (2, 2, 65, 32, 80), (1, 8, 48, 48, 96)])
def test_kept_aggregates_give_identical_results(ops, shape):
    """The memory-for-bandwidth variant (forward keeps the four aggregates, backward skips
    its recompute passes) must not change a single bit, with any workspace chunking."""
    x, g, go = sga_inputs(shape, seed=31 + sum(shape))
    xt, gt, got = cu(x), [cu(a) for a in g], cu(go)
    out, mask = ops.sga_forward(xt, *gt)
    out2, mask2, agg = ops.sga_forward(xt, *gt, keep_aggregates=True)
    assert torch.equal(out, out2) and torch.equal(mask, mask2)
    out3, mask3, agg3 = ops.sga_forward(xt, *gt, keep_aggregates=True, workspace_bytes=1)
    assert torch.equal(out, out3) and torch.equal(mask, mask3) and torch.equal(agg, agg3)
    for d in (0, 1):
        assert torch.equal(agg[d].view_as(xt), ops.sga_direction(xt, gt[d], d))
    if agg.shape[0] == 4:        # horizontal scans in the standard layout (W % 16 == 0, D <= 256)
        assert shape[4] % 16 == 0
        for d in (2, 3):
            assert torch.equal(agg[d].view_as(xt), ops.sga_direction(xt, gt[d], d))
    else:                        # transposed path: right^T, left^T, x^T
        assert agg.shape[0] == 5
        for d in (2, 3):
            a = ops.sga_direction(xt, gt[d], d)
            assert torch.equal(agg[d].view(*shape[:3], shape[4], shape[3]), a.transpose(3, 4).contiguous())
        assert torch.equal(agg[4].view(*shape[:3], shape[4], shape[3]), xt.transpose(3, 4).contiguous())
    ref = ops.sga_backward(xt, *gt, mask, got, want_max_idx=True)
    for wsb in (None, 1):
        got2 = ops.sga_backward(xt, *gt, mask, got, want_max_idx=True, aggregates=agg, workspace_bytes=wsb)
        assert torch.equal(ref[0], got2[0]) and torch.equal(ref[2], got2[2])
        assert all(torch.equal(p, q) for p, q in zip(ref[1], got2[1]))


def test_sga_module_keeps_aggregates_by_policy(monkeypatch):
    from ganet_b200.modules import SGA
    x, g, go = sga_inputs((1, 2, 8, 6, 7), seed=5)
    grads = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("GANET_B200_KEEP_AGGREGATES", mode)
        xt = cu(x).requires_grad_()
        gt = [cu(a).requires_grad_() for a in g]
        out = SGA()(xt, *gt)
        assert len(out.grad_fn.saved_tensors) == (7 if mode == "1" else 6)
        out.backward(cu(go))
        grads[mode] = [xt.grad] + [t.grad for t in gt]
    assert all(torch.equal(a, b) for a, b in zip(grads["0"], grads["1"]))


def test_sga_against_golden_vectors(ops):
    z = np.load(os.path.join(GOLD, "sga_ref_cpu.npz"))
    for k in range(int(z["n"])):
        x, go = z[f"x{k}"], z[f"go{k}"]
        g = [z[f"g{k}_{d}"] for d in range(4)]
        xt, gt = cu(x), [cu(a) for a in g]
        out, mask = ops.sga_forward(xt, *gt)
        assert_close(npy(out), z[f"out{k}"], RTOL, "out")
        # the golden vectors carry the host's unfused rounding: the mask may differ
        # only where the two best directions are within rounding distance
        bad = npy(mask) != z[f"mask{k}"]
        assert bad.mean() <= 0.01
        gi, gg = ops.sga_backward(xt, *gt, cu(z[f"mask{k}"]), cu(go))
        assert_close(npy(gi), z[f"gi{k}"], RTOL, "gradInput")
        for d in range(4):
            assert_close(npy(gg[d]), z[f"gg{k}_{d}"], RTOL, "guidance grad")


def test_tma_and_ldg_kernels_agree_bitwise(ops, tmp_path):
    """The code paths behind the process-wide switches (read once per process, hence subprocesses):
    horizontal scans in the standard layout (default), the H<->W transposed TMA path with and without
    its transpose-free small-call forward, the plain load/store kernels, and gradInput accumulated by
    TMA reduce-add or by load + add + store.  `out` and `mask` must be the same bits on every path;
    the transposed-family paths must also agree bit for bit on every gradient (same summation order),
    and the standard-layout path -- which sums over depth inside one warp -- within 1e-4."""
    import subprocess
    import sys
    code = (
        "import sys, torch, hashlib, numpy as np; sys.path.insert(0, %r); sys.path.insert(0, %r);"
        "from ganet_b200 import ops; from util import sga_inputs;"
        "x, g, go = sga_inputs((1, 2, 24, 32, 48), seed=77);"
        "cu = lambda a: torch.from_numpy(a).cuda();"
        "xt, gt = cu(x), [cu(a) for a in g];"
        "out, mask = ops.sga_forward(xt, *gt);"
        "gi, gg = ops.sga_backward(xt, *gt, mask, cu(go));"
        "h = hashlib.sha256();"
        "[h.update(t.cpu().numpy().tobytes()) for t in (out, mask)];"
        "h2 = hashlib.sha256();"
        "[h2.update(t.cpu().numpy().tobytes()) for t in (gi,) + tuple(gg)];"
        "np.savez(sys.argv[1], gi=gi.cpu().numpy(), **{'gg%%d' %% k: t.cpu().numpy() for k, t in enumerate(gg)});"
        "print(h.hexdigest(), h2.hexdigest())"
    ) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)))
    no_h = {"GANET_NO_HSCAN": "1"}
    knob_sets = [{}, no_h, dict(no_h, GANET_NO_DIRECT="1"), {"GANET_NO_TMA": "1"},
                 dict(no_h, GANET_TMA_REDUCE="1"), dict(no_h, GANET_TMA_REDUCE="0")]
    fwd, grad, files = [], [], []
    for i, knobs in enumerate(knob_sets):
        env = dict(os.environ)
        for k in ("GANET_NO_TMA", "GANET_NO_DIRECT", "GANET_FORCE_DIRECT", "GANET_TMA_REDUCE", "GANET_NO_HSCAN"):
            env.pop(k, None)
        env.update(knobs)
        f = str(tmp_path / ("grads%d.npz" % i))
        r = subprocess.run([sys.executable, "-c", code, f], env=env, capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stderr[-2000:]
        a, b = r.stdout.strip().splitlines()[-1].split()
        fwd.append(a); grad.append(b); files.append(f)
    assert len(set(fwd)) == 1, fwd
    assert len(set(grad[1:])) == 1, grad
    new, old = np.load(files[0]), np.load(files[1])
    for k in new.files:
        assert_close(new[k], old[k], RTOL, "standard-layout vs transposed path: " + k)


def test_lga_tiled_and_per_pixel_kernels_agree_bitwise(ops):
    """The TMA-tiled LGA kernels (lga_tile.cuh) keep the summation order of the per-pixel
    kernels (lga.cu): same bits.  GANET_LGA_NO_TILE is read once per process -> subprocess."""
    import subprocess
    import sys
    code = (
        "import sys, torch, hashlib; sys.path.insert(0, %r); sys.path.insert(0, %r);"
        "from ganet_b200 import ops; from util import lga_inputs;"
        "h = hashlib.sha256();"
        "cu = lambda a: torch.from_numpy(a).cuda();\n"
        "for shape in [(1, 9, 12, 40), (2, 6, 9, 44), (1, 33, 20, 152)]:\n"
        "    x, f, go = lga_inputs(shape, seed=13)\n"
        "    xt, ft, got = cu(x), cu(f), cu(go)\n"
        "    y = ops.lga_forward(xt, ft, 2)\n"
        "    gx, gf = ops.lga_backward(xt, ft, got, 2)\n"
        "    gx2, gf = ops.lga_backward(y, ft, got, 2, gf)\n"
        "    [h.update(t.cpu().numpy().tobytes()) for t in (y, gx, gx2, gf)]\n"
        "print(h.hexdigest())"
    ) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)))
    digests = []
    for knobs in ({}, {"GANET_LGA_NO_TILE": "1"}):
        env = dict(os.environ)
        env.pop("GANET_LGA_NO_TILE", None)
        env.update(knobs)
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
        assert r.returncode == 0, r.stderr[-2000:]
        digests.append(r.stdout.strip().splitlines()[-1])
    assert digests[0] == digests[1]


def test_sga_ties_and_constant_input(ops):
    x = torch.full((1, 2, 6, 5, 7), 0.75, device="cuda")
    g = [torch.full((1, 2, 5, 5, 7), 0.2, device="cuda") for _ in range(4)]
    out, mask = ops.sga_forward(x, *g)
    assert int(mask.max()) == 0                     # ties keep the lowest direction id
    _, _, idx = ops.sga_backward(x, *g, mask, torch.ones_like(x), want_max_idx=True)
    assert int(idx.max()) == 0                      # ties keep the lowest depth


# ---- LGA ---------------------------------------------------------------------
LGA_SHAPES = [(2, 7, 5, 6), (1, 3, 9, 11), (1, 1, 1, 1), (1, 5, 1, 40), (1, 4, 37, 3),
              (1, 33, 20, 150), (2, 2, 3, 5, 4),
              # W a multiple of 4, W >= 40, H >= 8, D >= 4: the TMA-tiled radius-2 kernels run;
              # partial tiles in both directions, depth not a multiple of the 4-plane stage,
              # more stages than the ring holds, the 5-D (lga3d) form
              (1, 9, 12, 40), (2, 6, 9, 44), (1, 33, 20, 152), (1, 4, 8, 72), (2, 2, 5, 8, 40)]


@pytest.mark.parametrize("shape", LGA_SHAPES)
def test_lga2_vs_reference_cuda(ops, ref_values, shape):
    x, f, go = lga_inputs(shape, seed=5)
    xt, ft, got = cu(x), cu(f), cu(go)
    y1 = ops.lga_forward(xt, ft, 2)
    y = ops.lga_forward(y1, ft, 2)
    g1, gf = ops.lga_backward(y1, ft, got, 2)
    gx, gf = ops.lga_backward(xt, ft, g1, 2, grad_f=gf)
    key = "lga2/%s/" % case_id(shape)
    assert_close_to_golden(y1, ref_values, key + "y1", RTOL, what="y1")
    assert_close_to_golden(y, ref_values, key + "y", RTOL, what="y")
    assert_close_to_golden(gx, ref_values, key + "gx", RTOL, what="grad_x")
    assert_close_to_golden(gf, ref_values, key + "gf", RTOL, what="grad_f")


@pytest.mark.parametrize("shape", LGA_SHAPES)
@pytest.mark.parametrize("radius", [2, 1, 0])
def test_lga_vs_oracle(ops, shape, radius):
    x, f, go = lga_inputs(shape, seed=6, radius=radius)
    xt, ft, got = cu(x), cu(f), cu(go)
    y = ops.lga_forward(xt, ft, radius)
    oy, _ = oracle.lga_forward(x, f, radius, 1)
    assert_close(npy(y), oy, RTOL, "y")
    gx, gf = ops.lga_backward(xt, ft, got, radius)
    ogx, ogf = oracle.lga_backward(x, f, None, go, radius, 1)
    assert_close(npy(gx), ogx, RTOL, "grad_x")
    assert_close(npy(gf), ogf, RTOL, "grad_f")


def test_lga_against_golden_vectors(ops):
    z = np.load(os.path.join(GOLD, "lga_ref_cpu.npz"))
    from ganet_b200.functions import Lga2Function, Lga3d2Function
    for k in range(int(z["n"])):
        x = cu(z[f"x{k}"]).requires_grad_()
        f = cu(z[f"f{k}"]).requires_grad_()
        fn = Lga2Function if x.dim() == 4 else Lga3d2Function
        y = fn.apply(x, f, 2)
        y.backward(cu(z[f"go{k}"]))
        assert_close(npy(y), z[f"y{k}"], RTOL, "y")
        assert_close(npy(x.grad), z[f"gx{k}"], RTOL, "grad_x")
        assert_close(npy(f.grad), z[f"gf{k}"], RTOL, "grad_f")


# ---- cost volume / regression ---------------------------------------------------
def _ref_cost_volume(x, y, dm):
    """libs/GANet/modules/GANet.py:119-134 run as written (stock torch ops)."""
    num, channels, height, width = x.size()
    cost = x.new().resize_(num, channels * 2, dm, height, width).zero_()
    for i in range(dm):
        if i > 0:
            cost[:, :channels, i, :, i:] = x[:, :, :, i:]
            cost[:, channels:, i, :, i:] = y[:, :, :, :-i]
        else:
            cost[:, :channels, i, :, :] = x
            cost[:, channels:, i, :, :] = y
    return cost.contiguous()


@pytest.mark.parametrize("shape,dm", [((2, 3, 4, 9), 6), ((1, 32, 10, 26), 65), ((1, 2, 3, 5), 9)])
def test_cost_volume_bit_exact_vs_torch_slices(shape, dm):
    from ganet_b200.modules import GetCostVolume
    torch.manual_seed(0)
    x = torch.randn(shape, device="cuda", requires_grad=True)
    y = torch.randn(shape, device="cuda", requires_grad=True)
    cost = GetCostVolume(dm - 1)(x, y)
    x2, y2 = x.detach().clone().requires_grad_(), y.detach().clone().requires_grad_()
    ref = _ref_cost_volume(x2, y2, dm)
    assert torch.equal(cost, ref)                  # pure copy: bit-exact
    gc = torch.randn_like(cost)
    cost.backward(gc)
    ref.backward(gc)
    assert_close(npy(x.grad), npy(x2.grad), RTOL, "grad_x")
    assert_close(npy(y.grad), npy(y2.grad), RTOL, "grad_y")


@pytest.mark.parametrize("shape", [(2, 7, 3, 5), (1, 193, 12, 40), (1, 1, 2, 2)])
def test_disparity_regression_vs_torch(shape):
    from ganet_b200.modules import DisparityRegression
    torch.manual_seed(1)
    p = torch.softmax(torch.randn(shape, device="cuda"), 1).requires_grad_()
    out = DisparityRegression(shape[1] - 1)(p)
    # modules/GANet.py:145-147 as written
    disp = torch.arange(shape[1], device="cuda", dtype=torch.float32).reshape(1, -1, 1, 1)
    disp = disp.repeat(p.size()[0], 1, p.size()[2], p.size()[3])
    p2 = p.detach().clone().requires_grad_()
    ref = torch.sum(p2 * disp, 1)
    assert_close(npy(out), npy(ref), RTOL, "disparity")
    g = torch.randn_like(out)
    out.backward(g)
    ref.backward(g)
    assert torch.equal(p.grad, p2.grad)


@pytest.mark.parametrize("shape,dm", [((1, 32, 80, 208), 65), ((1, 32, 128, 416), 65)])
def test_cost_volume_at_model_shapes(shape, dm):
    """GetCostVolume at the shapes GANet-11 (240x624) and GANet-deep (384x1248) feed it
    (models/GANet_deep.py:399): bit-exact forward, gradients vs the reference's slice-assign autograd.
    Prints device time and algorithmic DRAM bytes (profiles/r02_volume_ops.txt is this output)."""
    from ganet_b200.modules import GetCostVolume
    torch.manual_seed(2)
    x = torch.randn(shape, device="cuda", requires_grad=True)
    y = torch.randn(shape, device="cuda", requires_grad=True)
    mod = GetCostVolume(dm - 1)
    cost = mod(x, y)
    x2, y2 = x.detach().clone().requires_grad_(), y.detach().clone().requires_grad_()
    ref = _ref_cost_volume(x2, y2, dm)
    assert torch.equal(cost, ref)
    gc = torch.randn_like(cost)
    cost.backward(gc)
    ref.backward(gc)
    assert_close(npy(x.grad), npy(x2.grad), RTOL, "grad_x")
    assert_close(npy(y.grad), npy(y2.grad), RTOL, "grad_y")
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    with torch.no_grad():
        mod(x, y)
    e[0].record()
    for _ in range(10):
        c = mod(x, y)
    e[1].record()
    for _ in range(10):
        torch.autograd.grad(c, (x, y), gc, retain_graph=True)
    e[2].record()
    torch.cuda.synchronize()
    nb = cost.numel() * 4
    print("\nGetCostVolume %s dm=%d: fwd %.3f ms (%.0f GB/s of %d MB written), bwd %.3f ms (%.0f GB/s read)"
          % (shape, dm, e[0].elapsed_time(e[1]) / 10, nb / (e[0].elapsed_time(e[1]) / 10) / 1e6, nb >> 20,
             e[1].elapsed_time(e[2]) / 10, nb / (e[1].elapsed_time(e[2]) / 10) / 1e6))


@pytest.mark.parametrize("shape", [(1, 193, 240, 624), (1, 193, 384, 1248)])
def test_disparity_regression_at_model_shapes(shape):
    """DisparityRegression at full resolution (models/GANet_deep.py:219,247), forward and backward,
    against the reference's repeat * sum lines; prints device time and achieved bandwidth."""
    from ganet_b200.modules import DisparityRegression
    torch.manual_seed(3)
    p = torch.softmax(torch.randn(shape, device="cuda"), 1).requires_grad_()
    mod = DisparityRegression(shape[1] - 1)
    out = mod(p)
    disp = torch.arange(shape[1], device="cuda", dtype=torch.float32).reshape(1, -1, 1, 1)
    disp = disp.repeat(p.size()[0], 1, p.size()[2], p.size()[3])
    p2 = p.detach().clone().requires_grad_()
    ref = torch.sum(p2 * disp, 1)
    assert_close(npy(out), npy(ref), RTOL, "disparity")
    g = torch.randn_like(out)
    out.backward(g)
    ref.backward(g)
    assert torch.equal(p.grad, p2.grad)
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    e[0].record()
    for _ in range(10):
        o = mod(p)
    e[1].record()
    for _ in range(10):
        torch.autograd.grad(o, p, g, retain_graph=True)
    e[2].record()
    torch.cuda.synchronize()
    nb = p.numel() * 4
    print("\nDisparityRegression %s: fwd %.3f ms (%.0f GB/s of %d MB read), bwd %.3f ms (%.0f GB/s written)"
          % (shape, e[0].elapsed_time(e[1]) / 10, nb / (e[0].elapsed_time(e[1]) / 10) / 1e6, nb >> 20,
             e[1].elapsed_time(e[2]) / 10, nb / (e[1].elapsed_time(e[2]) / 10) / 1e6))


LGA_PASSES = [("LgaFunction", 1), ("Lga3Function", 3), ("Lga3d3Function", 3)]


@pytest.mark.parametrize("fname,passes", LGA_PASSES)
def test_lga_1_and_3_pass_functions_through_autograd(ref_values, fname, passes):
    """LgaFunction / Lga3Function (broken upstream: functions/GANet.py:155,241-242) and Lga3d3Function
    through torch.autograd on the GPU, against `passes` chained calls of the reference extension's
    lga_cuda_forward / backward with its accumulate-into-gradFilters contract."""
    import ganet_b200.functions as Fn
    fn = getattr(Fn, fname)
    shape = (1, 2, 6, 9, 12) if "3d" in fname else (2, 6, 9, 12)
    x, f, go = lga_inputs(shape, seed=21 + passes)
    xt, ft = cu(x).requires_grad_(), cu(f).requires_grad_()
    y = fn.apply(xt, ft, 2)
    y.backward(cu(go))
    key = "lga_passes/%s/" % fname
    assert_close_to_golden(y, ref_values, key + "y", RTOL, what=fname + " output")
    assert_close_to_golden(xt.grad, ref_values, key + "gx", RTOL, what=fname + " grad_x")
    assert_close_to_golden(ft.grad, ref_values, key + "gf", RTOL, what=fname + " grad_filters")


# ---- autograd / API behaviour -----------------------------------------------------
def test_sga_module_autograd_matches_oracle():
    from ganet_b200.modules import SGA
    shape = (1, 2, 8, 6, 7)
    x, g, go = sga_inputs(shape, seed=12)
    xt = cu(x).requires_grad_()
    gt = [cu(a).requires_grad_() for a in g]
    out = SGA()(xt, *gt)
    out.backward(cu(go), retain_graph=True)
    gi1 = xt.grad.clone()
    xt.grad = None
    out.backward(cu(go))                     # backward twice: saved state is not clobbered
    assert torch.equal(gi1, xt.grad)
    oo, om = oracle.sga_forward(x, *g, fused=True)
    ogi, ogg, _ = oracle.sga_backward(x, *g, om, go, fused=True)
    assert np.array_equal(npy(out), oo)
    assert_close(npy(gi1), ogi, RTOL, "gradInput")
    for d in range(4):
        assert_close(npy(gt[d].grad) / 2, ogg[d], RTOL, "guidance grad")   # accumulated twice


def test_lga2_backward_leaves_grad_output_intact():
    from ganet_b200.modules import LGA2
    x, f, go = lga_inputs((1, 6, 7, 8), seed=13)
    xt, ft = cu(x).requires_grad_(), cu(f).requires_grad_()
    got = cu(go)
    keep = got.clone()
    LGA2(2)(xt, ft).backward(got)
    assert torch.equal(got, keep)            # the reference overwrites it (functions/GANet.py:199)


def test_non_default_stream_and_threads(ops):
    """The reference launches on legacy stream 0 only; here the current stream is used
    and two host threads may call concurrently (DataParallel pattern)."""
    import threading
    shape = (1, 2, 10, 12, 14)
    x, g, _ = sga_inputs(shape, seed=14)
    oo, om = oracle.sga_forward(x, *g, fused=True)
    results = {}

    def work(i):
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            xt, gt = cu(x), [cu(a) for a in g]
            for _ in range(3):
                out, mask = ops.sga_forward(xt, *gt)
            st.synchronize()
            results[i] = (npy(out), npy(mask))

    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    for i in range(2):
        assert np.array_equal(results[i][0], oo) and np.array_equal(results[i][1], om)


def test_cuda_graph_capture_and_replay(ops):
    """Every launch goes to the current stream and nothing synchronises, so a forward +
    backward can be captured in a CUDA graph and replayed on new data (the reference's
    synchronous cudaMemcpy calls on the legacy stream cannot)."""
    shape = (1, 2, 24, 32, 48)
    x, g, go = sga_inputs(shape, seed=21)
    xs, gs, gos = cu(x), [cu(a) for a in g], cu(go)
    ops.sga_forward(xs, *gs)                       # warm-up outside capture (allocator, tensor maps)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out, mask = ops.sga_forward(xs, *gs)
        gi, gg = ops.sga_backward(xs, *gs, mask, gos)
    x2, g2, go2 = sga_inputs(shape, seed=22)
    xs.copy_(cu(x2)); gos.copy_(cu(go2))
    for dst, src in zip(gs, g2):
        dst.copy_(cu(src))
    graph.replay()
    torch.cuda.synchronize()
    oo, om = oracle.sga_forward(x2, *g2, fused=True)
    ogi, ogg, _ = oracle.sga_backward(x2, *g2, om, go2, fused=True)
    assert np.array_equal(npy(out), oo) and np.array_equal(npy(mask), om)
    assert_close(npy(gi), ogi, RTOL, "gradInput")
    for d in range(4):
        assert_close(npy(gg[d]), ogg[d], RTOL, "guidance grad")


def _pybind_module():
    import glob
    import importlib.util
    hits = sorted(glob.glob(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                         "ganet_b200", "lib", "GANet*.so")))
    if not hits:
        pytest.skip("pybind module not built (python -m ganet_b200.build --pybind)")
    spec = importlib.util.spec_from_file_location("GANet", hits[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_legacy_surface(mod):
    """SGA forward + backward through a module with the reference's native surface, buffers as the
    reference's Python layer allocates them -> out, temp, mask, gradInput, guidance grads, max_idx."""
    shape = (1, 2, 6, 5, 7)
    x, g, go = sga_inputs(shape, seed=15)
    xt, gt, got = cu(x), [cu(a) for a in g], cu(go)
    out, temp, mask = (torch.zeros_like(xt) for _ in range(3))
    assert mod.sga_cuda_forward(xt, *gt, temp, out, mask) == 1
    gi, tg = torch.zeros_like(xt), torch.zeros_like(xt)
    gg = [torch.zeros_like(gt[0]) for _ in range(4)]
    idx = torch.zeros(shape[0], shape[1], shape[3], shape[4], device="cuda")
    assert mod.sga_cuda_backward(xt, *gt, temp.clone(), mask, idx, got, tg, gi, *gg) == 1
    return out, temp, mask, gi, gg, idx


def run_legacy_lga(mod):
    xl, fl, _ = lga_inputs((1, 5, 6, 7), seed=16)
    xl, fl = cu(xl), cu(fl)
    y = torch.zeros_like(xl)
    mod.lga_cuda_forward(xl, fl, y, 2)
    return y


@pytest.mark.parametrize("surface", ["legacy_native", "pybind"])
def test_legacy_native_surface_matches_reference_extension(ref_digests, ref_values, surface):
    """The reference's native module surface -- as Python adapters (ganet_b200.legacy_native) and as the
    compiled pybind11 module `GANet` (csrc/ganet_pybind.cpp) -- honours the reference's buffer contract
    (caller-zeroed buffers, accumulate, fp32 mask, temp_out = left aggregate)."""
    if surface == "pybind":
        mine = _pybind_module()
    else:
        from ganet_b200 import legacy_native as mine
    a = run_legacy_surface(mine)
    for k, t in zip(("out", "temp", "mask"), a[:3]):
        assert digest(t) == ref_digests["legacy_surface/" + k], k
    assert digest(a[5]) == ref_digests["legacy_surface/idx"]
    assert_close_to_golden(a[3], ref_values, "legacy_surface/gi", RTOL, what="gradInput")
    for d in range(4):
        assert_close_to_golden(a[4][d], ref_values, "legacy_surface/gg%d" % d, RTOL, what="guidance grad")
    assert_close_to_golden(run_legacy_lga(mine), ref_values, "legacy_surface/lga", RTOL, what="lga forward")


@needs_ref
def test_reference_python_layer_runs_on_the_pybind_module():
    """The drop-in test of the NATIVE boundary: the reference's OWN libs/GANet/functions/GANet.py and
    modules/GANet.py (copied byte for byte to baseline/_ref/reflibs at build time) import
    `from ..build.lib import GANet` and get this repository's pybind11 module; their SgaFunction and
    Lga2Function -- the reference's buffer allocation, zero-filling and save_for_backward logic, unmodified --
    must then give the reference extension's results."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.exists(os.path.join(root, "baseline", "_ref", "reflibs", "GANet", "functions", "GANet.py")):
        pytest.skip("reference Python layer not copied (oracle/build_ref.py)")
    _pybind_module()
    import sys
    sys.path.insert(0, os.path.join(root, "baseline", "_ref"))
    try:
        from reflibs.GANet.modules.GANet import SGA as RefModuleSGA, LGA2 as RefModuleLGA2
    finally:
        sys.path.remove(os.path.join(root, "baseline", "_ref"))
    shape = (1, 2, 24, 16, 48)
    x, g, go = sga_inputs(shape, seed=23)
    xt = cu(x).requires_grad_()
    gt = [cu(a).requires_grad_() for a in g]
    out = RefModuleSGA()(xt, *gt)                       # reference SgaFunction.forward on our kernels
    out.backward(cu(go))
    ro, rm, rtemp = ref_gpu.sga_forward(cu(x), *[cu(a) for a in g])
    rgi, rgg, _ = ref_gpu.sga_backward(cu(x), *[cu(a) for a in g], rtemp, rm, cu(go))
    assert torch.equal(out.detach(), ro)
    assert_close(npy(xt.grad), npy(rgi), RTOL, "gradInput")
    for d in range(4):
        assert_close(npy(gt[d].grad), npy(rgg[d]), RTOL, "guidance grad %d" % d)
    xl, fl, gol = lga_inputs((1, 9, 10, 16), seed=24)
    xlt, flt = cu(xl).requires_grad_(), cu(fl).requires_grad_()
    y = RefModuleLGA2(2)(xlt, flt)                      # reference Lga2Function on our kernels
    y.backward(cu(gol).clone())                         # (the reference's backward overwrites gradOutput)
    ry, ry1 = ref_gpu.lga2_forward(cu(xl), cu(fl))
    rgx, rgf = ref_gpu.lga2_backward(cu(xl), cu(fl), ry1, cu(gol).clone())
    assert_close(npy(y), npy(ry), RTOL, "LGA2 output")
    assert_close(npy(xlt.grad), npy(rgx), RTOL, "LGA2 grad_x")
    assert_close(npy(flt.grad), npy(rgf), RTOL, "LGA2 grad_filters")


def test_error_reporting(ops):
    x = torch.zeros(1, 1, 2, 3, 4, device="cuda")
    g = torch.zeros(1, 1, 5, 3, 4, device="cuda")
    with pytest.raises(ValueError):
        ops.sga_forward(x, g, g, g, torch.zeros(1, 1, 4, 3, 4, device="cuda"))
    with pytest.raises(TypeError):
        ops.sga_forward(x.double(), g, g, g, g)
    from ganet_b200.functions import SgaFunction
    with pytest.raises(AssertionError):               # the reference's contiguity assert
        SgaFunction.apply(x.transpose(3, 4), g, g, g, g)
