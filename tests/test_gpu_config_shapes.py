"""GPU parity at the EXACT shapes BASELINE.json's configs put on the hot path (SURVEY.md
Appendix B), against the UNMODIFIED reference CUDA extension run on the same seeded inputs
(tests/golden/ref_cuda_*, written by tests/golden/make_golden.py --cuda on a B200) -- so even
the headline microbench sample is compared with the reference rather than through properties:

  config 2 (GANet-11, 240x624)      SGA 1x32x65x80x208 (M3), 1x48x33x40x104 (M6); LGA2 1x193x240x624
  config 3 (GANet-deep, 384x1248)   SGA 1x32x65x128x416 (K3), 1x48x33x64x208 (K6); LGA2 1x193x384x1248
  config 4 (training step)          the shapes of config 2, forward and backward
  config 5 (microbench sweep)       SGA 1x32x{96,192}x240x624 and 1x16x288x240x624 (the reference
                                    indexes with int: one call must stay below 2^31 elements),
                                    LGA2 1x{96,192,288}x240x624

Criteria (SURVEY.md 8c): SGA forward values, direction mask and depth arg-max bit-exact
(SHA-256 digests of the reference's results); gradients and LGA within 1e-4 relative fp32
(max|a-b| / max|b| and allclose(rtol=1e-4, atol=1e-5 * scale) at the sample positions the
golden file keeps, and the largest magnitudes).  Both backward variants (recompute / kept
aggregates) are checked.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from util import assert_close_to_golden, digest, golden_json, golden_values

pytestmark = pytest.mark.gpu
RTOL = 1e-4          # north_star: 1e-4 relative fp32

SGA_CONFIG_SHAPES = {
    "M3": (1, 32, 65, 80, 208), "M6": (1, 48, 33, 40, 104),
    "K3": (1, 32, 65, 128, 416), "K6": (1, 48, 33, 64, 208),
    "sweep_D96": (1, 32, 96, 240, 624), "headline_D192": (1, 32, 192, 240, 624),
    "sweep_D288": (1, 16, 288, 240, 624),
}
LGA_CONFIG_SHAPES = {
    "L": (1, 193, 240, 624), "L_kitti": (1, 193, 384, 1248),
    "sweep_D96": (1, 96, 240, 624), "headline_D192": (1, 192, 240, 624), "sweep_D288": (1, 288, 240, 624),
}


def _need(nbytes):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip("needs %.0f GB of free device memory" % (nbytes / 2 ** 30))


def _close(a, gold, key, what):
    """SURVEY.md 8c, both halves: per-tensor max|a-b| / max|b| <= 1e-4 AND the element-wise
    allclose(rtol=1e-4, atol=1e-5 * scale)."""
    assert_close_to_golden(a, gold, key, RTOL, atol=1e-5, what=what)


def sga_config_inputs(shape):
    N, C, D, H, W = shape
    torch.manual_seed(11 + D)
    x = torch.randn(shape, device="cuda")
    g = [F.normalize(torch.randn(N, C, 5, H, W, device="cuda"), p=1, dim=2) for _ in range(4)]
    go = torch.randn(shape, device="cuda")
    return x, g, go


def lga_config_inputs(shape):
    N, D, H, W = shape
    torch.manual_seed(5 + D)
    x = torch.randn(shape, device="cuda")
    f = F.normalize(torch.randn(N, 75, H, W, device="cuda"), p=1, dim=1)
    go = torch.randn(shape, device="cuda")
    return x, f, go


@pytest.fixture(scope="module")
def ops():
    from ganet_b200 import ops as o
    return o


@pytest.fixture(scope="module")
def ref_digests():
    return golden_json("ref_cuda_digests.json")


@pytest.fixture(scope="module")
def ref_values():
    return golden_values("ref_cuda_values.npz")


@pytest.mark.parametrize("name", list(SGA_CONFIG_SHAPES))
def test_sga_config_shape_vs_reference_cuda(ops, ref_digests, ref_values, name):
    shape = SGA_CONFIG_SHAPES[name]
    N, C, D, H, W = shape
    numel = N * C * D * H * W
    assert numel < 2 ** 31
    _need(70 * numel)                 # ~17 volumes live at the peak
    x, g, go = sga_config_inputs(shape)
    key = "config_sga/%s/" % name

    out, mask = ops.sga_forward(x, *g)
    assert digest(out) == ref_digests[key + "out"], "SGA forward values are not bit-identical"
    assert digest(mask) == ref_digests[key + "mask"], "direction mask differs"        # as float32, like the reference's
    out2, mask2, agg = ops.sga_forward(x, *g, keep_aggregates=True)
    assert torch.equal(out2, out) and torch.equal(mask2, mask)
    del out, mask, out2

    gi, gg, idx = ops.sga_backward(x, *g, mask2, go, want_max_idx=True)
    assert digest(idx, np.int32) == ref_digests[key + "idx"], "depth arg-max differs"
    _close(gi, ref_values, key + "gi", "gradInput")
    for k in range(4):
        _close(gg[k], ref_values, key + "gg%d" % k, "guidance gradient %d" % k)
    gi2, gg2 = ops.sga_backward(x, *g, mask2, go, aggregates=agg)
    assert torch.equal(gi2, gi) and all(torch.equal(a, b) for a, b in zip(gg2, gg))


@pytest.mark.parametrize("name", list(LGA_CONFIG_SHAPES))
def test_lga2_config_shape_vs_reference_cuda(ops, ref_values, name):
    x, f, go = lga_config_inputs(LGA_CONFIG_SHAPES[name])
    key = "config_lga2/%s/" % name
    y1 = ops.lga_forward(x, f, 2)
    y = ops.lga_forward(y1, f, 2)
    _close(y1, ref_values, key + "y1", "LGA pass 1")
    _close(y, ref_values, key + "y", "LGA2 output")
    g1, gf = ops.lga_backward(y1, f, go, 2)
    gx, gf = ops.lga_backward(x, f, g1, 2, gf)
    _close(gx, ref_values, key + "gx", "LGA2 grad_x")
    _close(gf, ref_values, key + "gf", "LGA2 grad_filters")
