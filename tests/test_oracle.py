"""CPU tests: the oracle (oracle/ganet_oracle.c) against the committed golden
vectors, against the results of the reference's own kernel bodies compiled for the
host (kept as digests in tests/golden/ref_cpu_digests.json), and against the
closed-form properties of SURVEY.md Appendix A.  No GPU needed."""
import os

import numpy as np
import pytest

from oracle import api
from util import GOLD, assert_close, case_id, digest, golden_json, lga_inputs, sga_inputs

SGA_BODY_SHAPES = [(1, 2, 5, 7, 9), (2, 1, 2, 3, 4), (1, 1, 1, 1, 1),
                   (1, 3, 12, 1, 6), (1, 1, 4, 9, 1), (1, 8, 48, 48, 96)]
LGA_BODY_SHAPES = [(1, 4, 6, 7), (2, 1, 3, 3), (1, 2, 1, 8), (2, 2, 3, 4, 5)]


def _ref_cpu():
    return golden_json("ref_cpu_digests.json")


def _check_sga_against_reference(ref, x, g, go):
    """Forward, mask, the left aggregate (the reference's temp_out) and, where `ref` has them, every gradient
    and the depth arg-max, bit for bit against the reference's kernel bodies."""
    oo, om, od = api.sga_forward(x, *g, fused=False, want_dirs=True)
    assert digest(oo) == ref["out"] and digest(om, np.uint8) == ref["mask"]
    assert digest(od[3]) == ref["left"]
    if "gi" in ref:
        ogi, ogg, oidx = api.sga_backward(x, *g, om, go, fused=False)
        assert digest(ogi) == ref["gi"]
        assert all(digest(ogg[k]) == ref["gg%d" % k] for k in range(4))
        assert digest(oidx, np.int32) == ref["idx"]


def _check_lga_against_reference(ref, x, f, go):
    oy, otmp = api.lga_forward(x, f, 2, 2)
    assert digest(oy) == ref["y"] and digest(otmp[0]) == ref["y1"]
    ogx, ogf = api.lga_backward(x, f, otmp, go, 2, 2)
    assert digest(ogx) == ref["gx"] and digest(ogf) == ref["gf"]


def test_sga_against_golden_vectors_bit_exact():
    z = np.load(os.path.join(GOLD, "sga_ref_cpu.npz"))
    for k in range(int(z["n"])):
        x, go = z[f"x{k}"], z[f"go{k}"]
        g = [z[f"g{k}_{d}"] for d in range(4)]
        out, mask, dirs = api.sga_forward(x, *g, fused=False, want_dirs=True)
        assert np.array_equal(out, z[f"out{k}"])
        assert np.array_equal(mask, z[f"mask{k}"])
        assert np.array_equal(dirs[3], z[f"left{k}"])          # reference temp_out = left aggregate
        gi, gg, idx = api.sga_backward(x, *g, mask, go, fused=False)
        assert np.array_equal(gi, z[f"gi{k}"])
        for d in range(4):
            assert np.array_equal(gg[d], z[f"gg{k}_{d}"])
        assert np.array_equal(idx, z[f"idx{k}"])


def test_lga_against_golden_vectors_bit_exact():
    z = np.load(os.path.join(GOLD, "lga_ref_cpu.npz"))
    for k in range(int(z["n"])):
        x, f, go = z[f"x{k}"], z[f"f{k}"], z[f"go{k}"]
        y, tmp = api.lga_forward(x, f, 2, 2)
        assert np.array_equal(y, z[f"y{k}"])
        assert np.array_equal(tmp[0], z[f"y1_{k}"])
        gx, gf = api.lga_backward(x, f, tmp, go, 2, 2)
        assert np.array_equal(gx, z[f"gx{k}"])
        assert np.array_equal(gf, z[f"gf{k}"])


@pytest.mark.parametrize("shape", SGA_BODY_SHAPES)
def test_oracle_equals_reference_kernel_bodies(shape):
    """config 1 of BASELINE.json is the last shape: SGA on 1x8x48x48x96, CPU only."""
    x, g, go = sga_inputs(shape, seed=sum(shape))
    ref = _ref_cpu()["sga_kernel_bodies"][case_id(shape)]
    assert ("gi" in ref) == (np.prod(shape) < 200000)
    _check_sga_against_reference(ref, x, g, go)


@pytest.mark.parametrize("shape", LGA_BODY_SHAPES)
def test_oracle_lga_equals_reference_kernel_bodies(shape):
    x, f, go = lga_inputs(shape, seed=3)
    _check_lga_against_reference(_ref_cpu()["lga_kernel_bodies"][case_id(shape)], x, f, go)


def test_golden_sample_catches_an_error_in_one_slice():
    """assert_close_to_golden on a tensor kept as a sample: an error of 1 % of the scale confined to the last depth
    plane of gradInput (what a wrong tail of the D > 288 line kernels would give) is caught, the exact tensor and one
    within rounding distance of it pass."""
    from util import assert_close_to_golden, sampled
    shape = (1, 2, 513, 3, 5)
    x, g, go = sga_inputs(shape, seed=3 + sum(shape))
    _, mask = api.sga_forward(x, *g, fused=True)
    gi, _, _ = api.sga_backward(x, *g, mask, go, fused=True)
    vals, scale = sampled(gi)
    assert vals.size < gi.size
    gold = {"gi": vals, "gi/scale": scale}
    assert_close_to_golden(gi, gold, "gi")
    assert_close_to_golden(gi * np.float32(1 + 1e-6), gold, "gi")
    bad = gi.copy()
    bad[:, :, -1] += np.float32(0.01 * scale)
    with pytest.raises(AssertionError):
        assert_close_to_golden(bad, gold, "gi")


def test_fused_rounding_differs_only_in_last_bits():
    x, g, _ = sga_inputs((1, 2, 9, 12, 10), seed=5)
    a, ma = api.sga_forward(x, *g, fused=False)
    b, mb = api.sga_forward(x, *g, fused=True)
    assert np.abs(a - b).max() < 1e-5
    assert (ma != mb).mean() < 0.01


def test_constant_input_ties_keep_lowest_direction_and_depth():
    """Constant x and identical weights make all four aggregates equal everywhere:
    Max keeps direction 0 (GANet_kernel.cu:31 strict <) and MaxDepth keeps depth 0."""
    N, C, D, H, W = 1, 2, 4, 5, 6
    x = np.full((N, C, D, H, W), 0.75, np.float32)
    g = [np.full((N, C, 5, H, W), 0.2, np.float32) for _ in range(4)]
    out, mask = api.sga_forward(x, *g)
    assert (mask == 0).all()
    go = np.ones_like(x)
    _, _, idx = api.sga_backward(x, *g, mask, go)
    assert (idx == 0).all()


def test_direction_geometry_by_flips():
    """up(x) == flipH(down(flipH x)), left(x) == flipW(right(flipW x)),
    right(x) == transpose(down(transpose x))."""
    x, g, _ = sga_inputs((1, 2, 5, 6, 7), seed=11)
    _, _, d = api.sga_forward(x, g[0], g[0], g[0], g[0], fused=False, want_dirs=True)
    xf = np.ascontiguousarray(x[:, :, :, ::-1]); gf = np.ascontiguousarray(g[0][:, :, :, ::-1])
    _, _, df = api.sga_forward(xf, gf, gf, gf, gf, fused=False, want_dirs=True)
    assert np.array_equal(d[1], df[0][:, :, :, ::-1])
    xw = np.ascontiguousarray(x[..., ::-1]); gw = np.ascontiguousarray(g[0][..., ::-1])
    _, _, dw = api.sga_forward(xw, gw, gw, gw, gw, fused=False, want_dirs=True)
    assert np.array_equal(d[3], dw[2][..., ::-1])
    xt = np.ascontiguousarray(x.swapaxes(3, 4)); gt = np.ascontiguousarray(g[0].swapaxes(3, 4))
    _, _, dt = api.sga_forward(xt, gt, gt, gt, gt, fused=False, want_dirs=True)
    assert np.array_equal(d[2], dt[0].swapaxes(3, 4))


def test_first_step_gradient_quirk():
    """Appendix A.3: with a single scan step per direction irrelevant, check the
    H=1 case by hand: down/up have T=1, so gradInput gets only T*w0 (+ depth-edge
    terms) from them and their w1..w4 gradients are exactly zero."""
    x, g, go = sga_inputs((1, 1, 3, 1, 4), seed=2)
    _, mask = api.sga_forward(x, *g)
    gi, gg, _ = api.sga_backward(x, *g, mask, go)
    for d in (0, 1):                       # vertical directions have one scan step
        assert np.all(gg[d][:, :, 1:] == 0)
        sel = (mask == d) * go
        assert np.allclose(gg[d][:, :, 0], (sel * x).sum(2), rtol=1e-5, atol=1e-6)


def test_lga_backward_is_the_adjoint():
    """<go, J v> == <J^T go, v> for the data path and the filter path."""
    rng = np.random.default_rng(0)
    x, f, go = lga_inputs((2, 5, 6, 7), seed=4)
    v = rng.standard_normal(x.shape).astype(np.float32)
    vf = rng.standard_normal(f.shape).astype(np.float32)
    y_v, _ = api.lga_forward(v, f, 2, 1)
    gx, gf = api.lga_backward(x, f, None, go, 2, 1)
    assert abs((go.astype(np.float64) * y_v).sum() - (gx.astype(np.float64) * v).sum()) < 1e-3
    y_vf, _ = api.lga_forward(x, vf, 2, 1)       # LGA is linear in the filters too
    assert abs((go.astype(np.float64) * y_vf).sum() - (gf.astype(np.float64) * vf).sum()) < 1e-3


def test_lga_out_of_range_taps_use_centre_voxel():
    """A 1x1x1 volume: every one of the 75 taps falls back to the centre voxel."""
    x = np.array([[[[2.0]]]], np.float32)
    f = np.arange(75, dtype=np.float32).reshape(1, 75, 1, 1) / 100
    y, _ = api.lga_forward(x, f, 2, 1)
    assert np.isclose(y[0, 0, 0, 0], 2.0 * f.sum(), rtol=1e-6)


def test_cost_volume_matches_slice_definition():
    """modules/GANet.py:125-131 restated with numpy slicing."""
    rng = np.random.default_rng(1)
    N, C, H, W, Dm = 2, 3, 4, 9, 6
    x = rng.standard_normal((N, C, H, W)).astype(np.float32)
    y = rng.standard_normal((N, C, H, W)).astype(np.float32)
    ref = np.zeros((N, 2 * C, Dm, H, W), np.float32)
    for i in range(Dm):
        if i > 0:
            ref[:, :C, i, :, i:] = x[:, :, :, i:]
            ref[:, C:, i, :, i:] = y[:, :, :, :-i]
        else:
            ref[:, :C, i] = x
            ref[:, C:, i] = y
    cost = api.cost_volume_forward(x, y, Dm)
    assert np.array_equal(cost, ref)
    gc = rng.standard_normal(cost.shape).astype(np.float32)
    gx, gy = api.cost_volume_backward(gc)
    # adjoint identity
    lhs = (gc.astype(np.float64) * cost).sum()
    rhs = (gx.astype(np.float64) * x).sum() + (gy.astype(np.float64) * y).sum()
    assert abs(lhs - rhs) < 1e-3


def test_cost_volume_wider_than_image():
    """maxdisp+1 > W: planes i >= W are all zero (the reference's empty slices)."""
    x = np.ones((1, 1, 2, 3), np.float32)
    cost = api.cost_volume_forward(x, x, 5)
    assert cost[:, :, 3:].sum() == 0 and cost[0, 0, 2, 0].tolist() == [0, 0, 1]


def test_disparity_regression():
    rng = np.random.default_rng(2)
    p = rng.random((2, 7, 3, 5)).astype(np.float32)
    p /= p.sum(1, keepdims=True)
    d = api.disp_regression_forward(p)
    ref = (p.astype(np.float64) * np.arange(7).reshape(1, 7, 1, 1)).sum(1)
    assert np.allclose(d, ref, rtol=1e-5, atol=1e-6)
    g = rng.standard_normal((2, 3, 5)).astype(np.float32)
    gp = api.disp_regression_backward(g, 7)
    assert np.array_equal(gp, g[:, None] * np.arange(7, dtype=np.float32).reshape(1, 7, 1, 1))


# ---- size-independent properties of the path (the ones test_gpu_fullsize.py relies on) ------
@pytest.mark.parametrize("fused", [False, True])
def test_power_of_two_scaling_is_exact(fused):
    """Every operation of the recurrence is a multiply, add, fma or max: scaling x (and the
    incoming gradient) by 2^k scales every result by 2^k bit for bit and leaves the direction
    mask and the depth arg-max untouched."""
    x, g, go = sga_inputs((1, 2, 9, 6, 7), seed=21)
    out, mask = api.sga_forward(x, *g, fused=fused)
    gi, gg, idx = api.sga_backward(x, *g, mask, go, fused=fused)
    out8, mask8 = api.sga_forward(8.0 * x, *g, fused=fused)
    assert np.array_equal(out8, 8.0 * out) and np.array_equal(mask8, mask)
    gi4, gg4, idx4 = api.sga_backward(8.0 * x, *g, mask, 0.5 * go, fused=fused)
    assert np.array_equal(gi4, 0.5 * gi) and np.array_equal(idx4, idx)
    # guidance gradients are bilinear in (gradOut, x / A): 0.5 * 8 = 4
    assert all(np.array_equal(a, 4.0 * b) for a, b in zip(gg4, gg))


def test_depth_flip_symmetry():
    """Flipping the depth axis and exchanging the d-1 / d+1 weights (w2 <-> w3) flips the result."""
    x, g, _ = sga_inputs((1, 2, 8, 5, 6), seed=22)
    out, mask = api.sga_forward(x, *g, fused=False)
    gs = [np.ascontiguousarray(a[:, :, [0, 1, 3, 2, 4]]) for a in g]
    outf, maskf = api.sga_forward(np.ascontiguousarray(x[:, :, ::-1]), *gs, fused=False)
    assert_close(outf[:, :, ::-1], out, 1e-5, "depth-flipped forward")
    assert (maskf[:, :, ::-1] != mask).mean() < 0.01        # only fp32 near-ties may flip


def test_slices_are_independent():
    """Nothing couples different (n, c): a batch equals its slices computed alone (what lets the
    path shard over the batch with no collective, and the native side chunk its workspace)."""
    x, g, go = sga_inputs((2, 3, 5, 4, 6), seed=23)
    out, mask = api.sga_forward(x, *g)
    gi, gg, idx = api.sga_backward(x, *g, mask, go)
    for n in range(2):
        for c in range(3):
            sl = (slice(n, n + 1), slice(c, c + 1))
            o1, m1 = api.sga_forward(x[sl], *[a[sl] for a in g])
            assert np.array_equal(o1, out[sl]) and np.array_equal(m1, mask[sl])
            gi1, gg1, idx1 = api.sga_backward(x[sl], *[a[sl] for a in g], m1, go[sl])
            assert np.array_equal(gi1, gi[sl]) and np.array_equal(idx1, idx[sl])
            assert all(np.array_equal(a, b[sl]) for a, b in zip(gg1, gg))


# ---- randomised shapes against the reference's own kernel bodies ----------------------------
def test_oracle_equals_reference_kernel_bodies_on_random_shapes():
    """Ragged and degenerate volumes (any of D, H, W down to 1), 30 seeded shapes: forward, mask, all gradients
    and the depth arg-max bit for bit against the reference's kernel bodies compiled for the host."""
    cases = _ref_cpu()["sga_random"]
    assert len(cases) == 30 and {tuple(c["shape"]) for c in cases} >= {(1, 1, 1, 1, 1), (2, 3, 13, 9, 9)}
    for c in cases:
        x, g, go = sga_inputs(tuple(c["shape"]), seed=c["seed"])
        _check_sga_against_reference(c, x, g, go)


def test_oracle_lga_equals_reference_kernel_bodies_on_random_shapes():
    cases = _ref_cpu()["lga_random"]
    assert len(cases) == 20
    for c in cases:
        x, f, go = lga_inputs(tuple(c["shape"]), seed=c["seed"])
        _check_lga_against_reference(c, x, f, go)
